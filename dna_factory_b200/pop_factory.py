"""pop_factory on the B200 path: same command line, same input / output files as ochrzan/dna-factory.

What stays host Python (cold, O(samples) or O(SNPs) bookkeeping the reference also does in Python):
  argument parsing                      pop_factory.py:638-670   (ArgParserTest pins the flag -> attribute map)
  SnpFactory / snps.json.gz             pop_factory.py:136-193,258-272      -> dna_factory_b200.snp
  DeleteriousGroup / deleterious.json   pop_factory.py:515-635
  .fam / pop_deleterious.txt            pop_factory.py:341-383, SampleInfo :47-71
  VCF header                            pop_factory.py:36-44
What moves to the GPU: write_vcf_snps (pop_factory.py:417-469) -- the worker pool, the row loop
queue_vcf_snps (:471-513) and the BgzfWriter behind `file.write` -- through dna_factory_b200._native.

Random streams: host-side draws use numpy's global RandomState and Python's `random` in the reference's
order, so a run seeded like the reference selects the same SNPs, deleterious sets, sexes and mutations.
Genotype draws use the counter-based Philox stream (DESIGN.md 3) keyed by --seed (default: the same
HHMMSS clock value the reference seeds numpy with).
"""
import argparse
import gc
import json
import os
import random
import sys
import threading
import time
from datetime import datetime

import numpy

from . import _native, assoc, fisher, model, mperm, partition, host
from . import tabix
from .tabix import TabixBuilder
from .snp import (CHROMOSOME_LIST, CHROMOSOME_MAX_POSITION, CHROMOSOME_PROB, SNPTuples, SnpFactory, SnpTable,  # noqa: F401
                  is_haploid, split_list, stripe_list)

MIN_SNP_FREQ = 0.005
MIN_TOTAL_COUNT = 1000
OUTPUT_DIR = os.path.join(os.getcwd(), "populations")
BED_MAGIC = b"\x6c\x1b\x01"     # PLINK 1 .bed, SNP-major


def validate_biallelic_table(table, flag, what):
    """`flag` needs a column-form SNP table (SnpTable) without rows of more than 2 alleles: checked before the VCF is
    written, so a table the output cannot hold fails at once instead of after the whole generation."""
    if not isinstance(table, SnpTable):
        raise ValueError("%s needs SNP records that fit the column form (integer ids, one-letter alleles)" % flag)
    bad = numpy.nonzero(table.n_alleles > 2)[0]
    if len(bad):
        raise ValueError("%s: SNP rs%d (row %d) has %d alleles; %s" % (
            flag, int(table.ids[bad[0]]), int(bad[0]), int(table.n_alleles[bad[0]]), what))


def validate_bed_table(table):
    validate_biallelic_table(table, "--bed", "PLINK 1 .bed / .bim hold biallelic SNPs only")


def validate_assoc_table(table):
    validate_biallelic_table(table, "--assoc", "the allelic test counts biallelic SNPs only")


def validate_assoc_population(control_size, test_size, flag="--assoc"):
    """--assoc, --model, --fisher and --mperm compare cases with controls: both groups must be non-empty."""
    if control_size <= 0 or test_size <= 0:
        raise ValueError("%s needs cases and controls (-s %d, -c %d)" % (flag, test_size, control_size))


def gen_vcf_header(fam_data):
    lines = ["##fileformat=VCFv4.3",
             "##filedate=%s" % datetime.now().strftime("%Y%m%d %H:%M"),
             "##source=PopFactory",
             '##FILTER=<ID=q10,Description="Quality below 10">',
             '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
             "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(str(s.person_id) for s in fam_data)]
    return "\n".join(lines) + "\n"


class SampleInfo:
    """One row of the .fam file plus the sample's deleterious SNP set."""

    def __init__(self, family_id, person_id, father_id, mother_id, sex: int, is_control: bool, deleterious_snps: dict):
        assert person_id
        self.person_id = person_id
        self.family_id = family_id
        self.father_id = father_id
        self.mother_id = mother_id
        self.sex = sex
        self.is_control = is_control
        self.deleterious_snps = deleterious_snps

    def to_fam_format(self):
        return "%i\t%i\t%i\t%i\t%i\t%i\t\n" % (self.family_id, self.person_id, self.father_id, self.mother_id, self.sex,
                                               1 if self.is_control else 2)

    def is_male(self):
        return self.sex == 1


class BgzfSink:
    """Stand-in for the Bio.bgzf.BgzfWriter the reference opens at pop_factory.py:403: text handed to
    write() is buffered and BGZF-encoded on the GPU; write_blocks() appends ready-made BGZF blocks."""

    def __init__(self, filename, engine, compresslevel=6, index=False):
        self._handle = open(filename, "wb")
        self._engine = engine
        self._pending = []
        self.compresslevel = compresslevel
        self.index = TabixBuilder() if index else None   # block + row table of everything appended (--tbi)

    def write(self, data):
        self._pending.append(data.encode("latin-1") if isinstance(data, str) else bytes(data))

    def flush(self):
        if self._pending:
            blob, _ = self._engine.bgzf_compress(b"".join(self._pending))
            self._pending = []
            self._handle.write(blob)
            if self.index is not None:
                self.index.add_blocks(*_native.bgzf_scan(blob))
        self._handle.flush()

    def write_blocks(self, blob):
        self.flush()
        self._handle.write(blob)
        if self.index is not None:
            self.index.add_blocks(*_native.bgzf_scan(blob))

    def close(self):
        self.flush()
        self._handle.write(_native.bgzf_eof())
        self._handle.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class DeleteriousGroup:
    def __init__(self, name, population_weight):
        self.deleterious = {}
        self.name = name
        self.population_weight = population_weight

    @classmethod
    def snp_ids_from_list(cls, snp_data, min_minor_allele_freq=0, max_minor_allele_freq=1):
        """Ids of the candidate SNPs (pop_factory.py:549-558); snp_data is a SnpTable or a list of SNPTuples."""
        filtering = min_minor_allele_freq > 0 or max_minor_allele_freq < 0.5
        if isinstance(snp_data, SnpTable):
            if not filtering:
                return snp_data.ids.tolist()
            maf = snp_data.minor_allele_freq()
            keep = (min_minor_allele_freq <= maf) & (maf <= max_minor_allele_freq)
            return snp_data.ids[keep].tolist()
        if not filtering:
            return [s.id for s in snp_data]
        return [s.id for s in snp_data
                if min_minor_allele_freq <= (s.minor_allele_tuple()[1] - s.ref_allele_tuple()[1]) <= max_minor_allele_freq]

    @classmethod
    def init_with_snps(cls, name, mutation_weights, snp_id_list, population_weight):
        group = cls(name, population_weight)
        if not snp_id_list:
            raise Exception("No SNPs in list to choose from. SNPs must have all been filtered out by deleterious config.")
        picked = numpy.random.choice(a=snp_id_list, size=len(mutation_weights), replace=False)
        for snp_id, weight in zip(picked, mutation_weights):
            group.deleterious[int(snp_id)] = weight
        return group

    @classmethod
    def from_yml(cls, yml_attr, snp_data, name):
        bounds = {"min_minor_allele_freq": 0, "max_minor_allele_freq": 1}
        for key in bounds:
            if yml_attr.get(key):
                if not 0 < yml_attr[key] < 0.5:
                    raise Exception("%s must be between 0 and 0.5. yml value = %s" % (key, yml_attr[key]))
                bounds[key] = yml_attr[key]
        instances = int(yml_attr["num_instances"]) if yml_attr.get("num_instances") else 1
        candidates = cls.snp_ids_from_list(snp_data, bounds["min_minor_allele_freq"], bounds["max_minor_allele_freq"])
        return [cls.init_with_snps("%s-%s" % (name, i), yml_attr["mutation_weights"], candidates,
                                   yml_attr["population_weight"]) for i in range(instances)]

    def to_json(self):
        return json.dumps(vars(self))

    @classmethod
    def from_json(cls, json_line):
        rec = json.loads(json_line)
        group = cls(rec["name"], rec["population_weight"])
        group.deleterious.update(rec["deleterious"])     # keys stay strings, as upstream (SURVEY R8)
        return group

    def select_mutations(self):
        """Shuffle the group's SNPs and take them until the weights add up to 1 (pop_factory.py:621-635)."""
        shuffled = list(self.deleterious.items())
        random.shuffle(shuffled)
        chosen, total = {}, 0
        for snp_id, weight in shuffled:
            chosen[snp_id] = weight
            total += weight
            if total >= 1:
                break
        return chosen


class PopulationFactory:
    def __init__(self, num_processes=1, generate_snps=False, male_odds=0.5, deleterious_config=None,
                 deleterious_list_path=None, sample_id_offset=0, snps_path=None, output_path=None, seed=None,
                 gpus=1, gpu_select=False, tbi=False, bed=False, assoc=False, model=False,
                 hardy=False, fisher=False, mperm=None):
        self.deleterious = {}
        self.ordered_snps = []
        self.snp_table = None
        self.snp_count = 0
        if output_path:
            self.population_dir = output_path if output_path.endswith(os.path.sep) else output_path + os.path.sep
        else:
            self.population_dir = os.path.join(OUTPUT_DIR, datetime.now().strftime("%Y%m%d%H%M")) + os.path.sep
        self.male_odds = male_odds
        self.num_processes = num_processes if num_processes > 0 else 1   # kept for CLI parity; the GPU path ignores it
        self.generate_snps = generate_snps
        self.deleterious_config = deleterious_config
        self.sample_id_offset = sample_id_offset or 0
        self.deleterious_list_path = deleterious_list_path
        self.snps_path = snps_path
        self.seed = seed
        self.gpus = max(1, gpus or 1)
        self.gpu_select = bool(gpu_select)
        self.tbi = bool(tbi)
        self.bed = bool(bed)
        self.stats = []
        self.bed_stats = []      # dnaf_stats of the .bed calls (--bed)
        self.assoc = bool(assoc)
        self.assoc_counts = None     # uint32[rows, 4] allele counts of the last write_vcf_snps (--assoc)
        self.override_rows = None    # global row of every override pair of the last write_vcf_snps
        self.model = bool(model)
        self.hardy = bool(hardy)
        self.geno_counts = None      # uint32[rows, 10] genotype counts of the last write_vcf_snps (--model / --hardy)
        self.hwe_p = None            # float64[rows, 3] Hardy-Weinberg exact P (ALL, AFF, UNAFF) of the same rows
        self.fisher = bool(fisher)
        self.fisher_log10p = None    # float64[rows, 4] Fisher log10 P (GENO, ALLELIC, DOM, REC) of the same rows (--fisher)
        self.mperm = mperm           # permutations of --mperm (None: no permutation tests)
        self.mperm_result = None     # (T_obs [rows, 2], exceedances [rows, 2], maxima [N, 2]) of ALLELIC and REC (--mperm)

    # ------------------------------------------------------------------------------------------ orchestration
    def generate_population(self, control_size, test_size, min_freq, max_snps, compression_level=6):
        t0 = time.time()
        if self.assoc:
            validate_assoc_population(control_size, test_size)
        if self.model:
            validate_assoc_population(control_size, test_size, "--model")
        if self.fisher:
            validate_assoc_population(control_size, test_size, "--fisher")
        if self.mperm is not None:
            if self.mperm < 1:
                raise ValueError("--mperm needs at least 1 permutation (got %d)" % self.mperm)
            validate_assoc_population(control_size, test_size, "--mperm")
        clock_seed = int(datetime.now().strftime("%H%M%S"))
        numpy.random.seed(clock_seed)
        if self.seed is None:
            self.seed = clock_seed
        os.makedirs(self.population_dir, exist_ok=True)
        presorted = False
        if self.snps_path:
            self.load_snps_file()
        elif self.generate_snps and self.gpu_select:
            # SnpFactory.random_snp_tuples + the sort of pop_factory.py:245 on the GPU, keyed by --seed
            with _native.Engine(0) as eng:
                self.snp_table = SnpFactory.init_from_cdf_file().random_snp_table_device(eng, max_snps, self.seed,
                                                                                         min_maf=min_freq)
            presorted = True
        elif self.generate_snps:
            self.snp_table = SnpFactory.init_from_cdf_file().random_snp_table(max_snps, min_maf=min_freq)
        else:
            self.load_snps_db(min_freq, max_snps)
        if self.snp_table is not None:
            if not presorted:
                self.snp_table = self.snp_table.sorted()
        else:
            self.ordered_snps.sort(key=lambda x: (x.chromosome, x.position))
        if not self.snps_path:
            self.output_snps()
        gc.collect()
        if self.deleterious_list_path:
            self.load_deleterious()
        else:
            self.pick_deleterious_snps(self.snp_table if self.snp_table is not None else self.ordered_snps,
                                       self.deleterious_config)
        self.output_vcf_population(control_size, test_size, self.male_odds, compression_level)
        print("Finished Generating Population in {:0.4f} secs.".format(time.time() - t0))

    def _n_snps(self):
        return len(self.snp_table) if self.snp_table is not None else len(self.ordered_snps)

    def output_snps(self):
        t0 = time.time()
        table = self.snp_table if self.snp_table is not None else SnpTable.from_snps(self.ordered_snps)
        table.write_json_gz(self.population_dir + "snps.json.gz", compresslevel=5)
        print("Time to write snps file {:0.4f} seconds".format(time.time() - t0))

    def load_snps_file(self):
        self.snp_table = SnpTable.read_json_gz_table(self.snps_path)   # native parser, columns only
        if self.snp_table is not None:
            self.snp_count = len(self.snp_table)
            return
        self.ordered_snps = SnpTable.read_json_gz(self.snps_path)
        self.snp_count = len(self.ordered_snps)
        try:
            self.snp_table = SnpTable.from_snps(self.ordered_snps)
        except ValueError:
            self.snp_table = None      # exotic records (string ids, multi-character alleles): keep the object list

    def load_snps_db(self, min_freq, max_snps):
        raise NotImplementedError("-l (RefSNP database mode, pop_factory.py:274-311) needs the reference's SQL "
                                  "database layer, which is outside the B200 hot path; export snps.json.gz with the "
                                  "reference and pass it with --snps_file")

    @classmethod
    def pick_deleterious_groups(cls, deleterious_groups, pop_size):
        groups = list(deleterious_groups)
        return random.choices(population=groups, weights=[g.population_weight for g in groups], k=pop_size)

    def generate_fam_file(self, control_size, test_size, male_odds, deleterious_group_list):
        control_id = 100000 + self.sample_id_offset
        test_id = 500000 + self.sample_id_offset
        rolls = numpy.random.rand(control_size + test_size)
        samples = []
        with open(self.population_dir + "population.fam", "w") as fam, \
                open(self.population_dir + "pop_deleterious.txt", "w") as pop_del:
            for i in range(control_size + test_size):
                is_control = i < control_size
                sex_code = 1 if rolls[i] <= male_odds else 2
                if is_control:
                    control_id += 1
                    iid, chosen = control_id, None
                else:
                    test_id += 1
                    iid = test_id
                    group = deleterious_group_list[i - control_size]
                    chosen = group.select_mutations()
                    pop_del.write("%i\t%s\t" % (test_id, group.name) + "\t".join("rs" + str(k) for k in chosen) + "\n")
                sample = SampleInfo(i + 1 + self.sample_id_offset * 2, iid, 0, 0, sex_code, is_control, chosen)
                samples.append(sample)
                fam.write(sample.to_fam_format())
        return samples

    def output_vcf_population(self, control_size, test_size, male_odds, compression_level):
        if not self._n_snps():
            raise Exception("No SNPs to Process! Exiting.")
        snps = self.snp_table if self.snp_table is not None else self.ordered_snps
        if self.bed:
            validate_bed_table(snps)
        if self.assoc:
            validate_assoc_table(snps)
        if self.model:
            validate_biallelic_table(snps, "--model", "the genotypic tests count biallelic SNPs only")
        if self.hardy:
            validate_biallelic_table(snps, "--hardy", "the Hardy-Weinberg tests count biallelic SNPs only")
        if self.fisher:
            validate_biallelic_table(snps, "--fisher", "the Fisher exact tests count biallelic SNPs only")
        if self.mperm:
            validate_biallelic_table(snps, "--mperm", "the permutation tests count biallelic SNPs only")
        groups = PopulationFactory.pick_deleterious_groups(list(self.deleterious.values()), test_size)
        fam_data = self.generate_fam_file(control_size, test_size, male_odds, groups)
        main_file = self.population_dir + "population.vcf.gz"
        self._level = compression_level
        engine = _native.Engine(0)
        bed_fd = None
        try:
            if self.bed:
                # population.bed / .bim beside population.fam: `plink --bfile population` reads the same population
                bed_fd = os.open(self.population_dir + "population.bed", os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
                os.write(bed_fd, BED_MAGIC)
            with BgzfSink(main_file, engine, compresslevel=compression_level, index=self.tbi) as f:
                f.write(gen_vcf_header(fam_data))
                print("Outputing VCF lines", flush=True)
                # the reference cuts the list into ~1 M-SNP chunks to bound its memory (pop_factory.py:402-413);
                # the GPU path streams, so one call covers the whole list
                self.write_vcf_snps(fam_data, snps, f, engine=engine, bed_fd=bed_fd)
                print("%s Finished work chunk 1 of 1." % datetime.now().strftime("%Y-%m-%d %H:%M"), flush=True)
            if self.tbi:
                # what `bcftools index -t` (README.md:98-99) would derive by inflating the file again
                blob, _ = engine.bgzf_compress(f.index.payload())
                with open(main_file + ".tbi", "wb") as t:
                    t.write(blob + _native.bgzf_eof())
            if self.bed:
                with open(self.population_dir + "population.bim", "wb") as b:
                    b.write(snps.bim_bytes())
            if self.assoc:
                self.output_assoc(snps)
            if self.model or self.hardy:
                self.output_model(snps)
            if self.fisher:
                self.output_fisher(snps)
            if self.mperm:
                self.output_mperm(snps)
        finally:
            engine.close()
            if bed_fd is not None:
                os.close(bed_fd)
        print("Finished VCF file output.", flush=True)

    def output_assoc(self, table):
        """population.assoc (the allelic test of every SNP) and deleterious_assoc.txt (how the planted SNPs fare) from
        the allele counts write_vcf_snps took on the GPU."""
        with open(self.population_dir + "population.assoc", "wb") as f:
            f.write(assoc.assoc_bytes(table, self.assoc_counts))
        text, summary = assoc.deleterious_report(table, self.deleterious, self.assoc_counts, self.override_rows)
        with open(self.population_dir + "deleterious_assoc.txt", "wb") as f:
            f.write(text)
        print(summary, flush=True)

    def output_model(self, table):
        """population.model and deleterious_model.txt (--model) and population.hwe (--hardy) from the genotype counts
        and exact-test P write_vcf_snps took on the GPU."""
        if self.model:
            with open(self.population_dir + "population.model", "wb") as f:
                f.write(model.model_bytes(table, self.geno_counts))
            text, summary = model.deleterious_model_report(table, self.deleterious, self.geno_counts, self.hwe_p,
                                                           self.override_rows)
            with open(self.population_dir + "deleterious_model.txt", "wb") as f:
                f.write(text)
            print(summary, flush=True)
        if self.hardy:
            with open(self.population_dir + "population.hwe", "wb") as f:
                f.write(model.hardy_bytes(table, self.geno_counts, self.hwe_p))

    def output_fisher(self, table):
        """population.assoc.fisher, population.model.fisher and deleterious_fisher.txt (--fisher) from the genotype
        counts and Fisher log10 P write_vcf_snps took on the GPU."""
        with open(self.population_dir + "population.assoc.fisher", "wb") as f:
            f.write(fisher.assoc_fisher_bytes(table, self.geno_counts, self.fisher_log10p))
        with open(self.population_dir + "population.model.fisher", "wb") as f:
            f.write(fisher.model_fisher_bytes(table, self.geno_counts, self.fisher_log10p))
        text, summary = fisher.deleterious_fisher_report(table, self.deleterious, self.geno_counts, self.fisher_log10p,
                                                         self.override_rows)
        with open(self.population_dir + "deleterious_fisher.txt", "wb") as f:
            f.write(text)
        print(summary, flush=True)

    def output_mperm(self, table):
        """population.assoc.mperm, population.model.rec.mperm and deleterious_mperm.txt (--mperm) from the permutation
        results write_vcf_snps took on the GPU."""
        t_obs, exceed, max_t = self.mperm_result
        emp1, emp2 = mperm.empirical(t_obs, exceed, max_t)
        with open(self.population_dir + "population.assoc.mperm", "wb") as f:
            f.write(mperm.mperm_bytes(table, emp1, emp2, 0))
        with open(self.population_dir + "population.model.rec.mperm", "wb") as f:
            f.write(mperm.mperm_bytes(table, emp1, emp2, 1))
        text, summary = mperm.deleterious_mperm_report(table, self.deleterious, t_obs, exceed, max_t, self.override_rows)
        with open(self.population_dir + "deleterious_mperm.txt", "wb") as f:
            f.write(text)
        print(summary, flush=True)

    def _geno_tests(self):
        return self.model or self.hardy or self.fisher

    def _genotype_tests(self, eng, rows, seed):
        """One dnaf_genotype_tests call for --model / --hardy / --fisher: (counts, HWE P or None, log10 P or None)."""
        return eng.genotype_tests(0, rows, seed, hwe=self.model or self.hardy, fisher=self.fisher)

    # ------------------------------------------------------------------------------------------ the GPU seam
    def write_vcf_snps(self, fam_data, snps, file, engine=None, bed_fd=None):
        """Rows of `snps` (in order) for `fam_data`, appended to `file` -- the reference's seam
        (pop_factory.py:417-469).  `snps` is a list of SNPTuples or a SnpTable; `file` a BgzfSink.  With `bed_fd`
        (an open population.bed that holds the 3 magic bytes) the same rows also go there as PLINK 1 .bed rows.  With
        --assoc the case/control allele counts of the same rows land in self.assoc_counts, with --model / --hardy /
        --fisher their genotype counts and exact-test P in self.geno_counts / self.hwe_p / self.fisher_log10p, with
        --mperm the permutation results in self.mperm_result."""
        t0 = time.time()
        level = getattr(file, "compresslevel", getattr(self, "_level", 6))
        seed = self.seed if self.seed is not None else int(datetime.now().strftime("%H%M%S"))
        n_rows = len(snps)
        sex, ctl = host.flatten_samples(fam_data)
        arrays = snps.device_arrays() if isinstance(snps, SnpTable) else host.flatten_snps(snps)
        if not _any_overrides(fam_data):
            orow, osamp = numpy.zeros(0, numpy.uint64), numpy.zeros(0, numpy.uint32)
        elif isinstance(snps, SnpTable):
            orow, osamp = host.override_pairs_table(fam_data, snps)
        else:
            orow, osamp = host.override_pairs(fam_data, snps)
        self.override_rows = orow
        gpus = min(self.gpus, max(1, n_rows))
        index = getattr(file, "index", None)
        if index is not None:
            table = snps if isinstance(snps, SnpTable) else SnpTable.from_snps(snps)
            index_rows = (table.chrom_labels, table.chrom_idx, table.position)
            tabix.validate_rows(table.chrom_idx, table.position)    # fail before the generation, not after it
        if gpus == 1:
            own = engine is None
            eng = engine or _native.Engine(0)
            try:
                eng.set_samples(sex, ctl)
                eng.set_snps(**arrays)
                eng.set_overrides(orow, osamp)
                file.flush()
                if index is not None:
                    index.add_rows(*index_rows, eng.row_offsets(0, n_rows))
                    eng.block_log(True)
                st = eng.generate_fd(0, n_rows, seed, file._handle.fileno(), level=level)   # the handle was just flushed
                self.stats.append(st)
                if index is not None:
                    index.add_blocks(*eng.block_log_get())
                    eng.block_log(False)
                if bed_fd is not None:
                    self.bed_stats.append(eng.generate_bed_fd_at(0, n_rows, seed, bed_fd, len(BED_MAGIC)))
                if self.assoc:
                    self.assoc_counts = eng.allele_counts(0, n_rows, seed)
                if self._geno_tests():
                    self.geno_counts, self.hwe_p, self.fisher_log10p = self._genotype_tests(eng, n_rows, seed)
                if self.mperm:
                    self.mperm_result = eng.mperm(0, n_rows, seed, self.mperm)
            finally:
                if own:
                    eng.close()
        else:
            self._write_multi_gpu(sex, ctl, arrays, orow, osamp, n_rows, seed, level, file, gpus,
                                  index_rows if index is not None else None, bed_fd)
        print("Finished write_vcf_snps chunk Elapsed time: {:0.4f} seconds".format(time.time() - t0))

    def _write_multi_gpu(self, sex, ctl, arrays, orow, osamp, n_rows, seed, level, file, gpus, index_rows=None, bed_fd=None):
        """Contiguous SNP ranges per GPU, no collective (SURVEY 8e; the reference stripes SNPs over its workers the
        same way, pop_factory.py:426).  BGZF blocks concatenate and the kernels are deterministic, so every rank
        first SIZES its stream on the device (dnaf_generate_device: no host traffic), the exclusive sum of the sizes
        gives every rank its offset in population.vcf.gz, and then all ranks pwrite() their streams side by side --
        nothing is spooled or copied twice.  Every rank holds only its own slice of the SNP table; the Philox row
        counter of its local row r is bounds[g] + r (dnaf_set_row_base).  .bed rows have a fixed size, so rank g
        pwrite()s its rows at 3 + bounds[g] * ceil(N/4) of population.bed without a sizing pass.  With --assoc every
        rank counts its own rows after its VCF write; the slices are joined in rank order (so do --model / --hardy /
        --fisher / --mperm; the --mperm maxima of the ranks join by elementwise max: a maximum composes over row
        ranges)."""
        bounds = partition.row_bounds(n_rows, gpus)
        n_dev = max(1, _native.device_count())      # more ranks than devices: ranks share devices round-robin
        errors = []
        index = getattr(file, "index", None)
        blocks, row_off, sizes, engines = [None] * gpus, [None] * gpus, [0] * gpus, [None] * gpus
        counts, geno, perm = [None] * gpus, [None] * gpus, [None] * gpus
        barrier = threading.Barrier(gpus)
        file.flush()   # the header blocks must be in the file: the ranks write behind them
        base = file._handle.tell()
        fd = file._handle.fileno()

        def run(g):
            try:
                lo, hi = bounds[g], bounds[g + 1]
                eng = engines[g] = _native.Engine(g % n_dev)
                eng.set_samples(sex, ctl)
                eng.set_snps(**host.slice_snps(arrays, lo, hi))
                eng.set_overrides(*host.slice_overrides(orow, osamp, lo, hi))
                eng.set_row_base(lo)
                if index is not None:
                    row_off[g] = eng.row_offsets(0, hi - lo)
                sizes[g] = eng.generate_device(0, hi - lo, seed, level=level)["bgzf_bytes"]
            except BaseException as e:  # noqa: re-raised on the caller's thread
                errors.append(e)
            try:
                barrier.wait()      # every rank's size is known
            except threading.BrokenBarrierError:
                return
            if errors:
                return
            try:
                lo, hi = bounds[g], bounds[g + 1]
                eng = engines[g]
                if index is not None:
                    eng.block_log(True)
                st = eng.generate_fd_at(0, hi - lo, seed, fd, base + sum(sizes[:g]), level=level)
                if st["bgzf_bytes"] != sizes[g]:
                    raise RuntimeError("rank %d: stream is %d bytes, its sizing pass said %d" % (g, st["bgzf_bytes"], sizes[g]))
                self.stats.append(st)
                if bed_fd is not None:
                    self.bed_stats.append(eng.generate_bed_fd_at(0, hi - lo, seed, bed_fd, len(BED_MAGIC) + lo * eng.bed_pitch()))
                if index is not None:
                    blocks[g] = eng.block_log_get()
                if self.assoc:
                    counts[g] = eng.allele_counts(0, hi - lo, seed)
                if self._geno_tests():
                    geno[g] = self._genotype_tests(eng, hi - lo, seed)
                if self.mperm:
                    perm[g] = eng.mperm(0, hi - lo, seed, self.mperm)
            except BaseException as e:  # noqa
                errors.append(e)

        threads = [threading.Thread(target=run, args=(g,)) for g in range(gpus)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for eng in engines:
            if eng is not None:
                eng.close()
        if errors:
            raise errors[0]
        file._handle.seek(base + sum(sizes))      # the sink appends the EOF block behind the last rank's stream
        if self.assoc:
            self.assoc_counts = numpy.concatenate(counts)
        if self._geno_tests():
            self.geno_counts = numpy.concatenate([q[0] for q in geno])
            if self.model or self.hardy:
                self.hwe_p = numpy.concatenate([q[1] for q in geno])
            if self.fisher:
                self.fisher_log10p = numpy.concatenate([q[2] for q in geno])
        if self.mperm:
            self.mperm_result = (numpy.concatenate([q[0] for q in perm]), numpy.concatenate([q[1] for q in perm]),
                                 numpy.maximum.reduce([q[2] for q in perm]))
        if index is not None:
            off = numpy.concatenate([numpy.zeros(1, numpy.uint64)] +
                                    [r[1:] + numpy.uint64(sum(int(q[-1]) for q in row_off[:g])) for g, r in enumerate(row_off)])
            index.add_rows(*index_rows, off)
            for cs, us in blocks:
                index.add_blocks(cs, us)

    # ------------------------------------------------------------------------------------------ deleterious sets
    def load_deleterious(self):
        with open(self.deleterious_list_path, "rt") as f:
            for line in f:
                group = DeleteriousGroup.from_json(line)
                self.deleterious[group.name] = group

    def pick_deleterious_snps(self, snp_data, deleterious_config):
        from yaml import load
        try:
            from yaml import CLoader as Loader
        except ImportError:
            from yaml import Loader
        t0 = time.time()
        with open(deleterious_config, "r") as p:
            for name, attr in load(p, Loader=Loader).items():
                for group in DeleteriousGroup.from_yml(attr, snp_data, name):
                    self.deleterious[group.name] = group
        with open(self.population_dir + "deleterious.json", "w") as f:
            for group in self.deleterious.values():
                f.write(group.to_json() + "\n")
        print("Elapsed pick_deleterious_snps {:0.2f} sec".format(time.time() - t0))


def _any_overrides(fam_data):
    return any((not s.is_control) and s.deleterious_snps for s in fam_data)


def parse_cmd_args(args):
    ap = argparse.ArgumentParser(fromfile_prefix_chars="@", prog="DNA Factory",
                                 description="Generates genetic populations using simulated SNP data.")
    ap.add_argument("-s", type=int, dest="size", help="size of afflicted/case group", required=True)
    ap.add_argument("-c", type=int, dest="control_size", help="size of control group", required=True)
    ap.add_argument("-x", type=int, dest="max_snps", help="max number of snps to load/generate")
    ap.add_argument("-p", type=str, default="deleterious.yml", dest="deleterious_config",
                    help="location of deleterious config yaml file (default is deleterious.yml)")
    ap.add_argument("-f", type=float, default=0.005, dest="min_freq",
                    help="min minor allele frequency for a SNP to be included, default is 0.005")
    ap.add_argument("-m", type=float, default=0.5, dest="male_odds",
                    help="odds of a population member being male (default 0.5)")
    ap.add_argument("-n", type=int, default=2, dest="num_processes",
                    help="Number of worker processes to use (accepted for compatibility; rows are drawn on the GPU)")
    ap.add_argument("-z", type=int, dest="compression_level", default=6, choices=range(1, 10),
                    help="gzip compression level (1=least 9=most) default 6")
    ap.add_argument("-l", action="store_const", const=False, default=True, dest="generate_snps",
                    help="load from refSNP datababse instead of using simulated snps (connection config in db.yml)")
    ap.add_argument("--deleterious_file", type=str,
                    help="<path> to a deleterious.json file that specifies the exact snps to use as deleterious")
    ap.add_argument("--snps_file", type=str, help="<path> location of snps.json.gz file to use as selected snps")
    ap.add_argument("--outdir", type=str, help="<path> directory to use for output files")
    ap.add_argument("--offset", type=int,
                    help="offset to add to all sample ids. Useful for creating VCF files that can be merged")
    # opt-in extras of the B200 path
    ap.add_argument("--seed", type=int, default=None, help="Philox seed of the genotype draws (default: HHMMSS clock)")
    ap.add_argument("--gpus", type=int, default=1, help="GPUs to spread contiguous SNP ranges over (default 1)")
    ap.add_argument("--gpu_select", action="store_true",
                    help="draw and sort the simulated SNPs on the GPU from the --seed stream instead of numpy's global state")
    ap.add_argument("--tbi", action="store_true",
                    help="also write population.vcf.gz.tbi (tabix index) from the row and block sizes the writer already knows")
    ap.add_argument("--bed", action="store_true",
                    help="also write population.bed / population.bim (PLINK 1 binary fileset beside population.fam, "
                         "A1 = ALT); every SNP must be biallelic")
    ap.add_argument("--assoc", action="store_true",
                    help="also write population.assoc (case/control allelic test of every SNP, counted on the GPU) and "
                         "deleterious_assoc.txt (rank of every planted deleterious SNP); every SNP must be biallelic")
    ap.add_argument("--model", action="store_true",
                    help="also write population.model (GENO, TREND, ALLELIC, DOM, REC case/control tests of every SNP, "
                         "genotypes counted on the GPU) and deleterious_model.txt (how every planted deleterious SNP "
                         "fares under them); every SNP must be biallelic")
    ap.add_argument("--hardy", action="store_true",
                    help="also write population.hwe (Hardy-Weinberg exact tests of every SNP in all samples, cases and "
                         "controls, on the GPU); every SNP must be biallelic")
    ap.add_argument("--fisher", action="store_true",
                    help="also write population.assoc.fisher and population.model.fisher (Fisher's exact case/control "
                         "tests of every SNP: ALLELIC, GENO, DOM, REC, no cell rule, on the GPU) and deleterious_fisher.txt "
                         "(how every planted deleterious SNP fares under them); every SNP must be biallelic")
    ap.add_argument("--mperm", type=int, default=None, metavar="N",
                    help="also write population.assoc.mperm and population.model.rec.mperm (max(T) permutation tests of "
                         "ALLELIC and REC over N case/control permutations, on the GPU: EMP1 pointwise, EMP2 family-wise "
                         "empirical P) and deleterious_mperm.txt (how every planted deleterious SNP fares under them); "
                         "every SNP must be biallelic")
    return ap.parse_args(args)


def main(sys_args):
    args = parse_cmd_args(sys_args)
    if not args.generate_snps and not args.snps_file:
        # with --snps_file the reference never touches its database either (pop_factory.py:221-231)
        raise SystemExit("-l needs the reference's RefSNP database layer; use --snps_file with an exported snps.json.gz")
    factory = PopulationFactory(num_processes=args.num_processes, generate_snps=args.generate_snps,
                                deleterious_list_path=args.deleterious_file, sample_id_offset=args.offset,
                                male_odds=args.male_odds, deleterious_config=args.deleterious_config,
                                snps_path=args.snps_file, output_path=args.outdir, seed=args.seed, gpus=args.gpus,
                                gpu_select=args.gpu_select, tbi=args.tbi, bed=args.bed, assoc=args.assoc,
                                model=args.model, hardy=args.hardy, fisher=args.fisher, mperm=args.mperm)
    factory.generate_population(args.control_size, args.size, args.min_freq, args.max_snps, args.compression_level)


if __name__ == "__main__":
    main(sys.argv[1:])
