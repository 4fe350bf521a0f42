"""CPU tests of the host-side mirror of the reference interface (no GPU compute)."""
import gzip
import json
import os
import random

import numpy as np
import pytest

from tests.cases import GOLDEN, load_case


def test_library_loads_and_exports_every_declared_symbol():
    import re
    from dna_factory_b200 import _native, build
    build.build()
    lib = _native.load()
    header = open(os.path.join(os.path.dirname(GOLDEN), "..", "include", "dnaf_b200.h")).read()
    declared = set(re.findall(r"\b(dnaf_[a-z0-9_]+)\s*\(", header)) - {"dnaf_sink_fn"}
    assert declared == set(_native.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.dnaf_abi_version() == 5
    assert _native.bgzf_eof() == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def test_missing_gpu_fails_loudly():
    """No visible CUDA device: creating a context raises.  The devices are hidden from a child process, so that the
    check runs on a machine with a GPU as well."""
    import subprocess
    import sys
    code = ("from dna_factory_b200 import _native\n"
            "try:\n    _native.Engine(0)\nexcept _native.DnafError as e:\n    print(e)\n"
            "else:\n    raise SystemExit('a context was created without a visible device')\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and "no CPU fallback" in r.stdout, r.stdout + r.stderr


def test_arg_parser_matches_reference_surface():
    # test/unit/pop_factory_test.py:78-104
    from dna_factory_b200 import pop_factory
    cmd = ("-s 10 -c 20 -n 5 -z 3 -p path_config.yml -f 0.1 -m 0.7 -x 2500 -l "
           "--deleterious_file /home/ochrzan/workspace/deleterious.json --offset 300 --snps_file my_snps.json "
           "--outdir myoutput/tuesday")
    a = pop_factory.parse_cmd_args(cmd.split(" "))
    assert (a.size, a.control_size, a.num_processes, a.compression_level) == (10, 20, 5, 3)
    assert (a.deleterious_config, a.min_freq, a.male_odds, a.max_snps) == ("path_config.yml", 0.1, 0.7, 2500)
    assert a.generate_snps is False and a.offset == 300
    assert a.deleterious_file == "/home/ochrzan/workspace/deleterious.json"
    assert a.snps_file == "my_snps.json" and a.outdir == "myoutput/tuesday"
    b = pop_factory.parse_cmd_args("-s 10 -c 20 -x 2500".split(" "))
    assert b.deleterious_file is None and b.compression_level == 6 and b.num_processes == 2
    assert b.deleterious_config == "deleterious.yml" and b.min_freq == 0.005 and b.male_odds == 0.5
    assert b.generate_snps is True


def test_snp_tuple_known_answers():
    # test/unit/pop_factory_test.py:5-28
    from dna_factory_b200.snp import SNPTuples
    s = SNPTuples(100, "1", 50000)
    for nt, c in (("G", 0.70), ("A", 0.90), ("T", 1.0)):
        s.add_tuple(nt, c)
    assert s.pick_snp_value(0.95) == "T" and s.pick_snp_value(0.4) == "G"
    assert s.pick_allele_index(0.95) == 2 and s.pick_allele_index(0.4) == 0
    assert s.alt_alleles() == "A,T"
    assert SNPTuples.from_json(str(s)).tuples == s.tuples


def test_split_list_and_ploidy():
    # test/unit/common_util_test.py:7-12, common/snp.py:102-109
    from dna_factory_b200.snp import is_haploid, split_list, stripe_list
    y = list(split_list(list(range(100)), 3))
    assert [len(v) for v in y] == [33, 33, 34]
    assert stripe_list(list(range(7)), 3) == [[0, 3, 6], [1, 4], [2, 5]]
    assert is_haploid("X", True) and not is_haploid("X", False)
    assert is_haploid("Y", False) and is_haploid("MT", False) and not is_haploid("7", True)


def test_deleterious_group_from_yml():
    # test/unit/pop_factory_test.py:31-44
    from dna_factory_b200.pop_factory import DeleteriousGroup
    from dna_factory_b200.snp import SNPTuples
    data = []
    for i in range(1, 5):
        s = SNPTuples(i, "1", 50000)
        for nt, c in (("G", 0.70), ("A", 0.90), ("T", 1.0)):
            s.add_tuple(nt, c)
        data.append(s)
    groups = DeleteriousGroup.from_yml({"mutation_weights": [0.5, 0.5, 0.5], "num_instances": 2,
                                        "population_weight": 5, "min_minor_allele_freq": 0.01}, data, "groupA")
    assert len(groups) == 2 and groups[0].population_weight == 5
    assert len(groups[0].deleterious) == 3 and len(groups[0].select_mutations()) == 2


def test_snp_factory_distribution():
    # test/unit/snp_factory_test.py:14-37 (tolerances as upstream)
    from dna_factory_b200.snp import CHROMOSOME_PROB, SnpFactory
    np.random.seed(7)
    random.seed(7)
    fac = SnpFactory.init_from_cdf_file()
    n, min_maf = 100000, 0.16
    t = fac.random_snp_table(n, min_maf=min_maf)
    assert len(t) == n and (t.n_alleles == 2).all()
    largest = fac.sorted_maf[-1]
    assert ((1 - t.cum[:, 0]) >= min_maf - 1e-12).all()
    assert (t.nts[:, 0] != t.nts[:, 1]).all()
    assert abs((t.cum[:, 0] == 1 - largest).mean() - fac.pdf[-1] / fac.pdf[fac._first_bin(min_maf):].sum()) < 0.01
    assert abs((t.chrom_idx == 0).mean() - CHROMOSOME_PROB[0]) < 0.01


def test_host_files_match_reference_cli_golden(tmp_path, monkeypatch):
    """snps.json.gz, deleterious.json, population.fam and pop_deleterious.txt byte for byte against the
    reference CLI run pinned in tests/golden/cli_small (the VCF itself needs the GPU: test_gpu_cli.py)."""
    from dna_factory_b200 import pop_factory
    gold = os.path.join(GOLDEN, "cli_small")
    meta = json.load(open(os.path.join(gold, "meta.json")))

    class FixedDatetime(pop_factory.datetime):
        @classmethod
        def now(cls, tz=None):
            return cls(2026, 1, 1, 12, 34, 56)

    monkeypatch.setattr(pop_factory, "datetime", FixedDatetime)
    captured = {}

    def fake_output(self, control_size, test_size, male_odds, level):
        groups = pop_factory.PopulationFactory.pick_deleterious_groups(list(self.deleterious.values()), test_size)
        captured["fam"] = self.generate_fam_file(control_size, test_size, male_odds, groups)
        captured["header"] = pop_factory.gen_vcf_header(captured["fam"])

    monkeypatch.setattr(pop_factory.PopulationFactory, "output_vcf_population", fake_output)
    random.seed(meta["python_random_seed"])
    args = meta["args"] + ["-p", os.path.join(gold, "deleterious_config.yml"), "--outdir", str(tmp_path)]
    pop_factory.main(args)
    with gzip.open(tmp_path / "snps.json.gz", "rb") as f:
        assert f.read() == open(os.path.join(gold, "snps.json"), "rb").read()
    for name in ("deleterious.json", "population.fam", "pop_deleterious.txt"):
        assert (tmp_path / name).read_bytes() == open(os.path.join(gold, name), "rb").read(), name
    with gzip.open(os.path.join(gold, "population.vcf.rows.gz"), "rb") as f:
        vcf = f.read()
    assert vcf.startswith(captured["header"].encode())


def test_override_pairs_table_equals_object_path():
    from dna_factory_b200 import host
    from dna_factory_b200.snp import SnpTable
    case = load_case("mixed64")
    biallelic = [s for s in case.snps if len(s.tuples) <= 4]
    table = SnpTable.from_snps(biallelic)
    a = host.override_pairs(case.samples, biallelic)
    b = host.override_pairs_table(case.samples, table)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and len(a[0]) > 0
    r8 = load_case("r8_strkeys")
    t8 = SnpTable.from_snps(r8.snps)
    assert len(host.override_pairs_table(r8.samples, t8)[0]) == 0


def test_threshold_is_exact_for_inclusive_compare():
    from dna_factory_b200 import host
    # cum >= U/2^32  <=>  U <= threshold(cum), checked around awkward values
    for cum in (0.0, 2.0 ** -32, 0.3, 0.9299999999999999, 1 - 2.0 ** -32, 1 - 2.0 ** -33, 1.0, 1.5):
        t = host.threshold(cum)
        for U in {0, 1, max(t - 1, 0), t, min(t + 1, 0xFFFFFFFF), 0xFFFFFFFF}:
            assert (cum >= U * 2.0 ** -32) == (U <= t), (cum, U)
    with pytest.raises(ValueError):
        host.threshold(-0.1)


def test_native_snps_json_parser_matches_json_loads(tmp_path):
    """dnaf_parse_snps_jsonl against SNPTuples.from_json (pop_factory.py:126-133) on the reference's own snps.json
    (tests/golden/cli_small), on multi-allelic records, and its refusal of records outside the column form."""
    import gzip
    from dna_factory_b200 import _native, snp
    from tests.cases import GOLDEN
    raw = open(os.path.join(GOLDEN, "cli_small", "snps.json"), "rb").read()
    cols = _native.parse_snps_jsonl(raw)
    want = [snp.SNPTuples.from_json(line) for line in raw.decode().splitlines()]
    assert cols is not None and len(cols["ids"]) == len(want)
    tab = snp.SnpTable(cols["ids"], cols["chrom_idx"], cols["chrom_labels"], cols["position"], cols["n_alleles"], cols["nts"],
                       cols["cum"])
    assert [(s.id, s.chromosome, s.position, s.tuples) for s in tab.to_snps()] == \
        [(s.id, s.chromosome, s.position, s.tuples) for s in want]
    multi = (b'{"id": 7, "chromosome": "MT", "position": 5, "tuples": {"G": 0.4, "A": 0.7000000000000001, "T": 0.9, "C": 1.0}}\n'
             b'{"id": 8, "chromosome": "X", "position": 0, "tuples": {"C": 1.0}}\n')
    cols = _native.parse_snps_jsonl(multi)
    assert cols["chrom_labels"] == ["MT", "X"] and list(cols["n_alleles"]) == [4, 1]
    assert cols["cum"][0].tolist() == [0.4, 0.7000000000000001, 0.9, 1.0] and bytes(cols["nts"][0]) == b"GATC"
    for bad in (b'{"id": "rs5", "chromosome": "1", "position": 1, "tuples": {"A": 1.0}}\n',       # string id
                b'{"id": 5, "chromosome": "1", "position": 1, "tuples": {"AT": 1.0}}\n',          # multi-character allele
                b'{"id": 5, "chromosome": "1", "position": 1}\n'):                                # no tuples
        assert _native.parse_snps_jsonl(bad) is None
    path = tmp_path / "snps.json.gz"
    with gzip.open(path, "wb") as f:
        f.write(raw)
    assert len(snp.SnpTable.read_json_gz_table(str(path))) == len(want)


def test_native_formatters_match_the_python_ones(tmp_path):
    """dnaf_format_prefixes / dnaf_format_snps_jsonl against the numpy / json.dumps implementations they replace
    (row lead of pop_factory.py:503-507, SNPTuples.__str__ of pop_factory.py:118-124), incl. K = 1, 3, 4 records."""
    import gzip
    from dna_factory_b200 import snp
    from tests.cases import synth_case
    case = synth_case(3, 400, seed=9, chroms=['1', '12', 'X', 'Y', 'MT'], exotic=True)
    tab = snp.SnpTable.from_snps(case.snps).sorted()
    a, b = tab.prefix_bytes(), tab.prefix_bytes_numpy()
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    want = b"".join(("%s\t%i\trs%s\t%s\t%s\t40\tPASS\t.\tGT\t" % (s.chromosome, s.position, s.id, s.ref_allele_tuple()[0],
                                                                  s.alt_alleles() if len(s.tuples) > 1 else s.tuples[0][0])
                     ).encode() for s in tab.to_snps())
    assert a[0][:-1].tobytes() == want
    tab.write_json_gz(str(tmp_path / "a.gz"))
    tab.write_json_gz_python(str(tmp_path / "b.gz"))
    got = gzip.open(tmp_path / "a.gz", "rb").read()
    assert got == gzip.open(tmp_path / "b.gz", "rb").read()
    assert got.decode().splitlines() == [str(s) for s in tab.to_snps()]


def test_offset_replay_host_files_match_reference(tmp_path, monkeypatch):
    """The README's multi-run recipe (README.md:88-94, pop_factory.py:350-351,378): `--offset 300` replayed from
    snps.json.gz / deleterious.json -- population.fam, pop_deleterious.txt and the VCF header's sample ids byte for
    byte against the pinned reference run (tests/golden/cli_offset; the rows need the GPU: test_gpu_cli.py)."""
    from dna_factory_b200 import pop_factory
    gold = os.path.join(GOLDEN, "cli_offset")
    src = os.path.join(GOLDEN, "cli_small")
    meta = json.load(open(os.path.join(gold, "meta.json")))

    class FixedDatetime(pop_factory.datetime):
        @classmethod
        def now(cls, tz=None):
            return cls(2026, 1, 1, 12, 34, 56)

    monkeypatch.setattr(pop_factory, "datetime", FixedDatetime)
    captured = {}

    def fake_output(self, control_size, test_size, male_odds, level):
        groups = pop_factory.PopulationFactory.pick_deleterious_groups(list(self.deleterious.values()), test_size)
        captured["fam"] = self.generate_fam_file(control_size, test_size, male_odds, groups)
        captured["header"] = pop_factory.gen_vcf_header(captured["fam"])

    monkeypatch.setattr(pop_factory.PopulationFactory, "output_vcf_population", fake_output)
    snps_gz = tmp_path / "snps_in.json.gz"
    with open(os.path.join(src, "snps.json"), "rb") as f, gzip.open(snps_gz, "wb") as g:
        g.write(f.read())
    random.seed(meta["python_random_seed"])
    out = tmp_path / "out"
    pop_factory.main(meta["args"] + ["--snps_file", str(snps_gz), "--deleterious_file", os.path.join(src, "deleterious.json"),
                                     "--outdir", str(out)])
    for name in ("population.fam", "pop_deleterious.txt"):
        assert (out / name).read_bytes() == open(os.path.join(gold, name), "rb").read(), name
    with gzip.open(os.path.join(gold, "population.vcf.rows.gz"), "rb") as f:
        vcf = f.read()
    assert vcf.startswith(captured["header"].encode())
    assert [s.person_id for s in captured["fam"]][:2] == [100301, 100302] and captured["fam"][0].family_id == 601


def test_slices_of_the_snp_table_and_overrides():
    """What a rank of `--gpus N` uploads: its own rows, offsets rebased, overrides made local."""
    from dna_factory_b200 import host
    case = load_case("mixed64")
    flat = host.flatten_snps(case.snps)
    orow, osamp = host.override_pairs(case.samples, case.snps)
    S = len(case.snps)
    pieces, opieces = [], 0
    for lo, hi in ((0, 7), (7, 7), (7, S)):
        a = host.slice_snps(flat, lo, hi)
        assert len(a["chrom_class"]) == hi - lo == len(a["prefix_off"]) - 1 and a["prefix_off"][0] == 0
        pieces.append(bytes(a["prefix_bytes"][:int(a["prefix_off"][-1])]))
        assert np.array_equal(a["thresholds"], flat["thresholds"][lo:hi])
        r, s = host.slice_overrides(orow, osamp, lo, hi)
        assert all(0 <= int(x) < hi - lo for x in r)
        opieces += len(r)
    assert b"".join(pieces) == bytes(flat["prefix_bytes"][:int(flat["prefix_off"][-1])])
    assert opieces == len(orow) > 0


def test_override_pairs_table_handles_duplicate_ids_and_odd_keys():
    from types import SimpleNamespace
    from dna_factory_b200 import host
    table = SimpleNamespace(ids=np.array([5, 9, 5, 12], dtype=np.int64))
    fam = [SimpleNamespace(is_control=True, deleterious_snps={5: 1.0}),
           SimpleNamespace(is_control=False, deleterious_snps={5: 0.5, "9": 0.5, 12.0: 0.1, 7: 0.2, True: 0.3, 9.5: 0.1}),
           SimpleNamespace(is_control=False, deleterious_snps=None),
           SimpleNamespace(is_control=False, deleterious_snps={9: 0.5})]
    rows, samples = host.override_pairs_table(fam, table, row_base=100)
    assert list(zip(rows.tolist(), samples.tolist())) == [(100, 1), (101, 3), (102, 1), (103, 1)]


def test_tabix_rows_are_validated_up_front():
    from dna_factory_b200 import tabix
    tabix.validate_rows([0, 0, 1, 1], [5, 9, 1, 1])
    tabix.validate_rows([], [])
    for chrom, pos in (([0, 1, 0], [1, 2, 3]), ([0, 0], [9, 5]), ([0], [1 << 30]), ([0], [-1])):
        with pytest.raises(ValueError):
            tabix.validate_rows(chrom, pos)


def test_chi_square_tail_known_answers():
    """chi2_sf replaces scipy.stats.chi2.sf (whose import costs minutes on a cold box); values from scipy 1.x."""
    from dna_factory_b200.allele_stats import chi2_sf
    for x, k, want in ((5064.3, 5049, 0.4369388816951934), (2458.0, 2475, 0.5920034834051018), (100.0, 51, 4.998131371998267e-05),
                       (20.0, 51, 0.9999710569766698), (3.0, 1, 0.08326451666355042), (60.0, 1, 9.485737571073857e-15),
                       (5600, 5049, 5.7232768619912364e-08), (0.5, 3, 0.9188914116546758)):
        assert abs(chi2_sf(x, k) - want) <= 1e-9 * max(want, 1e-6), (x, k)


def test_bgzf_inflater_checks_every_block():
    import zlib
    from dna_factory_b200.allele_stats import inflate_bgzf
    from oracle import oracle
    text = (b"1\t100\trs1\tA\tC\t40\tPASS\t.\tGT\t" + b"0/1\t" * 5000 + b"\n") * 9
    blob = oracle.bgzf(text, level=6, with_eof=False)
    assert inflate_bgzf(blob) == text
    bad = bytearray(blob)
    bad[-6] ^= 1                                   # CRC32 of the last block
    with pytest.raises(ValueError):
        inflate_bgzf(bytes(bad))


def test_reference_copy_is_byte_identical_and_runs():
    """oracle/make_ref.py materialises the UNMODIFIED reference for the CPU baselines; where /root/reference is
    mounted the copy must match it byte for byte and its CLI must run under the shims."""
    import hashlib
    from oracle import make_ref, ref_cli
    if not os.path.exists(os.path.join(make_ref.REFERENCE_DIR, "pop_factory.py")):
        pytest.skip("reference tree not mounted")
    assert make_ref.materialise()
    man = json.load(open(os.path.join(make_ref.DEST, "MANIFEST.json")))["sha256"]
    for rel, digest in man.items():
        assert hashlib.sha256(open(os.path.join(make_ref.REFERENCE_DIR, rel), "rb").read()).hexdigest() == digest
        assert hashlib.sha256(open(os.path.join(make_ref.DEST, rel), "rb").read()).hexdigest() == digest
    r = ref_cli.run(20, 20, 300, 2, procs=2)
    assert r["calls"] == 12000 and r["write_s"] > 0 and r["vcf_bytes"] > 1000


def test_bench_population_windows_do_not_depend_on_what_follows():
    """bench.py's multi-GPU parity check regenerates a rank's FIRST window alone: the window's SNP rows and forced
    cells must be the same whether 1 or 3 windows are drawn for that rank."""
    import bench
    one = bench.synth_population(64, rank=3, window=64)
    three = bench.synth_population(192, rank=3, window=64)
    assert np.array_equal(one[0], three[0]) and np.array_equal(one[1], three[1])
    a, b = one[2].device_arrays(), three[2].device_arrays()
    from dna_factory_b200 import host
    b0 = host.slice_snps(b, 0, 64)
    for k in ("chrom_class", "n_alleles", "thresholds", "prefix_off"):
        assert np.array_equal(a[k], b0[k]), k
    n = int(a["prefix_off"][-1])
    assert bytes(a["prefix_bytes"][:n]) == bytes(b0["prefix_bytes"][:n])
    r1, s1 = host.slice_overrides(one[3], one[4], 0, 64)
    r3, s3 = host.slice_overrides(three[3], three[4], 0, 64)
    assert np.array_equal(r1, r3) and np.array_equal(s1, s3) and len(r1) >= 2


def test_bench_dump_outputs_hold_the_stream_and_its_text(tmp_path):
    """bench.py --dump-outputs: float .npy files of at most 64 MB in all; the sampled windows are the bytes of the BGZF
    stream and of its text at the stored offsets, the block table covers the text, and the same stream gives the same
    files."""
    import bench
    from dna_factory_b200 import _native
    from oracle import oracle
    from tests.cases import synth_case
    case = synth_case(2000, 300, seed=4)
    text, _ = oracle.rows(case.samples, case.snps, case.seed, n_threads=4)
    blob = np.frombuffer(oracle.bgzf(text, level=2, with_eof=False), np.uint8)
    assert len(blob) > 2 * bench.DUMP_WINDOW
    st = {"rows": 300, "calls": 600000, "text_bytes": len(text), "bgzf_bytes": len(blob),
          "bgzf_blocks": len(_native.bgzf_scan(blob)[0]), "crc_xor": 0xDEADBEEF, "ms_total": 1.5}
    bench.dump_outputs(str(tmp_path / "a"), st, st, blob)
    got = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    assert {a.dtype for a in got.values()} <= {np.dtype(np.float32), np.dtype(np.float64)}
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert list(got["e2e_stats"]) == [300, 600000, len(text), len(blob), st["bgzf_blocks"], 0xDEADBEEF]
    assert got["e2e_bgzf_blocks"].shape == (st["bgzf_blocks"], 2) and got["e2e_bgzf_blocks"][:, 1].sum() == len(text)
    assert got["e2e_text"].shape == (128, bench.DUMP_WINDOW) and got["e2e_bgzf"].shape == (64, bench.DUMP_WINDOW)
    for o, w in zip(got["e2e_text_offsets"].astype(np.int64), got["e2e_text"]):
        assert w.astype(np.uint8).tobytes() == text[o:o + bench.DUMP_WINDOW]
    for o, w in zip(got["e2e_bgzf_offsets"].astype(np.int64), got["e2e_bgzf"]):
        assert w.astype(np.uint8).tobytes() == blob[o:o + bench.DUMP_WINDOW].tobytes()
    bench.dump_outputs(str(tmp_path / "b"), st, st, blob.copy())
    for name, a in got.items():
        assert np.array_equal(np.load(tmp_path / "b" / (name + ".npy")), a), name


def test_header_is_plain_c_and_links(tmp_path):
    """include/dnaf_b200.h must be consumable by the reference's side of an FFI without a C++ compiler: a C99 program
    includes it, links the library and calls the GPU-free entry points (tests/c/abi_smoke.c)."""
    import shutil
    import subprocess
    from dna_factory_b200 import _native
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    _native.load()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "abi_smoke"
    lib_dir = os.path.dirname(_native.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(root, "include"),
                           os.path.join(root, "tests", "c", "abi_smoke.c"), "-o", str(exe), "-L", lib_dir, "-ldnaf_b200",
                           "-Wl,-rpath," + lib_dir])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert r.stdout.startswith("abi 5 ok")


def test_bench_reference_arm_runs_the_unmodified_reference():
    """bench.py --impl reference / cpu_baseline: the reference CLI from oracle/_ref, timed by its own write_vcf_snps
    timer (pop_factory.py:417), at a toy size here."""
    import bench
    from oracle import make_ref
    make_ref.materialise()
    if not make_ref.available():
        pytest.skip("oracle/_ref not materialised (no reference tree here)")
    saved = bench.N_CASES, bench.N_CONTROLS
    bench.N_CASES = bench.N_CONTROLS = 50
    try:
        r = bench.python_reference_run(1, 0, rows=200)
    finally:
        bench.N_CASES, bench.N_CONTROLS = saved
    assert r["value"] > 0 and r["procs"] >= 1 and "unmodified reference CLI" in r["sample"]
