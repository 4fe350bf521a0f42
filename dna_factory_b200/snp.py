"""SNP records, genome constants and SNP selection (host side of the path).

Mirrors the reference's interface for this path -- same names, argument meaning and outputs -- so code
and tests written against ochrzan/dna-factory read the same here:
  CHROMOSOME_LIST / CHROMOSOME_PROB / CHROMOSOME_MAX_POSITION, split_list, stripe_list, is_haploid
                                                                    common/snp.py:8-60,71-88,102-109
  SNPTuples                                                         pop_factory.py:74-133
  SnpFactory (frequency-CDF SNP selection)                          pop_factory.py:136-193
The records are additionally kept in column form (SnpTable) because the GPU path consumes flat arrays
and 10^7 Python objects are the reference's own bottleneck (SURVEY 8a/a4, a8).
"""
import gzip
import json
import random

import numpy as np

from . import _native
from .maf_cdf import MAF_CDF

CHROMOSOME_LIST = [str(i) for i in range(1, 23)] + ["X", "Y"]

# share of reported SNPs per chromosome, order of CHROMOSOME_LIST (data, common/snp.py:10-34)
CHROMOSOME_PROB = [
    0.07426087261566, 0.07930487311426, 0.06669253502772, 0.068216704579376, 0.060859452377757,
    0.061620602417568, 0.056436996345677, 0.052745283940636, 0.041811456817423, 0.047572674763057,
    0.046903788666524, 0.045558978461098, 0.033875108161329, 0.030837930905743, 0.028329099437382,
    0.030535626281104, 0.026508783521902, 0.026711126377244, 0.022471493713103, 0.021115686613365,
    0.013429462318399, 0.013635819040166, 0.048111412615406, 0.002454231888101,
]

# GRCh38 chromosome lengths (data, common/snp.py:36-60)
CHROMOSOME_MAX_POSITION = dict(zip(CHROMOSOME_LIST, [
    248946339, 242765766, 198235509, 190181952, 181477687, 170744571, 159335932, 145571444, 138258771,
    133787363, 135076614, 133265032, 114352979, 107270972, 101981181, 90228323, 83247315, 80262386,
    58607512, 64333614, 46699955, 50806829, 156040000, 57217333]))

NUCLEOTIDES = ["A", "T", "C", "G"]


def split_list(l, n):
    """n consecutive chunks of round(len/n) items, the remainder going to the last (common/snp.py:71-79)."""
    size = round(len(l) / n)
    for i in range(n):
        yield l[i * size:(len(l) if i + 1 == n else (i + 1) * size)]


def stripe_list(l, num_stripes):
    """Round-robin striping (common/snp.py:82-88); kept for API parity, the GPU path does not stripe."""
    return [list(l[i::num_stripes]) for i in range(num_stripes)]


def is_haploid(chromo, is_male):
    """One allele per person on this chromosome? (common/snp.py:102-109)"""
    return (chromo == "X" and is_male) or chromo == "MT" or chromo == "Y"


class SNPTuples:
    """One SNP: id, chromosome, position and (nucleotide, cumulative probability) tuples."""

    def __init__(self, snp_id, chromosome, position):
        self.id = snp_id
        self.chromosome = chromosome
        self.position = position
        self.tuples = []

    def add_tuple(self, inserted, range_end):
        self.tuples.append((inserted, range_end))

    def pick_snp_value(self, random_roll):
        for nt, cum in self.tuples:
            if cum > random_roll:
                return nt
        return None

    def pick_allele_index(self, random_roll):
        """First allele whose cumulative probability is >= the roll (inclusive, as upstream)."""
        for i, (_, cum) in enumerate(self.tuples):
            if cum >= random_roll:
                return i
        return None

    def ref_allele_tuple(self):
        return self.tuples[0]

    def minor_allele_tuple(self):
        return self.tuples[1]

    def alt_alleles(self):
        if len(self.tuples) <= 2:
            return self.tuples[-1][0]
        return ",".join(t[0] for t in self.tuples[1:])

    def __str__(self):
        rec = {"id": self.id, "chromosome": self.chromosome, "position": self.position}
        if self.tuples:
            rec["tuples"] = {nt: cum for nt, cum in self.tuples}
        return json.dumps(rec)

    @classmethod
    def from_json(cls, json_line):
        rec = json.loads(json_line)
        snp = cls(rec["id"], rec["chromosome"], rec["position"])
        for nt, cum in rec.get("tuples", {}).items():
            snp.add_tuple(nt, cum)
        return snp


def _label_matrix(labels):
    """Chromosome labels as a zero-padded uint8 matrix, one row per label."""
    lab = np.zeros((len(labels), max(len(c.encode("latin-1")) for c in labels)), np.uint8)
    for i, c in enumerate(labels):
        b = c.encode("latin-1")
        lab[i, :len(b)] = np.frombuffer(b, np.uint8)
    return lab


def _digits(v):
    """Decimal digits of non-negative ints, right-aligned in a fixed width, with the mask of the printed ones."""
    width = max(1, len(str(int(v.max()))))
    p = 10 ** np.arange(width - 1, -1, -1, dtype=np.int64)
    d = (v[:, None] // p[None, :]) % 10
    nd = 1 + (v[:, None] >= p[None, :-1]).sum(axis=1) if width > 1 else np.ones(len(v), np.int64)
    ok = np.arange(width)[None, :] >= (width - nd)[:, None]
    return (d + 48).astype(np.uint8), ok


def _const(b, rows):
    a = np.frombuffer(b, np.uint8)
    return np.broadcast_to(a, (rows, len(a))), np.ones((rows, len(a)), bool)


def _join_fields(fields, rows):
    """Row-major concatenation of (bytes, mask) field matrices -> (flat bytes, row offsets[rows + 1])."""
    data = np.concatenate([f[0] for f in fields], axis=1)
    mask = np.concatenate([f[1] for f in fields], axis=1)
    off = np.zeros(rows + 1, np.uint64)
    off[1:] = np.cumsum(mask.sum(axis=1))
    return data[mask], off


class SnpTable:
    """Column form of a SNP list (biallelic fast path + generic K <= 4)."""

    def __init__(self, ids, chrom_idx, chrom_labels, position, n_alleles, nts, cum):
        self.ids = np.asarray(ids, dtype=np.int64)
        self.chrom_idx = np.asarray(chrom_idx, dtype=np.int32)
        self.chrom_labels = list(chrom_labels)
        self.position = np.asarray(position, dtype=np.int64)
        self.n_alleles = np.asarray(n_alleles, dtype=np.uint8)
        self.nts = np.asarray(nts, dtype=np.uint8).reshape(len(self.ids), _native.KMAX)      # ASCII codes
        self.cum = np.asarray(cum, dtype=np.float64).reshape(len(self.ids), _native.KMAX)

    def __len__(self):
        return len(self.ids)

    # ---- conversions -----------------------------------------------------------------------------
    @classmethod
    def from_snps(cls, snps):
        labels, index = [], {}
        S = len(snps)
        ids = np.zeros(S, np.int64)
        ci = np.zeros(S, np.int32)
        pos = np.zeros(S, np.int64)
        k = np.zeros(S, np.uint8)
        nts = np.zeros((S, _native.KMAX), np.uint8)
        cum = np.full((S, _native.KMAX), 2.0)
        for r, s in enumerate(snps):
            if s.chromosome not in index:
                index[s.chromosome] = len(labels)
                labels.append(s.chromosome)
            if not 1 <= len(s.tuples) <= _native.KMAX or any(len(t[0]) != 1 for t in s.tuples) \
                    or not isinstance(s.id, (int, np.integer)):
                raise ValueError("SNP %r does not fit the column form" % (s.id,))
            ids[r], ci[r], pos[r], k[r] = s.id, index[s.chromosome], s.position, len(s.tuples)
            for j, (nt, c) in enumerate(s.tuples):
                nts[r, j] = ord(nt)
                cum[r, j] = c
        return cls(ids, ci, labels, pos, k, nts, cum)

    def snp(self, r):
        s = SNPTuples(int(self.ids[r]), self.chrom_labels[self.chrom_idx[r]], int(self.position[r]))
        for j in range(int(self.n_alleles[r])):
            s.add_tuple(chr(self.nts[r, j]), float(self.cum[r, j]))
        return s

    def to_snps(self):
        return [self.snp(r) for r in range(len(self))]

    def take(self, order):
        return SnpTable(self.ids[order], self.chrom_idx[order], self.chrom_labels, self.position[order],
                        self.n_alleles[order], self.nts[order], self.cum[order])

    @classmethod
    def concat(cls, tables):
        labels = tables[0].chrom_labels
        if any(t.chrom_labels != labels for t in tables):
            raise ValueError("tables use different chromosome label lists")
        cat = np.concatenate
        return cls(cat([t.ids for t in tables]), cat([t.chrom_idx for t in tables]), labels,
                   cat([t.position for t in tables]), cat([t.n_alleles for t in tables]), cat([t.nts for t in tables]),
                   cat([t.cum for t in tables]))

    def sorted(self):
        """Order of `ordered_snps.sort(key=lambda x: (x.chromosome, x.position))` (pop_factory.py:245):
        chromosome compared as a STRING, ties keep insertion order (stable)."""
        rank_of_label = np.argsort(np.argsort(np.asarray(self.chrom_labels, dtype=object).astype(str), kind="stable"),
                                   kind="stable")
        # equal labels cannot occur in chrom_labels, so ranks are a permutation
        key = rank_of_label[self.chrom_idx]
        return self.take(np.lexsort((self.position, key)))

    def minor_allele_freq(self):
        """minor_allele_tuple()[1] - ref_allele_tuple()[1] (pop_factory.py:555-556); NaN for K == 1."""
        out = self.cum[:, 1] - self.cum[:, 0]
        return np.where(self.n_alleles >= 2, out, np.nan)

    # ---- flat arrays for the C ABI ---------------------------------------------------------------
    def chrom_class(self):
        lab = np.asarray([{"X": _native.CLASS_X, "Y": _native.CLASS_Y, "MT": _native.CLASS_MT}.get(c, _native.CLASS_AUTO)
                          for c in self.chrom_labels], dtype=np.uint8)
        return lab[self.chrom_idx]

    def thresholds(self):
        cum = self.cum
        if np.any(~(cum >= 0.0)):
            raise ValueError("negative or NaN cumulative allele probability")
        t = np.floor(np.minimum(cum, 1.0) * 4294967296.0)
        t = np.where(cum >= 1.0, 4294967295.0, np.minimum(t, 4294967295.0)).astype(np.uint32)
        col = np.arange(_native.KMAX)[None, :]
        return np.where(col < self.n_alleles[:, None], t, np.uint32(0xFFFFFFFF)).astype(np.uint32)

    def prefix_bytes(self):
        """Row leads "%s\\t%i\\trs%s\\t%s\\t%s\\t40\\tPASS\\t.\\tGT\\t" (pop_factory.py:503-507): the native formatter
        (dnaf_format_prefixes), or the numpy one for chromosome labels longer than 7 bytes."""
        S = len(self)
        if S == 0:
            return np.zeros(1, np.uint8), np.zeros(1, np.uint64)
        if np.any(self.position < 0) or np.any(self.ids < 0):
            raise ValueError("negative position / id")
        if all(0 < len(c.encode("latin-1")) <= 7 for c in self.chrom_labels):
            return _native.format_prefixes(self.ids, self.chrom_idx, self.chrom_labels, self.position, self.n_alleles, self.nts)
        return self.prefix_bytes_numpy()

    def prefix_bytes_numpy(self):
        """The same bytes, vectorised in numpy: fixed-width fields with a validity mask, flattened row-major."""
        S = len(self)
        if S == 0:
            return np.zeros(1, np.uint8), np.zeros(1, np.uint64)
        if np.any(self.position < 0) or np.any(self.ids < 0):
            raise ValueError("negative position / id")
        lab = _label_matrix(self.chrom_labels)
        pd, pok = _digits(self.position)
        idd, iok = _digits(self.ids)
        alt_w = 2 * (_native.KMAX - 1) - 1
        alt = np.zeros((S, alt_w), np.uint8)
        aok = np.zeros((S, alt_w), bool)
        k = self.n_alleles
        # ALT column: tuples[1] for K == 2, the REF itself for K == 1, comma-joined tuples[1:] for K > 2
        alt[:, 0] = np.where(k == 1, self.nts[:, 0], self.nts[:, 1])
        aok[:, 0] = True
        for j in range(2, _native.KMAX):
            alt[:, 2 * (j - 1) - 1] = ord(",")
            alt[:, 2 * (j - 1)] = self.nts[:, j]
            aok[:, 2 * (j - 1) - 1] = k > j
            aok[:, 2 * (j - 1)] = k > j
        tail = np.frombuffer(b"\t40\tPASS\t.\tGT\t", np.uint8)
        cl = lab[self.chrom_idx]
        fields = [(cl, cl != 0), _const(b"\t", S), (pd, pok), _const(b"\trs", S), (idd, iok), _const(b"\t", S),
                  (self.nts[:, :1], np.ones((S, 1), bool)), _const(b"\t", S), (alt, aok), (np.broadcast_to(tail, (S, len(tail))),
                                                                                          np.ones((S, len(tail)), bool))]
        flat, off = _join_fields(fields, S)
        return np.concatenate([flat, np.zeros(1, np.uint8)]), off

    def bim_bytes(self):
        """PLINK .bim text, one line per row: "chrom\trs<id>\t0\tposition\tA1\tA2\n" with A1 = ALT ('0' for K == 1)
        and A2 = REF, the allele order of the .bed codes (dnaf_generate_bed).  Rows with K > 2 have no .bim form."""
        S = len(self)
        if S == 0:
            return b""
        if np.any(self.n_alleles > 2):
            raise ValueError("SNP %d has %d alleles: PLINK 1 filesets hold biallelic rows only" % (
                int(self.ids[np.argmax(self.n_alleles > 2)]), int(self.n_alleles[np.argmax(self.n_alleles > 2)])))
        if np.any(self.position < 0) or np.any(self.ids < 0):
            raise ValueError("negative position / id")
        cl = _label_matrix(self.chrom_labels)[self.chrom_idx]
        pd, pok = _digits(self.position)
        idd, iok = _digits(self.ids)
        a1 = np.where(self.n_alleles == 1, ord("0"), self.nts[:, 1]).astype(np.uint8)[:, None]
        one = np.ones((S, 1), bool)
        fields = [(cl, cl != 0), _const(b"\trs", S), (idd, iok), _const(b"\t0\t", S), (pd, pok), _const(b"\t", S),
                  (a1, one), _const(b"\t", S), (self.nts[:, :1], one), _const(b"\n", S)]
        return _join_fields(fields, S)[0].tobytes()

    def device_arrays(self):
        pre, off = self.prefix_bytes()
        return dict(chrom_class=self.chrom_class(), n_alleles=self.n_alleles, thresholds=self.thresholds(),
                    prefix_bytes=pre, prefix_off=off)

    # ---- snps.json.gz (pop_factory.py:118-133,258-272) -------------------------------------------
    def write_json_gz(self, path, compresslevel=5):
        if len(self) and all(0 < len(c.encode("latin-1")) <= 7 and c.isalnum() for c in self.chrom_labels):
            data = _native.format_snps_jsonl(self.ids, self.chrom_idx, self.chrom_labels, self.position, self.n_alleles,
                                             self.nts, self.cum)
            with gzip.open(path, "wb", compresslevel=compresslevel) as f:
                f.write(data)
            return
        self.write_json_gz_python(path, compresslevel)

    def write_json_gz_python(self, path, compresslevel=5):
        with gzip.open(path, "wt", compresslevel=compresslevel) as f:
            reprs = {}
            for r in range(len(self)):
                k = int(self.n_alleles[r])
                parts = []
                for j in range(k):
                    c = float(self.cum[r, j])
                    s = reprs.get(c)
                    if s is None:
                        s = reprs[c] = json.dumps(c)
                    parts.append('"%s": %s' % (chr(self.nts[r, j]), s))
                f.write('{"id": %d, "chromosome": %s, "position": %d%s}\n' % (
                    self.ids[r], json.dumps(self.chrom_labels[self.chrom_idx[r]]), self.position[r],
                    (', "tuples": {%s}' % ", ".join(parts)) if k else ""))

    @classmethod
    def read_json_gz(cls, path):
        with gzip.open(path, "rt") as f:
            return [SNPTuples.from_json(line) for line in f]

    @classmethod
    def read_json_gz_table(cls, path):
        """The same file straight into column form (native parser, no object per SNP); None when some record
        does not fit the column form (string ids, multi-character alleles, ...): use read_json_gz then."""
        with gzip.open(path, "rb") as f:
            cols = _native.parse_snps_jsonl(f.read())
        if cols is None:
            return None
        return cls(cols["ids"], cols["chrom_idx"], cols["chrom_labels"], cols["position"], cols["n_alleles"], cols["nts"],
                   cols["cum"])


class SnpFactory:
    """Frequency-CDF SNP selection (pop_factory.py:136-193).

    The draws use numpy's global legacy RandomState and Python's `random` in the reference's own order
    (chromosomes, MAFs, position uniforms, reference nucleotides, then one `random.choice` per SNP for
    the alternate allele), so a run seeded like the reference selects the same SNPs.
    """

    def __init__(self, cdf_matrix):
        cdf_matrix = np.asarray(cdf_matrix, dtype=np.float64)
        self.sorted_maf = cdf_matrix[:, 0]
        self.cdf = cdf_matrix[:, 1]
        self.pdf = self.cdf - np.concatenate(([0.0], self.cdf[:-1]))

    @classmethod
    def init_from_cdf_file(cls, file=None):
        if file is None:
            return cls(np.asarray(MAF_CDF, dtype=np.float64))
        return cls(np.loadtxt(file, skiprows=1, delimiter=","))

    def _first_bin(self, min_maf):
        hits = np.nonzero(min_maf <= self.sorted_maf)[0]
        return int(hits[0]) if len(hits) else 0

    def gen_mafs(self, size, min_maf):
        start = self._first_bin(min_maf)
        p = self.pdf[start:]
        return np.random.choice(self.sorted_maf[start:], size=size, p=p * 1 / np.sum(p))

    def gen_chromosomes(self, size):
        return np.random.choice(CHROMOSOME_LIST, size=size, p=CHROMOSOME_PROB)

    def random_snp_table(self, size, min_maf=0.005, vector_alt=False):
        """SnpTable of `size` random SNPs.  vector_alt=True draws the alternate allele with numpy in one
        call instead of `size` calls to random.choice (faster; no longer stream-compatible upstream)."""
        chromosomes = self.gen_chromosomes(size)
        mafs = self.gen_mafs(size, min_maf)
        position_randoms = np.random.random(size)
        nt_randoms = np.random.choice(NUCLEOTIDES, size=size)
        labels = np.asarray(CHROMOSOME_LIST)
        order = np.argsort(labels, kind="stable")
        ci = order[np.searchsorted(labels[order], chromosomes)].astype(np.int32)
        max_pos = np.asarray([CHROMOSOME_MAX_POSITION[c] for c in CHROMOSOME_LIST], dtype=np.float64)
        position = (position_randoms * max_pos[ci]).astype(np.int64)          # int(u * max_position)
        ref = nt_randoms.astype("S1").view(np.uint8) if size else np.zeros(0, np.uint8)
        codes = np.frombuffer(b"ATCG", dtype=np.uint8)
        ref_idx = np.argsort(codes, kind="stable")[np.searchsorted(np.sort(codes), ref)]
        if vector_alt:
            pick = np.random.randint(0, 3, size=size)
        else:
            pick = np.fromiter((random.choice((0, 1, 2)) for _ in range(size)), dtype=np.int64, count=size)
        # remaining nucleotides keep A,T,C,G order with the reference removed (list.remove semantics)
        alt_idx = pick + (pick >= ref_idx)
        alt = codes[alt_idx] if size else np.zeros(0, np.uint8)
        nts = np.zeros((size, _native.KMAX), np.uint8)
        nts[:, 0] = ref
        nts[:, 1] = alt
        cum = np.full((size, _native.KMAX), 2.0)
        cum[:, 0] = 1 - mafs
        cum[:, 1] = 1.0
        return SnpTable(np.arange(1, size + 1), ci, CHROMOSOME_LIST, position, np.full(size, 2, np.uint8), nts, cum)

    def random_snp_tuples(self, size, min_maf=0.005):
        return self.random_snp_table(size, min_maf).to_snps()

    # ---- the same selection on the GPU (counter-based stream instead of numpy's global state) ---------
    def selection_tables(self, min_maf=0.005):
        """What the device sampler needs: the two cumulative tables exactly as numpy.random.choice builds them
        (cdf = p.cumsum(); cdf /= cdf[-1]), chromosome lengths and the string-order rank of every label."""
        start = self._first_bin(min_maf)
        p = self.pdf[start:]
        p = p * 1 / np.sum(p)                                   # pop_factory.py:166-167
        maf_cdf = p.cumsum()
        maf_cdf /= maf_cdf[-1]
        chrom_cdf = np.asarray(CHROMOSOME_PROB, dtype=np.float64).cumsum()
        chrom_cdf /= chrom_cdf[-1]
        labels = np.asarray(CHROMOSOME_LIST)
        rank = np.argsort(np.argsort(labels, kind="stable"), kind="stable").astype(np.uint8)
        max_pos = np.asarray([CHROMOSOME_MAX_POSITION[c] for c in CHROMOSOME_LIST], dtype=np.float64)
        return dict(start=start, maf_cdf=maf_cdf, chrom_cdf=chrom_cdf, chrom_rank=rank, chrom_max_pos=max_pos)

    def table_from_columns(self, cols, start, first_id=1):
        """SnpTable from the sampler's columns (device or oracle): tuples [(ref, 1 - maf), (alt, 1.0)]."""
        size = len(cols["order"])
        mafs = self.sorted_maf[start:][cols["maf_bin"]]
        nts = np.zeros((size, _native.KMAX), np.uint8)
        nts[:, 0] = cols["ref"]
        nts[:, 1] = cols["alt"]
        cum = np.full((size, _native.KMAX), 2.0)
        cum[:, 0] = 1 - mafs                                    # pop_factory.py:187
        cum[:, 1] = 1.0
        return SnpTable(cols["order"].astype(np.int64) + first_id, cols["chrom_idx"].astype(np.int32), CHROMOSOME_LIST,
                        cols["position"].astype(np.int64), np.full(size, 2, np.uint8), nts, cum)

    def random_snp_table_device(self, engine, size, seed, min_maf=0.005, sort=True):
        """`size` random SNPs drawn (and, by default, sorted like pop_factory.py:245) on the GPU."""
        t = self.selection_tables(min_maf)
        cols = engine.select_snps(size, seed, t["chrom_cdf"], t["chrom_max_pos"], t["chrom_rank"], t["maf_cdf"], sort=sort)
        return self.table_from_columns(cols, t["start"])
