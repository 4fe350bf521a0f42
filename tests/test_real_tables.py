"""SNP tables shaped like a real --snps_file against the row kernels (k_auto, k_lz, k_x, k_fused_text) and the oracle.

SnpFactory output has single-base alleles, short positions and ids and at most 99 distinct MAFs, so its row leads are
26 to 38 bytes long and its first thresholds fit in one MAF bucket each.  Records exported from RefSNP differ on both
counts: leads of 39 to 64 bytes (9-digit positions, 10-digit ids, indels, ALT lists) and longer ones, and thousands
of distinct, continuous first thresholds, which make prepare_buckets (host_tables.h) coarsen its keys and build every
table for the midpoint of a key range.  Each population here is built once as flat arrays; the same arrays go to the
Engine and to oracle.rows_from_flat, which prints whatever prefix bytes it is given, so the tests choose the prefix
length and content of every row exactly.

Assertions: the decompressed text equals the oracle's; every BGZF block is well formed (magic, BSIZE, CRC32 and ISIZE
of what it inflates to: oracle.bgzf_decompress) and their count is the call's `bgzf_blocks`; compressed bytes are
compared only between two calls on one context state."""
import gzip
import json
import os
import random
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest

from tests.cases import Sample, Snp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AUTO, X, Y, MT = 0, 1, 2, 3
CHROM = {AUTO: b"1", X: b"X", Y: b"Y", MT: b"MT"}
TWO32 = 1 << 32
LAST = 0xFFFFFFFF
BASES = "ACGT"
PASS_RE = re.compile(r"\[dnaf\] pass rows \d+ implicit \d+ blocks \d+ auto (\d+) x (\d+) text (\d+) generic (\d+):")


# ----------------------------------------------------------------------------------------------------------- helpers
def lead(L, chrom="1", seed=0):
    """A row lead "CHROM\\tPOS\\trsID\\tREF\\tALT\\t40\\tPASS\\t.\\tGT\\t" (pop_factory.py:503-507) of exactly L bytes, as
    real records make them: the position grows to 9 digits, the id to 10, then REF and ALT grow (an indel, or an
    ALT list such as "C,G,T")."""
    rs = random.Random(L * 7919 + seed)
    room = L - len(chrom) - 20 - 4        # bytes beyond a 1-digit position, 1-digit id, 1-base REF and ALT
    if room < 0:
        raise ValueError("a %r lead needs at least %d bytes" % (chrom, len(chrom) + 24))
    pos_d = 1 + min(room, 8)
    room -= pos_d - 1
    id_d = 1 + min(room, 9)
    room -= id_d - 1
    ref_len = 1 + room // 2
    alt_len = 1 + room - room // 2
    pos = rs.randint(10 ** (pos_d - 1) if pos_d > 1 else 1, 10 ** pos_d - 1)
    rsid = rs.randint(10 ** (id_d - 1) if id_d > 1 else 1, 10 ** id_d - 1)
    ref = "".join(rs.choice(BASES) for _ in range(ref_len))
    if alt_len in (3, 5, 7):                # an ALT list of single bases
        alt = ",".join(rs.choice(BASES) for _ in range((alt_len + 1) // 2))
    else:
        alt = "".join(rs.choice(BASES) for _ in range(alt_len))
    out = ("%s\t%d\trs%d\t%s\t%s\t40\tPASS\t.\tGT\t" % (chrom, pos, rsid, ref, alt)).encode()
    assert len(out) == L
    return out


def arbitrary_prefix(L, rs, tab=True):
    """L bytes that are no row lead (any byte but '\\n'); the last one is a tab, or never one."""
    b = bytearray(rs.choice([c for c in range(1, 256) if c != 10], size=L).astype(np.uint8).tobytes())
    if L:
        b[-1] = 9 if tab else rs.choice([c for c in range(33, 127)])
        if not tab:
            assert b[-1] != 9
    return bytes(b)


def body_bytes(cls, sex):
    """Text bytes of a row's genotype cells (dnaf_set_samples: 0/0 per sample, haploid X cells of males, Y and MT)."""
    n = len(sex)
    if n == 0:
        return 1
    if cls == AUTO:
        return 4 * n
    if cls == X:
        return int(sum(2 if s == 1 else 4 for s in sex))
    return 2 * n


def row_kind(cls, k, prefix, sex):
    """Which kernel takes a row (row_kind, host_plan.h, with the fused path on): 0 the generic three-kernel path,
    1 k_auto (k_lz at -z 3..9), 2 k_fused_text, 3 k_x."""
    if len(sex) == 0 or not 1 <= len(prefix) <= 64 or body_bytes(cls, sex) < 4096:
        return 0
    if k <= 2 and cls == AUTO:
        return 1 if prefix.endswith(b"\t") else 2
    if k <= 2 and cls == X:
        return 3
    return 2


def auto_segments(n):
    """Sample segments of an autosome or X row (build_segments): at most 254 spans of 64 samples each."""
    spans = (n + 63) // 64
    return (spans + 253) // 254


def text_segments(body):
    """k_fused_text segments of a class body (build_segments): balanced multiples of 256 bytes."""
    sp = (body + 255) // 256
    ns = (sp + 253) // 254
    pr = (sp + ns - 1) // ns
    return sum(1 for sg in range(ns) if sg * pr * 256 < body)


def first_threshold(maf):
    return min(int((1.0 - maf) * TWO32), TWO32 - 2)


def thresholds(rs, k, t0=None):
    """Sorted thresholds of a K-allele row (the last allele takes what is left: 2^32 - 1)."""
    if k == 1:
        return [LAST] * 4
    if t0 is None:
        t0 = int(rs.randint(1, TWO32 - 2))
    t = [t0] + sorted(int(x) for x in rs.randint(t0, TWO32 - 1, size=k - 2)) + [LAST]
    return t + [LAST] * (4 - k)


def population(n, seed, male_frac=0.5):
    """Samples (odd ones are cases, so both the first and the last span of a row hold cases) as oracle.flatten lays
    them out."""
    from oracle import oracle
    rs = np.random.RandomState(seed)
    samples = [Sample(family_id=i + 1, person_id=100001 + i, father_id=0, mother_id=0,
                      sex=1 if rs.rand() < male_frac else 2, is_control=i % 2 == 0,
                      deleterious_snps=None if i % 2 == 0 else {}) for i in range(n)]
    return oracle.flatten(samples, [])


def build_table(pop, rows, overrides):
    """rows: (class, K, thresholds[4], prefix bytes); overrides: (row, sample) pairs.  -> (oracle flat dict, Engine
    set_snps arguments, override rows, override samples)."""
    S = len(rows)
    cls = np.array([r[0] for r in rows], np.uint8)
    k = np.array([r[1] for r in rows], np.uint8)
    thr = np.array([r[2] for r in rows], np.uint32).reshape(S, 4)
    cum = np.full((S, 4), 2.0)
    for i in range(S):
        for j in range(k[i]):
            cum[i, j] = 1.0 if j == k[i] - 1 else thr[i, j] / float(TWO32)    # exact: threshold(cum) == thr
    pre = [r[3] for r in rows]
    off = np.zeros(S + 1, np.uint64)
    off[1:] = np.cumsum([len(p) for p in pre])
    pre_b = np.frombuffer(b"".join(pre) + b"\0", np.uint8).copy()
    chrom = [CHROM[int(c)] for c in cls]
    coff = np.zeros(S + 1, np.uint64)
    coff[1:] = np.cumsum([len(c) for c in chrom])
    pairs = sorted(set((int(r), int(s)) for r, s in overrides))
    orow = np.array([p[0] for p in pairs], np.uint64)
    osamp = np.array([p[1] for p in pairs], np.uint32)
    assert all(pop["is_control"][s] == 0 for s in osamp), "forced minors fall on cases only"
    flat = dict(pop, chrom_bytes=np.frombuffer(b"".join(chrom) + b"\0", np.uint8).copy(), chrom_off=coff,
                prefix_bytes=pre_b, prefix_off=off, K=k, cum=cum, over_row=orow, over_sample=osamp)
    arrays = dict(chrom_class=cls, n_alleles=k, thresholds=thr, prefix_bytes=pre_b, prefix_off=off)
    return flat, arrays, orow, osamp


def oracle_text(flat, seed):
    from oracle import oracle
    return oracle.rows_from_flat(flat, seed, 0, n_threads=8)[0].tobytes()


def engine(pop, arrays, orow, osamp, chunk=None):
    from dna_factory_b200 import _native
    eng = _native.Engine(0)
    eng.set_samples(pop["sex"], pop["is_control"])
    eng.set_snps(**arrays)
    eng.set_overrides(orow, osamp)
    if chunk:
        eng.set_chunk_bytes(chunk)
    return eng


def check_blob(blob, st, want):
    """Every block well formed, as many as the call reports, inflating to the oracle's text."""
    from oracle import oracle
    text, blocks, eof = oracle.bgzf_decompress(blob)
    assert blocks == st["bgzf_blocks"] and not eof
    assert text == want


# ------------------------------------------------------------------------------------------------------------- CPU
def test_lead_has_its_length_and_fields():
    from dna_factory_b200 import host
    for chrom in ("1", "X", "MT", "22"):
        for L in range(27, 81):
            b = lead(L, chrom, seed=L)
            assert len(b) == L
            f = b.decode().split("\t")
            assert len(f) == 10 and f[0] == chrom and f[5:] == ["40", "PASS", ".", "GT", ""]
            assert f[1].isdigit() and f[2].startswith("rs") and f[2][2:].isdigit()
            assert set(f[3]) <= set(BASES) and set(f[4]) <= set(BASES + ",")
            alts = f[4].split(",")
            tuples = [(f[3], 0.5)] + [(a, 0.5 + 0.1 * (i + 1)) for i, a in enumerate(alts[:-1])] + [(alts[-1], 1.0)]
            snp = Snp(id=int(f[2][2:]), chromosome=chrom, position=int(f[1]), tuples=tuples)
            assert host.row_prefix(snp).encode() == b
    # the position and the id reach real widths before the alleles grow
    f = lead(64).decode().split("\t")
    assert (len(f[1]), len(f[2]) - 2) == (9, 10) and len(f[3]) + len(f[4]) == 64 - 20 - 1 - 9 - 10
    with pytest.raises(ValueError):
        lead(24)


def test_row_kind_edges():
    tab, notab = b"1\t2\trs3\tA\tC\t40\tPASS\t.\tGT\t", b"x" * 30
    f1023, f1024 = [2] * 1023, [2] * 1024
    m2047, m2048 = [1] * 2047, [1] * 2048
    cases = [
        ((AUTO, 2, b"\t", f1024), 1), ((AUTO, 2, b"a\t" * 32, f1024), 1), ((AUTO, 2, b"a" + b"\t" * 64, f1024), 0),
        ((AUTO, 2, b"", f1024), 0), ((AUTO, 2, b"y", f1024), 2), ((AUTO, 2, notab, f1024), 2),
        ((AUTO, 2, tab, f1023), 0), ((AUTO, 2, tab, f1024), 1), ((AUTO, 1, tab, f1024), 1), ((AUTO, 3, tab, f1024), 2),
        ((AUTO, 4, tab, f1024), 2), ((X, 2, tab, f1024), 3), ((X, 2, notab, f1024), 3), ((X, 3, tab, f1024), 2),
        ((X, 2, tab, m2047), 0), ((X, 2, tab, m2048), 3), ((X, 2, b"\t" * 65, m2048), 0),
        ((Y, 2, tab, f1024), 0), ((Y, 2, tab, [2] * 2048), 2), ((MT, 1, tab, m2047), 0), ((MT, 2, tab, m2048), 2),
        ((AUTO, 2, tab, []), 0),
    ]
    for args, want in cases:
        assert row_kind(*args) == want, (args[:2], len(args[2]), len(args[3]))
    assert [auto_segments(n) for n in (4096, 4097, 16256, 16257, 20000)] == [1, 1, 1, 2, 2]
    assert [text_segments(b) for b in (8192, 65024, 65025, 80000)] == [1, 1, 2, 2]


def _segment(n_cells, p, seed, lead_tab, ends_row):
    """Allele bits of one autosome segment at minor-allele rate p and its text (k_lz's block body)."""
    rs = np.random.RandomState(seed)
    alleles = (rs.rand(2 * n_cells) < p).astype(np.uint8)
    bits = np.zeros((2 * n_cells + 31) // 32 + 1, dtype=np.uint32)
    idx = np.nonzero(alleles)[0]
    np.bitwise_or.at(bits, idx >> 5, (np.uint32(1) << (idx & 31).astype(np.uint32)))
    t = np.empty(4 * n_cells, np.uint8)
    t[0::4] = alleles[0::2] + 48
    t[1::4] = ord("/")
    t[2::4] = alleles[1::2] + 48
    t[3::4] = 9
    body = t.tobytes()[:-1] + (b"\n" if ends_row else b"")
    return bits, (b"\t" if lead_tab else b"") + body


def _lz_roundtrip(p_table, level, bits, n_cells, prefix, text, ends_row):
    from dna_factory_b200 import _native
    enc = _native.debug_lz_block(p_table, level, bits, n_cells, prefix, ends_row)
    assert zlib.decompress(enc, -15) == prefix + text, (p_table, level, len(prefix), n_cells)


@pytest.mark.parametrize("level", [3, 6, 9])
def test_lz_twin_every_prefix_length(level):
    """The host twin of k_lz with row leads of 0 (a segment that does not start its row) to 64 bytes."""
    rs = np.random.RandomState(level)
    for L in range(0, 65):
        n_cells = (1000, 64, 16256)[L % 3] if L != 64 else 16256       # 64 + 4 * 16256 bytes: the largest block
        prefix = lead(L, seed=level) if L >= 27 else arbitrary_prefix(L, rs)
        bits, text = _segment(n_cells, 0.03 + 0.005 * L, 1000 * level + L, L == 0, L % 2 == 0)
        _lz_roundtrip(0.03 + 0.005 * L, level, bits, n_cells, prefix, text, L % 2 == 0)


@pytest.mark.parametrize("level", [3, 6, 9])
def test_lz_twin_prefixes_with_high_bytes(level):
    """Latin-1 bytes in the lead (an id or a label exported in Latin-1): each needs a literal code of its own."""
    rs = np.random.RandomState(100 + level)
    for L in (1, 2, 17, 33, 40, 63, 64):
        high = bytes(rs.randint(0x80, 0x100, size=L - 1).astype(np.uint8)) + b"\t"
        latin = (b"1\t123456789\trs98765\xe9_ab\tA\tC\t40\tPASS\t.\tGT\t" * 2)[-L:]
        for j, prefix in enumerate((high, latin)):
            bits, text = _segment(2000, 0.1, L + 7 * j, False, True)
            _lz_roundtrip(0.1, level, bits, 2000, prefix, text, True)


@pytest.mark.parametrize("level", [3, 4, 6, 9])
def test_lz_twin_rates_off_the_table(level):
    """A coarsened bucket builds its tables for the midpoint p of a key range (0.00049 for the last range at a 22-bit
    shift) and holds rows far from it, K = 1 rows among them; a bucket of K = 1 rows alone has p = 0 and may still
    carry forced minors."""
    prefix = lead(44, seed=level)
    for p_table, rates in ((0.00049, (0.0, 0.001, 0.01)), (0.0, (0.0, 0.01)), (0.00098, (0.0, 0.004)),
                           (0.49, (0.0, 0.001))):
        for i, p_data in enumerate(rates):
            for n_cells, starts in ((16256, True), (777, False)):
                bits, text = _segment(n_cells, p_data, 10 * level + i, not starts, True)
                _lz_roundtrip(p_table, level, bits, n_cells, prefix if starts else b"", text, True)


# ------------------------------------------------------------------------------------------------------------- GPU
LENGTH_SIZES = [4096, 4097, 16256, 16257, 20000]
NOTAB_LENGTHS = [1, 31, 32, 33, 63, 64, 65]
BIG_LENGTHS = [0, 65000, 70000]


def prefix_rows(n, seed):
    """One row per prefix length 1..80 in each of three classes (autosome K = 2; X K = 2; Y, MT, or autosome K = 3 / 4
    in turn), autosome rows without a final tab, autosome rows with 0, 65 000 and 70 000-byte prefixes, and forced
    minors on the first and last case of some long-prefix rows.  The autosome rows of leads up to 32 bytes open the
    table (an implicit k_auto run); the rest is shuffled, so generic rows sit between k_auto rows."""
    rs = np.random.RandomState(seed)
    head, rest = [], []
    for L in range(1, 81):
        maf = float(np.exp(rs.uniform(np.log(1e-3), np.log(0.5))))
        pre = lead(L, "1", seed) if L >= 27 else arbitrary_prefix(L, rs)
        (head if L <= 32 else rest).append((AUTO, 2, thresholds(rs, 2, first_threshold(maf)), pre))
        pre = lead(L, "X", seed) if L >= 27 else arbitrary_prefix(L, rs)
        rest.append((X, 2, thresholds(rs, 2, first_threshold(maf)), pre))
        cls, k = [(Y, 2), (MT, 2), (AUTO, 3), (AUTO, 4)][L % 4]
        chrom = {Y: "Y", MT: "MT", AUTO: "1"}[cls]
        pre = lead(L, chrom, seed) if L >= 27 else arbitrary_prefix(L, rs)
        rest.append((cls, k, thresholds(rs, k), pre))
    for L in NOTAB_LENGTHS:
        rest.append((AUTO, 2, thresholds(rs, 2), arbitrary_prefix(L, rs, tab=False)))
    for L in BIG_LENGTHS:
        pre = lead(L, "1", seed) if L else b""
        rest.append((AUTO, 2, thresholds(rs, 2, first_threshold(0.2)), pre))
    order = rs.permutation(len(rest))
    rows = head + [rest[i] for i in order]
    first_case, last_case = 1, n - 1 if (n - 1) % 2 == 1 else n - 2
    over = []
    for r, row in enumerate(rows):
        if len(row[3]) >= 33 and r % 3 == 0:
            over += [(r, first_case), (r, last_case), (r, 63 if row[0] != X else 65)]
    return rows, over


def length_case(n):
    seed = 0x5EED0 + n
    pop = population(n, seed)
    rows, over = prefix_rows(n, seed)
    flat, arrays, orow, osamp = build_table(pop, rows, over)
    return seed, pop, rows, flat, arrays, orow, osamp


@pytest.fixture(scope="module")
def oracle_mod():
    from oracle import oracle
    oracle.build()
    return oracle


@pytest.mark.gpu
@pytest.mark.parametrize("n", LENGTH_SIZES)
def test_every_prefix_length_through_every_kernel(n, oracle_mod):
    seed, pop, rows, flat, arrays, orow, osamp = length_case(n)
    sex = pop["sex"]
    kinds = [row_kind(c, k, p, sex) for c, k, _, p in rows]
    # the table covers every prefix length on every class
    hist = {}
    for (c, k, _, p), kind in zip(rows, kinds):
        hist.setdefault((c == AUTO and k <= 2 and p.endswith(b"\t"), c == X, c in (Y, MT) or k > 2), set()).add(len(p))
    for key in ((True, False, False), (False, True, False), (False, False, True)):
        assert hist[key] >= set(range(1, 81)), key
    assert {len(p) for (c, k, _, p) in rows if c == AUTO and k == 2 and not p.endswith(b"\t")} >= set(NOTAB_LENGTHS)
    on = {kd: {len(p) for (_, _, _, p), kind in zip(rows, kinds) if kind == kd} for kd in (0, 1, 2, 3)}
    assert on[1] >= set(range(33, 65)) and on[3] >= set(range(33, 65)) and on[2] >= set(range(33, 65))
    assert on[0] >= {0, 65, 80, 65000, 70000} and not on[1] & {0, 65}
    assert any(len(rows[int(r)][3]) > 32 for r in orow)
    auto_text = sum(len(p) + body_bytes(AUTO, sex) for (_, _, _, p), kind in zip(rows, kinds) if kind == 1)
    want = oracle_text(flat, seed)
    S = len(rows)
    eng = engine(pop, arrays, orow, osamp)
    try:
        for chunk in (64 << 20, len(want) // 6):
            eng.set_chunk_bytes(chunk)
            for level in (1, 2, 3, 6, 9):
                blob, st = eng.generate(0, S, seed, level=level)
                check_blob(blob, st, want)
                # k_auto (k_lz at -z 3..9) took exactly the rows row_kind gives it: prefix + cells of each
                assert st["auto_text_bytes"] == auto_text, (chunk, level)
                assert st["ms_fused"] > 0 and st["text_bytes"] == len(want)
                if chunk < len(want):
                    assert st["auto_launches"] > 1
    finally:
        eng.close()


def trace_child(n, out_path):
    """Runs in a child process with DNAF_TRACE=1: the length table of n samples at -z 2 and -z 6, a chunk for the whole
    table and one that cuts passes; the pass lines go to stderr, the blobs to out_path."""
    seed, pop, rows, flat, arrays, orow, osamp = length_case(n)
    blobs = []
    for chunk in (64 << 20, 1 << 20):
        eng = engine(pop, arrays, orow, osamp, chunk)
        for level in (2, 6):
            sys.stderr.write("[run] %d %d\n" % (chunk, level))
            sys.stderr.flush()
            blobs.append(eng.generate(0, len(rows), seed, level=level)[0])
            sys.stderr.flush()
        eng.close()
    with open(out_path, "wb") as f:
        f.write(json.dumps([len(b) for b in blobs]).encode() + b"\n" + b"".join(blobs))


@pytest.mark.gpu
def test_kernel_block_counts(tmp_path, oracle_mod):
    """DNAF_TRACE=1 prints the blocks each pass gives k_auto (k_lz), k_x, k_fused_text and the generic path: their
    sums are what row_kind and the segment rules give, so the 33-64-byte rows of the table run on the fused kernels."""
    n = 16257    # two sample segments per autosome and X row
    seed, pop, rows, flat, arrays, orow, osamp = length_case(n)
    sex = pop["sex"]
    kinds = [row_kind(c, k, p, sex) for c, k, _, p in rows]
    want_auto = sum(kd == 1 for kd in kinds) * auto_segments(n)
    want_x = sum(kd == 3 for kd in kinds) * auto_segments(n)
    want_text = sum(text_segments(body_bytes(c, sex)) for (c, _, _, _), kd in zip(rows, kinds) if kd == 2)
    assert sum(kd == 1 and 33 <= len(p) <= 64 for (_, _, _, p), kd in zip(rows, kinds)) == 32
    assert sum(kd == 3 and 33 <= len(p) <= 64 for (_, _, _, p), kd in zip(rows, kinds)) == 32
    out = str(tmp_path / "blobs")
    env = dict(os.environ, DNAF_TRACE="1", DNAF_RAMP="0")
    env.pop("DNAF_FULL_PLAN", None)
    code = "import sys; sys.path.insert(0, %r); from tests.test_real_tables import trace_child; trace_child(%d, %r)" % (
        ROOT, n, out)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    runs, cur = [], None
    for line in r.stderr.splitlines():
        if line.startswith("[run] "):
            cur = [0, 0, 0, 0, 0]
            runs.append(cur)
        m = PASS_RE.search(line)
        if m and cur is not None:
            for i in range(4):
                cur[i] += int(m.group(i + 1))
            cur[4] += 1
    assert len(runs) == 4
    for auto, x, text, generic, passes in runs:
        assert (auto, x, text) == (want_auto, want_x, want_text)
        assert generic > 0
    assert runs[2][4] > 1 and runs[3][4] > 1, "the 1 MiB chunk must cut the table into several passes"
    with open(out, "rb") as f:
        sizes = json.loads(f.readline())
        data = f.read()
    want = oracle_text(flat, seed)
    pos = 0
    for size in sizes:
        assert oracle_mod.bgzf_decompress(data[pos:pos + size])[0] == want
        pos += size


def coarse_rows(seed, S=2400):
    """A real-file mix: continuous, log-uniform MAFs from 1e-5 to 0.5, thresholds next to 0 and next to 2^32 - 1,
    K = 1, 3 and 4 rows, X, Y and MT rows, leads of 26 to 70 bytes; sorted by chromosome label like a VCF."""
    rs = np.random.RandomState(seed)
    rows = []
    edge = [0, 1, 2, 3, 1 << 20, TWO32 - 2, TWO32 - 3, TWO32 - 5, TWO32 - (1 << 21)]
    for i in range(S):
        u = rs.rand()
        chrom = "1" if u < 0.88 else ("X" if u < 0.94 else ("Y" if u < 0.97 else "MT"))
        cls = {"X": X, "Y": Y, "MT": MT}.get(chrom, AUTO)
        v = rs.rand()
        k = 1 if v < 0.02 else (3 if v < 0.04 else (4 if v < 0.05 else 2))
        if i < len(edge):
            k = 2
        if i < len(edge):
            t = thresholds(rs, 2, edge[i])
        elif k >= 2:
            maf = float(np.exp(rs.uniform(np.log(1e-5), np.log(0.5))))
            t = thresholds(rs, k, first_threshold(maf) if k == 2 else None)
        else:
            t = thresholds(rs, 1)
        L = int(rs.choice([26, 30, 38, 42, 44, 47, 52, 58, 64, 66, 70])) + (len(chrom) - 1)
        rows.append((chrom, cls, k, t, lead(L, chrom, seed=i)))
    rows.sort(key=lambda r: r[0])
    return [r[1:] for r in rows]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4096, 20000])
def test_coarsened_buckets_in_one_call(n, oracle_mod):
    """More than 2 048 distinct first thresholds: prepare_buckets raises its shift until at most 512 keys remain, and
    every table is built for the midpoint p of its key range."""
    seed = 0xC0A5E + n
    pop = population(n, seed, male_frac=0.4)
    rows = coarse_rows(seed)
    rs = np.random.RandomState(seed)
    cases = np.nonzero(pop["is_control"] == 0)[0]
    over = [(int(r), int(s)) for r in rs.choice(len(rows), 60, replace=False) for s in rs.choice(cases, 5, replace=False)]
    flat, arrays, orow, osamp = build_table(pop, rows, over)
    first = {r[2][0] for r in rows if r[1] >= 2}
    assert len(first) > 2048
    assert {r[0] for r in rows} == {AUTO, X, Y, MT} and {r[1] for r in rows} == {1, 2, 3, 4}
    assert min(first) <= 3 and max(first) >= TWO32 - 3
    want = oracle_text(flat, seed)
    S = len(rows)
    cuts = [0, S // 3, S // 3 + 1, S]
    eng = engine(pop, arrays, orow, osamp)
    try:
        for level in range(1, 10):
            blob, st = eng.generate(0, S, seed, level=level)
            check_blob(blob, st, want)
            assert st["ms_fused"] > 0
            parts = b""
            for a, b in zip(cuts, cuts[1:]):
                part, st_part = eng.generate(a, b, seed, level=level)
                assert oracle_mod.bgzf_decompress(part)[1] == st_part["bgzf_blocks"]
                parts += part
            assert oracle_mod.bgzf_decompress(parts)[0] == want, "level %d: ranges do not concatenate" % level
            if level == 2:
                st_f = st
        eng.set_fused(False)
        plain, st_p = eng.generate(0, S, seed, level=2)
        assert st_p["ms_fused"] == 0
        check_blob(plain, st_p, want)
        # the static codes of coarsened buckets must stay close to the per-block dynamic codes
        assert st_f["bgzf_bytes"] < 1.10 * st_p["bgzf_bytes"] + 4096, (st_f["bgzf_bytes"], st_p["bgzf_bytes"])
    finally:
        eng.close()


def batch_rows(seed, S, x_rows, new_bytes):
    rs = np.random.RandomState(seed)
    rows = []
    for i in range(S):
        cls = X if (x_rows and i % 7 == 3) else AUTO
        chrom = "X" if cls == X else str(1 + i % 22)
        maf = float(rs.uniform(0.001, 0.5))
        pre = lead(int(rs.randint(27, 60)), chrom, seed=seed + i)
        if new_bytes and i % 5 == 0:
            f = pre.split(b"\t")
            f[2] += b"_a\xe9"[: 1 + i % 3]
            f[3] = f[3].lower()
            pre = b"\t".join(f)
        rows.append((cls, 2, thresholds(rs, 2, first_threshold(maf)), pre))
    return rows


@pytest.mark.gpu
def test_bucket_map_across_set_snps_calls(oracle_mod):
    """One context, batches A, B, A: B's thresholds take the key -> bucket map past 512 (the shift rises and every
    bucket is renumbered mid-session), B brings the first X rows and new prefix bytes (lowercase, '_', a Latin-1
    byte) that the literal codes must gain, and A again runs on the coarsened map."""
    from dna_factory_b200 import _native
    n = 4500
    seed = 0xB0C4E7
    pop = population(n, seed)
    a = batch_rows(11, 420, False, False)
    b = batch_rows(12, 420, True, True)
    ta, tb = {r[2][0] for r in a}, {r[2][0] for r in b}
    assert len(ta) < 512 < len(ta | tb)                 # distinct keys at the unshifted start: A fits, A then B does not
    cases = np.nonzero(pop["is_control"] == 0)[0]
    batches = []
    for name, rows in (("A", a), ("B", b), ("C", a)):
        over = [(r, int(cases[(7 * r) % len(cases)])) for r in range(0, len(rows), 9)] + [(5, int(cases[-1]))]
        flat, arrays, orow, osamp = build_table(pop, rows, over)
        batches.append((name, arrays, orow, osamp, oracle_text(flat, seed)))
    pb = set(b"".join(r[3] for r in b))
    assert not pb <= set(b"".join(r[3] for r in a)) and {ord("_"), 0xE9, ord("a")} <= pb
    eng = _native.Engine(0)
    eng.set_samples(pop["sex"], pop["is_control"])
    try:
        for name, arrays, orow, osamp, want in batches:
            eng.set_snps(**arrays)
            eng.set_overrides(orow, osamp)
            S = len(arrays["n_alleles"])
            for level in (2, 6):
                blob, st = eng.generate(0, S, seed, level=level)
                check_blob(blob, st, want)
                assert st["ms_fused"] > 0
                again, _ = eng.generate(0, S, seed, level=level)
                assert again == blob, "%s -z %d: a repeated call on the same state differs" % (name, level)
                with _native.Engine(0) as fresh:
                    fresh.set_samples(pop["sex"], pop["is_control"])
                    fresh.set_snps(**arrays)
                    fresh.set_overrides(orow, osamp)
                    blob2, st2 = fresh.generate(0, S, seed, level=level)
                    check_blob(blob2, st2, want)
    finally:
        eng.close()


def _fixed_clock(monkeypatch):
    from dna_factory_b200 import pop_factory

    class FixedDatetime(pop_factory.datetime):
        @classmethod
        def now(cls, tz=None):
            return cls(2026, 1, 1, 12, 34, 56)

    monkeypatch.setattr(pop_factory, "datetime", FixedDatetime)


def real_snps(seed, S, multibase):
    """SNP records as a RefSNP export gives them: continuous frequencies, 9-digit positions on chromosome 1, 10-digit
    ids, ALT lists; with `multibase`, indels (multi-base REF / ALT) too."""
    rs = np.random.RandomState(seed)
    chroms = ["1", "10", "22", "MT", "X", "Y"]
    snps, used = [], set()
    for i in range(S):
        chrom = chroms[int(rs.choice(6, p=[0.5, 0.2, 0.15, 0.03, 0.09, 0.03]))]
        pos = int(rs.randint(100_000_000, 248_000_000)) if chrom == "1" else int(rs.randint(1, 150_000_000))
        if (chrom, pos) in used:
            continue
        used.add((chrom, pos))
        k = int(rs.choice([2, 3, 4], p=[0.9, 0.07, 0.03]))
        nts = list(rs.permutation(list(BASES)))[:k]
        if multibase and i % 3 == 0:
            nts = [nts[0] + "".join(rs.choice(list(BASES), size=rs.randint(1, 30)))] + nts[1:]
        if multibase and i % 4 == 1:
            nts[-1] = nts[-1] + "".join(rs.choice(list(BASES), size=rs.randint(1, 9)))
        maf = float(np.exp(rs.uniform(np.log(0.002), np.log(0.5))))
        cum = sorted(float(x) for x in rs.uniform(1 - maf, 1, size=k - 1))
        cum[0] = round(1 - maf, 12)
        tuples = [(nt, c) for nt, c in zip(nts, cum + [1.0])]
        snps.append(Snp(id=int(rs.randint(1_000_000_000, 4_000_000_000)), chromosome=chrom, position=pos, tuples=tuples))
    return snps


@pytest.mark.gpu
@pytest.mark.parametrize("multibase", [False, True])
def test_cli_snps_file_real_records(tmp_path, monkeypatch, multibase, oracle_mod):
    """pop_factory --snps_file at -z 6 on 2 100 cases and 2 100 controls (fused kernels): a file the native parser
    keeps in column form, and one with indels that read_json_gz_table refuses (the json.loads object path).  The VCF
    body is the oracle's rows for the run's population.fam, forced minors (pop_deleterious.txt) and seed."""
    from dna_factory_b200 import pop_factory
    from dna_factory_b200.snp import SnpTable
    snps = real_snps(77 + multibase, 300, multibase)
    path = tmp_path / "snps_in.json.gz"
    with gzip.open(path, "wb") as g:
        for s in snps:
            g.write((json.dumps({"id": s.id, "chromosome": s.chromosome, "position": s.position,
                                 "tuples": {nt: c for nt, c in s.tuples}}) + "\n").encode())
    assert (SnpTable.read_json_gz_table(str(path)) is None) == multibase
    cfg = tmp_path / "groups.yml"
    cfg.write_text("rare:\n  mutation_weights:\n  - 1\n  - 1\n  num_instances: 2\n  population_weight: 1\n"
                   "  max_minor_allele_freq: 0.05\ncommon:\n  mutation_weights:\n  - 0.5\n  - 0.5\n  - 0.5\n"
                   "  num_instances: 2\n  population_weight: 1\n  min_minor_allele_freq: 0.05\n")
    out = tmp_path / "out"
    _fixed_clock(monkeypatch)
    random.seed(5)
    pop_factory.main(["-s", "2100", "-c", "2100", "-z", "6", "--snps_file", str(path), "-p", str(cfg),
                      "--outdir", str(out), "--seed", "4711"])
    blob = (out / "population.vcf.gz").read_bytes()
    vcf, blocks, eof = oracle_mod.bgzf_decompress(blob)
    assert eof and blocks > 3
    lines = vcf.split(b"\n")
    n_head = sum(1 for ln in lines if ln.startswith(b"#"))
    body = b"\n".join(lines[n_head:])
    forced = {}
    for ln in (out / "pop_deleterious.txt").read_text().splitlines():
        f = ln.split("\t")
        forced[int(f[0])] = {int(x[2:]): 1 for x in f[2:] if x}
    fam = []
    for ln in (out / "population.fam").read_text().splitlines():
        f = ln.split("\t")
        ctl = f[5] == "1"
        fam.append(Sample(family_id=int(f[0]), person_id=int(f[1]), father_id=0, mother_id=0, sex=int(f[4]),
                          is_control=ctl, deleterious_snps=None if ctl else forced[int(f[1])]))
    assert len(fam) == 4200 and sum(bool(s.deleterious_snps) for s in fam) > 0
    ordered = sorted(snps, key=lambda s: (s.chromosome, s.position))
    flat = oracle_mod.flatten(fam, ordered)
    assert len(flat["over_row"]) > 0
    plen = np.diff(flat["prefix_off"].astype(np.int64))
    assert plen.max() > (64 if multibase else 40) and (plen[flat["K"] <= 2] >= 39).mean() > 0.5
    want = oracle_mod.rows_from_flat(flat, 4711, 0, n_threads=8)[0].tobytes()
    assert body == want
