"""Case/control allelic association (--assoc): allele counts from k_assoc (dnaf_allele_counts*), the .assoc text from
dnaf_format_assoc, and the planted-SNP report of dna_factory_b200.assoc.

The counts are checked against recounts written from the counting rule (every allele the VCF text prints counts
once) over independent sources: the three-kernel genotype export (dnaf_genotypes), the reference's own golden rows and
the CLI's own population.vcf.gz.  The formatter is checked against a per-line Python rendering and scipy."""
import gzip
import json
import math
import os
import random

import numpy as np
import pytest

from tests.cases import GOLDEN, ROW_CASES, Snp, load_case, synth_case


# ------------------------------------------------------------------------------------------------------------ helpers
def counts_from_genotypes(g, is_control):
    """[rows][4] counts from dnaf_genotypes' [rows][n][2] allele indices (0xFF = allele not printed)."""
    obs = g != 0xFF
    alt = g == 1
    case = ~np.asarray(is_control, bool)[None, :, None]
    return np.stack([(alt & case).sum((1, 2)), (obs & case).sum((1, 2)), (alt & ~case).sum((1, 2)),
                     (obs & ~case).sum((1, 2))], axis=1).astype(np.uint32)


def counts_from_text(text, is_control):
    """The same from VCF rows: '.' prints no allele, a haploid 'a' one, 'a/b' two; allele 1 is ALT."""
    case = ~np.asarray(is_control, bool)
    out = []
    for line in text.split(b"\n")[:-1]:
        cells = line.split(b"\t")[9:] if len(case) else []
        assert len(cells) == len(case)
        row = [0, 0, 0, 0]
        for c, is_case in zip(cells, case):
            alleles = [] if c == b"." else c.split(b"/")
            j = 0 if is_case else 2
            row[j] += sum(a == b"1" for a in alleles)
            row[j + 1] += len(alleles)
        out.append(row)
    return np.asarray(out, np.uint32).reshape(-1, 4)


CHR_CODE = {"X": "23", "Y": "24", "MT": "26"}


def _g(v):
    return "NA" if v is None else "%.4g" % v


def assoc_line_python(label, snp_id, pos, k, ref, alt, cnt):
    """One .assoc body line written from the definitions, independent of the C formatter."""
    a, ca, c, cu = (float(x) for x in cnt)
    b, d = ca - a, cu - c
    f_a = a / ca if ca else None
    f_u = c / cu if cu else None
    den = (a + b) * (c + d) * (a + c) * (b + d)
    x2 = (a + b + c + d) * (a * d - b * c) * (a * d - b * c) / den if den else None
    p = math.erfc(math.sqrt(x2 / 2)) if x2 is not None else None
    odds = a * d / (b * c) if b * c else None
    a1 = chr(alt) if k == 2 else "0"
    return "%4s %12s %10d %4s %8s %8s %4s %12s %12s %12s\n" % (
        CHR_CODE.get(label, label), "rs%d" % snp_id, pos, a1, _g(f_a), _g(f_u), chr(ref), _g(x2), _g(p), _g(odds))


def _table(S, rs, labels=("1", "22", "X", "Y", "MT", "10")):
    from dna_factory_b200.snp import SnpTable
    labels = list(labels)
    k = np.where(rs.rand(S) < 0.2, 1, 2).astype(np.uint8)
    nts = np.zeros((S, 4), np.uint8)
    nts[:, 0] = rs.choice(np.frombuffer(b"ACGT", np.uint8), S)
    nts[:, 1] = np.where(k == 2, rs.choice(np.frombuffer(b"ACGT", np.uint8), S), 0)
    cum = np.full((S, 4), 2.0)
    cum[:, 0] = np.where(k == 1, 1.0, 0.9)
    cum[:, 1] = 1.0
    return SnpTable(rs.randint(1, 10 ** 9, S), rs.randint(0, len(labels), S), labels, rs.randint(0, 250_000_000, S), k,
                    nts, cum)


# ------------------------------------------------------------------------------------------------------------- CPU
def test_format_assoc_matches_per_line_rendering():
    from dna_factory_b200 import assoc
    rs = np.random.RandomState(5)
    S = 400
    t = _table(S, rs)
    ca = rs.randint(0, 3000, S)
    cu = rs.randint(0, 3000, S)
    a = (ca * rs.rand(S)).astype(np.int64)
    c = (cu * rs.rand(S)).astype(np.int64)
    counts = np.stack([a, ca, c, cu], 1).astype(np.uint32)
    counts[0] = [0, 0, 0, 0]            # nothing observed
    counts[1] = [0, 500, 0, 400]        # all-REF row: a + c = 0
    counts[2] = [300, 300, 200, 200]    # all-ALT row: b + d = 0
    counts[3] = [5, 10, 0, 0]           # no controls observed
    counts[4] = [0, 0, 7, 9]            # no cases observed
    counts[5] = [10, 20, 0, 30]         # c = 0: OR is NA, CHISQ is not
    counts[6] = [0, 20, 10, 30]         # a = 0: OR = 0
    counts[7] = [3000, 3000, 0, 3000]   # P underflows far below 1e-300
    counts[8] = [2 ** 31, 2 ** 32 - 1, 2 ** 30, 2 ** 32 - 1]   # large counts stay exact in double
    k1 = np.nonzero(t.n_alleles == 1)[0]
    assert len(k1)
    counts[k1] = [[0, 40, 0, 50]] * len(k1)   # K = 1 rows without forced minors
    counts[k1[0]] = [4, 40, 0, 50]           # ... and one with
    got = assoc.assoc_bytes(t, counts)
    want = "".join(assoc_line_python(t.chrom_labels[t.chrom_idx[r]], int(t.ids[r]), int(t.position[r]), int(t.n_alleles[r]),
                                     int(t.nts[r, 0]), int(t.nts[r, 1]), counts[r]) for r in range(S))
    assert got == assoc.ASSOC_HEADER + want.encode()
    lines = got.decode().splitlines()
    assert lines[0].split() == ["CHR", "SNP", "BP", "A1", "F_A", "F_U", "A2", "CHISQ", "P", "OR"]
    stats = [[f[i] for i in (4, 5, 7, 8, 9)] for f in (ln.split() for ln in lines[1:])]   # F_A F_U CHISQ P OR
    assert stats[0] == ["NA"] * 5
    assert stats[1] == ["0", "0", "NA", "NA", "NA"]
    assert lines[1 + 5].split()[9] == "NA" and lines[1 + 5].split()[7] != "NA"
    assert lines[1 + 7].split()[8] == "0"
    assert {len(ln) for ln in lines[1:]} == {len(lines[0])}     # aligned columns (ids below 10^10)
    assert assoc.assoc_bytes(t.take(np.arange(0)), np.zeros((0, 4), np.uint32)) == assoc.ASSOC_HEADER


def test_chisq_and_p_agree_with_scipy():
    from scipy.stats import chi2_contingency
    from dna_factory_b200 import assoc
    from dna_factory_b200.snp import SnpTable
    tables = [(30, 100, 10, 100), (1, 2000, 0, 2000), (500, 1000, 480, 1000), (7, 9, 2, 11), (900, 1000, 100, 1000)]
    counts = np.asarray(tables, np.uint32)
    n = len(tables)
    t = SnpTable(np.arange(1, n + 1), np.zeros(n, np.int32), ["1"], np.arange(n) * 10, np.full(n, 2, np.uint8),
                 np.tile(np.frombuffer(b"ACGT", np.uint8), (n, 1)), np.tile([0.9, 1.0, 2.0, 2.0], (n, 1)))
    lines = assoc.assoc_bytes(t, counts).decode().splitlines()[1:]
    x2 = assoc.chisq(counts)
    for (a, ca, c, cu), line, x in zip(tables, lines, x2):
        ref = chi2_contingency([[a, ca - a], [c, cu - c]], correction=False)
        stat, p = ref[0], ref[1]
        assert x == pytest.approx(stat, rel=1e-12)
        f = line.split()
        assert float(f[7]) == pytest.approx(stat, rel=1e-3)
        assert float(f[8]) == pytest.approx(p, rel=1e-3, abs=1e-300)
        assert assoc.row_stats(a, ca, c, cu)[3] == pytest.approx(p, rel=1e-9, abs=1e-300)


def test_chr_codes_and_alleles():
    from dna_factory_b200 import assoc
    from dna_factory_b200.snp import SnpTable
    labels = ["1", "X", "Y", "MT", "GL0001"]
    t = SnpTable([11, 12, 13, 14, 15], [0, 1, 2, 3, 4], labels, [5, 6, 7, 8, 9], [2, 2, 2, 1, 2],
                 [[65, 67, 0, 0], [71, 84, 0, 0], [67, 65, 0, 0], [84, 0, 0, 0], [65, 71, 0, 0]],
                 [[0.9, 1.0, 2.0, 2.0]] * 3 + [[1.0, 2.0, 2.0, 2.0], [0.9, 1.0, 2.0, 2.0]])
    rows = [ln.split() for ln in assoc.assoc_bytes(t, np.tile([1, 4, 2, 4], (5, 1))).decode().splitlines()[1:]]
    assert [r[0] for r in rows] == ["1", "23", "24", "26", "GL0001"]
    assert [r[1] for r in rows] == ["rs11", "rs12", "rs13", "rs14", "rs15"]
    assert [(r[3], r[6]) for r in rows] == [("C", "A"), ("T", "G"), ("A", "C"), ("0", "T"), ("G", "A")]


def test_deleterious_report_ranks_and_forced_counts():
    from dna_factory_b200 import assoc
    from dna_factory_b200.pop_factory import DeleteriousGroup
    rs = np.random.RandomState(2)
    S = 50
    t = _table(S, rs, labels=("1", "2"))
    t.n_alleles[:] = 2
    counts = np.tile(np.asarray([10, 100, 10, 100], np.uint32), (S, 1))
    counts[7] = [60, 100, 10, 100]      # strongest
    counts[9] = [30, 100, 10, 100]      # second
    counts[11] = [0, 100, 0, 100]       # NA
    g1 = DeleteriousGroup("g1", 1)
    g1.deleterious = {int(t.ids[7]): 1, int(t.ids[9]): 0.5}
    g2 = DeleteriousGroup.from_json(json.dumps({"name": "g2", "population_weight": 1, "deleterious": {str(t.ids[11]): 1}}))
    orow = np.asarray([7, 7, 7, 9], np.uint64)
    text, summary = assoc.deleterious_report(t, {"g1": g1, "g2": g2}, counts, orow)
    lines = [ln.split("\t") for ln in text.decode().splitlines()]
    assert lines[0] == ["GROUP", "SNP", "CHR", "BP", "WEIGHT", "FORCED", "F_A", "F_U", "CHISQ", "P", "OR", "RANK"]
    rec = {ln[1]: ln for ln in lines[1:]}
    assert rec["rs%d" % t.ids[7]][5] == "3" and rec["rs%d" % t.ids[7]][11] == "1"
    assert rec["rs%d" % t.ids[9]][5] == "1" and rec["rs%d" % t.ids[9]][11] == "2"
    assert rec["rs%d" % t.ids[11]][0] == "g2" and rec["rs%d" % t.ids[11]][5] == "0"     # string key: found, forces nothing
    assert rec["rs%d" % t.ids[11]][8] == "NA" and rec["rs%d" % t.ids[11]][11] == str(S)   # behind the 49 tested rows
    assert summary.startswith("2 of 3 planted deleterious SNPs pass P < 0.05 / 50")


def test_assoc_flag_parses():
    from dna_factory_b200 import pop_factory
    base = ["-s", "3", "-c", "4"]
    assert pop_factory.parse_cmd_args(base + ["--assoc"]).assoc is True
    assert pop_factory.parse_cmd_args(base).assoc is False


def _snps_gz(tmp_path, extra=None):
    with open(os.path.join(GOLDEN, "cli_small", "snps.json"), "rb") as f:
        lines = f.read().splitlines(keepends=True)
    if extra:
        lines.insert(5, extra)
    path = tmp_path / "snps_in.json.gz"
    with gzip.open(path, "wb") as g:
        g.write(b"".join(lines))
    return path


@pytest.mark.parametrize("sizes,match", [(("-s", "5", "-c", "4"), "rs9001"), (("-s", "0", "-c", "4"), "cases and controls"),
                                         (("-s", "5", "-c", "0"), "cases and controls")])
def test_assoc_refusals_before_the_vcf(tmp_path, sizes, match):
    """A multi-allelic table, a population without cases and one without controls fail before any output."""
    from dna_factory_b200 import pop_factory
    extra = b'{"id": 9001, "chromosome": "1", "position": 7000000, "tuples": {"A": 0.5, "C": 0.8, "G": 1.0}}\n'
    snps_gz = _snps_gz(tmp_path, extra if match == "rs9001" else None)
    out = tmp_path / "out"
    random.seed(1)
    with pytest.raises(ValueError, match=match):
        pop_factory.main(list(sizes) + ["--snps_file", str(snps_gz), "-p",
                                        os.path.join(GOLDEN, "cli_small", "deleterious_config.yml"), "--outdir", str(out),
                                        "--seed", "7", "--assoc"])
    assert not (out / "population.vcf.gz").exists()
    assert not (out / "population.assoc").exists()


# ------------------------------------------------------------------------------------------------------------- GPU
def _engine(case, chunk=None, row_base=None):
    from dna_factory_b200 import _native, host
    eng = _native.Engine(0)
    host.configure(eng, case.samples, case.snps)
    eng.set_row_base(case.row_begin if row_base is None else row_base)
    if chunk:
        eng.set_chunk_bytes(chunk)
    return eng


def _ctl(case):
    return np.asarray([bool(s.is_control) for s in case.samples], bool)


def _runs(ks):
    """Maximal runs [a, b) of rows with at most 2 alleles."""
    runs, a = [], None
    for r, k in enumerate(list(ks) + [9]):
        if k <= 2 and a is None:
            a = r
        elif k > 2 and a is not None:
            runs.append((a, r))
            a = None
    return runs


def _dense_case(n, seed, n_snps=24):
    """All four classes (one row of each is added), a K = 1 row, and forced minors on most cases of every X, Y and MT row (male haploid cells,
    female Y cells) and of the rarest rows."""
    case = synth_case(n, n_snps, seed=seed, chroms=["1", "2", "X", "Y", "MT", "22"], n_del=6)
    case.snps.append(Snp(id=100_001, chromosome="7", position=5, tuples=[("G", 1.0)]))
    case.snps.append(Snp(id=100_002, chromosome="Y", position=6, tuples=[("A", 0.995), ("C", 1.0)]))
    case.snps.append(Snp(id=100_003, chromosome="X", position=7, tuples=[("C", 0.8), ("T", 1.0)]))
    case.snps.append(Snp(id=100_004, chromosome="MT", position=8, tuples=[("T", 0.9), ("G", 1.0)]))
    case.snps.sort(key=lambda x: (x.chromosome, x.position))
    rare = sorted(case.snps, key=lambda s: -s.tuples[0][1])[:3]
    hap = [s for s in case.snps if s.chromosome in ("X", "Y", "MT")]
    for i, smp in enumerate(case.samples):
        if not smp.is_control and i % 3 != 0:
            for s in rare + hap + [case.snps[0]]:
                smp.deleterious_snps[s.id] = 0.5
    return case


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 15, 16, 17, 4095, 4096, 4097, 20000, 100003])
def test_counts_match_the_genotype_export(n):
    """k_assoc against counts taken from the three-kernel export (k_sample -> k_overrides -> k_export_genotypes), across
    the 16-sample word and the 4096-sample CTA tile, with a row counter offset and a chunk that makes many passes."""
    case = _dense_case(n, seed=n)
    S = len(case.snps)
    assert {s.chromosome for s in case.snps} >= {"X", "Y", "MT", "1"}
    eng = _engine(case, chunk=4096, row_base=1000 + n)
    want = counts_from_genotypes(eng.genotypes(0, S, case.seed), _ctl(case))
    got, st = eng.allele_counts_stats(0, S, case.seed)
    assert np.array_equal(got, want)
    assert st["rows"] == S and st["calls"] == S * n and st["kernel_launches"] == -(-S // 256)
    assert st["ms_sample"] > 0 and st["ms_total"] >= st["ms_sample"]
    assert (st["bgzf_bytes"], st["bgzf_blocks"], st["text_bytes"]) == (0, 0, 0)
    eng.close()


@pytest.mark.gpu
def test_counts_over_many_passes():
    """700 rows of all four classes at N = 4097 (two CTAs per row), 256 rows per pass: three passes."""
    case = synth_case(4097, 700, seed=44, chroms=["1", "X", "Y", "MT", "5"], n_del=40)
    S = len(case.snps)
    eng = _engine(case, chunk=4096, row_base=3 * 2 ** 32 + 17)
    want = counts_from_genotypes(eng.genotypes(0, S, case.seed), _ctl(case))
    got, st = eng.allele_counts_stats(0, S, case.seed)
    assert st["kernel_launches"] == 3
    assert np.array_equal(got, want)
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ROW_CASES)
def test_counts_match_the_reference_golden_rows(name):
    """X, Y and MT for both sexes, forced minors, K = 1 rows, a row counter above 2^32, N = 0; K > 2 rows skipped."""
    case = load_case(name)
    lines = case.text.split(b"\n")[:-1]
    eng = _engine(case)
    runs = _runs([len(s.tuples) for s in case.snps])
    assert runs
    for a, b in runs:
        got = eng.allele_counts(a, b, case.seed)
        want = counts_from_text(b"".join(ln + b"\n" for ln in lines[a:b]), _ctl(case))
        assert np.array_equal(got, want), (name, a, b)
    eng.close()


@pytest.mark.gpu
def test_ranges_and_repeats():
    case = _dense_case(2500, seed=11, n_snps=600)
    S = len(case.snps)
    eng = _engine(case, chunk=8192)
    whole = eng.allele_counts(0, S, case.seed)
    assert np.array_equal(eng.allele_counts(0, S, case.seed), whole)
    cut = [0, 1, 7, 7, S // 2, S - 1, S]
    assert np.array_equal(np.concatenate([eng.allele_counts(a, b, case.seed) for a, b in zip(cut, cut[1:])]), whole)
    _, st = eng.allele_counts_stats(0, S, case.seed)
    dev = eng.allele_counts_device(0, S, case.seed)
    assert {k: dev[k] for k in ("rows", "calls", "kernel_launches")} == {k: st[k] for k in ("rows", "calls", "kernel_launches")}
    assert whole[:, 0].sum() > 0 and whole[:, 2].sum() > 0
    eng.close()


@pytest.mark.gpu
def test_refuses_multiallelic_rows_before_any_work():
    import ctypes
    from dna_factory_b200 import _native
    case = synth_case(40, 20, seed=5, exotic=True)
    eng = _engine(case)
    k = [len(s.tuples) for s in case.snps]
    bad = next(r for r, kr in enumerate(k) if kr > 2)
    out = np.full((20, 4), 0xABABABAB, np.uint32)
    st = _native.Stats()
    rc = eng._lib.dnaf_allele_counts(eng._h, 0, 20, case.seed, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                     ctypes.byref(st))
    assert rc == _native.E_INPUT
    assert ("row %d " % bad) in eng._lib.dnaf_last_error(eng._h).decode()
    assert (out == 0xABABABAB).all() and st.kernel_launches == 0
    with pytest.raises(_native.DnafError) as e:
        eng.allele_counts_device(0, 20, case.seed)
    assert e.value.code == _native.E_INPUT
    a, b = _runs(k)[0]
    assert eng.allele_counts(a, b, case.seed).shape == (b - a, 4)     # the context is still usable
    eng.close()


def _fixed_clock(monkeypatch):
    from dna_factory_b200 import pop_factory

    class FixedDatetime(pop_factory.datetime):
        @classmethod
        def now(cls, tz=None):
            return cls(2026, 1, 1, 12, 34, 56)

    monkeypatch.setattr(pop_factory, "datetime", FixedDatetime)


def _cli_small(monkeypatch, out, extra):
    from dna_factory_b200 import pop_factory
    gold = os.path.join(GOLDEN, "cli_small")
    meta = json.load(open(os.path.join(gold, "meta.json")))
    _fixed_clock(monkeypatch)
    random.seed(meta["python_random_seed"])
    pop_factory.main(meta["args"] + ["-p", os.path.join(gold, "deleterious_config.yml"), "--outdir", str(out),
                                     "--seed", str(meta["philox_seed"]), "--assoc"] + extra)


def _vcf_recount(out):
    vcf = gzip.decompress((out / "population.vcf.gz").read_bytes())
    body = b"".join(ln + b"\n" for ln in vcf.split(b"\n")[:-1] if not ln.startswith(b"#"))
    ctl = [ln.split("\t")[5] == "1" for ln in (out / "population.fam").read_text().splitlines()]
    return counts_from_text(body, ctl)


@pytest.mark.gpu
def test_cli_assoc_matches_its_own_vcf(tmp_path, monkeypatch):
    """--assoc on the pinned reference CLI run: population.assoc is the text of the counts recounted from the run's own
    population.vcf.gz, and --gpus 2 writes the same population.assoc and deleterious_assoc.txt."""
    from dna_factory_b200 import assoc
    from dna_factory_b200.snp import SnpTable
    out = tmp_path / "g1"
    _cli_small(monkeypatch, out, [])
    table = SnpTable.read_json_gz_table(str(out / "snps.json.gz"))
    want = _vcf_recount(out)
    assert len(want) == len(table) == 400
    assert (out / "population.assoc").read_bytes() == assoc.assoc_bytes(table, want)
    report = (out / "deleterious_assoc.txt").read_text().splitlines()
    assert len(report) == 1 + sum(len(json.loads(ln)["deleterious"]) for ln in open(out / "deleterious.json"))
    _cli_small(monkeypatch, tmp_path / "g2", ["--gpus", "2"])
    for name in ("population.assoc", "deleterious_assoc.txt"):
        assert (tmp_path / "g2" / name).read_bytes() == (out / name).read_bytes(), name


@pytest.mark.gpu
def test_cli_planted_snps_come_out_on_top(tmp_path, monkeypatch, capsys):
    """One group of three planted SNPs, one forced per case: 2000 + 2000 samples find every one of them in the top 3."""
    from dna_factory_b200 import pop_factory
    cfg = tmp_path / "one_group.yml"
    cfg.write_text("planted:\n  mutation_weights:\n  - 1\n  - 1\n  - 1\n  num_instances: 1\n  population_weight: 1\n"
                   "  max_minor_allele_freq: 0.1\n")
    out = tmp_path / "out"
    _fixed_clock(monkeypatch)
    random.seed(99)
    pop_factory.main(["-s", "2000", "-c", "2000", "-x", "3000", "-f", "0.01", "-p", str(cfg), "--outdir", str(out),
                      "--seed", "2024", "--assoc"])
    assert "3 of 3 planted deleterious SNPs pass" in capsys.readouterr().out
    lines = [ln.split("\t") for ln in (out / "deleterious_assoc.txt").read_text().splitlines()]
    col = {name: i for i, name in enumerate(lines[0])}
    assert len(lines) == 4
    for ln in lines[1:]:
        assert ln[col["GROUP"]] == "planted-0"
        assert int(ln[col["FORCED"]]) > 0
        assert int(ln[col["RANK"]]) <= 3


@pytest.mark.gpu
def test_cli_replay_reports_forced_zero(tmp_path, monkeypatch):
    """A --deleterious_file replay keeps string keys, which force nothing (SURVEY R8): every line shows FORCED 0."""
    from dna_factory_b200 import pop_factory
    gold = os.path.join(GOLDEN, "cli_small")
    out = tmp_path / "out"
    _fixed_clock(monkeypatch)
    random.seed(3)
    pop_factory.main(["-s", "40", "-c", "40", "--snps_file", str(_snps_gz(tmp_path)), "--deleterious_file",
                      os.path.join(gold, "deleterious.json"), "--outdir", str(out), "--seed", "5", "--assoc"])
    lines = [ln.split("\t") for ln in (out / "deleterious_assoc.txt").read_text().splitlines()]
    n_planted = sum(len(json.loads(ln)["deleterious"]) for ln in open(os.path.join(gold, "deleterious.json")))
    assert len(lines) == 1 + n_planted
    assert all(ln[5] == "0" for ln in lines[1:])
    assert all(ln[3] != "NA" for ln in lines[1:])      # every key found its row through int(key)
