"""Fisher's exact tests (--fisher): log10 P from k_fisher (dnaf_fisher_exact, dnaf_genotype_tests*), the
.assoc.fisher / Fisher .model text from dnaf_format_assoc_fisher / dnaf_format_model_fisher, and the planted-SNP report
of dna_factory_b200.fisher.

The exact test is checked against full enumerations written from the definition (log-gamma in double for small tables,
40-digit mpmath for large ones) and against scipy.stats.fisher_exact on 2x2 tables; the count path against
dnaf_genotype_counts and dnaf_fisher_exact; the formatters against a per-line Python rendering; the CLI against the
text of the genotypes recounted from its own population.vcf.gz."""
import gzip
import json
import math
import os
import random

import numpy as np
import pytest

from tests.cases import GOLDEN, synth_case
from tests.test_assoc import _dense_case, _fixed_clock, _runs, _snps_gz, _table
from tests.test_model import CHR_CODE, _cli_small, _geno_engine, _random_counts, _trend_variance_form, geno_from_text

TIE = 1e-7   # the relative tie tolerance of dnaf_fisher_exact (kHweTie)


# ------------------------------------------------------------------------------------------------------------ helpers
def _margins(x, y):
    x, y = np.asarray(x, np.int64), np.asarray(y, np.int64)
    c = x + y
    return x, c, int(x.sum()), int(c.sum())


def _all_tables(c, R):
    """Every case row (x1, x2, x3) with column sums c and R cases, as int64[k, 3]."""
    x1 = np.arange(0, min(c[0], R) + 1)
    x2 = np.arange(0, min(c[1], R) + 1)
    a, b = np.meshgrid(x1, x2, indexing="ij")
    a, b = a.ravel(), b.ravel()
    x3 = R - a - b
    ok = (x3 >= 0) & (x3 <= c[2])
    return np.stack([a[ok], b[ok], x3[ok]], 1)


def _log_terms(tabs, c):
    from scipy.special import gammaln
    return (gammaln(c + 1.0) - gammaln(tabs + 1.0) - gammaln(c - tabs + 1.0)).sum(1)


def fisher_ref(x, y):
    """log10 of the two-sided Fisher P by full enumeration of the tables with the same margins: log P(table) from
    log-gamma, P = the sum of every P(table) <= P(observed) (1 + TIE) over the sum of all.  NaN when a row margin is 0
    or fewer than two columns are non-empty."""
    x, c, R, N = _margins(list(x) + [0] * (3 - len(x)), list(y) + [0] * (3 - len(y)))
    if R == 0 or R == N or (c > 0).sum() < 2:
        return math.nan
    tabs = _all_tables(c, R)
    lp = _log_terms(tabs, c)
    top = lp.max()
    p = np.exp(lp - top)
    obs = float(np.exp(_log_terms(x[None, :], c)[0] - top))
    return math.log10(min(1.0, p[p <= obs * (1 + TIE)].sum() / p.sum()))


def fisher_ref_exact(x, y, prune=1800.0):
    """The same in 40-digit mpmath, over the tables within exp(-prune) of the largest one and within exp(-120) of the
    observed one (the rest is below 10^-52 of the sums they would join): log10 P to far better than 1e-10, including P
    far below the double range."""
    import mpmath
    mpmath.mp.dps = 40
    x, c, R, N = _margins(list(x) + [0] * (3 - len(x)), list(y) + [0] * (3 - len(y)))
    tabs = _all_tables(c, R)
    lp = _log_terms(tabs, c)
    obs_lp = float(_log_terms(x[None, :], c)[0])
    keep = (lp - lp.max() > -prune) | (lp - obs_lp > -120.0)   # and the tail next to the observed table
    tabs = tabs[keep]

    def lt(t):
        return sum(mpmath.loggamma(int(cj) + 1) - mpmath.loggamma(int(tj) + 1) - mpmath.loggamma(int(cj - tj) + 1)
                   for tj, cj in zip(t, c))
    terms = [lt(t) for t in tabs.tolist()]
    obs = lt(x.tolist())
    tot = mpmath.fsum(mpmath.exp(v - obs) for v in terms)
    tail = mpmath.fsum(mpmath.exp(v - obs) for v in terms if mpmath.exp(v - obs) <= 1 + TIE)
    return float(mpmath.log10(tail / tot))


def _p(l):
    return "NA" if math.isnan(l) else "%.4g" % (10.0 ** l)


def _allele_tables(c):
    """[rows][4][6] Fisher tables (GENO, ALLELIC, DOM, REC) of [rows][10] counts, built in numpy."""
    c = np.asarray(c, np.int64).reshape(-1, 10)
    a11, a12, a22 = c[:, 2], c[:, 1], c[:, 0] - c[:, 1] - c[:, 2]
    u11, u12, u22 = c[:, 7], c[:, 6], c[:, 5] - c[:, 6] - c[:, 7]
    alt_a, alt_u = 2 * a11 + a12 + c[:, 4], 2 * u11 + u12 + c[:, 9]
    ref_a, ref_u = 2 * c[:, 0] + c[:, 3] - alt_a, 2 * c[:, 5] + c[:, 8] - alt_u
    z = np.zeros_like(a11)
    t = [(a11, a12, a22, u11, u12, u22), (alt_a, ref_a, z, alt_u, ref_u, z), (a11 + a12, a22, z, u11 + u12, u22, z),
         (a11, a12 + a22, z, u11, u12 + u22, z)]
    return np.stack([np.stack(q, 1) for q in t], 1).astype(np.uint32)


def model_fisher_lines_python(label, snp_id, k, ref, alt, c, l):
    """The five Fisher .model lines of one row, from the definitions."""
    a11, a12, a22 = c[2], c[1], c[0] - c[1] - c[2]
    u11, u12, u22 = c[7], c[6], c[5] - c[6] - c[7]
    alt_a, alt_u = 2 * a11 + a12 + c[4], 2 * u11 + u12 + c[9]
    ref_a, ref_u = 2 * c[0] + c[3] - alt_a, 2 * c[5] + c[8] - alt_u
    trend = _trend_variance_form([a11, a12, a22], [u11, u12, u22])
    rows = [("GENO", "%d/%d/%d" % (a11, a12, a22), "%d/%d/%d" % (u11, u12, u22), _p(l[0])),
            ("TREND", "%d/%d/%d" % (a11, a12, a22), "%d/%d/%d" % (u11, u12, u22),
             "NA" if trend is None else "%.4g" % math.erfc(math.sqrt(trend / 2))),
            ("ALLELIC", "%d/%d" % (alt_a, ref_a), "%d/%d" % (alt_u, ref_u), _p(l[1])),
            ("DOM", "%d/%d" % (a11 + a12, a22), "%d/%d" % (u11 + u12, u22), _p(l[2])),
            ("REC", "%d/%d" % (a11, a12 + a22), "%d/%d" % (u11, u12 + u22), _p(l[3]))]
    a1 = chr(alt) if k == 2 else "0"
    return "".join("%4s %12s %4s %4s %8s %14s %14s %12s\n" % (CHR_CODE.get(label, label), "rs%d" % snp_id, a1, chr(ref), test,
                                                            aff, unaff, p) for test, aff, unaff, p in rows)


def assoc_fisher_line_python(label, snp_id, pos, k, ref, alt, c, l):
    a11, a12, u11, u12 = c[2], c[1], c[7], c[6]
    a, ca = 2 * a11 + a12 + c[4], 2 * c[0] + c[3]
    cc, cu = 2 * u11 + u12 + c[9], 2 * c[5] + c[8]
    b, d = ca - a, cu - cc
    g = lambda v: "NA" if v is None else "%.4g" % v    # noqa: E731
    return "%4s %12s %10d %4s %8s %8s %4s %12s %12s\n" % (
        CHR_CODE.get(label, label), "rs%d" % snp_id, pos, chr(alt) if k == 2 else "0", g(a / ca if ca else None),
        g(cc / cu if cu else None), chr(ref), _p(l[1]), g(a * d / (b * cc) if b * cc else None))


# ------------------------------------------------------------------------------------------------------------- CPU
def test_fisher_reference_sanity():
    """The test's own references on tables worked by hand: the tea-tasting table 3/1 vs 1/3 has P = 34/70; a table
    with a single possible arrangement has P = 1; scipy agrees on a plain 2x2 table; the mpmath form agrees."""
    assert 10 ** fisher_ref([3, 1], [1, 3]) == pytest.approx(34 / 70, rel=1e-13)
    assert fisher_ref([2, 0], [0, 0]) != fisher_ref([2, 0], [0, 0])       # no controls: NaN
    assert fisher_ref([2, 0, 0], [3, 0, 0]) != fisher_ref([2, 0, 0], [3, 0, 0])   # one column: NaN
    assert fisher_ref([0, 2, 0], [1, 0, 0]) == pytest.approx(math.log10(1 / 3), rel=1e-13)
    from scipy.stats import fisher_exact
    assert 10 ** fisher_ref([12, 5], [3, 20]) == pytest.approx(fisher_exact([[12, 5], [3, 20]])[1], rel=1e-12)
    assert fisher_ref_exact([12, 5, 7], [3, 20, 4]) == pytest.approx(fisher_ref([12, 5, 7], [3, 20, 4]), abs=1e-12)


def test_format_assoc_and_model_fisher_match_per_line_rendering():
    from dna_factory_b200 import fisher
    rs = np.random.RandomState(11)
    S = 300
    t = _table(S, rs)
    counts = _random_counts(S, rs)
    counts[0] = 0                                          # nothing observed
    counts[1] = [40, 0, 0, 0, 0, 30, 0, 0, 0, 0]           # monomorphic REF
    counts[3] = [0, 0, 0, 0, 0, 50, 10, 10, 0, 0]          # no cases
    counts[6] = [0, 0, 0, 40, 12, 0, 0, 0, 35, 3]          # haploid only (Y / MT rows): ALLELIC only
    counts[7] = [3000, 0, 3000, 0, 0, 3000, 3000, 0, 0, 0]  # P far below the double range
    l = -rs.rand(S, 4) * 12
    l[0] = np.nan
    l[1] = np.nan
    l[3] = np.nan
    l[6] = [np.nan, -3.5, np.nan, np.nan]
    l[7] = [-2500.0, -1500.25, -400.0, -320.0]
    l[8] = [0.0, -0.0, -1e-17, -7.0]
    want_m, want_a = [], []
    for r in range(S):
        args = (t.chrom_labels[t.chrom_idx[r]], int(t.ids[r]), int(t.n_alleles[r]), int(t.nts[r, 0]), int(t.nts[r, 1]))
        cr = [int(v) for v in counts[r]]
        want_m.append(model_fisher_lines_python(*args, cr, l[r]))
        want_a.append(assoc_fisher_line_python(args[0], args[1], int(t.position[r]), *args[2:], cr, l[r]))
    got_m = fisher.model_fisher_bytes(t, counts, l)
    got_a = fisher.assoc_fisher_bytes(t, counts, l)
    assert got_m == fisher.MODEL_FISHER_HEADER + "".join(want_m).encode()
    assert got_a == fisher.ASSOC_FISHER_HEADER + "".join(want_a).encode()
    m = [ln.split() for ln in got_m.decode().splitlines()]
    assert m[0] == ["CHR", "SNP", "A1", "A2", "TEST", "AFF", "UNAFF", "P"]
    assert [ln[4] for ln in m[1:6]] == ["GENO", "TREND", "ALLELIC", "DOM", "REC"]
    row7 = {ln[4]: ln[7] for ln in m[1 + 5 * 7:1 + 5 * 8]}
    assert row7 == {"GENO": "0", "TREND": "0", "ALLELIC": "0", "DOM": "0", "REC": "1e-320"}
    row6 = {ln[4]: ln[7] for ln in m[1 + 5 * 6:1 + 5 * 7]}
    assert row6["ALLELIC"] == "0.0003162" and row6["GENO"] == row6["DOM"] == row6["REC"] == "NA"
    a = [ln.split() for ln in got_a.decode().splitlines()]
    assert a[0] == ["CHR", "SNP", "BP", "A1", "F_A", "F_U", "A2", "P", "OR"]
    assert a[1 + 8][7] == "1" and a[1 + 7][7] == "0" and [a[1][i] for i in (4, 5, 7, 8)] == ["NA"] * 4
    assert {ln[0] for ln in a[1:]} == {CHR_CODE.get(x, x) for x in t.chrom_labels}
    empty = t.take(np.arange(0))
    assert fisher.model_fisher_bytes(empty, np.zeros((0, 10), np.uint32), np.zeros((0, 4))) == fisher.MODEL_FISHER_HEADER
    assert fisher.assoc_fisher_bytes(empty, np.zeros((0, 10), np.uint32), np.zeros((0, 4))) == fisher.ASSOC_FISHER_HEADER


def test_deleterious_fisher_report_text():
    from dna_factory_b200 import fisher
    from dna_factory_b200.pop_factory import DeleteriousGroup
    rs = np.random.RandomState(2)
    S = 40
    t = _table(S, rs, labels=("1", "2"))
    t.n_alleles[:] = 2
    counts = np.tile(np.asarray([400, 160, 20, 0, 0, 400, 160, 20, 0, 0], np.uint32), (S, 1))
    counts[5] = [400, 150, 120, 0, 0, 400, 160, 20, 0, 0]   # recessive signal, every cell >= 5
    counts[6] = [400, 100, 30, 0, 0, 400, 160, 3, 0, 0]     # REC signal with 3 ALT/ALT controls: no chi-square REC
    counts[7] = [400, 200, 30, 0, 0, 400, 160, 20, 0, 0]    # weaker
    l = np.full((S, 4), -0.2)
    l[5] = [-40.0, -2000.5, -30.0, -1500.0]
    l[6] = [-9.0, -8.0, -1.0, -7.25]
    l[7] = [-1.0, -2.0, -0.5, np.nan]
    g1 = DeleteriousGroup("g1", 1)
    g1.deleterious = {int(t.ids[5]): 1, int(t.ids[6]): 0.5, 999: 0.2}        # 999: not in the table
    g2 = DeleteriousGroup.from_json(json.dumps({"name": "g2", "population_weight": 1, "deleterious": {str(t.ids[7]): 1}}))
    orow = np.asarray([5, 5, 6], np.uint64)
    text, summary = fisher.deleterious_fisher_report(t, {"g1": g1, "g2": g2}, counts, l, orow)
    lines = [ln.split("\t") for ln in text.decode().splitlines()]
    assert tuple(lines[0]) == fisher.REPORT_COLUMNS
    col = {k: i for i, k in enumerate(lines[0])}
    rec = {ln[1]: ln for ln in lines[1:]}
    r5, r6, r7 = rec["rs%d" % t.ids[5]], rec["rs%d" % t.ids[6]], rec["rs%d" % t.ids[7]]
    assert r5[col["FORCED"]] == "2" and r6[col["FORCED"]] == "1" and r7[col["FORCED"]] == "0"
    assert (r5[col["AFF"]], r5[col["UNAFF"]]) == ("120/150/130", "20/160/220")
    assert (r5[col["P_ALLELIC"]], r5[col["P_GENO"]], r5[col["P_DOM"]], r5[col["P_REC"]]) == ("0", "1e-40", "1e-30", "0")
    assert (r5[col["LOG10P_ALLELIC"]], r5[col["LOG10P_REC"]]) == ("-2000.5", "-1500")
    assert (r5[col["RANK_REC"]], r5[col["RANK_ALLELIC"]]) == ("1", "1")
    assert (r6[col["RANK_REC"]], r6[col["RANK_ALLELIC"]]) == ("2", "2")
    assert r7[col["P_REC"]] == "NA" and r7[col["LOG10P_REC"]] == "NA" and r7[col["RANK_REC"]] == str(S)
    assert rec["rs999"][2:] == ["NA", "NA", "0.2", "0"] + ["NA"] * 10
    assert len(lines) == 5
    assert summary == ("2 of 4 planted deleterious SNPs pass P < 0.05 / 40 = 0.00125 under Fisher REC and 2 under "
                       "Fisher ALLELIC; 1 of the REC passes have no chi-square REC test (a genotype cell below 5)")


def test_fisher_flag_parses():
    from dna_factory_b200 import pop_factory
    assert pop_factory.parse_cmd_args(["-s", "3", "-c", "4", "--fisher"]).fisher is True
    assert pop_factory.parse_cmd_args(["-s", "3", "-c", "4"]).fisher is False


@pytest.mark.parametrize("sizes,multi,match", [
    (("-s", "5", "-c", "4"), True, "--fisher: SNP rs9001"),
    (("-s", "0", "-c", "4"), False, "--fisher needs cases and controls"),
    (("-s", "5", "-c", "0"), False, "--fisher needs cases and controls")])
def test_fisher_refusals_before_the_vcf(tmp_path, sizes, multi, match):
    """A multi-allelic table and a population without cases or controls fail before any output."""
    from dna_factory_b200 import pop_factory
    extra = b'{"id": 9001, "chromosome": "1", "position": 7000000, "tuples": {"A": 0.5, "C": 0.8, "G": 1.0}}\n'
    snps_gz = _snps_gz(tmp_path, extra if multi else None)
    out = tmp_path / "out"
    random.seed(1)
    with pytest.raises(ValueError, match=match):
        pop_factory.main(list(sizes) + ["--snps_file", str(snps_gz), "-p",
                                        os.path.join(GOLDEN, "cli_small", "deleterious_config.yml"), "--outdir", str(out),
                                        "--seed", "7", "--fisher"])
    for name in ("population.vcf.gz", "population.assoc.fisher", "population.model.fisher"):
        assert not (out / name).exists()


# ------------------------------------------------------------------------------------------------------------- GPU
def _fisher(tables):
    from dna_factory_b200 import _native
    with _native.Engine(0) as eng:
        return eng.fisher_exact(np.asarray(tables, np.uint32).reshape(-1, 6))


def _by_margins(tables):
    """The reference log10 P of every table, one enumeration per margin set (every table of a set at once)."""
    t = np.asarray(tables, np.int64)
    x, c = t[:, :3], t[:, :3] + t[:, 3:]
    R, N = x.sum(1), c.sum(1)
    lp_obs = _log_terms(x, c)
    want = np.full(len(t), np.nan)
    keys, inv = np.unique(np.concatenate([c, R[:, None]], 1), axis=0, return_inverse=True)
    inv = inv.ravel()
    order = np.argsort(inv, kind="stable")
    bounds = np.searchsorted(inv[order], np.arange(len(keys) + 1))
    for g, key in enumerate(keys):
        cg, Rg = key[:3], int(key[3])
        if Rg == 0 or Rg == int(cg.sum()) or (cg > 0).sum() < 2:
            continue
        idx = order[bounds[g]:bounds[g + 1]]
        lp = _log_terms(_all_tables(cg, Rg), cg)
        top = lp.max()
        p = np.sort(np.exp(lp - top))
        cum = np.cumsum(p)
        k = np.searchsorted(p, np.exp(lp_obs[idx] - top) * (1 + TIE), side="right")
        want[idx] = np.log10(np.minimum(1.0, cum[k - 1] / cum[-1]))
    return want


@pytest.mark.gpu
def test_fisher_exact_every_small_table():
    """Every 2x3 table up to N = 24 and every 2x2 table up to N = 60, ties included, against the log-gamma enumeration:
    relative 1e-12 in P; NaN exactly where a margin is 0 or fewer than two columns are non-empty."""
    t3 = [(a, b, c, d, e, f) for n in range(25) for a in range(n + 1) for b in range(n + 1 - a) for c in range(n + 1 - a - b)
          for d in range(n + 1 - a - b - c) for e in range(n + 1 - a - b - c - d) for f in [n - a - b - c - d - e]]
    t2 = [(a, b, 0, c, n - a - b - c, 0) for n in range(61) for a in range(n + 1) for b in range(n + 1 - a)
          for c in range(n + 1 - a - b)]
    tables = np.asarray(t3 + t2, np.int64)
    got = _fisher(tables)
    want = _by_margins(tables)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    err = np.abs(got[ok] - want[ok])
    assert err.max() <= 1e-12 / math.log(10) + 1e-15, tables[ok][np.argmax(err)]
    assert (got[ok] <= 0).all() and (got[ok] == 0).sum() > 1000       # P = 1 (ties at the mode) prints as 1


@pytest.mark.gpu
def test_fisher_exact_empty_column_is_the_2x2_test_and_nan_cases():
    rs = np.random.RandomState(4)
    t = rs.randint(0, 3000, (500, 4))
    t[:20] = rs.randint(0, 4, (20, 4))
    z = np.zeros(len(t), np.int64)
    a, b, c, d = t.T
    forms = [np.stack(q, 1) for q in ((a, b, z, c, d, z), (a, z, b, c, z, d), (z, a, b, z, c, d))]
    got = [_fisher(f) for f in forms]
    assert np.array_equal(got[0], got[1], equal_nan=True) and np.array_equal(got[0], got[2], equal_nan=True)
    nan_cases = [(0, 0, 0, 5, 6, 7), (5, 6, 7, 0, 0, 0), (3, 0, 0, 9, 0, 0), (0, 0, 4, 0, 0, 2), (0, 0, 0, 0, 0, 0)]
    assert np.isnan(_fisher(nan_cases)).all()
    assert len(_fisher(np.zeros((0, 6)))) == 0


@pytest.mark.gpu
def test_fisher_exact_2x2_agrees_with_scipy():
    """2x2 tables up to N = 10^4 against scipy.stats.fisher_exact, on the tables where no other table's probability
    lies between the two tie tolerances (scipy: 1e-14, here 1e-7), so the two definitions agree."""
    from scipy.stats import fisher_exact
    rs = np.random.RandomState(9)
    tabs = []
    for n in (10, 80, 500, 3000, 10000):
        for _ in range(40):
            R = rs.randint(1, n)
            c = rs.randint(1, n)
            lo, hi = max(0, R + c - n), min(R, c)
            x = rs.randint(lo, hi + 1)
            tabs.append((x, R - x, 0, c - x, n - R - c + x, 0))
    got = _fisher(tabs)
    checked = 0
    for t, g in zip(tabs, got):
        x, c, R, N = _margins(t[:3], t[3:])
        alls = _all_tables(c, R)
        lp = _log_terms(alls, c)
        obs = float(_log_terms(x[None, :], c)[0])
        d = lp - obs
        if ((d > 1e-14) & (d <= 2e-7)).any() or np.isnan(g):
            continue
        want = fisher_exact([[t[0], t[1]], [t[3], t[4]]])[1]
        if want < 1e-290:
            continue
        assert 10 ** g == pytest.approx(want, rel=1e-9), t
        checked += 1
    assert checked > 150


@pytest.mark.gpu
def test_fisher_exact_large_and_rare_tables_against_mpmath():
    """Random tables up to N = 10^5, the rare-variant shapes the generator plants (a column near 0) and tables with
    P < 1e-1000, against a 40-digit enumeration: |d log10 P| <= 1e-10."""
    rs = np.random.RandomState(23)
    tabs = []
    for n in (1000, 20000, 100000):                        # 2x2: allele tables
        for _ in range(4):
            R = rs.randint(n // 4, 3 * n // 4)
            f = rs.uniform(0.001, 0.5)
            x = rs.binomial(R, f)
            y = rs.binomial(n - R, f)
            tabs.append((x, R - x, 0, y, n - R - y, 0))
    tabs += [(400, 3600, 0, 5, 3995, 0),                   # planted REC shape: P ~ 1e-110
             (1500, 2500, 0, 3, 3997, 0),                  # P far below 1e-300
             (9000, 1000, 0, 10, 99990 - 9000, 0),         # P < 1e-1000
             (1, 49999, 0, 0, 50000, 0)]
    tabs += [(300, 700, 1000, 3, 720, 1277),               # 2x3 planted GENO shape, 2000 + 2000
             (12, 330, 658, 8, 310, 682),                  # 2x3 rare ALT/ALT column, near the null
             (1, 20, 979, 0, 15, 985),
             (40, 380, 580, 45, 360, 595),                 # common SNP, 1000 + 1000
             (1200, 0, 0, 0, 1, 1199)]                     # P far below the double range
    got = _fisher(tabs)
    for t, g in zip(tabs, got):
        want = fisher_ref_exact(t[:3], t[3:])
        assert abs(g - want) <= 1e-10, (t, g, want)
    assert got[14] < -1000 and got[-1] < -300


@pytest.mark.gpu
@pytest.mark.parametrize("n", [17, 4097, 20000])
def test_genotype_tests_match_counts_and_the_exact_kernel(n):
    """genotype_tests: counts and HWE P bitwise equal to genotype_counts over many passes and ranges; its Fisher output
    bitwise equal to dnaf_fisher_exact over tables built in numpy from those counts; the device-only call runs the same
    launches; Y and MT rows have only ALLELIC."""
    case = _dense_case(n, seed=n) if n != 4097 else synth_case(4097, 700, seed=44, chroms=["1", "X", "Y", "MT", "5"], n_del=40)
    S = len(case.snps)
    eng = _geno_engine(case, chunk=4096, row_base=77 + n)
    counts, hwe_p, st0 = eng.genotype_counts_stats(0, S, case.seed)
    got, p, l, st = eng.genotype_tests_stats(0, S, case.seed)
    assert np.array_equal(got, counts) and np.array_equal(p, hwe_p, equal_nan=True)
    assert st0["kernel_launches"] == 2 * -(-S // (4096 // 64))
    assert st["kernel_launches"] == 3 * -(-S // (4096 // 96)) and st["rows"] == S     # 96 bytes a row: 42-row passes
    want = eng.fisher_exact(_allele_tables(got).reshape(-1, 6)).reshape(-1, 4)
    assert np.array_equal(l, want, equal_nan=True)
    g2, p2, l2 = eng.genotype_tests(0, S, case.seed, hwe=False)
    assert p2 is None and np.array_equal(g2, got) and np.array_equal(l2, l, equal_nan=True)
    g3, p3, l3 = eng.genotype_tests(0, S, case.seed, fisher=False)
    assert l3 is None and np.array_equal(p3, p, equal_nan=True)
    cut = [0, 1, 7, 7, S // 2, S - 1, S]
    parts = [eng.genotype_tests(a, b, case.seed) for a, b in zip(cut, cut[1:])]
    assert np.array_equal(np.concatenate([q[2] for q in parts]), l, equal_nan=True)
    dev = eng.genotype_tests_device(0, S, case.seed)
    assert {k: dev[k] for k in ("rows", "calls", "kernel_launches")} == {k: st[k] for k in ("rows", "calls", "kernel_launches")}
    cls = np.asarray([{"X": 1, "Y": 2, "MT": 3}.get(s.chromosome, 0) for s in case.snps])
    hap = cls >= 2
    assert np.isnan(l[hap][:, [0, 2, 3]]).all()
    assert (l[~np.isnan(l)] <= 0).all()
    eng.close()


@pytest.mark.gpu
def test_genotype_tests_refuse_multiallelic_rows_before_any_work():
    import ctypes
    from dna_factory_b200 import _native
    case = synth_case(40, 20, seed=5, exotic=True)
    eng = _geno_engine(case)
    k = [len(s.tuples) for s in case.snps]
    bad = next(r for r, kr in enumerate(k) if kr > 2)
    out = np.full((20, 10), 0xABABABAB, np.uint32)
    l = np.full((20, 4), 7.0)
    st = _native.Stats()
    f64p = ctypes.POINTER(ctypes.c_double)
    rc = eng._lib.dnaf_genotype_tests(eng._h, 0, 20, case.seed, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), None,
                                      l.ctypes.data_as(f64p), ctypes.byref(st))
    assert rc == _native.E_INPUT
    assert ("row %d " % bad) in eng._lib.dnaf_last_error(eng._h).decode()
    assert (out == 0xABABABAB).all() and (l == 7.0).all() and st.kernel_launches == 0
    with pytest.raises(_native.DnafError) as e:
        eng.genotype_tests_device(0, 20, case.seed)
    assert e.value.code == _native.E_INPUT
    a, b = _runs(k)[0]
    assert eng.genotype_tests(a, b, case.seed)[2].shape == (b - a, 4)     # the context is still usable
    eng.close()


@pytest.mark.gpu
def test_cli_fisher_matches_its_own_vcf(tmp_path, monkeypatch):
    """--fisher on the pinned reference CLI run: population.assoc.fisher / .model.fisher are the text of the genotypes
    recounted from the run's own population.vcf.gz (log10 P by dnaf_fisher_exact of the recount); --gpus 2 writes the
    same bytes; the files of --assoc --model --hardy are byte-identical with and without --fisher."""
    from dna_factory_b200 import _native, fisher
    from dna_factory_b200.snp import SnpTable
    out = tmp_path / "f1"
    flags = ["--assoc", "--model", "--hardy"]
    _cli_small(monkeypatch, out, flags + ["--fisher"])
    table = SnpTable.read_json_gz_table(str(out / "snps.json.gz"))
    vcf = gzip.decompress((out / "population.vcf.gz").read_bytes())
    body = b"".join(ln + b"\n" for ln in vcf.split(b"\n")[:-1] if not ln.startswith(b"#"))
    ctl = [ln.split("\t")[5] == "1" for ln in (out / "population.fam").read_text().splitlines()]
    want = geno_from_text(body, ctl)
    assert len(want) == len(table) == 400
    with _native.Engine(0) as eng:
        l = eng.fisher_exact(_allele_tables(want).reshape(-1, 6)).reshape(-1, 4)
    assert (out / "population.assoc.fisher").read_bytes() == fisher.assoc_fisher_bytes(table, want, l)
    assert (out / "population.model.fisher").read_bytes() == fisher.model_fisher_bytes(table, want, l)
    report = (out / "deleterious_fisher.txt").read_text().splitlines()
    assert len(report) == 1 + sum(len(json.loads(ln)["deleterious"]) for ln in open(out / "deleterious.json"))
    _cli_small(monkeypatch, tmp_path / "f2", ["--fisher", "--gpus", "2"])
    for name in ("population.assoc.fisher", "population.model.fisher", "deleterious_fisher.txt"):
        assert (tmp_path / "f2" / name).read_bytes() == (out / name).read_bytes(), name
    _cli_small(monkeypatch, tmp_path / "n", flags)
    names = sorted(os.listdir(tmp_path / "n"))
    assert "population.assoc.fisher" not in names
    for name in names:
        got, ref = (tmp_path / "n" / name).read_bytes(), (out / name).read_bytes()
        if name.endswith(".json.gz"):      # gzip's MTIME field (bytes 4-7) holds the wall clock of each run
            got, ref = got[:4] + got[8:], ref[:4] + ref[8:]
        assert got == ref, name


@pytest.mark.gpu
def test_cli_planted_snps_under_fisher_rec(tmp_path, monkeypatch, capsys):
    """The one-group, three-SNP config of test_cli_planted_snps_under_rec: every planted SNP passes P < 0.05 / S under
    Fisher REC and ranks in the top 3 by it, with no NA, also where the chi-square REC test is NA by the cell rule."""
    import re
    from dna_factory_b200 import pop_factory
    cfg = tmp_path / "one_group.yml"
    cfg.write_text("planted:\n  mutation_weights:\n  - 1\n  - 1\n  - 1\n  num_instances: 1\n  population_weight: 1\n"
                   "  max_minor_allele_freq: 0.1\n")
    out = tmp_path / "out"
    _fixed_clock(monkeypatch)
    random.seed(99)
    pop_factory.main(["-s", "2000", "-c", "2000", "-x", "3000", "-f", "0.01", "-p", str(cfg), "--outdir", str(out),
                      "--seed", "2024", "--fisher"])
    printed = capsys.readouterr().out
    m = re.search(r"3 of 3 planted deleterious SNPs pass P < 0.05 / 3000 = \S+ under Fisher REC and \d under Fisher "
                  r"ALLELIC; (\d) of the REC passes have no chi-square REC test", printed)
    assert m, printed
    lines = [ln.split("\t") for ln in (out / "deleterious_fisher.txt").read_text().splitlines()]
    col = {name: i for i, name in enumerate(lines[0])}
    assert len(lines) == 4
    for ln in lines[1:]:
        assert int(ln[col["FORCED"]]) > 0
        assert ln[col["P_REC"]] != "NA" and int(ln[col["RANK_REC"]]) <= 3
        assert float(ln[col["LOG10P_REC"]]) < math.log10(0.05 / 3000)
    assert not (out / "population.model").exists()
