"""Genotypic tests (--model) and Hardy-Weinberg exact tests (--hardy): genotype counts from k_geno
(dnaf_genotype_counts*), exact-test P from k_hwe (dnaf_hwe_exact), the .model / .hwe text from dnaf_format_model /
dnaf_format_hardy, and the planted-SNP report of dna_factory_b200.model.

The counts are checked against recounts written from the counting rule (every cell the VCF text prints counts once)
over independent sources: the three-kernel genotype export (dnaf_genotypes), the reference's golden rows and the CLI's
own population.vcf.gz.  The exact test is checked against a log-space full enumeration; the formatters against a
per-line Python rendering, scipy and the variance form of the trend test."""
import json
import math
import os
import random

import numpy as np
import pytest

from tests.cases import GOLDEN, ROW_CASES, load_case, synth_case
from tests.test_assoc import _ctl, _dense_case, _engine, _fixed_clock, _runs, _snps_gz, _table, counts_from_text

TIE = 1e-7   # the relative tie tolerance of dnaf_hwe_exact


# ------------------------------------------------------------------------------------------------------------ helpers
def geno_from_genotypes(g, is_control):
    """[rows][10] counts from dnaf_genotypes' [rows][n][2] allele indices (0xFF = allele not printed)."""
    dip = (g[:, :, 0] != 0xFF) & (g[:, :, 1] != 0xFF)
    hap = (g[:, :, 0] != 0xFF) & (g[:, :, 1] == 0xFF)
    het = dip & (g[:, :, 0] != g[:, :, 1])
    hom = dip & (g[:, :, 0] == 1) & (g[:, :, 1] == 1)
    hap_alt = hap & (g[:, :, 0] == 1)
    case = ~np.asarray(is_control, bool)[None, :]
    cols = [m & grp for grp in (case, ~case) for m in (dip, het, hom, hap, hap_alt)]
    return np.stack([c.sum(1) for c in cols], 1).astype(np.uint32).reshape(-1, 10)


def geno_from_text(text, is_control):
    """The same from VCF rows: 'a/b' is a diploid cell, 'a' a haploid one, '.' nothing; allele 1 is ALT."""
    case = ~np.asarray(is_control, bool)
    out = []
    for line in text.split(b"\n")[:-1]:
        cells = line.split(b"\t")[9:] if len(case) else []
        assert len(cells) == len(case)
        row = [0] * 10
        for c, is_case in zip(cells, case):
            j = 0 if is_case else 5
            if c == b".":
                continue
            al = c.split(b"/")
            if len(al) == 2:
                row[j] += 1
                row[j + 1] += al[0] != al[1]
                row[j + 2] += al[0] == al[1] == b"1"
            else:
                row[j + 3] += 1
                row[j + 4] += al[0] == b"1"
        out.append(row)
    return np.asarray(out, np.uint32).reshape(-1, 10)


def triples(counts):
    """[rows][3][3]: (n11, n12, n22) of ALL, AFF, UNAFF per row."""
    c = np.asarray(counts, np.int64).reshape(-1, 10)
    aff = np.stack([c[:, 2], c[:, 1], c[:, 0] - c[:, 1] - c[:, 2]], 1)
    unaff = np.stack([c[:, 7], c[:, 6], c[:, 5] - c[:, 6] - c[:, 7]], 1)
    return np.stack([aff + unaff, aff, unaff], 1)


def hwe_ref(n11, n12, n22, exact=False):
    """Two-sided Hardy-Weinberg exact P by full enumeration in log space: every het count h of the same n and rare-allele
    count, log p(h) from log-gamma, P = sum of p(h) <= p(n12) (1 + TIE) over the sum of all.  exact=True evaluates the
    log-gamma terms with mpmath at 40 digits (float64 gammaln of arguments near 10^5 is only good to about 1e-10)."""
    from scipy.special import gammaln
    n = n11 + n12 + n22
    if n == 0:
        return math.nan
    r = 2 * min(n11, n22) + n12
    h = np.arange(r % 2, r + 1, 2)
    hr = (r - h) // 2
    hc = n - h - hr
    lp = -gammaln(h + 1.0) - gammaln(hr + 1.0) - gammaln(hc + 1.0) + h * math.log(2.0)
    if exact:
        import mpmath
        mpmath.mp.dps = 40
        keep = lp - lp.max() > -800          # the rest is below 1e-347 of the mode in any precision
        h, hr, hc = h[keep], hr[keep], hc[keep]
        lpm = [-mpmath.loggamma(a + 1) - mpmath.loggamma(b + 1) - mpmath.loggamma(c + 1) + a * mpmath.log(2)
               for a, b, c in zip(h.tolist(), hr.tolist(), hc.tolist())]
        top = max(lpm)
        p = np.asarray([float(mpmath.exp(v - top)) for v in lpm])
    else:
        p = np.exp(lp - lp.max())
    obs = p[h == n12]
    if len(obs) == 0:                        # the observed het count lies in the part dropped above: P is 0 in double
        return 0.0
    return float(p[p <= obs[0] * (1 + TIE)].sum() / p.sum())


def assert_p_close(got, want, rel=1e-12):
    """Relative agreement wherever the reference P >= 1e-290; below that the kernel may give 0."""
    if math.isnan(want):
        assert math.isnan(got)
    elif want >= 1e-290:
        assert got == pytest.approx(want, rel=rel, abs=0), (got, want)
    else:
        assert 0 <= got < 1e-280


def _g(v):
    return "NA" if v is None else "%.4g" % v


CHR_CODE = {"X": "23", "Y": "24", "MT": "26"}


def _chi2_table(obs):
    """Pearson chi-square of a 2 x k table, None for any zero margin."""
    obs = np.asarray(obs, float)
    rt, ct, n = obs.sum(1), obs.sum(0), obs.sum()
    if (rt <= 0).any() or (ct <= 0).any():
        return None
    e = np.outer(rt, ct) / n
    return float(((obs - e) ** 2 / e).sum())


def _trend_variance_form(case, ctrl):
    """Cochran-Armitage T^2 / Var(T) with scores x = 2, 1, 0 (ALT copies), from its definition."""
    x = np.asarray([2.0, 1.0, 0.0])
    r, s = np.asarray(case, float), np.asarray(ctrl, float)
    R, S = r.sum(), s.sum()
    if R <= 0 or S <= 0:
        return None
    N = R + S
    c = r + s
    T = float((x * (r * S - s * R)).sum())
    var = R * S / N * (float((x * x * c * (N - c)).sum()) - 2 * sum(x[i] * x[j] * c[i] * c[j]
                                                                      for i in range(3) for j in range(i + 1, 3)))
    return T * T / var if var > 0 else None


def model_lines_python(label, snp_id, k, ref, alt, c):
    """The five .model body lines of one row, written from the definitions, independent of the C formatter."""
    a11, a12, a22 = c[2], c[1], c[0] - c[1] - c[2]
    u11, u12, u22 = c[7], c[6], c[5] - c[6] - c[7]
    alt_a, alt_u = 2 * a11 + a12 + c[4], 2 * u11 + u12 + c[9]
    ref_a, ref_u = 2 * c[0] + c[3] - alt_a, 2 * c[5] + c[8] - alt_u
    cells_ok = min(a11, a12, a22, u11, u12, u22) >= 5
    geno = _chi2_table([[a11, a12, a22], [u11, u12, u22]]) if cells_ok else None
    trend = _trend_variance_form([a11, a12, a22], [u11, u12, u22])
    allelic = _chi2_table([[alt_a, ref_a], [alt_u, ref_u]])
    dom = _chi2_table([[a11 + a12, a22], [u11 + u12, u22]]) if cells_ok else None
    rec = _chi2_table([[a11, a12 + a22], [u11, u12 + u22]]) if cells_ok else None
    rows = [("GENO", "%d/%d/%d" % (a11, a12, a22), "%d/%d/%d" % (u11, u12, u22), geno, 2),
            ("TREND", "%d/%d/%d" % (a11, a12, a22), "%d/%d/%d" % (u11, u12, u22), trend, 1),
            ("ALLELIC", "%d/%d" % (alt_a, ref_a), "%d/%d" % (alt_u, ref_u), allelic, 1),
            ("DOM", "%d/%d" % (a11 + a12, a22), "%d/%d" % (u11 + u12, u22), dom, 1),
            ("REC", "%d/%d" % (a11, a12 + a22), "%d/%d" % (u11, u12 + u22), rec, 1)]
    a1 = chr(alt) if k == 2 else "0"
    out = []
    for test, aff, unaff, x, df in rows:
        p = None if x is None else (math.erfc(math.sqrt(x / 2)) if df == 1 else math.exp(-x / 2))
        out.append("%4s %12s %4s %4s %8s %14s %14s %12s %4s %12s\n" % (
            CHR_CODE.get(label, label), "rs%d" % snp_id, a1, chr(ref), test, aff, unaff, _g(x),
            "NA" if x is None else str(df), _g(p)))
    return "".join(out)


def hardy_lines_python(label, snp_id, k, ref, alt, c, p):
    out = []
    for t, (n11, n12, n22) in zip(("ALL", "AFF", "UNAFF"), triples(c)[0]):
        n = n11 + n12 + n22
        f = (2 * n11 + n12) / (2 * n) if n else None
        out.append("%4s %12s %8s %4s %4s %20s %8s %8s %12s\n" % (
            CHR_CODE.get(label, label), "rs%d" % snp_id, t, chr(alt) if k == 2 else "0", chr(ref),
            "%d/%d/%d" % (n11, n12, n22), _g(n12 / n if n else None), _g(2 * f * (1 - f) if n else None),
            "NA" if math.isnan(p[{"ALL": 0, "AFF": 1, "UNAFF": 2}[t]]) else _g(p[{"ALL": 0, "AFF": 1, "UNAFF": 2}[t]])))
    return "".join(out)


def _random_counts(S, rs, big=3000):
    """uint32[S, 10] counts that obey the counter relations (het + hom <= dip)."""
    c = np.zeros((S, 10), np.int64)
    for j in (0, 5):
        c[:, j] = rs.randint(0, big, S)
        c[:, j + 1] = (c[:, j] * rs.rand(S) * 0.6).astype(np.int64)
        c[:, j + 2] = ((c[:, j] - c[:, j + 1]) * rs.rand(S) * 0.5).astype(np.int64)
        c[:, j + 3] = rs.randint(0, 50, S) * (rs.rand(S) < 0.3)
        c[:, j + 4] = (c[:, j + 3] * rs.rand(S)).astype(np.int64)
    return c.astype(np.uint32)


# ------------------------------------------------------------------------------------------------------------- CPU
def test_format_model_and_hardy_match_per_line_rendering():
    from dna_factory_b200 import model
    rs = np.random.RandomState(8)
    S = 300
    t = _table(S, rs)
    counts = _random_counts(S, rs)
    counts[0] = 0                                          # nothing observed
    counts[1] = [40, 0, 0, 0, 0, 30, 0, 0, 0, 0]           # monomorphic REF
    counts[2] = [40, 0, 40, 0, 0, 30, 0, 30, 0, 0]         # monomorphic ALT
    counts[3] = [0, 0, 0, 0, 0, 50, 10, 10, 0, 0]          # no cases
    counts[4] = [60, 20, 10, 0, 0, 0, 0, 0, 0, 0]          # no controls
    counts[5] = [100, 30, 4, 0, 0, 100, 40, 20, 0, 0]      # one cell below 5: GENO / DOM / REC NA, TREND not
    counts[6] = [0, 0, 0, 40, 12, 0, 0, 0, 35, 3]          # haploid only (Y / MT rows): ALLELIC only
    counts[7] = [3000, 0, 3000, 0, 0, 3000, 3000, 0, 0, 0]  # P far below 1e-300
    p = rs.rand(S, 3)
    p[0] = np.nan
    p[6] = np.nan
    p[7] = [0.0, 1.0, 1e-200]
    want_m, want_h = [], []
    for r in range(S):
        args = (t.chrom_labels[t.chrom_idx[r]], int(t.ids[r]), int(t.n_alleles[r]), int(t.nts[r, 0]), int(t.nts[r, 1]))
        want_m.append(model_lines_python(*args, [int(v) for v in counts[r]]))
        want_h.append(hardy_lines_python(*args, counts[r], p[r]))
    got_m = model.model_bytes(t, counts)
    got_h = model.hardy_bytes(t, counts, p)
    assert got_m == model.MODEL_HEADER + "".join(want_m).encode()
    assert got_h == model.HWE_HEADER + "".join(want_h).encode()
    m = [ln.split() for ln in got_m.decode().splitlines()]
    assert m[0] == ["CHR", "SNP", "A1", "A2", "TEST", "AFF", "UNAFF", "CHISQ", "DF", "P"]
    assert [ln[4] for ln in m[1:6]] == ["GENO", "TREND", "ALLELIC", "DOM", "REC"]
    row5 = {ln[4]: ln for ln in m[1 + 5 * 5:1 + 5 * 6]}
    assert [row5[k][7] for k in ("GENO", "DOM", "REC")] == ["NA"] * 3 and row5["TREND"][7] != "NA"
    row6 = {ln[4]: ln for ln in m[1 + 5 * 6:1 + 5 * 7]}
    assert [row6[k][7:] for k in ("GENO", "TREND", "DOM", "REC")] == [["NA"] * 3] * 4 and row6["ALLELIC"][7] != "NA"
    assert {ln[7:] == ["NA"] * 3 for ln in m[1:6]} == {True}               # empty row
    assert {ln[7:] == ["NA"] * 3 for ln in m[6:16]} == {True}              # monomorphic rows
    assert {ln[7:] == ["NA"] * 3 for ln in m[16:26]} == {True}             # no cases / no controls
    assert m[1 + 5 * 7 + 2][9] == "0"                                      # ALLELIC P underflows
    h = [ln.split() for ln in got_h.decode().splitlines()]
    assert h[0] == ["CHR", "SNP", "TEST", "A1", "A2", "GENO", "O(HET)", "E(HET)", "P"]
    assert [ln[2] for ln in h[1:4]] == ["ALL", "AFF", "UNAFF"]
    assert h[1 + 3 * 6][5:] == ["0/0/0", "NA", "NA", "NA"]
    assert model.model_bytes(t.take(np.arange(0)), np.zeros((0, 10), np.uint32)) == model.MODEL_HEADER
    assert model.hardy_bytes(t.take(np.arange(0)), np.zeros((0, 10), np.uint32), np.zeros((0, 3))) == model.HWE_HEADER


def test_allelic_geno_dom_rec_agree_with_scipy_and_trend_with_its_variance_form():
    from scipy.stats import chi2, chi2_contingency
    from dna_factory_b200 import model
    rs = np.random.RandomState(3)
    counts = _random_counts(200, rs, big=800)
    counts[:, [0, 5]] += 60                                     # most rows pass the cell rule
    counts[:, [1, 6]] += 10
    counts[:, [2, 7]] += 10
    x2 = model.model_chisq(counts)
    t = _table(200, rs, labels=("1",))
    t.n_alleles[:] = 2
    lines = [ln.split() for ln in model.model_bytes(t, counts).decode().splitlines()[1:]]
    checked = 0
    for r, c in enumerate(counts.astype(np.int64)):
        a = [c[2], c[1], c[0] - c[1] - c[2]]
        u = [c[7], c[6], c[5] - c[6] - c[7]]
        alt_a, alt_u = 2 * a[0] + a[1] + c[4], 2 * u[0] + u[1] + c[9]
        tables = {2: [[alt_a, 2 * c[0] + c[3] - alt_a], [alt_u, 2 * c[5] + c[8] - alt_u]]}
        if min(a + u) >= 5:
            tables[0] = [a, u]
            tables[3] = [[a[0] + a[1], a[2]], [u[0] + u[1], u[2]]]
            tables[4] = [[a[0], a[1] + a[2]], [u[0], u[1] + u[2]]]
            checked += 1
        else:
            assert np.isnan(x2[r, [0, 3, 4]]).all()
        for j, tab in tables.items():
            stat, p = chi2_contingency(tab, correction=False)[:2]
            assert x2[r, j] == pytest.approx(stat, rel=1e-10)
            assert float(lines[5 * r + j][9]) == pytest.approx(p, rel=1e-3, abs=1e-300)
            assert model.chi2_p(x2[r, j], 2 if j == 0 else 1) == pytest.approx(chi2.sf(stat, 2 if j == 0 else 1), rel=1e-9,
                                                                               abs=1e-300)
        assert x2[r, 1] == pytest.approx(_trend_variance_form(a, u), rel=1e-10)
    assert checked > 150


def test_cell_rule_and_na_cases_of_model_chisq():
    from dna_factory_b200 import model
    c = np.zeros((5, 10), np.uint32)
    c[1] = [50, 10, 5, 0, 0, 50, 10, 5, 0, 0]      # every cell >= 5: every test
    c[2] = [50, 10, 4, 0, 0, 50, 10, 5, 0, 0]      # a11 = 4: GENO / DOM / REC NA
    c[3] = [0, 0, 0, 30, 10, 0, 0, 0, 30, 20]      # Y / MT shape: ALLELIC only
    c[4] = [50, 10, 5, 0, 0, 0, 0, 0, 0, 0]        # no controls: NA everywhere
    x = model.model_chisq(c)
    assert np.isnan(x[0]).all() and np.isnan(x[4]).all()
    assert not np.isnan(x[1]).any()
    assert np.isnan(x[2, [0, 3, 4]]).all() and not np.isnan(x[2, [1, 2]]).any()
    assert np.isnan(x[3, [0, 1, 3, 4]]).all() and not np.isnan(x[3, 2])


def test_deleterious_model_report_text():
    from dna_factory_b200 import model
    from dna_factory_b200.pop_factory import DeleteriousGroup
    rs = np.random.RandomState(2)
    S = 40
    t = _table(S, rs, labels=("1", "2"))
    t.n_alleles[:] = 2
    counts = np.tile(np.asarray([400, 160, 20, 0, 0, 400, 160, 20, 0, 0], np.uint32), (S, 1))
    counts[5] = [400, 150, 120, 0, 0, 400, 160, 20, 0, 0]   # recessive signal: top under REC
    counts[6] = [400, 200, 30, 0, 0, 400, 160, 20, 0, 0]    # weaker, mostly additive
    counts[7] = [400, 160, 3, 0, 0, 400, 160, 20, 0, 0]     # a cell below 5: REC NA
    hwe = np.full((S, 3), 0.5)
    hwe[5] = [1e-9, 1e-30, 0.3]
    g1 = DeleteriousGroup("g1", 1)
    g1.deleterious = {int(t.ids[5]): 1, int(t.ids[6]): 0.5, 999: 0.2}        # 999: not in the table
    g2 = DeleteriousGroup.from_json(json.dumps({"name": "g2", "population_weight": 1, "deleterious": {str(t.ids[7]): 1}}))
    orow = np.asarray([5, 5, 6], np.uint64)
    text, summary = model.deleterious_model_report(t, {"g1": g1, "g2": g2}, counts, hwe, orow)
    lines = [ln.split("\t") for ln in text.decode().splitlines()]
    assert tuple(lines[0]) == model.REPORT_COLUMNS
    col = {k: i for i, k in enumerate(lines[0])}
    rec = {ln[1]: ln for ln in lines[1:]}
    r5, r6, r7 = rec["rs%d" % t.ids[5]], rec["rs%d" % t.ids[6]], rec["rs%d" % t.ids[7]]
    assert r5[col["FORCED"]] == "2" and r6[col["FORCED"]] == "1"
    assert (r5[col["AFF"]], r5[col["UNAFF"]]) == ("120/150/130", "20/160/220")
    assert r5[col["RANK_REC"]] == "1" and r5[col["RANK_ALLELIC"]] == "1"
    assert r6[col["RANK_REC"]] == "2"
    assert (r5[col["HWE_ALL"]], r5[col["HWE_AFF"]], r5[col["HWE_UNAFF"]]) == ("1e-09", "1e-30", "0.3")
    assert r7[col["GROUP"]] == "g2" and r7[col["FORCED"]] == "0"          # string key: found, forces nothing
    assert r7[col["P_REC"]] == "NA" and r7[col["RANK_REC"]] == str(S)   # behind the 39 tested rows
    assert r7[col["P_ALLELIC"]] != "NA"
    assert rec["rs999"][2:] == ["NA", "NA", "0.2", "0"] + ["NA"] * 12
    assert len(lines) == 5
    assert summary == ("1 of 4 planted deleterious SNPs pass P < 0.05 / 40 = 0.00125 under REC and 2 under ALLELIC; "
                       "1 have no REC test (a genotype cell below 5); 1 have HWE P < 1e-06 in ALL and 0 in UNAFF")


def test_model_and_hardy_flags_parse():
    from dna_factory_b200 import pop_factory
    base = ["-s", "3", "-c", "4"]
    a = pop_factory.parse_cmd_args(base + ["--model", "--hardy"])
    assert a.model is True and a.hardy is True
    a = pop_factory.parse_cmd_args(base)
    assert a.model is False and a.hardy is False


@pytest.mark.parametrize("flags,sizes,match", [
    (["--model"], ("-s", "5", "-c", "4"), "--model: SNP rs9001"),
    (["--hardy"], ("-s", "5", "-c", "4"), "--hardy: SNP rs9001"),
    (["--model"], ("-s", "0", "-c", "4"), "--model needs cases and controls"),
    (["--model", "--hardy"], ("-s", "5", "-c", "0"), "--model needs cases and controls")])
def test_model_refusals_before_the_vcf(tmp_path, flags, sizes, match):
    """A multi-allelic table (both flags) and a population without cases or controls (--model) fail before any output."""
    from dna_factory_b200 import pop_factory
    extra = b'{"id": 9001, "chromosome": "1", "position": 7000000, "tuples": {"A": 0.5, "C": 0.8, "G": 1.0}}\n'
    snps_gz = _snps_gz(tmp_path, extra if "rs9001" in match else None)
    out = tmp_path / "out"
    random.seed(1)
    with pytest.raises(ValueError, match=match):
        pop_factory.main(list(sizes) + ["--snps_file", str(snps_gz), "-p",
                                        os.path.join(GOLDEN, "cli_small", "deleterious_config.yml"), "--outdir", str(out),
                                        "--seed", "7"] + flags)
    for name in ("population.vcf.gz", "population.model", "population.hwe"):
        assert not (out / name).exists()


def test_hwe_reference_sanity():
    """The test's own reference on cases worked by hand: n = 2 with two rare alleles has p(h=0) = 1/3 and p(h=2) = 2/3;
    a monomorphic sample has one table; the observed het count at the mode gives P = 1."""
    assert hwe_ref(1, 0, 1) == pytest.approx(1 / 3, rel=1e-12)
    assert hwe_ref(0, 2, 0) == pytest.approx(1.0, rel=1e-12)
    assert hwe_ref(0, 0, 10) == 1.0
    assert hwe_ref(25, 50, 25) == pytest.approx(1.0, rel=1e-12)
    assert 0 < hwe_ref(7, 21, 72) < 1
    assert math.isnan(hwe_ref(0, 0, 0))


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_hwe_exact_every_small_table():
    """Every (n11, n12, n22) with n11 + n12 + n22 <= 40, ties included, against the log-space enumeration."""
    from dna_factory_b200 import _native
    geno = np.asarray([(a, b, n - a - b) for n in range(41) for a in range(n + 1) for b in range(n - a + 1)], np.uint32)
    with _native.Engine(0) as eng:
        got = eng.hwe_exact(geno)
    ties = 0
    for (a, b, c), p in zip(geno.tolist(), got):
        want = hwe_ref(a, b, c)
        assert_p_close(p, want)
        ties += want == 1.0 and b != 0
    assert np.isnan(got[0]) and ties > 10


@pytest.mark.gpu
def test_hwe_exact_random_counts_up_to_1e5():
    """Random tables up to N = 10^5 around HWE and far from it, against the enumeration in 40-digit log-gamma."""
    from dna_factory_b200 import _native
    rs = np.random.RandomState(17)
    rows = []
    for n in (57, 1000, 20000, 100000):
        for _ in range(3):
            f = rs.uniform(0.01, 0.5)
            a = rs.binomial(n, f * f)
            b = rs.binomial(n - a, 2 * f * (1 - f) / (1 - f * f))
            rows.append((a, b, n - a - b))                              # near HWE
        rows.append((n // 10, n // 100, n - n // 10 - n // 100))        # far too few hets: P tiny or 0
        rows.append((n // 400, n // 4, n - n // 400 - n // 4))          # too many hets
    rows.append((0, 100000, 0))
    rows.append((0, 1, 99999))
    with _native.Engine(0) as eng:
        got = eng.hwe_exact(np.asarray(rows, np.uint32))
    for (a, b, c), p in zip(rows, got):
        assert_p_close(p, hwe_ref(a, b, c, exact=True))


def _geno_engine(case, chunk=None, row_base=None):
    return _engine(case, chunk=chunk, row_base=row_base)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 15, 16, 17, 4095, 4096, 4097, 20000, 100003])
def test_genotype_counts_match_the_genotype_export(n):
    """k_geno against counts taken from the three-kernel export, across the 16-sample word and the 4096-sample CTA
    tile, with a row counter offset and a chunk that makes many passes; the P of every pass equals dnaf_hwe_exact of
    its counts, and the allele invariant holds against dnaf_allele_counts."""
    case = _dense_case(n, seed=n)
    S = len(case.snps)
    eng = _geno_engine(case, chunk=4096, row_base=1000 + n)
    want = geno_from_genotypes(eng.genotypes(0, S, case.seed), _ctl(case))
    got, p, st = eng.genotype_counts_stats(0, S, case.seed)
    assert np.array_equal(got, want)
    assert np.array_equal(p, eng.hwe_exact(triples(got).reshape(-1, 3)).reshape(-1, 3), equal_nan=True)
    assert st["rows"] == S and st["calls"] == S * n and st["kernel_launches"] == 2 * -(-S // 64)
    assert st["ms_sample"] > 0 and st["ms_total"] >= st["ms_sample"]
    g = got.astype(np.int64)
    alleles = np.stack([2 * g[:, 2] + g[:, 1] + g[:, 4], 2 * g[:, 0] + g[:, 3],
                        2 * g[:, 7] + g[:, 6] + g[:, 9], 2 * g[:, 5] + g[:, 8]], 1)
    assert np.array_equal(alleles, eng.allele_counts(0, S, case.seed))
    eng.close()


@pytest.mark.gpu
def test_genotype_counts_over_many_passes_and_ranges():
    """700 rows of all four classes at N = 4097 (two CTAs per row): 11 passes with the exact tests, 7 without; ranges
    concatenate; the device-only call does the same launches; the allele invariant holds on every row."""
    case = synth_case(4097, 700, seed=44, chroms=["1", "X", "Y", "MT", "5"], n_del=40)
    S = len(case.snps)
    eng = _geno_engine(case, chunk=4096, row_base=3 * 2 ** 32 + 17)
    want = geno_from_genotypes(eng.genotypes(0, S, case.seed), _ctl(case))
    got, p, st = eng.genotype_counts_stats(0, S, case.seed)
    assert st["kernel_launches"] == 2 * 11
    assert np.array_equal(got, want)
    got2, p2, st2 = eng.genotype_counts_stats(0, S, case.seed, hwe=False)
    assert p2 is None and st2["kernel_launches"] == 7 and np.array_equal(got2, want)
    cut = [0, 1, 7, 7, S // 2, S - 1, S]
    parts = [eng.genotype_counts(a, b, case.seed) for a, b in zip(cut, cut[1:])]
    assert np.array_equal(np.concatenate([q[0] for q in parts]), got)
    assert np.array_equal(np.concatenate([q[1] for q in parts]), p, equal_nan=True)
    dev = eng.genotype_counts_device(0, S, case.seed)
    assert {k: dev[k] for k in ("rows", "calls", "kernel_launches")} == {k: st[k] for k in ("rows", "calls", "kernel_launches")}
    cls = np.asarray([{"X": 1, "Y": 2, "MT": 3}.get(s.chromosome, 0) for s in case.snps])
    assert np.isnan(p[cls >= 2]).all() and not np.isnan(p[cls <= 1]).any()
    assert (got[cls >= 2][:, [0, 5]] == 0).all() and (got[cls == 0][:, [3, 8]] == 0).all()
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ROW_CASES)
def test_genotype_counts_match_the_reference_golden_rows(name):
    """X, Y and MT for both sexes, forced minors, K = 1 rows, a row counter above 2^32, N = 0; K > 2 rows skipped."""
    case = load_case(name)
    lines = case.text.split(b"\n")[:-1]
    eng = _geno_engine(case)
    runs = _runs([len(s.tuples) for s in case.snps])
    assert runs
    for a, b in runs:
        got, _ = eng.genotype_counts(a, b, case.seed)
        want = geno_from_text(b"".join(ln + b"\n" for ln in lines[a:b]), _ctl(case))
        assert np.array_equal(got, want), (name, a, b)
    eng.close()


@pytest.mark.gpu
def test_genotype_counts_refuse_multiallelic_rows_before_any_work():
    import ctypes
    from dna_factory_b200 import _native
    case = synth_case(40, 20, seed=5, exotic=True)
    eng = _geno_engine(case)
    k = [len(s.tuples) for s in case.snps]
    bad = next(r for r, kr in enumerate(k) if kr > 2)
    out = np.full((20, 10), 0xABABABAB, np.uint32)
    p = np.full((20, 3), 7.0)
    st = _native.Stats()
    rc = eng._lib.dnaf_genotype_counts(eng._h, 0, 20, case.seed, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                       p.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ctypes.byref(st))
    assert rc == _native.E_INPUT
    assert ("row %d " % bad) in eng._lib.dnaf_last_error(eng._h).decode()
    assert (out == 0xABABABAB).all() and (p == 7.0).all() and st.kernel_launches == 0
    with pytest.raises(_native.DnafError) as e:
        eng.genotype_counts_device(0, 20, case.seed)
    assert e.value.code == _native.E_INPUT
    a, b = _runs(k)[0]
    assert eng.genotype_counts(a, b, case.seed)[0].shape == (b - a, 10)     # the context is still usable
    eng.close()


def _cli_small(monkeypatch, out, extra):
    from dna_factory_b200 import pop_factory
    gold = os.path.join(GOLDEN, "cli_small")
    meta = json.load(open(os.path.join(gold, "meta.json")))
    _fixed_clock(monkeypatch)
    random.seed(meta["python_random_seed"])
    pop_factory.main(meta["args"] + ["-p", os.path.join(gold, "deleterious_config.yml"), "--outdir", str(out),
                                     "--seed", str(meta["philox_seed"])] + extra)


@pytest.mark.gpu
def test_cli_model_hardy_match_their_own_vcf(tmp_path, monkeypatch):
    """--model --hardy --assoc on the pinned reference CLI run: population.model / .hwe are the text of the genotypes
    recounted from the run's own population.vcf.gz (P of the exact tests by dnaf_hwe_exact of the recount),
    population.assoc is unchanged by the other flags, and --gpus 2 writes the same bytes."""
    import gzip
    from dna_factory_b200 import _native, assoc, model
    from dna_factory_b200.snp import SnpTable
    out = tmp_path / "g1"
    _cli_small(monkeypatch, out, ["--model", "--hardy", "--assoc"])
    table = SnpTable.read_json_gz_table(str(out / "snps.json.gz"))
    vcf = gzip.decompress((out / "population.vcf.gz").read_bytes())
    body = b"".join(ln + b"\n" for ln in vcf.split(b"\n")[:-1] if not ln.startswith(b"#"))
    ctl = [ln.split("\t")[5] == "1" for ln in (out / "population.fam").read_text().splitlines()]
    want = geno_from_text(body, ctl)
    assert len(want) == len(table) == 400
    with _native.Engine(0) as eng:
        p = eng.hwe_exact(triples(want).reshape(-1, 3)).reshape(-1, 3)
    assert (out / "population.model").read_bytes() == model.model_bytes(table, want)
    assert (out / "population.hwe").read_bytes() == model.hardy_bytes(table, want, p)
    assert (out / "population.assoc").read_bytes() == assoc.assoc_bytes(table, counts_from_text(body, ctl))
    report = (out / "deleterious_model.txt").read_text().splitlines()
    assert len(report) == 1 + sum(len(json.loads(ln)["deleterious"]) for ln in open(out / "deleterious.json"))
    _cli_small(monkeypatch, tmp_path / "a", ["--assoc"])
    for name in ("population.assoc", "deleterious_assoc.txt"):
        assert (tmp_path / "a" / name).read_bytes() == (out / name).read_bytes(), name
    _cli_small(monkeypatch, tmp_path / "g2", ["--model", "--hardy", "--gpus", "2"])
    for name in ("population.model", "population.hwe", "deleterious_model.txt"):
        assert (tmp_path / "g2" / name).read_bytes() == (out / name).read_bytes(), name
    _cli_small(monkeypatch, tmp_path / "h", ["--hardy"])
    assert (tmp_path / "h" / "population.hwe").read_bytes() == (out / "population.hwe").read_bytes()
    assert not (tmp_path / "h" / "population.model").exists()


@pytest.mark.gpu
def test_cli_planted_snps_under_rec(tmp_path, monkeypatch, capsys):
    """One group of three planted SNPs, one forced per case: each ranks in the top 3 under REC, or its REC test is NA by
    the cell rule (fewer than 5 ALT/ALT controls at MAF <= 0.1) and ALLELIC finds it; its cases leave Hardy-Weinberg
    equilibrium."""
    import re
    from dna_factory_b200 import pop_factory
    cfg = tmp_path / "one_group.yml"
    cfg.write_text("planted:\n  mutation_weights:\n  - 1\n  - 1\n  - 1\n  num_instances: 1\n  population_weight: 1\n"
                   "  max_minor_allele_freq: 0.1\n")
    out = tmp_path / "out"
    _fixed_clock(monkeypatch)
    random.seed(99)
    pop_factory.main(["-s", "2000", "-c", "2000", "-x", "3000", "-f", "0.01", "-p", str(cfg), "--outdir", str(out),
                      "--seed", "2024", "--model"])
    printed = capsys.readouterr().out
    m = re.search(r"(\d) of 3 planted deleterious SNPs pass P < 0.05 / 3000 = \S+ under REC and 3 under ALLELIC; "
                  r"(\d) have no REC test", printed)
    assert m and int(m.group(1)) + int(m.group(2)) == 3, printed
    lines = [ln.split("\t") for ln in (out / "deleterious_model.txt").read_text().splitlines()]
    col = {name: i for i, name in enumerate(lines[0])}
    assert len(lines) == 4
    for ln in lines[1:]:
        assert int(ln[col["FORCED"]]) > 0
        assert int(ln[col["RANK_REC"]]) <= 3 or ln[col["P_REC"]] == "NA"
        assert int(ln[col["RANK_ALLELIC"]]) <= 3
        assert float(ln[col["HWE_AFF"]]) < 1e-6
    assert not (out / "population.hwe").exists()


@pytest.mark.gpu
def test_cli_replay_reports_forced_zero(tmp_path, monkeypatch):
    """A --deleterious_file replay keeps string keys, which force nothing (SURVEY R8): every line shows FORCED 0."""
    from dna_factory_b200 import pop_factory
    gold = os.path.join(GOLDEN, "cli_small")
    out = tmp_path / "out"
    _fixed_clock(monkeypatch)
    random.seed(3)
    pop_factory.main(["-s", "40", "-c", "40", "--snps_file", str(_snps_gz(tmp_path)), "--deleterious_file",
                      os.path.join(gold, "deleterious.json"), "--outdir", str(out), "--seed", "5", "--model"])
    lines = [ln.split("\t") for ln in (out / "deleterious_model.txt").read_text().splitlines()]
    n_planted = sum(len(json.loads(ln)["deleterious"]) for ln in open(os.path.join(gold, "deleterious.json")))
    assert len(lines) == 1 + n_planted
    assert all(ln[5] == "0" for ln in lines[1:])
    assert all(ln[3] != "NA" for ln in lines[1:])      # every key found its row through int(key)

