"""max(T) permutation tests (--mperm): the permutation masks of k_perm_masks (dnaf_perm_case_masks), the statistics,
exceedances and maxima of k_mperm (dnaf_mperm*), the .mperm text of dnaf_format_mperm and the planted-SNP report of
dna_factory_b200.mperm.

The permutations are checked against a numpy restatement of Algorithm S over oracle/philox_np; the statistics against
a numpy brute force over the three-kernel genotype export (dnaf_genotypes) and those permutations; the CLI against
EMP1 / EMP2 recomputed from its own population.vcf.gz."""
import gzip
import json
import math
import os
import random

import numpy as np
import pytest

from oracle.philox_np import philox4x32_10
from tests.cases import GOLDEN, synth_case
from tests.test_assoc import _dense_case, _fixed_clock, _runs, _snps_gz, _table
from tests.test_model import CHR_CODE, _cli_small, _geno_engine, geno_from_genotypes

TIE = 1e-7
TAG = 0x4D505200


# ------------------------------------------------------------------------------------------------------------ helpers
def perm_masks_np(seed, n, ncase, first, n_perm):
    """bool[n_perm, n] case sets of permutations first .. first + n_perm - 1 by Algorithm S (include/dnaf_b200.h)."""
    p = np.arange(first, first + n_perm, dtype=np.uint64)
    q = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.zeros((n_perm, len(q), 4), np.uint64)
    ctr[..., 0] = q[None, :]
    ctr[..., 1] = p[:, None]
    ctr[..., 2] = TAG
    ctr[..., 3] = 0xFFFFFFFF
    U = philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32)).reshape(n_perm, -1)[:, :n].astype(np.uint64)
    need = np.full(n_perm, ncase, np.uint64)
    case = np.zeros((n_perm, n), bool)
    for i in range(n):
        c = U[:, i] * np.uint64(n - i) < (need << np.uint64(32))
        case[:, i] = c
        need -= c.astype(np.uint64)
    return case


def pack(case):
    """bool[P, n] -> uint32[P, ceil(n/32)] (bit i & 31 of word i >> 5)."""
    P, n = case.shape
    W = (n + 31) // 32
    b = np.zeros((P, W * 32), np.uint64)
    b[:, :n] = case
    return (b.reshape(P, W, 32) << np.arange(32, dtype=np.uint64)).sum(2).astype(np.uint32)


def chi2(a, b, c, d):
    """The 2x2 Pearson statistic in the operation order of chi2_2x2; NaN where the denominator is 0."""
    den = (a + b) * (c + d) * (a + c) * (b + d)
    x = a * d - b * c
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den > 0, (a + b + c + d) * x * x / np.where(den > 0, den, 1.0), np.nan)


def stats_np(g, cls, case, male):
    """T[P, rows, 2] of the permutations `case` (bool[P, n]) over the genotype export g ([rows][n][2]):
    ALLELIC and REC with the case margins of each row class."""
    dip = (g[:, :, 0] != 0xFF) & (g[:, :, 1] != 0xFF)
    hap = (g[:, :, 0] != 0xFF) & (g[:, :, 1] == 0xFF)
    A = (dip & ((g[:, :, 0] == 1) | (g[:, :, 1] == 1))) | (hap & (g[:, :, 0] == 1))
    B = dip & (g[:, :, 0] == 1) & (g[:, :, 1] == 1)
    C = case.astype(np.int64)
    sa, sb = C @ A.T.astype(np.int64), C @ B.T.astype(np.int64)        # [P, rows]
    alt = (A.sum(1) + B.sum(1)).astype(np.float64)
    obs = (2 * dip.sum(1) + hap.sum(1)).astype(np.float64)
    hom, dipn = B.sum(1).astype(np.float64), dip.sum(1).astype(np.float64)
    m = (case & male[None, :]).sum(1).astype(np.float64)[:, None]
    f = (case & ~male[None, :]).sum(1).astype(np.float64)[:, None]
    cls = np.asarray(cls)[None, :]
    ca = np.where(cls == 0, 2.0 * (m + f), np.where(cls == 1, 2.0 * f + m, np.where(cls == 2, m, m + f)))
    cd = np.where(cls == 0, m + f, np.where(cls == 1, f, 0.0))
    a = (sa + sb).astype(np.float64)
    h = sb.astype(np.float64)
    t0 = chi2(a, ca - a, alt - a, (obs - ca) - (alt - a))
    t1 = chi2(h, cd - h, hom - h, (dipn - cd) - (hom - h))
    return np.stack([t0, t1], 2)


def brute_force(t_obs, t_perm):
    """(exceed[rows, 2], max_t[P, 2]) of the observed statistics and T[P, rows, 2] by the definitions."""
    thr = t_obs * (1 - TIE)
    with np.errstate(invalid="ignore"):
        exceed = (t_perm >= thr[None]).sum(0).astype(np.uint32)
    live = ~np.isnan(thr)[None] & ~np.isnan(t_perm)
    max_t = np.where(live, t_perm, 0.0).max(1)
    return exceed, max_t


def _cls(snps):
    return np.asarray([{"X": 1, "Y": 2, "MT": 3}.get(s.chromosome, 0) for s in snps])


# ------------------------------------------------------------------------------------------------------------- CPU
def test_algorithm_s_selects_exactly_ncase_uniformly():
    """Exactly ncase cases in every permutation, for every ncase; at N = 7, ncase = 3 the inclusion frequencies and the
    frequencies of all 35 subsets pass a chi-square test of uniformity over 20 000 permutations."""
    from scipy.stats import chi2 as chi2_dist
    for n, ncase in ((1, 0), (1, 1), (5, 2), (33, 1), (33, 32), (100, 50)):
        c = perm_masks_np(42, n, ncase, 3, 50)
        assert (c.sum(1) == ncase).all()
    P = 20000
    c = perm_masks_np(7, 7, 3, 0, P)
    inc = c.sum(0)
    e = P * 3 / 7
    assert chi2_dist.sf(((inc - e) ** 2 / e).sum(), 6) > 1e-4
    keys = (c.astype(np.int64) << np.arange(7)).sum(1)
    _, sub = np.unique(keys, return_counts=True)
    assert len(sub) == 35
    e = P / 35
    assert chi2_dist.sf(((sub - e) ** 2 / e).sum(), 34) > 1e-4
    assert not np.array_equal(perm_masks_np(7, 7, 3, 0, 10), perm_masks_np(8, 7, 3, 0, 10))


def test_format_mperm_matches_per_line_rendering():
    from dna_factory_b200 import mperm
    rs = np.random.RandomState(5)
    S = 200
    t = _table(S, rs)
    emp1 = rs.rand(S, 2)
    emp2 = np.maximum(emp1, rs.rand(S, 2))
    emp1[3] = emp2[3] = np.nan
    emp1[4, 1] = emp2[4, 1] = np.nan
    emp1[5] = emp2[5] = 1.0 / 1001
    g = lambda v: "NA" if math.isnan(v) else "%.4g" % v    # noqa: E731
    for test in (0, 1):
        got = mperm.mperm_bytes(t, emp1, emp2, test)
        want = "".join("%4s %12s %12s %12s\n" % (CHR_CODE.get(t.chrom_labels[t.chrom_idx[r]], t.chrom_labels[t.chrom_idx[r]]),
                                                 "rs%d" % t.ids[r], g(emp1[r, test]), g(emp2[r, test])) for r in range(S))
        assert got == mperm.MPERM_HEADER + want.encode()
    lines = [ln.split() for ln in mperm.mperm_bytes(t, emp1, emp2, 1).decode().splitlines()]
    assert lines[0] == ["CHR", "SNP", "EMP1", "EMP2"]
    assert lines[1 + 4][2:] == ["NA", "NA"] and lines[1 + 5][2] == "0.000999"
    assert mperm.mperm_bytes(t.take(np.arange(0)), np.zeros((0, 2)), np.zeros((0, 2)), 0) == mperm.MPERM_HEADER


def test_empirical_p_and_threshold():
    from dna_factory_b200 import mperm
    t_obs = np.asarray([[10.0, np.nan], [2.0, 3.0], [0.0, 50.0], [np.nan, np.nan]])
    exceed = np.asarray([[0, 0], [3, 2], [9, 0], [0, 0]], np.uint32)
    max_t = np.asarray([[12.0, 4.0], [9.0, 3.0 * (1 - 1e-7)], [10.0 * (1 - 5e-8), 2.0], [1.0, 8.0]] + [[5.0, 5.0]] * 5)
    emp1, emp2 = mperm.empirical(t_obs, exceed, max_t)
    assert emp1[0, 0] == 1 / 10 and emp1[1, 0] == 4 / 10 and emp1[2, 0] == 1.0 and emp1[1, 1] == 3 / 10
    assert emp2[0, 0] == 3 / 10               # 12 and the tie at 10 (1 - 5e-8)
    assert emp2[1, 1] == 9 / 10               # 4, the tie at 3 (1 - 1e-7), 8 and five 5s
    assert emp2[2, 1] == 1 / 10 and emp2[2, 0] == 1.0
    assert np.isnan(emp1[0, 1]) and np.isnan(emp2[3]).all() and np.isnan(emp1[3]).all()
    assert list(mperm.threshold(max_t)) == [12.0, 8.0]
    assert list(mperm.threshold(np.arange(40.0).reshape(20, 2))) == [36.0, 37.0]   # ceil(0.95 * 20) = 19th smallest


def test_deleterious_mperm_report_text():
    from dna_factory_b200 import mperm
    from dna_factory_b200.pop_factory import DeleteriousGroup
    rs = np.random.RandomState(3)
    S = 30
    t = _table(S, rs, labels=("1", "2"))
    t_obs = np.full((S, 2), 1.0)
    t_obs[4] = [60.0, 400.0]
    t_obs[5] = [3.0, np.nan]
    exceed = np.full((S, 2), 500, np.uint32)
    exceed[4] = [0, 0]
    exceed[5] = [40, 0]
    max_t = np.stack([np.linspace(1, 50, 999), np.linspace(2, 100, 999)], 1)
    g1 = DeleteriousGroup("g1", 1)
    g1.deleterious = {int(t.ids[4]): 1, int(t.ids[5]): 0.5, 999: 0.2}
    g2 = DeleteriousGroup.from_json(json.dumps({"name": "g2", "population_weight": 1, "deleterious": {str(t.ids[4]): 1}}))
    orow = np.asarray([4, 4, 5], np.uint64)
    text, summary = mperm.deleterious_mperm_report(t, {"g1": g1, "g2": g2}, t_obs, exceed, max_t, orow)
    lines = [ln.split("\t") for ln in text.decode().splitlines()]
    assert tuple(lines[0]) == mperm.REPORT_COLUMNS and len(lines) == 5
    assert lines[1][2:] == [t.chrom_labels[t.chrom_idx[4]], "%d" % t.position[4], "1", "2", "60", "0.001", "0.001", "400",
                            "0.001", "0.001"]
    assert lines[2][5:] == ["1", "3", "0.041", "0.959", "NA", "NA", "NA"]   # 958 maxima of 999 reach 3
    assert lines[3] == ["g1", "rs999", "NA", "NA", "0.2", "0"] + ["NA"] * 6
    assert lines[4][:2] == ["g2", "rs%d" % t.ids[4]] and lines[4][5] == "2"
    thr = mperm.threshold(max_t)
    assert summary == ("2 of 4 planted deleterious SNPs have EMP2 < 0.05 under REC and 2 under ALLELIC (999 permutations); "
                       "genome-wide 5%% threshold: CHISQ %.4g (P %.3g) under REC and CHISQ %.4g (P %.3g) under ALLELIC, "
                       "Bonferroni P < 0.05 / 30 = 0.00167" % (thr[1], math.erfc(math.sqrt(thr[1] / 2)), thr[0],
                                                                math.erfc(math.sqrt(thr[0] / 2))))


def test_mperm_flag_parses():
    from dna_factory_b200 import pop_factory
    assert pop_factory.parse_cmd_args(["-s", "3", "-c", "4", "--mperm", "200"]).mperm == 200
    assert pop_factory.parse_cmd_args(["-s", "3", "-c", "4"]).mperm is None


MULTI = b'{"id": 9001, "chromosome": "1", "position": 7000000, "tuples": {"A": 0.5, "C": 0.8, "G": 1.0}}\n'
NON_COLUMN = b'{"id": 9002, "chromosome": "1", "position": 7000001, "tuples": {"AT": 0.9, "C": 1.0}}\n'


@pytest.mark.parametrize("sizes,extra,n,match", [
    (("-s", "5", "-c", "4"), MULTI, "100", "--mperm: SNP rs9001"),
    (("-s", "5", "-c", "4"), NON_COLUMN, "100", "--mperm needs SNP records that fit the column form"),
    (("-s", "0", "-c", "4"), None, "100", "--mperm needs cases and controls"),
    (("-s", "5", "-c", "0"), None, "100", "--mperm needs cases and controls"),
    (("-s", "5", "-c", "4"), None, "0", "--mperm needs at least 1 permutation")])
def test_mperm_refusals_before_any_file(tmp_path, sizes, extra, n, match):
    from dna_factory_b200 import pop_factory
    snps_gz = _snps_gz(tmp_path, extra)
    out = tmp_path / "out"
    random.seed(1)
    with pytest.raises(ValueError, match=match):
        pop_factory.main(list(sizes) + ["--snps_file", str(snps_gz), "-p",
                                        os.path.join(GOLDEN, "cli_small", "deleterious_config.yml"), "--outdir", str(out),
                                        "--seed", "7", "--mperm", n])
    for name in ("population.vcf.gz", "population.fam", "population.assoc.mperm", "population.model.rec.mperm"):
        assert not (out / name).exists()


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 15, 16, 17, 31, 33, 1003, 20000])
def test_perm_case_masks_match_algorithm_s(n):
    """dnaf_perm_case_masks bit for bit against the numpy restatement, for ncase = 1, N - 1 and about N / 2 and a
    nonzero first permutation; the (male, female) counts match the sex vector."""
    from dna_factory_b200 import _native
    rs = np.random.RandomState(n)
    sex = rs.randint(1, 3, n).astype(np.uint8)
    seed = 0x1234567890AB + n
    n_perm = 40 if n <= 1003 else 6
    with _native.Engine(0) as eng:
        for ncase in sorted({1, max(n - 1, 0), n // 2}):
            ctl = np.ones(n, np.uint8)
            ctl[rs.permutation(n)[:ncase]] = 0
            eng.set_samples(sex, ctl)
            for first in (0, 1000003):
                masks, sexc = eng.perm_case_masks(seed, first, n_perm)
                want = perm_masks_np(seed, n, ncase, first, n_perm)
                assert np.array_equal(masks, pack(want)), (n, ncase, first)
                male = sex == 1
                assert np.array_equal(sexc, np.stack([(want & male).sum(1), (want & ~male).sum(1)], 1))
            part = eng.perm_case_masks(seed, first + 7, 3)[0]
            assert np.array_equal(part, eng.perm_case_masks(seed, first, 10)[0][7:])


def _mperm_case(n):
    case = _dense_case(n, seed=n)
    sex = np.asarray([s.sex for s in case.samples])
    return case, sex == 1, _cls(case.snps)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [17, 1003, 4099])
def test_mperm_matches_brute_force(n):
    """t_obs, exceed and max_t against the numpy brute force over dnaf_genotypes and the restated permutations: all four
    chromosome classes, dense forced minors, a nonzero row base, many passes, N_perm across the 64-permutation tile."""
    from dna_factory_b200 import _native, assoc
    case, male, cls = _mperm_case(n)
    S = len(case.snps)
    eng = _geno_engine(case, chunk=4096, row_base=91 + n)
    g = eng.genotypes(0, S, case.seed)
    counts = geno_from_genotypes(g, [bool(s.is_control) for s in case.samples])
    ncase = sum(not s.is_control for s in case.samples)
    for n_perm in (1, 31, 64, 257):
        t_obs, exceed, max_t, st = eng.mperm_stats(0, S, case.seed, n_perm)
        assert st["rows"] == S and st["kernel_launches"] > 4    # several passes
        # observed: ALLELIC is the .assoc CHISQ of the same counts, REC the no-cell-rule 2x2
        c = counts.astype(np.float64)
        alt_a, alt_u = 2 * c[:, 2] + c[:, 1] + c[:, 4], 2 * c[:, 7] + c[:, 6] + c[:, 9]
        want_a = assoc.chisq(np.stack([alt_a, 2 * c[:, 0] + c[:, 3], alt_u, 2 * c[:, 5] + c[:, 8]], 1))
        want_r = chi2(c[:, 2], c[:, 0] - c[:, 2], c[:, 7], c[:, 5] - c[:, 7])
        for got, want in ((t_obs[:, 0], want_a), (t_obs[:, 1], want_r)):
            assert np.array_equal(np.isnan(got), np.isnan(want))
            ok = ~np.isnan(want)
            assert np.allclose(got[ok], want[ok], rtol=1e-12, atol=0)
        assert np.isnan(t_obs[cls >= 2, 1]).all()
        perms = perm_masks_np(case.seed, n, ncase, 0, n_perm)
        t_perm = stats_np(g, cls, perms, male)
        thr = t_obs * (1 - TIE)
        with np.errstate(invalid="ignore", divide="ignore"):
            rel = np.abs(t_perm - thr[None]) / thr[None]
        assert not (rel < 1e-12).any()                        # exact comparison is well posed
        want_ex, want_max = brute_force(t_obs, t_perm)
        assert np.array_equal(exceed, want_ex), n_perm
        assert np.array_equal(max_t, want_max), n_perm
        assert (exceed[np.isnan(t_obs)] == 0).all()
    eng.close()


@pytest.mark.gpu
def test_mperm_composes_over_row_ranges_and_repeats():
    """Two calls over row halves give the concatenated t_obs / exceed and the elementwise-max max_t of one whole call;
    a repeated call is bit-identical; the device-only call runs the same launches."""
    case = synth_case(2500, 300, seed=8, chroms=["1", "X", "Y", "MT", "5"], n_del=30)
    S = len(case.snps)
    eng = _geno_engine(case, chunk=1 << 16)
    whole = eng.mperm_stats(0, S, case.seed, 100)
    again = eng.mperm(0, S, case.seed, 100)
    for a, b in zip(whole[:3], again):
        assert np.array_equal(a, b, equal_nan=True)
    h = S // 2 + 3
    lo, hi = eng.mperm(0, h, case.seed, 100), eng.mperm(h, S, case.seed, 100)
    assert np.array_equal(np.concatenate([lo[0], hi[0]]), whole[0], equal_nan=True)
    assert np.array_equal(np.concatenate([lo[1], hi[1]]), whole[1])
    assert np.array_equal(np.maximum(lo[2], hi[2]), whole[2])
    dev = eng.mperm_device(0, S, case.seed, 100)
    assert {k: dev[k] for k in ("rows", "calls", "kernel_launches")} == \
        {k: whole[3][k] for k in ("rows", "calls", "kernel_launches")}
    assert (whole[2] > 0).all() and (whole[1] <= 100).all()
    eng.close()


@pytest.mark.gpu
def test_mperm_refusals():
    """A K > 2 row is refused with DNAF_E_INPUT before any launch; n_perm == 0 and a population without controls
    with DNAF_E_ARG."""
    import ctypes
    from dna_factory_b200 import _native
    case = synth_case(40, 20, seed=5, exotic=True)
    eng = _geno_engine(case)
    k = [len(s.tuples) for s in case.snps]
    bad = next(r for r, kr in enumerate(k) if kr > 2)
    t = np.full((20, 2), 7.0)
    ex = np.full((20, 2), 0xABABABAB, np.uint32)
    mx = np.full((10, 2), 7.0)
    st = _native.Stats()
    f64p = ctypes.POINTER(ctypes.c_double)
    rc = eng._lib.dnaf_mperm(eng._h, 0, 20, case.seed, 10, t.ctypes.data_as(f64p),
                             ex.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), mx.ctypes.data_as(f64p), ctypes.byref(st))
    assert rc == _native.E_INPUT
    assert ("row %d " % bad) in eng._lib.dnaf_last_error(eng._h).decode()
    assert (t == 7.0).all() and (ex == 0xABABABAB).all() and (mx == 7.0).all() and st.kernel_launches == 0
    with pytest.raises(_native.DnafError) as e:
        eng.mperm_device(0, 20, case.seed, 10)
    assert e.value.code == _native.E_INPUT
    a, b = _runs(k)[0]
    with pytest.raises(_native.DnafError) as e:
        eng.mperm(a, b, case.seed, 0)
    assert e.value.code == _native.E_ARG
    assert eng.mperm(a, b, case.seed, 5)[0].shape == (b - a, 2)      # the context is still usable
    eng.set_samples(np.ones(40, np.uint8), np.ones(40, np.uint8))
    with pytest.raises(_native.DnafError) as e:
        eng.mperm(a, b, case.seed, 5)
    assert e.value.code == _native.E_ARG
    eng.close()


def _emp_np(t_obs, t_perm):
    exceed, max_t = brute_force(t_obs, t_perm)
    from dna_factory_b200 import mperm
    return mperm.empirical(t_obs, exceed, max_t)


@pytest.mark.gpu
def test_cli_mperm_matches_its_own_vcf(tmp_path, monkeypatch):
    """--mperm 200 on the pinned reference CLI run: both files hold every SNP with 1/(N+1) <= EMP1 <= EMP2 <= 1 on
    every tested row, and equal EMP1 / EMP2 recomputed in numpy from the run's own population.vcf.gz and the restated
    permutations; --gpus 2 writes the same files; every other file is byte-identical to the run without --mperm."""
    from dna_factory_b200 import mperm
    from dna_factory_b200.snp import SnpTable
    from tests.test_model import geno_from_text
    out = tmp_path / "m1"
    _cli_small(monkeypatch, out, ["--mperm", "200"])
    table = SnpTable.read_json_gz_table(str(out / "snps.json.gz"))
    vcf = gzip.decompress((out / "population.vcf.gz").read_bytes())
    body = [ln for ln in vcf.split(b"\n")[:-1] if not ln.startswith(b"#")]
    fam = [ln.split("\t") for ln in (out / "population.fam").read_text().splitlines()]
    ctl = np.asarray([f[5] == "1" for f in fam])
    male = np.asarray([f[4] == "1" for f in fam])
    # the genotype export layout from the VCF text: 'a/b' diploid, 'a' haploid, '.' nothing
    g = np.full((len(body), len(fam), 2), 0xFF, np.uint8)
    for r, ln in enumerate(body):
        for i, cell in enumerate(ln.split(b"\t")[9:]):
            if cell != b".":
                for s, al in enumerate(cell.split(b"/")):
                    g[r, i, s] = int(al)
    counts = geno_from_text(b"".join(ln + b"\n" for ln in body), ctl)
    assert np.array_equal(geno_from_genotypes(g, ctl), counts)
    cls = np.asarray([{"X": 1, "Y": 2, "MT": 3}.get(table.chrom_labels[c], 0) for c in table.chrom_idx])
    c = counts.astype(np.float64)
    alt_a, alt_u = 2 * c[:, 2] + c[:, 1] + c[:, 4], 2 * c[:, 7] + c[:, 6] + c[:, 9]
    t_obs = np.stack([chi2(alt_a, 2 * c[:, 0] + c[:, 3] - alt_a, alt_u, 2 * c[:, 5] + c[:, 8] - alt_u),
                      chi2(c[:, 2], c[:, 0] - c[:, 2], c[:, 7], c[:, 5] - c[:, 7])], 1)
    meta = json.load(open(os.path.join(GOLDEN, "cli_small", "meta.json")))
    perms = perm_masks_np(meta["philox_seed"], len(fam), int((~ctl).sum()), 0, 200)
    emp1, emp2 = _emp_np(t_obs, stats_np(g, cls, perms, male))
    for t, name in enumerate(("population.assoc.mperm", "population.model.rec.mperm")):
        text = (out / name).read_bytes()
        assert text == mperm.mperm_bytes(table, emp1, emp2, t), name
        rows = [ln.split() for ln in text.decode().splitlines()[1:]]
        assert len(rows) == len(table)
        for r in rows:
            if r[2] != "NA":
                assert 1 / 201 - 1e-12 <= float(r[2]) <= float(r[3]) <= 1
    report = (out / "deleterious_mperm.txt").read_text().splitlines()
    assert len(report) == 1 + sum(len(json.loads(ln)["deleterious"]) for ln in open(out / "deleterious.json"))
    _cli_small(monkeypatch, tmp_path / "m2", ["--mperm", "200", "--gpus", "2"])
    for name in ("population.assoc.mperm", "population.model.rec.mperm", "deleterious_mperm.txt"):
        assert (tmp_path / "m2" / name).read_bytes() == (out / name).read_bytes(), name
    _cli_small(monkeypatch, tmp_path / "n", [])
    names = sorted(os.listdir(tmp_path / "n"))
    assert "population.assoc.mperm" not in names
    for name in names:
        got, ref = (tmp_path / "n" / name).read_bytes(), (out / name).read_bytes()
        if name.endswith(".json.gz"):      # gzip's MTIME field (bytes 4-7) holds the wall clock of each run
            got, ref = got[:4] + got[8:], ref[:4] + ref[8:]
        assert got == ref, name


@pytest.mark.gpu
def test_cli_planted_snps_under_mperm_rec(tmp_path, monkeypatch, capsys):
    """Planted SNPs with hundreds of forced 1/1 cases beat every permutation's maximum under REC: EMP2_REC = 1/(N+1)."""
    import re
    from dna_factory_b200 import pop_factory
    cfg = tmp_path / "one_group.yml"
    cfg.write_text("planted:\n  mutation_weights:\n  - 1\n  - 1\n  - 1\n  num_instances: 1\n  population_weight: 1\n"
                   "  max_minor_allele_freq: 0.1\n")
    out = tmp_path / "out"
    _fixed_clock(monkeypatch)
    random.seed(99)
    pop_factory.main(["-s", "2000", "-c", "2000", "-x", "3000", "-f", "0.01", "-p", str(cfg), "--outdir", str(out),
                      "--seed", "2024", "--mperm", "200"])
    printed = capsys.readouterr().out
    assert re.search(r"3 of 3 planted deleterious SNPs have EMP2 < 0.05 under REC and \d under ALLELIC \(200 "
                     r"permutations\); genome-wide 5% threshold: CHISQ \S+ \(P \S+\) under REC", printed), printed
    lines = [ln.split("\t") for ln in (out / "deleterious_mperm.txt").read_text().splitlines()]
    col = {name: i for i, name in enumerate(lines[0])}
    assert len(lines) == 4
    for ln in lines[1:]:
        assert int(ln[col["FORCED"]]) >= 100
        assert ln[col["EMP2_REC"]] == "%.4g" % (1 / 201) and ln[col["EMP1_REC"]] == "%.4g" % (1 / 201)
