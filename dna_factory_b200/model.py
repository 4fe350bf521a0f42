"""Genotypic case/control tests (pop_factory --model), Hardy-Weinberg exact tests (pop_factory --hardy) and the report
on the planted deleterious SNPs under the genotypic tests.

The genotype counts and the exact-test P come from the GPU (Engine.genotype_counts, kernels k_geno and k_hwe); this
module turns them into
  population.model          five tests per SNP in the column names and order of PLINK 1.9's plink.model
                            (CHR SNP A1 A2 TEST AFF UNAFF CHISQ DF P; GENO, TREND, ALLELIC, DOM, REC), A1 = ALT
  population.hwe            three exact tests per SNP in the columns of plink.hwe (CHR SNP TEST A1 A2 GENO O(HET)
                            E(HET) P; ALL, AFF, UNAFF)
  deleterious_model.txt     one line per (deleterious group, planted SNP): its genotype counts, the P of every test,
                            its rank by REC and by ALLELIC CHISQ, and its Hardy-Weinberg P
Statistics (also dnaf_format_model): ALLELIC is the .assoc test on the allele counts (haploid cells included); TREND
the Cochran-Armitage trend test on diploid cells; GENO the 2x3 Pearson test (2 df); DOM (n11+n12 vs n22) and REC (n11
vs n12+n22) 2x2 Pearson tests; no continuity correction; GENO, DOM and REC are NA when any of the six genotype cells is
below 5 (PLINK's --cell 5); a zero denominator is NA.
"""
import math

import numpy as np

from . import _native
from .assoc import planted_rows, rank_of

MODEL_COLUMNS = ("CHR", "SNP", "A1", "A2", "TEST", "AFF", "UNAFF", "CHISQ", "DF", "P")
MODEL_HEADER = ("%4s %12s %4s %4s %8s %14s %14s %12s %4s %12s\n" % MODEL_COLUMNS).encode()
HWE_COLUMNS = ("CHR", "SNP", "TEST", "A1", "A2", "GENO", "O(HET)", "E(HET)", "P")
HWE_HEADER = ("%4s %12s %8s %4s %4s %20s %8s %8s %12s\n" % HWE_COLUMNS).encode()
DF = (2, 1, 1, 1, 1)
REPORT_COLUMNS = ("GROUP", "SNP", "CHR", "BP", "WEIGHT", "FORCED", "AFF", "UNAFF", "P_ALLELIC", "P_TREND", "P_GENO", "P_DOM",
                  "P_REC", "RANK_REC", "RANK_ALLELIC", "HWE_ALL", "HWE_AFF", "HWE_UNAFF")
HWE_STRICT = 1e-6


def _counts(counts, n):
    counts = np.asarray(counts, np.uint32).reshape(-1, 10)
    if len(counts) != n:
        raise ValueError("%d rows of counts for a table of %d SNPs" % (len(counts), n))
    return counts


def model_bytes(table, counts):
    """population.model text (header line + five lines per row) of a SnpTable and its uint32[rows, 10] counts."""
    counts = _counts(counts, len(table))
    return MODEL_HEADER + _native.format_model(table.ids, table.chrom_idx, table.chrom_labels, table.n_alleles, table.nts,
                                               counts)


def hardy_bytes(table, counts, hwe_p):
    """population.hwe text (header line + three lines per row) of a SnpTable, its counts and float64[rows, 3] P."""
    counts = _counts(counts, len(table))
    return HWE_HEADER + _native.format_hardy(table.ids, table.chrom_idx, table.chrom_labels, table.n_alleles, table.nts,
                                             counts, hwe_p)


def genotypes(counts):
    """float64[rows, 2, 3]: (n11, n12, n22) = ALT/ALT, het, REF/REF diploid counts of the cases and of the controls."""
    c = np.asarray(counts, np.float64).reshape(-1, 10)
    return np.stack([np.stack([c[:, 2 + 5 * g], c[:, 1 + 5 * g], c[:, 5 * g] - c[:, 1 + 5 * g] - c[:, 2 + 5 * g]], 1)
                     for g in (0, 1)], 1)


def model_chisq(counts):
    """float64[rows, 5]: CHISQ of GENO, TREND, ALLELIC, DOM, REC per row, NaN where it is NA (the formatter's rules)."""
    c = np.asarray(counts, np.float64).reshape(-1, 10)
    g = genotypes(c)
    a11, a12, a22, u11, u12, u22 = g[:, 0, 0], g[:, 0, 1], g[:, 0, 2], g[:, 1, 0], g[:, 1, 1], g[:, 1, 2]
    alt_a, alt_u = 2 * a11 + a12 + c[:, 4], 2 * u11 + u12 + c[:, 9]
    ref_a, ref_u = 2 * c[:, 0] + c[:, 3] - alt_a, 2 * c[:, 5] + c[:, 8] - alt_u
    ok = (g >= 5).all(axis=(1, 2))
    R, S = a11 + a12 + a22, u11 + u12 + u22
    N = R + S

    def two_by_two(a, b, cc, d):
        den = (a + b) * (cc + d) * (a + cc) * (b + d)
        x = a * d - b * cc
        return np.where(den > 0, (a + b + cc + d) * x * x / np.where(den > 0, den, 1.0), np.nan)

    with np.errstate(divide="ignore", invalid="ignore"):
        geno = np.zeros(len(c))
        for a, u in ((a11, u11), (a12, u12), (a22, u22)):
            nj = a + u
            ea, eu = R * nj / N, S * nj / N
            geno = geno + (a - ea) ** 2 / ea + (u - eu) ** 2 / eu
        geno = np.where(ok & (R > 0) & (S > 0), geno, np.nan)
        sxr, sxn, sx2n = 2 * a11 + a12, 2 * (a11 + u11) + (a12 + u12), 4 * (a11 + u11) + (a12 + u12)
        den = R * S * (N * sx2n - sxn * sxn)
        t = N * sxr - R * sxn
        trend = np.where(den > 0, N * t * t / np.where(den > 0, den, 1.0), np.nan)
        allelic = two_by_two(alt_a, ref_a, alt_u, ref_u)
        dom = np.where(ok, two_by_two(a11 + a12, a22, u11 + u12, u22), np.nan)
        rec = np.where(ok, two_by_two(a11, a12 + a22, u11, u12 + u22), np.nan)
    return np.stack([geno, trend, allelic, dom, rec], 1)


def chi2_p(x, df):
    """Chi-square survival of x at 1 or 2 df; None for NA."""
    if x is None or math.isnan(x):
        return None
    return math.erfc(math.sqrt(x / 2.0)) if df == 1 else math.exp(-x / 2.0)


def _g(v):
    return "NA" if v is None or (isinstance(v, float) and math.isnan(v)) else "%.4g" % v


def deleterious_model_report(table, groups, counts, hwe_p, orow):
    """deleterious_model.txt text and its summary.

    One line per (group, planted SNP) (assoc.planted_rows: FORCED, and FORCED 0 for the string keys of a replay):
    AFF / UNAFF are the n11/n12/n22 genotype counts of cases and controls, then the P of ALLELIC, TREND, GENO, DOM and
    REC, the rank by REC CHISQ and by ALLELIC CHISQ among all rows (NA ranks behind every tested row), and the
    Hardy-Weinberg P of ALL, AFF and UNAFF.  The summary counts the planted SNPs that pass P < 0.05 / S under REC and
    under ALLELIC, those whose REC test is NA by the cell rule, and those with HWE P < 1e-6 in ALL and in UNAFF.
    -> (text bytes, summary str)."""
    counts = _counts(counts, len(table))
    hwe_p = np.asarray(hwe_p, np.float64).reshape(-1, 3)
    S = len(table)
    x2 = model_chisq(counts)
    g = genotypes(counts).astype(np.int64)
    tested = {t: np.sort(x2[:, t][~np.isnan(x2[:, t])]) for t in (2, 4)}
    alpha = 0.05 / max(S, 1)
    lines = ["\t".join(REPORT_COLUMNS)]
    planted = hits_rec = hits_allelic = rec_na = hwe_all = hwe_unaff = 0
    for name, snp_id, weight, r, forced in planted_rows(table, groups, orow):
        planted += 1
        if r is None:
            lines.append("\t".join([name, "rs%d" % snp_id, "NA", "NA", "%g" % weight, "0"] + ["NA"] * 12))
            continue
        x = [None if math.isnan(v) else float(v) for v in x2[r]]
        p = [chi2_p(v, df) for v, df in zip(x, DF)]
        hits_rec += p[4] is not None and p[4] < alpha
        hits_allelic += p[2] is not None and p[2] < alpha
        rec_na += x[4] is None and bool((g[r] < 5).any())
        hwe_all += hwe_p[r, 0] < HWE_STRICT
        hwe_unaff += hwe_p[r, 2] < HWE_STRICT
        lines.append("\t".join([name, "rs%d" % snp_id, table.chrom_labels[table.chrom_idx[r]], "%d" % table.position[r],
                                "%g" % weight, "%d" % forced, "%d/%d/%d" % tuple(g[r, 0]), "%d/%d/%d" % tuple(g[r, 1]),
                                _g(p[2]), _g(p[1]), _g(p[0]), _g(p[3]), _g(p[4]),
                                "%d" % rank_of(tested[4], x[4]), "%d" % rank_of(tested[2], x[2])] +
                               [_g(float(v)) for v in hwe_p[r]]))
    summary = ("%d of %d planted deleterious SNPs pass P < 0.05 / %d = %.3g under REC and %d under ALLELIC; "
               "%d have no REC test (a genotype cell below 5); %d have HWE P < %g in ALL and %d in UNAFF" % (
                   hits_rec, planted, S, alpha, hits_allelic, rec_na, hwe_all, HWE_STRICT, hwe_unaff))
    return ("\n".join(lines) + "\n").encode(), summary
