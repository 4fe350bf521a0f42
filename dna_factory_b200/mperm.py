"""max(T) permutation tests of ALLELIC and REC (pop_factory --mperm N) and the report on the planted deleterious SNPs
under them.

The observed statistics, the per-row exceedance counts and the per-permutation maxima come from the GPU
(Engine.mperm, kernels k_perm_masks, k_geno, k_mperm_planes and k_mperm); this module turns them into
  population.assoc.mperm       CHR SNP EMP1 EMP2 of the ALLELIC test (the .assoc statistic), the columns of PLINK 1.9's
                               plink.assoc.mperm
  population.model.rec.mperm   the same for REC (2x2 Pearson n11 | n12 + n22 on diploid cells, no cell rule)
  deleterious_mperm.txt        one line per (deleterious group, planted SNP): CHISQ, EMP1 and EMP2 of ALLELIC and REC
Permutation p is a uniformly random subset of exactly ncase samples (Algorithm S over a Philox stream of the run's
seed; include/dnaf_b200.h, dnaf_perm_case_masks).  With N permutations, T_obs the observed statistic of a row and T_p
its value under permutation p, T_p counts as at least T_obs when T_p >= T_obs (1 - 1e-7), and
  EMP1 = (#{p : T_p >= T_obs} + 1) / (N + 1)      pointwise
  EMP2 = (#{p : max_rows T_p >= T_obs} + 1) / (N + 1)      family-wise (max(T))
EMP prints "%.4g", NA where the row has no test (a zero denominator; Y and MT rows have no REC).
"""
import math

import numpy as np

from . import _native
from .assoc import planted_rows

TIE = 1e-7   # relative tie tolerance (kHweTie)
TESTS = ("ALLELIC", "REC")
MPERM_COLUMNS = ("CHR", "SNP", "EMP1", "EMP2")
MPERM_HEADER = ("%4s %12s %12s %12s\n" % MPERM_COLUMNS).encode()
REPORT_COLUMNS = ("GROUP", "SNP", "CHR", "BP", "WEIGHT", "FORCED", "CHISQ_ALLELIC", "EMP1_ALLELIC", "EMP2_ALLELIC",
                  "CHISQ_REC", "EMP1_REC", "EMP2_REC")


def empirical(t_obs, exceed, max_t):
    """(EMP1, EMP2), each float64[rows, 2] (ALLELIC, REC), of the observed statistics float64[rows, 2], their
    exceedance counts uint32[rows, 2] and the per-permutation maxima float64[n_perm, 2]; NaN where T_obs is NaN."""
    t_obs = np.asarray(t_obs, np.float64).reshape(-1, 2)
    exceed = np.asarray(exceed, np.float64).reshape(-1, 2)
    max_t = np.asarray(max_t, np.float64).reshape(-1, 2)
    if len(exceed) != len(t_obs):
        raise ValueError("%d rows of exceedances for %d rows of statistics" % (len(exceed), len(t_obs)))
    n = len(max_t)
    thr = t_obs * (1.0 - TIE)
    r2 = np.stack([n - np.searchsorted(np.sort(max_t[:, t]), thr[:, t], side="left") for t in range(2)], 1)
    na = np.isnan(t_obs)
    emp1 = np.where(na, np.nan, (exceed + 1.0) / (n + 1.0))
    emp2 = np.where(na, np.nan, (r2 + 1.0) / (n + 1.0))
    return emp1, emp2


def threshold(max_t):
    """The permutation genome-wide 5 % threshold of each test: the ceil(0.95 N)-th smallest per-permutation maximum,
    float64[2] (ALLELIC, REC)."""
    max_t = np.asarray(max_t, np.float64).reshape(-1, 2)
    k = max(1, math.ceil(0.95 * len(max_t)))
    return np.sort(max_t, 0)[k - 1]


def mperm_bytes(table, emp1, emp2, test):
    """population.assoc.mperm (test 0, ALLELIC) or population.model.rec.mperm (test 1, REC) text: header line + one
    line per row."""
    emp = np.stack([np.asarray(emp1, np.float64).reshape(-1, 2)[:, test], np.asarray(emp2, np.float64).reshape(-1, 2)[:, test]], 1)
    if len(emp) != len(table):
        raise ValueError("%d rows of EMP for a table of %d SNPs" % (len(emp), len(table)))
    return MPERM_HEADER + _native.format_mperm(table.ids, table.chrom_idx, table.chrom_labels, emp)


def _g(v):
    return "NA" if math.isnan(v) else "%.4g" % v


def _p1(x):
    return math.erfc(math.sqrt(x / 2.0))


def deleterious_mperm_report(table, groups, t_obs, exceed, max_t, orow):
    """deleterious_mperm.txt text and its summary.

    One line per (group, planted SNP) (assoc.planted_rows: FORCED, and FORCED 0 for the string keys of a replay):
    CHISQ, EMP1 and EMP2 of ALLELIC, then of REC.  The summary counts the planted SNPs with EMP2 < 0.05 under REC and
    under ALLELIC and gives the permutation genome-wide 5 % threshold of each test (threshold(), as a CHISQ and as its
    nominal 1-df P) next to Bonferroni's 0.05 / S.
    -> (text bytes, summary str)."""
    t_obs = np.asarray(t_obs, np.float64).reshape(-1, 2)
    if len(t_obs) != len(table):
        raise ValueError("%d rows of statistics for a table of %d SNPs" % (len(t_obs), len(table)))
    emp1, emp2 = empirical(t_obs, exceed, max_t)
    S, n = len(table), len(np.asarray(max_t).reshape(-1, 2))
    lines = ["\t".join(REPORT_COLUMNS)]
    planted, hits = 0, [0, 0]
    for name, snp_id, weight, r, forced in planted_rows(table, groups, orow):
        planted += 1
        if r is None:
            lines.append("\t".join([name, "rs%d" % snp_id, "NA", "NA", "%g" % weight, "0"] + ["NA"] * 6))
            continue
        cols = []
        for t in range(2):
            hits[t] += bool(emp2[r, t] < 0.05)
            cols += [_g(t_obs[r, t]), _g(emp1[r, t]), _g(emp2[r, t])]
        lines.append("\t".join([name, "rs%d" % snp_id, table.chrom_labels[table.chrom_idx[r]], "%d" % table.position[r],
                                "%g" % weight, "%d" % forced] + cols))
    thr = threshold(max_t)
    summary = ("%d of %d planted deleterious SNPs have EMP2 < 0.05 under REC and %d under ALLELIC (%d permutations); "
               "genome-wide 5%% threshold: CHISQ %.4g (P %.3g) under REC and CHISQ %.4g (P %.3g) under ALLELIC, "
               "Bonferroni P < 0.05 / %d = %.3g" % (hits[1], planted, hits[0], n, thr[1], _p1(thr[1]), thr[0], _p1(thr[0]),
                                                      S, 0.05 / max(S, 1)))
    return ("\n".join(lines) + "\n").encode(), summary
