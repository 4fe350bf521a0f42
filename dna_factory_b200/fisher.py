"""Fisher's exact case/control tests (pop_factory --fisher) and the report on the planted deleterious SNPs under them.

The genotype counts and log10 of the exact P come from the GPU (Engine.genotype_tests, kernels k_geno and k_fisher);
this module turns them into
  population.assoc.fisher   the allelic test per SNP in the columns of PLINK 1.9's plink.assoc.fisher
                            (CHR SNP BP A1 F_A F_U A2 P OR), A1 = ALT as in the .bim
  population.model.fisher   five tests per SNP in the columns of plink --model fisher (CHR SNP A1 A2 TEST AFF UNAFF P;
                            GENO, TREND, ALLELIC, DOM, REC)
  deleterious_fisher.txt    one line per (deleterious group, planted SNP): its genotype counts, the Fisher P of
                            ALLELIC, GENO, DOM and REC, and its rank by Fisher REC and ALLELIC
Tests (also dnaf_fisher_exact): GENO is the 2x3 table of diploid genotypes, ALLELIC the ALT / REF allele table with
haploid cells (the .assoc counts), DOM n11+n12 vs n22, REC n11 vs n12+n22; no cell rule.  TREND keeps its asymptotic
chi-square P, as plink --model fisher does.  P prints "%.4g", 0 where it is below the double range, NA where a margin is
0.  Ranks use log10 P, which never underflows, so they stay exact where P prints 0.
"""
import math

import numpy as np

from . import _native
from .assoc import planted_rows, rank_of
from .model import genotypes, model_chisq

ASSOC_FISHER_COLUMNS = ("CHR", "SNP", "BP", "A1", "F_A", "F_U", "A2", "P", "OR")
ASSOC_FISHER_HEADER = ("%4s %12s %10s %4s %8s %8s %4s %12s %12s\n" % ASSOC_FISHER_COLUMNS).encode()
MODEL_FISHER_COLUMNS = ("CHR", "SNP", "A1", "A2", "TEST", "AFF", "UNAFF", "P")
MODEL_FISHER_HEADER = ("%4s %12s %4s %4s %8s %14s %14s %12s\n" % MODEL_FISHER_COLUMNS).encode()
REPORT_COLUMNS = ("GROUP", "SNP", "CHR", "BP", "WEIGHT", "FORCED", "AFF", "UNAFF", "P_ALLELIC", "P_GENO", "P_DOM", "P_REC",
                  "LOG10P_ALLELIC", "LOG10P_REC", "RANK_REC", "RANK_ALLELIC")


def _inputs(table, counts, log10p):
    counts = np.asarray(counts, np.uint32).reshape(-1, 10)
    log10p = np.asarray(log10p, np.float64).reshape(-1, 4)
    if len(counts) != len(table) or len(log10p) != len(table):
        raise ValueError("%d rows of counts and %d of log10 P for a table of %d SNPs" % (len(counts), len(log10p), len(table)))
    return counts, log10p


def assoc_fisher_bytes(table, counts, log10p):
    """population.assoc.fisher text (header line + one line per row) of a SnpTable, its uint32[rows, 10] genotype counts
    and float64[rows, 4] Fisher log10 P."""
    counts, log10p = _inputs(table, counts, log10p)
    return ASSOC_FISHER_HEADER + _native.format_assoc_fisher(table.ids, table.chrom_idx, table.chrom_labels, table.position,
                                                             table.n_alleles, table.nts, counts, log10p)


def model_fisher_bytes(table, counts, log10p):
    """population.model.fisher text (header line + five lines per row) of the same inputs."""
    counts, log10p = _inputs(table, counts, log10p)
    return MODEL_FISHER_HEADER + _native.format_model_fisher(table.ids, table.chrom_idx, table.chrom_labels, table.n_alleles,
                                                             table.nts, counts, log10p)


def _p(l):
    return "NA" if math.isnan(l) else "%.4g" % (10.0 ** l)


def _l(l):
    return "NA" if math.isnan(l) else "%.6g" % l


def deleterious_fisher_report(table, groups, counts, log10p, orow):
    """deleterious_fisher.txt text and its summary.

    One line per (group, planted SNP) (assoc.planted_rows: FORCED, and FORCED 0 for the string keys of a replay):
    AFF / UNAFF are the n11/n12/n22 genotype counts of cases and controls, then the Fisher P of ALLELIC, GENO, DOM and
    REC, log10 P of ALLELIC and REC, and the rank by Fisher REC and ALLELIC among all rows (smaller log10 P first; NA
    ranks behind every tested row).  The summary counts the planted SNPs that pass P < 0.05 / S under Fisher REC and
    under Fisher ALLELIC, and the REC passes whose chi-square REC test is NA by the cell rule (a genotype cell below 5).
    -> (text bytes, summary str)."""
    counts, log10p = _inputs(table, counts, log10p)
    S = len(table)
    g = genotypes(counts).astype(np.int64)
    no_chisq_rec = np.isnan(model_chisq(counts)[:, 4])
    tested = {t: np.sort(-log10p[:, t][~np.isnan(log10p[:, t])]) for t in (1, 3)}
    alpha = 0.05 / max(S, 1)
    lines = ["\t".join(REPORT_COLUMNS)]
    planted = hits_rec = hits_allelic = rec_no_chisq = 0
    for name, snp_id, weight, r, forced in planted_rows(table, groups, orow):
        planted += 1
        if r is None:
            lines.append("\t".join([name, "rs%d" % snp_id, "NA", "NA", "%g" % weight, "0"] + ["NA"] * 10))
            continue
        l = [float(v) for v in log10p[r]]
        rec = not math.isnan(l[3]) and l[3] < math.log10(alpha)
        hits_rec += rec
        hits_allelic += not math.isnan(l[1]) and l[1] < math.log10(alpha)
        rec_no_chisq += rec and bool(no_chisq_rec[r])
        lines.append("\t".join([name, "rs%d" % snp_id, table.chrom_labels[table.chrom_idx[r]], "%d" % table.position[r],
                                "%g" % weight, "%d" % forced, "%d/%d/%d" % tuple(g[r, 0]), "%d/%d/%d" % tuple(g[r, 1]),
                                _p(l[1]), _p(l[0]), _p(l[2]), _p(l[3]), _l(l[1]), _l(l[3])] +
                               ["%d" % rank_of(tested[t], None if math.isnan(l[t]) else -l[t]) for t in (3, 1)]))
    summary = ("%d of %d planted deleterious SNPs pass P < 0.05 / %d = %.3g under Fisher REC and %d under Fisher ALLELIC; "
               "%d of the REC passes have no chi-square REC test (a genotype cell below 5)" % (
                   hits_rec, planted, S, alpha, hits_allelic, rec_no_chisq))
    return ("\n".join(lines) + "\n").encode(), summary
