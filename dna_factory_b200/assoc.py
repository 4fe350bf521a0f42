"""Case/control allelic association test (pop_factory --assoc) and the report on the planted deleterious SNPs.

The allele counts come from the GPU (Engine.allele_counts, kernel k_assoc); this module turns them into
  population.assoc          the 1-df allelic test per SNP, in the column names and order of PLINK 1.9's plink.assoc
                            (CHR SNP BP A1 F_A F_U A2 CHISQ P OR), A1 = ALT and A2 = REF as in the .bim
  deleterious_assoc.txt     one line per (deleterious group, planted SNP): how strongly the scan finds it and where it
                            ranks among all SNPs
Statistics (also dnaf_format_assoc): with a / b the ALT / REF alleles in cases and c / d in controls,
F_A = a/(a+b), F_U = c/(c+d), CHISQ = n(ad-bc)^2 / ((a+b)(c+d)(a+c)(b+d)) without continuity correction,
P = erfc(sqrt(CHISQ/2)), OR = ad/(bc); NA where a denominator is 0.
"""
import math

import numpy as np

from . import _native

ASSOC_COLUMNS = ("CHR", "SNP", "BP", "A1", "F_A", "F_U", "A2", "CHISQ", "P", "OR")
ASSOC_HEADER = ("%4s %12s %10s %4s %8s %8s %4s %12s %12s %12s\n" % ASSOC_COLUMNS).encode()
REPORT_COLUMNS = ("GROUP", "SNP", "CHR", "BP", "WEIGHT", "FORCED", "F_A", "F_U", "CHISQ", "P", "OR", "RANK")


def assoc_bytes(table, counts):
    """population.assoc text (header line + one line per row) of a SnpTable and its uint32[rows, 4] counts."""
    counts = np.asarray(counts, np.uint32).reshape(-1, 4)
    if len(counts) != len(table):
        raise ValueError("%d rows of counts for a table of %d SNPs" % (len(counts), len(table)))
    return ASSOC_HEADER + _native.format_assoc(table.ids, table.chrom_idx, table.chrom_labels, table.position,
                                               table.n_alleles, table.nts, counts)


def chisq(counts):
    """float64[rows]: the allelic CHISQ of every row, NaN where it is NA (same formula and order as the formatter)."""
    c = np.asarray(counts, np.float64).reshape(-1, 4)
    a, ca, cc, cu = c[:, 0], c[:, 1], c[:, 2], c[:, 3]
    b, d = ca - a, cu - cc
    den = ca * cu * (a + cc) * (b + d)
    x = a * d - b * cc
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den > 0, (a + b + cc + d) * x * x / np.where(den > 0, den, 1.0), np.nan)


def row_stats(a, ca, c, cu):
    """(F_A, F_U, CHISQ, P, OR) of one row from its four counts; None for NA."""
    a, ca, c, cu = float(a), float(ca), float(c), float(cu)
    b, d = ca - a, cu - c
    den = ca * cu * (a + c) * (b + d)
    x2 = (a + b + c + d) * (a * d - b * c) * (a * d - b * c) / den if den > 0 else None
    return (a / ca if ca > 0 else None, c / cu if cu > 0 else None, x2,
            math.erfc(math.sqrt(x2 / 2.0)) if x2 is not None else None, a * d / (b * c) if b * c > 0 else None)


def _g(v):
    return "NA" if v is None else "%.4g" % v


def planted_rows(table, groups, orow):
    """(group name, SNP id, weight, row or None, forced) of every (group, planted SNP), in the groups' order.

    groups: {name: DeleteriousGroup}.  orow: the global row of every override pair (host.override_pairs*), so `forced`
    is the number of cases whose minor allele was forced on that row.  A key of a --deleterious_file replay is a string,
    which forces nothing upstream either (SURVEY R8): it still finds its row through int(key), with forced 0.  row is
    None for an id the table does not hold."""
    S = len(table)
    forced = np.bincount(np.asarray(orow, np.int64), minlength=S) if len(orow) else np.zeros(S, np.int64)
    ids = np.asarray(table.ids, np.int64)
    order = np.argsort(ids, kind="stable")
    for name, group in groups.items():
        for key, weight in group.deleterious.items():
            snp_id = int(key)
            j = int(np.searchsorted(ids[order], snp_id))
            if j >= S or ids[order[j]] != snp_id:
                yield name, snp_id, weight, None, 0
            else:
                r = int(order[j])
                yield name, snp_id, weight, r, int(forced[r])


def rank_of(tested, x):
    """1 + the number of values of the sorted array `tested` above x; behind all of them when x is None (NA)."""
    return len(tested) + 1 if x is None else 1 + len(tested) - int(np.searchsorted(tested, x, side="right"))


def deleterious_report(table, groups, counts, orow):
    """deleterious_assoc.txt text and its one-line summary.

    One line per (group, planted SNP) (planted_rows): FORCED is the number of cases whose minor allele was forced on
    that row.  RANK is 1 + the rows with a larger CHISQ (ranked by CHISQ, not P, which underflows to 0 for strong
    effects); a row whose CHISQ is NA ranks behind every tested row.
    -> (text bytes, summary str)."""
    counts = np.asarray(counts, np.uint32).reshape(-1, 4)
    S = len(table)
    x2 = chisq(counts)
    tested = np.sort(x2[~np.isnan(x2)])
    lines = ["\t".join(REPORT_COLUMNS)]
    planted = hits = 0
    alpha = 0.05 / max(S, 1)
    for name, snp_id, weight, r, forced in planted_rows(table, groups, orow):
        planted += 1
        if r is None:
            lines.append("\t".join([name, "rs%d" % snp_id, "NA", "NA", "%g" % weight, "0"] + ["NA"] * 6))
            continue
        f_a, f_u, x, p, odds = row_stats(*counts[r])
        hits += p is not None and p < alpha
        lines.append("\t".join([name, "rs%d" % snp_id, table.chrom_labels[table.chrom_idx[r]], "%d" % table.position[r],
                                "%g" % weight, "%d" % forced, _g(f_a), _g(f_u), _g(x), _g(p), _g(odds),
                                "%d" % rank_of(tested, x)]))
    summary = "%d of %d planted deleterious SNPs pass P < 0.05 / %d = %.3g" % (hits, planted, S, alpha)
    return ("\n".join(lines) + "\n").encode(), summary
