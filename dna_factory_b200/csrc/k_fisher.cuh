// k_fisher: Fisher's exact test of case/control tables, as log10 P (dnaf_genotype_tests, dnaf_fisher_exact,
// dnaf_format_assoc_fisher, dnaf_format_model_fisher).
//
// Definition (PLINK's and scipy.stats.fisher_exact's): with both margins fixed, a 2x3 table with case row (x1, x2, x3),
// control row (y1, y2, y3), column sums c_j = x_j + y_j, R cases and N in all has probability
//   prod_j C(c_j, x_j) / C(N, R)                                   (the multivariate hypergeometric)
// and the two-sided P is the sum of the probabilities of every table whose probability is <= (1 + kHweTie) times the
// observed one.  A table with one empty column is the 2x2 test over the other two (the same conditional distribution),
// so a 2x2 test is the 2x3 table with x3 = y3 = 0.  NaN (no test) when a row margin is 0 or fewer than two columns are
// non-empty: then only one table exists.
//
// Numerics (as hwe_exact_p): every term is a product of ratios started at the mode, so no term exceeds the mode's ~1.
// Moving one case from column j to column i multiplies the term by y_i x_j / ((x_i + 1)(y_j + 1)).  Scales are kept in
// a separate integer exponent: a running term is renormalised by 2^512 whenever it falls below 2^-512, the observed
// term fixes the scale e_obs of the tail sum, and log10 P = log10(tail / total) + e_obs log10 2.  So log10 P stays
// exact far below the double range.  Each tail stops once its terms are below the observed one and below 2^-64 of the
// tail sum.
//
// Two columns (2x2): one walk over x1 from its mode, as hwe_exact_p.
// Three columns (2x3): the tables form a plane (u = cases in the outer column, v = cases in the first inner column).
// The sum of row u's terms is proportional to the hypergeometric marginal of u, so one full walk of the mode row gives
// every row sum by a 1-D recurrence, and the total costs one row plus the marginal.  Every row's largest term (its
// anchor) follows from the previous row's in O(1) moves.  A row whose anchor is <= the threshold belongs to the tail
// whole (its row sum); only the rows whose anchor is above it are walked term by term, from the anchor out to both of
// their tails.  For a P near 0.5 that is a few rows around the mode instead of the whole plane.
#pragma once
#include "k_geno.cuh"

namespace dnaf {

constexpr double kFisherLo = 0x1p-512, kFisherUp = 0x1p512;
constexpr int kFisherExp = 512;
constexpr double kLog10_2 = 0.30102999566398119521;

__device__ __forceinline__ double fisher_nan() { return __longlong_as_double(0x7FF8000000000000ll); }

// one case from column j to column i: y_i x_j / ((x_i + 1)(y_j + 1))
__device__ __forceinline__ double fisher_mv(int64_t xi, int64_t yi, int64_t xj, int64_t yj) {
    return (double)yi * (double)xj / ((double)(xi + 1) * (double)(yj + 1));
}

__device__ __forceinline__ void fisher_renorm(double& t, int& e) {
    if (t < kFisherLo) {
        t *= kFisherUp;
        e -= kFisherExp;
    }
}

// t 2^e expressed in the scale 2^s
__device__ __forceinline__ double fisher_at(double t, int e, int s) { return e == s ? t : ldexp(t, e - s); }

__device__ __forceinline__ double fisher_log10(double tail, double total, int e_obs) {
    return fmin(0.0, log10(tail / total) + (double)e_obs * kLog10_2);
}

// 2x2: x cases of the c cases + controls in column a, R cases, N in all
__device__ double fisher_1d(int64_t x, int64_t c, int64_t R, int64_t N) {
    const int64_t lo = max((int64_t)0, R - (N - c)), hi = min(c, R);
    // t(k+1) / t(k) with k cases in column a: (c - k)(R - k) / ((k + 1)(N - c - R + k + 1))
    auto up = [&](int64_t k) { return fisher_mv(k, c - k, R - k, N - c - R + k); };
    auto down = [&](int64_t k) { return fisher_mv(R - k, N - c - R + k, k, c - k); };
    int64_t m = min(hi, max(lo, (int64_t)(((double)R + 1.0) * ((double)c + 1.0) / ((double)N + 2.0))));
    while (m < hi && up(m) > 1.0) ++m;
    while (m > lo && down(m) > 1.0) --m;
    double p = 1.0;
    int e_obs = 0;
    for (int64_t k = m; k < x; ++k) p *= up(k), fisher_renorm(p, e_obs);
    for (int64_t k = m; k > x; --k) p *= down(k), fisher_renorm(p, e_obs);
    const double thr = p * (1.0 + kHweTie);
    double total = 1.0, tail = 0.0;
    if (e_obs == 0 && 1.0 <= thr) tail = 1.0;
    for (int dir = 0; dir < 2; ++dir) {
        double t = 1.0;
        int e = 0;
        for (int64_t k = m; dir ? k < hi : k > lo; k += dir ? 1 : -1) {
            t *= dir ? up(k) : down(k);
            fisher_renorm(t, e);
            if (e == 0) total += t;
            const double v = fisher_at(t, e, e_obs);
            if (v <= thr) {
                tail += v;
                if (v <= tail * 0x1p-64) break;
            }
        }
    }
    return fisher_log10(tail, total, e_obs);
}

// 2x3, all three columns non-empty: x0 cases of the c0 in the outer column, x1 of the c1 in the first inner one
__device__ double fisher_2d(int64_t x0, int64_t x1, int64_t c0, int64_t c1, int64_t c2, int64_t R, int64_t N) {
    const int64_t S = N - R;
    const int64_t x[2] = {x0, x1}, c[3] = {c0, c1, c2};
    const int64_t ulo = max((int64_t)0, R - c[1] - c[2]), uhi = min(c[0], R);
    // row u: v cases in column 1, w = R - u - v in column 2
    auto vlo = [&](int64_t u) { return max((int64_t)0, R - u - c[2]); };
    auto vhi = [&](int64_t u) { return min(c[1], R - u); };
    auto vup = [&](int64_t u, int64_t v) { const int64_t w = R - u - v; return fisher_mv(v, c[1] - v, w, c[2] - w); };
    auto vdown = [&](int64_t u, int64_t v) { const int64_t w = R - u - v; return fisher_mv(w, c[2] - w, v, c[1] - v); };
    // row sums: the hypergeometric marginal of u (u of the c[0] in column 0 among R cases)
    auto rup = [&](int64_t u) { return fisher_mv(u, c[0] - u, R - u, S - (c[0] - u)); };
    auto rdown = [&](int64_t u) { return fisher_mv(R - u, S - (c[0] - u), u, c[0] - u); };
    // anchor of row u +- 1 from the anchor (u, v) of row u: one case in or out of column 0 through column 2 when it
    // can (else column 1), then uphill along the row to its largest term
    auto step = [&](int dir, int64_t& u, int64_t& v, double& a, int& ae) {
        const int64_t w = R - u - v;
        if (dir) {
            if (w > 0) a *= fisher_mv(u, c[0] - u, w, c[2] - w);
            else a *= fisher_mv(u, c[0] - u, v, c[1] - v), --v;
            ++u;
        } else {
            if (w < c[2]) a *= fisher_mv(w, c[2] - w, u, c[0] - u);
            else a *= fisher_mv(v, c[1] - v, u, c[0] - u), ++v;
            --u;
        }
        double r;
        while (v < vhi(u) && (r = vup(u, v)) > 1.0) a *= r, ++v;
        while (v > vlo(u) && (r = vdown(u, v)) > 1.0) a *= r, --v;
        fisher_renorm(a, ae);
    };
    int64_t m0 = min(uhi, max(ulo, (int64_t)(((double)R + 1.0) * ((double)c[0] + 1.0) / ((double)N + 2.0))));
    while (m0 < uhi && rup(m0) > 1.0) ++m0;
    while (m0 > ulo && rdown(m0) > 1.0) --m0;
    int64_t v0 = min(vhi(m0), max(vlo(m0), (int64_t)(((double)(R - m0) + 1.0) * ((double)c[1] + 1.0) /
                                                        ((double)(c[1] + c[2]) + 2.0))));
    while (v0 < vhi(m0) && vup(m0, v0) > 1.0) ++v0;
    while (v0 > vlo(m0) && vdown(m0, v0) > 1.0) --v0;
    // the observed term, relative to the anchor of row m0
    double p = 1.0;
    int e_obs = 0;
    {
        int64_t u = m0, v = v0;
        while (u != x[0]) step(u < x[0], u, v, p, e_obs);
        for (; v < x[1]; ++v) p *= vup(u, v), fisher_renorm(p, e_obs);
        for (; v > x[1]; --v) p *= vdown(u, v), fisher_renorm(p, e_obs);
    }
    const double thr = p * (1.0 + kHweTie);
    // the mode row in full: its sum, relative to its anchor
    double rs0 = 1.0;
    for (int dir = 0; dir < 2; ++dir) {
        double t = 1.0;
        for (int64_t v = v0; dir ? v < vhi(m0) : v > vlo(m0); v += dir ? 1 : -1) {
            t *= dir ? vup(m0, v) : vdown(m0, v);
            rs0 += t;
            if (t <= rs0 * 0x1p-64) break;
        }
    }
    double total = 0.0, tail = 0.0;
    for (int dir = 0; dir < 2; ++dir) {   // rows below m0, then m0 and above
        int64_t u = m0, v = v0;
        double a = 1.0, rs = rs0;
        int ae = 0, re = 0;
        if (!dir) {
            if (u == ulo) continue;
            step(0, u, v, a, ae);
            rs *= rdown(m0);
            fisher_renorm(rs, re);
        }
        for (;;) {
            if (re == 0) total += rs;
            if (fisher_at(a, ae, e_obs) <= thr) {   // the whole row is in the tail
                const double r = fisher_at(rs, re, e_obs);
                tail += r;
                if (r <= tail * 0x1p-64) break;
            } else {                                // the row's terms from its anchor (> thr) out to both tails
                for (int side = 0; side < 2; ++side) {
                    double t = a;
                    int e = ae;
                    for (int64_t w = v; side ? w < vhi(u) : w > vlo(u); w += side ? 1 : -1) {
                        t *= side ? vup(u, w) : vdown(u, w);
                        fisher_renorm(t, e);
                        const double q = fisher_at(t, e, e_obs);
                        if (q <= thr) {
                            tail += q;
                            if (q <= tail * 0x1p-64) break;
                        }
                    }
                }
            }
            if (dir ? u == uhi : u == ulo) break;
            rs *= dir ? rup(u) : rdown(u);
            fisher_renorm(rs, re);
            step(dir, u, v, a, ae);
        }
    }
    return fisher_log10(tail, total, e_obs);
}

// log10 of the two-sided Fisher exact P of the table with case row (x1, x2, x3) and control row (y1, y2, y3)
__device__ double fisher_exact_log10p(uint32_t x1, uint32_t x2, uint32_t x3, uint32_t y1, uint32_t y2, uint32_t y3) {
    const int64_t c1 = (int64_t)x1 + y1, c2 = (int64_t)x2 + y2, c3 = (int64_t)x3 + y3;
    const int64_t R = (int64_t)x1 + x2 + x3, N = c1 + c2 + c3;
    const int k = (c1 > 0) + (c2 > 0) + (c3 > 0);
    if (k < 2 || R == 0 || R == N) return fisher_nan();
    if (k == 2) return c1 ? fisher_1d(x1, c1, R, N) : fisher_1d(x2, c2, R, N);   // the first non-empty column
    // the smallest column is the outer one, the other two keep their order
    if (c1 <= c2 && c1 <= c3) return fisher_2d(x1, x2, c1, c2, c3, R, N);
    if (c2 <= c3) return fisher_2d(x2, x1, c2, c1, c3, R, N);
    return fisher_2d(x3, x1, c3, c1, c2, R, N);
}

constexpr uint32_t kFisherThreads = 128;
constexpr uint32_t kFisherTests = 4;   // per row: GENO, ALLELIC, DOM, REC

struct FisherArgs {
    const uint32_t* counts;   // rows: [rows][10] of k_geno; tables: [items][6] = (x1, x2, x3, y1, y2, y3)
    uint64_t items;           // rows: 4 * rows; tables: items
    int rows;                 // layout of counts
    double* log10p;           // rows: [rows][4] (GENO, ALLELIC, DOM, REC); tables: [items]
};

// rows layout: items [0, rows) are the GENO tests (the long ones go first), then ALLELIC, DOM, REC of every row
__global__ void __launch_bounds__(kFisherThreads) k_fisher(const FisherArgs a) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.items) return;
    if (!a.rows) {
        const uint32_t* t = a.counts + 6 * i;
        a.log10p[i] = fisher_exact_log10p(t[0], t[1], t[2], t[3], t[4], t[5]);
        return;
    }
    const uint64_t rows = a.items / kFisherTests;
    uint64_t row;
    uint32_t test;
    if (i < rows) {
        row = i;
        test = 0;
    } else {
        row = (i - rows) / 3;
        test = 1 + (uint32_t)(i - rows - 3 * row);
    }
    const uint32_t* c = a.counts + kGenoWords * row;
    // the diploid genotypes (n11, n12, n22) and the alleles (haploid cells included) of the cases and the controls
    const uint32_t a11 = c[2], a12 = c[1], a22 = c[0] - c[1] - c[2], u11 = c[7], u12 = c[6], u22 = c[5] - c[6] - c[7];
    double r;
    if (test == 0) {
        r = fisher_exact_log10p(a11, a12, a22, u11, u12, u22);
    } else if (test == 1) {
        const uint32_t alt_a = 2 * a11 + a12 + c[4], alt_u = 2 * u11 + u12 + c[9];
        r = fisher_exact_log10p(alt_a, 2 * c[0] + c[3] - alt_a, 0, alt_u, 2 * c[5] + c[8] - alt_u, 0);
    } else if (test == 2) {
        r = fisher_exact_log10p(a11 + a12, a22, 0, u11 + u12, u22, 0);
    } else {
        r = fisher_exact_log10p(a11, a12 + a22, 0, u11, u12 + u22, 0);
    }
    a.log10p[kFisherTests * row + test] = r;
}

}  // namespace dnaf
