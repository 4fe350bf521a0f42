// Host side of the case/control genotype counts (k_geno), the Hardy-Weinberg exact tests (k_hwe) and Fisher's exact
// tests (k_fisher), and the .model, .hwe and Fisher text formatters.  The counts run through count_passes
// (host_assoc.h): 40 bytes of counters a row, plus 24 bytes of P a row when the call also runs k_hwe over the pass's
// counters (three tests a row: ALL, AFF, UNAFF), plus 32 bytes of log10 P a row when it also runs k_fisher (four tests
// a row: GENO, ALLELIC, DOM, REC).  Included by dnaf_api.cu after host_assoc.h.
#pragma once

namespace {

// k_geno's arguments for the context's samples, SNPs and forced minors (row0 and counts are set per pass)
GenoArgs geno_args(const dnaf_ctx* c, uint64_t seed) {
    GenoArgs a;
    a.cls = c->d_cls.as<uint8_t>();
    a.k = c->d_k.as<uint8_t>();
    a.thr = c->d_thr.as<uint32_t>();
    a.sexmask = c->d_sexmask.as<uint2>();
    a.casemask = c->d_casemask.as<uint32_t>();
    a.orow = c->d_orow.as<uint64_t>();
    a.osamp = c->d_osamp.as<uint32_t>();
    a.n_over = c->P;
    a.row_base = c->row_base;
    a.n = c->n;
    a.groups = (c->n + 15u) / 16u;
    a.tiles = std::max<uint32_t>(1u, (a.groups + kGenoThreads - 1u) / kGenoThreads);
    a.k0 = (uint32_t)seed;
    a.k1 = (uint32_t)(seed >> 32);
    return a;
}

int geno_passes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* out, double* hwe_out,
                bool with_hwe, double* fisher_out, bool with_fisher, dnaf_stats* st) {
    int rc = check_biallelic(c, row_begin, row_end, "the genotype count");
    if (rc) return rc;
    GenoArgs a = geno_args(c, seed);
    constexpr uint64_t kCountBytes = 4u * kGenoWords, kFisherBytes = kFisherTests * sizeof(double);
    const uint64_t row_bytes = kCountBytes + (with_hwe ? 3u * sizeof(double) : 0u) + (with_fisher ? kFisherBytes : 0u);
    if ((with_hwe || with_fisher) && row_end > row_begin) {
        const uint64_t per_pass = std::max<uint64_t>(1, std::min<uint64_t>(c->chunk_bytes / row_bytes, 0x7FFFFFFFull / a.tiles));
        const uint64_t rows = std::min(row_end - row_begin, per_pass);
        if (with_hwe) CU(c, c->d_hwe.reserve(rows * 3u * sizeof(double)));
        if (with_fisher) CU(c, c->d_fisher.reserve(rows * kFisherBytes));
    }
    auto launch = [&](uint64_t r0, uint64_t r1) {
        a.row0 = r0;
        a.counts = c->d_counts.as<uint32_t>();
        k_geno<<<(uint32_t)((r1 - r0) * a.tiles), kGenoThreads, 0, c->stream>>>(a);
        uint32_t n = 1;
        if (with_hwe) {
            HweArgs h;
            h.counts = a.counts;
            h.items = 3 * (r1 - r0);
            h.rows = 1;
            h.p = c->d_hwe.as<double>();
            k_hwe<<<(uint32_t)((h.items + 255) / 256), 256, 0, c->stream>>>(h);
            ++n;
        }
        if (with_fisher) {
            FisherArgs f;
            f.counts = a.counts;
            f.items = kFisherTests * (r1 - r0);
            f.rows = 1;
            f.log10p = c->d_fisher.as<double>();
            k_fisher<<<(uint32_t)((f.items + kFisherThreads - 1) / kFisherThreads), kFisherThreads, 0, c->stream>>>(f);
            ++n;
        }
        return n;
    };
    auto fetch = [&](uint64_t r0, uint64_t r1) {
        cudaError_t e = cudaSuccess;
        if (out)
            e = cudaMemcpyAsync(out + kGenoWords * (r0 - row_begin), c->d_counts.p, (r1 - r0) * kCountBytes,
                                cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess && with_hwe && hwe_out)
            e = cudaMemcpyAsync(hwe_out + 3 * (r0 - row_begin), c->d_hwe.p, (r1 - r0) * 3u * sizeof(double),
                                cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess && with_fisher && fisher_out)
            e = cudaMemcpyAsync(fisher_out + kFisherTests * (r0 - row_begin), c->d_fisher.p, (r1 - r0) * kFisherBytes,
                                cudaMemcpyDeviceToHost, c->stream);
        return e;
    };
    return count_passes(c, row_begin, row_end, a.tiles, kGenoWords, row_bytes, st, launch, fetch);
}

int geno_impl(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* out, double* hwe_out,
              bool with_hwe, double* fisher_out, bool with_fisher, dnaf_stats* st) {
    if (!c) return DNAF_E_ARG;
    const int rc = geno_passes(c, row_begin, row_end, seed, out, hwe_out, with_hwe, fisher_out, with_fisher, st);
    if (rc) quiesce(c);
    return rc;
}

int hwe_exact_impl(dnaf_ctx* c, uint64_t n, const uint32_t* geno, double* p) {
    if (n == 0) return DNAF_OK;
    if (n > 0x7FFFFFFFull * 256u) return fail(c, DNAF_E_ARG, "too many triples for one grid");
    CU(c, cudaSetDevice(c->dev));
    int rc = upload(c, c->d_counts, geno, 3 * n, false);
    if (rc) return rc;
    CU(c, c->d_hwe.reserve(n * sizeof(double)));
    HweArgs h;
    h.counts = c->d_counts.as<uint32_t>();
    h.items = n;
    h.rows = 0;
    h.p = c->d_hwe.as<double>();
    k_hwe<<<(uint32_t)((n + 255) / 256), 256, 0, c->stream>>>(h);
    CU(c, cudaGetLastError());
    CU(c, cudaMemcpyAsync(p, c->d_hwe.p, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return DNAF_OK;
}

int fisher_exact_impl(dnaf_ctx* c, uint64_t n, const uint32_t* tables, double* log10p) {
    if (n == 0) return DNAF_OK;
    if (n > 0x7FFFFFFFull * kFisherThreads) return fail(c, DNAF_E_ARG, "too many tables for one grid");
    CU(c, cudaSetDevice(c->dev));
    int rc = upload(c, c->d_counts, tables, 6 * n, false);
    if (rc) return rc;
    CU(c, c->d_fisher.reserve(n * sizeof(double)));
    FisherArgs f;
    f.counts = c->d_counts.as<uint32_t>();
    f.items = n;
    f.rows = 0;
    f.log10p = c->d_fisher.as<double>();
    k_fisher<<<(uint32_t)((n + kFisherThreads - 1) / kFisherThreads), kFisherThreads, 0, c->stream>>>(f);
    CU(c, cudaGetLastError());
    CU(c, cudaMemcpyAsync(log10p, c->d_fisher.p, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return DNAF_OK;
}

}  // namespace

// .model and .hwe body lines: pure host code (no context, no GPU).
namespace modelfmt {

// One row's diploid genotype counts (ALT/ALT, het, REF/REF) and allele counts, cases (a) and controls (u), from its
// ten k_geno counters.
struct RowCounts {
    double a11, a12, a22, u11, u12, u22;   // diploid genotypes
    double alt_a, ref_a, alt_u, ref_u;     // alleles, haploid cells included (the .assoc counts)
    explicit RowCounts(const uint32_t* c)
        : a11(c[2]), a12(c[1]), a22((double)c[0] - c[1] - c[2]), u11(c[7]), u12(c[6]), u22((double)c[5] - c[6] - c[7]) {
        alt_a = 2 * a11 + a12 + c[4];
        ref_a = 2.0 * c[0] + c[3] - alt_a;
        alt_u = 2 * u11 + u12 + c[9];
        ref_u = 2.0 * c[5] + c[8] - alt_u;
    }
    bool cells_ok() const { return a11 >= 5 && a12 >= 5 && a22 >= 5 && u11 >= 5 && u12 >= 5 && u22 >= 5; }
};

inline double nan_() { return std::nan(""); }

// chi2_2x2, the Pearson 2x2 of .assoc, ALLELIC, DOM and REC: k_mperm.cuh (shared with the permutation kernel)

// Pearson 2x3 over the genotype cells
inline double chi2_geno(const RowCounts& g) {
    const double R = g.a11 + g.a12 + g.a22, S = g.u11 + g.u12 + g.u22, N = R + S;
    const double a[3] = {g.a11, g.a12, g.a22}, u[3] = {g.u11, g.u12, g.u22};
    if (R <= 0 || S <= 0) return nan_();
    double x = 0;
    for (int j = 0; j < 3; ++j) {
        const double nj = a[j] + u[j];
        if (nj <= 0) return nan_();
        const double ea = R * nj / N, eu = S * nj / N;
        x += (a[j] - ea) * (a[j] - ea) / ea + (u[j] - eu) * (u[j] - eu) / eu;
    }
    return x;
}

// Cochran-Armitage trend, x = ALT copies: N (N sum x r_x - R sum x n_x)^2 / (R S (N sum x^2 n_x - (sum x n_x)^2))
inline double chi2_trend(const RowCounts& g) {
    const double R = g.a11 + g.a12 + g.a22, S = g.u11 + g.u12 + g.u22, N = R + S;
    const double sxr = 2 * g.a11 + g.a12, sxn = 2 * (g.a11 + g.u11) + (g.a12 + g.u12), sx2n = 4 * (g.a11 + g.u11) + (g.a12 + g.u12);
    const double den = R * S * (N * sx2n - sxn * sxn);
    const double t = N * sxr - R * sxn;
    return den > 0 ? N * t * t / den : nan_();
}

// CHISQ of GENO, TREND, ALLELIC, DOM, REC (PLINK's order), NaN = NA
inline void model_chisq(const uint32_t* c, double x[5]) {
    const RowCounts g(c);
    const bool ok = g.cells_ok();
    x[0] = ok ? chi2_geno(g) : nan_();
    x[1] = chi2_trend(g);
    x[2] = chi2_2x2(g.alt_a, g.ref_a, g.alt_u, g.ref_u);
    x[3] = ok ? chi2_2x2(g.a11 + g.a12, g.a22, g.u11 + g.u12, g.u22) : nan_();
    x[4] = ok ? chi2_2x2(g.a11, g.a12 + g.a22, g.u11, g.u12 + g.u22) : nan_();
}

inline double chi2_sf(double x, int df) { return df == 1 ? std::erfc(std::sqrt(x / 2.0)) : std::exp(-x / 2.0); }

inline char a1_of(const uint8_t* nts, const uint8_t* n_alleles, uint64_t r) {
    return n_alleles[r] >= 2 ? (char)nts[4 * r + 1] : '0';   // A1 = ALT ('0' when the row has none), as in the .bim
}

// The columns a .model line and a Fisher .model line share: CHR, SNP, A1, A2 and the AFF / UNAFF cells of GENO, TREND,
// ALLELIC, DOM, REC
struct ModelFields {
    char lab[8], snp[32], aff[5][40], unaff[5][40];
    const char* chr;
    char a1, a2;
    ModelFields(uint64_t r, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const uint8_t* nts,
                const uint8_t* n_alleles, const uint32_t* c, const RowCounts& g) {
        chr = assocfmt::chr_code(labels, chrom_idx[r], lab);
        snprintf(snp, sizeof snp, "rs%lld", (long long)ids[r]);
        a1 = a1_of(nts, n_alleles, r);
        a2 = (char)nts[4 * r];
        const unsigned A11 = c[2], A12 = c[1], A22 = c[0] - c[1] - c[2], U11 = c[7], U12 = c[6], U22 = c[5] - c[6] - c[7];
        snprintf(aff[0], 40, "%u/%u/%u", A11, A12, A22);
        snprintf(unaff[0], 40, "%u/%u/%u", U11, U12, U22);
        memcpy(aff[1], aff[0], 40);
        memcpy(unaff[1], unaff[0], 40);
        snprintf(aff[2], 40, "%.0f/%.0f", g.alt_a, g.ref_a);
        snprintf(unaff[2], 40, "%.0f/%.0f", g.alt_u, g.ref_u);
        snprintf(aff[3], 40, "%u/%u", A11 + A12, A22);
        snprintf(unaff[3], 40, "%u/%u", U11 + U12, U22);
        snprintf(aff[4], 40, "%u/%u", A11, A12 + A22);
        snprintf(unaff[4], 40, "%u/%u", U11, U12 + U22);
    }
};

static const char* const kModelTest[5] = {"GENO", "TREND", "ALLELIC", "DOM", "REC"};

inline char* model_serial(uint64_t r0, uint64_t r1, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                          const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, char* o) {
    static const int kDf[5] = {2, 1, 1, 1, 1};
    for (uint64_t r = r0; r < r1; ++r) {
        const uint32_t* c = counts + (uint64_t)kGenoWords * r;
        const RowCounts g(c);
        const ModelFields f(r, chrom_idx, labels, ids, nts, n_alleles, c, g);
        double x[5];
        model_chisq(c, x);
        for (int t = 0; t < 5; ++t) {
            const bool na = std::isnan(x[t]);
            char vx[32], vp[32], df[8];
            assocfmt::num(vx, 32, x[t]);
            assocfmt::num(vp, 32, na ? x[t] : chi2_sf(x[t], kDf[t]));
            snprintf(df, sizeof df, na ? "NA" : "%d", kDf[t]);
            o += sprintf(o, "%4s %12s %4c %4c %8s %14s %14s %12s %4s %12s\n", f.chr, f.snp, f.a1, f.a2, kModelTest[t], f.aff[t],
                         f.unaff[t], vx, df, vp);
        }
    }
    return o;
}

// "%.4g" of the P whose log10 is l: 0 where 10^l underflows, NA for NaN
inline int fisher_p(char* p, size_t cap, double l) { return assocfmt::num(p, cap, std::isnan(l) ? l : std::pow(10.0, l)); }

// Fisher .model lines: GENO, TREND, ALLELIC, DOM, REC; TREND keeps its asymptotic P, the others print the Fisher P of
// `log10p` ([rows][4]: GENO, ALLELIC, DOM, REC)
inline char* model_fisher_serial(uint64_t r0, uint64_t r1, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                                 const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, const double* log10p,
                                 char* o) {
    for (uint64_t r = r0; r < r1; ++r) {
        const uint32_t* c = counts + (uint64_t)kGenoWords * r;
        const RowCounts g(c);
        const ModelFields f(r, chrom_idx, labels, ids, nts, n_alleles, c, g);
        const double* l = log10p + 4 * r;
        for (int t = 0; t < 5; ++t) {
            char vp[32];
            if (t == 1) {
                const double x = chi2_trend(g);
                assocfmt::num(vp, 32, std::isnan(x) ? x : chi2_sf(x, 1));
            } else {
                fisher_p(vp, 32, l[t == 0 ? 0 : t - 1]);
            }
            o += sprintf(o, "%4s %12s %4c %4c %8s %14s %14s %12s\n", f.chr, f.snp, f.a1, f.a2, kModelTest[t], f.aff[t],
                         f.unaff[t], vp);
        }
    }
    return o;
}

// .assoc.fisher lines: F_A, F_U and OR of the allele counts (haploid cells included), as in .assoc; P = Fisher ALLELIC
inline char* assoc_fisher_serial(uint64_t r0, uint64_t r1, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                                 const int64_t* position, const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts,
                                 const double* log10p, char* o) {
    for (uint64_t r = r0; r < r1; ++r) {
        const RowCounts g(counts + (uint64_t)kGenoWords * r);
        const assocfmt::AlleleStats s(g.alt_a, g.alt_a + g.ref_a, g.alt_u, g.alt_u + g.ref_u);
        char lab[8], snp[32], v[4][32];
        const char* chr = assocfmt::chr_code(labels, chrom_idx[r], lab);
        snprintf(snp, sizeof snp, "rs%lld", (long long)ids[r]);
        assocfmt::num(v[0], 32, s.f_a);
        assocfmt::num(v[1], 32, s.f_u);
        fisher_p(v[2], 32, log10p[4 * r + 1]);
        assocfmt::num(v[3], 32, s.odds);
        o += sprintf(o, "%4s %12s %10lld %4c %8s %8s %4c %12s %12s\n", chr, snp, (long long)position[r], a1_of(nts, n_alleles, r),
                     v[0], v[1], (char)nts[4 * r], v[2], v[3]);
    }
    return o;
}

inline char* hardy_serial(uint64_t r0, uint64_t r1, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                          const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, const double* hwe_p, char* o) {
    static const char* const kTest[3] = {"ALL", "AFF", "UNAFF"};
    for (uint64_t r = r0; r < r1; ++r) {
        const uint32_t* c = counts + (uint64_t)kGenoWords * r;
        char lab[8];
        const char* chr = assocfmt::chr_code(labels, chrom_idx[r], lab);
        char snp[32];
        snprintf(snp, sizeof snp, "rs%lld", (long long)ids[r]);
        const char a1 = a1_of(nts, n_alleles, r), a2 = (char)nts[4 * r];
        for (int t = 0; t < 3; ++t) {   // ALL = cases + controls, AFF = cases, UNAFF = controls
            const uint64_t dip = (t != 2 ? (uint64_t)c[0] : 0u) + (t != 1 ? c[5] : 0u);
            const uint64_t n12 = (t != 2 ? (uint64_t)c[1] : 0u) + (t != 1 ? c[6] : 0u);
            const uint64_t n11 = (t != 2 ? (uint64_t)c[2] : 0u) + (t != 1 ? c[7] : 0u);
            const uint64_t n22 = dip - n12 - n11;
            const double n = (double)dip, f = n > 0 ? (2.0 * n11 + n12) / (2.0 * n) : nan_();
            char geno[64], oh[32], eh[32], vp[32];
            snprintf(geno, sizeof geno, "%llu/%llu/%llu", (unsigned long long)n11, (unsigned long long)n12, (unsigned long long)n22);
            assocfmt::num(oh, 32, n > 0 ? n12 / n : nan_());
            assocfmt::num(eh, 32, 2.0 * f * (1.0 - f));
            assocfmt::num(vp, 32, hwe_p[3 * r + t]);
            o += sprintf(o, "%4s %12s %8s %4c %4c %20s %8s %8s %12s\n", chr, snp, kTest[t], a1, a2, geno, oh, eh, vp);
        }
    }
    return o;
}

constexpr uint64_t kModelLineBytes = 5 * 192, kHardyLineBytes = 3 * 192, kAssocLineBytes = 192;   // output room a row

}  // namespace modelfmt
