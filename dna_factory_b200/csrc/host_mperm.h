// Host side of the max(T) permutation tests (k_mperm.cuh) and the .mperm text formatter.  The permutation case masks
// are drawn once per call (k_perm_masks, in the first pass); rows then run through count_passes (host_assoc.h), every
// pass k_geno (the row totals) -> k_mperm_planes -> k_mperm.  A row costs 40 bytes of counters, 8 * pitch bytes of
// planes (two bits a sample) and 24 bytes of T_obs and exceedances; the per-permutation maxima accumulate across passes
// in d_maxt.  Included by dnaf_api.cu after host_geno.h.
#pragma once

namespace {

// words per plane / mask row: ceil(n / 32), padded to whole staging steps of k_mperm
uint32_t mperm_pitch(uint32_t n) {
    const uint32_t w = (n + 31u) / 32u;
    return std::max(kMpermKw, (w + kMpermKw - 1) / kMpermKw * kMpermKw);
}

int check_perms(dnaf_ctx* c, uint64_t first, uint64_t n_perm) {
    if (!c->have_samples) return fail(c, DNAF_E_ARG, "set_samples must be called first");
    if (n_perm == 0) return fail(c, DNAF_E_ARG, "n_perm must be at least 1");
    if (first + n_perm > (1ull << 32)) return fail(c, DNAF_E_ARG, "permutation indices must stay below 2^32");
    return DNAF_OK;
}

PermMaskArgs perm_mask_args(const dnaf_ctx* c, uint64_t seed, uint64_t first, uint32_t n_perm, uint64_t pitch_p,
                            uint64_t pitch_w, uint32_t* masks, uint32_t* sexcnt) {
    PermMaskArgs m;
    m.sex = c->d_sex.as<uint8_t>();
    m.n = c->n;
    m.ncase = c->ncase;
    m.first = (uint32_t)first;
    m.n_perm = n_perm;
    m.pitch_p = pitch_p;
    m.pitch_w = pitch_w;
    m.k0 = (uint32_t)seed;
    m.k1 = (uint32_t)(seed >> 32);
    m.masks = masks;
    m.sexcnt = sexcnt;
    return m;
}

int perm_masks_impl(dnaf_ctx* c, uint64_t seed, uint64_t first, uint32_t n_perm, uint32_t* masks, uint32_t* sexcnt) {
    int rc = check_perms(c, first, n_perm);
    if (rc) return rc;
    CU(c, cudaSetDevice(c->dev));
    const uint64_t W = (c->n + 31u) / 32u, mask_bytes = (uint64_t)n_perm * W * 4u;
    CU(c, c->d_pmask.reserve(mask_bytes + (uint64_t)n_perm * 8u));
    uint32_t* d_sex = reinterpret_cast<uint32_t*>(c->d_pmask.as<uint8_t>() + mask_bytes);
    const PermMaskArgs m = perm_mask_args(c, seed, first, n_perm, W, 1, c->d_pmask.as<uint32_t>(), d_sex);
    k_perm_masks<<<(n_perm + kPermMaskThreads - 1) / kPermMaskThreads, kPermMaskThreads, 0, c->stream>>>(m);
    CU(c, cudaGetLastError());
    if (masks) CU(c, cudaMemcpyAsync(masks, c->d_pmask.p, mask_bytes, cudaMemcpyDeviceToHost, c->stream));
    if (sexcnt) CU(c, cudaMemcpyAsync(sexcnt, d_sex, (uint64_t)n_perm * 8u, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return DNAF_OK;
}

int mperm_passes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t n_perm, double* t_obs,
                 uint32_t* exceed, double* max_t, dnaf_stats* st) {
    int rc = check_biallelic(c, row_begin, row_end, "the permutation test");
    if (!rc) rc = check_perms(c, 0, n_perm);
    if (rc) return rc;
    if (c->ncase == 0 || c->ncase == c->n)
        return fail(c, DNAF_E_ARG, "the permutation test needs cases and controls (%u cases of %u samples)", c->ncase, c->n);
    CU(c, cudaSetDevice(c->dev));
    const GenoArgs g = geno_args(c, seed);
    const uint32_t pitch = mperm_pitch(c->n), ptiles = (n_perm + kMpermTile - 1) / kMpermTile;
    const uint64_t perms = (uint64_t)ptiles * kMpermTile, mask_bytes = perms * pitch * 4u;
    const uint64_t row_bytes = 4u * kGenoWords + 8ull * pitch + 24u;
    const uint32_t tiles = std::max(g.tiles, ptiles);   // bounds k_geno's and k_mperm's grids alike
    const uint64_t per_pass = std::max<uint64_t>(1, std::min<uint64_t>(c->chunk_bytes / row_bytes, 0x7FFFFFFFull / tiles));
    const uint64_t rows = std::min(row_end - row_begin, per_pass);
    const uint64_t rows_pad = (rows + kMpermTile - 1) / kMpermTile * kMpermTile;
    CU(c, c->d_pmask.reserve(mask_bytes + perms * 8u));
    CU(c, c->d_maxt.reserve((uint64_t)n_perm * 16u));
    if (rows) {
        CU(c, c->d_planes.reserve(2 * rows_pad * pitch * 4u));
        CU(c, c->d_mrow.reserve(rows * 24u));
    }
    uint32_t* d_sexcnt = reinterpret_cast<uint32_t*>(c->d_pmask.as<uint8_t>() + mask_bytes);
    CU(c, cudaMemsetAsync(c->d_pmask.p, 0, mask_bytes, c->stream));   // padding words and permutations: empty masks
    CU(c, cudaMemsetAsync(c->d_maxt.p, 0, (uint64_t)n_perm * 16u, c->stream));
    MpermPlaneArgs pl;
    pl.cls = g.cls;
    pl.k = g.k;
    pl.thr = g.thr;
    pl.sexmask = g.sexmask;
    pl.orow = g.orow;
    pl.osamp = g.osamp;
    pl.n_over = g.n_over;
    pl.row_base = g.row_base;
    pl.n = g.n;
    pl.groups = g.groups;
    pl.tiles = g.tiles;
    pl.k0 = g.k0;
    pl.k1 = g.k1;
    pl.pitch = pitch;
    pl.plane_a = c->d_planes.as<uint32_t>();
    pl.plane_b = pl.plane_a + rows_pad * pitch;
    pl.exceed = reinterpret_cast<uint32_t*>(c->d_mrow.as<double>() + 2 * rows);
    MpermArgs m;
    m.plane_a = pl.plane_a;
    m.plane_b = pl.plane_b;
    m.masks = c->d_pmask.as<uint32_t>();
    m.sexcnt = d_sexcnt;
    m.cls = g.cls;
    m.n_perm = n_perm;
    m.ptiles = ptiles;
    m.pitch = pitch;
    m.t_obs = c->d_mrow.as<double>();
    m.exceed = pl.exceed;
    m.max_t = c->d_maxt.as<unsigned long long>();
    bool masks_drawn = false;
    auto launch = [&](uint64_t r0, uint64_t r1) {
        uint32_t n = 3;
        if (!masks_drawn) {   // once per call, timed with the first pass
            const PermMaskArgs pm = perm_mask_args(c, seed, 0, n_perm, pitch, 1, c->d_pmask.as<uint32_t>(), d_sexcnt);
            k_perm_masks<<<(n_perm + kPermMaskThreads - 1) / kPermMaskThreads, kPermMaskThreads, 0, c->stream>>>(pm);
            masks_drawn = true;
            ++n;
        }
        GenoArgs ga = g;
        ga.row0 = r0;
        ga.counts = c->d_counts.as<uint32_t>();
        k_geno<<<(uint32_t)((r1 - r0) * g.tiles), kGenoThreads, 0, c->stream>>>(ga);
        pl.row0 = r0;
        k_mperm_planes<<<(uint32_t)((r1 - r0) * g.tiles), kGenoThreads, 0, c->stream>>>(pl);
        m.counts = ga.counts;
        m.row0 = r0;
        m.rows = (uint32_t)(r1 - r0);
        const uint64_t rtiles = (r1 - r0 + kMpermTile - 1) / kMpermTile;
        k_mperm<<<(uint32_t)(rtiles * ptiles), kMpermThreads, 0, c->stream>>>(m);
        return n;
    };
    auto fetch = [&](uint64_t r0, uint64_t r1) {
        cudaError_t e = cudaSuccess;
        if (t_obs)
            e = cudaMemcpyAsync(t_obs + 2 * (r0 - row_begin), m.t_obs, (r1 - r0) * 16u, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess && exceed)
            e = cudaMemcpyAsync(exceed + 2 * (r0 - row_begin), m.exceed, (r1 - r0) * 8u, cudaMemcpyDeviceToHost, c->stream);
        return e;
    };
    rc = count_passes(c, row_begin, row_end, tiles, kGenoWords, row_bytes, st, launch, fetch);
    if (rc) return rc;
    if (max_t) {   // the bit patterns of non-negative doubles are the doubles
        CU(c, cudaMemcpyAsync(max_t, c->d_maxt.p, (uint64_t)n_perm * 16u, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    return DNAF_OK;
}

int mperm_impl(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t n_perm, double* t_obs,
               uint32_t* exceed, double* max_t, dnaf_stats* st) {
    if (!c) return DNAF_E_ARG;
    const int rc = mperm_passes(c, row_begin, row_end, seed, n_perm, t_obs, exceed, max_t, st);
    if (rc) quiesce(c);
    return rc;
}

}  // namespace

// .mperm body lines: pure host code (no context, no GPU).
namespace mpermfmt {

// CHR SNP EMP1 EMP2 of rows [r0,r1); emp = [rows][2] (EMP1, EMP2), NaN = NA
inline char* lines_serial(uint64_t r0, uint64_t r1, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                          const double* emp, char* o) {
    for (uint64_t r = r0; r < r1; ++r) {
        char lab[8], snp[32], v[2][32];
        const char* chr = assocfmt::chr_code(labels, chrom_idx[r], lab);
        snprintf(snp, sizeof snp, "rs%lld", (long long)ids[r]);
        assocfmt::num(v[0], 32, emp[2 * r]);
        assocfmt::num(v[1], 32, emp[2 * r + 1]);
        o += sprintf(o, "%4s %12s %12s %12s\n", chr, snp, v[0], v[1]);
    }
    return o;
}

constexpr uint64_t kLineBytes = 96;   // output room a row

}  // namespace mpermfmt
