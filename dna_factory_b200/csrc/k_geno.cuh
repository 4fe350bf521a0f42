// k_geno: case/control genotype counts per row straight from the allele draws (draw -> forced minors -> count), the
// input of the genotypic tests of .model and the Hardy-Weinberg exact tests of .hwe (dnaf_genotype_counts,
// dnaf_format_model, dnaf_format_hardy).  k_hwe: the two-sided Hardy-Weinberg exact P of a (n11, n12, n22) triple.
//
// Counting rule (DESIGN.md 5, "Genotypic tests and Hardy-Weinberg"): every cell the VCF text prints
// (pop_factory.py:481-499) counts once --
//   diploid cells: everybody on autosome rows, females on X rows
//   haploid cells: males on X and Y rows, everybody on MT rows           female Y cells ('.') count nothing
// A forced minor sets both slots of its cell to ALT, so a diploid cell becomes 1/1 and a haploid cell ALT.  With the
// draw word w of a 16-sample group (bit 2i+s = allele slot s of sample i, set = ALT; rows have K <= 2, checked by the
// host), the diploid bit-pair mask D and the haploid slot-0 mask H of the row's class, E = slot 0 of every cell and
// the case bit pairs cs, the five counts of the group's cases are
//   dip = popc(D & E & cs), het = popc((w ^ w>>1) & E & D & cs), hom = popc(w & w>>1 & E & D & cs),
//   hap = popc(H & cs),     hap_alt = popc(w & H & cs)
// and the same five with ~cs for the controls.  One CTA covers (row, 256 groups) like k_assoc; its sums go to the
// pass's [row][10] array with one atomicAdd per counter (integer adds: the result does not depend on their order).
#pragma once
#include "k_bed.cuh"

namespace dnaf {

constexpr uint32_t kGenoThreads = 256;   // one thread per 16-sample word, one CTA per (row, 256 words)
constexpr uint32_t kGenoWords = 10;      // counters per row: dip, het, hom, hap, hap_alt of the cases, then of the controls

struct GenoArgs {
    const uint8_t* cls;       // chromosome class per row
    const uint8_t* k;         // alleles per row (<= 2: checked by the host)
    const uint32_t* thr;      // [row][4]
    const uint2* sexmask;     // per 16-sample group: x = bit pairs of the males, y = of the females (dnaf_set_samples)
    const uint32_t* casemask; // per 16-sample group: bit pairs of the cases (is_control == 0)
    const uint64_t* orow;     // override pairs, sorted by row
    const uint32_t* osamp;
    uint64_t n_over;
    uint64_t row0;            // first row of the pass
    uint64_t row_base;        // Philox row counter = row_base + row
    uint32_t n;               // samples
    uint32_t groups;          // ceil(n / 16)
    uint32_t tiles;           // CTAs per row: ceil(groups / kGenoThreads)
    uint32_t k0, k1;          // seed
    uint32_t* counts;         // [rows of the pass][10], zeroed before the launch; row 0 = row0
};

__global__ void __launch_bounds__(kGenoThreads) k_geno(const GenoArgs a) {
    __shared__ uint32_t s_w[kGenoThreads];
    __shared__ uint64_t s_ovr[2];
    __shared__ uint32_t s_sum[kGenoThreads / 32][kGenoWords];
    const uint32_t rl = blockIdx.x / a.tiles, tile = blockIdx.x - rl * a.tiles;
    const uint64_t row = a.row0 + rl;
    const uint32_t tid = threadIdx.x;
    const uint32_t g = tile * kGenoThreads + tid;
    const bool live = g < a.groups;
    if (tid < 2) s_ovr[tid] = bed_lower_bound(a.orow, a.n_over, row + tid);
    const uint8_t cls = __ldg(&a.cls[row]);
    const uint2 sm = live ? __ldg(&a.sexmask[g]) : make_uint2(0u, 0u);
    const uint32_t cs = live ? __ldg(&a.casemask[g]) : 0u;
    const uint32_t valid = sm.x | sm.y;
    uint32_t w = 0;
    if (live) {
        const uint4 t4 = __ldg(reinterpret_cast<const uint4*>(a.thr) + row);
        const uint32_t thr[4] = {t4.x, t4.y, t4.z, t4.w};
        uint32_t p1;
        draw_group_k(__ldg(&a.k[row]), g, a.row_base + row, a.k0, a.k1, thr, valid, w, p1);
    }
    s_w[tid] = w;
    __syncthreads();
    // forced minors, as in k_bed: the CTA walks the row's override list together
    const uint64_t o0 = s_ovr[0], o1 = s_ovr[1];
    if (o1 > o0) {
        const uint32_t s0 = tile * kGenoThreads * 16u;
        for (uint64_t o = o0 + tid; o < o1; o += kGenoThreads) {
            const uint32_t i = __ldg(&a.osamp[o]);
            const uint32_t li = i - s0;   // wraps for samples before this tile
            if (i < a.n && li < kGenoThreads * 16u) atomicOr(&s_w[li >> 4], 3u << (2u * (li & 15u)));
        }
        __syncthreads();
        w = s_w[tid];
    }
    constexpr uint32_t E = 0x55555555u;   // slot 0 of every cell
    uint32_t D = valid, H = 0u;
    if (cls == kX) D = sm.y, H = sm.x & E;
    else if (cls == kY) D = 0u, H = sm.x & E;
    else if (cls == kMT) D = 0u, H = valid & E;
    const uint32_t d0 = D & E, het = (w ^ (w >> 1)) & d0, hom = w & (w >> 1) & d0, halt = w & H;
    uint32_t c[kGenoWords] = {(uint32_t)__popc(d0 & cs),  (uint32_t)__popc(het & cs),  (uint32_t)__popc(hom & cs),
                              (uint32_t)__popc(H & cs),   (uint32_t)__popc(halt & cs),
                              (uint32_t)__popc(d0 & ~cs), (uint32_t)__popc(het & ~cs), (uint32_t)__popc(hom & ~cs),
                              (uint32_t)__popc(H & ~cs),  (uint32_t)__popc(halt & ~cs)};
#pragma unroll
    for (uint32_t j = 0; j < kGenoWords; ++j) c[j] = __reduce_add_sync(0xFFFFFFFFu, c[j]);
    if ((tid & 31u) == 0) {
#pragma unroll
        for (uint32_t j = 0; j < kGenoWords; ++j) s_sum[tid >> 5][j] = c[j];
    }
    __syncthreads();
    if (tid < kGenoWords) {
        uint32_t v = 0;
#pragma unroll
        for (uint32_t q = 0; q < kGenoThreads / 32; ++q) v += s_sum[q][tid];
        if (v) atomicAdd(&a.counts[(uint64_t)kGenoWords * rl + tid], v);
    }
}

// ------------------------------------------------------------------------------------------ Hardy-Weinberg exact P
// Two-sided exact test of Wigginton, Cutler & Abecasis (2005) (the SNPHWE definition plink --hardy reports): given
// n = n11 + n12 + n22 genotypes with r = 2 min(n11, n22) + n12 rare alleles, the het counts h = r mod 2, ..., r have
// probabilities p(h) proportional to n! / (h! hom_r! hom_c!) 2^h with hom_r = (r-h)/2, hom_c = n - h - hom_r, linked by
//   p(h+2) / p(h) = 4 hom_r hom_c / ((h+2)(h+1)).
// P = sum of p(h) over every h with p(h) <= p(n12) (1 + kHweTie) divided by the sum of all p(h).  The relative tie
// tolerance kHweTie makes the result independent of the order of the floating-point operations: terms equal to the
// observed one in exact arithmetic (a symmetric distribution) differ from it by a few ulps here.
// One thread runs the recurrence in double from the mode (term 1, so no term exceeds 1): first to the observed h for
// p(n12), then down and up from the mode for the sums; each tail stops once its terms are below p(n12)(1 + kHweTie)
// and below 2^-64 of the tail sum (the omitted terms shrink faster than geometrically).  When the walk to the observed
// h falls below 1e-295 / (terms), P < 1e-290 and 0 is returned.  n = 0: NaN (no test).
constexpr double kHweTie = 1e-7;

__device__ __forceinline__ double hwe_up(int64_t h, int64_t r, int64_t n) {       // p(h+2) / p(h)
    const int64_t hr = (r - h) >> 1, hc = n - h - hr;
    return 4.0 * (double)hr * (double)hc / ((double)(h + 2) * (double)(h + 1));
}
__device__ __forceinline__ double hwe_down(int64_t h, int64_t r, int64_t n) {     // p(h-2) / p(h)
    const int64_t hr = (r - h) >> 1, hc = n - h - hr;
    return (double)h * (double)(h - 1) / (4.0 * (double)(hr + 1) * (double)(hc + 1));
}

__device__ double hwe_exact_p(uint32_t n11, uint32_t n12, uint32_t n22) {
    const int64_t n = (int64_t)n11 + n12 + n22;
    if (n == 0) return __longlong_as_double(0x7FF8000000000000ll);   // NaN
    const int64_t r = 2 * (int64_t)min(n11, n22) + n12, obs = n12;
    int64_t m = (int64_t)((double)r * (double)(2 * n - r) / (double)(2 * n));   // near the mode (Wigginton's start)
    if ((m ^ r) & 1) ++m;
    m = min(m, r);
    while (m + 2 <= r && hwe_up(m, r, n) > 1.0) m += 2;
    while (m >= 2 && hwe_down(m, r, n) > 1.0) m -= 2;
    const double floor_p = 1e-295 / (double)(r / 2 + 1);
    double p_obs = 1.0;
    for (int64_t h = m; h < obs && p_obs >= floor_p; h += 2) p_obs *= hwe_up(h, r, n);
    for (int64_t h = m; h > obs && p_obs >= floor_p; h -= 2) p_obs *= hwe_down(h, r, n);
    if (p_obs < floor_p) return 0.0;
    const double thr = p_obs * (1.0 + kHweTie);
    double total = 1.0, tail = 1.0 <= thr ? 1.0 : 0.0;
    double t = 1.0;
    for (int64_t h = m; h >= 2; h -= 2) {
        t *= hwe_down(h, r, n);
        total += t;
        if (t <= thr) {
            tail += t;
            if (t <= tail * 0x1p-64) break;
        }
    }
    t = 1.0;
    for (int64_t h = m; h + 2 <= r; h += 2) {
        t *= hwe_up(h, r, n);
        total += t;
        if (t <= thr) {
            tail += t;
            if (t <= tail * 0x1p-64) break;
        }
    }
    return tail / total;
}

struct HweArgs {
    const uint32_t* counts;   // rows: [rows][10] of k_geno; triples: [items][3] = (n11, n12, n22)
    uint64_t items;           // rows: 3 * rows (ALL, AFF, UNAFF of every row); triples: items
    int rows;                 // layout of counts
    double* p;                // [items]
};

__global__ void __launch_bounds__(256) k_hwe(const HweArgs a) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.items) return;
    uint32_t n11, n12, n22;
    if (a.rows) {   // test 0 = ALL (cases + controls), 1 = AFF (cases), 2 = UNAFF (controls)
        const uint64_t row = i / 3;
        const uint32_t t = (uint32_t)(i - 3 * row);
        const uint32_t* c = a.counts + kGenoWords * row;
        const uint32_t dip = (t != 2 ? c[0] : 0u) + (t != 1 ? c[5] : 0u);
        n12 = (t != 2 ? c[1] : 0u) + (t != 1 ? c[6] : 0u);
        n11 = (t != 2 ? c[2] : 0u) + (t != 1 ? c[7] : 0u);
        n22 = dip - n12 - n11;
    } else {
        n11 = a.counts[3 * i];
        n12 = a.counts[3 * i + 1];
        n22 = a.counts[3 * i + 2];
    }
    a.p[i] = hwe_exact_p(n11, n12, n22);
}

}  // namespace dnaf
