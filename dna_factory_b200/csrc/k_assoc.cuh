// k_assoc: case/control allele counts per row straight from the allele draws (draw -> forced minors -> count), the
// input of the 1-df allelic association test (dnaf_allele_counts, dnaf_format_assoc).
//
// Counting rule (DESIGN.md 5, "Allelic association"): every allele the VCF text prints (pop_factory.py:481-499)
// counts once --
//   autosome: slots 0 and 1 of everybody     X: slot 0 of males, slots 0 and 1 of females
//   Y:        slot 0 of males, nothing of females ('.')              MT: slot 0 of everybody
// A forced minor sets both slots of its cell to ALT, so it counts as ALT on every slot of the cell that is counted
// (none on a female's Y cell).  With the draw word w of a 16-sample group (bit 2i+s = allele slot s of sample i, set
// = ALT; rows have K <= 2, checked by the host), the observed-slot mask `obs` of the row's class and the case bit
// pairs `cs`, the four counts of the group are
//   popcount(w & obs & cs), popcount(obs & cs), popcount(w & obs & ~cs), popcount(obs & ~cs).
// One CTA covers (row, 256 groups) like k_bed; its sums go to the pass's [row][4] array with one atomicAdd per
// counter (integer adds: the result does not depend on their order).
#pragma once
#include "k_bed.cuh"

namespace dnaf {

constexpr uint32_t kAssocThreads = 256;   // one thread per 16-sample word, one CTA per (row, 256 words)

struct AssocArgs {
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
    uint32_t tiles;           // CTAs per row: ceil(groups / kAssocThreads)
    uint32_t k0, k1;          // seed
    uint32_t* counts;         // [rows of the pass][4], zeroed before the launch; row 0 = row0
};

__global__ void __launch_bounds__(kAssocThreads) k_assoc(const AssocArgs a) {
    __shared__ uint32_t s_w[kAssocThreads];
    __shared__ uint64_t s_ovr[2];
    __shared__ uint4 s_sum[kAssocThreads / 32];
    const uint32_t rl = blockIdx.x / a.tiles, tile = blockIdx.x - rl * a.tiles;
    const uint64_t row = a.row0 + rl;
    const uint32_t tid = threadIdx.x;
    const uint32_t g = tile * kAssocThreads + tid;
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
        const uint32_t s0 = tile * kAssocThreads * 16u;
        for (uint64_t o = o0 + tid; o < o1; o += kAssocThreads) {
            const uint32_t i = __ldg(&a.osamp[o]);
            const uint32_t li = i - s0;   // wraps for samples before this tile
            if (i < a.n && li < kAssocThreads * 16u) atomicOr(&s_w[li >> 4], 3u << (2u * (li & 15u)));
        }
        __syncthreads();
        w = s_w[tid];
    }
    constexpr uint32_t E = 0x55555555u;   // slot 0 of every cell
    uint32_t obs = valid;
    if (cls == kX) obs = (sm.x & E) | sm.y;
    else if (cls == kY) obs = sm.x & E;
    else if (cls == kMT) obs = valid & E;
    const uint32_t alt = w & obs;
    uint32_t c0 = __popc(alt & cs), c1 = __popc(obs & cs), c2 = __popc(alt & ~cs), c3 = __popc(obs & ~cs);
    c0 = __reduce_add_sync(0xFFFFFFFFu, c0);
    c1 = __reduce_add_sync(0xFFFFFFFFu, c1);
    c2 = __reduce_add_sync(0xFFFFFFFFu, c2);
    c3 = __reduce_add_sync(0xFFFFFFFFu, c3);
    if ((tid & 31u) == 0) s_sum[tid >> 5] = make_uint4(c0, c1, c2, c3);
    __syncthreads();
    if (tid < 4) {
        uint32_t v = 0;
#pragma unroll
        for (uint32_t j = 0; j < kAssocThreads / 32; ++j) {
            const uint4 q = s_sum[j];
            v += tid == 0 ? q.x : tid == 1 ? q.y : tid == 2 ? q.z : q.w;
        }
        if (v) atomicAdd(&a.counts[4ull * rl + tid], v);
    }
}

}  // namespace dnaf
