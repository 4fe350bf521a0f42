// k_bed: PLINK 1 .bed genotype matrix straight from the allele draws (draw -> forced minors -> encode -> store).
//
// Encoding (DESIGN.md 5, "PLINK 1 fileset"):
//   * the file is the magic 6C 1B 01 (SNP-major), then per row in VCF order B = ceil(N/4) bytes; sample i sits in
//     byte i/4, bits 2(i%4) (low) and 2(i%4)+1 (high); the padding bits of a row's last byte are 0.  The library
//     writes the rows only, like dnaf_generate writes no VCF header.
//   * the 2-bit value counts ALT copies, with .bim A1 = ALT and A2 = REF (plink2's default, plink 1.9
//     --keep-allele-order): 2 copies -> 0, 1 copy -> 2, 0 copies -> 3, missing -> 1.
//   * cells follow the VCF text rules (pop_factory.py:481-499): haploid cells (X and Y for males, MT for everybody)
//     use slot 0 only and are written homozygous; females on Y are missing; forced minors are two ALT copies, except on
//     a female's Y cell, which stays missing ('.' wins, as in k_overrides -> k_format).
//
// The draw word of one group of 16 samples (draw_group, bit 2i+s = allele slot s of sample i) and the .bed codes of
// the same 16 samples are both one 32-bit word, 4 little-endian bytes in the same sample order.  With E = 0x55555555:
//   lo = ~(w | w >> 1) & E       (0 ALT copies, or missing after the mask below)
//   hi = (~(w & w >> 1) & E) << 1    (fewer than 2 ALT copies)
// Rows with K > 2 cannot be written in PLINK 1; the host refuses them before any launch.
#pragma once
#include "dnaf_device.cuh"

namespace dnaf {

constexpr uint32_t kBedThreads = 256;   // one thread per 16-sample word, one CTA per (row, 256 words)

struct BedArgs {
    const uint8_t* cls;       // chromosome class per row
    const uint8_t* k;         // alleles per row (<= 2: checked by the host)
    const uint32_t* thr;      // [row][4]
    const uint2* sexmask;     // per 16-sample group: x = bit pairs of the males, y = of the females (dnaf_set_samples)
    const uint64_t* orow;     // override pairs, sorted by row
    const uint32_t* osamp;
    uint64_t n_over;
    uint64_t row0;            // first row of the pass
    uint64_t row_base;        // Philox row counter = row_base + row
    uint32_t n;               // samples
    uint32_t groups;          // ceil(n / 16)
    uint32_t tiles;           // CTAs per row: ceil(groups / kBedThreads)
    uint32_t pitch;           // bytes per row: ceil(n / 4)
    uint32_t k0, k1;          // seed
    uint8_t* out;             // rows x pitch bytes, row 0 = row0
};

__device__ __forceinline__ uint64_t bed_lower_bound(const uint64_t* __restrict__ v, uint64_t n, uint64_t key) {
    uint64_t lo = 0;
    while (n) {
        const uint64_t h = n >> 1;
        if (__ldg(&v[lo + h]) < key) {
            lo += h + 1;
            n -= h + 1;
        } else {
            n = h;
        }
    }
    return lo;
}

__global__ void __launch_bounds__(kBedThreads) k_bed(const BedArgs a) {
    __shared__ uint32_t s_w[kBedThreads];
    __shared__ uint64_t s_ovr[2];
    const uint32_t rl = blockIdx.x / a.tiles, tile = blockIdx.x - rl * a.tiles;
    const uint64_t row = a.row0 + rl;
    const uint32_t tid = threadIdx.x;
    const uint32_t g = tile * kBedThreads + tid;
    const bool live = g < a.groups;
    // the row's forced minors: [first override of row, first override of row + 1) in the sorted list
    if (tid < 2) s_ovr[tid] = bed_lower_bound(a.orow, a.n_over, row + tid);
    const uint8_t cls = __ldg(&a.cls[row]);
    const uint2 sm = live ? __ldg(&a.sexmask[g]) : make_uint2(0u, 0u);
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
    // forced minors, applied to the draw words before encoding.  All threads of the CTA share the row's list, so a row
    // with thousands of overrides (deleterious SNPs at the C4 shape) costs count / 256 trips, not count.
    const uint64_t o0 = s_ovr[0], o1 = s_ovr[1];
    if (o1 > o0) {
        const uint32_t s0 = tile * kBedThreads * 16u;
        for (uint64_t o = o0 + tid; o < o1; o += kBedThreads) {
            const uint32_t i = __ldg(&a.osamp[o]);
            const uint32_t li = i - s0;   // wraps for samples before this tile
            if (i < a.n && li < kBedThreads * 16u) atomicOr(&s_w[li >> 4], 3u << (2u * (li & 15u)));
        }
        __syncthreads();
        w = s_w[tid];
    }
    if (!live) return;
    constexpr uint32_t E = 0x55555555u;
    uint32_t hap = 0, miss = 0;
    if (cls == kX) hap = sm.x;
    else if (cls == kY) { hap = sm.x; miss = sm.y; }
    else if (cls == kMT) hap = valid;
    const uint32_t s0bits = w & hap & E;           // slot 0 of the haploid cells, copied to slot 1: homozygous
    w = (w & ~hap) | s0bits | (s0bits << 1);
    uint32_t code = (~(w | (w >> 1)) & E) | ((~(w & (w >> 1)) & E) << 1);
    code = (code & ~miss) | (miss & E);            // missing = 01
    code &= valid;                                 // padding bits of the last byte are 0
    uint8_t* dst = a.out + (uint64_t)rl * a.pitch + 4ull * g;
    if ((a.pitch & 3u) == 0) {                     // rows are word aligned (N = 20 000, 100 000, ...): 4g + 4 <= pitch
        *reinterpret_cast<uint32_t*>(dst) = code;
    } else {
        const uint32_t nb = min(4u, a.pitch - 4u * g);
        for (uint32_t b = 0; b < nb; ++b) dst[b] = (uint8_t)(code >> (8u * b));
    }
}

}  // namespace dnaf
