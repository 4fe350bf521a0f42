// k_auto: the hot-path kernel for autosome rows with K <= 2 alleles (96 % of the bytes of a population).
// One CTA per BGZF block (a balanced segment of one row), one thread per span of 64 genotype cells.
// Allele draws -> (virtual) VCF text -> deflate tokens -> BGZF block; the text is never materialised.
//
// Reference behaviour restated: pop_factory.py:471-508 (row loop + row text), the BgzfWriter framing
// (call site pop_factory.py:449).
//
// Differences from the first fused kernel (k_fused.cuh, kept for the X / text kernels' shared pieces):
//   * tokens come from a BYTE lookup table: 8 allele slots (16 text bytes) per step instead of one mismatching
//     byte per step.  For a byte b of the span's allele mask m, the 10 bits  m'[8b .. 8b+10)  of
//     m' = (m << 2) | carry  determine every token between the first and the last mismatching text byte of those
//     16 bytes; the host stores that bit string per (Huffman table, 10-bit pattern).  The kernel only walks the
//     non-empty bytes, looks the interior up, and computes the one data-dependent token itself: the distance-4
//     match that bridges the gap since the previous mismatch.
//   * a span OWNS the separator that precedes its first cell and not the one that ends its last cell, so every
//     gap the loop sees has odd length (>= 3: a match, 1: that separator as a literal) -- no special cases
//   * no sorting of spans: the trip count is the number of non-empty mask bytes (<= 16), nearly equal within a row
//   * draws: two Philox calls per 32-slot group unconditionally, then one shared residual loop
//   * CRC32: the span-local linear CRC of the mask (16 lookups) is moved to the block end with 4 lookups into a
//     per-distance table instead of a 32-step GF(2) multiply; prefix CRCs come from a pre-kernel
#pragma once
#include "k_fused.cuh"

namespace dnaf {

constexpr int kAStage = 16;          // staged words per span before the block falls back to direct emission
#ifndef DNAF_LUT_MAX_BITS
#define DNAF_LUT_MAX_BITS 43
#endif
constexpr uint32_t kLutMaxBits = DNAF_LUT_MAX_BITS;   // interior bits a LUT entry can hold (a <= 21-bit match token rides along in 64)
constexpr uint32_t kLutLong = 1u << 17;               // flag of a LUT entry whose bit string does not fit

// Static code tables of one (MAF bucket, with/without prefix) pair.
struct AutoTable {
    // ---- first kATabWords words + the LUT are copied to shared memory by every block (bulk copies, 16-byte units)
    uint32_t len_tok[264];   // [g] token bridging g predicted bytes: 0 empty, 1 '\t' literal, 3..258 match; [259 + bit]: '/' + allele literal
    uint32_t lit[8];         // cell literals by id: code | bits << 24
    uint32_t eob;
    uint32_t hdr_bits;
    uint32_t hdr[62];        // serialized dynamic-block header
    uint2 lut[1024];         // x: code bits 0..31; y: code bits 32..42 | nbits << 11 | long << 17 | 2*first << 24 | (2*last+1) << 28
    uint32_t pre_lit[256];   // literal codes of prefix bytes
};
constexpr uint32_t kATabWords = 264 + 8 + 2 + 62;   // 336 words = 84 x 16 bytes
static_assert(kATabWords % 4 == 0 && sizeof(AutoTable) % 16 == 0, "AutoTable must copy in 16-byte units");

struct AutoArgs {
    SampleView sv;
    SnpView nv;
    const FusedDesc* desc;     // one per block, or NULL: the launch covers a run of autosome rows opening the pass and
                               // block b is segment b % nseg of row row0 + b / nseg, at slot b (no host planning, nothing to upload)
    uint64_t row0;
    uint32_t nseg;
    uint32_t nseg_magic;       // ceil(2^32 / nseg): block / nseg == umulhi(block, magic) while block * nseg < 2^32
    const uint32_t* seginfo;   // [nseg][3]: first cell, cells, template CRC of the segment
    const uint16_t* bucket;    // per row: MAF bucket (tables 2*bucket, 2*bucket + 1)
    const uint32_t* ovr_first; // [rows + 1]: first override of every row
    const AutoTable* tables;
    const uint32_t* etab;      // [16][256] span-local CRC contributions of mask bytes, measured to ONE BYTE BEFORE the span's cell end
    const uint32_t* mtab;      // [254][4][256] multiply by x^(8*256*j)
    const uint32_t* mtail;     // [4][256] multiply by x^(8*4*(n mod 64)) (rows whose last span is partial)
    const uint32_t* mpre;      // [2][4][256] multiply by x^(8*body bytes of segment 0): [0] segment does not end the row, [1] it does
    const uint32_t* crctab;    // [256]
    const uint32_t* xinit;     // [kBlk+1] 0xFFFFFFFF * x^(8n)
    const uint32_t* pre_crc;   // per row: linear CRC of the prefix
    const uint64_t* orow;
    const uint32_t* osamp;
    uint64_t row_base;
    uint32_t k0, k1;
    uint8_t* slots;
    uint32_t slot_stride;      // bytes per output slot of this pass (>= the longest block's text + 96)
    uint32_t* sizes;
    uint32_t* crcs;
};

// ---- span grammar (shared by the host's table builder, the LUT builder and the device slow paths) ----
// Own coordinates: byte q = 4*cell + {0,1,2,3}; byte -1 is the separator before the first cell.
//   first span of a block: ['\t' unless the block starts a row] a0 '/' a1, then prev_end = 3; else prev_end = -1
//   every mismatching allele byte 2s: [gap = 2s - prev_end predicted bytes][literal allele], prev_end = 2s + 1
//   tail: 4*nc - 1 - prev_end predicted bytes (even): 0 nothing, 2 -> '/' + allele literal, >= 4 one match
//   ['\n' if the span ends the row] [EOB if the span ends the block]
// Sink: tok(gap) (gap 0 -> nothing, >= 3 -> match), lit(id), eob().
template <class Sink>
__host__ __device__ inline void span_tokens_ref(const uint32_t m[4], uint32_t carry, bool first_in_block, bool starts_row,
                                                int nc, bool ends_row, bool ends_block, Sink& sink) {
    auto bit = [&](int s) { return (int)((pick4(m, s >> 5) >> (s & 31)) & 1u); };
    int prev_end = -1;
    int s0 = 0;
    if (first_in_block) {
        if (!starts_row) sink.lit(kLitTab);
        sink.lit(bit(0));
        sink.lit(kLitSlash);
        sink.lit(bit(1));
        prev_end = 3;
        s0 = 2;
    }
    for (int s = s0; s < 2 * nc; ++s) {
        const int prev = s >= 2 ? bit(s - 2) : (int)((carry >> s) & 1u);
        if (bit(s) == prev) continue;
        const int gap = 2 * s - prev_end;
        if (gap == 1) sink.lit((s & 1) ? kLitSlash : kLitTab);   // the separator between two mismatching alleles
        else sink.tok(gap);
        sink.lit(bit(s));
        prev_end = 2 * s + 1;
    }
    const int tail = 4 * nc - 1 - prev_end;
    if (tail == 2) {
        sink.lit(kLitSlash);
        sink.lit(bit(2 * nc - 1));
    } else if (tail) {
        sink.tok(tail);
    }
    if (ends_row) sink.lit(kLitNl);
    if (ends_block) sink.eob();
}

// ---- bit sinks ----
// Staging sink: appends up to 64 bits at a time to the thread's private words stage[k * stride] (word-interleaved
// across threads: conflict-free).  Branch-free: the three words an append can touch are stored every time.
template <int CAP>
struct AStageT {
    uint32_t* p;        // &stage[wi * stride + tid]
    uint32_t stride;    // in words
    uint32_t a0, nacc, wi;
    __device__ __forceinline__ void put64(uint32_t lo, uint32_t hi, uint32_t n) {   // n <= 64
        const uint32_t w0 = a0 | (lo << nacc);
        const uint32_t w1 = __funnelshift_l(lo, hi, nacc);
        const uint32_t w2 = __funnelshift_l(hi, 0u, nacc);
        if (wi < (uint32_t)CAP) {
            p[0] = w0;
            p[stride] = w1;
            p[2 * stride] = w2;
        }
        nacc += n;
        const uint32_t adv = nacc >> 5;
        uint32_t t01;
        asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\tselp.b32 %0, %2, %3, p;\n\t}" : "=r"(t01) : "r"(adv), "r"(w1), "r"(w0));
        asm("{\n\t.reg .pred p;\n\tsetp.gt.u32 p, %1, 1;\n\tselp.b32 %0, %2, %3, p;\n\t}" : "=r"(a0) : "r"(adv), "r"(w2), "r"(t01));
        wi += adv;
        p += adv * stride;
        nacc &= 31u;
    }
    // [token t1 (code | bits << 24)][c_lo:c_hi of nb bits], t1 bits + nb <= 64
    __device__ __forceinline__ void put_tok_code(uint32_t t1, uint32_t c_lo, uint32_t c_hi, uint32_t nb) {
        const uint32_t n1 = t1 >> 24;
        put64((t1 & 0xFFFFFFu) | (c_lo << n1), __funnelshift_l(c_lo, c_hi, n1), n1 + nb);
    }
    __device__ __forceinline__ uint32_t bits() const { return 32u * wi + nacc; }
};
using AStage = AStageT<kAStage>;

// Direct sink (a span overflowed its staging area): ORs the bits into the zeroed output words.
struct AEmit {
    uint32_t* words;
    uint32_t pos;
    __device__ void put64(uint32_t lo, uint32_t hi, uint32_t n) {
        if (!n) return;
        const uint32_t wi = pos >> 5, sh = pos & 31u;
        const uint32_t w0 = lo << sh, w1 = __funnelshift_l(lo, hi, sh), w2 = __funnelshift_l(hi, 0u, sh);
        if (w0) atomicOr(&words[wi], w0);
        if (w1) atomicOr(&words[wi + 1], w1);
        if (w2) atomicOr(&words[wi + 2], w2);
        pos += n;
    }
    __device__ void put_tok_code(uint32_t t1, uint32_t c_lo, uint32_t c_hi, uint32_t nb) {
        const uint32_t n1 = t1 >> 24;
        put64((t1 & 0xFFFFFFu) | (c_lo << n1), __funnelshift_l(c_lo, c_hi, n1), n1 + nb);
    }
};

// token-level adapter of a bit sink for span_tokens_ref-style slow paths
template <class Bits>
struct ATokSink {
    Bits& b;
    const uint32_t* len_tok;
    const uint32_t* lits;
    uint32_t eob_tok;
    __device__ void tok(int gap) { const uint32_t t = len_tok[gap]; b.put64(t & 0xFFFFFFu, 0u, t >> 24); }
    __device__ void lit(int id) { const uint32_t t = lits[id]; b.put64(t & 0xFFFFFFu, 0u, t >> 24); }
    __device__ void eob() { b.put64(eob_tok & 0xFFFFFFu, 0u, eob_tok >> 24); }
};

// The tokens of one span through the byte LUT.  mpb: the thread's 20 bytes of m' in shared memory.
template <class Bits>
__device__ __forceinline__ void emit_span(Bits& out, const uint2* __restrict__ lut, const uint32_t* __restrict__ len_tok,
                                          const uint32_t* __restrict__ lits, uint32_t eob_tok, const uint8_t* __restrict__ mpb,
                                          uint32_t nz, uint32_t m0, uint32_t mlast_bit, bool first_in_block, bool starts_row,
                                          int nc, bool ends_row, bool ends_block) {
    int prev_end = -1;
    if (first_in_block) {
        const uint32_t ta = lits[m0 & 1u], tb = lits[(m0 >> 1) & 1u], ts = lits[kLitSlash];
        uint32_t t1 = starts_row ? 0u : lits[kLitTab];
        // ['\t'] a0   then   '/' a1 : two <= 20-bit halves
        const uint32_t n1 = t1 >> 24;
        const uint32_t h1 = (t1 & 0xFFFFFFu) | ((ta & 0xFFFFFFu) << n1), h1n = n1 + (ta >> 24);
        const uint32_t h2 = (ts & 0xFFFFFFu) | ((tb & 0xFFFFFFu) << (ts >> 24)), h2n = (ts >> 24) + (tb >> 24);
        out.put_tok_code(h1 | (h1n << 24), h2, 0u, h2n);
        prev_end = 3;
    }
    while (nz) {
        const int b = __ffs((int)nz) - 1;
        nz &= nz - 1u;
        const uint32_t idx = (uint32_t)mpb[b] | (((uint32_t)mpb[b + 1] & 3u) << 8);
        const uint2 e = lut[idx];
        const uint32_t nb = (e.y >> 11) & 63u;
        const int pos = 16 * b;
        const int gap = pos + (int)((e.y >> 24) & 15u) - prev_end;
        const uint32_t t1 = len_tok[gap];
        if (!(e.y & kLutLong)) {
            out.put_tok_code(t1, e.x, e.y & 0x7FFu, nb);
        } else {
            // rare: the interior of this byte does not fit a LUT entry -- spell it out mismatch by mismatch
            out.put64(t1 & 0xFFFFFFu, 0u, t1 >> 24);
            const uint32_t mb = idx >> 2, xb = (mb ^ idx) & 0xFFu;   // idx = (m byte << 2) | carry: x = m ^ (m << 2 | carry)
            int pe = -1;
            for (int s = 0; s < 8; ++s) {
                if (!((xb >> s) & 1u)) continue;
                if (pe >= 0) {
                    const int g = 2 * s - pe;
                    const uint32_t t = g == 1 ? lits[(s & 1) ? kLitSlash : kLitTab] : len_tok[g];
                    out.put64(t & 0xFFFFFFu, 0u, t >> 24);
                }
                const uint32_t t = lits[(mb >> s) & 1u];
                out.put64(t & 0xFFFFFFu, 0u, t >> 24);
                pe = 2 * s + 1;
            }
        }
        prev_end = pos + (int)(e.y >> 28);
    }
    {
        const int tail = 4 * nc - 1 - prev_end;
        const uint32_t t1 = len_tok[tail == 2 ? 259 + (int)mlast_bit : tail];
        const uint32_t tn = ends_row ? lits[kLitNl] : 0u;
        const uint32_t te = ends_block ? eob_tok : 0u;
        const uint32_t nn = tn >> 24;
        out.put_tok_code(t1, (tn & 0xFFFFFFu) | ((te & 0xFFFFFFu) << nn), 0u, nn + (te >> 24));
    }
}

// 16-bit mask of the non-zero bytes of four words
__device__ __forceinline__ uint32_t nonzero_bytes(const uint32_t x[4]) {
    uint32_t nz = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        const uint32_t t = (((x[w] & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x[w]) & 0x80808080u;
        nz |= ((t * 0x00204081u) >> 28) << (4 * w);
    }
    return nz;
}

// compare four Philox words (bit depths d0 .. d0+3, MSB first) of one 32-slot group against the threshold
__device__ __forceinline__ void cmp_words(const uint4 r, uint32_t thr, uint32_t d0, uint32_t& eq, uint32_t& lt) {
    const uint32_t ww[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t mk = 0u - ((thr >> (31u - (d0 + i))) & 1u);
        const uint32_t d = eq & (ww[i] ^ mk);
        lt |= d & mk;
        eq &= ~d;
    }
}

// Linear CRC of every row prefix (register starts at 0, no final xor), and the set of byte values that occur in
// the prefixes (the code tables must hold a literal for each); run once per set_snps.
// state: [0..7] presence bits, [8] blocks finished (zeroed by the host); the last block stores the set to
// host_present (mapped page-locked memory), so that no DMA read-back is needed.
__global__ void __launch_bounds__(256) k_prefix_crc(const uint8_t* __restrict__ prefix, const uint64_t* __restrict__ pre_off,
                                                   uint64_t n_rows, const uint32_t* __restrict__ crctab,
                                                   uint32_t* __restrict__ out, uint32_t* __restrict__ state,
                                                   volatile uint32_t* __restrict__ host_present) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t seen[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (r < n_rows) {
        uint32_t c = 0;
        for (uint64_t i = pre_off[r]; i < pre_off[r + 1]; ++i) {
            const uint32_t v = prefix[i];
            c = __ldg(&crctab[(c ^ v) & 0xFFu]) ^ (c >> 8);
#pragma unroll
            for (int w = 0; w < 8; ++w)
                if ((v >> 5) == (uint32_t)w) seen[w] |= 1u << (v & 31u);
        }
        out[r] = c;
    }
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        const uint32_t m = __reduce_or_sync(0xFFFFFFFFu, seen[w]);
        if ((threadIdx.x & 31u) == 0 && m) atomicOr(&state[w], m);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&state[8], 1u) + 1u == gridDim.x) {
            __threadfence();
            for (int w = 0; w < 8; ++w) host_present[w] = *reinterpret_cast<volatile uint32_t*>(&state[w]);
            __threadfence_system();
        }
    }
}

__device__ __forceinline__ uint32_t mul_tab(const uint32_t* __restrict__ t, uint32_t v) {   // t: [4][256]
    return __ldg(&t[v & 0xFFu]) ^ __ldg(&t[256u + ((v >> 8) & 0xFFu)]) ^ __ldg(&t[512u + ((v >> 16) & 0xFFu)]) ^
           __ldg(&t[768u + (v >> 24)]);
}

// dynamic shared memory carve-up, nthr = blockDim.x
__host__ __device__ inline uint32_t auto_smem_bytes(uint32_t nthr) {
    return 8192u + kATabWords * 4u + ((uint32_t)(kAStage + 2) * nthr + nthr + 24u) * 4u + 20u * nthr + 16u;
}

// 1-D bulk copy global -> shared (cp.async.bulk, the TMA engine): 16-byte aligned both sides, size a multiple of 16;
// the bytes are counted on the mbarrier at `mbar` (shared-window address)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(mbar)
                 : "memory");
}

// Wait for phase `parity` of an mbarrier (try_wait sleeps in hardware); a copy that never lands traps instead of hanging.
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    for (uint32_t spins = 0;; ++spins) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(mbar), "r"(parity)
                     : "memory");
        if (ok) return;
        if (spins > (1u << 20)) __trap();
    }
}

// The 128 allele bits of one span (64 cells from cell `cs`, nc of them real): replay-stream draws (dnaf_device.cuh) and the
// forced-minor cells of the row (pop_factory.py:495-499).  Shared by k_auto and k_lz.
__device__ __forceinline__ void auto_draw_span(const AutoArgs& a, const FusedDesc& d, uint32_t cs, int nc, uint32_t m[4]) {
    if (nc > 0 && a.nv.k[d.row] == 2) {
        const uint32_t thr = a.nv.thr[d.row * 4];
        const uint64_t prow = a.row_base + d.row;
        const uint32_t r_lo = (uint32_t)prow, r_hi = (uint32_t)(prow >> 32);
        const uint32_t g0 = cs >> 4;
        uint32_t eq[4], lt[4];
        const int slots0 = (int)(2u * a.sv.n) - (int)(32u * g0);   // allele slots from this span's first group to the row's end
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            // lanes beyond the last sample start out decided ("U <= T": reference allele, mask bit 0)
            eq[w] = __funnelshift_lc(0xFFFFFFFFu, 0u, (uint32_t)max(slots0 - 32 * w, 0));
            lt[w] = ~eq[w];
        }
        // the first 8 bits of every lane decide 99.6 % of them: two calls per group, no divergence
#pragma unroll
        for (uint32_t q = 0; q < 2; ++q)
#pragma unroll
            for (int w = 0; w < 4; ++w) cmp_words(philox4x32_10(g0 + w, q, r_lo, r_hi, a.k0, a.k1), thr, 4u * q, eq[w], lt[w]);
        // residual: one call per trip on the first group of this thread that still has an undecided lane, groups in
        // order, calls q = 2..7 in order.  That group is rotated into slot 0 (decided groups go to the back), so that
        // no array is indexed by a runtime group number: such an index puts eq / lt in local memory.
        uint32_t rot = 0, q = 2;   // slot 0 holds group g0 + rot; q: its next call
        for (;;) {
            if (!(eq[0] | eq[1])) {
                uint32_t t = eq[0]; eq[0] = eq[2]; eq[2] = t; t = eq[1]; eq[1] = eq[3]; eq[3] = t;
                t = lt[0]; lt[0] = lt[2]; lt[2] = t; t = lt[1]; lt[1] = lt[3]; lt[3] = t;
                rot += 2; q = 2;
            }
            if (!eq[0]) {
                uint32_t t = eq[0]; eq[0] = eq[1]; eq[1] = eq[2]; eq[2] = eq[3]; eq[3] = t;
                t = lt[0]; lt[0] = lt[1]; lt[1] = lt[2]; lt[2] = lt[3]; lt[3] = t;
                rot += 1; q = 2;
            }
            if (!eq[0]) break;   // every group decided
            cmp_words(philox4x32_10(g0 + rot, q, r_lo, r_hi, a.k0, a.k1), thr, 4u * q, eq[0], lt[0]);
            if (q == 7u) {   // all 32 bits compared: lanes still equal have U == T, i.e. U <= T
                lt[0] |= eq[0];
                eq[0] = 0;
            }
            ++q;
        }
        // every eq is 0 now; rotate lt back by rot (mod 4)
        if (rot & 2u) {
            uint32_t t = lt[0]; lt[0] = lt[2]; lt[2] = t; t = lt[1]; lt[1] = lt[3]; lt[3] = t;
        }
        if (rot & 1u) {
            const uint32_t t = lt[3]; lt[3] = lt[2]; lt[2] = lt[1]; lt[1] = lt[0]; lt[0] = t;
        }
#pragma unroll
        for (int w = 0; w < 4; ++w) m[w] = ~lt[w];   // U <= T -> reference allele
    }
    // forced-minor cells (pop_factory.py:495-499)
    if (nc > 0) {
        for (uint32_t o = 0; o < d.ovr_count; ++o) {
            const uint32_t i = a.osamp[d.ovr_first + o];
            if (i >= cs && i < cs + (uint32_t)nc) {
                const uint32_t j = 2u * (i - cs);
                const uint32_t bit = 3u << (j & 31u);
                // selects, not m[j >> 5]: an indexed m lives in local memory for the whole kernel
#pragma unroll
                for (int w = 0; w < 4; ++w) m[w] |= (j >> 5) == (uint32_t)w ? bit : 0u;
            }
        }
    }
}

// CRC32 share of one span: the span-local linear CRC of its allele mask, moved to the end of the block's cells.
// Two halves, so that a caller can issue the loads early and consume them late: _gather reads the E table and issues
// the four lookups of the multiply table (1 MB, from L2), _finish XORs them and applies the short-last-span move.
struct SpanCrc {
    uint32_t t[4];   // mtab lookups of the span-local CRC's bytes; all 0 when the span has no share
    bool tail;       // the span's share still moves across the block's short last span
};

__device__ __forceinline__ SpanCrc auto_span_crc_gather(const AutoArgs& a, const FusedDesc& d, const uint32_t m[4], int nc,
                                                        uint32_t tid, uint32_t nspans) {
    // ---- CRC32 share of this span: template ^ delta (affine); delta's span-local CRC moved to the block end
    SpanCrc c{{0u, 0u, 0u, 0u}, false};
    const bool partial_tail = (d.ncells & 63u) != 0u;   // the block's last span is short
    if (nc > 0 && (m[0] | m[1] | m[2] | m[3])) {
        uint32_t mm[4] = {m[0], m[1], m[2], m[3]};
        if (nc < 64) {  // partial last span: align its end with the table's span end (128-bit left shift)
            const uint32_t sh = 2u * (64u - (uint32_t)nc);
            const uint32_t ws = sh >> 5, bs = sh & 31u;
#pragma unroll
            for (int k = 0; k < 3; ++k)
                if (ws > (uint32_t)k) { mm[3] = mm[2]; mm[2] = mm[1]; mm[1] = mm[0]; mm[0] = 0; }
            mm[3] = __funnelshift_l(mm[2], mm[3], bs);
            mm[2] = __funnelshift_l(mm[1], mm[2], bs);
            mm[1] = __funnelshift_l(mm[0], mm[1], bs);
            mm[0] = mm[0] << bs;
        }
        uint32_t sp = 0;
#pragma unroll
        for (int w = 0; w < 4; ++w)
#pragma unroll
            for (int k = 0; k < 4; ++k) sp ^= __ldg(&a.etab[(4 * w + k) * 256 + ((mm[w] >> (8 * k)) & 0xFFu)]);
        // whole spans between the end of this span's cells and the end of the block's cells (mtab + 0 multiplies by
        // 1: the last span's share, and the one before a short last span, are sp itself), then the short last span
        const uint32_t last = nspans - 1u;
        const uint32_t j = tid == last ? 0u : (partial_tail ? last - 1u - tid : last - tid);
        const uint32_t* t = a.mtab + (size_t)j * 1024u;
#pragma unroll
        for (int k = 0; k < 4; ++k) c.t[k] = __ldg(&t[256 * k + ((sp >> (8 * k)) & 0xFFu)]);
        c.tail = partial_tail && tid != last;
    }
    return c;
}

__device__ __forceinline__ uint32_t auto_span_crc_finish(const AutoArgs& a, const SpanCrc& c) {
    const uint32_t crc = c.t[0] ^ c.t[1] ^ c.t[2] ^ c.t[3];
    return c.tail ? mul_tab(a.mtail, crc) : crc;
}

__device__ __forceinline__ uint32_t auto_span_crc(const AutoArgs& a, const FusedDesc& d, const uint32_t m[4], int nc, uint32_t tid,
                                                  uint32_t nspans) {
    return auto_span_crc_finish(a, auto_span_crc_gather(a, d, m, nc, tid, nspans));
}

#ifndef DNAF_AUTO_REGS
#define DNAF_AUTO_REGS 56   // 7 blocks of 160 threads per SM; 64 (6 blocks) and 48 (spills) measured slower
#endif
__global__ void __maxnreg__(DNAF_AUTO_REGS) k_auto(const AutoArgs a) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31u, wid = tid >> 5;
    uint2* s_lut = reinterpret_cast<uint2*>(smem_raw);
    uint32_t* s_len = reinterpret_cast<uint32_t*>(s_lut + 1024);   // len_tok | lit | eob | hdr_bits | hdr
    uint32_t* s_stage = s_len + kATabWords;
    uint32_t* s_last2 = s_stage + (kAStage + 2) * nthr;
    uint32_t* s_misc = s_last2 + nthr;      // [0..7] warp span bits, [8..9] warp prefix bits, [10] constant crc terms, [16] crc, [17] overflow
    uint8_t* s_mp = reinterpret_cast<uint8_t*>(s_misc + 24);
    const uint32_t* s_lits = s_len + 264;
    const uint32_t* s_hdr = s_len + 274;

    FusedDesc d;
    if (a.desc) {
        d = a.desc[blockIdx.x];
    } else {
        const uint32_t rl = a.nseg_magic ? __umulhi(blockIdx.x, a.nseg_magic) : blockIdx.x, sg = blockIdx.x - rl * a.nseg;   // magic 0: one segment per row
        d.row = a.row0 + rl;
        d.cell0 = __ldg(&a.seginfo[3u * sg]);
        d.ncells = __ldg(&a.seginfo[3u * sg + 1u]);
        d.body_crc = __ldg(&a.seginfo[3u * sg + 2u]);
        d.slot = blockIdx.x;
        d.flags = (sg == 0u ? 1u : 0u) | (sg + 1u == a.nseg ? 2u : 0u);
        d.ovr_first = __ldg(&a.ovr_first[d.row]);
        d.ovr_count = __ldg(&a.ovr_first[d.row + 1]) - d.ovr_first;
        d.table = 2u * __ldg(&a.bucket[d.row]) + (sg == 0u ? 0u : 1u);
    }
    const AutoTable* __restrict__ tb = a.tables + d.table;
    // code tables of this block's bucket -> shared memory by two bulk copies (TMA, one thread issues them) that land
    // under the draws; completion is counted in bytes on an mbarrier every thread waits on before the token pass
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(s_misc + 22);   // 8-byte aligned: nthr is a multiple of 32
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"(8192u + kATabWords * 4u) : "memory");
        bulk_g2s(s_lut, tb->lut, 8192u, mbar);
        bulk_g2s(s_len, tb->len_tok, kATabWords * 4u, mbar);
    }
    if (tid == 6) { s_misc[16] = 0; s_misc[17] = 0; }
    const bool starts_row = d.flags & 1u, ends_row = (d.flags >> 1) & 1u;
    const uint32_t nspans = (d.ncells + 63u) / 64u;

    // ---- draw this span's 128 allele bits (replay RNG spec: dnaf_device.cuh)
    const uint32_t cs = d.cell0 + 64u * tid;
    int nc = 0;
    if (tid < nspans) nc = (int)min(64u, d.ncells - 64u * tid);
    uint32_t m[4] = {0, 0, 0, 0};
    auto_draw_span(a, d, cs, nc, m);
    const SpanCrc crc_part = auto_span_crc_gather(a, d, m, nc, tid, nspans);
    // the prefix is read after the draws: live across them, its offsets pushed the draw loop into spills
    const uint64_t pb = a.nv.pre_off[d.row];
    const uint32_t plen = starts_row ? (uint32_t)(a.nv.pre_off[d.row + 1] - pb) : 0u;
    // text bytes of this block: [prefix | the separator that ended the previous segment] cells, minus the last
    // separator unless the row ends here
    const uint32_t lead = starts_row ? plen : 1u;
    const uint32_t n = lead + 4u * d.ncells - (ends_row ? 0u : 1u);
    // prefix literal of this thread (blocks that start a row)
    uint32_t pre_tok = 0;
    if (tid < plen) pre_tok = __ldg(&tb->pre_lit[a.nv.prefix[pb + tid]]);
    if (tid == 0) {   // the terms that do not depend on the draws: init, prefix, all-reference template
        uint32_t c0 = d.body_crc ^ __ldg(&a.xinit[n]);
        if (starts_row) c0 ^= mul_tab(ends_row ? a.mpre + 1024 : a.mpre, __ldg(&a.pre_crc[d.row]));
        s_misc[10] = c0;
    }

    // ---- m' = (m << 2) | carry in shared memory, mismatch bytes
    // slots past the span's last cell repeat that cell, so that they never mismatch
    uint32_t mp[4] = {m[0], m[1], m[2], m[3]};
    if (nc > 0 && nc < 64) {
        const int s = 2 * nc - 2;
        const uint32_t l2 = (pick4(m, s >> 5) >> (s & 31)) & 3u;
        const uint32_t pat = ((l2 & 1u) ? 0x55555555u : 0u) | ((l2 & 2u) ? 0xAAAAAAAAu : 0u);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int lo = 2 * nc - 32 * w;  // slots of this word that exist
            const uint32_t keep = lo >= 32 ? 0xFFFFFFFFu : (lo <= 0 ? 0u : ((1u << lo) - 1u));
            mp[w] = (m[w] & keep) | (pat & ~keep);
        }
    }
    s_last2[tid] = mp[3] >> 30;
    __syncthreads();        // also orders the mbarrier's initialisation before the waits
    mbar_wait(mbar, 0u);    // the code tables have landed
    const uint32_t carry = tid ? s_last2[tid - 1] : (mp[0] & 3u);
    uint32_t nz = 0;
    if (nc > 0) {
        uint32_t q[5];
        q[0] = (mp[0] << 2) | carry;
        q[1] = __funnelshift_l(mp[0], mp[1], 2);
        q[2] = __funnelshift_l(mp[1], mp[2], 2);
        q[3] = __funnelshift_l(mp[2], mp[3], 2);
        q[4] = mp[3] >> 30;
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_mp + 20u * tid);
#pragma unroll
        for (int k = 0; k < 5; ++k) dst[k] = q[k];
        const uint32_t x[4] = {mp[0] ^ q[0], mp[1] ^ q[1], mp[2] ^ q[2], mp[3] ^ q[3]};
        nz = nonzero_bytes(x);
    }
    // ---- pass 1: this span's tokens, staged privately
    const uint32_t eob = s_len[272];
    const bool worker = nc > 0;
    const bool p_last = worker && 64u * tid + (uint32_t)nc == d.ncells;
    const bool p_end = ends_row && p_last;
    const uint32_t mlast_bit = worker ? (pick4(m, (2 * nc - 1) >> 5) >> ((2 * nc - 1) & 31)) & 1u : 0u;
    AStage st{s_stage + tid, nthr, 0u, 0u, 0u};
    if (worker) {
        emit_span(st, s_lut, s_len, s_lits, eob, s_mp + 20u * tid, nz, mp[0], mlast_bit, tid == 0, starts_row, nc, p_end, p_last);
        if (st.bits() > 32u * kAStage) s_misc[17] = 1;
    }
    // the CRC share is consumed only now: its mtab lookups (L2), issued before the first barrier, land under the token
    // pass instead of holding the CTA at that barrier; XOR is order-free and the trailer reads s_misc[16] two barriers on
    const uint32_t crc = warp_xor(auto_span_crc_finish(a, crc_part));
    if (lane == 0 && crc) atomicXor(&s_misc[16], crc);
    // ---- exclusive scans over the CTA: prefix literal bits (warps 0-1) and span bits
    const uint32_t pre_bits = pre_tok >> 24;
    const uint32_t my_bits = worker ? st.bits() : 0u;
    uint32_t v0 = pre_bits, v1 = my_bits;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u1 = __shfl_up_sync(0xFFFFFFFFu, v1, o);
        if (lane >= (uint32_t)o) v1 += u1;
    }
    if (wid < 2) {
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u0 = __shfl_up_sync(0xFFFFFFFFu, v0, o);
            if (lane >= (uint32_t)o) v0 += u0;
        }
    }
    if (lane == 31u) {
        s_misc[wid] = v1;
        if (wid < 2) s_misc[8 + wid] = v0;
    }
    __syncthreads();
    uint32_t span_off = v1 - my_bits, total_span = 0;
    const uint32_t nw = nthr >> 5;
    for (uint32_t w = 0; w < nw; ++w) {
        const uint32_t t = s_misc[w];
        if (w < wid) span_off += t;
        total_span += t;
    }
    const uint32_t total_pre = plen ? s_misc[8] + s_misc[9] : 0u;   // plen <= 64: two warps
    const uint32_t pre_off = v0 - pre_bits + (wid == 1 ? s_misc[8] : 0u);
    const uint32_t hdr_bits = s_len[273];
    const uint32_t data_bits = hdr_bits + total_pre + total_span;
    const uint32_t payload = (data_bits + 7u) / 8u;
    const uint32_t out_words = (data_bits + 31u) / 32u;
    const bool stored = payload > n + 5u;  // cannot happen with sane tables; keeps BSIZE <= 64 KiB regardless
    uint8_t* blk = a.slots + (uint64_t)d.slot * a.slot_stride + kSlotLead;
    uint32_t* words = reinterpret_cast<uint32_t*>(blk + 18);  // 16-byte aligned

    uint32_t out_payload;
    if (!stored) {
        // header words are written, the words after them zeroed (they are OR-ed into)
        const uint32_t hdr_words = (hdr_bits + 31u) / 32u;
        const uint32_t hw4 = (hdr_words + 3u) & ~3u;   // <= 64 <= nthr
        if (tid < hw4) words[tid] = tid < hdr_words ? s_hdr[tid] : 0u;
        const bool overflow = s_misc[17] != 0;   // final: pass 1 ended before the scan's barrier
        const uint32_t ppos = hdr_bits + pre_off;                 // first bit of this thread's prefix literal
        const uint32_t dst = hdr_bits + total_pre + span_off;     // first bit of this span in the block
        if (overflow) {   // the slow pass 2 ORs every word
            uint4* w4 = reinterpret_cast<uint4*>(words + hw4);
            const uint32_t n4 = out_words + 2u > hw4 ? (out_words + 2u - hw4 + 3u) / 4u : 0u;
            for (uint32_t i = tid; i < n4; i += nthr) w4[i] = make_uint4(0u, 0u, 0u, 0u);
        } else {
            // Only words that two writers share are OR-ed into -- the words of the prefix literals and the first and last
            // word of every span; words in between belong to one span and are stored whole.  Zero just those (the words
            // up to hw4 are initialised by the header store above).
            if (pre_bits) {
                const uint32_t wi = ppos >> 5;
                if (wi >= hw4) words[wi] = 0u;
                if (wi + 1u >= hw4) words[wi + 1u] = 0u;
            }
            if (worker) {
                const uint32_t first = dst >> 5, last = (dst + my_bits - 1u) >> 5;
                if (first >= hw4) words[first] = 0u;
                if (last >= hw4) words[last] = 0u;
            }
        }
        __syncthreads();
        if (pre_bits) {  // prefix literal: at most 15 bits
            const uint32_t wi = ppos >> 5, sh = ppos & 31u, v = pre_tok & 0xFFFFFFu;
            atomicOr(&words[wi], v << sh);
            if (sh + pre_bits > 32) atomicOr(&words[wi + 1], v >> (32 - sh));
        }
        if (worker) {
            if (!overflow) {
                // ---- pass 2 (fast): move the staged bits to their final position; only the first and the last
                // destination word can be shared with a neighbour
                const uint32_t sh = dst & 31u;
                const uint32_t nsrc = (my_bits + 31u) / 32u;
                const uint32_t ndst = (sh + my_bits + 31u) / 32u;
                uint32_t* o = words + (dst >> 5);
                const uint32_t* sp = s_stage + tid;
                uint32_t prev = my_bits ? sp[0] : 0u;
                atomicOr(&o[0], prev << sh);
                uint32_t k = 1;
                for (; k + 1u < ndst; ++k) {
                    const uint32_t cur = sp[k * nthr];
                    o[k] = __funnelshift_l(prev, cur, sh);
                    prev = cur;
                }
                if (k < ndst) {
                    const uint32_t cur = k < nsrc ? sp[k * nthr] : 0u;
                    atomicOr(&o[k], __funnelshift_l(prev, cur, sh));
                }
            } else {
                // ---- pass 2 (slow): some span overflowed its staging words -- emit straight into the output words
                AEmit em{words, dst};
                ATokSink<AEmit> ts{em, s_len, s_lits, eob};
                span_tokens_ref(mp, carry, tid == 0, starts_row, nc, p_end, p_last, ts);
            }
        }
        out_payload = payload;
    } else {
        // stored deflate block: format the text itself (rare safety net)
        if (tid == 0) {
            blk[18] = 1;
            blk[19] = (uint8_t)n; blk[20] = (uint8_t)(n >> 8);
            blk[21] = (uint8_t)~n; blk[22] = (uint8_t)((~n) >> 8);
            if (!starts_row) blk[23] = '\t';
        }
        if (tid < plen) blk[23 + tid] = a.nv.prefix[pb + tid];
        if (nc > 0) {
            uint8_t* p = blk + 23 + lead + 256u * tid;
            for (int c = 0; c < nc; ++c) {
                const uint32_t bits = (pick4(m, c >> 4) >> (2 * (c & 15))) & 3u;
                p[4 * c] = '0' + (bits & 1u);
                p[4 * c + 1] = '/';
                p[4 * c + 2] = '0' + (bits >> 1);
                if (!(p_last && c == nc - 1)) p[4 * c + 3] = '\t';
                else if (ends_row) p[4 * c + 3] = '\n';
            }
        }
        out_payload = n + 5u;
    }
    __syncthreads();
    if (tid < 26) {  // 18-byte BGZF header, CRC32, ISIZE
        // the E table measures distances to one byte before the cell boundary, where blocks that do not end the row
        // stop; a block that ends the row is one byte ('\n') longer
        uint32_t delta = s_misc[16];
        if (ends_row) delta = __ldg(&a.crctab[delta & 0xFFu]) ^ (delta >> 8);
        const uint32_t crc32 = ~(delta ^ s_misc[10]);
        const uint32_t bsize = out_payload + 25u;
        if (tid < 16) {   // 1f 8b 08 04 | 00 00 00 00 | 00 ff 06 00 | 42 43 02 00, from words (an indexed byte array is local memory)
            const uint32_t hw = tid < 4u ? 0x04088b1fu : (tid < 8u ? 0u : (tid < 12u ? 0x0006ff00u : 0x00024342u));
            blk[tid] = (uint8_t)(hw >> (8u * (tid & 3u)));
        } else if (tid < 18) {
            blk[tid] = (uint8_t)(bsize >> (8 * (tid - 16)));
        } else if (tid < 22) {
            blk[18 + out_payload + (tid - 18)] = (uint8_t)(crc32 >> (8 * (tid - 18)));
        } else {
            blk[18 + out_payload + (tid - 18)] = (uint8_t)(n >> (8 * (tid - 22)));
        }
        if (tid == 0) {
            a.sizes[d.slot] = out_payload + 26u;
            a.crcs[d.slot] = crc32;
        }
    }
}

}  // namespace dnaf
