// k_x: fused kernel for X-chromosome rows (K <= 2), the byte-LUT design of k_auto carried over to rows whose cells
// have two widths.
//
// On X a male prints "a\t" (2 bytes, slot 2i only) and a female "a/b\t" (4 bytes) -- pop_factory.py:488-494,
// common/snp.py:109.  In the COMPACTED allele sequence c[k] (slots of the row with the unused second slot of males
// removed) the text is  c[0] S[0] c[1] S[1] ...  with S[k] in {'/', '\t'} fixed by the sex vector alone, and under
// the byte-4-back predictor
//     byte 2k   mismatches  <=>  c[k] != c[k-2]          (data)
//     byte 2k+1 mismatches  <=>  S[k] != S[k-2]          (static per population)
// A UNIT is four compacted positions = 8 text bytes.  Its tokens depend only on 6 allele bits c[4u-2 .. 4u+3] and
// 6 separator bits S[4u-2 .. 4u+3]: a 4096-entry table per Huffman code (in L2; the separator half of the key is
// precomputed per span).  Entries are normalised so that the gap a unit leaves to its neighbours is never 1 or 2
// bytes (those bytes are spelled out as literals inside the entry): the kernel only ever bridges gaps of 0 or >= 3
// bytes, one match token, with no data-dependent literal of its own.  The positions after a span's last whole
// unit (0..3, plus the '\n' that ends a row) go through a short event-by-event tail.
//
// Reference behaviour restated: pop_factory.py:471-508 (row loop + row text), BgzfWriter framing (pop_factory.py:449).
#pragma once
#include "k_auto.cuh"

namespace dnaf {

struct XSpan {          // static per population, one per 64 samples
    uint32_t used[4];   // slots that print: bit 2i always, bit 2i+1 when sample i is female (existing samples only)
    uint32_t mv[4][5];  // move masks of the 5 compress steps, per 32-slot word
    uint32_t len[4];    // compacted bits per word (16..32)
    uint32_t sk[4];     // separator kind over compacted positions: 1 = '/', 0 = '\t'
    uint32_t skc;       // kinds of the two positions before the span (bits 0,1)
    uint32_t snz;       // units with a static separator mismatch
    uint32_t L;         // compacted positions of the span
    uint32_t byte_off;  // body byte offset of the span's first sample
    uint8_t sk6[32];    // per unit u: separator kinds of positions 4u-2 .. 4u+3 (positions past L repeat, no mismatch)
};
static_assert(offsetof(XSpan, sk6) % 16 == 0 && sizeof(XSpan) % 16 == 0, "k_x loads XSpan::sk6 as two 16-byte words");

// compacted allele bits of one span (4 words -> 128-bit little-endian sequence of total length L)
__host__ __device__ __forceinline__ uint32_t compact_span(const uint32_t m[4], const XSpan& xs, uint32_t c[4]) {
    uint32_t cw[4];
    for (int w = 0; w < 4; ++w) {
        uint32_t x = m[w] & xs.used[w];
        for (int i = 0; i < 5; ++i) {
            const uint32_t t = x & xs.mv[w][i];
            x = (x ^ t) | (t >> (1 << i));
        }
        cw[w] = x;
    }
    const uint32_t l0 = xs.len[0], l1 = xs.len[1], l2 = xs.len[2], l3 = xs.len[3];
    const uint64_t lo = (uint64_t)cw[0] | ((uint64_t)cw[1] << l0);      // l0 + l1 <= 64
    const uint64_t hi = (uint64_t)cw[2] | ((uint64_t)cw[3] << l2);
    const uint32_t sl = l0 + l1;                                         // 0..64
    uint64_t c01 = lo, c23 = 0;
    if (sl < 64) {
        c01 |= hi << sl;
        c23 = sl ? (hi >> (64 - sl)) : 0;
    } else {
        c23 = hi;
    }
    c[0] = (uint32_t)c01; c[1] = (uint32_t)(c01 >> 32); c[2] = (uint32_t)c23; c[3] = (uint32_t)(c23 >> 32);
    return l0 + l1 + l2 + l3;
}

// Static code tables of one (MAF bucket, with/without prefix) pair for X rows.
struct XTable {
    uint32_t len_tok[264];   // [g] match token for g = 3..258 predicted bytes; [0] empty
    uint32_t lit[8];
    uint32_t eob;
    uint32_t hdr_bits;
    uint32_t hdr[62];
    uint32_t pre_lit[256];
    uint2 lut[4096];         // key = c6 | s6 << 6; x: code bits 0..31; y: code bits 32..42 | nbits << 11 | long << 17 | lead << 24 | lastp << 28
};

// ---- the tokens of one unit; shared by the LUT builder, the host's statistics and the device slow paths ----
// c6 / s6: alleles / separator kinds of positions 4u-2 .. 4u+3 (bit j+2 = position 4u+j).
// Sink: lit(id), tok(len >= 3).  lead = bytes the unit leaves untouched at its start (0, 3..7; -1: no mismatch at
// all), lastp = end of the last byte it emitted (1..5, 8).
template <class Sink>
__host__ __device__ inline void xunit_tokens(uint32_t c6, uint32_t s6, Sink& sink, int& lead, int& lastp) {
    auto ev = [&](int b) {
        const uint32_t v = (b & 1) ? s6 : c6;
        const int j = b >> 1;
        return (int)(((v >> (j + 2)) ^ (v >> j)) & 1u);
    };
    auto lit_of = [&](int b) {
        const int j = b >> 1;
        if (b & 1) return ((s6 >> (j + 2)) & 1u) ? (int)kLitSlash : (int)kLitTab;
        return (int)((c6 >> (j + 2)) & 1u);
    };
    int pe = -1;
    lead = -1;
    lastp = 0;
    for (int b = 0; b < 8; ++b) {
        if (!ev(b)) continue;
        if (pe < 0) {
            if (b == 1 || b == 2) {
                for (int q = 0; q < b; ++q) sink.lit(lit_of(q));
                lead = 0;
            } else {
                lead = b;
            }
        } else {
            const int g = b - pe;
            if (g >= 3) sink.tok(g);
            else
                for (int q = pe; q < b; ++q) sink.lit(lit_of(q));
        }
        sink.lit(lit_of(b));
        pe = b + 1;
    }
    if (pe < 0) return;
    if (8 - pe == 1 || 8 - pe == 2) {
        for (int q = pe; q < 8; ++q) sink.lit(lit_of(q));
        pe = 8;
    }
    lastp = pe;
}

__host__ __device__ __forceinline__ uint32_t bit128(const uint32_t v[4], int k) { return (pick4(v, k >> 5) >> (k & 31)) & 1u; }

// 6-bit window of (v << 2 | carry) at unit u, i.e. positions 4u-2 .. 4u+3
__host__ __device__ __forceinline__ uint32_t win6(const uint32_t v[4], uint32_t carry, int u) {
    uint32_t r = 0;
    for (int j = -2; j < 4; ++j) {
        const int k = 4 * u + j;
        const uint32_t b = k < 0 ? (carry >> (k + 2)) & 1u : (k < 128 ? bit128(v, k) : 0u);
        r |= b << (j + 2);
    }
    return r;
}

// ---- the span grammar (host statistics + device slow path).  c: compacted alleles, L of them; positions past L repeat. ----
//   first span of a block: unit 0 as eight literals
//   whole units (nfull = (L - row_end) / 4): xunit_tokens, bridged by matches of 0 or >= 3 bytes
//   the rest, event by event; ['\n' when the span ends the row]; [EOB when it ends the block]
template <class Sink>
__host__ __device__ inline void xspan_tokens_ref(const uint32_t c[4], uint32_t carry, const XSpan& xs, int L,
                                                 bool first_in_block, bool ends_row, bool ends_block, Sink& sink) {
    const int nfull = (L - (ends_row ? 1 : 0)) / 4;
    const int nb = 2 * L - (ends_row ? 1 : 0);
    int prev_end = 0;
    auto lit_at = [&](int q) {
        const int k = q >> 1;
        if (q & 1) return bit128(xs.sk, k) ? (int)kLitSlash : (int)kLitTab;
        return (int)bit128(c, k);
    };
    auto gap_to = [&](int q) {
        const int g = q - prev_end;
        if (g >= 3) sink.tok(g);
        else
            for (int t = prev_end; t < q; ++t) sink.lit(lit_at(t));
    };
    for (int u = 0; u < nfull; ++u) {
        if (u == 0 && first_in_block) {
            for (int q = 0; q < 8; ++q) sink.lit(lit_at(q));
            prev_end = 8;
            continue;
        }
        const uint32_t c6 = win6(c, carry, u), s6 = xs.sk6[u];
        // peek: does the unit have any mismatch?
        const uint32_t xa = ((c6 >> 2) ^ c6) & 15u, xsm = ((s6 >> 2) ^ s6) & 15u;
        if (!(xa | xsm)) continue;
        // the bridge comes first: bytes up to the unit's first mismatch (a mismatch at byte 1 or 2 makes the unit
        // spell its first bytes out, so the bridge stops at the unit's start)
        const uint32_t evs = (xa & 1u) | ((xsm & 1u) << 1) | ((xa & 2u) << 1) | ((xsm & 2u) << 2) | ((xa & 4u) << 2) |
                             ((xsm & 4u) << 3) | ((xa & 8u) << 3) | ((xsm & 8u) << 4);   // mismatch flags by byte
        int first = 0;
        while (!((evs >> first) & 1u)) ++first;
        const int g = 8 * u + ((first == 1 || first == 2) ? 0 : first) - prev_end;
        if (g) sink.tok(g);
        int lead, lastp;
        xunit_tokens(c6, s6, sink, lead, lastp);
        prev_end = 8 * u + lastp;
    }
    for (int k = 4 * nfull; k < L; ++k) {
        const uint32_t ck2 = k >= 2 ? bit128(c, k - 2) : (carry >> k) & 1u;
        const uint32_t sk2 = k >= 2 ? bit128(xs.sk, k - 2) : (xs.skc >> k) & 1u;
        const bool force = first_in_block && k < 2;   // (cannot happen: a block's first span has whole units)
        if (force || bit128(c, k) != ck2) {
            gap_to(2 * k);
            sink.lit((int)bit128(c, k));
            prev_end = 2 * k + 1;
        }
        if (ends_row && k == L - 1) break;
        if (force || bit128(xs.sk, k) != sk2) {
            gap_to(2 * k + 1);
            sink.lit(bit128(xs.sk, k) ? (int)kLitSlash : (int)kLitTab);
            prev_end = 2 * k + 2;
        }
    }
    gap_to(nb);
    if (ends_row) sink.lit(kLitNl);
    if (ends_block) sink.eob();
}

struct XArgs {
    SampleView sv;
    SnpView nv;
    const FusedDesc* desc;
    const XTable* tables;
    const XSpan* xspans;       // [ceil(N/64)]
    const uint32_t* etab;      // [16][256] span-local CRC contributions of compacted allele bytes (span end aligned)
    const uint32_t* mspan;     // [spans][4][256] multiply by x^(8 * bytes from the span's end to its block's end)
    const uint32_t* mpre;      // [4][256] multiply by x^(8 * body bytes of segment 0)
    const uint32_t* xinit;     // [kBlk+1]
    const uint32_t* pre_crc;   // per row
    const uint64_t* orow;
    const uint32_t* osamp;
    uint64_t row_base;
    uint32_t k0, k1;
    uint8_t* slots;
    uint32_t slot_stride;      // bytes per output slot of this pass (>= the longest block's text + 96)
    uint32_t* sizes;
    uint32_t* crcs;
};

constexpr int kXStage = 24;   // staged words per span: X spans carry the static separator mismatches on top of the data
__host__ __device__ inline uint32_t x_smem_bytes(uint32_t nthr) {
    return kATabWords * 4u + ((uint32_t)(kXStage + 2) * nthr + nthr + 24u) * 4u + 20u * nthr + 32u * nthr + 16u;
}

// 32-bit mask of the non-zero nibbles of four words
__device__ __forceinline__ uint32_t nonzero_nibbles(const uint32_t x[4]) {
    uint32_t nz = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        uint32_t t = x[w] | (x[w] >> 1);
        t |= t >> 2;
        t &= 0x11111111u;                       // bit 4j = nibble j non-zero
        t = (t | (t >> 3)) & 0x03030303u;       // two flags per byte
        t = (t | (t >> 6)) & 0x000F000Fu;       // four per half word
        t = (t | (t >> 12)) & 0xFFu;
        nz |= t << (8 * w);
    }
    return nz;
}

#ifndef DNAF_X_REGS
#define DNAF_X_REGS 56   // as k_auto: 7 blocks of 160 threads per SM, no spills
#endif
__global__ void __maxnreg__(DNAF_X_REGS) k_x(const XArgs a) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31u, wid = tid >> 5;
    uint32_t* s_len = reinterpret_cast<uint32_t*>(smem_raw);   // len_tok | lit | eob | hdr_bits | hdr
    uint32_t* s_stage = s_len + kATabWords;
    uint32_t* s_last2 = s_stage + (kXStage + 2) * nthr;
    uint32_t* s_misc = s_last2 + nthr;
    uint8_t* s_cp = reinterpret_cast<uint8_t*>(s_misc + 24);
    uint32_t* s_sk6 = reinterpret_cast<uint32_t*>(s_cp + 20u * nthr);   // [8][nthr]: the span's XSpan::sk6, word-interleaved
    const uint32_t* s_lits = s_len + 264;
    const uint32_t* s_hdr = s_len + 274;

    const FusedDesc d = a.desc[blockIdx.x];
    const XTable* __restrict__ tb = a.tables + d.table;
    // match / literal tokens and the block header -> shared memory by one TMA bulk copy (see k_auto); the unit LUT stays in L2
    static_assert(sizeof(XTable) % 16 == 0, "XTable must be 16-byte aligned for the bulk copy");
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(s_misc + 22);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"(kATabWords * 4u) : "memory");
        bulk_g2s(s_len, tb->len_tok, kATabWords * 4u, mbar);
    }
    if (tid == 6) { s_misc[16] = 0; s_misc[17] = 0; }
    const uint32_t nspans = (d.ncells + 63u) / 64u;

    // ---- draw this span's 128 slots (as k_auto), force the overrides, compact to the printed alleles
    const uint32_t cs = d.cell0 + 64u * tid;
    int nc = 0;
    if (tid < nspans) nc = (int)min(64u, d.ncells - 64u * tid);
    uint32_t m[4] = {0, 0, 0, 0};
    if (nc > 0 && a.nv.k[d.row] == 2) {
        const uint32_t thr = a.nv.thr[d.row * 4];
        const uint64_t prow = a.row_base + d.row;
        const uint32_t r_lo = (uint32_t)prow, r_hi = (uint32_t)(prow >> 32);
        const uint32_t g0 = cs >> 4;
        uint32_t eq[4], lt[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            // slots beyond the last sample start out decided ("U <= T": reference allele, mask bit 0)
            const uint32_t g = g0 + w;
            const uint32_t slots = 32u * g < 2u * a.sv.n ? 2u * a.sv.n - 32u * g : 0u;
            eq[w] = slots >= 32u ? 0xFFFFFFFFu : ((1u << slots) - 1u);
            lt[w] = ~eq[w];
        }
#pragma unroll
        for (uint32_t q = 0; q < 2; ++q)
#pragma unroll
            for (int w = 0; w < 4; ++w) cmp_words(philox4x32_10(g0 + w, q, r_lo, r_hi, a.k0, a.k1), thr, 4u * q, eq[w], lt[w]);
        uint32_t qn = 0x02020202u;
        for (;;) {
            const int w = eq[0] ? 0 : (eq[1] ? 1 : (eq[2] ? 2 : (eq[3] ? 3 : 4)));
            if (w == 4) break;
            const uint32_t q = (qn >> (8 * w)) & 0xFFu;
            uint32_t e = pick4(eq, w), l = pick4(lt, w);
            cmp_words(philox4x32_10(g0 + w, q, r_lo, r_hi, a.k0, a.k1), thr, 4u * q, e, l);
            if (q == 7u) {
                l |= e;
                e = 0;
            }
            qn += 1u << (8 * w);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k == w) { eq[k] = e; lt[k] = l; }
        }
#pragma unroll
        for (int w = 0; w < 4; ++w) m[w] = ~(lt[w] | eq[w]);
    }
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
    const XSpan* __restrict__ xs = &a.xspans[min(cs >> 6, (a.sv.n + 63u) / 64u - 1u)];
    uint32_t c[4] = {0, 0, 0, 0};
    uint32_t L = 0;
    if (nc > 0) L = compact_span(m, *xs, c);

    // ---- CRC32 share of this span: template ^ delta (affine)
    uint32_t crc = 0;
    if (nc > 0 && (c[0] | c[1] | c[2] | c[3])) {
        uint32_t mm[4] = {c[0], c[1], c[2], c[3]};
        if (L < 128) {  // align the span's end with the table's span end (128-bit left shift by 128 - L)
            const uint32_t sh = 128u - L;
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
        crc = mul_tab(a.mspan + (size_t)(cs >> 6) * 1024u, sp);
    }
    // the block's prefix and text length, needed from here on (loaded after the draws: fewer live registers there)
    const bool starts_row = d.flags & 1u, ends_row = (d.flags >> 1) & 1u;
    const uint64_t pb = a.nv.pre_off[d.row];
    const uint32_t plen = starts_row ? (uint32_t)(a.nv.pre_off[d.row + 1] - pb) : 0u;
    const uint32_t body0 = a.sv.xoff[d.cell0];
    const uint32_t n = plen + (a.sv.xoff[d.cell0 + d.ncells] - body0);  // text bytes of this block
    uint32_t pre_tok = 0;
    if (tid < plen) pre_tok = __ldg(&tb->pre_lit[a.nv.prefix[pb + tid]]);
    if (tid == 0) {
        uint32_t c0 = d.body_crc ^ __ldg(&a.xinit[n]);
        if (starts_row) c0 ^= mul_tab(a.mpre, __ldg(&a.pre_crc[d.row]));
        crc ^= c0;
    }
    crc = warp_xor(crc);

    // ---- positions past L repeat the last two, so that they never mismatch; c' = (c << 2) | carry to shared memory
    uint32_t cpad[4] = {c[0], c[1], c[2], c[3]};
    if (nc > 0 && L < 128u) {
        const uint32_t l2 = L >= 2 ? ((bit128(c, (int)L - 1) << 1) | bit128(c, (int)L - 2)) : 0u;
        // position k >= L takes the value of position k - 2: the pattern of the last two positions, phase-aligned
        const uint32_t even = (L & 1u) ? (l2 >> 1) : (l2 & 1u), odd = (L & 1u) ? (l2 & 1u) : (l2 >> 1);
        const uint32_t pat = (even ? 0x55555555u : 0u) | (odd ? 0xAAAAAAAAu : 0u);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int lo = (int)L - 32 * w;
            const uint32_t keep = lo >= 32 ? 0xFFFFFFFFu : (lo <= 0 ? 0u : ((1u << lo) - 1u));
            cpad[w] = (c[w] & keep) | (pat & ~keep);
        }
    }
    s_last2[tid] = L >= 2 ? ((bit128(c, (int)L - 1) << 1) | bit128(c, (int)L - 2)) : 0u;
    __syncthreads();        // also orders the mbarrier's initialisation before the waits
    mbar_wait(mbar, 0u);
    if (lane == 0 && crc) atomicXor(&s_misc[16], crc);
    const uint32_t carry = tid ? s_last2[tid - 1] : (cpad[0] & 3u);
    const bool worker = nc > 0;
    const bool p_last = worker && 64u * tid + (uint32_t)nc == d.ncells;
    const bool p_end = ends_row && p_last;
    const int nfull = worker ? ((int)L - (p_end ? 1 : 0)) / 4 : 0;
    uint32_t nz = 0;
    if (worker) {
        uint32_t q[5];
        q[0] = (cpad[0] << 2) | carry;
        q[1] = __funnelshift_l(cpad[0], cpad[1], 2);
        q[2] = __funnelshift_l(cpad[1], cpad[2], 2);
        q[3] = __funnelshift_l(cpad[2], cpad[3], 2);
        q[4] = cpad[3] >> 30;
        uint32_t* dst = reinterpret_cast<uint32_t*>(s_cp + 20u * tid);
#pragma unroll
        for (int k = 0; k < 5; ++k) dst[k] = q[k];
        // the unit loop's separator keys come from shared memory: one global round trip here instead of one per unit
        // in front of the dependent LUT load
        const uint4* sk = reinterpret_cast<const uint4*>(xs->sk6);
        const uint4 k0 = sk[0], k1 = sk[1];
        s_sk6[0 * nthr + tid] = k0.x; s_sk6[1 * nthr + tid] = k0.y; s_sk6[2 * nthr + tid] = k0.z; s_sk6[3 * nthr + tid] = k0.w;
        s_sk6[4 * nthr + tid] = k1.x; s_sk6[5 * nthr + tid] = k1.y; s_sk6[6 * nthr + tid] = k1.z; s_sk6[7 * nthr + tid] = k1.w;
        const uint32_t x[4] = {cpad[0] ^ q[0], cpad[1] ^ q[1], cpad[2] ^ q[2], cpad[3] ^ q[3]};
        nz = (nonzero_nibbles(x) | xs->snz) & (nfull >= 32 ? 0xFFFFFFFFu : ((1u << nfull) - 1u));
    }
    // ---- pass 1: this span's tokens, staged privately
    const uint32_t eob = s_len[272];
    AStageT<kXStage> st{s_stage + tid, nthr, 0u, 0u, 0u};
    ATokSink<AStageT<kXStage>> ts{st, s_len, s_lits, eob};
    if (worker) {
        const uint8_t* cpb = s_cp + 20u * tid;
        auto sk6_at = [&](int u) { return (s_sk6[(u >> 2) * nthr + tid] >> (8 * (u & 3))) & 0xFFu; };
        const uint2* __restrict__ lut = tb->lut;
        int prev_end = 0;
        if (tid == 0) {   // first span of the block: unit 0 as eight literals
            uint32_t lo = 0, hi = 0, nlo = 0, nhi = 0;
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                const uint32_t t = s_lits[(b & 1) ? (((xs->sk[0] >> (b >> 1)) & 1u) ? kLitSlash : kLitTab) : ((cpad[0] >> (b >> 1)) & 1u)];
                if (b < 4) { lo |= (t & 0xFFFFFFu) << nlo; nlo += t >> 24; }     // cell literals: <= 10 bits each
                else { hi |= (t & 0xFFFFFFu) << nhi; nhi += t >> 24; }
            }
            st.put64(lo, 0u, nlo);
            st.put64(hi, 0u, nhi);
            prev_end = 8;
            nz &= ~1u;
        }
        while (nz) {
            const int u = __ffs((int)nz) - 1;
            nz &= nz - 1u;
            const uint32_t v = (uint32_t)cpb[u >> 1] | ((uint32_t)cpb[(u >> 1) + 1] << 8);
            const uint32_t c6 = (v >> (4 * (u & 1))) & 63u;
            const uint32_t s6 = sk6_at(u);
            const uint32_t key = c6 | (s6 << 6);
            const uint2 e = __ldg(&lut[key]);
            const uint32_t nb = (e.y >> 11) & 63u;
            const int pos = 8 * u;
            const int gap = pos + (int)((e.y >> 24) & 15u) - prev_end;
            const uint32_t t1 = s_len[gap];
            if (!(e.y & kLutLong)) {
                st.put_tok_code(t1, e.x, e.y & 0x7FFu, nb);
            } else {
                st.put64(t1 & 0xFFFFFFu, 0u, t1 >> 24);
                int lead, lastp;
                xunit_tokens(c6, s6, ts, lead, lastp);
            }
            prev_end = pos + (int)(e.y >> 28);
        }
        // the positions after the last whole unit, event by event: they all lie in the 6-position window of unit `nfull`
        // (bit j + 2 = position 4 * nfull + j, j = -2 .. 3), read like the loop above reads its units
        {
            const int k0 = 4 * nfull;
            const uint32_t vt = (uint32_t)cpb[nfull >> 1] | ((uint32_t)cpb[(nfull >> 1) + 1] << 8);
            const uint32_t c6 = (vt >> (4 * (nfull & 1))) & 63u;
            const uint32_t s6 = nfull < 32 ? sk6_at(nfull) : (xs->sk[3] >> 30);
            auto lit_at = [&](int q) {
                const int j = (q >> 1) - k0 + 2;
                if (q & 1) return s_lits[((s6 >> j) & 1u) ? kLitSlash : kLitTab];
                return s_lits[(c6 >> j) & 1u];
            };
            auto gap_to = [&](int q) {
                const int g = q - prev_end;
                if (g >= 3) {
                    const uint32_t t = s_len[g];
                    st.put64(t & 0xFFFFFFu, 0u, t >> 24);
                } else {
                    for (int t = prev_end; t < q; ++t) {
                        const uint32_t tk = lit_at(t);
                        st.put64(tk & 0xFFFFFFu, 0u, tk >> 24);
                    }
                }
            };
            for (int k = k0; k < (int)L; ++k) {
                const int j = k - k0;   // window bit j + 2 = position k, bit j = position k - 2
                const uint32_t cb = (c6 >> (j + 2)) & 1u, sb = (s6 >> (j + 2)) & 1u;
                if (cb != ((c6 >> j) & 1u)) {
                    gap_to(2 * k);
                    const uint32_t tk = s_lits[cb];
                    st.put64(tk & 0xFFFFFFu, 0u, tk >> 24);
                    prev_end = 2 * k + 1;
                }
                if (p_end && k == (int)L - 1) break;
                if (sb != ((s6 >> j) & 1u)) {
                    gap_to(2 * k + 1);
                    const uint32_t tk = s_lits[sb ? kLitSlash : kLitTab];
                    st.put64(tk & 0xFFFFFFu, 0u, tk >> 24);
                    prev_end = 2 * k + 2;
                }
            }
            gap_to(2 * (int)L - (p_end ? 1 : 0));
            const uint32_t tn = p_end ? s_lits[kLitNl] : 0u;
            const uint32_t te = p_last ? eob : 0u;
            const uint32_t nn = tn >> 24;
            st.put64((tn & 0xFFFFFFu) | ((te & 0xFFFFFFu) << nn), 0u, nn + (te >> 24));
        }
        if (st.bits() > 32u * kXStage) s_misc[17] = 1;
    }
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
    const uint32_t total_pre = plen ? s_misc[8] + s_misc[9] : 0u;
    const uint32_t pre_off = v0 - pre_bits + (wid == 1 ? s_misc[8] : 0u);
    const uint32_t hdr_bits = s_len[273];
    const uint32_t data_bits = hdr_bits + total_pre + total_span;
    const uint32_t payload = (data_bits + 7u) / 8u;
    const uint32_t out_words = (data_bits + 31u) / 32u;
    const bool stored = payload > n + 5u;
    uint8_t* blk = a.slots + (uint64_t)d.slot * a.slot_stride + kSlotLead;
    uint32_t* words = reinterpret_cast<uint32_t*>(blk + 18);  // 16-byte aligned

    uint32_t out_payload;
    if (!stored) {
        const uint32_t hdr_words = (hdr_bits + 31u) / 32u;
        const uint32_t hw4 = (hdr_words + 3u) & ~3u;   // <= 64 <= nthr
        if (tid < hw4) words[tid] = tid < hdr_words ? s_hdr[tid] : 0u;
        {
            uint4* w4 = reinterpret_cast<uint4*>(words + hw4);
            const uint32_t n4 = out_words + 2u > hw4 ? (out_words + 2u - hw4 + 3u) / 4u : 0u;
            for (uint32_t i = tid; i < n4; i += nthr) w4[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        __syncthreads();
        const bool overflow = s_misc[17] != 0;
        if (pre_bits) {
            const uint32_t pos = hdr_bits + pre_off, wi = pos >> 5, sh = pos & 31u, v = pre_tok & 0xFFFFFFu;
            atomicOr(&words[wi], v << sh);
            if (sh + pre_bits > 32) atomicOr(&words[wi + 1], v >> (32 - sh));
        }
        if (worker) {
            const uint32_t dst = hdr_bits + total_pre + span_off;
            if (!overflow) {
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
                // some span overflowed its staging words: every span re-emits straight into the output words
                AEmit em{words, dst};
                ATokSink<AEmit> te{em, s_len, s_lits, eob};
                xspan_tokens_ref(cpad, carry, *xs, (int)L, tid == 0, p_end, p_last, te);
            }
        }
        out_payload = payload;
    } else {
        // stored deflate block: format the text itself (rare safety net)
        if (tid == 0) {
            blk[18] = 1;
            blk[19] = (uint8_t)n; blk[20] = (uint8_t)(n >> 8);
            blk[21] = (uint8_t)~n; blk[22] = (uint8_t)((~n) >> 8);
        }
        if (tid < plen) blk[23 + tid] = a.nv.prefix[pb + tid];
        if (nc > 0) {
            uint8_t* p = blk + 23 + plen + (xs->byte_off - body0);
            for (uint32_t k = 0; k < L; ++k) {
                p[2 * k] = '0' + bit128(c, (int)k);
                p[2 * k + 1] = (p_end && k + 1 == L) ? '\n' : (bit128(xs->sk, (int)k) ? '/' : '\t');
            }
        }
        out_payload = n + 5u;
    }
    __syncthreads();
    if (tid < 26) {
        const uint32_t crc32 = ~s_misc[16];
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
