// k_lz: the autosome-row kernel of the higher compression tiers (-z 3..9).  Same job, block geometry, draws, CRC
// and output slots as k_auto (k_auto.cuh); what changes is the deflate parse.  k_auto predicts every byte by the byte
// 4 back ("P4"); here a block is parsed with real LZ77 matches over its whole 32 KiB window -- in the ALLELE-BIT
// domain: the text of an autosome row is  a0 '/' a1 '\t' ...  with a_j in {'0','1'}, so the block is a string of
// allele bits with fixed separators, and a deflate match (length 2k [+1], distance 4D bytes) is a run of k equal bits
// 2D positions back.  Comparing 32 alleles (64 text bytes) costs one XOR and one find-first-set.
//
// Reference behaviour restated: Bio.bgzf.BgzfWriter(compresslevel=z) -- pop_factory.py:403 passes the -z value
// (default 6, pop_factory.py:656-658) to zlib.compressobj(level, DEFLATED, -15) for every 64 KiB block.  zlib's
// levels are hash chains of growing depth (16, 32, 128, 256, 1024, 4096 candidates at levels 4 .. 9, lazy
// evaluation from level 4 on); the tiers here follow that ladder (lz_cfg).  Compressed bytes are outside the parity
// contract (SURVEY R5, 8c); the decompressed text is identical at every level.
//
// Match finder (deterministic, built per block in shared memory):
//   * key of allele position a = its next L alleles (L = 8 or 9, per MAF bucket) and a's parity (distances are even)
//   * a block is cut into REGIONS of 4096 alleles = the 32 spans of one warp.  Every warp links the positions of its
//     region into per-key chains in position order, 32 consecutive positions per step: every lane reads
//     head[region][key] (the last occurrence before this step) into prev[a], then the step's positions go into the
//     heads with atomicMax.  Positions of one step that share a key all point at the same predecessor and only the
//     last of them is reachable from later steps -- which thins exactly the over-populated keys (the inside of a long
//     run of reference alleles) and loses ~1 % of the entries elsewhere.  max() does not depend on the order the
//     lanes arrive in and reads and updates are separated by a warp barrier: the same block always gives the same
//     chains.  (A first version linked equal keys inside a step exactly with __match_any_sync; MATCH.ANY takes time
//     proportional to the number of distinct keys in the warp and made this phase 4x the cost of everything else.)
//   * a lookup at position s walks prev[] in its own region, then enters the regions before it through their heads
//     (all of a previous region precedes s): candidates come nearest first, like zlib's hash chains, at most
//     `chain` of them; plus the two near distances 4 and 8 bytes that need no table.
//   * one thread parses one span (64 cells) sequentially, greedy longest match (ties: nearest), one-step lazy
//     evaluation from -z 6 on; tokens never cross spans, sources may lie anywhere earlier in the block.
//   * per MAF bucket the host fits the codes of this parse AND of the near-distances-only parse and keeps the
//     smaller (fused_host.h make_lz_table): blocks of such buckets (LzTable.chain == 0) skip the chain build.
#pragma once
#include "k_auto.cuh"

namespace dnaf {

constexpr int kLStage = 14;            // staged words per span before the block falls back to direct emission
constexpr uint32_t kLzNone = 0xFFFFu;      // prev[] entry / head value of "no earlier position" (heads hold 0 = none, position + 1 otherwise)
constexpr uint32_t kLzRegion = 4096;   // alleles per region (one warp's 32 spans)
constexpr uint32_t kLzMaxKey = 9;      // alleles in a key (head tables have 2^(key+1) 32-bit entries per region)
constexpr uint32_t kLzMaxDist = 16384; // alleles = 32768 bytes
constexpr uint32_t kLzGood = 8;        // alleles: with a near match this long in hand the key chain is not walked

struct LzCfg {
    uint32_t chain;   // far candidates examined per lookup
    uint32_t lazy;    // 0 / 1: one-step lazy evaluation
    uint32_t key;     // alleles per key (<= kLzMaxKey)
    uint32_t nice;    // alleles: a match this long ends the search
};

// -z level -> parse parameters.  3: the two near distances only (no tables are built); 4..9: zlib's own ladder shape
// (its max_chain is 16 / 32 / 128 / 256 / 1024 / 4096 there; shorter here because every chain entry is already a
// >= 2*key byte match), lazy evaluation from 6 on; like zlib, the lookup behind a match searches a quarter as deep.
__host__ __device__ inline LzCfg lz_cfg(int level, uint32_t key) {
    LzCfg c;
    c.key = key;
    c.chain = level <= 3 ? 0u : level == 4 ? 1u : level == 5 ? 4u : level == 6 ? 20u : level == 7 ? 32u : level == 8 ? 64u : 128u;
    c.lazy = level >= 6 ? 1u : 0u;
    c.nice = level <= 4 ? 16u : level == 5 ? 32u : level <= 7 ? 64u : 128u;   // zlib: 16, 32, 128, 128, 258, 258 bytes
    return c;
}

// Static code tables of one (MAF bucket, with/without prefix, tier).
struct LzTable {
    // ---- the first kLTabWords words are copied to shared memory by every block (one bulk copy)
    uint32_t len_tok[260];   // [len 3..258]: length code | extra << code bits | total bits << 24 (no distance part)
    uint32_t lit[8];         // cell literals by id: code | bits << 24
    uint32_t eob;
    uint32_t hdr_bits;
    uint32_t dist_tok[32];   // [distance symbol]: code | bits << 24
    uint32_t key_alleles;    // the parse parameters this table's codes were fitted to (LzCfg): a bucket whose rows
    uint32_t chain;          // compress no better with the key chains (rare minor alleles: the dynamic-block header
    uint32_t lazy;           // of a code with 27 distance symbols outweighs what far matches save) keeps chain = 0
    uint32_t nice;           // and its blocks skip the chain build
    uint32_t hdr[94];        // serialized dynamic-block header
    // ----
    uint32_t pre_lit[256];   // literal codes of prefix bytes
};
constexpr uint32_t kLTabWords = 260 + 8 + 2 + 32 + 4 + 94;   // 400 words = 100 x 16 bytes
static_assert(kLTabWords % 4 == 0 && sizeof(LzTable) % 16 == 0, "LzTable must copy in 16-byte units");

__host__ __device__ __forceinline__ uint32_t lz_fsr(uint32_t lo, uint32_t hi, uint32_t sh) {
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, sh);
#else
    sh &= 31u;
    return sh ? (lo >> sh) | (hi << (32u - sh)) : lo;
#endif
}
// distance (bytes, 1..32768) -> deflate distance symbol, number of extra bits, extra value
__host__ __device__ __forceinline__ void lz_dist_sym(uint32_t d, uint32_t& sym, uint32_t& eb, uint32_t& ev) {
    if (d <= 4u) { sym = d - 1u; eb = 0; ev = 0; return; }
    const uint32_t x = d - 1u;
#ifdef __CUDA_ARCH__
    const uint32_t hb = 31u - (uint32_t)__clz((int)x);
#else
    const uint32_t hb = 31u - (uint32_t)__builtin_clz(x);
#endif
    sym = 2u * hb + ((x >> (hb - 1u)) & 1u);
    eb = hb - 1u;
    ev = x & ((1u << eb) - 1u);
}

// ---- the span grammar of the LZ tiers (host table builder, device fast and slow paths all run this function) ----
// Block coordinates: allele a of the block is text byte 2a, its separator byte 2a+1 ('/' after even a, '\t' after
// odd a); byte -1 is the separator before the block's first allele (the prefix's last tab, or the tab that ended
// the previous segment -- the block owns it).  A span of nc cells starting at allele a0 owns bytes 2*a0 - 1 ..
// 2*(a0 + 2nc) - 2 (its last allele): the separator BEFORE its first cell, not the one after its last.
//   first span of a block: ['\t' unless the block starts a row] a0 '/' a1 as literals (no history yet)
//   then greedy: at byte p, s = first allele at or after p; candidates = distances 4, 8 and the key chain of s;
//   k = most alleles equal to those 2D back (up to the span's end); the match covers bytes p .. 2(s+k)-1, without
//   that last separator when it is not the span's; >= 3 bytes -> match, else one literal byte.
//   ['\n' if the span ends the row] [EOB if it ends the block]
// Mem: word(i) = allele bits 32i .. 32i+31 of the block (zero past the end), prev(a), head(region, key).
// Sink: emit(is_match, literal id, len bytes, dist bytes), eob().
template <class Mem>
__host__ __device__ __forceinline__ uint32_t lz_win32(const Mem& mem, uint32_t a) {
    const uint32_t w = a >> 5;
    return lz_fsr(mem.word(w), mem.word(w + 1u), a & 31u);
}

__host__ __device__ __forceinline__ uint32_t lz_ctz32(uint32_t x) {   // x != 0
#ifdef __CUDA_ARCH__
    return (uint32_t)__ffs((int)x) - 1u;
#else
    return (uint32_t)__builtin_ctz(x);
#endif
}

// alleles from s + 32 on that equal those from j + 32 on, given that the first 32 are equal: 32 + ... (<= limit)
template <class Mem>
__host__ __device__ __forceinline__ uint32_t lz_extend(const Mem& mem, uint32_t s, uint32_t j, uint32_t limit) {
    uint32_t off = 32u;
    for (;;) {
        const uint32_t x = lz_win32(mem, s + off) ^ lz_win32(mem, j + off);
        const uint32_t room = limit - off;
        uint32_t c = x ? lz_ctz32(x) : 32u;
        c = c < room ? c : room;
        if (c == 32u && room > 32u) off += 32u;
        else return off + c;
    }
}

// Best match at allele s (k alleles at distance `da` alleles; k = 0: none), and s's own 32-allele window.
// Set-up and the two near distances (4 and 8 bytes: j = s-2, s-4) are compared from the same three words that hold
// s's own window, then the key chain of s is walked nearest first (own region, then the regions before it through
// their heads), at most `depth` entries -- unless a near match of kLzGood alleles is already in hand.
template <class Mem>
__host__ __device__ __forceinline__ void lz_lookup(const Mem& mem, uint32_t s, uint32_t aend, uint32_t nall, const LzCfg cfg,
                                                  uint32_t depth, uint32_t& best_k, uint32_t& best_da, uint32_t& ws0) {
    const uint32_t limit = aend - s;
    // alleles lo .. lo+63 with lo = s - 4 (s >= 4 everywhere but in the first cells of a block)
    const uint32_t lo = s >= 4u ? s - 4u : 0u, sh0 = s - lo;
    const uint32_t w = lo >> 5, sh = lo & 31u;
    const uint32_t x0 = mem.word(w), x1 = mem.word(w + 1u), x2 = mem.word(w + 2u);
    const uint32_t v0 = lz_fsr(x0, x1, sh), v1 = lz_fsr(x1, x2, sh);
    ws0 = lz_fsr(v0, v1, sh0);
    const uint32_t room = limit < 32u ? limit : 32u;
    uint32_t k1 = 0, k2 = 0;
    if (s >= 2u) {
        const uint32_t d1 = ws0 ^ lz_fsr(v0, v1, sh0 - 2u);
        k1 = d1 ? lz_ctz32(d1) : 32u;
        k1 = k1 < room ? k1 : room;
    }
    if (s >= 4u) {
        const uint32_t d2 = ws0 ^ v0;
        k2 = d2 ? lz_ctz32(d2) : 32u;
        k2 = k2 < room ? k2 : room;
    }
    best_k = k2 > k1 ? k2 : k1;
    best_da = k2 > k1 ? 4u : 2u;
    if (best_k == 32u && limit > 32u) best_k = lz_extend(mem, s, s - best_da, limit);   // the nearer one goes on
    // not with a near match of kLzGood alleles in hand (zlib's good_length idea taken to its end: on the host twin,
    // walking a quarter of the chain there or none of it gives the same ratio)
    if (depth && best_k < limit && best_k < kLzGood && s + cfg.key <= nall) {
        const uint32_t key = (ws0 & ((1u << cfg.key) - 1u)) | ((s & 1u) << cfg.key);
        uint32_t reg = s / kLzRegion;
        uint32_t j = mem.prev(s);
        for (uint32_t n = 0; n < depth; ++n) {
            while (j == kLzNone && reg) {
                --reg;
                j = mem.head(reg, key);
            }
            if (j == kLzNone || s - j > kLzMaxDist) break;
            const uint32_t x = ws0 ^ lz_win32(mem, j);
            uint32_t k = x ? lz_ctz32(x) : 32u;
            k = k < room ? k : room;
            if (k == 32u && limit > 32u) k = lz_extend(mem, s, j, limit);
            if (k > best_k) {
                best_k = k;
                best_da = s - j;
                if (k >= limit || k >= cfg.nice) break;
            }
            j = mem.prev(j);
        }
    }
}

// One trip of the loop = one TOKEN: the lookup at byte p and, with lazy evaluation, the lookup one allele on (searched
// a quarter as deep, zlib's rule behind a good match) -- both in the same trip, so that the lanes of a warp walk their
// chains together.  (Earlier shapes, measured: nested per-token loops left 18 of 32 threads active; a fully flat
// one-candidate-per-trip state machine 13 of 32 -- every trip ran the code of every state some lane was in; one lookup
// per trip with the lazy second lookup as a trip of its own 16 of 32 at -z 6 -- full-depth and quarter-depth lanes
// mixed.  A two-phase variant -- near-match tokens emitted in a tight loop until the thread stands at an allele that
// needs its chain, then all lanes walk together -- was 7 % faster at -z 3 and 3 % slower at -z 6: the rows that cost
// the time are the common-minor-allele ones, where every token needs its chain.)
// nice: a match of that many alleles ends the search (zlib's nice_length).
template <class Mem, class Sink>
__host__ __device__ __forceinline__ void lz_span_tokens(const Mem& mem, uint32_t a0, int nc, bool first_in_block, bool starts_row,
                                                        bool ends_row, bool ends_block, uint32_t nall, const LzCfg cfg, Sink& sink) {
    const uint32_t aend = a0 + 2u * (uint32_t)nc;   // one past the span's last allele
    auto bit = [&](uint32_t a) { return (int)((mem.word(a >> 5) >> (a & 31u)) & 1u); };
    int p = 2 * (int)a0 - 1;                        // next byte to emit (block coordinates)
    if (first_in_block) {
        if (!starts_row) sink.emit(false, kLitTab, 0, 0);
        sink.emit(false, bit(a0), 0, 0);
        sink.emit(false, kLitSlash, 0, 0);
        sink.emit(false, bit(a0 + 1u), 0, 0);
        p = 2 * (int)a0 + 3;
    }
    const int pend = 2 * (int)aend - 1;             // one past the span's last byte
    while (p < pend) {
        const uint32_t s = (uint32_t)(p + 1) >> 1;   // s < aend here: the span's last byte is an allele
        const uint32_t odd = (uint32_t)p & 1u;
        uint32_t best_k, best_da, ws0;
        lz_lookup(mem, s, aend, nall, cfg, cfg.chain, best_k, best_da, ws0);
        // bytes p .. 2(s+k)-1, minus the separator after the span's last allele
        int len = 2 * (int)(s + best_k) - p - (s + best_k == aend ? 1 : 0);
        bool lit_first = false;
        if (cfg.lazy && len >= 3 && !odd && s + 1u < aend && s + best_k < aend && best_k < cfg.nice) {
            // would a literal now buy a longer match from the next byte on?
            uint32_t k2, da2, w2;
            lz_lookup(mem, s + 1u, aend, nall, cfg, (cfg.chain + 3u) >> 2, k2, da2, w2);
            const int len2 = 2 * (int)(s + 1u + k2) - (p + 1) - (s + 1u + k2 == aend ? 1 : 0);
            if (len2 > len + 1) {
                lit_first = true;
                len = len2;
                best_da = da2;
            }
        }
        if (lit_first) {
            sink.emit(false, (int)(ws0 & 1u), 0, 0);
            p += 1;
        }
        const bool is_match = len >= 3;
        const int id = odd ? ((s & 1u) ? kLitSlash : kLitTab) : (int)(ws0 & 1u);   // separator before allele s / allele s
        sink.emit(is_match, id, len, 2 * (int)best_da);
        p += is_match ? len : 1;
    }
    if (ends_row) sink.emit(false, kLitNl, 0, 0);
    if (ends_block) sink.eob();
}

#ifdef __CUDACC__
struct LzArgs {
    AutoArgs a;
    const LzTable* tables;   // [2 * bucket + (segment 0 ? 0 : 1)]; parse parameters come from the table
};

struct LzMemDev {
    const uint32_t* bits;
    const uint16_t* prv;
    const uint32_t* hd;      // [region][2^hbits]: last position of the key in the region + 1, 0 = none
    uint32_t hbits;
    __device__ __forceinline__ uint32_t word(uint32_t i) const { return bits[i]; }
    __device__ __forceinline__ uint32_t prev(uint32_t a) const { return prv[a]; }
    __device__ __forceinline__ uint32_t head(uint32_t reg, uint32_t key) const { return (hd[(reg << hbits) + key] - 1u) & 0xFFFFu; }
};

// token-level adapter of the bit sinks (AStageT / AEmit, k_auto.cuh): literal or match through ONE append
template <class Bits>
struct LzTokSink {
    Bits& b;
    const uint32_t* len_tok;
    const uint32_t* lits;
    const uint32_t* dist_tok;
    uint32_t eob_tok;
    __device__ __forceinline__ void emit(bool is_match, int id, int len, int dist) {
        const uint32_t t1 = is_match ? len_tok[len] : lits[id];
        uint32_t c = 0, nb = 0;
        if (is_match) {
            uint32_t sym, eb, ev;
            lz_dist_sym((uint32_t)dist, sym, eb, ev);
            const uint32_t dt = dist_tok[sym];
            const uint32_t dn = dt >> 24;
            c = (dt & 0xFFFFFFu) | (ev << dn);
            nb = dn + eb;
        }
        b.put_tok_code(t1, c, 0u, nb);   // <= 20 + 28 bits
    }
    __device__ __forceinline__ void eob() { b.put64(eob_tok & 0xFFFFFFu, 0u, eob_tok >> 24); }
};

// dynamic shared memory carve-up
__host__ __device__ inline uint32_t lz_smem_bytes(uint32_t nthr, uint32_t hbits, bool with_chains) {
    return kLTabWords * 4u + (4u * nthr + 8u) * 4u + ((uint32_t)(kLStage + 2) * nthr + 24u) * 4u + 16u +
           (with_chains ? (nthr / 32u) * (4u << hbits) + nthr * 256u : 0u);   // heads + prev[] come last
}

// 64 registers, as before the shared draw lost its stack frame (left free, ptxas takes 80 for the register-only draw)
__global__ void __launch_bounds__(256, 4) k_lz(const LzArgs la) {
    const AutoArgs& a = la.a;
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31u, wid = tid >> 5;
    uint32_t* s_tab = reinterpret_cast<uint32_t*>(smem_raw);     // LzTable's first kLTabWords words
    uint32_t* s_bits = s_tab + kLTabWords;                       // allele bits of the block + 8 zero guard words
    uint32_t* s_stage = s_bits + 4u * nthr + 8u;
    uint32_t* s_misc = s_stage + (kLStage + 2) * nthr;           // as in k_auto: [0..7] warp bits, [8..9] prefix bits, [10] const crc, [16] crc, [17] overflow, [22..23] mbarrier
    uint16_t* s_prev = reinterpret_cast<uint16_t*>(s_misc + 24u + 4u);
    const uint32_t* s_len = s_tab;
    const uint32_t* s_lits = s_tab + 260;
    const uint32_t* s_dist = s_tab + 270;
    const uint32_t* s_hdr = s_tab + 306;

    FusedDesc d;
    if (a.desc) {
        d = a.desc[blockIdx.x];
    } else {
        const uint32_t rl = a.nseg_magic ? __umulhi(blockIdx.x, a.nseg_magic) : blockIdx.x, sg = blockIdx.x - rl * a.nseg;
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
    const LzTable* __restrict__ tb = la.tables + d.table;
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(s_misc + 22);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"(kLTabWords * 4u) : "memory");
        bulk_g2s(s_tab, tb->len_tok, kLTabWords * 4u, mbar);
    }
    if (tid == 6) { s_misc[16] = 0; s_misc[17] = 0; }
    const bool starts_row = d.flags & 1u, ends_row = (d.flags >> 1) & 1u;
    const uint64_t pb = a.nv.pre_off[d.row];
    const uint32_t plen = starts_row ? (uint32_t)(a.nv.pre_off[d.row + 1] - pb) : 0u;
    const uint32_t lead = starts_row ? plen : 1u;
    const uint32_t n = lead + 4u * d.ncells - (ends_row ? 0u : 1u);
    const uint32_t nspans = (d.ncells + 63u) / 64u;
    const uint32_t nall = 2u * d.ncells;

    // ---- draws, overrides, CRC share: exactly k_auto's (shared functions)
    const uint32_t cs = d.cell0 + 64u * tid;
    int nc = 0;
    if (tid < nspans) nc = (int)min(64u, d.ncells - 64u * tid);
    uint32_t m[4] = {0, 0, 0, 0};
    auto_draw_span(a, d, cs, nc, m);
    uint32_t crc = auto_span_crc(a, d, m, nc, tid, nspans);
    uint32_t pre_tok = 0;
    if (tid < plen) pre_tok = __ldg(&tb->pre_lit[a.nv.prefix[pb + tid]]);
    if (tid == 0) {
        uint32_t c0 = d.body_crc ^ __ldg(&a.xinit[n]);
        if (starts_row) c0 ^= mul_tab(ends_row ? a.mpre + 1024 : a.mpre, __ldg(&a.pre_crc[d.row]));
        s_misc[10] = c0;
    }
    crc = warp_xor(crc);

    // ---- allele bits of the block -> shared memory (bits past the block's last cell are zero)
    {
        uint32_t mm[4] = {m[0], m[1], m[2], m[3]};
        if (nc < 64) {
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const int lo = 2 * nc - 32 * w;
                mm[w] &= lo >= 32 ? 0xFFFFFFFFu : (lo <= 0 ? 0u : ((1u << lo) - 1u));
            }
        }
        *reinterpret_cast<uint4*>(s_bits + 4u * tid) = make_uint4(mm[0], mm[1], mm[2], mm[3]);
        if (tid < 8) s_bits[4u * nthr + tid] = 0u;
    }
    const uint32_t key_alleles = __ldg(&tb->key_alleles), chain = __ldg(&tb->chain);
    const uint32_t hbits = key_alleles + 1u;
    uint32_t* s_head = reinterpret_cast<uint32_t*>(s_prev + 128u * nthr);
    if (chain) {   // heads of this warp's region start empty
        uint32_t* h32 = s_head + ((size_t)wid << hbits);
        for (uint32_t i = lane; i < (1u << hbits); i += 32u) h32[i] = 0u;
    }
    __syncthreads();        // bits complete; also orders the mbarrier's initialisation before the waits
    if (lane == 0 && crc) atomicXor(&s_misc[16], crc);

    // ---- chains of this warp's region, 32 consecutive positions per step (see the header comment).  Positions whose
    // key runs past the block's end are linked too (their keys hold guard zeros): no lookup can reach them, every
    // candidate lies before a position whose own key fits.
    if (chain) {
        const uint32_t rbase = kLzRegion * wid;                  // first allele of the region
        const uint32_t rend = min(nall, rbase + kLzRegion);
        uint32_t* hd = s_head + ((size_t)wid << hbits);
        const uint32_t kmask = (1u << key_alleles) - 1u, par = (lane & 1u) << key_alleles;
        uint32_t w0 = s_bits[rbase >> 5];
        for (uint32_t pos = rbase; pos < rend; pos += 32u) {
            const uint32_t w1 = s_bits[(pos >> 5) + 1u];
            const uint32_t key = (__funnelshift_r(w0, w1, lane) & kmask) | par;
            w0 = w1;
            const uint32_t before = hd[key];                     // last occurrence in the steps before this one (+ 1)
            s_prev[pos + lane] = (uint16_t)(before - 1u);        // 0 -> kLzNone
            __syncwarp();
            atomicMax(&hd[key], pos + lane + 1u);
            __syncwarp();
        }
    }
    mbar_wait(mbar, 0u);    // the code tables have landed
    __syncthreads();        // every region's chains are complete

    // ---- pass 1: this span's tokens, staged privately
    const uint32_t eob = s_tab[268];
    const bool worker = nc > 0;
    const bool p_last = worker && 64u * tid + (uint32_t)nc == d.ncells;
    const bool p_end = ends_row && p_last;
    const LzCfg cfg{chain, s_tab[304], key_alleles, s_tab[305]};
    const LzMemDev mem{s_bits, s_prev, s_head, hbits};
    AStageT<kLStage> st{s_stage + tid, nthr, 0u, 0u, 0u};
    if (worker) {
        LzTokSink<AStageT<kLStage>> ts{st, s_len, s_lits, s_dist, eob};
        lz_span_tokens(mem, 128u * tid, nc, tid == 0, starts_row, p_end, p_last, nall, cfg, ts);
        if (st.bits() > 32u * kLStage) s_misc[17] = 1;
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
    const uint32_t hdr_bits = s_tab[269];
    const uint32_t data_bits = hdr_bits + total_pre + total_span;
    const uint32_t payload = (data_bits + 7u) / 8u;
    const uint32_t out_words = (data_bits + 31u) / 32u;
    const bool stored = payload > n + 5u;
    uint8_t* blk = a.slots + (uint64_t)d.slot * a.slot_stride + kSlotLead;
    uint32_t* words = reinterpret_cast<uint32_t*>(blk + 18);

    uint32_t out_payload;
    if (!stored) {
        const uint32_t hdr_words = (hdr_bits + 31u) / 32u;
        const uint32_t hw4 = (hdr_words + 3u) & ~3u;   // <= 96 <= nthr is NOT guaranteed: loop
        for (uint32_t i = tid; i < hw4; i += nthr) words[i] = i < hdr_words ? s_hdr[i] : 0u;
        const bool overflow = s_misc[17] != 0;
        const uint32_t ppos = hdr_bits + pre_off;
        const uint32_t dst = hdr_bits + total_pre + span_off;
        if (overflow) {
            uint4* w4 = reinterpret_cast<uint4*>(words + hw4);
            const uint32_t n4 = out_words + 2u > hw4 ? (out_words + 2u - hw4 + 3u) / 4u : 0u;
            for (uint32_t i = tid; i < n4; i += nthr) w4[i] = make_uint4(0u, 0u, 0u, 0u);
        } else {
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
        if (pre_bits) {
            const uint32_t wi = ppos >> 5, sh = ppos & 31u, v = pre_tok & 0xFFFFFFu;
            atomicOr(&words[wi], v << sh);
            if (sh + pre_bits > 32) atomicOr(&words[wi + 1], v >> (32 - sh));
        }
        if (worker) {
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
                AEmit em{words, dst};
                LzTokSink<AEmit> ts{em, s_len, s_lits, s_dist, eob};
                lz_span_tokens(mem, 128u * tid, nc, tid == 0, starts_row, p_end, p_last, nall, cfg, ts);
            }
        }
        out_payload = payload;
    } else {
        // stored deflate block (rare safety net), as in k_auto
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
    if (tid < 26) {
        uint32_t delta = s_misc[16];
        if (ends_row) delta = __ldg(&a.crctab[delta & 0xFFu]) ^ (delta >> 8);
        const uint32_t crc32 = ~(delta ^ s_misc[10]);
        const uint32_t bsize = out_payload + 25u;
        if (tid < 16) {
            const uint8_t head[16] = {0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0x00, 0x42, 0x43, 0x02, 0x00};
            blk[tid] = head[tid];
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
#endif  // __CUDACC__

}  // namespace dnaf
