// Host-side set-up for the fused kernels: static Huffman codes per minor-allele-frequency bucket, their
// serialized deflate dynamic-block headers, the token lookup tables and CRC helper tables.
//
// The codes are built from token statistics obtained by running the kernels' own span grammars
// (span_tokens_ref, xspan_tokens_ref, tokenize_words) over Bernoulli(maf) masks from a fixed-seed generator,
// which is the model the reference's row loop samples from (pop_factory.py:477-494).  Every symbol a block can
// need gets a code (add-one smoothing), so any mask pattern -- including forced-minor cells -- stays encodable.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cmath>
#include <cstring>
#include <queue>
#include <vector>

#include "k_fused.cuh"
#include "k_auto.cuh"
#include "k_fused_text.cuh"
#include "k_x.cuh"
#include "k_lz.cuh"

namespace dnaf {
namespace hosttab {

inline uint32_t mulmod(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int i = 0; i < 32; ++i) {
        if (a & 0x80000000u) p ^= b;
        a <<= 1;
        b = (b & 1u) ? (b >> 1) ^ kCrcPoly : (b >> 1);
    }
    return p;
}

inline int len_index(int len) {
    static const int base[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23, 27,
                                 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
    for (int i = 28; i >= 0; --i)
        if (len >= base[i]) return i;
    return 0;
}
static const int kLenBase[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23, 27,
                                 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
static const int kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};

// Huffman code lengths limited to maxbits (frequencies are halved until the tree is shallow enough).
inline std::vector<uint8_t> huff_lengths(const std::vector<uint64_t>& freq_in, int maxbits) {
    const int n = (int)freq_in.size();
    std::vector<uint8_t> lens(n, 0);
    std::vector<int> used;
    for (int i = 0; i < n; ++i)
        if (freq_in[i]) used.push_back(i);
    if (used.empty()) return lens;
    if (used.size() == 1) {
        lens[used[0]] = 1;
        return lens;
    }
    for (int shift = 0;; ++shift) {
        struct Node { uint64_t w; int id; };
        auto cmp = [](const Node& a, const Node& b) { return a.w > b.w || (a.w == b.w && a.id > b.id); };
        std::priority_queue<Node, std::vector<Node>, decltype(cmp)> pq(cmp);
        std::vector<int> parent(2 * used.size(), -1);
        for (size_t i = 0; i < used.size(); ++i) pq.push({std::max<uint64_t>(1, freq_in[used[i]] >> shift), (int)i});
        int next = (int)used.size();
        while (pq.size() > 1) {
            Node a = pq.top(); pq.pop();
            Node b = pq.top(); pq.pop();
            parent[a.id] = next;
            parent[b.id] = next;
            pq.push({a.w + b.w, next});
            ++next;
        }
        int maxd = 0;
        std::vector<int> depth(used.size());
        for (size_t i = 0; i < used.size(); ++i) {
            int d = 0;
            for (int v = (int)i; parent[v] >= 0; v = parent[v]) ++d;
            depth[i] = d;
            maxd = std::max(maxd, d);
        }
        if (maxd <= maxbits) {
            for (size_t i = 0; i < used.size(); ++i) lens[used[i]] = (uint8_t)depth[i];
            return lens;
        }
    }
}

inline uint32_t reverse_bits(uint32_t code, int len) {
    uint32_t r = 0;
    for (int i = 0; i < len; ++i) r |= ((code >> i) & 1u) << (len - 1 - i);
    return r;
}

// canonical codes, bit-reversed; out[i] = code | len << 24
inline std::vector<uint32_t> huff_codes(const std::vector<uint8_t>& lens) {
    uint32_t count[16] = {0}, next[16] = {0};
    for (uint8_t l : lens) count[l]++;
    count[0] = 0;
    uint32_t code = 0;
    for (int b = 1; b < 16; ++b) {
        code = (code + count[b - 1]) << 1;
        next[b] = code;
    }
    std::vector<uint32_t> out(lens.size(), 0);
    for (size_t i = 0; i < lens.size(); ++i)
        if (lens[i]) out[i] = reverse_bits(next[lens[i]]++, lens[i]) | ((uint32_t)lens[i] << 24);
    return out;
}

struct BitString {
    std::vector<uint32_t> words;
    uint32_t bits = 0;
    void put(uint32_t v, int n) {
        for (int i = 0; i < n; ++i, ++bits) {
            if ((bits >> 5) >= words.size()) words.push_back(0);
            if ((v >> i) & 1u) words[bits >> 5] |= 1u << (bits & 31);
        }
    }
};

// BFINAL=1, BTYPE=2 header for literal/length lengths `ll` (286) and the single distance code 3.
inline BitString dynamic_header(const std::vector<uint8_t>& ll) {
    static const int order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    int nlit = 286;
    while (nlit > 257 && ll[nlit - 1] == 0) --nlit;
    std::vector<uint8_t> seq(ll.begin(), ll.begin() + nlit);
    const uint8_t dist[4] = {0, 0, 0, 1};
    seq.insert(seq.end(), dist, dist + 4);
    std::vector<std::pair<int, int>> rl;  // (symbol, extra)
    for (size_t i = 0; i < seq.size();) {
        const int v = seq[i];
        size_t run = 1;
        while (i + run < seq.size() && seq[i + run] == v) ++run;
        i += run;
        if (v == 0) {
            while (run >= 11) { const size_t c = std::min<size_t>(run, 138); rl.push_back({18, (int)c - 11}); run -= c; }
            if (run >= 3) { rl.push_back({17, (int)run - 3}); run = 0; }
            while (run-- > 0) rl.push_back({0, 0});
        } else {
            rl.push_back({v, 0});
            --run;
            while (run >= 3) { const size_t c = std::min<size_t>(run, 6); rl.push_back({16, (int)c - 3}); run -= c; }
            while (run-- > 0) rl.push_back({v, 0});
        }
    }
    std::vector<uint64_t> clf(19, 0);
    for (auto& p : rl) clf[p.first]++;
    std::vector<uint8_t> cll = huff_lengths(clf, 7);
    int used = 0, only = 0;
    for (int i = 0; i < 19; ++i)
        if (cll[i]) { ++used; only = i; }
    if (used == 1) cll[only == 0 ? 1 : 0] = 1;
    std::vector<uint32_t> clc = huff_codes(cll);
    int ncl = 19;
    while (ncl > 4 && cll[order[ncl - 1]] == 0) --ncl;
    BitString bs;
    bs.put(1, 1);
    bs.put(2, 2);
    bs.put(nlit - 257, 5);
    bs.put(4 - 1, 5);
    bs.put(ncl - 4, 4);
    for (int i = 0; i < ncl; ++i) bs.put(cll[order[i]], 3);
    for (auto& p : rl) {
        bs.put(clc[p.first] & 0xFFFFFFu, (int)(clc[p.first] >> 24));
        if (p.first == 16) bs.put(p.second, 2);
        else if (p.first == 17) bs.put(p.second, 3);
        else if (p.first == 18) bs.put(p.second, 7);
    }
    return bs;
}

struct HistSink {
    uint64_t nlit[8] = {0};
    uint64_t nlen[29] = {0};
    void lit(int id) { nlit[id]++; }
    void match(int l) { nlen[len_index(l)]++; }
};

// Codes for cell literals, all match lengths, EOB (+ prefix byte literals when `prefix_hist`) from token counts
// gathered over `blocks` blocks.
inline FusedTable finish_cell_table(const HistSink& h, uint64_t blocks, const uint64_t* prefix_hist) {
    std::vector<uint64_t> f(286, 0);
    const uint8_t lit_byte[5] = {'0', '1', '/', '\t', '\n'};
    const uint64_t scale = 16;  // fixed-point so that per-row prefix averages below one occurrence still count
    for (int i = 0; i < 5; ++i) f[lit_byte[i]] += (h.nlit[i] * scale) / blocks + 1;
    for (int i = 0; i < 29; ++i) f[257 + i] += (h.nlen[i] * scale) / blocks + 1;
    f[256] = scale;
    if (prefix_hist)
        for (int c = 0; c < 256; ++c)
            if (prefix_hist[c]) f[c] += std::max<uint64_t>(1, prefix_hist[c]);
    std::vector<uint8_t> ll = huff_lengths(f, 15);
    // the kernels fuse [match or separator][literal] into one 32-bit token: keep the cell literals <= 10 bits
    while (ll['0'] > 10 || ll['1'] > 10 || ll['/'] > 10 || ll['\t'] > 10) {
        for (uint8_t c : {(uint8_t)'0', (uint8_t)'1', (uint8_t)'/', (uint8_t)'\t'})
            if (ll[c] > 10) f[c] *= 4;
        ll = huff_lengths(f, 15);
    }
    std::vector<uint32_t> lc = huff_codes(ll);
    FusedTable t;
    memset(&t, 0, sizeof t);
    for (int len = 3; len <= 258; ++len) {
        const int ci = len_index(len);
        const uint32_t c = lc[257 + ci];
        const uint32_t cl = c >> 24, ex = (uint32_t)kLenExtra[ci];
        t.len_tok[len] = ((c & 0xFFFFFFu) | ((uint32_t)(len - kLenBase[ci]) << cl)) | ((cl + ex + 1u) << 24);
    }
    for (int i = 0; i < 5; ++i) t.lit[i] = lc[lit_byte[i]];
    t.eob = lc[256];
    for (int c = 0; c < 256; ++c) t.pre_lit[c] = lc[c];
    BitString hdr = dynamic_header(ll);
    t.hdr_bits = hdr.bits;
    for (size_t i = 0; i < hdr.words.size() && i < 62; ++i) t.hdr[i] = hdr.words[i];
    if (hdr.words.size() > 62) t.hdr_bits = 0xFFFFFFFFu;  // caller treats as "no table" (cannot happen: < 1 KiB)
    return t;
}

// ---- k_auto (k_auto.cuh): token statistics under its span grammar, code tables and the byte LUT ----
struct AutoHistSink {
    HistSink h;
    void tok(int gap) {
        if (gap == 1) h.lit(kLitTab);
        else if (gap >= 3) h.match(gap);
    }
    void lit(int id) { h.lit(id); }
    void eob() {}
};

// Token statistics of `blocks` blocks of `per_block` full spans of Bernoulli(p_minor) alleles.
inline HistSink simulate_auto(double p_minor, int blocks, int per_block, bool starts_row) {
    AutoHistSink s;
    uint64_t st = 0x9E3779B97F4A7C15ull ^ (uint64_t)(p_minor * 1e9);
    auto next = [&]() {
        st ^= st << 13; st ^= st >> 7; st ^= st << 17;
        return st;
    };
    const uint64_t thr = (uint64_t)(std::min(p_minor, 0.999999) * 18446744073709551615.0);
    for (int b = 0; b < blocks; ++b) {
        uint32_t carry = 0;
        for (int sp = 0; sp < per_block; ++sp) {
            uint32_t m[4];
            for (int w = 0; w < 4; ++w) {
                uint32_t v = 0;
                for (int i = 0; i < 32; ++i) v |= (uint32_t)(next() < thr) << i;
                m[w] = v;
            }
            span_tokens_ref(m, sp ? carry : (m[0] & 3u), sp == 0, starts_row, 64, false, sp + 1 == per_block, s);
            carry = m[3] >> 30;
        }
    }
    return s.h;
}

// Multiply-by-x^(8*bytes) table [4][256] for reflected CRC values (linear: built from the 32 basis bits).
inline void fill_mul_table(uint32_t xpow /* x^(8*bytes) */, uint32_t* out /* [1024] */) {
    uint32_t basis[32];
    for (int i = 0; i < 32; ++i) basis[i] = mulmod(xpow, 1u << i);
    for (int k = 0; k < 4; ++k)
        for (int b = 0; b < 256; ++b) {
            uint32_t v = 0;
            for (int i = 0; i < 8; ++i)
                if ((b >> i) & 1) v ^= basis[8 * k + i];
            out[256 * k + b] = v;
        }
}

inline AutoTable make_auto_table(double p_minor, const uint64_t* prefix_hist, int per_block, bool starts_row) {
    const int kBlocks = std::max(2, 1024 / std::max(1, per_block));
    const FusedTable f = finish_cell_table(simulate_auto(p_minor, kBlocks, std::max(1, per_block), starts_row), kBlocks, prefix_hist);
    AutoTable t;
    memset(&t, 0, sizeof t);
    if (f.hdr_bits == 0xFFFFFFFFu) {
        t.hdr_bits = f.hdr_bits;
        return t;
    }
    for (int i = 0; i < 260; ++i) t.len_tok[i] = f.len_tok[i];
    t.len_tok[0] = 0;
    t.len_tok[1] = f.lit[kLitTab];
    t.len_tok[2] = 0;  // even gaps of 2 never reach the table
    for (int bit = 0; bit < 2; ++bit) {
        const uint32_t a = f.lit[kLitSlash], b = f.lit[bit];
        t.len_tok[259 + bit] = ((a & 0xFFFFFFu) | ((b & 0xFFFFFFu) << (a >> 24))) | (((a >> 24) + (b >> 24)) << 24);
    }
    for (int i = 0; i < 8; ++i) t.lit[i] = f.lit[i];
    t.eob = f.eob;
    t.hdr_bits = f.hdr_bits;
    memcpy(t.hdr, f.hdr, sizeof t.hdr);
    memcpy(t.pre_lit, f.pre_lit, sizeof t.pre_lit);
    for (uint32_t idx = 0; idx < 1024; ++idx) {
        const uint32_t mb = idx >> 2, xb = (mb ^ idx) & 0xFFu;
        if (!xb) continue;
        unsigned __int128 code = 0;
        uint32_t nb = 0;
        int first = -1, pe = -1;
        auto put = [&](uint32_t tok) {
            if (nb < 100) code |= (unsigned __int128)(tok & 0xFFFFFFu) << nb;
            nb += tok >> 24;
        };
        for (int s = 0; s < 8; ++s) {
            if (!((xb >> s) & 1u)) continue;
            if (first < 0) first = s;
            else {
                const int g = 2 * s - pe;
                put(g == 1 ? f.lit[(s & 1) ? kLitSlash : kLitTab] : t.len_tok[g]);
            }
            put(f.lit[(mb >> s) & 1u]);
            pe = 2 * s + 1;
        }
        const bool is_long = nb > kLutMaxBits;
        const uint64_t c = is_long ? 0 : (uint64_t)code;
        t.lut[idx].x = (uint32_t)c;
        t.lut[idx].y = (uint32_t)((c >> 32) & 0x7FFu) | (is_long ? kLutLong : (nb << 11)) | ((uint32_t)(2 * first) << 24) |
                       ((uint32_t)pe << 28);
    }
    return t;
}

// Static per-population description of the X-row spans (k_x.cuh): compaction masks (Hacker's Delight 7-4
// "compress", move masks precomputed), separator kinds, the per-unit separator windows and static mismatches.
inline std::vector<XSpan> build_xspans(const uint8_t* sex, uint32_t n, const uint32_t* xoff) {
    const uint32_t nspans = (n + 63u) / 64u;
    std::vector<XSpan> out(nspans);
    // separator kinds over the whole row, in compacted-allele order
    std::vector<uint8_t> kinds;
    kinds.reserve((size_t)2 * n);
    for (uint32_t i = 0; i < n; ++i) {
        if (sex[i] == 1) kinds.push_back(0);             // "a\t"
        else { kinds.push_back(1); kinds.push_back(0); } // "a/b\t"
    }
    size_t k0 = 0;
    for (uint32_t sp = 0; sp < nspans; ++sp) {
        XSpan xs;
        memset(&xs, 0, sizeof xs);
        const uint32_t i0 = 64u * sp, i1 = std::min(n, i0 + 64u);
        for (uint32_t i = i0; i < i1; ++i) {
            const uint32_t j = 2u * (i - i0);
            xs.used[j >> 5] |= 1u << (j & 31u);
            if (sex[i] != 1) xs.used[(j + 1) >> 5] |= 1u << ((j + 1) & 31u);
        }
        uint32_t L = 0;
        for (int w = 0; w < 4; ++w) {
            uint32_t m = xs.used[w];
            xs.len[w] = (uint32_t)__builtin_popcount(m);
            uint32_t mk = ~m << 1;
            for (int i = 0; i < 5; ++i) {
                uint32_t mp = mk ^ (mk << 1);
                mp ^= mp << 2;
                mp ^= mp << 4;
                mp ^= mp << 8;
                mp ^= mp << 16;
                const uint32_t mv = mp & m;
                xs.mv[w][i] = mv;
                m = (m ^ mv) | (mv >> (1 << i));
                mk &= ~mp;
            }
            L += xs.len[w];
        }
        xs.L = L;
        // kinds of positions -2 .. 127 of the span; positions past L repeat the pair before them (no mismatch there)
        uint8_t kk[130];
        for (int k = -2; k < 128; ++k) {
            uint8_t v;
            if (k < 0) v = ((long long)k0 + k >= 0) ? kinds[(size_t)((long long)k0 + k)] : 0;
            else if ((uint32_t)k < L) v = kinds[k0 + k];
            else v = kk[k];                                             // = kind of position k - 2
            kk[k + 2] = v;
        }
        xs.skc = (uint32_t)kk[0] | ((uint32_t)kk[1] << 1);
        for (int k = 0; k < 128; ++k)
            if (kk[k + 2]) xs.sk[k >> 5] |= 1u << (k & 31);
        for (int u = 0; u < 32; ++u) {
            uint32_t s6 = 0;
            for (int j = 0; j < 6; ++j) s6 |= (uint32_t)kk[4 * u + j] << j;    // positions 4u-2 .. 4u+3
            xs.sk6[u] = (uint8_t)s6;
            if (((s6 >> 2) ^ s6) & 15u) xs.snz |= 1u << u;
        }
        xs.byte_off = xoff[i0];
        out[sp] = xs;
        k0 += L;
    }
    return out;
}

struct XHistSink {
    HistSink h;
    void tok(int gap) { if (gap >= 3) h.match(gap); }
    void lit(int id) { h.lit(id); }
    void eob() {}
};

// Table for k_x: token statistics of X rows with Bernoulli(p_minor) alleles over the population's real spans,
// the codes, and the 4096-entry unit table.
inline XTable make_x_table(double p_minor, const std::vector<XSpan>& xspans, int per_block, const uint64_t* prefix_hist) {
    XHistSink hs;
    uint64_t st = 0xA24BAED4963EE407ull ^ (uint64_t)(p_minor * 1e9);
    auto next = [&]() {
        st ^= st << 13; st ^= st >> 7; st ^= st << 17;
        return st;
    };
    const uint64_t thr = (uint64_t)(std::min(p_minor, 0.999999) * 18446744073709551615.0);
    const size_t ns = std::min<size_t>(xspans.size(), 512);
    uint32_t carry = 0;
    for (size_t sp = 0; sp < ns; ++sp) {
        const XSpan& xs = xspans[sp];
        uint32_t m[4], c[4];
        for (int w = 0; w < 4; ++w) {
            uint32_t v = 0;
            for (int i = 0; i < 32; ++i) v |= (uint32_t)(next() < thr) << i;
            m[w] = v;
        }
        const uint32_t L = compact_span(m, xs, c);
        if (!L) continue;
        // pad like the kernel: positions past L repeat the pair before them
        for (uint32_t k = L; k < 128; ++k) {
            const uint32_t v = k >= 2 ? bit128(c, (int)k - 2) : 0u;
            c[k >> 5] = (c[k >> 5] & ~(1u << (k & 31))) | (v << (k & 31));
        }
        const bool first = (sp % (size_t)std::max(1, per_block)) == 0;
        xspan_tokens_ref(c, first ? (c[0] & 3u) : carry, xs, (int)xs.L, first, false, false, hs);
        carry = L >= 2 ? ((bit128(c, (int)L - 1) << 1) | bit128(c, (int)L - 2)) : 0u;
    }
    const uint64_t blocks = std::max<uint64_t>(1, ns / (size_t)std::max(1, per_block));
    const FusedTable f = finish_cell_table(hs.h, blocks, prefix_hist);
    XTable t;
    memset(&t, 0, sizeof t);
    t.hdr_bits = f.hdr_bits;
    if (f.hdr_bits == 0xFFFFFFFFu) return t;
    for (int i = 3; i < 260; ++i) t.len_tok[i] = f.len_tok[i];
    for (int i = 0; i < 8; ++i) t.lit[i] = f.lit[i];
    t.eob = f.eob;
    memcpy(t.hdr, f.hdr, sizeof t.hdr);
    memcpy(t.pre_lit, f.pre_lit, sizeof t.pre_lit);
    struct CodeSink {
        const XTable& t;
        unsigned __int128 code = 0;
        uint32_t nb = 0;
        void put(uint32_t tok) {
            if (nb < 100) code |= (unsigned __int128)(tok & 0xFFFFFFu) << nb;
            nb += tok >> 24;
        }
        void lit(int id) { put(t.lit[id]); }
        void tok(int g) { put(t.len_tok[g]); }
    };
    for (uint32_t key = 0; key < 4096; ++key) {
        CodeSink cs{t};
        int lead, lastp;
        xunit_tokens(key & 63u, key >> 6, cs, lead, lastp);
        if (lead < 0) continue;
        const bool is_long = cs.nb > kLutMaxBits;
        const uint64_t c = is_long ? 0 : (uint64_t)cs.code;
        t.lut[key].x = (uint32_t)c;
        t.lut[key].y = (uint32_t)((c >> 32) & 0x7FFu) | (is_long ? kLutLong : (cs.nb << 11)) | ((uint32_t)lead << 24) |
                       ((uint32_t)lastp << 28);
    }
    return t;
}

struct ByteHist {
    uint64_t nlit[256] = {0};
    uint64_t nlen[29] = {0};
    void lit_byte(uint8_t b) { nlit[b]++; }
    void match(int l) { nlen[len_index(l)]++; }
};

// Table for k_fused_text: token statistics of rows of chromosome class `cls` whose alleles are
// Bernoulli(p_minor), laid out with the population's real sex vector (cell widths / '.' depend on it).
inline FusedTable make_text_table(int cls, double p_minor, const uint8_t* sex, uint32_t n,
                                  const uint64_t* prefix_hist) {
    ByteHist h;
    uint64_t st = 0xD1B54A32D192ED03ull ^ (uint64_t)(p_minor * 1e9) ^ ((uint64_t)cls << 56);
    auto next = [&]() {
        st ^= st << 13; st ^= st >> 7; st ^= st << 17;
        return st;
    };
    const uint64_t thr = (uint64_t)(std::min(p_minor, 0.999999) * 18446744073709551615.0);
    const uint32_t ns = std::min<uint32_t>(n, 32768);
    const int reps = ns < 8192 ? 4 : 2;
    uint64_t blocks = 0;
    std::vector<uint8_t> text;
    for (int rep = 0; rep < reps; ++rep) {
        text.clear();
        for (uint32_t i = 0; i < ns; ++i) {
            const bool male = sex[i] == 1;
            const bool wide = cls == kAuto || (cls == kX && !male);
            const uint8_t a0 = '0' + (next() < thr), a1 = '0' + (next() < thr);
            text.push_back((cls == kY && !male) ? '.' : a0);
            if (wide) { text.push_back('/'); text.push_back(a1); }
            text.push_back('\t');
        }
        while (text.size() % 4) text.push_back(0);
        const uint32_t* words = reinterpret_cast<const uint32_t*>(text.data());
        const size_t total = (size_t)ns * 0 + text.size();
        size_t pos = 0;
        int span_in_block = 0;
        while (pos < total) {
            const int nb = (int)std::min<size_t>(256, total - pos);
            const uint32_t* w = words + pos / 4;
            auto wat = [&](int k) { return w[k]; };
            tokenize_words(wat, nb, span_in_block > 0, span_in_block > 0 ? w[-1] : 0u, h);
            pos += nb;
            if (++span_in_block == 254) { span_in_block = 0; ++blocks; }
        }
        ++blocks;
    }
    std::vector<uint64_t> f(286, 0);
    const uint64_t scale = 16;
    for (int c = 0; c < 256; ++c)
        if (h.nlit[c]) f[c] += (h.nlit[c] * scale) / blocks + 1;
    for (const char* c = "0123./\t\n"; *c; ++c) f[(uint8_t)*c] += 1;
    for (int i = 0; i < 29; ++i) f[257 + i] += (h.nlen[i] * scale) / blocks + 1;
    f[256] = scale;
    if (prefix_hist)
        for (int c = 0; c < 256; ++c)
            if (prefix_hist[c]) f[c] += std::max<uint64_t>(1, prefix_hist[c]);
    std::vector<uint8_t> ll = huff_lengths(f, 15);
    std::vector<uint32_t> lc = huff_codes(ll);
    FusedTable t;
    memset(&t, 0, sizeof t);
    for (int len = 3; len <= 258; ++len) {
        const int ci = len_index(len);
        const uint32_t c = lc[257 + ci];
        const uint32_t cl = c >> 24, ex = (uint32_t)kLenExtra[ci];
        t.len_tok[len] = ((c & 0xFFFFFFu) | ((uint32_t)(len - kLenBase[ci]) << cl)) | ((cl + ex + 1u) << 24);
    }
    t.eob = lc[256];
    for (int c = 0; c < 256; ++c) t.pre_lit[c] = lc[c];
    BitString hdr = dynamic_header(ll);
    t.hdr_bits = hdr.bits;
    for (size_t i = 0; i < hdr.words.size() && i < 62; ++i) t.hdr[i] = hdr.words[i];
    if (hdr.words.size() > 62) t.hdr_bits = 0xFFFFFFFFu;
    return t;
}

// ---- k_lz (k_lz.cuh): the LZ tiers' chains on the host, token statistics under lz_span_tokens, code tables ----
// Host twin of the shared-memory structures k_lz builds per block: allele bits, prev[] and the per-region heads.
struct LzHostMem {
    std::vector<uint32_t> bits;     // + guard words
    std::vector<uint16_t> prv;
    std::vector<uint16_t> hd;       // [region][2^(key+1)]
    uint32_t hbits = 0;
    uint32_t word(uint32_t i) const { return bits[i]; }
    uint32_t prev(uint32_t a) const { return prv[a]; }
    uint32_t head(uint32_t reg, uint32_t key) const { return hd[((size_t)reg << hbits) + key]; }
    // bits must hold (nall + 31) / 32 words.  Same structure as the kernel builds: steps of 32 consecutive positions;
    // every position of a step points at the key's last occurrence BEFORE the step, the step's last occurrence of a
    // key becomes the head.
    void build(uint32_t nall, uint32_t key_alleles) {
        const uint32_t words = (nall + 31u) / 32u;
        bits.resize(words + 8u, 0u);
        for (uint32_t i = words; i < words + 8u; ++i) bits[i] = 0u;
        if (nall & 31u) bits[words - 1u] &= (1u << (nall & 31u)) - 1u;
        hbits = key_alleles + 1u;
        const uint32_t nreg = (nall + kLzRegion - 1u) / kLzRegion;
        prv.assign((size_t)nreg * kLzRegion, (uint16_t)kLzNone);
        hd.assign((size_t)nreg << hbits, (uint16_t)kLzNone);
        const uint32_t kmask = (1u << key_alleles) - 1u;
        uint32_t keys[32];
        for (uint32_t pos = 0; pos < nall; pos += 32u) {
            const uint32_t reg = pos / kLzRegion;
            const uint32_t n = std::min(32u, ((nall + 31u) & ~31u) - pos);
            for (uint32_t l = 0; l < n; ++l) {
                const uint32_t a = pos + l, w = a >> 5, sh = a & 31u;
                keys[l] = (lz_fsr(bits[w], bits[w + 1u], sh) & kmask) | ((a & 1u) << key_alleles);
                prv[a] = hd[((size_t)reg << hbits) + keys[l]];
            }
            for (uint32_t l = n; l-- > 0;) hd[((size_t)reg << hbits) + keys[l]] = (uint16_t)(pos + l);   // descending: the step's FIRST occurrence stays
        }
    }
};

struct LzHist {
    uint64_t nlit[8] = {0};
    uint64_t nlen[29] = {0};
    uint64_t ndist[30] = {0};
    uint64_t extra = 0;
    void emit(bool is_match, int id, int len, int dist) {
        if (!is_match) {
            nlit[id]++;
            return;
        }
        const int li = len_index(len);
        nlen[li]++;
        uint32_t sym, eb, ev;
        lz_dist_sym((uint32_t)dist, sym, eb, ev);
        ndist[sym]++;
        extra += (uint64_t)kLenExtra[li] + eb;
    }
    void eob() {}
};

// Token statistics of `blocks` blocks of `per_block` full spans of Bernoulli(p_minor) alleles under the LZ grammar.
inline LzHist simulate_lz(double p_minor, int blocks, int per_block, bool starts_row, const LzCfg cfg) {
    LzHist h;
    uint64_t st = 0x9E3779B97F4A7C15ull ^ (uint64_t)(p_minor * 1e9);
    auto next = [&]() {
        st ^= st << 13; st ^= st >> 7; st ^= st << 17;
        return st;
    };
    const uint64_t thr = (uint64_t)(std::min(p_minor, 0.999999) * 18446744073709551615.0);
    LzHostMem mem;
    const uint32_t nall = 128u * (uint32_t)per_block;
    for (int b = 0; b < blocks; ++b) {
        mem.bits.assign(4u * per_block + 8u, 0u);
        for (int w = 0; w < 4 * per_block; ++w) {
            uint32_t v = 0;
            for (int i = 0; i < 32; ++i) v |= (uint32_t)(next() < thr) << i;
            mem.bits[w] = v;
        }
        mem.build(nall, cfg.key);
        for (int sp = 0; sp < per_block; ++sp)
            lz_span_tokens(mem, 128u * sp, 64, sp == 0, starts_row, false, sp + 1 == per_block, nall, cfg, h);
    }
    return h;
}

// BFINAL=1, BTYPE=2 header for literal/length lengths `ll` (286) and distance lengths `dl` (30).
inline BitString dynamic_header2(const std::vector<uint8_t>& ll, const std::vector<uint8_t>& dl) {
    static const int order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    int nlit = 286, ndist = 30;
    while (nlit > 257 && ll[nlit - 1] == 0) --nlit;
    while (ndist > 1 && dl[ndist - 1] == 0) --ndist;
    std::vector<uint8_t> seq(ll.begin(), ll.begin() + nlit);
    seq.insert(seq.end(), dl.begin(), dl.begin() + ndist);
    std::vector<std::pair<int, int>> rl;  // (symbol, extra)
    for (size_t i = 0; i < seq.size();) {
        const int v = seq[i];
        size_t run = 1;
        while (i + run < seq.size() && seq[i + run] == v) ++run;
        i += run;
        if (v == 0) {
            while (run >= 11) { const size_t c = std::min<size_t>(run, 138); rl.push_back({18, (int)c - 11}); run -= c; }
            if (run >= 3) { rl.push_back({17, (int)run - 3}); run = 0; }
            while (run-- > 0) rl.push_back({0, 0});
        } else {
            rl.push_back({v, 0});
            --run;
            while (run >= 3) { const size_t c = std::min<size_t>(run, 6); rl.push_back({16, (int)c - 3}); run -= c; }
            while (run-- > 0) rl.push_back({v, 0});
        }
    }
    std::vector<uint64_t> clf(19, 0);
    for (auto& p : rl) clf[p.first]++;
    std::vector<uint8_t> cll = huff_lengths(clf, 7);
    int used = 0, only = 0;
    for (int i = 0; i < 19; ++i)
        if (cll[i]) { ++used; only = i; }
    if (used == 1) cll[only == 0 ? 1 : 0] = 1;
    std::vector<uint32_t> clc = huff_codes(cll);
    int ncl = 19;
    while (ncl > 4 && cll[order[ncl - 1]] == 0) --ncl;
    BitString bs;
    bs.put(1, 1);
    bs.put(2, 2);
    bs.put(nlit - 257, 5);
    bs.put(ndist - 1, 5);
    bs.put(ncl - 4, 4);
    for (int i = 0; i < ncl; ++i) bs.put(cll[order[i]], 3);
    for (auto& p : rl) {
        bs.put(clc[p.first] & 0xFFFFFFu, (int)(clc[p.first] >> 24));
        if (p.first == 16) bs.put(p.second, 2);
        else if (p.first == 17) bs.put(p.second, 3);
        else if (p.first == 18) bs.put(p.second, 7);
    }
    return bs;
}

// estimated payload bits of a histogram under its own optimal codes (for choosing the key length of a bucket)
inline double lz_hist_bits(const LzHist& h) {
    auto ent = [](const uint64_t* f, int n) {
        double tot = 0, bits = 0;
        for (int i = 0; i < n; ++i) tot += (double)f[i];
        for (int i = 0; i < n; ++i)
            if (f[i]) bits -= (double)f[i] * std::log2((double)f[i] / tot);
        return bits;
    };
    uint64_t ll[37];
    for (int i = 0; i < 8; ++i) ll[i] = h.nlit[i];
    for (int i = 0; i < 29; ++i) ll[8 + i] = h.nlen[i];
    return ent(ll, 37) + ent(h.ndist, 30) + (double)h.extra;
}

// Key length of a MAF bucket: rare minor alleles want long keys (few, long matches), common ones short keys.
inline uint32_t lz_key_for(double p_minor) {
    const double p = std::min(p_minor, 1.0 - p_minor);
    return std::min<uint32_t>(kLzMaxKey, p < 0.22 ? 9u : 8u);   // the kernel sizes its head tables for kLzMaxKey
}

// Codes + header of one candidate parse configuration; *total_bits = payload under these codes + the header, per block
inline LzTable fit_lz_table(double p_minor, const uint64_t* prefix_hist, int per_block, bool starts_row, const LzCfg cfg,
                            double* total_bits) {
    const int kBlocks = std::max(2, 512 / std::max(1, per_block));
    const LzHist h = simulate_lz(p_minor, kBlocks, std::max(1, per_block), starts_row, cfg);
    std::vector<uint64_t> f(286, 0), fd(30, 0);
    const uint8_t lit_byte[5] = {'0', '1', '/', '\t', '\n'};
    const uint64_t scale = 16, blocks = (uint64_t)kBlocks;
    for (int i = 0; i < 5; ++i) f[lit_byte[i]] += (h.nlit[i] * scale) / blocks + 1;
    for (int i = 0; i < 29; ++i) f[257 + i] += (h.nlen[i] * scale) / blocks + 1;
    f[256] = scale;
    if (prefix_hist)
        for (int c = 0; c < 256; ++c)
            if (prefix_hist[c]) f[c] += std::max<uint64_t>(1, prefix_hist[c]);
    // every distance a block can need gets a code: multiples of 4 up to 32768 (symbols 3 and 5..29) with the key
    // chains, only 4 and 8 (symbols 3 and 5) without
    for (int i = 3; i < (cfg.chain ? 30 : 6); ++i)
        if (i != 4) fd[i] = (h.ndist[i] * scale) / blocks + 1;
    std::vector<uint8_t> ll = huff_lengths(f, 15), dl = huff_lengths(fd, 15);
    std::vector<uint32_t> lc = huff_codes(ll), dc = huff_codes(dl);
    LzTable t;
    memset(&t, 0, sizeof t);
    for (int len = 3; len <= 258; ++len) {
        const int ci = len_index(len);
        const uint32_t c = lc[257 + ci];
        const uint32_t cl = c >> 24, ex = (uint32_t)kLenExtra[ci];
        t.len_tok[len] = ((c & 0xFFFFFFu) | ((uint32_t)(len - kLenBase[ci]) << cl)) | ((cl + ex) << 24);
    }
    for (int i = 0; i < 5; ++i) t.lit[i] = lc[lit_byte[i]];
    t.eob = lc[256];
    for (int i = 0; i < 30; ++i) t.dist_tok[i] = dc[i];
    t.key_alleles = cfg.key;
    t.chain = cfg.chain;
    t.lazy = cfg.lazy;
    t.nice = cfg.nice;
    for (int c = 0; c < 256; ++c) t.pre_lit[c] = lc[c];
    BitString hdr = dynamic_header2(ll, dl);
    t.hdr_bits = hdr.bits;
    for (size_t i = 0; i < hdr.words.size() && i < 94; ++i) t.hdr[i] = hdr.words[i];
    if (hdr.words.size() > 94) t.hdr_bits = 0xFFFFFFFFu;
    // payload under the codes just built
    double bits = (double)h.extra;
    for (int i = 0; i < 5; ++i) bits += (double)h.nlit[i] * ll[lit_byte[i]];
    for (int i = 0; i < 29; ++i) bits += (double)h.nlen[i] * ll[257 + i];
    for (int i = 0; i < 30; ++i) bits += (double)h.ndist[i] * dl[i];
    *total_bits = bits / (double)blocks + (double)hdr.bits;
    return t;
}

// The table of a bucket at a level: the level's own parse, or the near-distances-only parse when that compresses the
// bucket's rows at least as well (rare minor alleles: few far matches, and a 27-symbol distance code costs header
// bytes in every block) -- those blocks then skip the chain build altogether.
inline LzTable make_lz_table(double p_minor, const uint64_t* prefix_hist, int per_block, bool starts_row, int level) {
    const LzCfg full = lz_cfg(level, lz_key_for(p_minor));
    double bits_full = 0, bits_near = 0;
    LzTable t = fit_lz_table(p_minor, prefix_hist, per_block, starts_row, full, &bits_full);
    if (full.chain) {
        LzCfg near = full;
        near.chain = 0;
        const LzTable tn = fit_lz_table(p_minor, prefix_hist, per_block, starts_row, near, &bits_near);
        if (tn.hdr_bits != 0xFFFFFFFFu && (t.hdr_bits == 0xFFFFFFFFu || bits_near <= bits_full)) t = tn;
    }
    return t;
}

// Host-side deflate block of one autosome segment under an LzTable (self-test of grammar + codes + header; the
// product path is k_lz).  bits: the block's allele bits; returns the raw deflate bytes.
struct LzBitSink {
    BitString bs;
    const LzTable& t;
    explicit LzBitSink(const LzTable& tt) : t(tt) {}
    void tok(uint32_t v) { bs.put(v & 0xFFFFFFu, (int)(v >> 24)); }
    void emit(bool is_match, int id, int len, int dist) {
        if (!is_match) {
            tok(t.lit[id]);
            return;
        }
        tok(t.len_tok[len]);
        uint32_t sym, eb, ev;
        lz_dist_sym((uint32_t)dist, sym, eb, ev);
        tok(t.dist_tok[sym]);
        bs.put(ev, (int)eb);
    }
    void eob() { tok(t.eob); }
};

inline std::vector<uint8_t> lz_encode_block_host(const LzTable& t, const uint32_t* bits, uint32_t ncells, const uint8_t* prefix,
                                                 uint32_t plen, bool ends_row, int level) {
    LzHostMem mem;
    const uint32_t nall = 2u * ncells;
    mem.bits.assign(bits, bits + (nall + 31u) / 32u);
    mem.build(nall, t.key_alleles);
    LzBitSink sink(t);
    for (uint32_t i = 0; i < (t.hdr_bits + 31u) / 32u; ++i) {
        const uint32_t nb = std::min(32u, t.hdr_bits - 32u * i);
        sink.bs.put(t.hdr[i], (int)nb);
    }
    const bool starts_row = plen > 0;
    for (uint32_t i = 0; i < plen; ++i) sink.tok(t.pre_lit[prefix[i]]);
    (void)level;
    const LzCfg cfg{t.chain, t.lazy, t.key_alleles, t.nice};
    const uint32_t nspans = (ncells + 63u) / 64u;
    for (uint32_t sp = 0; sp < nspans; ++sp) {
        const int nc = (int)std::min(64u, ncells - 64u * sp);
        const bool last = sp + 1u == nspans;
        lz_span_tokens(mem, 128u * sp, nc, sp == 0, starts_row, ends_row && last, last, nall, cfg, sink);
    }
    std::vector<uint8_t> out((sink.bs.bits + 7u) / 8u);
    for (size_t i = 0; i < out.size(); ++i) out[i] = (uint8_t)(sink.bs.words[i >> 2] >> (8 * (i & 3)));
    return out;
}

}  // namespace hosttab
}  // namespace dnaf
