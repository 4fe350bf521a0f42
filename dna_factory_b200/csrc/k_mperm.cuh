// max(T) permutation tests of ALLELIC and REC (dnaf_mperm, pop_factory --mperm; DESIGN.md 5, "Permutation tests").
//
// Permutation p (0-based) is a uniformly random subset of exactly ncase of the N samples, drawn by selection sampling
// (Knuth's Algorithm S): for i = 0..N-1 with `need` starting at ncase, sample i is a case iff
//   (uint64)U(p,i) * (N - i) < (uint64)need << 32,   then need -= 1,
//   U(p,i) = philox4x32_10(ctr = (i >> 2, p, 0x4D505200, 0xFFFFFFFF), key = (seed_lo, seed_hi))[i & 3].
// Integer-only, always exactly ncase cases, bias at most 2^-32 a step.  Word 3 = 0xFFFFFFFF is never a genotype row's
// counter (DESIGN.md 3) and word 2 differs from SNP selection's 0x534E5000 / 0x534E5001, so the stream is disjoint
// from both; it depends on (seed, N, ncase, p) only.
//
// Statistics (T_obs of a row and T_p of every permutation): ALLELIC is the .assoc CHISQ (haploid cells count),
// REC the 2x2 Pearson n11 | n12 + n22 over the diploid cells, no cell rule; both through chi2_2x2 (shared with the
// .model formatter), NaN where a denominator is 0.  A permutation's case margins follow from the row class and its
// (male, female) case counts m, f:
//   case alleles:        autosome 2(m + f), X 2f + m, Y m, MT m + f
//   case diploid cells:  autosome m + f,    X f,      Y and MT 0 (no REC)
// and the row totals come from k_geno's counts of the same pass.  Case ALT alleles under p are popc(A & cs) +
// popc(B & cs) and case ALT/ALT cells popc(B & cs), with the one-bit-per-sample planes of k_mperm_planes:
//   A = the printed cell carries an ALT (diploid 0/1 or 1/1, haploid ALT),  B = diploid 1/1.
// T_p counts as at least T_obs when T_p >= T_obs (1 - kHweTie); a row whose T_obs is NaN has no test and takes no part
// in any maximum, and a NaN T_p counts nowhere.
//
// Kernels:
//   k_perm_masks    one thread per permutation runs Algorithm S; word w of permutation j goes to
//                   masks[j * pitch_p + w * pitch_w] (bit i & 31 of word i >> 5 = sample i is a case), and its (m, f)
//                   to sexcnt[j][2].
//   k_mperm_planes  k_geno's draw, row counter and forced minors, compacted to the A / B planes [rows][pitch].
//   k_mperm         a binary "GEMM": a CTA takes 64 rows x 64 permutations and walks the sample words in steps of 32,
//                   staged in shared memory; each thread keeps 4 x 4 (row, permutation) pairs of (popc(A & cs),
//                   popc(B & cs)) in registers, then computes T_p in double, adds per-row exceedance counts with
//                   integer atomicAdd and folds per-permutation maxima with atomicMax on the bit pattern of the
//                   non-negative double.  Both are order-independent, so the results are deterministic.
#pragma once
#include "k_geno.cuh"

namespace dnaf {

constexpr uint32_t kMpermTag = 0x4D505200u;   // Philox counter word 2 of the permutation stream
constexpr uint32_t kPermMaskThreads = 32;
constexpr uint32_t kMpermTile = 64;           // rows and permutations of one k_mperm CTA
constexpr uint32_t kMpermKw = 32;             // sample words staged a step; plane and mask rows are padded to a multiple
constexpr uint32_t kMpermThreads = 256;       // 16 x 16 threads, 4 x 4 (row, permutation) pairs each

// Pearson 2x2 (cases a, b / controls c, d), no continuity correction; the .assoc expression.  NaN: no test.
__host__ __device__ inline double chi2_2x2(double a, double b, double c, double d) {
    const double den = (a + b) * (c + d) * (a + c) * (b + d);
    return den > 0 ? (a + b + c + d) * (a * d - b * c) * (a * d - b * c) / den : nan("");
}

struct PermMaskArgs {
    const uint8_t* sex;       // per sample, 1 = male
    uint32_t n, ncase;
    uint32_t first;           // permutation index of thread 0
    uint32_t n_perm;
    uint64_t pitch_p, pitch_w;
    uint32_t k0, k1;          // seed
    uint32_t* masks;
    uint32_t* sexcnt;         // [n_perm][2]: male cases, female cases
};

__global__ void __launch_bounds__(kPermMaskThreads) k_perm_masks(const PermMaskArgs a) {
    const uint32_t j = blockIdx.x * kPermMaskThreads + threadIdx.x;
    if (j >= a.n_perm) return;
    const uint32_t p = a.first + j;
    uint32_t* dst = a.masks + (uint64_t)j * a.pitch_p;
    uint32_t need = a.ncase, word = 0, males = 0;
    for (uint32_t i4 = 0; i4 < a.n; i4 += 4) {
        const uint4 r = philox4x32_10(i4 >> 2, p, kMpermTag, 0xFFFFFFFFu, a.k0, a.k1);
        const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (uint32_t q = 0; q < 4; ++q) {
            const uint32_t i = i4 + q;
            if (i < a.n) {
                if ((uint64_t)u[q] * (a.n - i) < ((uint64_t)need << 32)) {
                    --need;
                    word |= 1u << (i & 31u);
                    males += __ldg(&a.sex[i]) == 1;
                }
                if ((i & 31u) == 31u || i + 1 == a.n) {
                    dst[(uint64_t)(i >> 5) * a.pitch_w] = word;
                    word = 0;
                }
            }
        }
    }
    a.sexcnt[2 * j] = males;
    a.sexcnt[2 * j + 1] = a.ncase - males;
}

struct MpermPlaneArgs {
    const uint8_t* cls;       // as in GenoArgs
    const uint8_t* k;
    const uint32_t* thr;
    const uint2* sexmask;
    const uint64_t* orow;
    const uint32_t* osamp;
    uint64_t n_over;
    uint64_t row0;            // first row of the pass
    uint64_t row_base;        // Philox row counter = row_base + row
    uint32_t n;
    uint32_t groups;          // ceil(n / 16)
    uint32_t tiles;           // CTAs per row: ceil(groups / kGenoThreads)
    uint32_t k0, k1;
    uint32_t pitch;           // words per plane row
    uint32_t* plane_a;        // [rows of the pass][pitch], row 0 = row0
    uint32_t* plane_b;
    uint32_t* exceed;         // [rows of the pass][2]: zeroed here, summed by k_mperm
};

// bits 0, 2, ..., 30 of x -> bits 0..15
__device__ __forceinline__ uint32_t even_bits(uint32_t x) {
    x &= 0x55555555u;
    x = (x | (x >> 1)) & 0x33333333u;
    x = (x | (x >> 2)) & 0x0F0F0F0Fu;
    x = (x | (x >> 4)) & 0x00FF00FFu;
    return (x | (x >> 8)) & 0x0000FFFFu;
}

__global__ void __launch_bounds__(kGenoThreads) k_mperm_planes(const MpermPlaneArgs a) {
    __shared__ uint32_t s_w[kGenoThreads];
    __shared__ uint64_t s_ovr[2];
    const uint32_t rl = blockIdx.x / a.tiles, tile = blockIdx.x - rl * a.tiles;
    const uint64_t row = a.row0 + rl;
    const uint32_t tid = threadIdx.x;
    const uint32_t g = tile * kGenoThreads + tid;
    const bool live = g < a.groups;
    if (tid < 2) s_ovr[tid] = bed_lower_bound(a.orow, a.n_over, row + tid);
    if (tile == 0 && tid < 2) a.exceed[2ull * rl + tid] = 0u;
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
    // forced minors, as in k_geno
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
    const uint32_t d0 = D & E;
    const uint32_t pa = even_bits(((w | (w >> 1)) & d0) | (w & H)), pb = even_bits(w & (w >> 1) & d0);
    // two 16-sample groups make one 32-sample word: the even thread writes it
    const uint32_t qa = __shfl_down_sync(0xFFFFFFFFu, pa, 1), qb = __shfl_down_sync(0xFFFFFFFFu, pb, 1);
    if (live && !(tid & 1u)) {
        const uint64_t at = (uint64_t)rl * a.pitch + (g >> 1);
        a.plane_a[at] = pa | (qa << 16);
        a.plane_b[at] = pb | (qb << 16);
    }
}

struct MpermArgs {
    const uint32_t* plane_a;  // [rows of the pass, padded to 64][pitch] (k_mperm_planes)
    const uint32_t* plane_b;
    const uint32_t* masks;    // [permutations, padded to 64 with empty masks][pitch] (k_perm_masks)
    const uint32_t* sexcnt;   // [permutations][2]
    const uint32_t* counts;   // [rows of the pass][10] (k_geno)
    const uint8_t* cls;
    uint64_t row0;            // first row of the pass
    uint32_t rows;            // rows of the pass
    uint32_t n_perm;
    uint32_t ptiles;          // permutation tiles: ceil(n_perm / 64)
    uint32_t pitch;           // words per plane / mask row, a multiple of kMpermKw
    double* t_obs;            // [rows of the pass][2] ALLELIC, REC (written by the CTAs of permutation tile 0)
    uint32_t* exceed;         // [rows of the pass][2] #{p : T_p >= T_obs (1 - kHweTie)}
    unsigned long long* max_t;   // [n_perm][2] max over rows of T_p (bit patterns of non-negative doubles)
};

// ALLELIC and REC of one row: a = case ALT alleles, h = case ALT/ALT cells, ca / cd = case alleles / diploid cells;
// alt, obs, hom, dip = the row's totals (cases + controls)
__device__ __forceinline__ void mperm_stats(double a, double h, double ca, double cd, const double* tot, double t[2]) {
    t[0] = chi2_2x2(a, ca - a, tot[0] - a, (tot[1] - ca) - (tot[0] - a));
    t[1] = chi2_2x2(h, cd - h, tot[2] - h, (tot[3] - cd) - (tot[2] - h));
}

__global__ void __launch_bounds__(kMpermThreads, 2) k_mperm(const MpermArgs a) {
    constexpr uint32_t T = kMpermTile, S = kMpermKw + 4;   // row stride: 16-byte aligned, conflict-free phases
    __shared__ __align__(16) uint32_t s_a[T][S];
    __shared__ __align__(16) uint32_t s_b[T][S];
    __shared__ __align__(16) uint32_t s_m[T][S];
    __shared__ double s_tot[T][4];      // alt, obs, hom, dip of the row
    __shared__ double s_thr[T][2];      // T_obs (1 - kHweTie), NaN: no test
    __shared__ uint32_t s_cls[T];
    __shared__ uint32_t s_mf[T][2];     // (male, female) cases of the permutation
    __shared__ unsigned long long s_max[kMpermThreads / 32][T][2];
    const uint32_t ptile = blockIdx.x % a.ptiles, rtile = blockIdx.x / a.ptiles;
    const uint32_t r0 = rtile * T, p0 = ptile * T;
    const uint32_t tid = threadIdx.x, tx = tid & 15u, ty = tid >> 4;
    if (tid < T) {
        const uint32_t r = r0 + tid;
        double thr[2] = {nan(""), nan("")};
        if (r < a.rows) {
            const uint32_t* c = a.counts + (uint64_t)kGenoWords * r;
            const double alt_a = 2.0 * c[2] + c[1] + c[4], alt_u = 2.0 * c[7] + c[6] + c[9];
            const double ca = 2.0 * c[0] + c[3], cu = 2.0 * c[5] + c[8];
            s_tot[tid][0] = alt_a + alt_u;
            s_tot[tid][1] = ca + cu;
            s_tot[tid][2] = (double)c[2] + c[7];
            s_tot[tid][3] = (double)c[0] + c[5];
            s_cls[tid] = __ldg(&a.cls[a.row0 + r]);
            double t[2];
            mperm_stats(alt_a, c[2], ca, c[0], s_tot[tid], t);
            if (ptile == 0) {
                a.t_obs[2ull * r] = t[0];
                a.t_obs[2ull * r + 1] = t[1];
            }
            thr[0] = t[0] * (1.0 - kHweTie);
            thr[1] = t[1] * (1.0 - kHweTie);
        }
        s_thr[tid][0] = thr[0];
        s_thr[tid][1] = thr[1];
    } else if (tid < 2 * T) {
        const uint32_t j = tid - T, p = p0 + j;
        s_mf[j][0] = p < a.n_perm ? __ldg(&a.sexcnt[2 * p]) : 0u;
        s_mf[j][1] = p < a.n_perm ? __ldg(&a.sexcnt[2 * p + 1]) : 0u;
    }
    uint32_t acc_a[4][4], acc_b[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc_a[i][j] = acc_b[i][j] = 0u;
    const uint32_t* ga = a.plane_a + (uint64_t)r0 * a.pitch;
    const uint32_t* gb = a.plane_b + (uint64_t)r0 * a.pitch;
    const uint32_t* gm = a.masks + (uint64_t)p0 * a.pitch;
    for (uint32_t k0 = 0; k0 < a.pitch; k0 += kMpermKw) {
        __syncthreads();
#pragma unroll
        for (uint32_t q = tid; q < T * kMpermKw / 4; q += kMpermThreads) {   // 8 threads a 128-byte row piece
            const uint32_t r = q >> 3, c4 = (q & 7u) * 4u;
            const uint64_t off = (uint64_t)r * a.pitch + k0 + c4;
            *reinterpret_cast<uint4*>(&s_a[r][c4]) = __ldg(reinterpret_cast<const uint4*>(ga + off));
            *reinterpret_cast<uint4*>(&s_b[r][c4]) = __ldg(reinterpret_cast<const uint4*>(gb + off));
            *reinterpret_cast<uint4*>(&s_m[r][c4]) = __ldg(reinterpret_cast<const uint4*>(gm + off));
        }
        __syncthreads();
#pragma unroll 2
        for (uint32_t k = 0; k < kMpermKw; k += 4) {
            uint4 M[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) M[j] = *reinterpret_cast<const uint4*>(&s_m[tx + 16 * j][k]);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint4 A = *reinterpret_cast<const uint4*>(&s_a[ty + 16 * i][k]);
                const uint4 B = *reinterpret_cast<const uint4*>(&s_b[ty + 16 * i][k]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    acc_a[i][j] += __popc(A.x & M[j].x) + __popc(A.y & M[j].y) + __popc(A.z & M[j].z) + __popc(A.w & M[j].w);
                    acc_b[i][j] += __popc(B.x & M[j].x) + __popc(B.y & M[j].y) + __popc(B.z & M[j].z) + __popc(B.w & M[j].w);
                }
            }
        }
    }
    // epilogue: rows ty + 16 i, permutations tx + 16 j
    uint32_t ex[4][2];
    unsigned long long mx[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i) ex[i][0] = ex[i][1] = 0u, mx[i][0] = mx[i][1] = 0ull;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t rr = ty + 16 * i;
        if (r0 + rr >= a.rows) continue;
        const uint32_t cls = s_cls[rr];
        const double thr0 = s_thr[rr][0], thr1 = s_thr[rr][1];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t pj = tx + 16 * j;
            if (p0 + pj >= a.n_perm) continue;
            const double m = s_mf[pj][0], f = s_mf[pj][1];
            const double ca = cls == kAuto ? 2.0 * (m + f) : cls == kX ? 2.0 * f + m : cls == kY ? m : m + f;
            const double cd = cls == kAuto ? m + f : cls == kX ? f : 0.0;
            double t[2];
            mperm_stats((double)acc_a[i][j] + acc_b[i][j], acc_b[i][j], ca, cd, s_tot[rr], t);
            ex[i][0] += t[0] >= thr0;
            ex[i][1] += t[1] >= thr1;
            if (!isnan(thr0) && !isnan(t[0])) mx[j][0] = max(mx[j][0], (unsigned long long)__double_as_longlong(t[0]));
            if (!isnan(thr1) && !isnan(t[1])) mx[j][1] = max(mx[j][1], (unsigned long long)__double_as_longlong(t[1]));
        }
    }
    // exceedance: the 16 threads of a row are one half-warp
    const uint32_t lane = tid & 31u, half = 0xFFFFu << (lane & 16u);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const uint32_t v = __reduce_add_sync(half, ex[i][t]);
            if (tx == 0 && v) atomicAdd(&a.exceed[2ull * (r0 + ty + 16 * i) + t], v);
        }
    // maxima: lanes l and l ^ 16 share the permutation, then the eight warps through shared memory
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int t = 0; t < 2; ++t) {
            const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, mx[j][t], 16);
            if (lane < 16) s_max[tid >> 5][tx + 16 * j][t] = max(mx[j][t], o);
        }
    __syncthreads();
    if (tid < 2 * T) {
        const uint32_t pj = tid >> 1, t = tid & 1u;
        unsigned long long v = 0;
#pragma unroll
        for (uint32_t w = 0; w < kMpermThreads / 32; ++w) v = max(v, s_max[w][pj][t]);
        if (v && p0 + pj < a.n_perm) atomicMax(&a.max_t[2ull * (p0 + pj) + t], v);
    }
}

}  // namespace dnaf
