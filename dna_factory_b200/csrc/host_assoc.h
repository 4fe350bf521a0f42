// Host side of the case/control allele counts (k_assoc.cuh) and the .assoc text formatter, and the pass driver of
// every per-row count kernel (k_assoc here, k_geno in host_geno.h).  Rows [row_begin,row_end) go in passes bounded by
// the 2^31-CTA grid and by chunk_bytes of device output (16 bytes a row for k_assoc); every pass zeroes its
// [rows][words] counters, runs its kernels and, unless the call is device-only, ends with the copies into the
// caller's buffers.  Included by dnaf_api.cu after host_bed.h.
#pragma once

#include <cmath>

namespace {

// Per 16-sample group: bit pairs (2i, 2i+1) of the cases (is_control[i] == 0) (dnaf_set_samples).
std::vector<uint32_t> assoc_case_masks(const uint8_t* is_control, uint32_t n) {
    std::vector<uint32_t> m((size_t)((n + 15u) / 16u), 0u);
    for (uint32_t i = 0; i < n; ++i)
        if (!is_control[i]) m[i / 16u] |= 3u << (2u * (i % 16u));
    return m;
}

// Refuses rows of more than 2 alleles before any launch (`test` names what counts them).
int check_biallelic(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, const char* test) {
    if (!c->have_samples || !c->have_snps) return fail(c, DNAF_E_ARG, "set_samples and set_snps must be called first");
    if (row_begin > row_end || row_end > c->S) return fail(c, DNAF_E_ARG, "row range out of bounds");
    for (uint64_t r = row_begin; r < row_end; ++r)
        if (c->h_k[r] > 2)
            return fail(c, DNAF_E_INPUT, "row %llu has %u alleles: %s counts biallelic rows only", (unsigned long long)r,
                        c->h_k[r], test);
    return DNAF_OK;
}

// One count kernel over rows [row_begin,row_end) (checked by the caller): `tiles` CTAs a row, `words` uint32 counters a
// row in c->d_counts (zeroed by every pass), `row_bytes` of device output a row (the pass-size bound).
// launch(r0, r1) queues the pass's kernels and returns how many; fetch(r0, r1) queues the pass's copies to the host
// (nothing for device-only calls).  stats: rows, calls, kernel_launches, ms_sample (the pass kernels), ms_total.
template <class Launch, class Fetch>
int count_passes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint32_t tiles, uint32_t words, uint64_t row_bytes,
                 dnaf_stats* st, Launch launch, Fetch fetch) {
    CU(c, cudaSetDevice(c->dev));
    dnaf_stats local;
    memset(&local, 0, sizeof local);
    const uint64_t per_pass = std::max<uint64_t>(1, std::min<uint64_t>(c->chunk_bytes / row_bytes, 0x7FFFFFFFull / tiles));
    const uint64_t rows = row_end - row_begin;
    if (rows) CU(c, c->d_counts.reserve(std::min(rows, per_pass) * 4u * words));
    bool timed[3] = {false, false, false};
    // the kernel time of the pass three back (its events are reused by this pass)
    auto retire = [&](int k) -> int {
        if (!timed[k]) return DNAF_OK;
        CU(c, cudaEventSynchronize(c->ob[k].ev[1]));
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ob[k].ev[0], c->ob[k].ev[1]);
        local.ms_sample += ms;
        timed[k] = false;
        return DNAF_OK;
    };
    CU(c, cudaEventRecord(c->ev_bed[0], c->stream));
    int npass = 0;
    for (uint64_t r0 = row_begin; r0 < row_end; ++npass) {
        const uint64_t r1 = std::min(row_end, r0 + per_pass);
        const int k = npass % 3;
        int rc = retire(k);
        if (rc) return rc;
        CU(c, cudaMemsetAsync(c->d_counts.p, 0, (r1 - r0) * 4u * words, c->stream));
        CU(c, cudaEventRecord(c->ob[k].ev[0], c->stream));
        local.kernel_launches += launch(r0, r1);
        CU(c, cudaGetLastError());
        CU(c, cudaEventRecord(c->ob[k].ev[1], c->stream));
        timed[k] = true;
        CU(c, fetch(r0, r1));
        local.rows += r1 - r0;
        r0 = r1;
    }
    CU(c, cudaEventRecord(c->ev_bed[1], c->stream));
    for (int k = 0; k < 3; ++k) {
        const int rc = retire(k);
        if (rc) return rc;
    }
    CU(c, cudaEventSynchronize(c->ev_bed[1]));   // the last copy has landed too: it precedes ev_bed[1] on the stream
    cudaEventElapsedTime(&local.ms_total, c->ev_bed[0], c->ev_bed[1]);
    local.calls = local.rows * c->n;
    if (st) *st = local;
    return DNAF_OK;
}

int assoc_passes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* out, dnaf_stats* st) {
    int rc = check_biallelic(c, row_begin, row_end, "the allelic test");
    if (rc) return rc;
    AssocArgs a;
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
    a.tiles = std::max<uint32_t>(1u, (a.groups + kAssocThreads - 1u) / kAssocThreads);
    a.k0 = (uint32_t)seed;
    a.k1 = (uint32_t)(seed >> 32);
    auto launch = [&](uint64_t r0, uint64_t r1) {
        a.row0 = r0;
        a.counts = c->d_counts.as<uint32_t>();
        k_assoc<<<(uint32_t)((r1 - r0) * a.tiles), kAssocThreads, 0, c->stream>>>(a);
        return 1u;
    };
    auto fetch = [&](uint64_t r0, uint64_t r1) {
        return out ? cudaMemcpyAsync(out + 4 * (r0 - row_begin), c->d_counts.p, (r1 - r0) * 16u, cudaMemcpyDeviceToHost,
                                     c->stream)
                   : cudaSuccess;
    };
    return count_passes(c, row_begin, row_end, a.tiles, 4u, 16u, st, launch, fetch);
}

int assoc_impl(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* out, dnaf_stats* st) {
    if (!c) return DNAF_E_ARG;
    const int rc = assoc_passes(c, row_begin, row_end, seed, out, st);
    if (rc) quiesce(c);
    return rc;
}

}  // namespace

// .assoc body lines: pure host code (no context, no GPU).
namespace assocfmt {

// "%.4g" of v, or "NA" when the statistic has a zero denominator (flagged by the caller as NaN)
inline int num(char* p, size_t cap, double v) {
    return std::isnan(v) ? snprintf(p, cap, "NA") : snprintf(p, cap, "%.4g", v);
}

// PLINK's CHR column of label `idx` (8 bytes a label): X, Y and MT are written 23, 24 and 26; `lab` holds the label
inline const char* chr_code(const char* labels, int32_t idx, char lab[8]) {
    memcpy(lab, labels + 8 * (size_t)idx, 8);
    lab[7] = 0;
    return !strcmp(lab, "X") ? "23" : !strcmp(lab, "Y") ? "24" : !strcmp(lab, "MT") ? "26" : lab;
}

// The allelic statistics of a row from a = ALT and ca = observed alleles in cases, c / cu the same in controls; NaN = NA
struct AlleleStats {
    double f_a, f_u, chisq, p, odds;
    AlleleStats(double a, double ca, double c, double cu) {
        const double b = ca - a, d = cu - c;   // REF in cases, REF in controls
        const double nan = std::nan("");
        f_a = ca > 0 ? a / ca : nan;
        f_u = cu > 0 ? c / cu : nan;
        const double den = ca * cu * (a + c) * (b + d);
        chisq = den > 0 ? (a + b + c + d) * (a * d - b * c) * (a * d - b * c) / den : nan;
        p = std::isnan(chisq) ? nan : std::erfc(std::sqrt(chisq / 2.0));
        odds = b * c > 0 ? a * d / (b * c) : nan;
    }
};

inline char* lines_serial(uint64_t r0, uint64_t r1, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                          const int64_t* position, const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, char* o) {
    for (uint64_t r = r0; r < r1; ++r) {
        char lab[8];
        const char* chr = chr_code(labels, chrom_idx[r], lab);
        const AlleleStats s(counts[4 * r], counts[4 * r + 1], counts[4 * r + 2], counts[4 * r + 3]);
        char v[5][32];
        num(v[0], 32, s.f_a);
        num(v[1], 32, s.f_u);
        num(v[2], 32, s.chisq);
        num(v[3], 32, s.p);
        num(v[4], 32, s.odds);
        char snp[32];
        snprintf(snp, sizeof snp, "rs%lld", (long long)ids[r]);
        const char a1 = n_alleles[r] >= 2 ? (char)nts[4 * r + 1] : '0';   // A1 = ALT ('0' when the row has none), as in the .bim
        const char a2 = (char)nts[4 * r];
        o += sprintf(o, "%4s %12s %10lld %4c %8s %8s %4c %12s %12s %12s\n", chr, snp, (long long)position[r], a1, v[0], v[1],
                     a2, v[2], v[3], v[4]);
    }
    return o;
}

// Rows [0,n) in slices of 64 Ki over the host's cores: serial(r0, r1, o) writes the lines of rows [r0,r1) at o (at most
// `line` bytes a row) and returns their end; every slice is written to its own buffer and the slices are joined in order.
template <class Serial>
uint64_t sliced(uint64_t n, uint64_t line, char* out, Serial serial) {
    constexpr uint64_t kSlice = 1ull << 16;
    const uint64_t slices = (n + kSlice - 1) / kSlice;
    if (slices <= 1) return (uint64_t)(serial(0, n, out) - out);
    std::vector<std::vector<char>> buf(slices);
    std::atomic<uint64_t> next{0};
    auto work = [&]() {
        for (uint64_t k; (k = next.fetch_add(1)) < slices;) {
            const uint64_t r0 = k * kSlice, r1 = std::min(n, r0 + kSlice);
            buf[k].resize((r1 - r0) * line);
            char* e = serial(r0, r1, buf[k].data());
            buf[k].resize((size_t)(e - buf[k].data()));
        }
    };
    const unsigned nt = (unsigned)std::min<uint64_t>(slices, std::max(1u, std::min(32u, std::thread::hardware_concurrency())));
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < nt; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    char* o = out;
    for (const auto& b : buf) {
        memcpy(o, b.data(), b.size());
        o += b.size();
    }
    return (uint64_t)(o - out);
}

// about 1.7 us of printf per row
inline uint64_t lines(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const int64_t* position,
                      const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, char* out) {
    return sliced(n, 192, out, [&](uint64_t r0, uint64_t r1, char* o) {
        return lines_serial(r0, r1, chrom_idx, labels, ids, position, nts, n_alleles, counts, o);
    });
}

}  // namespace assocfmt
