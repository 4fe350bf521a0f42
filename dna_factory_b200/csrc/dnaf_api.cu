// C ABI (include/dnaf_b200.h) and host orchestration of the B200 hot path.
//
// Replaces, for the population-generation path of ochrzan/dna-factory:
//   PopulationFactory.write_vcf_snps   pop_factory.py:417-469  (worker pool + ordered writer)
//   PopulationFactory.queue_vcf_snps   pop_factory.py:471-513  (row loop)
//   Bio.bgzf.BgzfWriter.write          call site pop_factory.py:449
// Work is cut into passes of at most `chunk_bytes` of uncompressed text; each pass is
//   sample -> (overrides) -> format -> BGZF encode -> scan -> compact -> D2H -> sink      (generic path)
// or the fused kernel (k_fused.cuh) followed by scan -> compact -> D2H -> sink.  The PLINK 1 .bed writer
// (dnaf_generate_bed*) is one kernel per pass, k_bed -> D2H -> sink (host_bed.h); the case/control allele counts
// (dnaf_allele_counts*) are one kernel per pass too, k_assoc -> D2H (host_assoc.h), and the genotype counts
// (dnaf_genotype_counts*) k_geno -> (k_hwe) -> D2H through the same pass driver (host_geno.h), and the permutation
// tests (dnaf_mperm*) k_geno -> k_mperm_planes -> k_mperm through it too (host_mperm.h).
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/dnaf_b200.h"
#include "dnaf_device.cuh"
#include "fused_host.h"
#include "k_assoc.cuh"
#include "k_bed.cuh"
#include "k_deflate.cuh"
#include "k_fisher.cuh"
#include "k_fused.cuh"
#include "k_fused_text.cuh"
#include "k_geno.cuh"
#include "k_mperm.cuh"
#include "k_sample_format.cuh"
#include "k_select.cuh"
#include "snps_json.h"
#include <map>
#include <mutex>
#include <unordered_map>

using namespace dnaf;

#include "host_ctx.h"
#include "host_tables.h"
#include "host_plan.h"
#include "host_sink.h"
#include "host_passes.h"
#include "host_bed.h"
#include "host_assoc.h"
#include "host_geno.h"
#include "host_mperm.h"


// ================================================================================================ C ABI
extern "C" {

int dnaf_abi_version(void) { return DNAF_ABI_VERSION; }

int dnaf_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return count;
}

const char* dnaf_last_error(const dnaf_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int dnaf_create(int device_ordinal, dnaf_ctx** out) {
    if (!out) return fail(nullptr, DNAF_E_ARG, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, DNAF_E_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    cudaGetErrorString(e));
    if (device_ordinal < 0 || device_ordinal >= count) return fail(nullptr, DNAF_E_ARG, "device ordinal out of range");
    dnaf_ctx* c = new dnaf_ctx();
    c->dev = device_ordinal;
    auto bail = [&](const char* what, cudaError_t err) {
        fail(nullptr, DNAF_E_CUDA, "%s: %s", what, cudaGetErrorString(err));
        delete c;
        return DNAF_E_CUDA;
    };
    if ((e = cudaSetDevice(device_ordinal)) != cudaSuccess) return bail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    c->own_stream = true;
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if ((e = cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, hi)) != cudaSuccess) return bail("cudaStreamCreate", e);
        if ((e = cudaStreamCreateWithPriority(&c->side2, cudaStreamNonBlocking, hi)) != cudaSuccess) return bail("cudaStreamCreate", e);
    }
    if ((e = cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    {   // high priority: the compaction of pass i must not queue behind the blocks of pass i+1's kernels
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if ((e = cudaStreamCreateWithPriority(&c->comp, cudaStreamNonBlocking, hi)) != cudaSuccess) return bail("cudaStreamCreate", e);
    }
    for (auto& sbf : c->sbuf)
        if ((e = cudaEventCreateWithFlags(&sbf.ev_free, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto& b : c->ob) {
        for (auto& ev : b.ev)
            if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail("cudaEventCreate", e);
        for (auto& ev : b.ev_auto)
            if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail("cudaEventCreate", e);
        if ((e = cudaEventCreateWithFlags(&b.ev_copied, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    }
    if ((e = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&c->ev_join2, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (auto& ev : c->ev_bed)
        if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail("cudaEventCreate", e);
    // CRC tables: byte table and x^(8k) mod P for k = 0..kBlk
    std::vector<uint32_t> tab(256), xp(kBlk + 1);
    for (uint32_t i = 0; i < 256; ++i) {
        uint32_t v = i;
        for (int k = 0; k < 8; ++k) v = (v & 1u) ? (v >> 1) ^ kCrcPoly : (v >> 1);
        tab[i] = v;
    }
    xp[0] = 0x80000000u;  // x^0
    for (uint32_t k = 1; k <= kBlk; ++k) xp[k] = host_mulmod(xp[k - 1], 0x00800000u /* x^8 */);
    int rc = upload(c, c->d_crctab, tab.data(), tab.size());
    if (!rc) rc = upload(c, c->d_xpow8, xp.data(), xp.size());
    if (rc) {
        g_create_error = c->err;
        delete c;
        return rc;
    }
    *out = c;
    return DNAF_OK;
}

void dnaf_destroy(dnaf_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->dev);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->side) { cudaStreamSynchronize(c->side); cudaStreamDestroy(c->side); }
    if (c->side2) { cudaStreamSynchronize(c->side2); cudaStreamDestroy(c->side2); }
    if (c->ev_join2) cudaEventDestroy(c->ev_join2);
    if (c->copy) { cudaStreamSynchronize(c->copy); cudaStreamDestroy(c->copy); }
    if (c->comp) { cudaStreamSynchronize(c->comp); cudaStreamDestroy(c->comp); }
    for (auto& sbf : c->sbuf)
        if (sbf.ev_free) cudaEventDestroy(sbf.ev_free);
    for (auto& b : c->ob) {
        for (auto& ev : b.ev)
            if (ev) cudaEventDestroy(ev);
        for (auto& ev : b.ev_auto)
            if (ev) cudaEventDestroy(ev);
        if (b.ev_copied) cudaEventDestroy(b.ev_copied);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    for (auto& ev : c->ev_bed)
        if (ev) cudaEventDestroy(ev);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int dnaf_set_stream(dnaf_ctx* c, void* cuda_stream) {
    if (!c) return DNAF_E_ARG;
    if (c->own_stream && c->stream) {
        cudaStreamSynchronize(c->stream);
        cudaStreamDestroy(c->stream);
    }
    c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    c->own_stream = false;
    return DNAF_OK;
}

int dnaf_set_chunk_bytes(dnaf_ctx* c, uint64_t text_bytes) {
    if (!c) return DNAF_E_ARG;
    if (text_bytes < 4096) return fail(c, DNAF_E_ARG, "chunk must be at least 4096 bytes");
    c->chunk_bytes = std::min<uint64_t>(text_bytes, 8ull << 30);
    return DNAF_OK;
}

int dnaf_set_row_base(dnaf_ctx* c, uint64_t row_base) {
    if (!c) return DNAF_E_ARG;
    c->row_base = row_base;
    return DNAF_OK;
}

int dnaf_set_fused(dnaf_ctx* c, int enable) {
    if (!c) return DNAF_E_ARG;
    c->fused = enable ? 1 : 0;
    c->layout_ok = false;   // which rows take which kernel changes
    return DNAF_OK;
}

int dnaf_set_samples(dnaf_ctx* c, uint32_t n, const uint8_t* sex, const uint8_t* is_control) {
    if (!c) return DNAF_E_ARG;
    if (n && (!sex || !is_control)) return fail(c, DNAF_E_ARG, "sex / is_control are NULL");
    if (n > (1u << 30)) return fail(c, DNAF_E_ARG, "too many samples");
    CU(c, cudaSetDevice(c->dev));
    std::vector<uint32_t> xoff(n + 1);
    uint32_t males = 0, acc = 0;
    for (uint32_t i = 0; i < n; ++i) {
        xoff[i] = acc;
        const bool male = sex[i] == 1;
        males += male;
        acc += male ? 2u : 4u;
    }
    xoff[n] = acc;
    c->n = n;
    c->males = males;
    c->ncase = 0;
    for (uint32_t i = 0; i < n; ++i) c->ncase += !is_control[i];
    // body bytes incl. the '\n' that replaces the last '\t' ("\t".join(...) + "\n", pop_factory.py:508)
    c->body[kAuto] = n ? 4u * n : 1u;
    c->body[kX] = n ? acc : 1u;
    c->body[kY] = n ? 2u * n : 1u;
    c->body[kMT] = n ? 2u * n : 1u;
    int rc = upload(c, c->d_sex, sex, n);
    if (!rc) rc = upload(c, c->d_xoff, xoff.data(), xoff.size());
    if (rc) return rc;
    c->h_sex.assign(sex, sex + n);
    c->h_xoff = xoff;
    c->samples_epoch++;
    {
        uint64_t h = 1469598103934665603ull ^ n;
        for (uint32_t i = 0; i < n; ++i) h = (h ^ sex[i]) * 1099511628211ull;
        c->samples_hash = h;
    }
    c->h_xspans = hosttab::build_xspans(sex, n, xoff.data());
    rc = upload(c, c->d_xspans, c->h_xspans.data(), c->h_xspans.size());
    if (rc) return rc;
    {   // k_bed: which cells of a 16-sample group are male / female (haploid on X and Y, missing on Y)
        const std::vector<uint32_t> m = bed_sex_masks(sex, n);
        rc = upload(c, c->d_sexmask, m.data(), m.size());
        if (rc) return rc;
    }
    {   // k_assoc: which cells of a 16-sample group are cases
        const std::vector<uint32_t> m = assoc_case_masks(is_control, n);
        rc = upload(c, c->d_casemask, m.data(), m.size());
        if (rc) return rc;
    }
    {   // X rows: the sample that holds body byte 256*k (for k_fused_text)
        std::vector<uint32_t> xspan((size_t)acc / 256 + 2, 0);
        uint32_t i = 0;
        for (size_t k = 0; k < xspan.size(); ++k) {
            const uint64_t byte = 256ull * k;
            while (i + 1 < n && xoff[i + 1] <= byte) ++i;
            xspan[k] = i;
        }
        rc = upload(c, c->d_xspan, xspan.data(), xspan.size());
        if (rc) return rc;
    }
    c->have_samples = true;
    c->layout_ok = false;
    return DNAF_OK;
}

int dnaf_set_snps(dnaf_ctx* c, uint64_t S, const uint8_t* cls, const uint8_t* k, const uint32_t* thr,
                  const uint8_t* prefix, const uint64_t* pre_off) {
    if (!c) return DNAF_E_ARG;
    if (S && (!cls || !k || !thr || !prefix || !pre_off)) return fail(c, DNAF_E_ARG, "NULL SNP array");
    CU(c, cudaSetDevice(c->dev));
    if (g_trace) { g_t0 = std::chrono::steady_clock::now(); trace("set_snps begins", 0); }
    bool multi = false;
    uint64_t short_rows = 0;
    for (uint64_t r = 0; r < S; ++r) {
        if (cls[r] > kMT) return fail(c, DNAF_E_ARG, "row %llu: bad chromosome class %u", (unsigned long long)r, cls[r]);
        if (k[r] < 1 || k[r] > kKmax)
            return fail(c, DNAF_E_ARG, "row %llu: %u alleles (supported: 1..%d)", (unsigned long long)r, k[r], kKmax);
        // The last allele absorbs whatever the table leaves above its last cumulative probability (the kernels never
        // compare against it).  The reference fails only when a roll actually lands there (pick_allele_index returns
        // None, pop_factory.py:92-95), so tables that merely round short of 1.0 (0.9999999 in an snps.json.gz) are
        // accepted with a note; a last value below 0.999 is a broken table and is refused.
        if (thr[r * 4 + k[r] - 1] != 0xFFFFFFFFu) {
            if (thr[r * 4 + k[r] - 1] < 0xFFBE76C8u)   // floor(0.999 * 2^32)
                return fail(c, DNAF_E_INPUT,
                            "row %llu: cumulative allele probabilities do not reach 1.0 "
                            "(the reference's pick_allele_index would return None)", (unsigned long long)r);
            ++short_rows;
        }
        if (pre_off[r + 1] < pre_off[r] || pre_off[r + 1] - pre_off[r] > (1u << 20))
            return fail(c, DNAF_E_ARG, "row %llu: bad prefix offsets", (unsigned long long)r);
        multi |= k[r] > 2;
    }
    if (short_rows)
        fprintf(stderr, "dnaf_set_snps: %llu row(s) whose cumulative allele probabilities stop within 0.001 of 1.0: "
                        "the last allele takes the remainder\n", (unsigned long long)short_rows);
    c->S = S;
    c->any_multi = multi;
    c->h_cls.assign(cls, cls + S);
    c->h_k.assign(k, k + S);
    c->h_plen.resize(S);
    c->h_pfx_tab.resize(S);
    for (uint64_t r = 0; r < S; ++r) {
        c->h_plen[r] = (uint32_t)(pre_off[r + 1] - pre_off[r]);
        c->h_pfx_tab[r] = c->h_plen[r] && prefix[pre_off[r + 1] - 1] == '\t';
    }
    trace("validated, host copies made", 0);
    // pageable sources: each copy returns once the data is staged, one synchronise covers them all
    int rc = upload(c, c->d_cls, cls, S, false);
    if (!rc) rc = upload(c, c->d_k, k, S, false);
    if (!rc) rc = upload(c, c->d_thr, thr, S * 4, false);
    if (!rc) rc = upload(c, c->d_prefix, prefix, S ? pre_off[S] : 0, false);
    if (!rc && S) rc = upload(c, c->d_pre_off, pre_off, S + 1, false);   // S == 0: pre_off may be NULL, a single 0 goes up below
    if (rc) return rc;
    if (S == 0) {
        const uint64_t zero = 0;
        rc = upload(c, c->d_pre_off, &zero, 1);
        if (rc) return rc;
    } else {   // per-row linear CRC of the prefix (k_auto adds it to its blocks' checksums with four lookups)
        CU(c, c->d_pre_crc.reserve(S * sizeof(uint32_t)));
        CU(c, c->d_pfx_state.reserve(16 * sizeof(uint32_t)));
        CU(c, c->h_present.reserve(8 * sizeof(uint32_t)));
        CU(c, cudaMemsetAsync(c->d_pfx_state.p, 0, 16 * sizeof(uint32_t), c->stream));
        k_prefix_crc<<<(uint32_t)((S + 255) / 256), 256, 0, c->stream>>>(c->d_prefix.as<uint8_t>(), c->d_pre_off.as<uint64_t>(), S,
                                                                       c->d_crctab.as<uint32_t>(), c->d_pre_crc.as<uint32_t>(),
                                                                       c->d_pfx_state.as<uint32_t>(), c->h_present.as<uint32_t>());
        CU(c, cudaGetLastError());
        CU(c, cudaStreamSynchronize(c->stream));   // the uploads above and the kernel
        uint32_t present[8];
        for (int w = 0; w < 8; ++w) present[w] = c->present_sticky[w] |= reinterpret_cast<volatile uint32_t*>(c->h_present.p)[w];
        prefix_model(c, present);
    }
    trace("uploaded", 0);
    c->have_snps = true;
    c->layout_ok = false;
    rc = prepare_buckets(c, k, thr);
    if (rc) return rc;
    trace("buckets prepared", 0);
    return DNAF_OK;
}

int dnaf_set_overrides(dnaf_ctx* c, uint64_t P, const uint64_t* rows, const uint32_t* samples) {
    if (!c) return DNAF_E_ARG;
    if (P && (!rows || !samples)) return fail(c, DNAF_E_ARG, "NULL override array");
    for (uint64_t i = 1; i < P; ++i)
        if (rows[i] < rows[i - 1]) return fail(c, DNAF_E_ARG, "override pairs must be sorted by row");
    CU(c, cudaSetDevice(c->dev));
    c->h_orow.assign(rows, rows + P);
    c->h_osamp.assign(samples, samples + P);
    int rc = upload(c, c->d_orow, rows, P);
    if (!rc) rc = upload(c, c->d_osamp, samples, P);
    if (rc) return rc;
    c->P = P;
    c->layout_ok = false;   // the per-row override index is part of the layout
    return DNAF_OK;
}

int dnaf_select_snps(dnaf_ctx* c, uint64_t n, uint64_t seed, uint32_t n_chrom, const double* chrom_cdf,
                     const double* chrom_max_pos, const uint8_t* chrom_rank, uint32_t n_maf, const double* maf_cdf,
                     int sorted, uint32_t* order, uint8_t* chrom_idx, uint8_t* maf_bin, uint32_t* position, uint8_t* ref,
                     uint8_t* alt) {
    if (!c) return DNAF_E_ARG;
    if (n == 0) return DNAF_OK;
    if (n > 0x7FFFFFFFull) return fail(c, DNAF_E_ARG, "at most 2^31-1 SNPs per call (the device sort counts its items in an int)");
    if (!chrom_cdf || !chrom_max_pos || !chrom_rank || !maf_cdf || !order || !chrom_idx || !maf_bin || !position || !ref || !alt)
        return fail(c, DNAF_E_ARG, "NULL array");
    if (n_chrom < 1 || n_chrom > (uint32_t)kSelMaxChrom || n_maf < 1 || n_maf > (uint32_t)kSelMaxMaf)
        return fail(c, DNAF_E_ARG, "1..%d chromosomes and 1..%d MAF bins", kSelMaxChrom, kSelMaxMaf);
    for (uint32_t i = 0; i < n_chrom; ++i)
        if (!(chrom_max_pos[i] >= 0.0) || chrom_max_pos[i] >= 4294967296.0) return fail(c, DNAF_E_ARG, "chromosome length out of range");
    CU(c, cudaSetDevice(c->dev));
    DevBuf d_par, d_key, d_key2, d_idx, d_idx2, d_col, d_col2, d_tmp;
    const size_t par_bytes = (2 * (size_t)n_chrom + n_maf) * sizeof(double) + n_chrom;
    std::vector<uint8_t> par(par_bytes);
    memcpy(par.data(), chrom_cdf, n_chrom * sizeof(double));
    memcpy(par.data() + n_chrom * sizeof(double), chrom_max_pos, n_chrom * sizeof(double));
    memcpy(par.data() + 2 * n_chrom * sizeof(double), maf_cdf, n_maf * sizeof(double));
    memcpy(par.data() + (2 * (size_t)n_chrom + n_maf) * sizeof(double), chrom_rank, n_chrom);
    int rc = upload(c, d_par, par.data(), par.size(), false);
    if (rc) return rc;
    const size_t col_bytes = n * 8 + 64;   // chrom, maf, ref, alt (1 byte each) + pos (4 bytes), 16-byte aligned pieces
    auto col_at = [&](DevBuf& b, int which) {   // 0 pos, 1 chrom, 2 maf, 3 ref, 4 alt
        uint8_t* p = b.as<uint8_t>();
        const size_t n4 = (n * 4 + 15) & ~size_t(15), n1 = (n + 15) & ~size_t(15);
        return which == 0 ? p : p + n4 + (size_t)(which - 1) * n1;
    };
    CU(c, d_key.reserve(n * 8));
    CU(c, d_key2.reserve(n * 8));
    CU(c, d_idx.reserve(n * 4));
    CU(c, d_idx2.reserve(n * 4));
    CU(c, d_col.reserve(col_bytes + 64));
    CU(c, d_col2.reserve(col_bytes + 64));
    SelectArgs a;
    a.n = n;
    a.k0 = (uint32_t)seed;
    a.k1 = (uint32_t)(seed >> 32);
    a.n_chrom = n_chrom;
    a.n_maf = n_maf;
    a.chrom_cdf = d_par.as<double>();
    a.chrom_max_pos = d_par.as<double>() + n_chrom;
    a.maf_cdf = d_par.as<double>() + 2 * n_chrom;
    a.chrom_rank = d_par.as<uint8_t>() + (2 * (size_t)n_chrom + n_maf) * sizeof(double);
    a.key = d_key.as<uint64_t>();
    a.idx = d_idx.as<uint32_t>();
    a.pos = reinterpret_cast<uint32_t*>(col_at(d_col, 0));
    a.chrom = col_at(d_col, 1);
    a.maf = col_at(d_col, 2);
    a.ref = col_at(d_col, 3);
    a.alt = col_at(d_col, 4);
    k_select_snps<<<(uint32_t)((n + 255) / 256), 256, 0, c->stream>>>(a);
    CU(c, cudaGetLastError());
    const DevBuf* res = &d_col;
    const uint32_t* d_order = d_idx.as<uint32_t>();
    if (sorted) {
        // stable LSD radix sort on (string rank of the chromosome, position): ties keep draw order, like list.sort
        size_t tmp = 0;
        CU(c, cub::DeviceRadixSort::SortPairs(nullptr, tmp, d_key.as<uint64_t>(), d_key2.as<uint64_t>(), d_idx.as<uint32_t>(),
                                              d_idx2.as<uint32_t>(), (int)n, 0, 40, c->stream));
        CU(c, d_tmp.reserve(tmp + 16));
        CU(c, cub::DeviceRadixSort::SortPairs(d_tmp.p, tmp, d_key.as<uint64_t>(), d_key2.as<uint64_t>(), d_idx.as<uint32_t>(),
                                              d_idx2.as<uint32_t>(), (int)n, 0, 40, c->stream));
        k_select_gather<<<(uint32_t)((n + 255) / 256), 256, 0, c->stream>>>(
            n, d_idx2.as<uint32_t>(), a.chrom, a.maf, a.pos, a.ref, a.alt, col_at(d_col2, 1), col_at(d_col2, 2),
            reinterpret_cast<uint32_t*>(col_at(d_col2, 0)), col_at(d_col2, 3), col_at(d_col2, 4));
        CU(c, cudaGetLastError());
        res = &d_col2;
        d_order = d_idx2.as<uint32_t>();
    }
    DevBuf& R = const_cast<DevBuf&>(*res);
    CU(c, cudaMemcpyAsync(order, d_order, n * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(position, col_at(R, 0), n * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(chrom_idx, col_at(R, 1), n, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(maf_bin, col_at(R, 2), n, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(ref, col_at(R, 3), n, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaMemcpyAsync(alt, col_at(R, 4), n, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
    return DNAF_OK;
}

int64_t dnaf_parse_snps_jsonl(const char* text, uint64_t n_bytes, uint64_t cap, int64_t* ids, int32_t* chrom_idx,
                              int64_t* position, uint8_t* n_alleles, uint8_t* nts, double* cum, char* chrom_labels,
                              uint32_t max_labels, uint32_t* n_labels) {
    if (!text || !ids || !chrom_idx || !position || !n_alleles || !nts || !cum || !chrom_labels || !n_labels) return 0;
    return snpsjson::parse(text, n_bytes, cap, ids, chrom_idx, position, n_alleles, nts, cum, chrom_labels, max_labels, n_labels);
}

uint64_t dnaf_format_prefixes(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* position,
                              const int64_t* ids, const uint8_t* n_alleles, const uint8_t* nts, char* out, uint64_t* off) {
    return snpsfmt::prefixes(n, chrom_idx, labels, position, ids, n_alleles, nts, out, off);
}

uint64_t dnaf_format_snps_jsonl(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* position,
                                const int64_t* ids, const uint8_t* n_alleles, const uint8_t* nts, const uint32_t* repr_idx,
                                const char* reprs, const uint32_t* repr_off, char* out) {
    return snpsfmt::jsonl(n, chrom_idx, labels, position, ids, n_alleles, nts, repr_idx, reprs, repr_off, out);
}

uint64_t dnaf_bgzf_bound(uint64_t text_bytes) {
    // every block carries <= kBlk bytes of text and at most 26 + 5 bytes of framing beyond them;
    // row-aligned cutting can leave blocks partly filled, so count blocks generously
    const uint64_t blocks = text_bytes / (kBlk / 2) + 2;
    return text_bytes + blocks * 64 + 1024;
}

int dnaf_block_log(dnaf_ctx* c, int enable) {
    if (!c) return DNAF_E_ARG;
    c->log_blocks = enable != 0;
    c->log_csize.clear();
    c->log_usize.clear();
    return DNAF_OK;
}

int dnaf_block_log_get(dnaf_ctx* c, const uint32_t** csize, const uint32_t** usize, uint64_t* n_blocks) {
    if (!c) return DNAF_E_ARG;
    if (!csize || !usize || !n_blocks) return fail(c, DNAF_E_ARG, "NULL output pointer");
    *csize = c->log_csize.data();
    *usize = c->log_usize.data();
    *n_blocks = c->log_csize.size();
    return DNAF_OK;
}

int dnaf_bgzf_scan(const uint8_t* data, uint64_t n_bytes, uint32_t* csize, uint32_t* usize, uint64_t cap,
                   uint64_t* n_blocks) {
    if (!n_blocks || (n_bytes && !data)) return DNAF_E_ARG;
    uint64_t k = 0;
    const uint64_t covered = walk_bgzf(data, n_bytes, [&](uint32_t cs, uint32_t us) {
        if (k < cap) {
            if (csize) csize[k] = cs;
            if (usize) usize[k] = us;
        }
        ++k;
    });
    *n_blocks = k;
    if (covered != n_bytes) return DNAF_E_INPUT;
    return k > cap && (csize || usize) ? DNAF_E_SPACE : DNAF_OK;
}

int64_t dnaf_debug_lz_block(double p_minor, int level, const uint32_t* allele_bits, uint32_t n_cells, const uint8_t* prefix,
                            uint32_t prefix_len, int ends_row, uint8_t* out, uint64_t out_cap) {
    if (level < 3 || level > 9 || !allele_bits || !out || n_cells == 0 || n_cells > 254u * 64u || prefix_len > 64 ||
        (prefix_len && !prefix))
        return DNAF_E_ARG;
    uint64_t hist[256] = {0};
    for (uint32_t i = 0; i < prefix_len; ++i) hist[prefix[i]] += 16;
    const int per_block = (int)((n_cells + 63u) / 64u);
    const LzTable t = hosttab::make_lz_table(p_minor, prefix_len ? hist : nullptr, per_block, prefix_len != 0, level);
    if (t.hdr_bits == 0xFFFFFFFFu) return DNAF_E_INPUT;
    const std::vector<uint8_t> enc = hosttab::lz_encode_block_host(t, allele_bits, n_cells, prefix, prefix_len, ends_row != 0, level);
    if (enc.size() > out_cap) return DNAF_E_SPACE;
    memcpy(out, enc.data(), enc.size());
    return (int64_t)enc.size();
}

int dnaf_bgzf_eof(uint8_t* out28) {
    static const uint8_t eof[28] = {0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0x00, 0x42, 0x43,
                                    0x02, 0x00, 0x1b, 0x00, 0x03, 0,    0, 0,    0,    0,    0,    0,    0, 0};
    if (!out28) return DNAF_E_ARG;
    memcpy(out28, eof, 28);
    return DNAF_OK;
}

int dnaf_plan(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t* text_bytes, uint64_t* bgzf_bound) {
    if (!c) return DNAF_E_ARG;
    int rc = ensure_layout(c);
    if (rc) return rc;
    if (row_begin > row_end || row_end > c->S) return fail(c, DNAF_E_ARG, "row range out of bounds");
    const uint64_t t = c->h_row_off[row_end] - c->h_row_off[row_begin];
    if (text_bytes) *text_bytes = t;
    if (bgzf_bound) *bgzf_bound = dnaf_bgzf_bound(t) + (row_end - row_begin) * 64;
    return DNAF_OK;
}

int dnaf_row_offsets(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t* out) {
    if (!c) return DNAF_E_ARG;
    int rc = ensure_layout(c);
    if (rc) return rc;
    if (row_begin > row_end || row_end > c->S) return fail(c, DNAF_E_ARG, "row range out of bounds");
    if (!out) return fail(c, DNAF_E_ARG, "out is NULL");
    const uint64_t base = c->h_row_off[row_begin];
    for (uint64_t r = row_begin; r <= row_end; ++r) out[r - row_begin] = c->h_row_off[r] - base;
    return DNAF_OK;
}

int dnaf_generate(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                  uint8_t* out, uint64_t out_cap, dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (!out && out_cap) return fail(c, DNAF_E_ARG, "out is NULL");
    Sink s;
    s.buf = out;
    s.cap = out_cap;
    return generate_impl(c, row_begin, row_end, seed, level, s, stats);
}

int dnaf_generate_stream(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                         dnaf_sink_fn sink, void* user, dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (!sink) return fail(c, DNAF_E_ARG, "sink is NULL");
    Sink s;
    s.fn = sink;
    s.user = user;
    return generate_impl(c, row_begin, row_end, seed, level, s, stats);
}

int dnaf_generate_fd(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level, int fd,
                     dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (fd < 0) return fail(c, DNAF_E_ARG, "bad file descriptor");
    Sink s;
    s.fd = fd;
    return generate_impl(c, row_begin, row_end, seed, level, s, stats);
}

int dnaf_generate_fd_at(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level, int fd, uint64_t file_offset,
                        dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (fd < 0) return fail(c, DNAF_E_ARG, "bad file descriptor");
    if (file_offset > (uint64_t)INT64_MAX) return fail(c, DNAF_E_ARG, "file offset out of range");
    Sink s;
    s.fd = fd;
    s.fd_off = (int64_t)file_offset;
    return generate_impl(c, row_begin, row_end, seed, level, s, stats);
}

int dnaf_generate_device(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                         dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    Sink s;
    s.device_only = true;
    return generate_impl(c, row_begin, row_end, seed, level, s, stats);
}

int dnaf_generate_bed(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint8_t* out, uint64_t out_cap,
                      dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (!out && out_cap) return fail(c, DNAF_E_ARG, "out is NULL");
    Sink s;
    s.buf = out;
    s.cap = out_cap;
    return bed_impl(c, row_begin, row_end, seed, s, stats);
}

int dnaf_generate_bed_fd_at(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int fd, uint64_t file_offset,
                            dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (fd < 0) return fail(c, DNAF_E_ARG, "bad file descriptor");
    if (file_offset > (uint64_t)INT64_MAX) return fail(c, DNAF_E_ARG, "file offset out of range");
    Sink s;
    s.fd = fd;
    s.fd_off = (int64_t)file_offset;
    return bed_impl(c, row_begin, row_end, seed, s, stats);
}

int dnaf_generate_bed_device(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    Sink s;
    s.device_only = true;
    return bed_impl(c, row_begin, row_end, seed, s, stats);
}

int dnaf_allele_counts(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* counts, dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (!counts && row_end > row_begin) return fail(c, DNAF_E_ARG, "counts is NULL");
    return assoc_impl(c, row_begin, row_end, seed, counts, stats);
}

int dnaf_allele_counts_device(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, dnaf_stats* stats) {
    return assoc_impl(c, row_begin, row_end, seed, nullptr, stats);
}

uint64_t dnaf_format_assoc(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const int64_t* position,
                           const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, char* out) {
    if (!n || !chrom_idx || !labels || !ids || !position || !nts || !n_alleles || !counts || !out) return 0;
    return assocfmt::lines(n, chrom_idx, labels, ids, position, nts, n_alleles, counts, out);
}

int dnaf_genotype_tests(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* counts, double* hwe_p,
                        double* fisher_log10p, dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (!counts && row_end > row_begin) return fail(c, DNAF_E_ARG, "counts is NULL");
    return geno_impl(c, row_begin, row_end, seed, counts, hwe_p, hwe_p != nullptr, fisher_log10p, fisher_log10p != nullptr,
                     stats);
}

int dnaf_genotype_tests_device(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int with_hwe,
                               int with_fisher, dnaf_stats* stats) {
    return geno_impl(c, row_begin, row_end, seed, nullptr, nullptr, with_hwe != 0, nullptr, with_fisher != 0, stats);
}

int dnaf_genotype_counts(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* counts, double* hwe_p,
                         dnaf_stats* stats) {
    return dnaf_genotype_tests(c, row_begin, row_end, seed, counts, hwe_p, nullptr, stats);
}

int dnaf_genotype_counts_device(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int with_hwe,
                                dnaf_stats* stats) {
    return dnaf_genotype_tests_device(c, row_begin, row_end, seed, with_hwe, 0, stats);
}

int dnaf_hwe_exact(dnaf_ctx* c, uint64_t n, const uint32_t* geno, double* p) {
    if (!c) return DNAF_E_ARG;
    if (n && (!geno || !p)) return fail(c, DNAF_E_ARG, "geno / p is NULL");
    const int rc = hwe_exact_impl(c, n, geno, p);
    if (rc) quiesce(c);
    return rc;
}

int dnaf_fisher_exact(dnaf_ctx* c, uint64_t n, const uint32_t* tables, double* log10p) {
    if (!c) return DNAF_E_ARG;
    if (n && (!tables || !log10p)) return fail(c, DNAF_E_ARG, "tables / log10p is NULL");
    const int rc = fisher_exact_impl(c, n, tables, log10p);
    if (rc) quiesce(c);
    return rc;
}

uint64_t dnaf_format_model(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const uint8_t* nts,
                           const uint8_t* n_alleles, const uint32_t* counts, char* out) {
    if (!n || !chrom_idx || !labels || !ids || !nts || !n_alleles || !counts || !out) return 0;
    return assocfmt::sliced(n, modelfmt::kModelLineBytes, out, [&](uint64_t r0, uint64_t r1, char* o) {
        return modelfmt::model_serial(r0, r1, chrom_idx, labels, ids, nts, n_alleles, counts, o);
    });
}

uint64_t dnaf_format_hardy(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const uint8_t* nts,
                           const uint8_t* n_alleles, const uint32_t* counts, const double* hwe_p, char* out) {
    if (!n || !chrom_idx || !labels || !ids || !nts || !n_alleles || !counts || !hwe_p || !out) return 0;
    return assocfmt::sliced(n, modelfmt::kHardyLineBytes, out, [&](uint64_t r0, uint64_t r1, char* o) {
        return modelfmt::hardy_serial(r0, r1, chrom_idx, labels, ids, nts, n_alleles, counts, hwe_p, o);
    });
}

uint64_t dnaf_format_assoc_fisher(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                                  const int64_t* position, const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts,
                                  const double* log10p, char* out) {
    if (!n || !chrom_idx || !labels || !ids || !position || !nts || !n_alleles || !counts || !log10p || !out) return 0;
    return assocfmt::sliced(n, modelfmt::kAssocLineBytes, out, [&](uint64_t r0, uint64_t r1, char* o) {
        return modelfmt::assoc_fisher_serial(r0, r1, chrom_idx, labels, ids, position, nts, n_alleles, counts, log10p, o);
    });
}

uint64_t dnaf_format_model_fisher(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                                  const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, const double* log10p,
                                  char* out) {
    if (!n || !chrom_idx || !labels || !ids || !nts || !n_alleles || !counts || !log10p || !out) return 0;
    return assocfmt::sliced(n, modelfmt::kModelLineBytes, out, [&](uint64_t r0, uint64_t r1, char* o) {
        return modelfmt::model_fisher_serial(r0, r1, chrom_idx, labels, ids, nts, n_alleles, counts, log10p, o);
    });
}

int dnaf_perm_case_masks(dnaf_ctx* c, uint64_t seed, uint64_t first_perm, uint32_t n_perm, uint32_t* masks,
                         uint32_t* sex_counts) {
    if (!c) return DNAF_E_ARG;
    const int rc = perm_masks_impl(c, seed, first_perm, n_perm, masks, sex_counts);
    if (rc) quiesce(c);
    return rc;
}

int dnaf_mperm(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t n_perm, double* t_obs,
               uint32_t* exceed, double* max_t, dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if ((!t_obs || !exceed) && row_end > row_begin) return fail(c, DNAF_E_ARG, "t_obs / exceed is NULL");
    if (!max_t && n_perm) return fail(c, DNAF_E_ARG, "max_t is NULL");
    return mperm_impl(c, row_begin, row_end, seed, n_perm, t_obs, exceed, max_t, stats);
}

int dnaf_mperm_device(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t n_perm, dnaf_stats* stats) {
    return mperm_impl(c, row_begin, row_end, seed, n_perm, nullptr, nullptr, nullptr, stats);
}

uint64_t dnaf_format_mperm(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const double* emp,
                           char* out) {
    if (!n || !chrom_idx || !labels || !ids || !emp || !out) return 0;
    return assocfmt::sliced(n, mpermfmt::kLineBytes, out, [&](uint64_t r0, uint64_t r1, char* o) {
        return mpermfmt::lines_serial(r0, r1, chrom_idx, labels, ids, emp, o);
    });
}

int dnaf_genotypes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint8_t* out, uint64_t cap) {
    if (!c) return DNAF_E_ARG;
    int rc = ensure_layout(c);
    if (rc) return rc;
    if (row_begin > row_end || row_end > c->S) return fail(c, DNAF_E_ARG, "row range out of bounds");
    const uint64_t need = (row_end - row_begin) * c->n * 2ull;
    if (need > cap) return fail(c, DNAF_E_SPACE, "genotype buffer too small: need %llu bytes", (unsigned long long)need);
    if (need == 0) return DNAF_OK;
    if (!out) return fail(c, DNAF_E_ARG, "out is NULL");
    CU(c, cudaSetDevice(c->dev));
    const uint64_t rows_per = std::max<uint64_t>(1, (64ull << 20) / (2ull * c->n));
    for (uint64_t r0 = row_begin; r0 < row_end; r0 += rows_per) {
        const uint64_t r1 = std::min(row_end, r0 + rows_per);
        uint64_t n_over = 0;
        stage_overrides_all(c, r0, r1, &n_over);
        rc = upload_overrides(c);
        if (!rc) rc = run_sample(c, r0, (uint32_t)(r1 - r0), nullptr, seed, n_over, c->d_olocal.as<uint32_t>(),
                                 c->d_osub.as<uint32_t>(), nullptr);
        if (rc) return rc;
        const uint64_t cells = (r1 - r0) * c->n;
        CU(c, c->d_geno.reserve(cells * 2));
        k_export_genotypes<<<(uint32_t)((cells + 255) / 256), 256, 0, c->stream>>>(
            sample_view(c), snp_view(c), r0, (uint32_t)(r1 - r0), c->d_plane0.as<uint32_t>(),
            c->any_multi ? c->d_plane1.as<uint32_t>() : nullptr, c->d_geno.as<uint8_t>());
        CU(c, cudaGetLastError());
        CU(c, cudaMemcpyAsync(out + (r0 - row_begin) * c->n * 2ull, c->d_geno.p, cells * 2, cudaMemcpyDeviceToHost,
                              c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
    }
    return DNAF_OK;
}

int dnaf_text(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint8_t* out, uint64_t cap,
              uint64_t* n_bytes) {
    if (!c) return DNAF_E_ARG;
    int rc = ensure_layout(c);
    if (rc) return rc;
    if (row_begin > row_end || row_end > c->S) return fail(c, DNAF_E_ARG, "row range out of bounds");
    const uint64_t need = c->h_row_off[row_end] - c->h_row_off[row_begin];
    if (n_bytes) *n_bytes = need;
    if (need > cap) return fail(c, DNAF_E_SPACE, "text buffer too small: need %llu bytes", (unsigned long long)need);
    if (need == 0) return DNAF_OK;
    if (!out) return fail(c, DNAF_E_ARG, "out is NULL");
    CU(c, cudaSetDevice(c->dev));
    uint64_t r0 = row_begin, done = 0;
    while (r0 < row_end) {
        const uint64_t r1 = next_chunk_end(c, r0, row_end, c->chunk_bytes);
        const uint64_t bytes = c->h_row_off[r1] - c->h_row_off[r0];
        uint64_t n_over = 0;
        stage_overrides_all(c, r0, r1, &n_over);
        rc = upload_overrides(c);
        if (!rc) rc = run_sample(c, r0, (uint32_t)(r1 - r0), nullptr, seed, n_over, c->d_olocal.as<uint32_t>(),
                                 c->d_osub.as<uint32_t>(), nullptr);
        if (!rc) rc = run_format(c, r0, (uint32_t)(r1 - r0), nullptr, nullptr, bytes, nullptr);
        if (rc) return rc;
        CU(c, cudaMemcpyAsync(out + done, c->d_text.p, bytes, cudaMemcpyDeviceToHost, c->stream));
        CU(c, cudaStreamSynchronize(c->stream));
        done += bytes;
        r0 = r1;
    }
    return DNAF_OK;
}

int dnaf_bgzf_compress(dnaf_ctx* c, const uint8_t* text, uint64_t n, uint8_t* out, uint64_t cap,
                       dnaf_stats* stats) {
    if (!c) return DNAF_E_ARG;
    if (n && !text) return fail(c, DNAF_E_ARG, "text is NULL");
    CU(c, cudaSetDevice(c->dev));
    dnaf_stats local;
    memset(&local, 0, sizeof local);
    Sink s;
    s.buf = out;
    s.cap = cap;
    uint64_t done = 0;
    while (done < n) {
        const uint64_t piece = std::min<uint64_t>(n - done, (c->chunk_bytes / kBlk + 1) * (uint64_t)kBlk);
        CU(c, c->d_text.reserve(piece + 64));
        CU(c, cudaMemcpyAsync(c->d_text.p, text + done, piece, cudaMemcpyHostToDevice, c->stream));
        c->plan.clear();
        c->gslot.clear();
        for (uint64_t o = 0; o < piece; o += kBlk)
            c->plan.push_back({o, (uint32_t)std::min<uint64_t>(kBlk, piece - o), 0});
        dnaf_ctx::OutBuf& B = c->ob[0];
        c->cur_ob = 0;
        c->slot_stride = kSlot;
        int rc = reserve_outputs(c, B, (uint32_t)c->plan.size(), piece);
        if (!rc) rc = reserve_stage(c, B);
        if (rc) return rc;
        CU(c, cudaStreamWaitEvent(c->stream, c->sbuf[c->sb].ev_free, 0));
        for (int e = 0; e < 3; ++e) CU(c, cudaEventRecord(B.ev[e], c->stream));
        B.rows = 0;
        B.text = 0;
        B.gen = false;
        B.fused = false;
        B.generic_blocks = true;
        B.auto_text = 0;
        rc = launch_generic(c, &local);
        if (rc) return rc;
        for (int e = 3; e < 5; ++e) CU(c, cudaEventRecord(B.ev[e], c->stream));   // ev[4]: the compaction stream waits for it
        rc = close_pass(c, B, (uint32_t)c->plan.size(), &local);
        if (!rc) rc = start_copy(c, B, s, &local);
        if (!rc) rc = finish_copy(c, B, s);
        if (rc) return rc;
        local.text_bytes += piece;
        done += piece;
    }
    local.ms_total = local.ms_deflate;
    if (stats) *stats = local;
    return DNAF_OK;
}

}  // extern "C"
