// Host side of the PLINK 1 .bed writer (k_bed.cuh): rows [row_begin,row_end) in passes of at most chunk_bytes of .bed
// output, through the same three output buffers, copy stream and sinks as the BGZF passes.  A pass's size is known on
// the host (rows x ceil(N/4)), so there is no totals read-back and no compaction.  Included by dnaf_api.cu after
// host_passes.h.
#pragma once

namespace {

// Per 16-sample group: bit pairs (2i, 2i+1) of the males and of the females (dnaf_set_samples).
std::vector<uint32_t> bed_sex_masks(const uint8_t* sex, uint32_t n) {
    std::vector<uint32_t> m(2 * (size_t)((n + 15u) / 16u), 0u);
    for (uint32_t i = 0; i < n; ++i) m[2 * (i / 16u) + (sex[i] == 1 ? 0 : 1)] |= 3u << (2u * (i % 16u));
    return m;
}

// Waits for the pass that last used B (kernel timing, then its copy) and hands its bytes to the sink.
int bed_retire(dnaf_ctx* c, dnaf_ctx::OutBuf& B, Sink& sink, dnaf_stats* st) {
    if (B.bed_timed) {
        CU(c, cudaEventSynchronize(B.ev[1]));
        float ms = 0;
        cudaEventElapsedTime(&ms, B.ev[0], B.ev[1]);
        st->ms_sample += ms;
        B.bed_timed = false;
    }
    return finish_copy(c, B, sink);
}

int bed_passes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, Sink& sink, dnaf_stats* st) {
    if (!c->have_samples || !c->have_snps) return fail(c, DNAF_E_ARG, "set_samples and set_snps must be called first");
    if (row_begin > row_end || row_end > c->S) return fail(c, DNAF_E_ARG, "row range out of bounds");
    for (uint64_t r = row_begin; r < row_end; ++r)
        if (c->h_k[r] > 2)
            return fail(c, DNAF_E_INPUT, "row %llu has %u alleles: a PLINK 1 .bed holds biallelic rows only",
                        (unsigned long long)r, c->h_k[r]);
    const uint64_t pitch = (c->n + 3u) / 4u;
    if (sink.buf && (row_end - row_begin) * pitch > sink.cap)
        return fail(c, DNAF_E_SPACE, "output buffer too small: need %llu bytes",
                    (unsigned long long)((row_end - row_begin) * pitch));
    CU(c, cudaSetDevice(c->dev));
    dnaf_stats local;
    memset(&local, 0, sizeof local);
    sink.log = false;
    if (sink.buf) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, sink.buf) == cudaSuccess) sink.pinned = attr.type == cudaMemoryTypeHost;
        else cudaGetLastError();
    }
    BedArgs a;
    a.cls = c->d_cls.as<uint8_t>();
    a.k = c->d_k.as<uint8_t>();
    a.thr = c->d_thr.as<uint32_t>();
    a.sexmask = c->d_sexmask.as<uint2>();
    a.orow = c->d_orow.as<uint64_t>();
    a.osamp = c->d_osamp.as<uint32_t>();
    a.n_over = c->P;
    a.row_base = c->row_base;
    a.n = c->n;
    a.groups = (c->n + 15u) / 16u;
    a.tiles = std::max<uint32_t>(1u, (a.groups + kBedThreads - 1u) / kBedThreads);
    a.pitch = (uint32_t)pitch;
    a.k0 = (uint32_t)seed;
    a.k1 = (uint32_t)(seed >> 32);
    // rows per pass: chunk_bytes of output, and a grid that stays below 2^31 CTAs
    const uint64_t per_pass = std::max<uint64_t>(1, std::min<uint64_t>(pitch ? c->chunk_bytes / pitch : ~0ull, 0x7FFFFFFFull / a.tiles));
    for (auto& b : c->ob) {
        b.copy_mode = 0;
        b.bed_timed = false;
    }
    CU(c, cudaEventRecord(c->ev_bed[0], c->stream));
    int npass = 0;
    for (uint64_t r0 = row_begin; r0 < row_end; ++npass) {
        const uint64_t r1 = std::min(row_end, r0 + per_pass);
        const uint64_t bytes = (r1 - r0) * pitch;
        dnaf_ctx::OutBuf& B = c->ob[npass % 3];
        int rc = bed_retire(c, B, sink, &local);   // the pass three back: its buffer is free again
        if (rc) return rc;
        if (bytes) {
            CU(c, B.d_out.reserve(bytes));
            a.row0 = r0;
            a.out = B.d_out.as<uint8_t>();
            CU(c, cudaEventRecord(B.ev[0], c->stream));
            k_bed<<<(uint32_t)((r1 - r0) * a.tiles), kBedThreads, 0, c->stream>>>(a);
            CU(c, cudaGetLastError());
            CU(c, cudaEventRecord(B.ev[1], c->stream));
            B.bed_timed = true;
            local.kernel_launches += 1;
            if (!sink.device_only) CU(c, cudaStreamWaitEvent(c->copy, B.ev[1], 0));
            rc = queue_copy(c, B, sink, bytes);
            if (rc) return rc;
        }
        local.rows += r1 - r0;
        r0 = r1;
    }
    CU(c, cudaEventRecord(c->ev_bed[1], c->stream));
    for (int k = std::max(0, npass - 3); k < npass; ++k) {   // in pass order: staged sinks are delivered here
        const int rc = bed_retire(c, c->ob[k % 3], sink, &local);
        if (rc) return rc;
    }
    CU(c, cudaEventSynchronize(c->ev_bed[1]));
    cudaEventElapsedTime(&local.ms_total, c->ev_bed[0], c->ev_bed[1]);
    local.calls = local.rows * c->n;
    if (st) *st = local;
    return DNAF_OK;
}

int bed_impl(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, Sink& sink, dnaf_stats* st) {
    if (!c) return DNAF_E_ARG;
    const int rc = bed_passes(c, row_begin, row_end, seed, sink, st);
    if (rc) {
        quiesce(c);
        for (auto& b : c->ob) b.bed_timed = false;
    }
    return rc;
}

}  // namespace
