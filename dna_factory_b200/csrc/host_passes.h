// The pass pipeline: generic-path launches and generate_passes(), which plans, launches and drains up to three
// passes in flight.  Included by dnaf_api.cu after host_sink.h.
#pragma once

namespace {

// sample (+ overrides) `rows` rows into the plane buffers; row list optional (d_grow), overrides as local pairs
int run_sample(dnaf_ctx* c, uint64_t r0, uint32_t rows, const uint32_t* d_row_idx, uint64_t seed, uint64_t n_over,
               const uint32_t* d_olocal, const uint32_t* d_osamp, dnaf_stats* st) {
    const SampleView sv = sample_view(c);
    const uint64_t words = (uint64_t)rows * sv.groups;
    CU(c, c->d_plane0.reserve(std::max<uint64_t>(words, 1) * 4));
    if (c->any_multi) CU(c, c->d_plane1.reserve(std::max<uint64_t>(words, 1) * 4));
    uint32_t* p1 = c->any_multi ? c->d_plane1.as<uint32_t>() : nullptr;
    if (words) {
        const uint32_t grid = (uint32_t)((words + 255) / 256);
        k_sample<<<grid, 256, 0, c->stream>>>(sv, snp_view(c), r0, d_row_idx, c->row_base, rows, (uint32_t)seed,
                                              (uint32_t)(seed >> 32), c->d_plane0.as<uint32_t>(), p1);
        if (st) st->kernel_launches += 1;
        if (n_over) {
            k_overrides<<<(uint32_t)((n_over + 255) / 256), 256, 0, c->stream>>>(d_olocal, d_osamp, n_over, sv.groups, c->n,
                                                                              c->d_plane0.as<uint32_t>(), p1);
            if (st) st->kernel_launches += 1;
        }
    }
    CU(c, cudaGetLastError());
    return DNAF_OK;
}

// overrides of rows [r0,r1) as (local row, sample) device arrays (all rows, no subset)
int stage_overrides_all(dnaf_ctx* c, uint64_t r0, uint64_t r1, uint64_t* n_over) {
    const size_t o0 = std::lower_bound(c->h_orow.begin(), c->h_orow.end(), r0) - c->h_orow.begin();
    const size_t o1 = std::lower_bound(c->h_orow.begin(), c->h_orow.end(), r1) - c->h_orow.begin();
    c->olocal.clear();
    c->osub.clear();
    for (size_t o = o0; o < o1; ++o) {
        c->olocal.push_back((uint32_t)(c->h_orow[o] - r0));
        c->osub.push_back(c->h_osamp[o]);
    }
    *n_over = o1 - o0;
    return DNAF_OK;
}

// uploads the (local row, sample) override pairs staged in c->olocal / c->osub
int upload_overrides(dnaf_ctx* c) {
    if (c->olocal.empty()) return DNAF_OK;
    int rc = upload_async(c, c->d_olocal, c->olocal);
    if (!rc) rc = upload_async(c, c->d_osub, c->osub);
    return rc;
}

int run_format(dnaf_ctx* c, uint64_t r0, uint32_t rows, const uint32_t* d_row_idx, const uint64_t* d_sub_off,
               uint64_t text_bytes, dnaf_stats* st) {
    CU(c, c->d_text.reserve(text_bytes + 64));
    if (!rows) return DNAF_OK;
    k_format<<<rows, 256, 0, c->stream>>>(sample_view(c), snp_view(c), r0, d_row_idx, d_sub_off,
                                          c->d_row_off.as<uint64_t>(), c->h_row_off[r0], c->d_plane0.as<uint32_t>(),
                                          c->any_multi ? c->d_plane1.as<uint32_t>() : nullptr, c->d_text.as<uint8_t>());
    if (st) st->kernel_launches += 1;
    CU(c, cudaGetLastError());
    return DNAF_OK;
}

uint64_t next_chunk_end(const dnaf_ctx* c, uint64_t r0, uint64_t row_end, uint64_t budget) {
    const uint64_t lim = c->h_row_off[r0] + budget;
    uint64_t r1 = std::upper_bound(c->h_row_off.begin() + r0, c->h_row_off.begin() + row_end + 1, lim) -
                  c->h_row_off.begin() - 1;
    if (r1 <= r0) r1 = r0 + 1;
    return std::min(r1, row_end);
}

int generate_passes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                    Sink& sink, dnaf_stats* st);

// The pass pipeline keeps up to three passes in flight.  When a call fails half way (sink error, caller's buffer
// too small, CUDA error) nothing of it may still be running when the error is returned: a copy could be landing in a
// caller buffer that is about to be freed, and the next call must find an idle pipeline.
void quiesce(dnaf_ctx* c) {
    cudaSetDevice(c->dev);
    cudaStreamSynchronize(c->stream);   // may be the caller's stream (dnaf_set_stream), NULL = the default stream
    for (cudaStream_t s : {c->side, c->side2, c->comp, c->copy})
        if (s) cudaStreamSynchronize(s);
    cudaGetLastError();
    for (auto& b : c->ob) b.copy_mode = 0;
}

int generate_impl(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                  Sink& sink, dnaf_stats* st) {
    const int rc = generate_passes(c, row_begin, row_end, seed, level, sink, st);
    if (rc && c) quiesce(c);
    return rc;
}

int generate_passes(dnaf_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                    Sink& sink, dnaf_stats* st) {
    if (!c) return DNAF_E_ARG;
    if (level < 1 || level > 9) return fail(c, DNAF_E_ARG, "level must be 1..9");
    int rc = ensure_layout(c);
    if (rc) return rc;
    if (row_begin > row_end || row_end > c->S) return fail(c, DNAF_E_ARG, "row range out of bounds");
    CU(c, cudaSetDevice(c->dev));
    // -z 1..2: the byte-4-back parse (k_auto); -z 3: distances 4 and 8, -z 4..9: hash-chain LZ77 tiers of growing search
    // depth (k_lz) on autosome rows
    static const int lz_off = getenv("DNAF_NO_LZ") ? 1 : 0;
    rc = ensure_lz_tables(c, lz_off ? 1 : level);
    if (rc) return rc;
    const bool use_lz = c->lz_ok;
    dnaf_stats local;
    memset(&local, 0, sizeof local);
    sink.log = c->log_blocks && !sink.device_only;
    if (sink.buf) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, sink.buf) == cudaSuccess) sink.pinned = attr.type == cudaMemoryTypeHost;
        else cudaGetLastError();
    }
    uint64_t r0 = row_begin;
    // Three output buffers in rotation.  Pass i is launched as soon as the copy of pass i-3 (same buffer) has landed,
    // i.e. without waiting for anything recent, so the GPU runs ahead; then the copy of pass i-1 is queued behind
    // the copy of pass i-2 that is still in flight, so the copy engine never waits for the host either.
    for (auto& b : c->ob) b.copy_mode = 0;
    int npass = 0;
    if (g_trace) { g_t0 = std::chrono::steady_clock::now(); trace("generate begins", 0); }
    // the side streams of k_fused_text / k_x start after what the main stream holds when the call begins (tables,
    // prefix CRCs, implicit descriptors); within the call they wait only for their pass's slot set
    CU(c, cudaEventRecord(c->ev_fork, c->stream));
    while (r0 < row_end) {
        const int cur = npass % 3;
        rc = finish_copy(c, c->ob[cur], sink);
        if (rc) return rc;
        // the first passes of a call are short (1/4, 1/2 of a chunk; 1/2 when nothing leaves the device): the GPU starts
        // while the host still plans and the first D2H copy starts early.  Measured (bench.py, 32768-row calls): ramp
        // 3 / 2 / 1 / 0 -> 4.90 / 5.00 / 5.09 / 5.09e11 calls/s on the device, end to end unchanged.
        static const int ramp_env = getenv("DNAF_RAMP") ? atoi(getenv("DNAF_RAMP")) : -1;
        const int ramp = ramp_env >= 0 ? ramp_env : (sink.device_only ? 1 : 2);
        const uint64_t r1 = next_chunk_end(c, r0, row_end, std::max<uint64_t>(c->chunk_bytes >> std::max(0, ramp - npass), 4096));
        dnaf_ctx::OutBuf& B = c->ob[cur];
        const auto t_plan0 = std::chrono::steady_clock::now();
        plan_pass(c, r0, r1, implicit_end(c, r0, r1), c->h_k.data());
        const auto t_plan1 = std::chrono::steady_clock::now();
        c->cur_ob = cur;
        rc = reserve_outputs(c, B, c->pass_blocks, c->pass_text);
        if (!rc) rc = reserve_stage(c, B);
        if (rc) return rc;
        CU(c, cudaStreamWaitEvent(c->stream, c->sbuf[c->sb].ev_free, 0));   // compaction two passes ago read this slot set
        CU(c, cudaEventRecord(B.ev[0], c->stream));
        const uint32_t grows = (uint32_t)c->grow.size();
        if (grows) {
            rc = upload_async(c, c->d_grow, c->grow);
            if (!rc) rc = upload_async(c, c->d_goff, c->goff);
            if (!rc) rc = upload_overrides(c);
            if (!rc) rc = run_sample(c, r0, grows, c->d_grow.as<uint32_t>(), seed, c->olocal.size(),
                                     c->d_olocal.as<uint32_t>(), c->d_osub.as<uint32_t>(), &local);
            if (rc) return rc;
        }
        // A timed event between two kernels of the main stream is not free on the GPU: record only the marks whose
        // intervals are read (start_copy), and let k_auto's interval share ev[3] / ev[4] when nothing else is queued
        // between them.  ev[1], ev[2] time the generic path (grows != 0 whenever a pass has generic blocks).
        if (grows) {
            CU(c, cudaEventRecord(B.ev[1], c->stream));
            rc = run_format(c, r0, grows, c->d_grow.as<uint32_t>(), c->d_goff.as<uint64_t>(), c->gen_text_bytes, &local);
            if (rc) return rc;
            CU(c, cudaEventRecord(B.ev[2], c->stream));
        }
        rc = launch_generic(c, &local);
        if (rc) return rc;
        CU(c, cudaEventRecord(B.ev[3], c->stream));
        // k_fused_text and k_x write only their own slots of this pass's slot set and read descriptors that go up on
        // their own high-priority streams, so they do not queue behind the previous pass's k_auto: they start as soon as
        // the slot set is free (the compaction two passes ago is done) and finish under that k_auto, and the upload of
        // their descriptors stays off the main stream.  k_auto's own descriptors (if any) go up on the main stream.
        if (!c->fplan.empty()) rc = upload_async(c, c->d_fdesc, c->fplan);
        if (rc) return rc;
        if (!c->tplan.empty()) {
            CU(c, cudaStreamWaitEvent(c->side, c->ev_fork, 0));
            CU(c, cudaStreamWaitEvent(c->side, c->sbuf[c->sb].ev_free, 0));
            rc = upload_async(c, c->d_tdesc, c->tplan, c->side);
            if (rc) return rc;
        }
        if (!c->xplan.empty()) {
            CU(c, cudaStreamWaitEvent(c->side2, c->ev_fork, 0));
            CU(c, cudaStreamWaitEvent(c->side2, c->sbuf[c->sb].ev_free, 0));
            rc = upload_async(c, c->d_xdesc, c->xplan, c->side2);
            if (rc) return rc;
        }
        if (!c->tplan.empty()) {
            if (!c->text_attr_done) {
                CU(c, cudaFuncSetAttribute(k_fused_text, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TextSmem)));
                c->text_attr_done = true;
            }
            TextArgs ta;
            ta.sv = sample_view(c);
            ta.nv = snp_view(c);
            ta.desc = c->d_tdesc.as<TextDesc>();
            ta.tables = c->d_ftables.as<FusedTable>();
            ta.crc4 = c->d_crc4.as<uint32_t>();
            ta.xpow8 = c->d_xpow8.as<uint32_t>();
            ta.osamp = c->d_osamp.as<uint32_t>();
            ta.xspan = c->d_xspan.as<uint32_t>();
            ta.row_base = c->row_base;
            ta.k0 = (uint32_t)seed;
            ta.k1 = (uint32_t)(seed >> 32);
            ta.slots = c->sbuf[c->sb].slots.as<uint8_t>();
            ta.slot_stride = c->slot_stride;
            ta.sizes = c->sbuf[c->sb].sizes.as<uint32_t>();
            ta.crcs = c->sbuf[c->sb].crcs.as<uint32_t>();
            k_fused_text<<<(uint32_t)c->tplan.size(), c->text_threads, sizeof(TextSmem), c->side>>>(ta);
            local.kernel_launches += 1;
            CU(c, cudaGetLastError());
        }
        if (!c->xplan.empty()) {
            XArgs xa;
            xa.sv = sample_view(c);
            xa.nv = snp_view(c);
            xa.desc = c->d_xdesc.as<FusedDesc>();
            xa.tables = c->d_xtables.as<XTable>();
            xa.xspans = c->d_xspans.as<XSpan>();
            xa.etab = c->d_etab.as<uint32_t>();
            xa.mspan = c->d_mspan.as<uint32_t>();
            xa.mpre = c->d_mpre_x.as<uint32_t>();
            xa.xinit = c->d_xinit.as<uint32_t>();
            xa.pre_crc = c->d_pre_crc.as<uint32_t>();
            xa.orow = c->d_orow.as<uint64_t>();
            xa.osamp = c->d_osamp.as<uint32_t>();
            xa.row_base = c->row_base;
            xa.k0 = (uint32_t)seed;
            xa.k1 = (uint32_t)(seed >> 32);
            xa.slots = c->sbuf[c->sb].slots.as<uint8_t>();
            xa.slot_stride = c->slot_stride;
            xa.sizes = c->sbuf[c->sb].sizes.as<uint32_t>();
            xa.crcs = c->sbuf[c->sb].crcs.as<uint32_t>();
            k_x<<<(uint32_t)c->xplan.size(), c->fused_threads, x_smem_bytes(c->fused_threads), c->side2>>>(xa);
            local.kernel_launches += 1;
            CU(c, cudaGetLastError());
        }
        if (!c->tplan.empty()) CU(c, cudaEventRecord(c->ev_join, c->side));
        if (!c->xplan.empty()) CU(c, cudaEventRecord(c->ev_join2, c->side2));
        // one k_auto launch: the implicit opening run of the pass, or else the planned blocks (implicit_end never leaves
        // k_auto rows to plan after an implicit run)
        if (!c->fplan.empty() || c->implicit_rows) {
            AutoArgs fa;
            fa.sv = sample_view(c);
            fa.nv = snp_view(c);
            fa.desc = c->implicit_rows ? nullptr : c->d_fdesc.as<FusedDesc>();
            fa.row0 = r0;
            fa.nseg = (uint32_t)c->h_seg_crc.size();
            fa.nseg_magic = fa.nseg > 1 ? (uint32_t)(((1ull << 32) + fa.nseg - 1) / fa.nseg) : 0u;
            fa.seginfo = c->d_seginfo.as<uint32_t>();
            fa.bucket = c->d_bucket.as<uint16_t>();
            fa.ovr_first = c->d_ovr_first.as<uint32_t>();
            fa.tables = c->d_atables.as<AutoTable>();
            fa.etab = c->d_etab2.as<uint32_t>();
            fa.mtab = c->d_mtab.as<uint32_t>();
            fa.mtail = c->d_mtail.as<uint32_t>();
            fa.mpre = c->d_mpre.as<uint32_t>();
            fa.crctab = c->d_crctab.as<uint32_t>();
            fa.xinit = c->d_xinit.as<uint32_t>();
            fa.pre_crc = c->d_pre_crc.as<uint32_t>();
            fa.orow = c->d_orow.as<uint64_t>();
            fa.osamp = c->d_osamp.as<uint32_t>();
            fa.row_base = c->row_base;
            fa.k0 = (uint32_t)seed;
            fa.k1 = (uint32_t)(seed >> 32);
            fa.slots = c->sbuf[c->sb].slots.as<uint8_t>();
            fa.slot_stride = c->slot_stride;
            fa.sizes = c->sbuf[c->sb].sizes.as<uint32_t>();
            fa.crcs = c->sbuf[c->sb].crcs.as<uint32_t>();
            B.auto_from = c->fplan.empty() ? B.ev[3] : B.ev_auto[0];   // k_auto's descriptors went up after ev[3]
            if (!c->fplan.empty()) CU(c, cudaEventRecord(B.ev_auto[0], c->stream));
            const uint32_t ablocks = c->implicit_rows ? (uint32_t)c->implicit_rows * fa.nseg : (uint32_t)c->fplan.size();
            if (use_lz) {
                const LzCfg cfg = lz_cfg(level, kLzMaxKey);
                const uint32_t smem = lz_smem_bytes(c->fused_threads, kLzMaxKey + 1u, cfg.chain != 0u);
                if (!c->lz_attr_done) {
                    CU(c, cudaFuncSetAttribute(k_lz, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lz_smem_bytes(256, kLzMaxKey + 1u, true)));
                    c->lz_attr_done = true;
                }
                LzArgs la;
                la.a = fa;
                la.tables = c->d_ltables.as<LzTable>();
                k_lz<<<ablocks, c->fused_threads, smem, c->stream>>>(la);
            } else {
                k_auto<<<ablocks, c->fused_threads, auto_smem_bytes(c->fused_threads), c->stream>>>(fa);
            }
            const bool joins = !c->tplan.empty() || !c->xplan.empty();
            B.auto_to = joins ? B.ev_auto[1] : B.ev[4];
            if (joins) CU(c, cudaEventRecord(B.ev_auto[1], c->stream));
            if (c->implicit_rows) {
                B.auto_text = c->h_row_off[r0 + c->implicit_rows] - c->h_row_off[r0];
            } else {   // text of the planned k_auto blocks: prefix on a row's first block, cells, '\n' for '\t' at the row's end
                uint64_t t = 0;
                for (const FusedDesc& d : c->fplan) t += 4ull * d.ncells + ((d.flags & 1u) ? c->h_plen[d.row] : 0u);
                B.auto_text = t;
            }
            local.kernel_launches += 1;
            CU(c, cudaGetLastError());
        }
        if (!c->tplan.empty()) CU(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));
        if (!c->xplan.empty()) CU(c, cudaStreamWaitEvent(c->stream, c->ev_join2, 0));
        CU(c, cudaEventRecord(B.ev[4], c->stream));
        if (c->fplan.empty() && !c->implicit_rows) B.auto_text = 0;
        B.rows = r1 - r0;
        B.text = c->h_row_off[r1] - c->h_row_off[r0];
        B.gen = grows != 0;
        B.generic_blocks = !c->plan.empty();
        B.fused = c->implicit_rows || !c->fplan.empty() || !c->tplan.empty() || !c->xplan.empty();
        rc = close_pass(c, B, c->pass_blocks, &local);
        if (rc) return rc;
        if (g_trace) {
            const auto t_l = std::chrono::steady_clock::now();
            fprintf(stderr, "[dnaf] pass rows %llu implicit %llu blocks %u auto %zu x %zu text %zu generic %zu: plan %.0f us, launch %.0f us\n",
                    (unsigned long long)(r1 - r0), (unsigned long long)c->implicit_rows, c->pass_blocks,
                    c->implicit_rows * c->h_seg_crc.size() + c->fplan.size(), c->xplan.size(), c->tplan.size(), c->plan.size(),
                    std::chrono::duration<double, std::micro>(t_plan1 - t_plan0).count(),
                    std::chrono::duration<double, std::micro>(t_l - t_plan1).count());
            trace("launched pass", npass);
        }
        if (npass >= 1) {
            rc = start_copy(c, c->ob[(npass - 1) % 3], sink, &local);
            if (rc) return rc;
        }
        ++npass;
        r0 = r1;
    }
    if (npass >= 1) {
        rc = start_copy(c, c->ob[(npass - 1) % 3], sink, &local);
        if (rc) return rc;
    }
    for (int k = std::max(0, npass - 3); k < npass; ++k) {   // in pass order: staged sinks are delivered here
        rc = finish_copy(c, c->ob[k % 3], sink);
        if (rc) return rc;
    }
    local.calls = local.rows * c->n;
    if (st) *st = local;
    return DNAF_OK;
}

}  // namespace
