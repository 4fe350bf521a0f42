// The sink side of a pass: output / staging buffers, compaction launch, D2H copies and delivery to the caller's
// buffer, callback or file descriptor (write / pwrite), the BGZF block log.  Included by dnaf_api.cu after host_plan.h.
#pragma once

namespace {

struct Sink {
    dnaf_sink_fn fn = nullptr;
    void* user = nullptr;
    uint8_t* buf = nullptr;  // host buffer mode
    uint64_t cap = 0, used = 0;
    bool device_only = false;
    bool pinned = false;     // buf is page-locked host memory
    int fd = -1;             // file descriptor mode: write() straight from the page-locked staging buffer
    int64_t fd_off = -1;     // >= 0: pwrite() at this file offset instead (advanced as pieces land)
    bool log = false;        // append the blocks to the context's block log as they reach the host
};

// Walks whole BGZF blocks in [data, data+n): compressed size from BSIZE (the BC subfield), text size from ISIZE.
// Returns the number of bytes covered by well-formed blocks (== n for a clean stream).
template <class F>
uint64_t walk_bgzf(const uint8_t* data, uint64_t n, F&& on_block) {
    uint64_t o = 0;
    while (o + 28 <= n) {
        const uint8_t* h = data + o;
        if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4) || h[12] != 'B' || h[13] != 'C') break;
        const uint32_t csize = (uint32_t)(h[16] | (h[17] << 8)) + 1u;
        if (csize < 26 || o + csize > n) break;
        const uint8_t* t = h + csize - 4;
        const uint32_t usize = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16) | ((uint32_t)t[3] << 24);
        on_block(csize, usize);
        o += csize;
    }
    return o;
}

int append_block_log(dnaf_ctx* c, const uint8_t* data, uint64_t n) {
    const uint64_t covered = walk_bgzf(data, n, [&](uint32_t cs, uint32_t us) {
        c->log_csize.push_back(cs);
        c->log_usize.push_back(us);
    });
    if (covered != n) return fail(c, DNAF_E_CUDA, "block log: pass output is not a whole number of BGZF blocks");
    return DNAF_OK;
}

int deliver(dnaf_ctx* c, Sink& s, const uint8_t* data, uint64_t n) {
    if (s.fd >= 0) {
        uint64_t done = 0;
        while (done < n) {
            const size_t piece = (size_t)std::min<uint64_t>(n - done, 1u << 30);
            const ssize_t w = s.fd_off >= 0 ? ::pwrite(s.fd, data + done, piece, (off_t)(s.fd_off + (int64_t)done)) : ::write(s.fd, data + done, piece);
            if (w < 0) {
                if (errno == EINTR) continue;
                return fail(c, DNAF_E_SINK, "write to file descriptor %d failed: %s", s.fd, strerror(errno));
            }
            done += (uint64_t)w;
        }
        if (s.fd_off >= 0) s.fd_off += (int64_t)n;
    } else if (s.fn) {
        if (s.fn(s.user, data, n) != 0) return fail(c, DNAF_E_SINK, "sink callback failed");
    } else if (s.buf) {
        if (s.used + n > s.cap) return fail(c, DNAF_E_SPACE, "output buffer too small: need more than %llu bytes",
                                            (unsigned long long)s.cap);
        memcpy(s.buf + s.used, data, n);
    }
    s.used += n;
    return DNAF_OK;
}

// Uploads a host vector through the pass's page-locked staging arena, so the copy is asynchronous and the
// host can go on planning while the previous pass still runs.  reserve_stage() sizes the arena up front.
template <class T>
int upload_async(dnaf_ctx* c, DevBuf& b, const std::vector<T>& v, cudaStream_t s = 0) {
    CU(c, b.reserve(std::max<size_t>(v.size(), 1) * sizeof(T)));
    if (v.empty()) return DNAF_OK;
    if (!s) s = c->stream;
    dnaf_ctx::OutBuf& B = c->ob[c->cur_ob];
    const size_t bytes = v.size() * sizeof(T);
    const size_t at = (B.stage_used + 63) & ~size_t(63);
    if (at + bytes > B.h_stage.cap) {  // not planned for: fall back to a pageable (synchronising) copy
        CU(c, cudaMemcpyAsync(b.p, v.data(), bytes, cudaMemcpyHostToDevice, s));
        return DNAF_OK;
    }
    memcpy(B.h_stage.as<uint8_t>() + at, v.data(), bytes);
    B.stage_used = at + bytes;
    CU(c, cudaMemcpyAsync(b.p, B.h_stage.as<uint8_t>() + at, bytes, cudaMemcpyHostToDevice, s));
    return DNAF_OK;
}

int reserve_stage(dnaf_ctx* c, dnaf_ctx::OutBuf& B) {
    const size_t need = (c->fplan.size() + c->xplan.size()) * sizeof(FusedDesc) + c->tplan.size() * sizeof(TextDesc) +
                        c->plan.size() * sizeof(BlockDesc) + (c->gslot.size() + c->grow.size() + c->olocal.size() +
                        c->osub.size()) * 4 + c->goff.size() * 8 + 1024;
    if (need > B.h_stage.cap) {
        CU(c, cudaEventSynchronize(B.ev[5]));  // the arena may still feed the previous use of this buffer
        CU(c, B.h_stage.reserve(need * 2));
    }
    B.stage_used = 0;
    return DNAF_OK;
}

int reserve_outputs(dnaf_ctx* c, dnaf_ctx::OutBuf& B, uint32_t nb_exact, uint64_t text_bytes) {
    // whole multiples of 2048 blocks: passes of a job differ a little in block count, buffers must not be
    // re-allocated (cudaMalloc synchronises the device) every time one is a few blocks larger than the last
    const uint32_t nb = nb_exact > 256u ? (nb_exact + 2047u) / 2048u * 2048u : nb_exact;
    CU(c, c->sbuf[c->sb].slots.reserve((size_t)nb * c->slot_stride + 256));
    CU(c, c->sbuf[c->sb].sizes.reserve(nb * sizeof(uint32_t)));
    CU(c, c->sbuf[c->sb].crcs.reserve(nb * sizeof(uint32_t)));
    CU(c, B.d_totals.reserve((2 + 2 * (size_t)((nb + kGroup - 1u) / kGroup)) * sizeof(uint64_t)));   // state of k_size_partials / k_gather
    CU(c, B.d_out.reserve(text_bytes + (size_t)nb * 64 + 256));   // worst case: every block stored
    CU(c, B.h_totals.reserve(2 * sizeof(uint64_t)));
    if (!c->attr_done) {
        CU(c, cudaFuncSetAttribute(k_bgzf_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DeflateSmem)));
        c->attr_done = true;
    }
    return DNAF_OK;
}

// generic encoder over c->plan (text in d_text), slots from c->gslot (or 0..n-1 when empty)
int launch_generic(dnaf_ctx* c, dnaf_stats* st) {
    const uint32_t nb = (uint32_t)c->plan.size();
    if (!nb) return DNAF_OK;
    int rc = upload_async(c, c->d_blocks, c->plan);
    if (!rc) rc = upload_async(c, c->d_gslot, c->gslot);
    if (rc) return rc;
    k_bgzf_generic<<<nb, 256, sizeof(DeflateSmem), c->stream>>>(
        c->d_text.as<uint8_t>(), c->d_blocks.as<BlockDesc>(), c->gslot.empty() ? nullptr : c->d_gslot.as<uint32_t>(),
        c->d_crctab.as<uint32_t>(), c->d_xpow8.as<uint32_t>(), c->sbuf[c->sb].slots.as<uint8_t>(), c->slot_stride, c->sbuf[c->sb].sizes.as<uint32_t>(),
        c->sbuf[c->sb].crcs.as<uint32_t>());
    if (st) st->kernel_launches += 1;
    CU(c, cudaGetLastError());
    return DNAF_OK;
}

// Compaction of the pass whose kernels were just queued on the main stream (ev[4] marks their end): sizes -> offsets ->
// gather into B.d_out, on the compaction stream, so that it overlaps the next pass's kernels.  ev[5] = pass done.
int close_pass(dnaf_ctx* c, dnaf_ctx::OutBuf& B, uint32_t nb, dnaf_stats* st) {
    B.nb = nb;
    dnaf_ctx::SlotBuf& S = c->sbuf[c->sb];
    CU(c, cudaStreamWaitEvent(c->comp, B.ev[4], 0));
    if (nb) {
        const uint32_t ntiles = (nb + kTile - 1u) / kTile, ngroups = (nb + kGroup - 1u) / kGroup;
        k_size_partials<<<ngroups, kGroup, 0, c->comp>>>(S.sizes.as<uint32_t>(), S.crcs.as<uint32_t>(), nb,
                                                         reinterpret_cast<unsigned long long*>(B.d_totals.p));
        k_gather<<<ntiles, 256, 0, c->comp>>>(S.slots.as<uint8_t>(), c->slot_stride, S.sizes.as<uint32_t>(), nb,
                                              reinterpret_cast<unsigned long long*>(B.d_totals.p),
                                              reinterpret_cast<unsigned long long*>(B.h_totals.p), B.d_out.as<uint8_t>());
        if (st) st->kernel_launches += 2;
    }
    CU(c, cudaEventRecord(B.ev[5], c->comp));
    CU(c, cudaEventRecord(S.ev_free, c->comp));
    CU(c, cudaGetLastError());
    c->sb ^= 1;   // the next pass writes the other slot set
    return DNAF_OK;
}

int queue_copy(dnaf_ctx* c, dnaf_ctx::OutBuf& B, Sink& sink, uint64_t bytes);

// A closed pass: wait for its kernels and totals, account it, and START moving its bytes to the host (straight
// into a page-locked caller buffer when there is one).  finish_copy() completes the move.
int start_copy(dnaf_ctx* c, dnaf_ctx::OutBuf& B, Sink& sink, dnaf_stats* st) {
    trace("start_copy: wait kernels", (int)B.nb);
    CU(c, cudaEventSynchronize(B.ev[5]));
    trace("start_copy: kernels done", (int)B.nb);
    const uint64_t bytes = B.nb ? *reinterpret_cast<volatile uint64_t*>(B.h_totals.p) : 0;
    if (st) {
        st->bgzf_bytes += bytes;
        st->bgzf_blocks += B.nb;
        if (B.nb) st->crc_xor ^= (uint32_t)reinterpret_cast<volatile uint64_t*>(B.h_totals.p)[1];
        // only the intervals that count: each query costs a few us of host time, and after a call's last pass they
        // sit between the GPU going idle and the caller's next call
        float t01 = 0, t12 = 0, t23 = 0, t34 = 0, t45 = 0, t05 = 0;
        if (B.gen) {
            cudaEventElapsedTime(&t01, B.ev[0], B.ev[1]);
            cudaEventElapsedTime(&t12, B.ev[1], B.ev[2]);
            st->ms_sample += t01;
            st->ms_format += t12;
        }
        if (B.generic_blocks) cudaEventElapsedTime(&t23, B.ev[2], B.ev[3]);
        cudaEventElapsedTime(&t45, B.ev[4], B.ev[5]);
        cudaEventElapsedTime(&t05, B.ev[0], B.ev[5]);
        st->ms_deflate += t23 + t45;
        if (B.fused) {
            cudaEventElapsedTime(&t34, B.ev[3], B.ev[4]);
            st->ms_fused += t34;
        }
        st->ms_total += t05;
        if (B.auto_text) {
            float ta = 0;
            cudaEventElapsedTime(&ta, B.auto_from, B.auto_to);
            st->ms_auto += ta;
            st->auto_launches += 1;
            st->auto_text_bytes += B.auto_text;
        }
        st->rows += B.rows;
        st->text_bytes += B.text;
    }
    return queue_copy(c, B, sink, bytes);
}

// Queues the D2H copy of `bytes` bytes of B.d_out on the copy stream: straight into a page-locked caller buffer, else into
// the page-locked staging buffer that finish_copy() delivers from.  Device-only sinks only count the bytes.
int queue_copy(dnaf_ctx* c, dnaf_ctx::OutBuf& B, Sink& sink, uint64_t bytes) {
    B.copy_mode = 0;
    B.copy_bytes = bytes;
    if (sink.device_only || !bytes) {
        sink.used += bytes;
        return DNAF_OK;
    }
    if (sink.buf && sink.pinned) {  // no staging copy: DMA straight into the caller's page-locked buffer
        if (sink.used + bytes > sink.cap)
            return fail(c, DNAF_E_SPACE, "output buffer too small: need more than %llu bytes", (unsigned long long)sink.cap);
        CU(c, cudaMemcpyAsync(sink.buf + sink.used, B.d_out.p, bytes, cudaMemcpyDeviceToHost, c->copy));
        CU(c, cudaEventRecord(B.ev_copied, c->copy));
        B.copy_dst = sink.buf + sink.used;
        sink.used += bytes;
        B.copy_mode = 1;
        return DNAF_OK;
    }
    CU(c, B.h_out.reserve(bytes));
    CU(c, cudaMemcpyAsync(B.h_out.p, B.d_out.p, bytes, cudaMemcpyDeviceToHost, c->copy));
    CU(c, cudaEventRecord(B.ev_copied, c->copy));
    B.copy_mode = 2;
    return DNAF_OK;
}

int finish_copy(dnaf_ctx* c, dnaf_ctx::OutBuf& B, Sink& sink) {
    const int mode = B.copy_mode;
    B.copy_mode = 0;
    if (!mode) return DNAF_OK;
    trace("finish_copy: wait", (int)B.nb);
    CU(c, cudaEventSynchronize(B.ev_copied));
    trace("finish_copy: done", (int)B.nb);
    if (sink.log) {
        const int rc = append_block_log(c, mode == 2 ? B.h_out.as<uint8_t>() : B.copy_dst, B.copy_bytes);
        if (rc) return rc;
    }
    if (mode == 2) return deliver(c, sink, B.h_out.as<uint8_t>(), B.copy_bytes);
    return DNAF_OK;
}

}  // namespace
