// The planner: which kernel takes which row, the implicit block descriptors of autosome runs and the BGZF block
// plan of one pass.  Included by dnaf_api.cu after host_tables.h.
#pragma once

namespace {

// 0 = generic three-kernel path, 1 = k_auto, 2 = k_fused_text, 3 = k_x
inline int row_kind(const dnaf_ctx* c, uint64_t r, const uint8_t* hk) {
    if (!c->fused || !c->fused_ok || c->h_plen[r] < 1 || c->h_plen[r] > 64 || c->n == 0) return 0;
    if (c->body[c->h_cls[r]] < kFusedMinRowBytes) return 0;
    if (hk[r] <= 2 && c->h_cls[r] == kAuto) return c->h_pfx_tab[r] ? 1 : 2;
    if (hk[r] <= 2 && c->h_cls[r] == kX) return 3;
    return 2;
}
inline bool row_is_fused(const dnaf_ctx* c, uint64_t r, const uint8_t* hk) { return row_kind(c, r, hk) != 0; }

// What k_auto needs to derive its block descriptors itself over a run of autosome rows: which rows those are (host:
// prefix count of the others), the bucket and first override of every row, the segment table.
int ensure_implicit(dnaf_ctx* c) {
    c->h_other.assign(c->S + 1, 0);
    uint32_t others = 0;
    for (uint64_t r = 0; r < c->S; ++r) {
        c->h_other[r] = others;
        others += row_kind(c, r, c->h_k.data()) != 1;
    }
    c->h_other[c->S] = others;
    if (!c->fused_ok || c->S == 0 || others == c->S) return DNAF_OK;
    std::vector<uint32_t> first(c->S + 1);
    size_t o = 0;
    for (uint64_t r = 0; r <= c->S; ++r) {
        while (o < c->h_orow.size() && c->h_orow[o] < r) ++o;
        first[r] = (uint32_t)o;
    }
    std::vector<uint32_t> seg;
    for (size_t sg = 0; sg + 1 < c->h_seg_cell0.size(); ++sg) {
        seg.push_back(c->h_seg_cell0[sg]);
        seg.push_back(c->h_seg_cell0[sg + 1] - c->h_seg_cell0[sg]);
        seg.push_back(c->h_seg_crc[sg]);
    }
    int rc = upload(c, c->d_bucket, c->h_bucket.data(), c->h_bucket.size(), false);
    if (!rc) rc = upload(c, c->d_ovr_first, first.data(), first.size(), false);
    if (!rc) rc = upload(c, c->d_seginfo, seg.data(), seg.size());
    return rc;
}

// End of the run of rows that opens the pass [r0,r1) and whose k_auto blocks derive their descriptors themselves.
// All-autosome passes run implicitly whole.  A pass that opens with autosome rows and holds none after its first
// other row (a sorted step window ends with its MT, X and Y rows) runs that opening run implicitly and plans only the
// rest, so that one k_auto launch covers the pass either way.  Any other pass is planned whole (r0), as is every mixed
// pass when DNAF_FULL_PLAN is set (the reference for tests of the split).
uint64_t implicit_end(const dnaf_ctx* c, uint64_t r0, uint64_t r1) {
    if (!c->fused_ok || c->h_seg_crc.empty()) return r0;
    const uint32_t o0 = c->h_other[r0];
    if (c->h_other[r1] == o0) return r1;
    static const bool full_plan = getenv("DNAF_FULL_PLAN") != nullptr;
    if (full_plan) return r0;
    // the first row that does not take k_auto: h_other first exceeds o0 one row after it
    const uint64_t rx = std::upper_bound(c->h_other.begin() + r0, c->h_other.begin() + r1 + 1, o0) - c->h_other.begin() - 1;
    return c->h_other[r1] - c->h_other[rx] == r1 - rx ? rx : r0;
}

// BGZF block plan of one pass (rows [r0,r1)): fused segments and generic blocks, slots in row order.  The k_auto blocks
// of rows [r0,rx) (implicit_end) take slots 0 .. (rx-r0)*nseg-1 without descriptors; rows [rx,r1) are planned.
void plan_pass(dnaf_ctx* c, uint64_t r0, uint64_t r1, uint64_t rx, const uint8_t* hk) {
    c->implicit_rows = rx - r0;
    c->fplan.clear();
    c->xplan.clear();
    c->tplan.clear();
    c->plan.clear();
    c->gslot.clear();
    c->grow.clear();
    c->goff.clear();
    c->olocal.clear();
    c->osub.clear();
    uint64_t gtext = 0;
    const uint32_t nseg_auto = (uint32_t)c->h_seg_crc.size();
    uint32_t slot = (uint32_t)(rx - r0) * nseg_auto;
    size_t o = std::lower_bound(c->h_orow.begin(), c->h_orow.end(), rx) - c->h_orow.begin();
    uint64_t r = rx;
    while (r < r1) {
        while (o < c->h_orow.size() && c->h_orow[o] < r) ++o;
        const int kind = row_kind(c, r, hk);
        if (kind == 2) {
            size_t oe = o;
            while (oe < c->h_orow.size() && c->h_orow[oe] == r) ++oe;
            const std::vector<uint32_t>& sb = c->seg_byte0[c->h_cls[r]];
            const size_t nseg = sb.size() - 1;
            for (size_t sgi = 0; sgi < nseg; ++sgi) {
                TextDesc d;
                d.row = r;
                d.byte0 = sb[sgi];
                d.nbytes = sb[sgi + 1] - sb[sgi];
                d.slot = slot++;
                d.flags = (sgi == 0 ? 1u : 0u) | (sgi + 1 == nseg ? 2u : 0u);
                d.ovr_first = (uint32_t)o;
                d.ovr_count = (uint32_t)(oe - o);
                d.table = (uint32_t)c->h_bucket[r] * kVariants + 2u + 2u * c->h_cls[r] + (sgi == 0 ? 0u : 1u);
                d.pad = 0;
                c->tplan.push_back(d);
            }
            o = oe;
            ++r;
            continue;
        }
        if (kind == 1 || kind == 3) {
            size_t oe = o;
            while (oe < c->h_orow.size() && c->h_orow[oe] == r) ++oe;
            const size_t nseg = c->h_seg_crc.size();
            for (size_t sgi = 0; sgi < nseg; ++sgi) {
                FusedDesc d;
                d.row = r;
                d.cell0 = c->h_seg_cell0[sgi];
                d.ncells = c->h_seg_cell0[sgi + 1] - d.cell0;
                d.slot = slot++;
                d.flags = (sgi == 0 ? 1u : 0u) | (sgi + 1 == nseg ? 2u : 0u);
                d.ovr_first = (uint32_t)o;
                d.ovr_count = (uint32_t)(oe - o);
                if (kind == 1) {
                    d.table = (uint32_t)c->h_bucket[r] * 2u + (sgi == 0 ? 0u : 1u);
                    d.body_crc = c->h_seg_crc[sgi];
                    c->fplan.push_back(d);
                } else {
                    d.table = (uint32_t)c->h_bucket[r] * 2u + (sgi == 0 ? 0u : 1u);
                    d.body_crc = c->h_seg_crc_x[sgi];
                    c->xplan.push_back(d);
                }
            }
            o = oe;
            ++r;
            continue;
        }
        // a run of consecutive generic rows: text laid out back to back in the generic text buffer
        const uint64_t run_begin = r;
        while (r < r1 && !row_is_fused(c, r, hk)) {
            c->grow.push_back((uint32_t)(r - r0));
            c->goff.push_back(gtext);
            while (o < c->h_orow.size() && c->h_orow[o] == r) {
                c->olocal.push_back((uint32_t)(c->grow.size() - 1));
                c->osub.push_back(c->h_osamp[o]);
                ++o;
            }
            gtext += c->h_row_off[r + 1] - c->h_row_off[r];
            ++r;
        }
        uint64_t q = run_begin;
        size_t gi = c->grow.size() - (size_t)(r - run_begin);
        while (q < r) {
            const uint64_t off = c->goff[gi];
            const uint64_t len = c->h_row_off[q + 1] - c->h_row_off[q];
            const uint32_t plen = c->h_plen[q];
            if (len > kBlk) {
                uint64_t done = 0;
                if (plen + kSpan <= kBlk) {
                    const uint64_t first = plen + (uint64_t)((kBlk - plen) / kSpan) * kSpan;
                    c->plan.push_back({off, (uint32_t)std::min<uint64_t>(first, len), plen});
                    c->gslot.push_back(slot++);
                    done = std::min<uint64_t>(first, len);
                }
                while (done < len) {
                    const uint32_t piece = (uint32_t)std::min<uint64_t>(kBlk, len - done);
                    c->plan.push_back({off + done, piece, 0});
                    c->gslot.push_back(slot++);
                    done += piece;
                }
                ++q;
                ++gi;
            } else {
                uint64_t acc = 0;
                while (q < r && acc + (c->h_row_off[q + 1] - c->h_row_off[q]) <= kBlk) {
                    acc += c->h_row_off[q + 1] - c->h_row_off[q];
                    ++q;
                    ++gi;
                }
                c->plan.push_back({off, (uint32_t)acc, std::min<uint32_t>(plen, (uint32_t)acc)});
                c->gslot.push_back(slot++);
            }
        }
    }
    c->gen_text_bytes = gtext;
    c->pass_blocks = slot;
    // Slot stride of the pass: the longest block's text (a stored block is the worst case: text + 5) plus the slot
    // lead, BGZF framing, the zero-fill / copy overrun of the kernels (< 64 bytes), rounded up to 256.
    uint32_t longest = 0;
    if (rx > r0)
        for (uint32_t sg = 0; sg < nseg_auto; ++sg) longest = std::max(longest, 4u * (c->h_seg_cell0[sg + 1] - c->h_seg_cell0[sg]) + 66u);
    for (const FusedDesc& d : c->fplan) longest = std::max(longest, 4u * d.ncells + 66u);           // prefix <= 64, +1 lead, +1
    for (const FusedDesc& d : c->xplan) longest = std::max(longest, 4u * d.ncells + 66u);
    for (const TextDesc& d : c->tplan) longest = std::max(longest, d.nbytes + 66u);
    for (const BlockDesc& b : c->plan) longest = std::max(longest, b.len);
    c->slot_stride = std::min<uint32_t>(kSlot, (longest + 128u + 255u) & ~255u);
    c->pass_text = c->h_row_off[r1] - c->h_row_off[r0];
}

}  // namespace
