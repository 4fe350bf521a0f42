// Host-side state of one GPU context (struct dnaf_ctx), error / trace helpers, uploads and the row layout.
// Part of the single translation unit dnaf_api.cu (included there, in order: host_ctx.h, host_tables.h,
// host_plan.h, host_sink.h, host_passes.h, host_bed.h, host_assoc.h, host_geno.h).
#pragma once

namespace {

thread_local std::string g_create_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        release();
        const size_t want = std::max<size_t>(bytes + bytes / 2, 64 << 10);   // geometric: sizes settle after a few passes
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    ~PinnedBuf() { release(); }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        release();
        const size_t want = std::max<size_t>(bytes + bytes / 2, 64 << 10);
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

uint32_t host_mulmod(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int i = 0; i < 32; ++i) {
        if (a & 0x80000000u) p ^= b;
        a <<= 1;
        b = (b & 1u) ? (b >> 1) ^ kCrcPoly : (b >> 1);
    }
    return p;
}

}  // namespace

// Code tables are pure functions of (MAF bucket, prefix byte model, spans per block, sample set[, level]): one cache per
// PROCESS, so that the contexts of a multi-GPU run (one per rank, pop_factory --gpus N) build every table once
// between them instead of once each (8 ranks x ~10 s of host CPU on a C4-shaped population).  g_tables_mu is held
// by ensure_tables / ensure_lz_tables while they look up, build and insert.
namespace {
std::mutex g_tables_mu;
std::map<std::pair<uint64_t, uint64_t>, FusedTable> g_table_cache;
std::map<std::pair<uint64_t, uint64_t>, XTable> g_xtable_cache;
std::map<std::pair<uint64_t, uint64_t>, AutoTable> g_atable_cache;
std::map<std::pair<std::pair<uint64_t, uint64_t>, int>, LzTable> g_ltable_cache;
}  // namespace

struct dnaf_ctx {
    int dev = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    uint64_t chunk_bytes = 1024ull << 20;
    int fused = 1;
    uint64_t row_base = 0;

    // samples
    bool have_samples = false;
    uint32_t n = 0, males = 0;
    DevBuf d_sex, d_xoff;
    uint32_t body[4] = {1, 1, 1, 1};

    // snps
    bool have_snps = false;
    uint64_t S = 0;
    bool any_multi = false;
    DevBuf d_cls, d_k, d_thr, d_prefix, d_pre_off, d_row_off;
    std::vector<uint8_t> h_cls, h_k;
    std::vector<uint32_t> h_thr0;
    std::vector<uint32_t> h_plen;
    std::vector<uint64_t> h_row_off;  // valid when layout_ok
    bool layout_ok = false;

    // overrides
    uint64_t P = 0;
    DevBuf d_orow, d_osamp;
    std::vector<uint64_t> h_orow;
    std::vector<uint32_t> h_osamp;

    // constant tables
    DevBuf d_crctab, d_xpow8;

    // scratch
    DevBuf d_plane0, d_plane1, d_text, d_blocks, d_geno;
    struct SlotBuf {                       // block slots of a pass; two sets, so that the compaction of pass i (own
        DevBuf slots, sizes, crcs;         // stream) overlaps the kernels of pass i+1
        cudaEvent_t ev_free = nullptr;     // compaction that read this set has finished
    } sbuf[2];
    int sb = 0;
    cudaStream_t comp = nullptr;           // k_size_partials + k_gather run here
    PinnedBuf h_blocks;
    std::vector<BlockDesc> plan;

    cudaStream_t side = nullptr;           // k_fused_text runs here, concurrently with k_auto
    cudaStream_t side2 = nullptr;          // k_x runs here
    cudaEvent_t ev_join2 = nullptr;
    cudaStream_t copy = nullptr;           // D2H of pass i overlaps the kernels of pass i+1
    struct OutBuf {                        // what must outlive a pass while the next one runs
        DevBuf d_out, d_totals;
        PinnedBuf h_totals, h_out, h_stage;  // h_stage: descriptor uploads of the pass (truly asynchronous H2D)
        size_t stage_used = 0;
        cudaEvent_t ev[6] = {};
        cudaEvent_t ev_auto[2] = {};         // around the k_auto launch
        cudaEvent_t auto_from = nullptr, auto_to = nullptr;   // what k_auto's time is read between: ev_auto[0/1], or
                                                              // ev[3] / ev[4] when nothing else is queued in between
        uint64_t auto_text = 0;              // text bytes of the pass's k_auto blocks (0: no k_auto launch)
        cudaEvent_t ev_copied = nullptr;
        uint32_t nb = 0;
        uint64_t rows = 0, text = 0;
        bool gen = false, fused = false, generic_blocks = false;
        int copy_mode = 0;                   // 0 nothing in flight, 1 DMA into the caller's pinned buffer, 2 via h_out
        uint64_t copy_bytes = 0;
        const uint8_t* copy_dst = nullptr;   // mode 1: where in the caller's buffer the pass lands
        bool bed_timed = false;              // a k_bed launch (ev[0] -> ev[1]) whose time is not counted yet
    } ob[3];
    // optional record of every BGZF block handed to a host sink by dnaf_generate* (dnaf_block_log)
    bool log_blocks = false;
    std::vector<uint32_t> log_csize, log_usize;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool attr_done = false;

    // fused path (k_fused.cuh): per-bucket static codes, CRC helper tables, per-segment template CRCs
    bool fused_ok = false;
    DevBuf d_ftables, d_etab, d_fdesc, d_gslot, d_grow, d_goff, d_olocal, d_osub;
    std::vector<uint16_t> h_bucket;        // per row
    std::vector<uint32_t> h_seg_crc;       // L(template body) per autosome segment index
    std::vector<uint32_t> h_seg_cell0;     // first cell of every segment (+ end sentinel)
    std::vector<FusedDesc> fplan;
    std::vector<uint32_t> gslot, grow, olocal, osub;
    std::vector<uint64_t> goff;
    uint64_t gen_text_bytes = 0;
    uint32_t pass_blocks = 0;
    uint32_t slot_stride = kSlot;          // per pass: the longest block's text + room for framing, rounded to 256
    uint64_t pass_text = 0;
    uint32_t fused_threads = 256;
    int cur_ob = 0;
    std::map<std::pair<uint64_t, uint64_t>, FusedTable>& table_cache = g_table_cache;
    bool etab_ok = false;
    std::vector<double> bucket_p;          // minor-allele probability per bucket
    std::unordered_map<uint32_t, int> bucket_of;
    int bucket_shift = 0;
    std::vector<uint64_t> ph;              // prefix byte model
    uint64_t ph_hash = 0;
    uint64_t samples_epoch = 0, seg_epoch = ~0ull;
    uint64_t samples_hash = 0;             // FNV-1a of (n, sex vector): keys the sample-dependent tables in the process-wide caches
    std::vector<uint64_t> tables_sig;      // what d_ftables currently holds
    std::vector<uint8_t> h_sex;
    DevBuf d_crc4, d_xspan, d_tdesc, d_xspans, d_xdesc;
    // k_auto (k_auto.cuh): code tables + byte LUTs per (bucket, starts-row), CRC move tables, per-row prefix CRCs
    DevBuf d_atables, d_etab2, d_mtab, d_mtail, d_mpre, d_xinit, d_pre_crc;
    DevBuf d_xtables, d_mspan, d_mpre_x;   // k_x (k_x.cuh)
    DevBuf d_bucket, d_ovr_first, d_seginfo;   // implicit block descriptors of autosome runs (k_auto.cuh)
    std::vector<uint32_t> h_other;          // [S+1]: rows before r that do NOT take k_auto
    uint64_t implicit_rows = 0;             // leading rows of the pass whose k_auto blocks derive their own descriptors
    std::map<std::pair<uint64_t, uint64_t>, XTable>& xtable_cache = g_xtable_cache;
    std::vector<uint32_t> h_mspan, h_mpre_x;
    std::map<std::pair<uint64_t, uint64_t>, AutoTable>& atable_cache = g_atable_cache;
    // k_lz (k_lz.cuh): code tables per (bucket, starts-row) of the LZ tier in use (-z 4..9)
    DevBuf d_ltables;
    std::map<std::pair<std::pair<uint64_t, uint64_t>, int>, LzTable>& ltable_cache = g_ltable_cache;
    std::vector<uint64_t> ltables_sig;     // what d_ltables currently holds
    bool lz_ok = false;
    bool lz_attr_done = false;
    std::vector<uint32_t> h_mtail, h_mpre;
    DevBuf d_pfx_state;
    PinnedBuf h_present;                   // byte values seen in the row prefixes (written by k_prefix_crc)
    uint32_t present_sticky[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // prefix byte values seen so far (a superset keeps table keys stable)
    std::vector<uint8_t> need_sticky;      // (bucket, variant) tables ever needed: the uploaded set only grows
    std::vector<uint32_t> bk_key; std::vector<int> bk_val;   // direct-mapped cache in front of bucket_of
    bool seg_tabs_dirty = false;
    std::vector<uint8_t> h_pfx_tab;        // per row: prefix ends with '\t' (k_auto's first match may reach into it)
    std::vector<XSpan> h_xspans;
    DevBuf d_sexmask;                      // k_bed: per 16-sample group, bit pairs of the males (x) and females (y)
    DevBuf d_casemask, d_counts;           // k_assoc: per 16-sample group, bit pairs of the cases; a pass's [rows][4] counts
                                           // (k_geno: [rows][10]; dnaf_hwe_exact: the uploaded triples)
    DevBuf d_hwe;                          // k_hwe: a pass's [rows][3] P (dnaf_hwe_exact: [n])
    DevBuf d_fisher;                       // k_fisher: a pass's [rows][4] log10 P (dnaf_fisher_exact: [n])
    uint32_t ncase = 0;                    // samples with is_control == 0
    DevBuf d_pmask;                        // k_perm_masks: case masks [perms][pitch], then (male, female) cases [perms][2]
    DevBuf d_planes;                       // k_mperm_planes: a pass's A and B planes, [rows][pitch] each
    DevBuf d_mrow;                         // k_mperm: a pass's T_obs [rows][2] (double), then exceedances [rows][2]
    DevBuf d_maxt;                         // k_mperm: [perms][2] maxima, zeroed once per call
    cudaEvent_t ev_bed[2] = {};            // k_bed calls: first launch, last kernel end
    std::vector<uint32_t> h_seg_crc_x;     // L(template body) per X segment
    std::vector<uint32_t> h_xoff;
    std::vector<FusedDesc> xplan;
    std::vector<TextDesc> tplan;
    std::vector<uint32_t> seg_byte0[4];    // k_fused_text segments per chromosome class (+ end sentinel)
    uint32_t text_threads = 64;
    bool text_attr_done = false;
};

namespace {

int fail(dnaf_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    else g_create_error = buf;
    return code;
}

#define CU(c, call)                                                                                   \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess)                                                                       \
            return fail((c), e__ == cudaErrorMemoryAllocation ? DNAF_E_NOMEM : DNAF_E_CUDA, "%s: %s", #call, \
                        cudaGetErrorString(e__));                                                     \
    } while (0)

static bool g_trace = getenv("DNAF_TRACE") != nullptr;
static std::chrono::steady_clock::time_point g_t0;
static void trace(const char* what, int pass) {
    if (!g_trace) return;
    fprintf(stderr, "[dnaf] %8.3f ms  %s %d\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - g_t0).count(), what, pass);
}

template <class T>
int upload(dnaf_ctx* c, DevBuf& b, const T* src, size_t count, bool sync = true) {
    CU(c, b.reserve(std::max<size_t>(count, 1) * sizeof(T) + 64));
    if (count) CU(c, cudaMemcpyAsync(b.p, src, count * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    if (sync) CU(c, cudaStreamSynchronize(c->stream));
    return DNAF_OK;
}

SampleView sample_view(const dnaf_ctx* c) {
    SampleView v;
    v.n = c->n;
    v.groups = (2u * c->n + 31u) / 32u;
    v.sex = c->d_sex.as<uint8_t>();
    v.xoff = c->d_xoff.as<uint32_t>();
    for (int i = 0; i < 4; ++i) v.body[i] = c->body[i];
    return v;
}

SnpView snp_view(const dnaf_ctx* c) {
    SnpView v;
    v.cls = c->d_cls.as<uint8_t>();
    v.k = c->d_k.as<uint8_t>();
    v.thr = c->d_thr.as<uint32_t>();
    v.prefix = c->d_prefix.as<uint8_t>();
    v.pre_off = c->d_pre_off.as<uint64_t>();
    return v;
}

void build_segments(dnaf_ctx* c);
int ensure_tables(dnaf_ctx* c);
int ensure_implicit(dnaf_ctx* c);

// Text offset of every row (prefix + class body), host and device copies.
int ensure_layout(dnaf_ctx* c) {
    if (!c->have_samples || !c->have_snps) return fail(c, DNAF_E_ARG, "set_samples and set_snps must be called first");
    if (c->layout_ok) return DNAF_OK;
    if (g_trace) { g_t0 = std::chrono::steady_clock::now(); trace("ensure_layout begins", 0); }
    c->h_row_off.resize(c->S + 1);
    uint64_t acc = 0;
    for (uint64_t r = 0; r < c->S; ++r) {
        c->h_row_off[r] = acc;
        acc += (uint64_t)c->h_plen[r] + c->body[c->h_cls[r]];
    }
    c->h_row_off[c->S] = acc;
    trace("row offsets summed", 0);
    int rc = upload(c, c->d_row_off, c->h_row_off.data(), c->S + 1);
    if (rc) return rc;
    trace("row offsets uploaded", 0);
    build_segments(c);
    if (c->seg_tabs_dirty) {
        rc = upload(c, c->d_mtail, c->h_mtail.data(), c->h_mtail.size());
        if (!rc) rc = upload(c, c->d_mpre, c->h_mpre.data(), c->h_mpre.size());
        if (!rc) rc = upload(c, c->d_mspan, c->h_mspan.data(), c->h_mspan.size());
        if (!rc) rc = upload(c, c->d_mpre_x, c->h_mpre_x.data(), c->h_mpre_x.size());
        if (rc) return rc;
        c->seg_tabs_dirty = false;
    }
    rc = ensure_tables(c);
    if (rc) return rc;
    trace("tables ensured", 0);
    rc = ensure_implicit(c);
    if (rc) return rc;
    trace("implicit descriptors ready", 0);
    c->layout_ok = true;
    return DNAF_OK;
}

}  // namespace
