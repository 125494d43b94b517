// api.cu -- context, memory helpers, table life cycle and the pci.ids entry points of the C ABI
// (include/kxpu.h).  The parse / finalize / join kernels live in this translation unit; comm.cu
// (sharded load) drives them through internal.cuh.
#include <algorithm>
#include <cstdlib>
#include <new>
#include <vector>

#include "internal.cuh"
#include "pciids5.cu"
#include "finalize.cuh"
#include "small.cuh"
#include "scan.cuh"

void kx_exchange_destroy(kxpu_ctx *ctx);  // comm.cu

static const char *kx_err_names[] = {
    "ok", "invalid argument", "CUDA error", "no sm_100 GPU available", "output buffer too small",
    "table capacity exceeded", "NCCL / peer exchange unavailable or failed", "input outside the supported domain", "out of memory"};

extern "C" const char *kxpu_strerror(int32_t status) {
    int i = -status;
    if (i < 0 || i > 8) return "unknown status";
    return kx_err_names[i];
}

extern "C" const char *kxpu_last_error(kxpu_ctx *ctx) {
    if (!ctx) return "null ctx";
    static thread_local char copy[sizeof(ctx->err)];
    std::lock_guard<std::mutex> g(ctx->mu);  // ctx->err is written under the same lock
    memcpy(copy, ctx->err, sizeof copy);
    copy[sizeof copy - 1] = 0;
    return copy;
}
extern "C" uint64_t kxpu_launch_count(kxpu_ctx *ctx) { return ctx ? ctx->launches : 0; }

int32_t kx_ctx_create_on(int32_t ordinal, kxpu_ctx **out) {
    if (!out) return KXPU_E_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || ordinal < 0 || ordinal >= count) {
        cudaGetLastError();
        return KXPU_E_NOGPU;  // no CPU fallback: the caller must treat this as fatal
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ordinal) != cudaSuccess) return KXPU_E_NOGPU;
    if (prop.major != 10) return KXPU_E_NOGPU;  // kernels are built for sm_100a only
    kxpu_ctx *c = new (std::nothrow) kxpu_ctx();
    if (!c) return KXPU_E_NOMEM;
    c->device = ordinal;
    c->sm_count = prop.multiProcessorCount;
    if (cudaSetDevice(ordinal) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete c;
        return KXPU_E_CUDA;
    }
    bool ok = true;
    for (int i = 0; i < 2 * KXPU_T_COUNT; i++) ok = ok && cudaEventCreate(&c->ev[i]) == cudaSuccess;
    ok = ok && cudaEventCreate(&c->ev_user[0]) == cudaSuccess && cudaEventCreate(&c->ev_user[1]) == cudaSuccess;
    ok = ok && cudaMallocHost((void **)&c->h_ctl, (KX_C_COUNT + 64) * sizeof(uint32_t)) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();
        kxpu_ctx_destroy(c);
        return KXPU_E_CUDA;
    }
    // keep stream-ordered allocations cached: host-buffer calls allocate/free scratch per call
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, ordinal) == cudaSuccess) {
        uint64_t thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    cudaFuncSetAttribute(kxparse5::parse_kernel_v5, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)(sizeof(kxparse5::WarpSmem5) * kxparse::WARPS));
    const char *fr = getenv("KXPU_RCH");
    c->force_rch = (fr && fr[0] >= '1' && fr[0] <= '8' && !fr[1]) ? fr[0] - '0' : 0;
    c->no_small = getenv("KXPU_NO_SMALL") != nullptr;
    *out = c;
    return KXPU_OK;
}

extern "C" int32_t kxpu_ctx_create(int32_t ordinal, kxpu_ctx **out) { return kx_ctx_create_on(ordinal, out); }

extern "C" int32_t kxpu_ctx_destroy(kxpu_ctx *ctx) {
    if (!ctx) return KXPU_E_INVALID;
    if (ctx->multi) return KXPU_E_INVALID;  // owned by its kxpu_multi group: kxpu_multi_destroy
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    kx_exchange_destroy(ctx);
    for (KxArena &a : ctx->pool) cudaFree(a.p);
    ctx->pool.clear();
    if (ctx->d_stage) cudaFree(ctx->d_stage);
    if (ctx->scan_state) cudaFree(ctx->scan_state);
    for (int i = 0; i < 2 * KXPU_T_COUNT; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->ev_user[0]) cudaEventDestroy(ctx->ev_user[0]);
    if (ctx->ev_user[1]) cudaEventDestroy(ctx->ev_user[1]);
    if (ctx->h_ctl) cudaFreeHost(ctx->h_ctl);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return KXPU_OK;
}

extern "C" int32_t kxpu_set_stage_timing(kxpu_ctx *ctx, int32_t on) {
    if (!ctx) return KXPU_E_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    ctx->stage_timing = on != 0;
    return KXPU_OK;
}

extern "C" int32_t kxpu_last_timings(kxpu_ctx *ctx, float ms_out[KXPU_T_COUNT]) {
    if (!ctx || !ms_out) return KXPU_E_INVALID;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaSetDevice(ctx->device);
    KX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < KXPU_T_COUNT; i++) {
        ms_out[i] = 0.f;
        if (ctx->ev_used[i]) cudaEventElapsedTime(&ms_out[i], ctx->ev[2 * i], ctx->ev[2 * i + 1]);
    }
    return KXPU_OK;
}

// ------------------------------------------------------------------ memory helpers
extern "C" int32_t kxpu_timer_begin(kxpu_ctx *ctx) {
    KX_ENTER(ctx);
    KX_CUDA(ctx, cudaEventRecord(ctx->ev_user[0], ctx->stream));
    return KXPU_OK;
}
extern "C" int32_t kxpu_timer_end(kxpu_ctx *ctx, float *ms_out) {
    KX_ENTER(ctx);
    if (!ms_out) return KXPU_E_INVALID;
    KX_CUDA(ctx, cudaEventRecord(ctx->ev_user[1], ctx->stream));
    KX_CUDA(ctx, cudaEventSynchronize(ctx->ev_user[1]));
    KX_CUDA(ctx, cudaEventElapsedTime(ms_out, ctx->ev_user[0], ctx->ev_user[1]));
    return KXPU_OK;
}

extern "C" int32_t kxpu_dev_alloc(kxpu_ctx *ctx, size_t bytes, void **d_out) {
    KX_ENTER(ctx);
    if (!d_out) return KXPU_E_INVALID;
    KX_CUDA(ctx, cudaMalloc(d_out, bytes ? bytes : 16));
    return KXPU_OK;
}
extern "C" int32_t kxpu_dev_free(kxpu_ctx *ctx, void *d_ptr) {
    KX_ENTER(ctx);
    KX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    KX_CUDA(ctx, cudaFree(d_ptr));
    return KXPU_OK;
}
extern "C" int32_t kxpu_dev_upload(kxpu_ctx *ctx, void *d_dst, const void *h_src, size_t bytes) {
    KX_ENTER(ctx);
    KX_CUDA(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    KX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KXPU_OK;
}
extern "C" int32_t kxpu_dev_download(kxpu_ctx *ctx, void *h_dst, const void *d_src, size_t bytes) {
    KX_ENTER(ctx);
    KX_CUDA(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    KX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KXPU_OK;
}
extern "C" int32_t kxpu_dev_replicate(kxpu_ctx *ctx, void *d_dst, const void *d_src, size_t n, size_t copies) {
    KX_ENTER(ctx);
    // doubling copy: log2(copies) device-to-device memcpys
    if (copies == 0 || n == 0) return KXPU_OK;
    uint8_t *dst = (uint8_t *)d_dst;
    if (dst != d_src) KX_CUDA(ctx, cudaMemcpyAsync(dst, d_src, n, cudaMemcpyDeviceToDevice, ctx->stream));
    size_t have = 1;
    while (have < copies) {
        size_t add = std::min(have, copies - have);
        KX_CUDA(ctx, cudaMemcpyAsync(dst + have * n, dst, add * n, cudaMemcpyDeviceToDevice, ctx->stream));
        have += add;
    }
    KX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KXPU_OK;
}
extern "C" int32_t kxpu_pinned_alloc(kxpu_ctx *ctx, size_t bytes, void **h_out) {
    KX_ENTER(ctx);
    if (!h_out) return KXPU_E_INVALID;
    KX_CUDA(ctx, cudaMallocHost(h_out, bytes ? bytes : 16));
    return KXPU_OK;
}
extern "C" int32_t kxpu_pinned_free(kxpu_ctx *ctx, void *h_ptr) {
    KX_ENTER(ctx);
    KX_CUDA(ctx, cudaFreeHost(h_ptr));
    return KXPU_OK;
}
extern "C" int32_t kxpu_sync(kxpu_ctx *ctx) {
    KX_ENTER(ctx);
    KX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return KXPU_OK;
}

// ------------------------------------------------------------------ look-back state (scan.cuh)
unsigned long long *kx_scan_state(kxpu_ctx *ctx, size_t words) {
    if (words <= ctx->scan_state_words) return ctx->scan_state;
    size_t want = 1u << 14;
    while (want < words) want <<= 1;
    unsigned long long *p = nullptr;
    cudaStreamSynchronize(ctx->stream);  // kernels in flight may still use the old words
    if (cudaMalloc((void **)&p, want * 8) != cudaSuccess || cudaMemset(p, 0, want * 8) != cudaSuccess) {
        cudaGetLastError();
        if (p) cudaFree(p);
        KX_SET_ERR(ctx, "cudaMalloc(%zu) for the look-back state failed", want * 8);
        return nullptr;
    }
    if (ctx->scan_state) cudaFree(ctx->scan_state);
    ctx->scan_state = p;
    ctx->scan_state_words = want;
    return p;
}

uint32_t kx_next_epoch(kxpu_ctx *ctx) {
    if (++ctx->scan_epoch >= (1u << 24)) {  // 24-bit tag wraps: forget every old word
        if (ctx->scan_state) cudaMemsetAsync(ctx->scan_state, 0, ctx->scan_state_words * 8, ctx->stream);
        ctx->scan_epoch = 1;
    }
    return ctx->scan_epoch;
}

// ------------------------------------------------------------------ table life cycle
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bytes of range words the parse needs for num_chunks chunks: range_state + range_carry (u64) and
// lead (u32) per range (a range is >= 1 chunk), the resolve queue (u32) per chunk
static inline size_t range_words_bytes(uint32_t num_chunks) { return ((size_t)num_chunks + 64) * 24; }

struct ArenaLayout {
    size_t o_slots, o_vfirst, o_trunc, ff_bytes, o_counters, o_range, o_row_key, o_row_line, o_row_anchor, o_row_noff, o_row_nlen,
        o_sel, o_blob, total;
};
static ArenaLayout arena_layout(uint32_t cap, uint32_t blob_cap, size_t range_bytes) {
    ArenaLayout L;
    const size_t slots = (size_t)cap + 1;
    size_t off = 0;
    L.o_slots = off;       off = align_up(off + slots * sizeof(KxSlot), 256);
    L.o_vfirst = off;      off = align_up(off + 65536 * 8, 256);
    L.o_trunc = off;       off = align_up(off + 8, 256);
    L.ff_bytes = off;      // everything up to here resets to 0xff bytes
    L.o_counters = off;    off = align_up(off + KX_C_COUNT * 4, 256);
    L.o_range = off;       off = align_up(off + range_bytes, 256);
    L.o_row_key = off;     off = align_up(off + slots * 4, 256);
    L.o_row_line = off;    off = align_up(off + slots * 8, 256);
    L.o_row_anchor = off;  off = align_up(off + slots * 8, 256);
    L.o_row_noff = off;    off = align_up(off + slots * 4, 256);
    L.o_row_nlen = off;    off = align_up(off + slots * 4, 256);
    L.o_sel = off;         off = align_up(off + slots * 4, 256);
    L.o_blob = off;        off = align_up(off + (size_t)blob_cap + 16, 256);
    L.total = off;
    return L;
}

static void arena_reset(kxpu_ctx *ctx, const KxArena &a) {
    const ArenaLayout L = arena_layout(a.cap, a.blob_cap, a.range_bytes);
    const size_t n16 = L.ff_bytes / 16;
    size_t blocks = (n16 + 255) / 256;
    const size_t maxb = (size_t)ctx->sm_count * 8;
    if (blocks > maxb) blocks = maxb;
    kxparse::arena_reset_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>((uint4 *)a.p, n16, (uint32_t *)((uint8_t *)a.p + L.o_counters));
    KX_LAUNCHED(ctx);
}

int32_t kx_table_acquire(kxpu_ctx *ctx, uint32_t cap, uint32_t blob_cap, uint32_t num_chunks, kxpu_table **out) {
    kxpu_table *t = new (std::nothrow) kxpu_table();
    if (!t) return KXPU_E_NOMEM;
    const size_t need_range = range_words_bytes(num_chunks);
    // a parked arena of the same geometry is clean already (reset when it was released)
    bool found = false;
    for (size_t i = 0; i < ctx->pool.size(); i++) {
        const KxArena &a = ctx->pool[i];
        if (a.cap == cap && a.blob_cap == blob_cap && a.range_bytes >= need_range && a.range_bytes <= 4 * need_range + (1u << 20)) {
            t->arena = a;
            ctx->pool.erase(ctx->pool.begin() + (long)i);
            found = true;
            break;
        }
    }
    if (!found) {
        KxArena a;
        a.cap = cap; a.blob_cap = blob_cap; a.range_bytes = need_range;
        a.bytes = arena_layout(cap, blob_cap, need_range).total;
        // cudaMalloc, not the stream-ordered pool: the arena outlives many calls and is reused as is
        cudaError_t e = cudaMalloc(&a.p, a.bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            // parked arenas of other geometries may be what is in the way
            for (KxArena &p : ctx->pool) cudaFree(p.p);
            ctx->pool.clear();
            e = cudaMalloc(&a.p, a.bytes);
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            KX_SET_ERR(ctx, "cudaMalloc(%zu) for a table arena -> %s", a.bytes, cudaGetErrorString(e));
            delete t;
            return e == cudaErrorMemoryAllocation ? KXPU_E_NOMEM : KXPU_E_CUDA;
        }
        arena_reset(ctx, a);
        t->arena = a;
    }
    const ArenaLayout L = arena_layout(cap, blob_cap, t->arena.range_bytes);
    uint8_t *b = (uint8_t *)t->arena.p;
    t->cap = cap;
    uint32_t lg = 0;
    while ((1u << lg) < cap) lg++;
    t->shift = 32 - lg;
    t->dev.slots = (KxSlot *)(b + L.o_slots);
    t->dev.vendor_first = (unsigned long long *)(b + L.o_vfirst);
    t->dev.trunc = (unsigned long long *)(b + L.o_trunc);
    t->dev.counters = (uint32_t *)(b + L.o_counters);
    t->dev.cap = cap;
    t->dev.shift = t->shift;
    t->dev.max_keys = cap / 2;
    t->range_words = (unsigned long long *)(b + L.o_range);
    t->row_key = (uint32_t *)(b + L.o_row_key);
    t->row_line = (unsigned long long *)(b + L.o_row_line);
    t->row_anchor = (unsigned long long *)(b + L.o_row_anchor);
    t->row_name_off = (uint32_t *)(b + L.o_row_noff);
    t->row_name_len = (uint32_t *)(b + L.o_row_nlen);
    t->sel = (uint32_t *)(b + L.o_sel);
    t->blob = b + L.o_blob;
    t->blob_cap = blob_cap;
    t->rows_cap = cap + 1;
    *out = t;
    return KXPU_OK;
}

void kx_table_release(kxpu_ctx *ctx, kxpu_table *t) {
    if (!t) return;
    if (t->arena.p) {
        if (ctx->pool.size() >= 4) {  // the stream may still use the oldest parked arena's successor: order the free behind it
            cudaStreamSynchronize(ctx->stream);
            cudaFree(ctx->pool.front().p);
            ctx->pool.erase(ctx->pool.begin());
        }
        arena_reset(ctx, t->arena);
        ctx->pool.push_back(t->arena);
    }
    delete t;
}

uint32_t kx_initial_blob_cap(kxpu_ctx *ctx, size_t n) {
    const uint32_t by_text = (uint32_t)std::min<size_t>(std::max<size_t>(n, 256), 4u << 20);
    return ctx->blob_hint > by_text ? ctx->blob_hint : by_text;
}

bool kx_grow_cap(uint32_t *cap, bool table_full) {
    if (*cap >= (1u << 28)) return false;
    // x4 when the load limit was crossed (the key count is known to be below cap), x16 when the
    // table ran full (the count is unknown)
    const uint32_t sh = table_full ? 4u : 2u;
    *cap = (*cap >> (28u - sh)) ? (1u << 28) : (*cap << sh);
    return true;
}

void kx_note_table_size(kxpu_ctx *ctx, uint32_t nkeys, uint32_t blob_used, uint32_t blob_cap) {
    uint32_t ideal = 1u << 16;
    while (ideal < (1u << 28) && ideal / 2 < nkeys + nkeys / 8) ideal <<= 1;
    ctx->cap_hint = ideal;
    ctx->blob_hint = blob_cap > (4u << 20) && blob_used > (2u << 20) ? blob_cap : 0u;
}

// ------------------------------------------------------------------ launches
int32_t kx_launch_parse(kxpu_ctx *ctx, kxpu_table *t, const uint8_t *d_text, size_t n, unsigned long long base,
                        unsigned long long carry_in, const KxXaHook *xa) {
    using namespace kxparse;
    const uint32_t num_chunks = (uint32_t)((n + CW - 1) / CW);
    kxparse5::Params5 P;
    memset(&P, 0, sizeof P);
    if (xa) { P.xa_on = 1; P.xa_done = xa->done; P.xa = xa->p; }
    if (num_chunks == 0) {
        if (xa) {  // an empty shard still takes part in the exchange
            P.tab = t->dev;
            P.task_ctas = 0;
            kxparse5::resolve_chunks_kernel<<<kxparse5::XA_CTAS, kxparse5::RES_WARPS * 32, 0, ctx->stream>>>(P);
            KX_LAUNCHED(ctx);
            KX_CUDA(ctx, cudaGetLastError());
        }
        return KXPU_OK;
    }
    P.text = d_text; P.n = n; P.base = base; P.num_chunks = num_chunks;
    P.tma_limit = n >= (size_t)STG_BYTES ? (uint32_t)((n - STG_BYTES) / CW) + 1u : 0u;
    static int per_sm = 0;
    const size_t smem = sizeof(kxparse5::WarpSmem5) * WARPS;
    if (per_sm == 0) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kxparse5::parse_kernel_v5, NT, smem);
        if (per_sm < 1) per_sm = 1;
    }
    // ranges of 8 chunks; shorter ones when the text is too small to give every warp about eight
    // ranges (with two or three 16 KiB ranges per warp the last wave is half empty, and a range of a
    // first-seen vendor block costs its warp ~10 us per chunk)
    const uint32_t wave_warps = (uint32_t)per_sm * ctx->sm_count * WARPS;
    P.rch = std::min<uint32_t>(std::max<uint32_t>(num_chunks / (wave_warps * 8u), 1u), kxparse5::RCH5_MAX);
    if (ctx->force_rch) P.rch = (uint32_t)ctx->force_rch;
    P.num_ranges = (num_chunks + P.rch - 1) / P.rch;
    P.range_state = t->range_words;                            // [num_ranges]
    P.range_carry = t->range_words + P.num_ranges;             // [num_ranges]
    P.lead = (uint32_t *)(t->range_words + 2 * P.num_ranges);  // [num_ranges]
    P.tasks = P.lead + P.num_ranges;                           // [num_chunks]
    P.tab = t->dev; P.carry_in = carry_in;
    // persistent grid, at most one warp per range
    uint32_t grid = (uint32_t)per_sm * ctx->sm_count;
    const uint32_t need = (P.num_ranges + WARPS - 1) / WARPS;
    if (grid > need) grid = need;
    {
        KxTimer tm(ctx, KXPU_T_PARSE);
        kxparse5::parse_kernel_v5<<<grid, NT, smem, ctx->stream>>>(P);
        KX_LAUNCHED(ctx);
    }
    {
        KxTimer tr(ctx, KXPU_T_RESOLVE);
        kxparse5::resolve_ranges_kernel<<<(P.num_ranges + 255u) / 256u, 256, 0, ctx->stream>>>(P);
        KX_LAUNCHED(ctx);
        const uint32_t rgrid = std::min<uint32_t>(4u * ctx->sm_count, (num_chunks + kxparse5::RES_WARPS - 1) / kxparse5::RES_WARPS);
        P.task_ctas = rgrid;
        kxparse5::resolve_chunks_kernel<<<rgrid + (xa ? kxparse5::XA_CTAS : 0u), kxparse5::RES_WARPS * 32, 0, ctx->stream>>>(P);
        KX_LAUNCHED(ctx);
    }
    KX_CUDA(ctx, cudaGetLastError());
    return KXPU_OK;
}

int32_t kx_launch_trunc(kxpu_ctx *ctx, kxpu_table *t, const uint8_t *d_text, size_t n, unsigned long long base) {
    kxparse::trunc_kernel<<<1, 1024, 0, ctx->stream>>>(d_text, n, base, t->dev.trunc, t->dev.counters);
    KX_LAUNCHED(ctx);
    KX_CUDA(ctx, cudaGetLastError());
    return KXPU_OK;
}

// finalize of table t over text[0, n) at global offset base: validity against the table's own first anchors and
// cut-off, rows and names into the table's arrays
static kxparse::FinalizeParams finalize_params(const kxpu_table *t, const uint8_t *text, size_t n, unsigned long long base) {
    kxparse::FinalizeParams F;
    memset(&F, 0, sizeof F);
    F.text = text; F.n = n; F.base = base; F.tab = t->dev;
    F.mv.a = t->dev.vendor_first; F.mv.stride = 0; F.mv.n = 1; F.mv.trunc1 = t->dev.trunc;
    F.row_key = t->row_key; F.row_line = t->row_line; F.row_anchor = t->row_anchor;
    F.row_name_off = t->row_name_off; F.row_name_len = t->row_name_len;
    F.blob = t->blob; F.blob_cap = t->blob_cap;
    return F;
}

int32_t kx_launch_finalize(kxpu_ctx *ctx, kxpu_table *t, const uint8_t *d_text, size_t n, unsigned long long base,
                           const kxx::MinView *mv, const kxx::WaitSpec *wait, const KxSlabOut *slab) {
    kxparse::FinalizeParams F = finalize_params(t, d_text, n, base);
    if (wait) F.wait = *wait;
    if (mv) F.mv = *mv;
    if (slab) {
        F.slab_rows = reinterpret_cast<kxx::SlabRow *>(slab->rows); F.slab_rows_cap = slab->rows_cap;
        F.blob = slab->blob; F.blob_cap = slab->blob_cap;
        F.tail = slab->tail;
    }
    KxTimer tm(ctx, KXPU_T_FINALIZE);
    // validity + names: a warp scans scan_w table slots per step, persistent grid.  Small tables: 8 slots per
    // warp keep every warp of the grid busy with one short chain; big ones scan 32 and work off full batches
    F.scan_w = t->cap >= (1u << 19) ? 32u : 8u;
    const unsigned batches = (t->cap + 1 + F.scan_w - 1) / F.scan_w;
    const unsigned grid = std::min<unsigned>((batches + kxparse::SF_WARPS - 1) / kxparse::SF_WARPS, 8u * ctx->sm_count);
    kxparse::select_finalize_kernel<<<grid, kxparse::SF_WARPS * 32, 0, ctx->stream>>>(F);
    KX_LAUNCHED(ctx);
    KX_CUDA(ctx, cudaGetLastError());
    return KXPU_OK;
}

int32_t kx_launch_lookup(kxpu_ctx *ctx, kxpu_table *t, const uint32_t *d_keys, size_t n, int32_t *d_rows) {
    if (n == 0) return KXPU_OK;
    KxTimer tm(ctx, KXPU_T_LOOKUP);
    size_t blocks = (n + 255) / 256;
    size_t maxb = (size_t)ctx->sm_count * 32;
    if (blocks > maxb) blocks = maxb;
    kxparse::lookup_kernel<<<(unsigned)blocks, 256, 0, ctx->stream>>>(d_keys, n, t->dev.slots, t->cap, t->shift, d_rows);
    KX_LAUNCHED(ctx);
    KX_CUDA(ctx, cudaGetLastError());
    return KXPU_OK;
}

// ------------------------------------------------------------------ single-text load
struct KxJoin {  // optional batched join enqueued behind the finalize, in front of the host round trip
    const uint32_t *d_keys;
    size_t n;
    int32_t *d_rows;
    int32_t *h_rows;  // optional: the row handles also go to this host buffer (inside the one round trip)
    // zero-copy ingest of a small text: the text sits in mapped pinned host memory (device address), d_keys / d_rows
    // are mapped host buffers too; the small-text kernel reads / writes them over PCIe, no copy is enqueued
    const uint8_t *src_text;
};

// device address of `p` if it points into mapped pinned host memory, else nullptr
static void *kx_mapped_host(const void *p) {
    if (!p) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

// chunks the cooperative small-text kernel can take: one per warp of a grid that is resident at once
// (KXPU_NO_SMALL=1, read when the ctx is created, sends small texts through the big-text kernels: tests)
static uint32_t small_text_chunks(kxpu_ctx *ctx) {
    if (ctx->small_chunks < 0) {
        int coop = 0, per_sm = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device);
        cudaFuncSetAttribute(kxsmall::small_load_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kxparse::WARPS * kxparse::STG_BYTES);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kxsmall::small_load_kernel, kxparse::NT, kxparse::WARPS * kxparse::STG_BYTES);
        cudaGetLastError();
        ctx->small_chunks = (coop && !ctx->no_small) ? per_sm * ctx->sm_count * kxparse::WARPS : 0;
    }
    return (uint32_t)ctx->small_chunks;
}

// the whole load (+ join) of a small text as one cooperative launch (small.cuh)
static int32_t launch_small(kxpu_ctx *ctx, kxpu_table *t, const uint8_t *d_text, size_t n, const KxJoin *join) {
    using namespace kxparse;
    kxsmall::SmallParams P;
    memset(&P, 0, sizeof P);
    P.text = d_text; P.n = n;
    P.num_chunks = (uint32_t)((n + CW - 1) / CW);
    P.tma_limit = n >= (size_t)STG_BYTES ? (uint32_t)((n - STG_BYTES) / CW) + 1u : 0u;
    P.state = t->range_words;
    P.F = finalize_params(t, d_text, n, 0);
    FinalizeParams &F = P.F;
    if (join) { P.keys = join->d_keys; P.nq = join->n; P.rows_out = join->d_rows; }
    if (join && join->src_text) { P.text_src = join->src_text; P.h_ctl = ctx->h_ctl; }
    void *args[] = {&P};
    // the whole resident grid: phases 1 / 2 use one warp per chunk, the names and the join every warp
    const unsigned grid = std::max<unsigned>((P.num_chunks + WARPS - 1) / WARPS, (unsigned)(ctx->small_chunks / WARPS));
    // names phase: as few table slots per warp and step as give every warp of the grid at most one step
    F.scan_w = 8u;
    while (F.scan_w < 32u && (size_t)(t->cap + 1 + F.scan_w - 1) / F.scan_w > (size_t)grid * SF_WARPS) F.scan_w *= 2u;
    // KXPU_TRACE_SMALL=1 (debug): SM clocks at the phase boundaries of every CTA, printed per launch
    static const bool trace_on = getenv("KXPU_TRACE_SMALL") != nullptr;
    long long *d_trace = nullptr;
    if (trace_on && cudaMalloc((void **)&d_trace, (size_t)grid * 64) == cudaSuccess) { cudaMemset(d_trace, 0, (size_t)grid * 64); P.trace = d_trace; }
    {
        KxTimer tm(ctx, KXPU_T_PARSE);
        KX_CUDA(ctx, cudaLaunchCooperativeKernel((const void *)kxsmall::small_load_kernel, dim3(grid), dim3(NT), args, (size_t)WARPS * STG_BYTES, ctx->stream));
        KX_LAUNCHED(ctx);
    }
    if (d_trace) {
        std::vector<long long> h((size_t)grid * 8);
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(h.data(), d_trace, h.size() * 8, cudaMemcpyDeviceToHost);
        cudaFree(d_trace);
        static const char *nm[7] = {"phase1", "barrier1", "phase2", "barrier2", "names", "barrier3", "join"};
        fprintf(stderr, "[kxpu small trace] %u CTAs, cycles min/avg/max per CTA:", grid);
        for (int k = 0; k < 7; k++) {
            long long mn = 1ll << 62, mx = 0, sum = 0, cnt = 0;
            for (unsigned b = 0; b < grid; b++) {
                if (!h[b * 8 + k + 1] || !h[b * 8 + k]) continue;
                const long long d = h[b * 8 + k + 1] - h[b * 8 + k];
                mn = std::min(mn, d); mx = std::max(mx, d); sum += d; cnt++;
            }
            if (cnt) fprintf(stderr, " %s %lld/%lld/%lld |", nm[k], mn, sum / cnt, mx);
        }
        fprintf(stderr, "\n");
    }
    return KXPU_OK;
}

// Parse d_text[0..n), finalize, optionally join; ONE host round trip at the end (counters).
static int32_t kx_build_table_join(kxpu_ctx *ctx, const uint8_t *d_text, size_t n, kxpu_table **out, const KxJoin *join) {
    if ((reinterpret_cast<uintptr_t>(d_text) & 15u) != 0) {
        KX_SET_ERR(ctx, "device text pointer must be 16-byte aligned");
        return KXPU_E_INVALID;
    }
    if (n >= (1ull << 44)) return KXPU_E_UNSUPPORTED;
    uint32_t cap = ctx->cap_hint;
    while (cap > (1u << 16) && (size_t)cap / 2 > n / 6 + 1) cap >>= 1;  // a device line is at least 6 bytes
    uint32_t blob_cap = kx_initial_blob_cap(ctx, n);
    const uint32_t num_chunks = (uint32_t)((n + kxparse::CW - 1) / kxparse::CW);
    bool have_trunc = false;
    for (int attempt = 0; attempt < 12; attempt++) {
        kxpu_table *t = nullptr;
        int32_t rc = kx_table_acquire(ctx, cap, blob_cap, num_chunks, &t);
        if (rc != KXPU_OK) return rc;
        const bool small_path = num_chunks > 0 && num_chunks <= small_text_chunks(ctx) && !have_trunc;
        if (small_path) {
            // a small text (the real pci.ids): parse, fold, names and join in ONE cooperative launch
            rc = launch_small(ctx, t, d_text, n, join);
        } else {
            // zero-copy call that cannot take the small-text kernel (any more): the text comes over with a plain copy
            if (join && join->src_text && attempt == 0) cudaMemcpyAsync(const_cast<uint8_t *>(d_text), join->src_text, n, cudaMemcpyDefault, ctx->stream);
            rc = kx_launch_parse(ctx, t, d_text, n, 0, 0, nullptr);
            // a text with a >= 2 KiB stretch without a newline was seen on an earlier attempt: the exact
            // bufio.ErrTooLong cut-off is computed before the finalize
            if (rc == KXPU_OK && have_trunc) rc = kx_launch_trunc(ctx, t, d_text, n, 0);
            if (rc == KXPU_OK) rc = kx_launch_finalize(ctx, t, d_text, n, 0, nullptr, nullptr, nullptr);
            // the join does not need anything from the host: enqueue it before the round trip below
            // (it is simply run again if the table has to be rebuilt)
            if (rc == KXPU_OK && join) rc = kx_launch_lookup(ctx, t, join->d_keys, join->n, join->d_rows);
        }
        if (rc != KXPU_OK) { kx_table_release(ctx, t); return rc; }
        const bool zero_copy = small_path && join && join->src_text;  // the kernel wrote rows and counters to host memory itself
        if (!zero_copy) {
            if (join && join->h_rows && join->n) cudaMemcpyAsync(join->h_rows, join->d_rows, join->n * 4, cudaMemcpyDeviceToHost, ctx->stream);
            cudaMemcpyAsync(ctx->h_ctl, t->dev.counters, KX_C_COUNT * 4, cudaMemcpyDeviceToHost, ctx->stream);
        }
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            KX_SET_ERR(ctx, "parse/finalize failed: %s", cudaGetErrorString(e));
            kx_table_release(ctx, t);
            return KXPU_E_CUDA;
        }
        const uint32_t *h = ctx->h_ctl;
        if (h[KX_C_OVERFLOW] || h[KX_C_NKEYS] > t->dev.max_keys) {
            kx_table_release(ctx, t);
            if (!kx_grow_cap(&cap, h[KX_C_OVERFLOW] != 0)) return KXPU_E_CAPACITY;
            continue;
        }
        if (h[KX_C_NEED_TRUNC] == 2u) {  // finalize stood back: run again with the cut-off (never for real pci.ids)
            kx_table_release(ctx, t);
            have_trunc = true;
            continue;
        }
        if (h[KX_C_BLOB_OVERFLOW]) {
            kx_table_release(ctx, t);
            if ((size_t)blob_cap >= n) return KXPU_E_CAPACITY;
            blob_cap = (uint32_t)std::min<size_t>(std::max<size_t>(n, 256), (size_t)blob_cap * 8);
            continue;
        }
        t->n_rows = h[KX_C_NSEL];  // row handle = index of the slot in the selection
        t->blob_used = h[KX_C_BLOB_CURSOR];
        kx_note_table_size(ctx, h[KX_C_NKEYS], t->blob_used, blob_cap);
        *out = t;
        return KXPU_OK;
    }
    return KXPU_E_CAPACITY;
}

extern "C" int32_t kxpu_pciids_load_device(kxpu_ctx *ctx, const void *d_text, size_t n, kxpu_table **out) {
    KX_ENTER(ctx);
    if (!out || (!d_text && n)) return KXPU_E_INVALID;
    kx_clear_timings(ctx);
    return kx_build_table_join(ctx, (const uint8_t *)d_text, n, out, nullptr);
}

extern "C" int32_t kxpu_pciids_join_device(kxpu_ctx *ctx, const void *d_text, size_t n, const uint32_t *d_keys, size_t nq,
                                           int32_t *d_rows_out, kxpu_table **out) {
    KX_ENTER(ctx);
    if (!out || (!d_text && n) || (nq && (!d_keys || !d_rows_out))) return KXPU_E_INVALID;
    kx_clear_timings(ctx);
    const KxJoin j{d_keys, nq, d_rows_out, nullptr, nullptr};
    return kx_build_table_join(ctx, (const uint8_t *)d_text, n, out, &j);
}

// device staging buffer of the host-buffer entry points: grown on demand, kept by the ctx
static int32_t stage_reserve(kxpu_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->d_stage_bytes) return KXPU_OK;
    if (ctx->d_stage) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(ctx->d_stage);
        ctx->d_stage = nullptr;
        ctx->d_stage_bytes = 0;
    }
    const size_t want = align_up(bytes + bytes / 8 + 4096, 4096);
    cudaError_t e = cudaMalloc(&ctx->d_stage, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        KX_SET_ERR(ctx, "cudaMalloc(%zu) for the host staging buffer -> %s", want, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? KXPU_E_NOMEM : KXPU_E_CUDA;
    }
    ctx->d_stage_bytes = want;
    return KXPU_OK;
}

extern "C" int32_t kxpu_pciids_load(kxpu_ctx *ctx, const uint8_t *text, size_t n, kxpu_table **out) {
    KX_ENTER(ctx);
    if (!out || (!text && n)) return KXPU_E_INVALID;
    kx_clear_timings(ctx);
    int32_t rc = stage_reserve(ctx, n + 16);
    if (rc != KXPU_OK) return rc;
    cudaError_t e = cudaMemcpyAsync(ctx->d_stage, text, n, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) {
        KX_SET_ERR(ctx, "H2D copy of the text failed: %s", cudaGetErrorString(e));
        return KXPU_E_CUDA;
    }
    return kx_build_table_join(ctx, (const uint8_t *)ctx->d_stage, n, out, nullptr);
}

extern "C" int32_t kxpu_pciids_join(kxpu_ctx *ctx, const uint8_t *text, size_t n, const uint32_t *keys, size_t nq, int32_t *rows_out,
                                    kxpu_table **out) {
    KX_ENTER(ctx);
    if (!out || (!text && n) || (nq && (!keys || !rows_out))) return KXPU_E_INVALID;
    kx_clear_timings(ctx);
    // staging: [text | pad to 16 | keys | rows]
    const size_t o_keys = align_up(n + 16, 256), o_rows = o_keys + align_up(nq * 4 + 16, 256);
    int32_t rc = stage_reserve(ctx, o_rows + nq * 4 + 16);
    if (rc != KXPU_OK) return rc;
    uint8_t *d = (uint8_t *)ctx->d_stage;
    // Small text in mapped pinned host memory (cudaHostAlloc / cudaHostRegister; what a host that reads /usr/pci.ids
    // into a pinned buffer passes): no copy at all.  The cooperative kernel pulls the text over PCIe in its first
    // phase (one TMA bulk copy per 2 KiB chunk, all in flight at once), reads the keys and writes the row handles and
    // the table counters straight to host memory; the call is one launch and one stream synchronisation.
    const uint32_t chunks = (uint32_t)((n + kxparse::CW - 1) / kxparse::CW);
    if (nq && chunks > 0 && chunks <= small_text_chunks(ctx)) {
        const uint8_t *m_text = (const uint8_t *)kx_mapped_host(text);
        const uint32_t *m_keys = (const uint32_t *)kx_mapped_host(keys);
        int32_t *m_rows = (int32_t *)kx_mapped_host(rows_out);
        if (m_text && m_keys && m_rows && (reinterpret_cast<uintptr_t>(m_text) & 15u) == 0) {
            const KxJoin j{m_keys, nq, m_rows, nullptr, m_text};
            return kx_build_table_join(ctx, d, n, out, &j);
        }
    }
    cudaError_t e = cudaMemcpyAsync(d, text, n, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && nq) e = cudaMemcpyAsync(d + o_keys, keys, nq * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) {
        KX_SET_ERR(ctx, "H2D copy of the text / keys failed: %s", cudaGetErrorString(e));
        return KXPU_E_CUDA;
    }
    const KxJoin j{(const uint32_t *)(d + o_keys), nq, (int32_t *)(d + o_rows), rows_out, nullptr};
    return kx_build_table_join(ctx, d, n, out, &j);
}

extern "C" int32_t kxpu_table_free(kxpu_ctx *ctx, kxpu_table *t) {
    KX_ENTER(ctx);
    kx_table_release(ctx, t);
    return KXPU_OK;
}

extern "C" int32_t kxpu_table_rows(kxpu_ctx *ctx, kxpu_table *t, uint32_t *n_rows) {
    if (!ctx || !t || !n_rows) return KXPU_E_INVALID;
    *n_rows = t->n_rows;
    return KXPU_OK;
}

extern "C" int32_t kxpu_table_export(kxpu_ctx *ctx, kxpu_table *t, uint32_t *keys, uint64_t *line_off, int32_t *rows,
                                     size_t cap, uint32_t *n_rows) {
    KX_ENTER(ctx);
    if (!t || !n_rows) return KXPU_E_INVALID;
    *n_rows = t->n_rows;
    if (cap < t->n_rows) return KXPU_E_NOSPACE;
    if (t->n_rows == 0) return KXPU_OK;
    if (!keys || !line_off || !rows) return KXPU_E_INVALID;
    std::vector<uint32_t> k(t->n_rows);
    std::vector<unsigned long long> l(t->n_rows);
    KX_CUDA(ctx, cudaMemcpyAsync(k.data(), t->row_key, t->n_rows * 4ull, cudaMemcpyDeviceToHost, ctx->stream));
    KX_CUDA(ctx, cudaMemcpyAsync(l.data(), t->row_line, t->n_rows * 8ull, cudaMemcpyDeviceToHost, ctx->stream));
    KX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<int32_t> order(t->n_rows);
    for (uint32_t i = 0; i < t->n_rows; i++) order[i] = (int32_t)i;
    std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return l[a] < l[b]; });  // file order
    for (uint32_t i = 0; i < t->n_rows; i++) {
        keys[i] = k[order[i]];
        line_off[i] = l[order[i]];
        rows[i] = order[i];
    }
    return KXPU_OK;
}

// ------------------------------------------------------------------ lookup / names
extern "C" int32_t kxpu_lookup_device(kxpu_ctx *ctx, kxpu_table *t, const uint32_t *d_keys, size_t n,
                                      int32_t *d_rows_out) {
    KX_ENTER(ctx);
    if (!t || (n && (!d_keys || !d_rows_out))) return KXPU_E_INVALID;
    kx_clear_timings(ctx);
    return kx_launch_lookup(ctx, t, d_keys, n, d_rows_out);
}

extern "C" int32_t kxpu_lookup(kxpu_ctx *ctx, kxpu_table *t, const uint32_t *keys, size_t n, int32_t *rows_out) {
    KX_ENTER(ctx);
    if (!t || (n && (!keys || !rows_out))) return KXPU_E_INVALID;
    kx_clear_timings(ctx);
    if (n == 0) return KXPU_OK;
    KxScratch sc(ctx);
    uint32_t *d_keys = nullptr;
    int32_t *d_rows = nullptr;
    KX_CUDA(ctx, sc.alloc((void **)&d_keys, n * 4));
    KX_CUDA(ctx, sc.alloc((void **)&d_rows, n * 4));
    cudaMemcpyAsync(d_keys, keys, n * 4, cudaMemcpyHostToDevice, ctx->stream);
    int32_t rc = kx_launch_lookup(ctx, t, d_keys, n, d_rows);
    cudaMemcpyAsync(rows_out, d_rows, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (rc == KXPU_OK && e != cudaSuccess) { KX_SET_ERR(ctx, "lookup failed: %s", cudaGetErrorString(e)); rc = KXPU_E_CUDA; }
    return rc;
}

extern "C" int32_t kxpu_names(kxpu_ctx *ctx, kxpu_table *t, const int32_t *rows, size_t n, uint8_t *out, size_t cap,
                              uint32_t *offsets, size_t *need) {
    KX_ENTER(ctx);
    if (!t || !offsets || (n && !rows)) return KXPU_E_INVALID;
    kx_clear_timings(ctx);
    if (n == 0) { offsets[0] = 0; if (need) *need = 0; return KXPU_OK; }
    KxScratch sc(ctx);
    int32_t *d_rows = nullptr;
    uint32_t *d_lens = nullptr, *d_offs = nullptr;
    uint8_t *d_out = nullptr;
    KX_CUDA(ctx, sc.alloc((void **)&d_rows, n * 4));
    KX_CUDA(ctx, sc.alloc((void **)&d_lens, (n + 1) * 4));
    KX_CUDA(ctx, sc.alloc((void **)&d_offs, (n + 1) * 4));
    cudaMemcpyAsync(d_rows, rows, n * 4, cudaMemcpyHostToDevice, ctx->stream);
    cudaMemsetAsync(d_lens + n, 0, 4, ctx->stream);
    int32_t rc = KXPU_OK;
    {
        KxTimer tm(ctx, KXPU_T_NAMES);
        kxparse::name_len_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d_rows, n, t->row_name_len,
                                                                                       t->n_rows, d_lens);
        KX_LAUNCHED(ctx);
        // scanning n+1 items makes offsets[n] the total
        kxscan::exclusive_scan<uint32_t>(ctx, d_lens, n + 1, d_offs, nullptr);
    }
    cudaMemcpyAsync(offsets, d_offs, (n + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { KX_SET_ERR(ctx, "names failed: %s", cudaGetErrorString(e)); rc = KXPU_E_CUDA; }
    size_t total = rc == KXPU_OK ? offsets[n] : 0;
    if (need) *need = total;
    if (rc == KXPU_OK && total > cap) rc = KXPU_E_NOSPACE;
    if (rc == KXPU_OK && total > 0) {
        if (!out) rc = KXPU_E_INVALID;
        else {
            e = sc.alloc((void **)&d_out, total);
            if (e == cudaSuccess) {
                kxparse::name_copy_kernel<<<(unsigned)((n * 8 + 255) / 256), 256, 0, ctx->stream>>>(
                    d_rows, n, t->row_name_off, t->row_name_len, t->n_rows, t->blob, d_offs, d_out, total);
                KX_LAUNCHED(ctx);
                cudaMemcpyAsync(out, d_out, total, cudaMemcpyDeviceToHost, ctx->stream);
                e = cudaStreamSynchronize(ctx->stream);
            }
            if (e != cudaSuccess) { KX_SET_ERR(ctx, "names copy failed: %s", cudaGetErrorString(e)); rc = KXPU_E_CUDA; }
        }
    }
    return rc;
}
