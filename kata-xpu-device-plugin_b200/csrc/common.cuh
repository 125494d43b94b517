// common.cuh -- context, error plumbing and small device helpers shared by the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/kxpu.h"

constexpr int KX_MAX_RANKS = 16;  // ranks of one sharded load (one NVSwitch domain)


struct KxArena {  // one pooled table arena (api.cu): reset on release, handed out clean
    void *p = nullptr;
    size_t bytes = 0;
    uint32_t cap = 0, blob_cap = 0;
    size_t range_bytes = 0;
};

struct KxExchange;  // comm.cu: peer-memory exchange state of a sharded load
struct kxpu_multi;

struct kxpu_ctx {
    int device = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[2 * KXPU_T_COUNT] = {};
    cudaEvent_t ev_user[2] = {};
    bool ev_used[KXPU_T_COUNT] = {};
    int force_rch = 0;         // KXPU_RCH: chunks per parse range (0 = automatic), for tests
    bool no_small = false;     // KXPU_NO_SMALL: never use the cooperative small-text kernel, for tests
    int small_chunks = -1;     // chunks the small-text kernel can take (-1: not asked yet)
    bool stage_timing = true;  // per-stage CUDA events (kxpu_last_timings); kxpu_set_stage_timing(ctx, 0) drops them
    uint64_t launches = 0;
    std::mutex mu;
    char err[512] = {0};
    // pinned staging for small H2D/D2H control words
    uint32_t *h_ctl = nullptr;  // KX_C_COUNT + 64 words, pinned
    // table arenas: released tables park their (already reset) arena here
    std::vector<KxArena> pool;
    uint32_t cap_hint = 1u << 16;       // table capacity the next load starts with (follows the last text)
    uint32_t blob_hint = 0;             // name blob capacity of the last load (0 = derive from the text size)
    // tile status words of the single-pass scans / look-backs (scan.cuh): zeroed once, epoch-tagged
    unsigned long long *scan_state = nullptr;
    size_t scan_state_words = 0;
    uint32_t scan_epoch = 0;
    // host staging of kxpu_pciids_load / kxpu_lookup (grown on demand, kept)
    void *d_stage = nullptr;
    size_t d_stage_bytes = 0;
    // NCCL (lazy) and the exchange of the sharded load (comm.cu)
    void *nccl_comm = nullptr;
    int nranks = 1, rank = 0;
    KxExchange *xch = nullptr;
    kxpu_multi *multi = nullptr;  // set when the ctx belongs to a kxpu_ctx_create_multi group
};

#define KX_SET_ERR(ctx, ...) snprintf((ctx)->err, sizeof((ctx)->err), __VA_ARGS__)

#define KX_CUDA(ctx, call)                                                                  \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            KX_SET_ERR(ctx, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return KXPU_E_CUDA;                                                             \
        }                                                                                   \
    } while (0)

#define KX_LAUNCHED(ctx) ((ctx)->launches++)

struct KxTimer {  // records a CUDA-event pair around a stage on the ctx stream
    kxpu_ctx *c;
    int idx;
    bool open = true;
    KxTimer(kxpu_ctx *ctx, int i) : c(ctx), idx(i) {
        open = c->stage_timing;
        if (open) cudaEventRecord(c->ev[2 * i], c->stream);
    }
    void stop() {
        if (open) { cudaEventRecord(c->ev[2 * idx + 1], c->stream); c->ev_used[idx] = true; open = false; }
    }
    ~KxTimer() { stop(); }
};

static inline void kx_clear_timings(kxpu_ctx *c) { memset(c->ev_used, 0, sizeof(c->ev_used)); }

// >= `words` zero-initialised-once status words for look-backs (nullptr on allocation failure) and
// the epoch of the next look-back (api.cu)
unsigned long long *kx_scan_state(kxpu_ctx *ctx, size_t words);
uint32_t kx_next_epoch(kxpu_ctx *ctx);

// stream-ordered scratch that is released on every path out of a call
struct KxScratch {
    kxpu_ctx *c;
    std::vector<void *> ptrs;
    explicit KxScratch(kxpu_ctx *ctx) : c(ctx) {}
    cudaError_t alloc(void **p, size_t bytes) {
        cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 16, c->stream);
        if (e == cudaSuccess) ptrs.push_back(*p);
        else *p = nullptr;
        return e;
    }
    ~KxScratch() {
        for (void *p : ptrs) cudaFreeAsync(p, c->stream);
    }
};

// ------------------------------------------------------------------ device helpers
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t kx_lane() { return threadIdx.x & 31u; }

// Release / acquire fences.  __threadfence() and __threadfence_system() are fence.sc (MEMBAR.SC): sequentially
// consistent, i.e. totally ordered against every other SC fence in flight -- with one per CTA at a phase
// boundary they queue up.  Every fence in this library orders data in front of a flag / counter (release) or a
// flag / counter in front of data (acquire): fence.acq_rel (MEMBAR.ALL + L1 invalidate) is what that needs.
__device__ __forceinline__ void kx_fence_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void kx_fence_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

__device__ __forceinline__ uint32_t kx_hash(uint32_t key) { return key * 0x9E3779B1u; }
#endif
