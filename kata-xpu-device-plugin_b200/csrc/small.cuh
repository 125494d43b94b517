// small.cuh -- the whole load of a SMALL pci.ids text (the real file is 1.4 MB: BASELINE configs[1])
// in ONE cooperative kernel: every warp keeps ONE 2 KiB chunk in shared memory through all phases,
// grid-wide barriers stand where the big-text path has kernel boundaries.
//   phase 1  newline masks, top-level lines, vendor_first minima, the chunk's last top-level line
//            (published for the chunks behind it)
//   phase 2  vendor_first is final: the governing line of the chunk's head comes from a look-back
//            over the published words; every device line under a FIRST anchor (device_plugin.go:265)
//            is folded into the table -- no deferred lines, no second staging of the chunk
//   phase 3  validity + names (select_finalize_body, the same code as the big-text kernel)
//   phase 4  the batched join, if the caller passed keys
// One launch instead of five; the latency chains of the phases remain (parse ~5 us, fold ~8 us,
// names ~15 us), the launch gaps and the second pass over the head lines go.
#pragma once
#include "finalize.cuh"
#include "pciids5.cu"

namespace kxsmall {

using namespace kxparse;

struct SmallParams {
    const uint8_t *text;
    unsigned long long n;
    uint32_t num_chunks, tma_limit;
    unsigned long long *state;  // [num_chunks] inclusive governing line at the end of the chunk (ST_* / CV_*)
    FinalizeParams F;           // F.tab is the table
    const uint32_t *keys;       // join (may be null)
    size_t nq;
    int32_t *rows_out;
    const uint8_t *text_src;    // zero-copy ingest: the text in mapped pinned HOST memory (phase 1 reads it over PCIe and leaves a
                                // device copy in `text` for the later phases); nullptr: `text` already is the device copy
    uint32_t *h_ctl;            // zero-copy: the table counters go straight to this mapped host buffer (after the names phase)
    long long *trace;           // KXPU_TRACE_SMALL: [gridDim.x][8] clock64 at the phase boundaries (thread 0 of every CTA)
};

__device__ __forceinline__ void grid_barrier(uint32_t *ctr, uint32_t target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        kx_fence_gpu();
        atomicAdd(ctr, 1u);
        while (*reinterpret_cast<volatile uint32_t *>(ctr) < target) {
        }
        kx_fence_gpu();
    }
    __syncthreads();
}

#define KX_SMALL_MARK(k) do { if (P.trace && threadIdx.x == 0) P.trace[blockIdx.x * 8u + (k)] = clock64(); } while (0)

__global__ void __launch_bounds__(NT, 4) small_load_kernel(const SmallParams P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    KX_SMALL_MARK(0);
    __shared__ __align__(8) unsigned long long bars[WARPS];
    __shared__ uint32_t s_list[WARPS][LIST_CAP];
    const KxTableDev &tab = P.F.tab;
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t g = blockIdx.x * WARPS + w;
    const bool have = g < P.num_chunks;
    uint8_t *stage = smem_raw + w * STG_BYTES;
    const uint32_t st = smem_u32(stage);
    uint32_t k7f = 0x7f7f7f7fu, k0a = 0x0a0a0a0au, k80 = 0x80808080u;
    const unsigned long long cbase = (unsigned long long)g * CW;

    // ---------------------------------------------------------------- phase 1
    uint32_t n_rel = CW + 1, nl[2] = {0, 0}, th[2] = {0, 0}, kh[2] = {0, 0}, rawnl = 0;
    uint32_t base_info = P_NONE;  // top-level line at offset 0 of the text (no newline in front of it)
    if (have) {
        const uint8_t *src = P.text_src ? P.text_src : P.text;
        if (g < P.tma_limit) {
            if (lane == 0) {
                mbar_init(&bars[w], 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            }
            __syncwarp();
            stage_chunk_tma(st, src + cbase, smem_u32(&bars[w]), 0u, lane, l2_evict_first_policy());
        } else {
            n_rel = stage_chunk_manual(src, P.n, g, lane, stage);
        }
        if (P.text_src) {
            // zero-copy ingest: the chunk came over PCIe; its 2 KiB go to the device copy the names phase reads
            // (the copy has 16 bytes of slack behind n; bytes behind the text are zero in the stage)
            uint8_t *dcopy = const_cast<uint8_t *>(P.text) + cbase;
#pragma unroll
            for (int k = 0; k < CW / 16 / 32; k++) {
                const uint32_t cc = lane + 32u * (uint32_t)k;
                if (cbase + 16ull * cc < P.n) *reinterpret_cast<uint4 *>(dcopy + 16u * cc) = *reinterpret_cast<const uint4 *>(stage + 16u * cc);
            }
        }
        nl_masks(st, lane, n_rel, k7f, k0a, k80, nl, rawnl);
        tops_of2(st + lane * 32u + 1u, nl[0], nl[1], th[0], th[1]);
        kh[0] = th[0] | devs_of(st + lane * 32u + 1u, nl[0] & ~th[0]);
        kh[1] = th[1] | devs_of(st + (uint32_t)HALF + lane * 32u + 1u, nl[1] & ~th[1]);
        // top-level lines: candidate vendor anchors (only the FIRST line with a prefix counts, :265)
        uint32_t last_mine = P_NONE;  // [31] hex ok, [30:15] vendor, [14:0] position
        for (int h = 0; h < 2; h++) {
            uint32_t t = th[h];
            while (t) {
                const uint32_t bit = t & (0u - t);
                t ^= bit;
                const uint32_t p = (uint32_t)h * HALF + lane * 32u + 1u + (31u - (uint32_t)__clz((int)bit));
                uint32_t val;
                const bool ok = hex4_swar(lds32_unaligned(st + p), val);
                if (ok && cbase + p < tab.vendor_first[val]) atomicMin(&tab.vendor_first[val], cbase + p);
                last_mine = (ok ? 0x80000000u : 0u) | ((ok ? val : 0u) << 15) | p;
            }
        }
        if (g == 0u && n_rel > 0u) {
            const uint32_t c0 = lds8(st);
            if (c0 != (uint32_t)'#' && c0 != (uint32_t)'\t') {
                uint32_t val;
                const bool ok = hex4_swar(lds32_unaligned(st), val);
                if (ok && lane == 0 && 0ull < tab.vendor_first[val]) atomicMin(&tab.vendor_first[val], 0ull);
                base_info = (ok ? 0x80000000u : 0u) | ((ok ? val : 0u) << 15);
            }
        }
        uint32_t last1;
        // a lane's windows: half 0 then half 1 -- the LAST top-level line of the chunk is the one at the
        // highest position, which need not sit in the highest lane: take the maximum position
        {
            uint32_t best = last_mine == P_NONE ? 0u : ((last_mine & 0x7fffu) + 1u);
            const uint32_t mx = __reduce_max_sync(0xffffffffu, best);
            const uint32_t who = __ballot_sync(0xffffffffu, best == mx && best != 0u);
            last1 = mx ? __shfl_sync(0xffffffffu, last_mine, (uint32_t)__ffs((int)who) - 1u) : base_info;
        }
        if (lane == 0) {
            unsigned long long v = ST_NONE;
            if (last1 != P_NONE)
                v = ST_PREFIX | CV_HAS_TOP | ((last1 >> 31) ? CV_VOK : 0ull) | ((unsigned long long)((last1 >> 15) & 0xffffu) << 44) |
                    ((cbase + (last1 & 0x7fffu)) & CV_ANCHOR_MASK);
            else if (g == 0u)
                v = ST_PREFIX;  // nothing governs the start of the text
            P.state[g] = v;
        }
        if (n_rel > (uint32_t)CW && __reduce_or_sync(0xffffffffu, rawnl) == 0u && lane == 0)
            atomicOr(&tab.counters[KX_C_LONGLINE_HINT], 1u);  // 2 KiB without a newline: maybe a >= 64 KiB line
    }
    KX_SMALL_MARK(1);
    grid_barrier(&tab.counters[KX_C_GRIDBAR], gridDim.x);
    KX_SMALL_MARK(2);

    // ---------------------------------------------------------------- phase 2
    uint32_t nfresh = 0;
    if (have) {
        // governing line at the start of the chunk: nearest published prefix in front of it
        unsigned long long carry = 0;
        if (g > 0u) {
            long long q0 = (long long)g - 1;
            for (;;) {
                const long long q = q0 - lane;
                const unsigned long long sv = q >= 0 ? P.state[q] : ST_NONE;
                const uint32_t m = __ballot_sync(0xffffffffu, (sv & ST_MASK) == ST_PREFIX);
                if (m) {
                    carry = __shfl_sync(0xffffffffu, sv, (uint32_t)__ffs((int)m) - 1u) & ~ST_MASK;
                    break;
                }
                q0 -= 32;  // chunk 0 always publishes a prefix: the loop ends there at the latest
            }
        }
        // my windows' top-level lines: alive iff the line is the FIRST of its vendor id (its offset is the final
        // vendor_first); linfo = last top-level line of the window
        uint32_t linfo[2] = {P_NONE, P_NONE}, at[2] = {0u, 0u};
        for (int h = 0; h < 2; h++) {
            uint32_t t = th[h];
            const uint32_t pbase = (uint32_t)h * HALF + lane * 32u + 1u;
            while (t) {
                const uint32_t bit = t & (0u - t);
                t ^= bit;
                const uint32_t p = pbase + (31u - (uint32_t)__clz((int)bit));
                uint32_t val;
                const bool ok = hex4_swar(lds32_unaligned(st + p), val);
                const bool alive = ok && cbase + p == tab.vendor_first[val];
                if (alive) at[h] |= bit;
                linfo[h] = (alive ? 0x80000000u : 0u) | ((ok ? val : 0u) << 15) | p;
            }
        }
        if (g == 0u && base_info != P_NONE)  // the line at offset 0: alive iff it is the first of its id
            base_info = (base_info & 0x7fffffffu) | (((base_info >> 31) && tab.vendor_first[(base_info >> 15) & 0xffffu] == 0ull) ? 0x80000000u : 0u);
        // device lines in front of a window's first top-level line: governed by the last top-level line of
        // an earlier window of this chunk, else by the carry
        const uint32_t bal0 = __ballot_sync(0xffffffffu, th[0] != 0u), bal1 = __ballot_sync(0xffffffffu, th[1] != 0u);
        const uint32_t s0 = bal0 & lt_mask, s1 = bal1 & lt_mask;
        const uint32_t x0 = __shfl_sync(0xffffffffu, linfo[0], s0 ? 31 - __clz((int)s0) : 0);
        const uint32_t l0 = __shfl_sync(0xffffffffu, linfo[0], bal0 ? 31 - __clz((int)bal0) : 0);
        const uint32_t x1 = __shfl_sync(0xffffffffu, linfo[1], s1 ? 31 - __clz((int)s1) : 0);
        const uint32_t last0 = bal0 ? l0 : base_info;
        const uint32_t cin[2] = {s0 ? x0 : base_info, s1 ? x1 : last0};
        const uint32_t cv = (uint32_t)(carry >> 44) & 0xffffu;
        const unsigned long long canchor = carry & CV_ANCHOR_MASK;
        const bool carry_alive = (carry & CV_HAS_TOP) && (carry & CV_VOK) && tab.vendor_first[cv] == canchor;
        uint32_t gov[2];  // governing line in front of window h
        for (int h = 0; h < 2; h++)
            gov[h] = cin[h] == P_NONE ? (carry_alive ? LIST_CARRY : LIST_DEAD) : ((cin[h] >> 31) ? (cin[h] & 0x7fffu) : LIST_DEAD);
        fold_list(tab, s_list[w], st, cbase, kh, th, at, gov, cv << 16, canchor, true, nfresh);
    }
    flush_fresh(tab, nfresh);
    KX_SMALL_MARK(3);
    grid_barrier(&tab.counters[KX_C_GRIDBAR], 2u * gridDim.x);
    KX_SMALL_MARK(4);

    // ---------------------------------------------------------------- phase 3
    select_finalize_body(P.F, P.F.scan_w);
    KX_SMALL_MARK(5);
    if (P.nq == 0) return;
    grid_barrier(&tab.counters[KX_C_GRIDBAR], 3u * gridDim.x);
    KX_SMALL_MARK(6);
    if (P.h_ctl && blockIdx.x == 0 && threadIdx.x < KX_C_COUNT) P.h_ctl[threadIdx.x] = __ldcg(&tab.counters[threadIdx.x]);  // final since the barrier

    // ---------------------------------------------------------------- phase 4
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < P.nq; i += stride)
        P.rows_out[i] = table_probe(tab.slots, tab.cap, tab.shift, P.keys[i]);
    KX_SMALL_MARK(7);
}

}  // namespace kxsmall
