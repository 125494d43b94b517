// pciids5.cu -- the pci.ids parse kernel: warp-autonomous, alive-first, nothing waits.
//
// Replaces the per-key file scan of getDeviceName / locateVendor (reference
// pkg/device_plugin/device_plugin.go:208-275): the text is streamed through shared memory ONCE
// and every (vendor,device) pair is folded into a hash table with "first occurrence wins"
// semantics; lookups are then O(1) probes.
//   * the text is cut into RANGES of 8 chunks (16 KiB; fewer for texts too small to give every
//     warp of the grid a range) handed out to WARPS by ticket (a static
//     split leaves the SM half empty at the end: the issue arbiter favours some warps, they
//     finish early); a warp streams its ranges 2 KiB at a time through a private 3-stage ring
//     of 1-D TMA bulk copies (cp.async.bulk + mbarrier) -- no CTA barrier, no shared status;
//   * per chunk: newline masks (SWAR + IDP.4A) and line classes, then the TOP-LEVEL lines only
//     (hex prefix, vendor_first check/update -> alive bit).  A device line matters only under
//     the FIRST line with its vendor id (device_plugin.go:265): lines under a dead line are
//     dropped unparsed, lines under an alive one are folded by the lane that owns them;
//   * lines in front of the chunk's first top-level line are governed by the carry the warp
//     keeps in two registers along its range; at the start of a range the carry is not known
//     (the range before belongs to another warp): the warp only counts how many leading chunks
//     are affected (one word per range);
//   * resolve_ranges_kernel: one lane per range looks back over the per-range status words
//     (all published by then), 32 ranges per step; only if the governing line is alive -- the
//     first copy of a vendor block -- the leading chunks are queued, and resolve_chunks_kernel
//     stages each of them again (one warp per chunk) and folds its head lines.
// Earlier generations (CTA-tiled, per-chunk look-back, super-chunks, CTA barrier per 16 KiB) are
// in the git history and in profiles/r01_parse_v*; DESIGN.md has the numbers.
#pragma once
#include "exchange.cuh"
#include "parse_common.cuh"

namespace kxparse5 {

using namespace kxparse;

constexpr int STAGES5 = 3;
constexpr int RCH5_MAX = 8;  // chunks per range (16 KiB); fewer for small texts so that every warp gets a range
constexpr int RES_WARPS = 8;

struct WarpSmem5 {
    alignas(16) uint8_t stage[STAGES5][STG_BYTES];
    alignas(8) unsigned long long bar[STAGES5];
};

struct Params5 {
    const uint8_t *text;
    unsigned long long n, base;
    uint32_t num_chunks;
    uint32_t tma_limit;               // chunks [0, tma_limit) can be staged with one bulk copy of STG_BYTES
    uint32_t rch;                     // chunks per range, 1..RCH5_MAX
    uint32_t num_ranges;
    unsigned long long *range_state;  // [num_ranges] inclusive carry at the end of the range (ST_*/CV_*)
    uint32_t *lead;                   // [num_ranges] leading chunks whose head lines wait for the resolve kernels
    unsigned long long *range_carry;  // [num_ranges] resolve: governing line at the start of an alive range
    uint32_t *tasks;                  // [num_chunks] resolve: chunks to stage again, count in counters[KX_C_DEFER]
    KxTableDev tab;
    unsigned long long carry_in;
    // sharded load, phase A: vendor_first is final when the parse kernel is through, so the push of this shard's minima
    // rides on resolve_chunks_kernel as extra CTAs (behind the task_ctas that fold) and runs while those fold
    uint32_t task_ctas;
    int xa_on;
    uint32_t *xa_done;
    kxx::XaParams xa;
};

__global__ void __launch_bounds__(NT, 4) parse_kernel_v5(const Params5 P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    WarpSmem5 *W = reinterpret_cast<WarpSmem5 *>(smem_raw);
    uint32_t lane = threadIdx.x & 31u;
    const uint32_t w = threadIdx.x >> 5;
    asm volatile("" : "+r"(lane));  // opaque: no S2R SR_TID.X in the loop
    const uint32_t lt_mask = (1u << lane) - 1u;

    if (lane == 0) {
        for (int s = 0; s < STAGES5; s++) mbar_init(&W[w].bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    uint32_t tk = 0;
    if (lane == 0) tk = atomicAdd(&P.tab.counters[KX_C_TICKET], 1u);
    uint32_t r = __shfl_sync(0xffffffffu, tk, 0);
    if (r >= P.num_ranges) return;

    // shared-window addresses (see kxparse::lds128)
    uint32_t a_stage0 = smem_u32(smem_raw) + w * (uint32_t)sizeof(WarpSmem5);  // stage s: + s * STG_BYTES
    asm volatile("" : "+r"(a_stage0));  // opaque: keep it in a register instead of re-deriving it (S2R + LEA + IMAD) at every use
    const uint32_t a_bar0 = a_stage0 + (uint32_t)offsetof(WarpSmem5, bar);     // bar s:   + 8 * s

    uint32_t k7f = 0x7f7f7f7fu, k0a = 0x0a0a0a0au, k80 = 0x80808080u;
    asm volatile("" : "+r"(k7f), "+r"(k0a), "+r"(k80));

    const unsigned long long pol = l2_evict_first_policy();
    auto issue = [&](uint32_t g, uint32_t s) {  // lane 0: start the TMA copy of chunk g into stage s
        if (g < P.tma_limit) {
            mbar_expect_tx_a(a_bar0 + 8u * s, STG_BYTES);
            tma_load_a(a_stage0 + s * (uint32_t)STG_BYTES, P.text + (unsigned long long)g * CW, STG_BYTES, a_bar0 + 8u * s, pol);
        }
    };
    const uint32_t rch = P.rch;
    bool staged = false;  // the first chunks of the coming range are already on their way

    uint32_t phase_bits = 0, s = 0;
    uint32_t nfresh = 0;  // table slots this lane claimed in the current chunk (flushed once per warp and chunk)
    for (;;) {
        // ticket of the next range, drawn one range early; looked at (shuffled) late in this range
        uint32_t tk2 = 0, r_next = 0xffffffffu;
        bool have_next = false;
        if (lane == 0) tk2 = atomicAdd(&P.tab.counters[KX_C_TICKET], 1u);
        // carry along the range: the governing line at the start of the next chunk as a status word
        // (LS_* of parse_common.cuh; 0 = not known) plus the chunk that holds the line (0xffffffff = the
        // shard's carry-in)
        uint32_t rc_x = 0, rc_g = 0;
        if (r == 0u) {
            rc_x = LS_PUB | (((P.carry_in & CV_HAS_TOP) && (P.carry_in & CV_VOK)) ? (LS_TOP | LS_VOK) : 0u);
            rc_g = 0xffffffffu;
        }
        uint32_t lead = r == 0u ? 0u : rch;  // chunks whose head lines nobody can judge yet
        // the table ran full (the host grows it and parses again): fold nothing more.  Looked at once per
        // range, early, so that nobody waits for it; a stale answer costs bounded probing (KX_MAX_PROBE)
        const bool table_dead = *reinterpret_cast<volatile uint32_t *>(&P.tab.counters[KX_C_OVERFLOW]) != 0u;
        const uint32_t gb = r * rch;
        const uint32_t cnt = P.num_chunks - gb < rch ? P.num_chunks - gb : rch;
        if (!staged && lane == 0) {
            for (uint32_t j = 0; j < (uint32_t)STAGES5 && j < cnt; j++) issue(gb + j, (s + j) % (uint32_t)STAGES5);
        }
        staged = false;
        for (uint32_t i = 0; i < cnt; i++) {
            if (!have_next && rch > (uint32_t)STAGES5 && i + (uint32_t)STAGES5 >= rch) {
                r_next = __shfl_sync(0xffffffffu, tk2, 0);
                have_next = true;
            }
            const uint32_t g = gb + i;
            const uint32_t st = a_stage0 + s * (uint32_t)STG_BYTES;
            const unsigned long long cbase = P.base + (unsigned long long)g * CW;
            uint32_t n_rel = CW + 1;  // line starts at p < n_rel are real (p == CW: first byte of the next chunk)
            if (g < P.tma_limit) {
                const uint32_t bar = a_bar0 + 8u * s, par = (phase_bits >> s) & 1u;
                while (!mbar_try_a(bar, par)) {
                }
                phase_bits ^= 1u << s;
            } else {
                n_rel = stage_chunk_manual(P.text, P.n, g, lane, W[w].stage[s]);
            }

            uint32_t nl[2], th[2], rawnl;
            nl_masks(st, lane, n_rel, k7f, k0a, k80, nl, rawnl);
            tops_of2(st + lane * 32u + 1u, nl[0], nl[1], th[0], th[1]);

            // top-level lines, by the lane that owns them: a candidate vendor anchor; only the FIRST
            // line with this prefix counts (:265).  If an earlier one is already known, this block
            // can never produce a hit (a hit needs min_anchor == vendor_first): it is dead.
            uint32_t linfo0 = P_NONE, linfo1 = P_NONE;  // last top-level line of my windows: alive<<31 | vendor<<15 | position
            bool any_alive = (g == 0u) || (rc_x & LS_VOK) != 0u;  // the shard's first chunk and alive carries take the full path
            {
                uint32_t t0 = th[0], t1 = th[1];
                while (t0 | t1) {
                    const bool second = t0 == 0u;
                    const uint32_t tmv = second ? t1 : t0;
                    const uint32_t bit = tmv & (0u - tmv);
                    if (second) t1 = tmv ^ bit; else t0 = tmv ^ bit;
                    const uint32_t p = (second ? (uint32_t)HALF : 0u) + lane * 32u + 1u + (31u - (uint32_t)__clz((int)bit));
                    uint32_t val;
                    const bool ok = hex4_swar(lds32_unaligned(st + p), val);
                    const unsigned long long line_g = cbase + p;
                    bool alive = ok;
                    if (ok) {
                        const unsigned long long vf = P.tab.vendor_first[val];
                        if (line_g < vf) atomicMin(&P.tab.vendor_first[val], line_g);
                        alive = line_g <= vf;
                    }
                    any_alive |= alive;
                    const uint32_t info = (alive ? 0x80000000u : 0u) | ((ok ? val : 0u) << 15) | p;
                    if (second) linfo1 = info; else linfo0 = info;
                }
            }
            const uint32_t bal0 = __ballot_sync(0xffffffffu, th[0] != 0u);
            const uint32_t bal1 = __ballot_sync(0xffffffffu, th[1] != 0u);
            uint32_t last1;  // the chunk's last top-level line
            if (!__any_sync(0xffffffffu, any_alive)) {
                // common case: nothing alive in or in front of this chunk -- no device line of it
                // can matter, none is looked at
                const uint32_t bl = bal1 ? bal1 : bal0;
                last1 = __shfl_sync(0xffffffffu, bal1 ? linfo1 : linfo0, bl ? 31 - __clz((int)bl) : 0);
                if (bl == 0u) last1 = P_NONE;
            } else {
                // full path: device line candidates, governing line of every window
                uint32_t kh[2];
                kh[0] = th[0] | devs_of(st + lane * 32u + 1u, nl[0] & ~th[0]);
                kh[1] = th[1] | devs_of(st + (uint32_t)HALF + lane * 32u + 1u, nl[1] & ~th[1]);
                if (table_dead) { kh[0] = th[0]; kh[1] = th[1]; }

                // the shard starts with a line start at p = 0 (no newline before it)
                uint32_t base_info = P_NONE;  // top-level line in front of the lane windows (only that one)
                if (g == 0u && n_rel > 0u) {
                    const uint32_t c0 = lds8(st), c1 = lds8(st + 1u);
                    if (c0 != (uint32_t)'#' && c0 != (uint32_t)'\t') {
                        uint32_t val;
                        const bool ok = hex4_swar(lds32_unaligned(st), val);
                        bool alive = ok;
                        if (ok) {
                            const unsigned long long vf = P.tab.vendor_first[val];
                            if (lane == 0 && cbase < vf) atomicMin(&P.tab.vendor_first[val], cbase);
                            alive = cbase <= vf;
                        }
                        base_info = (alive ? 0x80000000u : 0u) | ((ok ? val : 0u) << 15);
                    } else if (c0 == (uint32_t)'\t' && c1 != (uint32_t)'\t') {
                        // device line at the very start: governed by the shard's carry-in, which is known
                        uint32_t dv;
                        if (lane == 0 && !table_dead && (P.carry_in & CV_HAS_TOP) && (P.carry_in & CV_VOK) && hex4_swar(lds32_unaligned(st + 1u), dv))
                            table_fold(P.tab, (((uint32_t)(P.carry_in >> 44) & 0xffffu) << 16) | dv, cbase, P.carry_in & CV_ANCHOR_MASK, nfresh);
                    }
                }
                // device lines behind the top-level lines of my windows (alive ones only)
                linfo0 = linfo1 = P_NONE;
                {
                    uint32_t t0 = th[0], t1 = th[1];
                    while (t0 | t1) {
                        const bool second = t0 == 0u;
                        const uint32_t tmv = second ? t1 : t0;
                        const uint32_t bit = tmv & (0u - tmv);
                        const uint32_t rest = tmv ^ bit;
                        if (second) t1 = rest; else t0 = rest;
                        const uint32_t pbase = (second ? (uint32_t)HALF : 0u) + lane * 32u + 1u;
                        const uint32_t p = pbase + (31u - (uint32_t)__clz((int)bit));
                        uint32_t val;
                        const bool ok = hex4_swar(lds32_unaligned(st + p), val);
                        const unsigned long long line_g = cbase + p;
                        const bool alive = ok && line_g <= P.tab.vendor_first[val];  // updated by the loop above
                        if (alive) {
                            const uint32_t nxt = rest & (0u - rest);
                            const uint32_t seg = (second ? kh[1] & ~th[1] : kh[0] & ~th[0]) & ~(bit | (bit - 1u)) & (nxt ? nxt - 1u : 0xffffffffu);
                            fold_lines(P.tab, st, cbase, seg, pbase, val << 16, line_g, nfresh);
                        }
                        const uint32_t info = (alive ? 0x80000000u : 0u) | ((ok ? val : 0u) << 15) | p;
                        if (second) linfo1 = info; else linfo0 = info;
                    }
                }
                // device lines in front of a window's first top-level line
                const uint32_t pre0 = kh[0] & ~th[0] & (th[0] ? (th[0] & (0u - th[0])) - 1u : 0xffffffffu);
                const uint32_t pre1 = kh[1] & ~th[1] & (th[1] ? (th[1] & (0u - th[1])) - 1u : 0xffffffffu);
                const uint32_t s0 = bal0 & lt_mask, s1 = bal1 & lt_mask;
                const uint32_t x0 = __shfl_sync(0xffffffffu, linfo0, s0 ? 31 - __clz((int)s0) : 0);
                const uint32_t l0 = __shfl_sync(0xffffffffu, linfo0, bal0 ? 31 - __clz((int)bal0) : 0);
                const uint32_t x1 = __shfl_sync(0xffffffffu, linfo1, s1 ? 31 - __clz((int)s1) : 0);
                const uint32_t l1 = __shfl_sync(0xffffffffu, linfo1, bal1 ? 31 - __clz((int)bal1) : 0);
                const uint32_t last0 = bal0 ? l0 : base_info;
                const uint32_t cin0 = s0 ? x0 : base_info;
                const uint32_t cin1 = s1 ? x1 : last0;
                last1 = bal1 ? l1 : last0;
                // governed by an alive line of an earlier window of this chunk
                if (cin0 != P_NONE && (cin0 >> 31))
                    fold_lines(P.tab, st, cbase, pre0, lane * 32u + 1u, ((cin0 >> 15) & 0xffffu) << 16, cbase + (cin0 & 0x7fffu), nfresh);
                if (cin1 != P_NONE && (cin1 >> 31))
                    fold_lines(P.tab, st, cbase, pre1, (uint32_t)HALF + lane * 32u + 1u, ((cin1 >> 15) & 0xffffu) << 16, cbase + (cin1 & 0x7fffu), nfresh);
                // head lines (in front of the chunk's first top-level line): governed by the carry; if
                // that is not known yet, the resolve kernels look at them
                const uint32_t hw0 = cin0 == P_NONE ? pre0 : 0u;
                const uint32_t hw1 = cin1 == P_NONE ? pre1 : 0u;
                if (rc_x & LS_VOK) {
                    uint32_t key_hi = ((rc_x >> 12) & 0xffffu) << 16;
                    unsigned long long anchor = P.base + (unsigned long long)rc_g * CW + (rc_x & 0xfffu);
                    if (rc_g == 0xffffffffu) {
                        key_hi = ((uint32_t)(P.carry_in >> 44) & 0xffffu) << 16;
                        anchor = P.carry_in & CV_ANCHOR_MASK;
                    }
                    // still the first line of its id?
                    if ((hw0 | hw1) != 0u && P.tab.vendor_first[key_hi >> 16] >= anchor) {
                        fold_lines(P.tab, st, cbase, hw0, lane * 32u + 1u, key_hi, anchor, nfresh);
                        fold_lines(P.tab, st, cbase, hw1, (uint32_t)HALF + lane * 32u + 1u, key_hi, anchor, nfresh);
                    }
                }
                flush_fresh(P.tab, nfresh);  // full path only: the branch is warp-uniform (__any_sync above)
            }
            if (last1 != P_NONE) {
                if (rc_x == 0u) lead = i + 1u;  // chunks 0..i have head lines nobody judged
                rc_x = LS_PUB | LS_TOP | ((last1 >> 31) ? LS_VOK : 0u) | (((last1 >> 15) & 0xffffu) << 12) | (last1 & 0xfffu);
                rc_g = g;
            }
            // 2 KiB without a newline may belong to a >= 64 KiB line (bufio.ErrTooLong): raise the
            // hint, the exact cut-off is then computed by trunc_kernel (never for real pci.ids)
            if ((bal0 | bal1) == 0u && n_rel > (uint32_t)CW && __reduce_or_sync(0xffffffffu, rawnl) == 0u && lane == 0)
                atomicOr(&P.tab.counters[KX_C_LONGLINE_HINT], 1u);

            // the stage is free: prefetch the chunk three steps ahead into it -- of this range, or (ranges
            // longer than the ring only) of the next one
            __syncwarp();
            {
                const uint32_t fi = i + (uint32_t)STAGES5;
                uint32_t fg = 0xffffffffu;
                if (fi < rch) {
                    fg = g + (uint32_t)STAGES5;
                } else if (rch > (uint32_t)STAGES5 && cnt == rch && r_next < P.num_ranges) {
                    fg = r_next * rch + (fi - rch);
                    staged = true;
                }
                if (lane == 0) issue(fg, s);
            }
            s = s == (uint32_t)STAGES5 - 1u ? 0u : s + 1u;
        }
        // the range's inclusive carry and its unjudged leading chunks for the resolve kernel
        if (lane == 0) {
            unsigned long long v = ST_NONE;
            if (rc_x != 0u) {
                if (rc_g == 0xffffffffu)
                    v = ST_PREFIX | P.carry_in;
                else
                    v = ST_PREFIX | CV_HAS_TOP | ((rc_x & LS_VOK) ? CV_VOK : 0ull) | ((unsigned long long)((rc_x >> 12) & 0xffffu) << 44) |
                        ((P.base + (unsigned long long)rc_g * CW + (rc_x & 0xfffu)) & CV_ANCHOR_MASK);
            }
            P.range_state[r] = v;
            P.lead[r] = lead < cnt ? lead : cnt;
        }
        if (!have_next) r_next = __shfl_sync(0xffffffffu, tk2, 0);
        r = r_next;
        if (r >= P.num_ranges) break;
    }
}

// Resolve, step 1: the leading chunks of every range, whose governing line was not known to the
// warp that parsed them.  One lane per range; the governing line is the inclusive carry of the
// nearest earlier range that published one (all status words are final now).  The look-back is
// warp-cooperative: 32 status words per step, first inside the warp's own 32 ranges, then
// backwards 32 at a time -- one step for real data, at most num_ranges/32 steps for a text whose
// top-level lines are megabytes apart.  The governing line is dead for all but the first copy of
// a vendor block; only then the range's leading chunks are queued for step 2.
constexpr uint32_t XA_CTAS = 64;  // extra CTAs of resolve_chunks_kernel that push phase A

__global__ void __launch_bounds__(256) resolve_ranges_kernel(const Params5 P) {
    const uint32_t rr = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t rr0 = rr - lane;  // first range of this warp
    if (rr0 >= P.num_ranges) return;
    const bool live = rr < P.num_ranges;
    const uint32_t nlead = live ? P.lead[rr] : 0u;
    // my own status word serves the lanes behind me
    const unsigned long long own = live ? P.range_state[rr] : ST_NONE;
    const uint32_t pm = __ballot_sync(0xffffffffu, (own & ST_MASK) == ST_PREFIX);
    const uint32_t below = pm & ((1u << lane) - 1u);
    const unsigned long long from_warp = __shfl_sync(0xffffffffu, own, below ? 31 - __clz((int)below) : 0);
    // carry into the warp's first range (needed by the lanes in front of the warp's first prefix)
    unsigned long long warp_in = 0;
    const uint32_t first_p = pm ? (uint32_t)__ffs((int)pm) - 1u : 32u;
    const bool want = __any_sync(0xffffffffu, nlead != 0u && lane <= first_p);
    if (want) {
        long long q0 = (long long)rr0 - 32;
        for (;;) {
            const long long q = q0 + lane;
            const unsigned long long sv = q >= 0 ? P.range_state[q] : (q == -1 ? (ST_PREFIX | P.carry_in) : ST_NONE);
            const uint32_t m = __ballot_sync(0xffffffffu, (sv & ST_MASK) == ST_PREFIX);
            if (m) {
                warp_in = __shfl_sync(0xffffffffu, sv, 31 - __clz((int)m));
                break;
            }
            q0 -= 32;  // q == -1 (the shard's carry-in) always answers: the loop ends at the latest there
        }
    }
    // no top-level line between the start of the range and those chunks' head lines: the carry
    // into the range governs them
    const unsigned long long carry = (below ? from_warp : warp_in) & ~ST_MASK;
    const bool alive = nlead != 0u && (carry & CV_HAS_TOP) && (carry & CV_VOK) &&
                       P.tab.vendor_first[(uint32_t)(carry >> 44) & 0xffffu] >= (carry & CV_ANCHOR_MASK);  // vendor_first is final here
    // queue space: one atomic per warp (in a text without repeated blocks every range queues its chunks)
    const uint32_t mine = alive ? nlead : 0u;
    const uint32_t incl = warp_incl_scan(mine);
    const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t at0 = 0;
    if (lane == 0 && tot) at0 = atomicAdd(&P.tab.counters[KX_C_DEFER], tot);
    at0 = __shfl_sync(0xffffffffu, at0, 0);
    if (!alive) return;
    P.range_carry[rr] = carry;
    const uint32_t at = at0 + incl - mine;
    for (uint32_t j = 0; j < nlead; j++) P.tasks[at + j] = rr * P.rch + j;
}

// Resolve, step 2: one warp per queued chunk stages it again and folds its head lines (the
// device lines in front of its first top-level line) under the range's governing line.  Six CTAs
// per SM (40 registers): left to itself ptxas trades spills in the task loop for occupancy.
__global__ void __launch_bounds__(RES_WARPS * 32, 6) resolve_chunks_kernel(const Params5 P) {
    __shared__ __align__(16) uint8_t stg[RES_WARPS][STG_BYTES];
    __shared__ __align__(8) unsigned long long bars[RES_WARPS];
    __shared__ uint32_t s_list[RES_WARPS][LIST_CAP];
    if (blockIdx.x >= P.task_ctas) {
        // phase A of the sharded load: these CTAs push slices of the shard's vendor minima into every rank's region while
        // the others fold; the one that finishes last adds cut-off and status and raises the flags (the barrier +
        // thread 0's cumulative system fence order each CTA's pushes in front of its count).  What the folds may
        // still find out (table full) travels with phase B.
        kxx::xa_push_slice(P.xa, (blockIdx.x - P.task_ctas) * blockDim.x + threadIdx.x, XA_CTAS * blockDim.x);
        __syncthreads();
        if (threadIdx.x == 0) {
            kx_fence_sys();
            const uint32_t prev = atomicAdd(P.xa_done, 1u);
            if (prev == XA_CTAS - 1u) {
                *P.xa_done = 0u;
                kx_fence_sys();
                kxx::xa_finish(P.xa);
            }
        }
        return;
    }
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    uint32_t k7f = 0x7f7f7f7fu, k0a = 0x0a0a0a0au, k80 = 0x80808080u;
    asm volatile("" : "+r"(k7f), "+r"(k0a), "+r"(k80));
    const uint32_t st = smem_u32(stg[w]), bar = smem_u32(&bars[w]);
    if (lane == 0) {
        mbar_init(&bars[w], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const unsigned long long pol = l2_evict_first_policy();
    const uint32_t n_tasks = P.tab.counters[KX_C_DEFER];
    uint32_t par = 0, nfresh = 0;
    // L2-resident table: claim first (one round trip per probe step); a table in DRAM: load first -- measured 2.5x
    // faster there (12.4 M keys, 1 GB table: 0.55 ms against 1.4 ms)
    const bool small_tab = P.tab.cap <= (1u << 20);
    uint32_t it = 0;
    for (uint32_t t = blockIdx.x * RES_WARPS + w; t < n_tasks; t += P.task_ctas * RES_WARPS, it++) {
        // table full: the host grows it and parses again (polled every fourth task: a stale answer costs bounded probing)
        if ((it & 3u) == 0u && *reinterpret_cast<volatile uint32_t *>(&P.tab.counters[KX_C_OVERFLOW]) != 0u) break;
        const uint32_t gg = P.tasks[t];
        uint32_t n_rel = CW + 1;
        if (gg < P.tma_limit) {
            stage_chunk_tma(st, P.text + (unsigned long long)gg * CW, bar, par, lane, pol);
            par ^= 1u;
        } else {
            n_rel = stage_chunk_manual(P.text, P.n, gg, lane, stg[w]);
        }
        const unsigned long long cc = P.range_carry[gg / P.rch];
        uint32_t nl[2], th[2], rawnl;
        nl_masks(st, lane, n_rel, k7f, k0a, k80, nl, rawnl);
        tops_of2(st + lane * 32u + 1u, nl[0], nl[1], th[0], th[1]);
        const uint32_t bal0 = __ballot_sync(0xffffffffu, th[0] != 0u);
        const uint32_t bal1 = __ballot_sync(0xffffffffu, th[1] != 0u);
        // head lines: the device lines of the windows in front of the chunk's first top-level line
        const uint32_t pre0 = nl[0] & (th[0] ? (th[0] & (0u - th[0])) - 1u : 0xffffffffu);
        const uint32_t pre1 = nl[1] & (th[1] ? (th[1] & (0u - th[1])) - 1u : 0xffffffffu);
        const uint32_t head[2] = {(bal0 & lt_mask) == 0u ? devs_of(st + lane * 32u + 1u, pre0) : 0u,
                                  (bal0 == 0u && (bal1 & lt_mask) == 0u) ? devs_of(st + (uint32_t)HALF + lane * 32u + 1u, pre1) : 0u};
        const uint32_t none[2] = {0u, 0u}, gov[2] = {LIST_CARRY, LIST_CARRY};
        fold_list(P.tab, s_list[w], st, P.base + (unsigned long long)gg * CW, head, none, none, gov, ((uint32_t)(cc >> 44) & 0xffffu) << 16,
                  cc & CV_ANCHOR_MASK, small_tab, nfresh);
        flush_fresh(P.tab, nfresh);
    }
}

}  // namespace kxparse5
