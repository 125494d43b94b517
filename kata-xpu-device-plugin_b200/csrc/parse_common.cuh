// parse_common.cuh -- building blocks of the pci.ids parse kernels (pciids5.cu, small.cuh) and of
// the kernels behind them (finalize.cuh, comm.cu): chunk geometry, status-word encodings, mbarrier /
// 1-D TMA bulk copy wrappers and chunk staging, the SWAR newline and hex primitives, line classes,
// shared-window accessors, the table fold ("first occurrence wins", device_plugin.go:237,265) and
// the per-warp fold list.
#pragma once
#include "common.cuh"
#include "table.cuh"

namespace kxparse {

constexpr int CW = 2048;                 // chunk bytes per warp iteration
constexpr int HALF = 1024;
constexpr int TRAIL = 16;                // bytes staged after the chunk (line head reads)
constexpr int STG_BYTES = CW + TRAIL;
constexpr int WARPS = 8;                 // per CTA
constexpr int NT = WARPS * 32;

// range_state word: [63:62] status, [61] has_top, [60] vendor valid, [59:44] vendor, [43:0] anchor
constexpr unsigned long long ST_NONE = 1ull << 62;    // published: range holds no top-level line
constexpr unsigned long long ST_PREFIX = 2ull << 62;  // published: inclusive governing line
constexpr unsigned long long ST_MASK = 3ull << 62;
constexpr unsigned long long CV_HAS_TOP = 1ull << 61;
constexpr unsigned long long CV_VOK = 1ull << 60;
constexpr unsigned long long CV_ANCHOR_MASK = (1ull << 44) - 1;
constexpr uint32_t KX_MAX_PROBE = 1024;  // longest probe run a table within its load limit can show (inserts give up beyond)
constexpr uint32_t P_NONE = 0xFFFFFFFFu;  // packed top info: [31] alive, [30:15] vendor, [14:0] position
// carry along a range (one register): [31] known, [30] top-level line seen, [29] alive vendor line,
// [27:12] vendor, [11:0] position in its chunk
#define LS_PUB 0x80000000u
#define LS_TOP 0x40000000u
#define LS_VOK 0x20000000u

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

// The text is streamed exactly once, while the (vendor,device) table must stay L2 resident for
// the folds: bulk copies carry an L2 evict-first policy.
__device__ __forceinline__ unsigned long long l2_evict_first_policy() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}

__device__ __forceinline__ uint32_t lop3_and_xor(uint32_t a, uint32_t b, uint32_t c) {  // (a & b) ^ c
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x6A;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t lop3_nor_and(uint32_t a, uint32_t b, uint32_t c) {  // ~(a | b) & c
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x02;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// 16-bit mask of the bytes of v that equal '\n' (bit b = byte b).  Per word: the exact
// zero-byte test on y = x^0x0a..: t = (y & 0x7f..) + 0x7f..; flag = ~(t | y) & 0x80.. -- bit 7 of
// y equals bit 7 of x (0x0a has it clear), so x itself feeds the last LOP3 (3 ops), then IDP.4A
// gathers the four 0x80 flags, weighted 1,2,4,8 (or 16..128), straight into the accumulator.
__device__ __forceinline__ uint32_t nl_mask16(const uint4 v, uint32_t k7f, uint32_t k0a, uint32_t k80) {
    uint32_t f0 = lop3_nor_and(lop3_and_xor(v.x, k7f, k0a) + k7f, v.x, k80);
    uint32_t f1 = lop3_nor_and(lop3_and_xor(v.y, k7f, k0a) + k7f, v.y, k80);
    uint32_t f2 = lop3_nor_and(lop3_and_xor(v.z, k7f, k0a) + k7f, v.z, k80);
    uint32_t f3 = lop3_nor_and(lop3_and_xor(v.w, k7f, k0a) + k7f, v.w, k80);
    uint32_t lo = __dp4a(f0, 0x08040201u, 0u);
    lo = __dp4a(f1, 0x80402010u, lo);
    uint32_t hi = __dp4a(f2, 0x08040201u, 0u);
    hi = __dp4a(f3, 0x80402010u, hi);
    return (lo >> 7) | (hi << 1);  // flags are 0x80 = 128 * {0,1}
}

// Four ASCII bytes (first character in the low byte) -> 16-bit value, SWAR.  Only [0-9a-f]
// passes (sysfs ids are lowercase and the reference compares raw bytes, strings.HasPrefix,
// device_plugin.go:237,265): the value is converted back to text and compared with the input.
__device__ __forceinline__ bool hex4_swar(uint32_t x, uint32_t &val) {
    uint32_t v = (x & 0x0f0f0f0fu) + ((x >> 6) & 0x01010101u) * 9u;           // nibble values per byte
    uint32_t r = v + 0x30303030u + (((v + 0x06060606u) >> 4) & 0x01010101u) * 0x27u;  // back to lowercase hex
    uint32_t s = __byte_perm(v, 0u, 0x0123);                                  // first char -> high byte
    uint32_t u = s | (s >> 4);
    val = __byte_perm(u, 0u, 0x4420);                                         // (d0<<12)|(d1<<8)|(d2<<4)|d3
    return ((v & 0xf0f0f0f0u) == 0u) & (r == x);
}

// Fold one device line into the table (first occurrence wins).  The slot is one 32-byte
// sector: key and min_line arrive with one load.  `fresh` counts the slots this thread claimed:
// the caller adds it to counters[KX_C_NKEYS] once per warp and chunk (one same-address atomic per
// key would serialise in L2 when every block is a first occurrence).
__device__ __forceinline__ void table_fold(const KxTableDev &tb, uint32_t key, unsigned long long line_g,
                                           unsigned long long anchor_g, uint32_t &fresh_cnt) {
    uint32_t slot = key == KX_EMPTY_KEY ? tb.cap : (kx_hash(key) >> tb.shift);
    uint4 head = __ldcg(reinterpret_cast<const uint4 *>(&tb.slots[slot]));  // key, row, min_line (L2: where the atomics live)
    uint32_t k = head.x;
    unsigned long long ml = ((unsigned long long)head.w << 32) | head.z;
    if (key != KX_EMPTY_KEY && k != key) {
        uint32_t step = 0;
        bool fresh = false;
        for (;;) {
            if (k == KX_EMPTY_KEY) {
                uint32_t old = atomicCAS(&tb.slots[slot].key, KX_EMPTY_KEY, key);
                if (old == KX_EMPTY_KEY) {
                    fresh_cnt++;
                    fresh = true;
                    break;
                }
                if (old == key) break;
            }
            slot = (slot + 1) & (tb.cap - 1);
            // below the 50 % load limit a probe run of KX_MAX_PROBE is out of the question: the table is
            // (over)full, the host grows it and parses again -- do not crawl through a full table
            if (++step >= KX_MAX_PROBE) { tb.counters[KX_C_OVERFLOW] = 1u; return; }
            k = __ldcg(&tb.slots[slot].key);
            if (k == key) break;
        }
        // a slot this thread just claimed still holds the initial (maximal) minima: no need to read them
        ml = fresh ? KX_NO_OFF : __ldcg(&tb.slots[slot].min_line);
    }
    if (line_g < ml) {
        atomicMin(&tb.slots[slot].min_line, line_g);
        atomicMin(&tb.slots[slot].min_anchor, anchor_g);
    }
}

// The fold for the callers that run on a latency chain (resolve_chunks_kernel, the small-text kernel: few
// lines, every one of them under a FIRST anchor, so a key is hardly ever seen twice): claim first, never load.
// A probe step is ONE round trip (the CAS returns what the slot holds) instead of load + CAS, and a warp's step
// count is the maximum over its lanes -- with the load the 32 folds of a warp took ~7 000 cycles.  The minima
// go out unconditionally (no return value, nobody waits for them).  Two folds per lane (on1: the second one
// exists), their probe steps in flight together.
__device__ __forceinline__ void table_fold_claim2(const KxTableDev &tb, uint32_t key0, unsigned long long line0, unsigned long long anchor0,
                                                  bool on1, uint32_t key1, unsigned long long line1, unsigned long long anchor1,
                                                  uint32_t &fresh_cnt) {
    uint32_t slot0 = key0 == KX_EMPTY_KEY ? tb.cap : (kx_hash(key0) >> tb.shift);
    uint32_t slot1 = key1 == KX_EMPTY_KEY ? tb.cap : (kx_hash(key1) >> tb.shift);
    bool open0 = key0 != KX_EMPTY_KEY, open1 = on1 && key1 != KX_EMPTY_KEY, ok0 = true, ok1 = on1;
    for (uint32_t step = 0; open0 || open1; step++) {
        uint32_t old0 = 0, old1 = 0;
        if (open0) old0 = atomicCAS(&tb.slots[slot0].key, KX_EMPTY_KEY, key0);
        if (open1) old1 = atomicCAS(&tb.slots[slot1].key, KX_EMPTY_KEY, key1);
        if (open0) {
            if (old0 == KX_EMPTY_KEY) { fresh_cnt++; open0 = false; }
            else if (old0 == key0) open0 = false;
            else slot0 = (slot0 + 1) & (tb.cap - 1);
        }
        if (open1) {
            if (old1 == KX_EMPTY_KEY) { fresh_cnt++; open1 = false; }
            else if (old1 == key1) open1 = false;
            else slot1 = (slot1 + 1) & (tb.cap - 1);
        }
        if (step + 1 >= KX_MAX_PROBE && (open0 || open1)) {  // (over)full: the host grows the table
            tb.counters[KX_C_OVERFLOW] = 1u;
            ok0 = ok0 && !open0; ok1 = ok1 && !open1;
            break;
        }
    }
    if (ok0) { atomicMin(&tb.slots[slot0].min_line, line0); atomicMin(&tb.slots[slot0].min_anchor, anchor0); }
    if (ok1) { atomicMin(&tb.slots[slot1].min_line, line1); atomicMin(&tb.slots[slot1].min_anchor, anchor1); }
}

// row handle of `key` in a finished table (-1 = miss): key and row share one 8-byte load
__device__ __forceinline__ int32_t table_probe(const KxSlot *__restrict__ slots, uint32_t cap, uint32_t shift, uint32_t key) {
    if (key == KX_EMPTY_KEY) return slots[cap].row;
    uint32_t slot = kx_hash(key) >> shift;
    for (uint32_t step = 0; step < cap; step++) {
        const uint2 kr = __ldg(reinterpret_cast<const uint2 *>(&slots[slot]));  // key, row
        if (kr.x == key) return (int32_t)kr.y;
        if (kr.x == KX_EMPTY_KEY) return -1;
        slot = (slot + 1) & (cap - 1);
    }
    return -1;
}

// four keys at once: the probe loads of a step are in flight together (a probe is one L2 round trip; used where
// a thread has several keys anyway -- with one key per thread and the grid in several waves the plain probe is as fast)
__device__ __forceinline__ void table_probe4(const KxSlot *__restrict__ slots, uint32_t cap, uint32_t shift, const uint32_t (&key)[4],
                                             uint32_t on, int32_t (&row)[4]) {
    uint32_t slot[4], open = on & 0xfu;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        row[j] = -1;
        slot[j] = key[j] == KX_EMPTY_KEY ? cap : (kx_hash(key[j]) >> shift);
    }
    for (uint32_t step = 0; open && step < cap; step++) {
        uint2 kr[4];
#pragma unroll
        for (int j = 0; j < 4; j++)
            if ((open >> j) & 1u) kr[j] = __ldg(reinterpret_cast<const uint2 *>(&slots[slot[j]]));
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (!((open >> j) & 1u)) continue;
            if (slot[j] == cap || kr[j].x == key[j]) { row[j] = (int32_t)kr[j].y; open &= ~(1u << j); }
            else if (kr[j].x == KX_EMPTY_KEY) open &= ~(1u << j);
            else slot[j] = (slot[j] + 1) & (cap - 1);
        }
    }
}

// find or claim the slot of `key` while the table is being built (0xffffffff: table full);
// fresh_cnt as in table_fold
__device__ __forceinline__ uint32_t table_claim(const KxTableDev &tb, uint32_t key, uint32_t &fresh_cnt) {
    if (key == KX_EMPTY_KEY) return tb.cap;
    uint32_t slot = kx_hash(key) >> tb.shift;
    for (uint32_t step = 0; step < KX_MAX_PROBE; step++) {
        const uint32_t k = __ldcg(&tb.slots[slot].key);
        if (k == key) return slot;
        if (k == KX_EMPTY_KEY) {
            const uint32_t old = atomicCAS(&tb.slots[slot].key, KX_EMPTY_KEY, key);
            if (old == KX_EMPTY_KEY) { fresh_cnt++; return slot; }
            if (old == key) return slot;
        }
        slot = (slot + 1) & (tb.cap - 1);
    }
    tb.counters[KX_C_OVERFLOW] = 1u;
    return 0xffffffffu;
}

// slot of `key` in a finished table, or 0xffffffff
__device__ __forceinline__ uint32_t table_find(const KxTableDev &tb, uint32_t key) {
    if (key == KX_EMPTY_KEY) return tb.cap;
    uint32_t slot = kx_hash(key) >> tb.shift;
    for (uint32_t step = 0; step < tb.cap; step++) {
        const uint32_t k = __ldg(&tb.slots[slot].key);
        if (k == key) return slot;
        if (k == KX_EMPTY_KEY) return 0xffffffffu;
        slot = (slot + 1) & (tb.cap - 1);
    }
    return 0xffffffffu;
}

// ---- shared memory through explicit 32-bit shared-window addresses --------------------------
// The compiler re-derives the shared window base (S2R SR_CgaCtaId + LEA) at every use of a
// generic pointer into dynamic shared memory; the hot loop therefore keeps ONE base address in a
// register and goes through ld/st.shared with integer offsets.
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
// four bytes at an arbitrary shared-memory byte address
__device__ __forceinline__ uint32_t lds32_unaligned(uint32_t a) {
    const uint32_t al = a & ~3u;
    return __funnelshift_r(lds32(al), lds32(al + 4u), (a & 3u) * 8u);
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_a(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return ok != 0u;
}
// 1-D TMA bulk copy global -> shared, completion counted on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_a(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, unsigned long long pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar), "l"(pol)
                 : "memory");
}

// stage chunk g with bounded loads and zero fill (ragged tail of the text / the resolve kernel);
// returns n_rel: line starts at p < n_rel are real
__device__ __forceinline__ uint32_t stage_chunk_manual(const uint8_t *text, unsigned long long n, uint32_t g, uint32_t lane,
                                                       uint8_t *dst) {
    const unsigned long long chunk_start = (unsigned long long)g * CW;
    const unsigned long long remain = n - chunk_start;
    const uint32_t n_rel = remain < (unsigned long long)CW ? (uint32_t)remain : (uint32_t)CW + (remain > (unsigned long long)CW);
    for (int cc = (int)lane; cc < STG_BYTES / 16; cc += 32) {
        const unsigned long long q0 = chunk_start + 16ull * (unsigned)cc;
        uint4 v;
        if (q0 + 16 <= n) {
            v = *reinterpret_cast<const uint4 *>(text + q0);
        } else {
            uint8_t tmp[16];
#pragma unroll
            for (int b = 0; b < 16; b++) tmp[b] = q0 + b < n ? text[q0 + b] : (uint8_t)0;
            v = *reinterpret_cast<uint4 *>(tmp);
        }
        *reinterpret_cast<uint4 *>(dst + 16 * cc) = v;
    }
    __syncwarp();
    return n_rel;
}

// Stage one chunk (STG_BYTES from src) at shared address st with one bulk copy and wait for it: one
// copy instead of five dependent 16-byte round trips per lane.  The caller owns the mbarrier `bar`
// (initialised with count 1) and its phase parity.
__device__ __forceinline__ void stage_chunk_tma(uint32_t st, const uint8_t *src, uint32_t bar, uint32_t parity, uint32_t lane,
                                                unsigned long long pol) {
    if (lane == 0) {
        mbar_expect_tx_a(bar, STG_BYTES);
        tma_load_a(st, src, STG_BYTES, bar, pol);
    }
    while (!mbar_try_a(bar, parity)) {
    }
}

// Newline masks of the chunk staged at shared address st.  Lane owns bytes [32*lane, 32*lane+32)
// of each KiB half; the two 16-byte pieces are read in a lane-dependent order so that every
// LDS.128 phase hits all banks.  nl[h] bit b = a line starts after the newline at byte b of the
// lane's window in KiB half h, trimmed to real line starts (< n_rel).
__device__ __forceinline__ void nl_masks(uint32_t st, uint32_t lane, uint32_t n_rel, uint32_t k7f, uint32_t k0a, uint32_t k80,
                                         uint32_t (&nl)[2], uint32_t &rawnl) {
    const uint32_t swz = (lane >> 2) & 1u;
    rawnl = 0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const uint32_t o = (uint32_t)h * HALF + lane * 32u;
        const uint4 va = lds128(st + o + 16u * swz);
        const uint4 vb = lds128(st + o + 16u * (swz ^ 1u));
        const uint32_t ma = nl_mask16(va, k7f, k0a, k80), mb = nl_mask16(vb, k7f, k0a, k80);
        const uint32_t m2 = ma | (mb << 16);
        uint32_t mm = __funnelshift_l(m2, m2, swz << 4);  // swapped read order: swap the halves back
        rawnl |= mm;
        if (n_rel <= (uint32_t)CW) mm &= n_rel > o + 1u ? (n_rel - o - 1u >= 32u ? 0xffffffffu : ((1u << (n_rel - o - 1u)) - 1u)) : 0u;
        nl[h] = mm;
    }
}

// top-level line starts (first byte neither '\t' nor '#': device_plugin.go:229-236) among the line
// starts m0 / m1 of the lane's two windows (KiB halves), one loop, both loads in flight; lp0 =
// shared address of the byte after byte 0 of the first window
__device__ __forceinline__ void tops_of2(uint32_t lp0, uint32_t m0, uint32_t m1, uint32_t &t0, uint32_t &t1) {
    t0 = t1 = 0;
    while (m0 | m1) {
        const uint32_t b0 = m0 & (0u - m0), b1 = m1 & (0u - m1);
        m0 ^= b0;
        m1 ^= b1;
        // an exhausted mask reads the byte in front of the window (31 - clz(0) = -1) and ORs in nothing
        const uint32_t c0 = lds8(lp0 + (31u - (uint32_t)__clz((int)b0)));
        const uint32_t c1 = lds8(lp0 + (uint32_t)HALF + (31u - (uint32_t)__clz((int)b1)));
        if (c0 != 9u && c0 != 35u) t0 |= b0;
        if (c1 != 9u && c1 != 35u) t1 |= b1;
    }
}

// device line candidates ("\t" + non-tab, :237) among the line starts mm of one window; lp =
// shared address of the byte after the window's byte 0
__device__ __forceinline__ uint32_t devs_of(uint32_t lp, uint32_t mm) {
    uint32_t km = 0;
    while (mm) {
        const uint32_t bit = mm & (0u - mm);
        mm ^= bit;
        const uint32_t a = lp + (31u - (uint32_t)__clz((int)bit));
        if (lds8(a) == 9u && lds8(a + 1u) != 9u) km |= bit;
    }
    return km;
}

// device lines `m` (bit b: line starts at pbase + b) of the chunk staged at st, all governed by
// the alive top-level line (key_hi, anchor): parse the id, fold.  Per-lane loop: only blocks of
// a first-seen vendor id get here.
__device__ __forceinline__ void fold_lines(const KxTableDev &tab, uint32_t st, unsigned long long cbase, uint32_t m, uint32_t pbase,
                                           uint32_t key_hi, unsigned long long anchor, uint32_t &fresh_cnt) {
    while (m) {
        const uint32_t b = (uint32_t)__ffs((int)m) - 1u;
        m &= m - 1u;
        const uint32_t p = pbase + b;
        uint32_t dv;
        if (hex4_swar(lds32_unaligned(st + p + 1u), dv)) table_fold(tab, key_hi | dv, cbase + p, anchor, fresh_cnt);
    }
}

// inclusive prefix sum of v over the warp (all 32 lanes must call)
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v) {
    const uint32_t lane = threadIdx.x & 31u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= (uint32_t)d) v += y;
    }
    return v;
}

constexpr int LIST_CAP = 256;            // entries of a warp's fold list (a 2 KiB chunk of pci.ids has <= 111 device lines)
constexpr uint32_t LIST_CARRY = 0xfffu;  // governing line = the carry into the chunk
constexpr uint32_t LIST_DEAD = 0xffeu;   // no alive governing line

// Fold the device lines of the chunk staged at st (global offset cbase) that have an alive governing
// line (all 32 lanes must call).  Per lane and KiB half h: kh[h] the line starts that matter (device
// line candidates and top-level lines), th[h] the top-level lines among them, at[h] the alive ones
// among those, gov[h] the governing line in front of the window: the position of an alive top-level
// line of the chunk, LIST_CARRY (the carry: vendor carry_hi >> 16, anchor carry_anchor) or LIST_DEAD.
// Every device line to fold becomes one entry (line position | governing position << 12) of the
// warp's list (LIST_CAP words of shared memory; a chunk with more lines takes several passes), and
// the list is folded two entries per lane and round with their probe steps in flight together
// (`claim`: table_fold_claim2, for an L2-resident table) or one per lane with the load-first
// table_fold (a table in DRAM).  Folding straight from the windows left a lane's table inserts --
// two dependent L2 round trips each -- serialised: ~10 in a row for a chunk of short lines.
__device__ __forceinline__ void fold_list(const KxTableDev &tab, uint32_t *list, uint32_t st, unsigned long long cbase,
                                          const uint32_t (&kh)[2], const uint32_t (&th)[2], const uint32_t (&at)[2],
                                          const uint32_t (&gov)[2], uint32_t carry_hi, unsigned long long carry_anchor, bool claim,
                                          uint32_t &fresh_cnt) {
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t mine = 0;
    for (int h = 0; h < 2; h++) {
        // lines in front of the window's first top-level line count iff gov is alive, those behind an alive top always
        const uint32_t dl = kh[h] & ~th[h];
        const uint32_t first = th[h] & (0u - th[h]);
        const uint32_t pre = dl & (first ? first - 1u : 0xffffffffu);
        if (gov[h] != LIST_DEAD) mine += (uint32_t)__popc(pre);
        uint32_t t = th[h];
        while (t) {
            const uint32_t bit = t & (0u - t);
            t ^= bit;
            const uint32_t nxt = t & (0u - t);
            if (at[h] & bit) mine += (uint32_t)__popc(dl & ~(bit | (bit - 1u)) & (nxt ? nxt - 1u : 0xffffffffu));
        }
    }
    const uint32_t incl = warp_incl_scan(mine);
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t off = incl - mine;
    auto entry = [&](uint32_t e, uint32_t &key, unsigned long long &line, unsigned long long &anchor) -> bool {
        const uint32_t p = e & 0xfffu, gp = e >> 12;
        uint32_t key_hi = carry_hi, dv;
        anchor = carry_anchor;
        if (gp != LIST_CARRY) {
            uint32_t val;
            hex4_swar(lds32_unaligned(st + gp), val);  // an alive line: its id parsed fine before
            key_hi = val << 16;
            anchor = cbase + gp;
        }
        line = cbase + p;
        const bool ok = hex4_swar(lds32_unaligned(st + p + 1u), dv);
        key = key_hi | dv;
        return ok;
    };
    for (uint32_t base = 0; base < total; base += (uint32_t)LIST_CAP) {  // one pass unless the chunk has > LIST_CAP lines
        // my entries whose list index falls into [base, base + LIST_CAP)
        {
            uint32_t idx = off;
            for (int h = 0; h < 2; h++) {
                const uint32_t pbase = (uint32_t)h * HALF + lane * 32u + 1u;
                uint32_t g = gov[h];
                uint32_t m = kh[h];
                while (m) {
                    const uint32_t bit = m & (0u - m);
                    m ^= bit;
                    const uint32_t p = pbase + (31u - (uint32_t)__clz((int)bit));
                    if (th[h] & bit) {
                        g = (at[h] & bit) ? p : LIST_DEAD;
                    } else if (g != LIST_DEAD) {
                        if (idx >= base && idx < base + (uint32_t)LIST_CAP) list[idx - base] = p | (g << 12);
                        idx++;
                    }
                }
            }
        }
        __syncwarp();
        const uint32_t cnt = total - base < (uint32_t)LIST_CAP ? total - base : (uint32_t)LIST_CAP;
        if (claim) {
            for (uint32_t i = lane; i < cnt; i += 64u) {
                uint32_t k0, k1 = 0;
                unsigned long long l0, a0, l1 = 0, a1 = 0;
                bool v0 = entry(list[i], k0, l0, a0);
                bool v1 = i + 32u < cnt && entry(list[i + 32u], k1, l1, a1);
                if (!v0 && v1) { k0 = k1; l0 = l1; a0 = a1; v0 = true; v1 = false; }
                if (v0) table_fold_claim2(tab, k0, l0, a0, v1, k1, l1, a1, fresh_cnt);
            }
        } else {
            for (uint32_t i = lane; i < cnt; i += 32u) {
                uint32_t k;
                unsigned long long l, a;
                if (entry(list[i], k, l, a)) table_fold(tab, k, l, a, fresh_cnt);
            }
        }
        __syncwarp();
    }
}

}  // namespace kxparse

namespace kxparse {
// one atomic per warp for the keys its lanes claimed (all 32 lanes must call)
__device__ __forceinline__ void flush_fresh(const KxTableDev &tb, uint32_t &fresh_cnt) {
    const uint32_t tot = __reduce_add_sync(0xffffffffu, fresh_cnt);
    if (tot && (threadIdx.x & 31u) == 0u) atomicAdd(&tb.counters[KX_C_NKEYS], tot);
    fresh_cnt = 0;
}
}  // namespace kxparse
