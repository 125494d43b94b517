// finalize.cuh -- the kernels behind the parse: bufio.ErrTooLong cut-off, validity + name
// sanitiser (K4, device_plugin.go:241-251), batched join (K3) and name gather.
#pragma once
#include "exchange.cuh"
#include "parse_common.cuh"

namespace kxparse {

// ------------------------------------------------------------------------------
// bufio.ErrTooLong cut-off (slow path, only when the parse kernel raised the hint).
// trunc = global offset of the first line whose content is >= 65536 bytes.
// One CTA; every thread scans a contiguous byte range for newlines and reports the
// first/last newline and the longest gap inside; thread 0 stitches the ranges.
// ------------------------------------------------------------------------------
constexpr unsigned long long MAX_TOKEN = 65536ull;

__global__ void __launch_bounds__(1024) trunc_kernel(const uint8_t *__restrict__ text, unsigned long long n,
                                                      unsigned long long base, unsigned long long *trunc_out, uint32_t *counters) {
    __shared__ unsigned long long s_first[1024], s_last[1024], s_bad[1024];
    const unsigned long long per = (n + 1023ull) / 1024ull;
    const unsigned long long lo = per * threadIdx.x, hi = lo + per < n ? lo + per : n;
    unsigned long long first = KX_NO_OFF, last = KX_NO_OFF, bad = KX_NO_OFF;
    for (unsigned long long i = lo; i < hi; i++) {
        if (text[i] == (uint8_t)'\n') {
            if (first == KX_NO_OFF) first = i;
            else if (i - last - 1 >= MAX_TOKEN && bad == KX_NO_OFF) bad = last + 1;  // line (last, i)
            last = i;
        }
    }
    s_first[threadIdx.x] = first; s_last[threadIdx.x] = last; s_bad[threadIdx.x] = bad;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long prev_nl = KX_NO_OFF;  // offset of the last newline so far (none: line starts at 0)
        unsigned long long res = KX_NO_OFF;
        for (int k = 0; k < 1024 && res == KX_NO_OFF; k++) {
            if (s_first[k] != KX_NO_OFF) {
                unsigned long long start = prev_nl == KX_NO_OFF ? 0 : prev_nl + 1;
                if (s_first[k] - start >= MAX_TOKEN) { res = start; break; }
                if (s_bad[k] != KX_NO_OFF) { res = s_bad[k]; break; }
                prev_nl = s_last[k];
            }
        }
        if (res == KX_NO_OFF) {
            unsigned long long start = prev_nl == KX_NO_OFF ? 0 : prev_nl + 1;
            if (n - start >= MAX_TOKEN) res = start;  // unterminated final line
        }
        *trunc_out = res == KX_NO_OFF ? KX_NO_OFF : base + res;
        counters[KX_C_NEED_TRUNC] = 1u;  // the cut-off is there: finalize_select may proceed
    }
}

// ------------------------------------------------------------------------------
// K4 name sanitiser (device_plugin.go:241-251), warp-cooperative.
// ------------------------------------------------------------------------------
__device__ __forceinline__ bool is_re_space(uint32_t c) {  // RE2 \s
    return c == 0x20u || c == 0x09u || c == 0x0au || c == 0x0cu || c == 0x0du;
}
// length of a unicode.IsSpace rune starting at s[0] (0 = not a space); len = bytes available
__device__ __forceinline__ uint32_t uspace_len(const uint8_t *s, uint32_t len) {
    if (len == 0) return 0;
    uint32_t c = s[0];
    if (c == 0x20u || (c >= 0x09u && c <= 0x0du)) return 1;
    if (len >= 2 && c == 0xC2u && (s[1] == 0x85u || s[1] == 0xA0u)) return 2;
    if (len >= 3) {
        uint32_t d = s[1], e = s[2];
        if (c == 0xE1u && d == 0x9Au && e == 0x80u) return 3;
        if (c == 0xE2u && d == 0x80u && ((e >= 0x80u && e <= 0x8Au) || e == 0xA8u || e == 0xA9u || e == 0xAFu)) return 3;
        if (c == 0xE2u && d == 0x81u && e == 0x9Fu) return 3;
        if (c == 0xE3u && d == 0x80u && e == 0x80u) return 3;
    }
    return 0;
}
// strings.TrimSpace on buf[0..len): returns [start,end)
__device__ __forceinline__ void trim_space(const uint8_t *buf, uint32_t len, uint32_t &start, uint32_t &end) {
    uint32_t a = 0, b = len, k;
    while ((k = uspace_len(buf + a, b - a)) != 0) a += k;
    for (;;) {
        if (b > a && uspace_len(buf + b - 1, 1) == 1) { b -= 1; continue; }
        if (b - a >= 2 && uspace_len(buf + b - 2, 2) == 2) { b -= 2; continue; }
        if (b - a >= 3 && uspace_len(buf + b - 3, 3) == 3) { b -= 3; continue; }
        break;
    }
    start = a; end = b;
}
// output byte for position i of the trimmed range (0 = deleted)
__device__ __forceinline__ uint32_t sanitise_byte(const uint8_t *buf, uint32_t i, uint32_t start, uint32_t end) {
    uint32_t c = buf[i];
    if (is_re_space(c)) return (i > start && is_re_space(buf[i - 1])) ? 0u : (uint32_t)'_';
    if (c >= 'a' && c <= 'z') return c - 32u;
    if (c == '/' || c == '.') return (uint32_t)'_';
    if ((c >= 'A' && c <= 'Z') || (c >= '0' && c <= '9') || c == '_') return c;
    if (i + 1 < end) {
        if (c == 0xC4u && buf[i + 1] == 0xB1u) return (uint32_t)'I';  // U+0131 upper-cases to ASCII I
        if (c == 0xC5u && buf[i + 1] == 0xBFu) return (uint32_t)'S';  // U+017F upper-cases to ASCII S
    }
    return 0u;
}

constexpr int SF_WARPS = 8;
constexpr int SF_WIN = 128;  // bytes of a line a row group looks at (eight lanes x one aligned 16-byte load)
constexpr int SF_BATCH = 8;  // rows a warp works off per step (two rounds of four rows)

struct FinalizeParams {
    const uint8_t *text;  // shard text (local)
    unsigned long long n, base;
    KxTableDev tab;
    // validity is judged against the first anchors / cut-off of the WHOLE text: the table's own
    // (single text) or the minimum over every rank's phase-A block (sharded load, comm.cu)
    kxx::MinView mv;
    uint32_t *row_key;
    unsigned long long *row_line;
    unsigned long long *row_anchor;
    uint32_t *row_name_off;
    uint32_t *row_name_len;
    uint8_t *blob;
    uint32_t blob_cap;
    kxx::WaitSpec wait;       // sharded load: the all-reduced minima are complete when these flags are up
    kxx::SlabRow *slab_rows;  // sharded load: rows go here (this rank's slab, 32-byte records) instead of the row arrays
    uint32_t slab_rows_cap;
    uint32_t scan_w;          // table slots a warp scans per step: 8 (latency) or 32 (big tables)
    kxx::SlabTail tail;       // sharded load: header + "slab ready" flags by the last CTA
};

__device__ __forceinline__ void finalize_store_row(const FinalizeParams &F, uint32_t row, uint32_t slot, uint32_t key, unsigned long long line,
                                                   unsigned long long anchor, uint32_t name_off, uint32_t name_len) {
    F.tab.slots[slot].row = (int32_t)row;
    if (F.slab_rows) {
        if (row < F.slab_rows_cap) {
            kxx::SlabRow r;
            r.key = key; r.name_len = name_len; r.line = line; r.anchor = anchor; r.name_off = name_off; r.pad = 0u;
            F.slab_rows[row] = r;
        }
    } else {
        F.row_key[row] = key; F.row_line[row] = line; F.row_anchor[row] = anchor;
        F.row_name_off[row] = name_off; F.row_name_len[row] = name_len;
    }
}

// Validity + names in ONE kernel.  A warp scans `scan_w` consecutive table slots per step (8 for the
// small tables of pci.ids-sized vendor sets: ~8 000 warps each with a single chain of dependent loads;
// 32 for big tables, where the kernel is throughput bound) and queues the valid ones (min_anchor ==
// first anchor of the vendor, line in front of the ErrTooLong cut-off) in shared memory, prefetching
// their name windows into L2.  Queued rows are worked off SF_BATCH at a time -- full batches as long as
// the warp has slots left to scan, the remainder at the end -- four rows per round, eight lanes per
// row: one aligned 16-byte load per lane brings 128 bytes of the line, the lanes find the newline, trim
// (strings.TrimSpace), sanitise one byte per lane and step (device_plugin.go:241-251) and compact the
// result into a shared-memory staging row.  Per batch the CTA claims row handles and blob space with one
// atomic each and the warps copy the names out.  Lines whose rest does not end inside the window (19
// device lines of pci.ids) are taken by the whole warp one at a time.  KX_C_NEED_TRUNC: 0 = cut-off
// never computed, 1 = computed (trunc_kernel), 2 = asked for: when the parse raised the long-line hint
// and the cut-off is not there yet, every block leaves (the test does not depend on what block 0
// writes) and the host finalizes again.
struct SfEntry {
    unsigned long long line, anchor;
    uint32_t slot, key;
};
constexpr int SF_QCAP = SF_BATCH - 1 + 32;  // what is left of the queue + one scan

__device__ __forceinline__ void select_finalize_body(const FinalizeParams &F, const uint32_t scan_w) {
    __shared__ __align__(16) uint8_t s_raw[SF_WARPS][4][SF_WIN + 16];
    __shared__ uint8_t s_name[SF_WARPS][SF_BATCH][SF_WIN];
    __shared__ __align__(8) SfEntry s_q[SF_WARPS][SF_QCAP + 1];
    __shared__ uint32_t s_cnt[SF_WARPS], s_bytes[SF_WARPS], s_more[SF_WARPS], s_row0, s_blob0;
    if (F.tab.counters[KX_C_LONGLINE_HINT] != 0u && F.tab.counters[KX_C_NEED_TRUNC] != 1u) {
        if (blockIdx.x == 0 && threadIdx.x == 0) F.tab.counters[KX_C_NEED_TRUNC] = 2u;
        return;
    }
    const uint32_t lane = threadIdx.x & 31u, wl = threadIdx.x >> 5, sub = lane & 7u, grp = lane >> 3;
    const uint32_t nslots = F.tab.cap + 1u;
    const uint32_t nchunks = (nslots + scan_w - 1u) / scan_w;
    const uint32_t cstride = gridDim.x * (uint32_t)SF_WARPS;
    const unsigned long long trunc = kxx::min_view_trunc(F.mv);
    SfEntry *q = s_q[wl];
    uint32_t chunk = blockIdx.x * (uint32_t)SF_WARPS + wl;  // the CTA's warps take neighbouring chunks
    uint32_t qn = 0;                                        // queued rows of this warp
    // the CTA's warps step together: row handles and blob space are claimed once per CTA and step
    // (same-address atomics run at ~1 per ns: one pair per warp and step was the whole kernel time)
    for (;;) {
        while (qn < (uint32_t)SF_BATCH && chunk < nchunks) {  // scan until a full batch is queued (or nothing is left)
            const uint32_t slot = chunk * scan_w + lane;
            chunk += cstride;
            bool valid = false;
            uint32_t key = 0;
            unsigned long long line = 0, anchor = 0;
            if (lane < scan_w && slot < nslots) {
                // the slot is one 32-byte sector: both halves are asked for at once
                const uint4 head = *reinterpret_cast<const uint4 *>(&F.tab.slots[slot]);
                anchor = F.tab.slots[slot].min_anchor;
                line = ((unsigned long long)head.w << 32) | head.z;
                key = slot == F.tab.cap ? KX_EMPTY_KEY : head.x;
                valid = line != KX_NO_OFF && !(slot < F.tab.cap && key == KX_EMPTY_KEY);
                if (valid) {
                    // the name window of a candidate row: on its way into L2 while its first anchor is looked up
                    // (a candidate that loses wastes one prefetch)
                    const unsigned long long a0 = (line - F.base + 5ull) & ~15ull;
                    if (a0 < F.n) asm volatile("prefetch.global.L2 [%0];" ::"l"(F.text + a0));
                    if (a0 + 112ull < F.n && ((a0 + 112ull) >> 7) != (a0 >> 7)) asm volatile("prefetch.global.L2 [%0];" ::"l"(F.text + a0 + 112ull));
                    valid = anchor == kxx::min_view_first(F.mv, key >> 16) && line < trunc;
                }
            }
            const uint32_t vm = __ballot_sync(0xffffffffu, valid);
            if (valid) {
                SfEntry e;
                e.line = line; e.anchor = anchor; e.slot = slot; e.key = key;
                q[qn + (uint32_t)__popc(vm & ((1u << lane) - 1u))] = e;
            }
            qn += (uint32_t)__popc(vm);
            __syncwarp();
        }
        const bool have = chunk < nchunks;
        const uint32_t nvalid = qn >= (uint32_t)SF_BATCH ? (uint32_t)SF_BATCH : (have ? 0u : qn);  // rows of this batch: queue[0, nvalid)
        uint32_t my_len = 0;    // lane r (< nvalid): sanitised length of batch row r
        uint32_t slow_m = 0;    // batch rows that need the long-line path
        for (uint32_t r0 = 0; r0 < nvalid; r0 += 4u) {
            const uint32_t r = r0 + grp;  // batch row of my group
            const bool act = r < nvalid;
            const uint32_t gmask = 0xffu << (8u * grp);  // my row group: its eight lanes take every branch below together
            uint32_t total = 0, start = 0, end = 0;
            bool slow = false;
            const uint8_t *buf = s_raw[wl][grp];
            if (act) {
                const unsigned long long rs = q[r].line - F.base + 5ull;  // rest of the line after "\t" + 4 hex digits
                const unsigned long long a0 = rs & ~15ull;
                const uint32_t lead = (uint32_t)(rs - a0);
                const unsigned long long p0 = a0 + 16ull * sub;
                uint4 qd;
                if (p0 + 16ull <= F.n) {
                    qd = *reinterpret_cast<const uint4 *>(F.text + p0);
                } else {
                    uint8_t tmp[16];
#pragma unroll
                    for (int k = 0; k < 16; k++) tmp[k] = p0 + k < F.n ? F.text[p0 + k] : (uint8_t)0x0a;  // EOF terminates the last line
                    qd = *reinterpret_cast<uint4 *>(tmp);
                }
                uint8_t *raw = s_raw[wl][grp];
                *reinterpret_cast<uint4 *>(raw + 16u * sub) = qd;
                // first newline at or behind `lead`: SWAR byte-equality mask of my 16 bytes (bit k = byte k is '\n')
                uint32_t nlm = 0;
                {
                    const uint32_t w4[4] = {qd.x, qd.y, qd.z, qd.w};
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const uint32_t y = w4[k] ^ 0x0a0a0a0au;
                        const uint32_t z = ~(((y & 0x7f7f7f7fu) + 0x7f7f7f7fu) | y | 0x7f7f7f7fu);  // 0x80 where the byte is zero
                        nlm |= (((z >> 7) * 0x00204081u) >> 21 & 0xfu) << (4 * k);      // gather the four flags
                    }
                    if (sub == 0u) nlm &= 0xffffu << lead;
                }
                const uint32_t pos = nlm ? (uint32_t)__ffs((int)nlm) - 1u : 16u;
                uint32_t first = pos < 16u ? 16u * sub + pos : (uint32_t)SF_WIN;
#pragma unroll
                for (int d = 4; d > 0; d >>= 1) {
                    const uint32_t o = __shfl_xor_sync(gmask, first, d, 8);
                    first = o < first ? o : first;
                }
                __syncwarp(gmask);
                if (first >= (uint32_t)SF_WIN) {
                    slow = true;
                } else {
                    buf = raw + lead;
                    uint32_t len = first - lead;
                    if (len > 0 && buf[len - 1] == 0x0du) len--;  // bufio.ScanLines drops one trailing CR
                    if (sub == 0) trim_space(buf, len, start, end);
                    start = __shfl_sync(gmask, start, 0, 8);
                    end = __shfl_sync(gmask, end, 0, 8);
                }
            }
            // sanitise (device_plugin.go:241-251), one byte per lane and step, eight bytes per row and
            // step, all four rows of the warp in lock step; the surviving bytes are compacted with a
            // ballot into the row's staging line.  Branch free: every lane runs every step.
            {
                const uint32_t span = __reduce_max_sync(0xffffffffu, end - start);
                uint8_t *dst = s_name[wl][act ? r : 0u];
                for (uint32_t o = 0; o < span; o += 8u) {
                    const uint32_t i = start + o + sub;
                    const bool in = i < end;
                    const uint32_t c = in ? buf[i] : 0x41u;
                    const uint32_t prev = (in && i > start) ? buf[i - 1] : 0x41u;  // a space run never starts in front of the trimmed range
                    const uint32_t nx = (in && i + 1u < end) ? buf[i + 1] : 0u;
                    const bool sp = c <= 32u && ((0x100003600ull >> c) & 1ull);      // RE2 \s: [\t\n\f\r ]
                    const bool psp = prev <= 32u && ((0x100003600ull >> prev) & 1ull);
                    uint32_t ch = 0;
                    ch = (c - 0x61u < 26u) ? c - 32u : ch;                          // ToUpper
                    ch = (c - 0x41u < 26u || c - 0x30u < 10u || c == 0x5fu) ? c : ch;
                    ch = (c == 0x2fu || c == 0x2eu) ? 0x5fu : ch;                   // '/' '.' -> '_'
                    ch = sp ? (psp ? 0u : 0x5fu) : ch;                              // \s+ -> one '_'
                    ch = (c == 0xC4u && nx == 0xB1u) ? 0x49u : ch;                   // U+0131 upper-cases to ASCII I
                    ch = (c == 0xC5u && nx == 0xBFu) ? 0x53u : ch;                   // U+017F upper-cases to ASCII S
                    ch = in ? ch : 0u;
                    const uint32_t gm = (__ballot_sync(0xffffffffu, ch != 0u) >> (8u * grp)) & 0xffu;
                    if (ch) dst[total + (uint32_t)__popc(gm & ((1u << sub) - 1u))] = (uint8_t)ch;
                    total += (uint32_t)__popc(gm);
                }
            }
            // lane r0 + g learns the length of batch row r0 + g (from group g)
            const uint32_t gtot = __shfl_sync(0xffffffffu, total, (lane & 3u) * 8u);
            const uint32_t gslow = __ballot_sync(0xffffffffu, slow && sub == 0u);
            if (lane >= r0 && lane < r0 + 4u && lane < nvalid) my_len = gtot;
            for (uint32_t g = 0; g < 4u; g++)
                if ((gslow >> (8u * g)) & 1u) slow_m |= 1u << (r0 + g);
            __syncwarp();  // the next round overwrites the raw windows this round's lanes read from
        }
        __syncwarp();
        // one claim of row handles and of blob space per batch
        uint32_t len_r = (lane < nvalid && !((slow_m >> lane) & 1u)) ? my_len : 0u;
        const uint32_t incl = warp_incl_scan(len_r);
        const uint32_t wtot = __shfl_sync(0xffffffffu, incl, 31);
        if (lane == 0) { s_cnt[wl] = nvalid; s_bytes[wl] = wtot; s_more[wl] = (have || qn > nvalid) ? 1u : 0u; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t rows = 0, bytes = 0;
#pragma unroll
            for (int k = 0; k < SF_WARPS; k++) { rows += s_cnt[k]; bytes += s_bytes[k]; }
            s_row0 = rows ? atomicAdd(&F.tab.counters[KX_C_NSEL], rows) : 0u;
            uint32_t b0 = bytes ? atomicAdd(&F.tab.counters[KX_C_BLOB_CURSOR], bytes) : 0u;
            if (b0 + bytes > F.blob_cap) { F.tab.counters[KX_C_BLOB_OVERFLOW] = 1u; b0 = 0xFFFFFFFFu; }
            s_blob0 = b0;
        }
        __syncthreads();
        uint32_t row0 = s_row0, blob0 = s_blob0, more = 0;
        for (uint32_t k = 0; k < wl; k++) { row0 += s_cnt[k]; if (blob0 != 0xFFFFFFFFu) blob0 += s_bytes[k]; }
#pragma unroll
        for (int k = 0; k < SF_WARPS; k++) more |= s_more[k];
        const bool room = blob0 != 0xFFFFFFFFu;
        const uint32_t off_r = room ? blob0 + incl - len_r : 0u;
        // names out: one row at a time, 32 bytes per step
        for (uint32_t r = 0; r < nvalid; r++) {
            const uint32_t L = __shfl_sync(0xffffffffu, len_r, r), O = __shfl_sync(0xffffffffu, off_r, r);
            if (room)
                for (uint32_t j = lane; j < L; j += 32u) F.blob[O + j] = s_name[wl][r][j];
        }
        // row records: lane r writes batch row r
        if (lane < nvalid && !((slow_m >> lane) & 1u)) {
            const SfEntry e = q[lane];
            finalize_store_row(F, row0 + lane, e.slot, e.key, e.line, e.anchor, room ? off_r : 0u, room ? len_r : 0u);
        }
        // long lines (the rest does not end inside the 128-byte window; 19 device lines of pci.ids):
        // the whole warp takes them one at a time -- the line is staged into the (now free) name staging
        // area 32 bytes per step, then sanitised one byte per lane with ballot compaction
        __syncwarp();
        for (uint32_t sm = slow_m; sm; sm &= sm - 1u) {
            const uint32_t r = (uint32_t)__ffs((int)sm) - 1u;
            const unsigned long long l_line = q[r].line, l_anchor = q[r].anchor;
            const uint32_t l_key = q[r].key, l_slot = q[r].slot;
            const unsigned long long rs = l_line - F.base + 5ull;
            uint8_t *buf = &s_name[wl][0][0];
            constexpr uint32_t LONG_MAX_LEN = (uint32_t)(SF_BATCH * SF_WIN) - 32u;
            uint32_t len = 0;
            bool found = false;
            for (uint32_t o = 0; o < LONG_MAX_LEN + 32u && !found; o += 32u) {
                const unsigned long long pos = rs + o + lane;
                const uint32_t c = pos < F.n ? F.text[pos] : 0x0au;  // EOF terminates the last line
                buf[o + lane] = (uint8_t)c;
                const uint32_t nlm = __ballot_sync(0xffffffffu, c == 0x0au);
                if (nlm) { len = o + (uint32_t)__ffs((int)nlm) - 1u; found = true; }
            }
            __syncwarp();
            uint32_t start = 0, end = 0, out_len = 0, at = 0;
            bool ok = true;
            if (found) {
                if (len > 0 && buf[len - 1] == 0x0du) len--;  // bufio.ScanLines drops one trailing CR
                if (lane == 0) trim_space(buf, len, start, end);
                start = __shfl_sync(0xffffffffu, start, 0);
                end = __shfl_sync(0xffffffffu, end, 0);
                for (uint32_t o = start; o < end; o += 32u) {
                    const uint32_t i = o + lane;
                    const uint32_t ch = i < end ? sanitise_byte(buf, i, start, end) : 0u;
                    out_len += (uint32_t)__popc(__ballot_sync(0xffffffffu, ch != 0u));
                }
                if (lane == 0) {
                    at = out_len ? atomicAdd(&F.tab.counters[KX_C_BLOB_CURSOR], out_len) : 0u;
                    if (at + out_len > F.blob_cap) { F.tab.counters[KX_C_BLOB_OVERFLOW] = 1u; at = 0xFFFFFFFFu; }
                }
                at = __shfl_sync(0xffffffffu, at, 0);
                ok = at != 0xFFFFFFFFu;
                if (ok) {
                    uint32_t wr = at;
                    for (uint32_t o = start; o < end; o += 32u) {
                        const uint32_t i = o + lane;
                        const uint32_t ch = i < end ? sanitise_byte(buf, i, start, end) : 0u;
                        const uint32_t bm = __ballot_sync(0xffffffffu, ch != 0u);
                        if (ch) F.blob[wr + (uint32_t)__popc(bm & ((1u << lane) - 1u))] = (uint8_t)ch;
                        wr += (uint32_t)__popc(bm);
                    }
                }
            } else if (lane == 0) {
                // longer than the staging area (never in pci.ids): lane 0, serial, straight from global memory
                const uint8_t *g = F.text + rs;
                const unsigned long long avail = F.n - rs;
                unsigned long long l = 0;
                while (l < avail && g[l] != 0x0au) l++;
                len = (uint32_t)l;
                if (len > 0 && g[len - 1] == 0x0du) len--;
                trim_space(g, len, start, end);
                for (uint32_t i = start; i < end; i++) out_len += sanitise_byte(g, i, start, end) != 0u;
                at = out_len ? atomicAdd(&F.tab.counters[KX_C_BLOB_CURSOR], out_len) : 0u;
                if (at + out_len > F.blob_cap) { F.tab.counters[KX_C_BLOB_OVERFLOW] = 1u; ok = false; }
                if (ok) {
                    uint32_t wr = at;
                    for (uint32_t i = start; i < end; i++) {
                        const uint32_t ch = sanitise_byte(g, i, start, end);
                        if (ch) F.blob[wr++] = (uint8_t)ch;
                    }
                }
            }
            if (lane == 0) finalize_store_row(F, row0 + r, l_slot, l_key, l_line, l_anchor, ok ? at : 0u, ok ? out_len : 0u);
            __syncwarp();
        }
        // what is left of the queue moves to its front
        {
            const uint32_t rem = qn - nvalid;
            if (nvalid != 0u && rem != 0u) {
                SfEntry e;
                if (lane < rem) e = q[nvalid + lane];
                __syncwarp();
                if (lane < rem) q[lane] = e;
                __syncwarp();
            }
            qn = rem;
        }
        __syncthreads();  // the staging rows and the claim words are reused by the next step
        if (!more) break;
    }
}

__global__ void __launch_bounds__(SF_WARPS * 32, 8) select_finalize_kernel(const FinalizeParams F) {
    kxx::wait_flags_cta(F.wait);
    select_finalize_body(F, F.scan_w);
    if (F.tail.on) {
        // one fence per CTA: the barrier makes the CTA's rows visible to thread 0, whose (cumulative) fence orders them
        // in front of the counter and, in the last CTA, of the header and the flags
        __syncthreads();
        if (threadIdx.x == 0) {
            kx_fence_sys();
            const uint32_t prev = atomicAdd(F.tail.done, 1u);
            if (prev == gridDim.x - 1u) {
                *F.tail.done = 0u;
                kx_fence_gpu();
                const volatile uint32_t *c = F.tab.counters;
                const uint32_t n_sel = c[KX_C_NSEL], blob_used = c[KX_C_BLOB_CURSOR];
                const bool over = c[KX_C_BLOB_OVERFLOW] || n_sel > F.tail.rows_cap || blob_used > F.tail.blob_cap;
                kxx::SlabHeader h;
                memset(&h, 0, sizeof h);
                h.n_rows = over ? 0u : n_sel;
                h.blob_bytes = over ? 0u : blob_used;
                h.status = over ? kxx::XS_SLAB_OVERFLOW : 0u;
                // phase A left before the resolve pass: what that pass found out about the table travels here
                if (c[KX_C_OVERFLOW]) h.status |= kxx::XS_GROW | kxx::XS_FULL;
                if (c[KX_C_NKEYS] > F.tab.max_keys) h.status |= kxx::XS_GROW;
                h.nkeys = c[KX_C_NKEYS];
                *F.tail.header = h;
                kx_fence_sys();
                for (int k = 0; k < F.tail.tg.n; k++) *reinterpret_cast<volatile uint32_t *>(F.tail.tg.region[k] + F.tail.o_flag) = F.tail.epoch;
            }
        }
    }
}

// ------------------------------------------------------------------------------
// K3 batched join: one thread per key, probe the table (L2 resident; key and row handle share
// one 32-byte sector), return the row handle.
// ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lookup_kernel(const uint32_t *__restrict__ keys, size_t n, const KxSlot *__restrict__ slots,
                                                      uint32_t cap, uint32_t shift, int32_t *__restrict__ rows_out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) rows_out[i] = table_probe(slots, cap, shift, keys[i]);
}

// name gather: lengths, then copy
__global__ void __launch_bounds__(256) name_len_kernel(const int32_t *__restrict__ rows, size_t n,
                                                        const uint32_t *__restrict__ row_name_len, uint32_t n_rows,
                                                        uint32_t *__restrict__ lens) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        int32_t r = rows[i];
        lens[i] = (r >= 0 && (uint32_t)r < n_rows) ? row_name_len[r] : 0u;
    }
}
// 8 lanes per name
__global__ void __launch_bounds__(256) name_copy_kernel(const int32_t *__restrict__ rows, size_t n,
                                                         const uint32_t *__restrict__ row_name_off,
                                                         const uint32_t *__restrict__ row_name_len, uint32_t n_rows,
                                                         const uint8_t *__restrict__ blob,
                                                         const uint32_t *__restrict__ offsets, uint8_t *__restrict__ out,
                                                         size_t cap) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    uint32_t sub = threadIdx.x & 7u;
    if (i >= n) return;
    int32_t r = rows[i];
    if (r < 0 || (uint32_t)r >= n_rows) return;
    uint32_t len = row_name_len[r], src = row_name_off[r], dst = offsets[i];
    if ((size_t)dst + len > cap) return;
    for (uint32_t k = sub; k < len; k += 8u) out[dst + k] = blob[src + k];
}

// [slots | vendor_first | trunc] <- 0xff, counters <- 0: one launch per table arena (api.cu)
__global__ void __launch_bounds__(256) arena_reset_kernel(uint4 *ff, size_t n_ff16, uint32_t *counters) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = i; k < n_ff16; k += stride) ff[k] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    if (i < KX_C_COUNT) counters[i] = 0u;
}

}  // namespace kxparse
