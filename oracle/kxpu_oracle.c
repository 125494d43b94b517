/*
 * kxpu_oracle.c -- CPU restatement (plain C) of the reference's discovery hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg
 * may load this library, and only as the checker / the timed CPU baseline.
 *
 * PARITY UNPINNED: the reference (Apokleos/kata-xpu-device-plugin @ 482ee26) ships no
 * tests, golden files or fixtures, is written in Go, and no Go toolchain exists in this
 * image, so this restatement cannot be checked against reference outputs.  It follows
 * the reference line by line (citations below, paths relative to the reference root)
 * and the published behaviour of the Go packages it calls:
 *   bufio.Scanner / ScanLines   (go1.22 stdlib)      -- line splitting, 64 KiB token cap
 *   strings.TrimSpace/ToUpper   (go1.22 stdlib)      -- name sanitiser
 *   regexp (RE2) \s             (go1.22 stdlib)      -- [\t\n\f\r ]
 *   gopkg.in/yaml.v3 v3.0.1     (go.mod:78)          -- YAML emit
 *   encoding/json MarshalIndent (go1.22 stdlib)      -- JSON emit
 *   tags.cncf.io/container-device-interface v0.8.0 pkg/parser.QualifiedName (go.mod:13)
 * It is pinned against (a) the self-derived hashes recorded in SURVEY.md 8(c) and
 * (b) independent Python restatements (tests/test_oracle.py).
 */
#define _GNU_SOURCE
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "../include/kxpu.h"

#define KXO_MAX_TOKEN 65536 /* bufio.MaxScanTokenSize = 64*1024 */

/* ------------------------------------------------------------------------- */
/* bufio.Scanner with ScanLines over an in-memory file.                       */
/* Follows: device_plugin.go:262 (bufio.NewScanner), :263/:226 (Scan loop).   */
/* Returns 1 and the line [*ls,*le) (trailing '\r' dropped, '\n' excluded),   */
/* 0 at EOF, -1 on bufio.ErrTooLong.  *pos advances past the line.            */
/* ------------------------------------------------------------------------- */
static int kxo_next_line(const uint8_t *text, size_t n, size_t *pos, size_t *ls, size_t *le) {
    size_t p = *pos;
    if (p >= n) return 0;
    const uint8_t *nl = (const uint8_t *)memchr(text + p, '\n', n - p);
    size_t end = nl ? (size_t)(nl - text) : n;
    if (end - p >= KXO_MAX_TOKEN) return -1; /* buffer fills with no newline in it */
    *ls = p;
    *le = (end > p && text[end - 1] == '\r') ? end - 1 : end; /* dropCR */
    *pos = nl ? end + 1 : n;
    return 1;
}

static int has_prefix(const uint8_t *s, size_t len, const uint8_t *pre, size_t plen) {
    return len >= plen && memcmp(s, pre, plen) == 0;
}

/*
 * getDeviceName + locateVendor, literally (device_plugin.go:208-275), generalised from
 * the constant nvidiaVendorID to a per-call vendor string (locateVendor already takes
 * one, :261).  vendor/device are raw strings as read from sysfs.
 * Returns the offset of the matching device line, or -1 ("" in the reference).
 * rest_off/rest_len = line with the "\t"+deviceID prefix removed (input of the
 * sanitiser, :241).  *scanned accumulates the bytes the scanner consumed.
 */
int64_t kxo_scan_lookup(const uint8_t *text, size_t n, const uint8_t *vendor, size_t vlen,
                        const uint8_t *device, size_t dlen, size_t *rest_off, size_t *rest_len,
                        uint64_t *scanned) {
    size_t pos = 0, ls, le;
    int r, found = 0;
    /* locateVendor :263-268 */
    while ((r = kxo_next_line(text, n, &pos, &ls, &le)) == 1) {
        if (has_prefix(text + ls, le - ls, vendor, vlen)) { found = 1; break; }
    }
    if (!found) { if (scanned) *scanned += pos; return -1; } /* :219-222 */
    uint8_t prefix[64];
    if (dlen + 1 > sizeof prefix) return -1;
    prefix[0] = '\t';
    memcpy(prefix + 1, device, dlen); /* :225 */
    int64_t hit = -1;
    while ((r = kxo_next_line(text, n, &pos, &ls, &le)) == 1) { /* :226 */
        size_t len = le - ls;
        if (len >= 1 && text[ls] == '#') continue;           /* :229 */
        if (!(len >= 1 && text[ls] == '\t')) break;           /* :233 -> "" */
        if (!has_prefix(text + ls, len, prefix, dlen + 1)) continue; /* :237 */
        hit = (int64_t)ls;
        if (rest_off) *rest_off = ls + dlen + 1;              /* :241 TrimPrefix */
        if (rest_len) *rest_len = len - (dlen + 1);
        break;
    }
    if (scanned) *scanned += pos;
    return hit;
}

/* ------------------------------------------------------------------------- */
/* Name sanitiser, device_plugin.go:242-251.                                  */
/* ------------------------------------------------------------------------- */

/* unicode.IsSpace code points as UTF-8, for strings.TrimSpace (:242). */
static size_t space_at_start(const uint8_t *s, size_t len) {
    if (len == 0) return 0;
    uint8_t c = s[0];
    if (c == ' ' || (c >= 0x09 && c <= 0x0d)) return 1;
    if (len >= 2 && c == 0xC2 && (s[1] == 0x85 || s[1] == 0xA0)) return 2;
    if (len >= 3) {
        if (c == 0xE1 && s[1] == 0x9A && s[2] == 0x80) return 3;                 /* U+1680 */
        if (c == 0xE2 && s[1] == 0x80 &&
            ((s[2] >= 0x80 && s[2] <= 0x8A) || s[2] == 0xA8 || s[2] == 0xA9 || s[2] == 0xAF))
            return 3;                                             /* U+2000-200A,2028,2029,202F */
        if (c == 0xE2 && s[1] == 0x81 && s[2] == 0x9F) return 3;                 /* U+205F */
        if (c == 0xE3 && s[1] == 0x80 && s[2] == 0x80) return 3;                 /* U+3000 */
    }
    return 0;
}
static size_t space_at_end(const uint8_t *s, size_t len) {
    if (len == 0) return 0;
    uint8_t c = s[len - 1];
    if (c == ' ' || (c >= 0x09 && c <= 0x0d)) return 1;
    if (len >= 2 && space_at_start(s + len - 2, 2) == 2) return 2;
    if (len >= 3 && space_at_start(s + len - 3, 3) == 3) return 3;
    return 0;
}

/*
 * out must hold len bytes (the result never grows).  Byte-level statement of:
 *   TrimSpace -> ToUpper -> '/'->'_' -> '.'->'_' -> \s+ -> "_" -> delete [^a-zA-Z0-9_.]+
 * After these steps only [A-Z0-9_] survive.  Non-ASCII runes are all deleted by the last
 * step except the two whose simple upper-case mapping is ASCII: U+0131 (C4 B1) -> 'I'
 * and U+017F (C5 BF) -> 'S' (unicode.ToUpper).  RE2 \s is [\t\n\f\r ]; \v is deleted.
 */
size_t kxo_sanitise(const uint8_t *s, size_t len, uint8_t *out) {
    size_t k;
    while ((k = space_at_start(s, len)) != 0) { s += k; len -= k; }
    while ((k = space_at_end(s, len)) != 0) len -= k;
    size_t o = 0;
    int in_ws = 0;
    for (size_t i = 0; i < len; i++) {
        uint8_t c = s[i];
        if (c == '\t' || c == '\n' || c == '\f' || c == '\r' || c == ' ') {
            if (!in_ws) out[o++] = '_';
            in_ws = 1;
            continue;
        }
        in_ws = 0;
        if (c >= 'a' && c <= 'z') c = (uint8_t)(c - 32);
        if (c == '/' || c == '.') c = '_';
        if ((c >= 'A' && c <= 'Z') || (c >= '0' && c <= '9') || c == '_') { out[o++] = c; continue; }
        if (c == 0xC4 && i + 1 < len && s[i + 1] == 0xB1) { out[o++] = 'I'; i++; continue; }
        if (c == 0xC5 && i + 1 < len && s[i + 1] == 0xBF) { out[o++] = 'S'; i++; continue; }
        /* everything else is deleted */
    }
    return o;
}

static void hex4(uint32_t v, uint8_t out[4]) {
    static const char d[] = "0123456789abcdef";
    out[0] = d[(v >> 12) & 15]; out[1] = d[(v >> 8) & 15]; out[2] = d[(v >> 4) & 15]; out[3] = d[v & 15];
}

/* getDeviceName for key = (vendor<<16)|device; returns name length or -1 on miss. */
int64_t kxo_device_name(const uint8_t *text, size_t n, uint32_t key, uint8_t *out, size_t cap,
                        int64_t *line_off, uint64_t *scanned) {
    uint8_t v[4], d[4];
    hex4(key >> 16, v); hex4(key & 0xffff, d);
    size_t ro = 0, rl = 0;
    int64_t hit = kxo_scan_lookup(text, n, v, 4, d, 4, &ro, &rl, scanned);
    if (line_off) *line_off = hit;
    if (hit < 0) return -1;
    uint8_t *tmp = (uint8_t *)malloc(rl + 1);
    size_t m = kxo_sanitise(text + ro, rl, tmp);
    if (m > cap) m = cap;
    memcpy(out, tmp, m);
    free(tmp);
    return (int64_t)m;
}

/* ------------------------------------------------------------------------- */
/* Single-pass table build: an independent statement of "what every possible  */
/* getDeviceName call would return", used to cross-check the literal scan and  */
/* as the "best honest CPU" baseline.  Rows come out in file order.            */
/* ------------------------------------------------------------------------- */
typedef struct kxo_row { uint32_t key; uint64_t line_off; uint64_t anchor_off; } kxo_row;

static int is_lhex(uint8_t c) { return (c >= '0' && c <= '9') || (c >= 'a' && c <= 'f'); }
static int hexval(uint8_t c) { return c <= '9' ? c - '0' : c - 'a' + 10; }
static int parse_hex4(const uint8_t *s, size_t len, uint32_t *v) {
    if (len < 4) return 0;
    uint32_t x = 0;
    for (int i = 0; i < 4; i++) { if (!is_lhex(s[i])) return 0; x = x * 16 + (uint32_t)hexval(s[i]); }
    *v = x;
    return 1;
}

/* returns number of rows; rows written up to cap. */
size_t kxo_table_build(const uint8_t *text, size_t n, kxo_row *rows, size_t cap) {
    /* vendor_seen[v]: an anchor for v already occurred (only the first counts, :265) */
    uint8_t *vendor_seen = (uint8_t *)calloc(65536, 1);
    uint8_t *dev_seen = (uint8_t *)calloc(65536 / 8, 1); /* devices seen in the current block */
    size_t pos = 0, ls, le, nrows = 0;
    int cur_valid = 0; /* current block belongs to the first anchor of cur_v */
    uint32_t cur_v = 0;
    uint64_t cur_anchor = 0;
    while (kxo_next_line(text, n, &pos, &ls, &le) == 1) {
        size_t len = le - ls;
        const uint8_t *l = text + ls;
        if (len >= 1 && l[0] == '#') continue;
        if (len >= 1 && l[0] == '\t') {
            uint32_t d;
            if (cur_valid && parse_hex4(l + 1, len - 1, &d) && !(dev_seen[d >> 3] & (1u << (d & 7)))) {
                dev_seen[d >> 3] |= (uint8_t)(1u << (d & 7));
                if (nrows < cap) { rows[nrows].key = (cur_v << 16) | d; rows[nrows].line_off = ls; rows[nrows].anchor_off = cur_anchor; }
                nrows++;
            }
            continue;
        }
        /* top-level line: ends any block; may start a new one */
        cur_valid = 0;
        uint32_t v;
        if (parse_hex4(l, len, &v) && !vendor_seen[v]) {
            vendor_seen[v] = 1;
            cur_valid = 1; cur_v = v; cur_anchor = ls;
            memset(dev_seen, 0, 65536 / 8);
        }
    }
    free(vendor_seen); free(dev_seen);
    return nrows;
}

/* Rest-of-line (after "\t"+4 hex) of the line at line_off, as the scanner would return it. */
size_t kxo_line_rest(const uint8_t *text, size_t n, uint64_t line_off, size_t *rest_off) {
    size_t pos = (size_t)line_off, ls, le;
    if (kxo_next_line(text, n, &pos, &ls, &le) != 1 || le - ls < 5) { *rest_off = 0; return 0; }
    *rest_off = ls + 5;
    return le - ls - 5;
}

/* ------------------------------------------------------------------------- */
/* createIommuDeviceMap (device_plugin.go:126-180) over a flat record table,   */
/* + device-list build of createDevicePlugins (:91-98).                        */
/* ------------------------------------------------------------------------- */

/* readIDFromFileFunc :183-191: data[2:] with all leading/trailing '\n' trimmed.
 * Returns length (<= 8) or -1 for "would panic" (file < 2 bytes) / unsupported. */
static int kxo_read_id(const uint8_t *txt, unsigned flen, uint8_t id[8]) {
    memset(id, 0, 8);
    if (flen < 2 || flen > 8) return -1;
    const uint8_t *s = txt + 2;
    int len = (int)flen - 2;
    while (len > 0 && s[0] == '\n') { s++; len--; }
    while (len > 0 && s[len - 1] == '\n') len--;
    memcpy(id, s, (size_t)len);
    return len;
}

typedef struct { uint64_t *keys; uint32_t *vals; size_t cap; } kxo_map;
static void map_init(kxo_map *m, size_t n) {
    size_t c = 16; while (c < 2 * n + 2) c <<= 1;
    m->cap = c; m->keys = (uint64_t *)malloc(c * 8); m->vals = (uint32_t *)malloc(c * 4);
    memset(m->keys, 0xff, c * 8);
}
static void map_free(kxo_map *m) { free(m->keys); free(m->vals); }
static uint32_t *map_get(kxo_map *m, uint64_t k, int *fresh) {
    uint64_t h = k * 0x9E3779B97F4A7C15ull;
    size_t i = (size_t)(h >> 20) & (m->cap - 1);
    for (;;) {
        if (m->keys[i] == k) { *fresh = 0; return &m->vals[i]; }
        if (m->keys[i] == ~0ull) { m->keys[i] = k; *fresh = 1; return &m->vals[i]; }
        i = (i + 1) & (m->cap - 1);
    }
}

#define KXO_UNSEEN 0xFFFFFFFEu
int32_t kxo_classify(const kxpu_devrec *recs, size_t n, kxpu_classify_out *out) {
    kxo_map gmap, dmap;
    map_init(&gmap, n); map_init(&dmap, n);
    uint32_t *gcount = (uint32_t *)calloc(n + 1, 4);   /* members per group ordinal */
    uint32_t *gord = (uint32_t *)malloc((n + 1) * 4);  /* group ordinal of accepted record */
    uint32_t *dcount = (uint32_t *)calloc(n + 1, 4);
    uint32_t *g_dev = (uint32_t *)malloc((n + 1) * 4); /* devid ordinal of group ordinal, or ~0 */
    uint32_t bus_index = 0, n_groups = 0, n_devids = 0; /* :130 */
    for (size_t i = 0; i < n; i++) {
        const kxpu_devrec *r = &recs[i];
        out->accept_index[i] = KXPU_REJECTED;
        if (r->flags & KXPU_REC_IS_DIR) continue;                    /* :137 */
        if (r->flags & KXPU_REC_VENDOR_ERR) continue;                /* :143 */
        uint8_t id[8];
        int l = kxo_read_id(r->vendor_txt, r->vendor_len, id);
        if (!(l == 4 && memcmp(id, "10de", 4) == 0)) continue;       /* :149 */
        if (r->flags & KXPU_REC_DRIVER_ERR) continue;                /* :152 */
        if (strncmp(r->driver, "vfio-pci", 16) != 0) continue;       /* :156 */
        if (r->flags & KXPU_REC_IOMMU_ERR) continue;                 /* :158 */
        int fresh;
        uint32_t *g = map_get(&gmap, r->iommu_group, &fresh);        /* :162 */
        if (fresh) *g = KXO_UNSEEN;
        if (*g == KXO_UNSEEN) {
            /* iommuMap[group] is only created at :171, so when the device read fails
             * (:165-168) the record is skipped and the group stays unseen. */
            int dl = (r->flags & KXPU_REC_DEVICE_ERR) ? -1 : kxo_read_id(r->device_txt, r->device_len, id);
            if (dl < 0) continue;
            *g = n_groups;
            uint64_t dk = 0; memcpy(&dk, id, 8);
            int dfresh;
            uint32_t *d = map_get(&dmap, dk, &dfresh);
            if (dfresh) { *d = n_devids; out->dev_ids[n_devids] = dk; n_devids++; }
            g_dev[n_groups] = *d;
            dcount[*d]++;                                            /* :169 */
            out->group_ids[n_groups] = r->iommu_group;
            n_groups++;
        }
        gord[bus_index] = *g;
        gcount[*g]++;
        out->accept_index[i] = bus_index++;                          /* :171-175 */
    }
    /* CSR fill */
    out->group_off[0] = 0;
    for (uint32_t g = 0; g < n_groups; g++) out->group_off[g + 1] = out->group_off[g] + gcount[g];
    out->dev_off[0] = 0;
    for (uint32_t d = 0; d < n_devids; d++) out->dev_off[d + 1] = out->dev_off[d] + dcount[d];
    uint32_t *gfill = (uint32_t *)calloc(n_groups + 1, 4), *dfill = (uint32_t *)calloc(n_devids + 1, 4);
    for (size_t i = 0; i < n; i++) {
        uint32_t b = out->accept_index[i];
        if (b == KXPU_REJECTED) continue;
        uint32_t g = gord[b];
        out->group_members[out->group_off[g] + gfill[g]++] = (uint32_t)i;
    }
    for (uint32_t g = 0; g < n_groups; g++) {
        uint32_t d = g_dev[g];
        out->dev_groups[out->dev_off[d] + dfill[d]++] = out->group_ids[g];
    }
    out->n_accepted = bus_index; out->n_groups = n_groups; out->n_devids = n_devids;
    free(gfill); free(dfill); free(gcount); free(gord); free(dcount); free(g_dev);
    map_free(&gmap); map_free(&dmap);
    return 0;
}

/* ------------------------------------------------------------------------- */
/* CDI spec emit: generateCDISpec (device_plugin.go:55-80) + Save              */
/* (cdi/spec.go:85-127), canonical device order = array order.                 */
/* ------------------------------------------------------------------------- */
typedef struct { uint8_t *p; size_t cap, len; } kxo_buf;
static void put(kxo_buf *b, const void *s, size_t n) {
    if (b->p && b->len + n <= b->cap) memcpy(b->p + b->len, s, n);
    b->len += n;
}
static void puts_(kxo_buf *b, const char *s) { put(b, s, strlen(s)); }
static void putu(kxo_buf *b, uint64_t v) { char t[24]; int k = snprintf(t, sizeof t, "%llu", (unsigned long long)v); put(b, t, (size_t)k); }

/* yaml.v3 isBase60Float (resolve.go): ^[-+]?[0-9][0-9_]*(?::[0-5]?[0-9])+(?:\.[0-9_]*)?$
 * A plain string that matches must be double-quoted (encode.go stringv). */
int kxo_is_base60(const uint8_t *s, size_t len) {
    size_t i = 0;
    if (i < len && (s[i] == '-' || s[i] == '+')) i++;
    if (!(i < len && s[i] >= '0' && s[i] <= '9')) return 0;
    i++;
    while (i < len && ((s[i] >= '0' && s[i] <= '9') || s[i] == '_')) i++;
    /* (?::[0-5]?[0-9])+ -- one or two digits after each ':'; two only if the first is 0-5 */
    int groups = 0;
    while (i < len && s[i] == ':') {
        size_t j = i + 1;
        if (!(j < len && s[j] >= '0' && s[j] <= '9')) break;
        if (j + 1 < len && s[j + 1] >= '0' && s[j + 1] <= '9') {
            if (s[j] <= '5') j += 2; else j += 1; /* greedy [0-5]?[0-9]; backtracking cannot
                                                     help: the next char must be ':' '.' or end */
        } else j += 1;
        i = j; groups++;
    }
    if (!groups) return 0;
    if (i < len && s[i] == '.') { i++; while (i < len && ((s[i] >= '0' && s[i] <= '9') || s[i] == '_')) i++; }
    return i == len;
}

static size_t bdf_len(const char *bdf) { size_t l = 0; while (l < 16 && bdf[l]) l++; return l; }

size_t kxo_cdi_emit(int32_t format, const kxpu_cdidev *devs, size_t n, uint8_t *out, size_t cap) {
    kxo_buf b = { out, cap, 0 };
    if (format == KXPU_FMT_YAML) {
        /* yaml.v3: struct fields in order; top-level annotations (empty map) and
         * containerEdits (zero struct) dropped by omitempty; sequences indented. */
        puts_(&b, "cdiVersion: 0.6.0\nkind: nvidia.com/gpu\n");          /* spec.go:12-13,18-19 */
        if (n == 0) { puts_(&b, "devices: []\n"); return b.len; }          /* Devices nil -> [] */
        puts_(&b, "devices:\n");
        for (size_t i = 0; i < n; i++) {
            const kxpu_cdidev *d = &devs[i];
            size_t bl = bdf_len(d->bdf);
            puts_(&b, "  - name: \""); putu(&b, d->index); puts_(&b, "\"\n");  /* :75, int-like => quoted */
            puts_(&b, "    annotations:\n      attach-pci: \"true\"\n      bdf: "); /* :63,:68, sorted keys */
            if (kxo_is_base60((const uint8_t *)d->bdf, bl)) { puts_(&b, "\""); put(&b, d->bdf, bl); puts_(&b, "\""); }
            else put(&b, d->bdf, bl);
            puts_(&b, "\n      cdi.k8s.io/vfio"); putu(&b, d->iommu_group);   /* :65 */
            puts_(&b, ": nvidia.com/gpu="); putu(&b, d->index);              /* :66 */
            puts_(&b, "\n    containerEdits:\n      deviceNodes:\n        - path: /dev/vfio/"); /* :71-73 */
            putu(&b, d->iommu_group); puts_(&b, "\n");
        }
        return b.len;
    }
    /* encoding/json MarshalIndent(spec, "", "  "), no trailing newline (spec.go:115-120) */
    puts_(&b, "{\n  \"cdiVersion\": \"0.6.0\",\n  \"kind\": \"nvidia.com/gpu\",\n");
    if (n == 0) { puts_(&b, "  \"devices\": null,\n  \"containerEdits\": {}\n}"); return b.len; }
    puts_(&b, "  \"devices\": [\n");
    for (size_t i = 0; i < n; i++) {
        const kxpu_cdidev *d = &devs[i];
        size_t bl = bdf_len(d->bdf);
        puts_(&b, "    {\n      \"name\": \""); putu(&b, d->index);
        puts_(&b, "\",\n      \"annotations\": {\n        \"attach-pci\": \"true\",\n        \"bdf\": \"");
        put(&b, d->bdf, bl);
        puts_(&b, "\",\n        \"cdi.k8s.io/vfio"); putu(&b, d->iommu_group);
        puts_(&b, "\": \"nvidia.com/gpu="); putu(&b, d->index);
        puts_(&b, "\"\n      },\n      \"containerEdits\": {\n        \"deviceNodes\": [\n          {\n            \"path\": \"/dev/vfio/");
        putu(&b, d->iommu_group);
        puts_(&b, "\"\n          }\n        ]\n      }\n    }");
        puts_(&b, i + 1 < n ? ",\n" : "\n");
    }
    puts_(&b, "  ],\n  \"containerEdits\": {}\n}");
    return b.len;
}

/* updateResponseForCDI / QualifiedName (generic_device_plugin.go:274-299; cdi-utils.go:9) */
size_t kxo_alloc_names(const uint64_t *idx, size_t n, uint8_t *out, size_t cap, uint32_t *offsets) {
    kxo_buf b = { out, cap, 0 };
    for (size_t i = 0; i < n; i++) {
        offsets[i] = (uint32_t)b.len;
        puts_(&b, "nvidia.com/gpu="); putu(&b, idx[i]);
    }
    offsets[n] = (uint32_t)b.len;
    return b.len;
}

/* ListAndWatchResponse{Devices} protobuf wire form (generic_device_plugin.go:224;
 * k8s.io/kubelet v0.30.2 deviceplugin/v1beta1 api.proto: Device{ID=1, health=2}). */
size_t kxo_lw_encode(const uint32_t *group_ids, const uint8_t *healthy, size_t n, uint8_t *out, size_t cap) {
    kxo_buf b = { out, cap, 0 };
    for (size_t i = 0; i < n; i++) {
        char id[16];
        int il = snprintf(id, sizeof id, "%u", group_ids[i]);
        const char *h = (!healthy || healthy[i]) ? "Healthy" : "Unhealthy";
        size_t hl = strlen(h);
        uint8_t hdr[2] = { 0x0a, (uint8_t)(2 + il + 2 + hl) };
        put(&b, hdr, 2);
        uint8_t f1[2] = { 0x0a, (uint8_t)il }; put(&b, f1, 2); put(&b, id, (size_t)il);
        uint8_t f2[2] = { 0x12, (uint8_t)hl }; put(&b, f2, 2); put(&b, h, hl);
    }
    return b.len;
}

/* ------------------------------------------------------------------------- */
/* CPU baseline timing (bench.py cpu_baseline / --impl reference).             */
/* ------------------------------------------------------------------------- */
static double now_s(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }

typedef struct {
    const uint8_t *text; size_t n; const uint32_t *keys; size_t lo, hi;
    int64_t *line_off; uint64_t scanned; uint64_t name_bytes;
} kxo_job;

static void *scan_worker(void *arg) {
    kxo_job *j = (kxo_job *)arg;
    uint8_t name[512];
    for (size_t i = j->lo; i < j->hi; i++) {
        int64_t off;
        int64_t l = kxo_device_name(j->text, j->n, j->keys[i], name, sizeof name, &off, &j->scanned);
        if (j->line_off) j->line_off[i] = off;
        if (l > 0) j->name_bytes += (uint64_t)l;
    }
    return NULL;
}

/* The reference algorithm (one full getDeviceName per key), keys split over `threads`
 * host threads.  Returns elapsed seconds; *scanned = text bytes consumed by all scans. */
double kxo_bench_scan(const uint8_t *text, size_t n, const uint32_t *keys, size_t nkeys, int threads,
                      int64_t *line_off, uint64_t *scanned) {
    if (threads < 1) threads = 1;
    if ((size_t)threads > nkeys && nkeys > 0) threads = (int)nkeys;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    kxo_job *jobs = (kxo_job *)calloc((size_t)threads, sizeof(kxo_job));
    double t0 = now_s();
    for (int t = 0; t < threads; t++) {
        jobs[t].text = text; jobs[t].n = n; jobs[t].keys = keys; jobs[t].line_off = line_off;
        jobs[t].lo = nkeys * (size_t)t / (size_t)threads; jobs[t].hi = nkeys * (size_t)(t + 1) / (size_t)threads;
        pthread_create(&th[t], NULL, scan_worker, &jobs[t]);
    }
    uint64_t total = 0;
    for (int t = 0; t < threads; t++) { pthread_join(th[t], NULL); total += jobs[t].scanned; }
    double dt = now_s() - t0;
    if (scanned) *scanned = total;
    free(th); free(jobs);
    return dt;
}

/* "Best honest CPU": one pass builds a table (kxo_table_build), then keys are probed by
 * binary search over rows sorted by key.  Single pass is sequential by nature (carried
 * vendor state); reported beside the literal scan so the GPU is not flattered. */
static int row_cmp(const void *a, const void *b) {
    uint32_t x = ((const kxo_row *)a)->key, y = ((const kxo_row *)b)->key;
    return x < y ? -1 : x > y;
}
double kxo_bench_parse_once(const uint8_t *text, size_t n, const uint32_t *keys, size_t nkeys,
                            int64_t *line_off, double *parse_s) {
    double t0 = now_s();
    size_t cap = 1u << 16, nr;
    kxo_row *rows = (kxo_row *)malloc(cap * sizeof(kxo_row));
    nr = kxo_table_build(text, n, rows, cap);
    if (nr > cap) { cap = nr; rows = (kxo_row *)realloc(rows, cap * sizeof(kxo_row)); nr = kxo_table_build(text, n, rows, cap); }
    double t1 = now_s();
    qsort(rows, nr, sizeof(kxo_row), row_cmp);
    for (size_t i = 0; i < nkeys; i++) {
        kxo_row k; k.key = keys[i];
        kxo_row *r = (kxo_row *)bsearch(&k, rows, nr, sizeof(kxo_row), row_cmp);
        if (line_off) line_off[i] = r ? (int64_t)r->line_off : -1;
    }
    double t2 = now_s();
    free(rows);
    if (parse_s) *parse_s = t1 - t0;
    return t2 - t0;
}

/* ------------------------------------------------------------------------- */
/* "Best honest CPU" on ALL host threads: the text is cut into one shard per    */
/* thread where a top-level line starts (the same rule as kxpu_plan_shards),    */
/* every thread runs the single pass of kxo_table_build on its shard (device    */
/* lines under a vendor id it has already seen are skipped unparsed, exactly    */
/* the first-occurrence shortcut the GPU kernel uses), then the shards' first   */
/* anchors are min-merged and the rows whose anchor is the global first one are */
/* concatenated in shard (= file) order.  Equals kxo_table_build on the whole   */
/* text (tests/test_oracle.py).  Keys are probed by binary search, in parallel. */
/* ------------------------------------------------------------------------- */
static size_t kxo_next_top(const uint8_t *text, size_t n, size_t pos) {
    if (pos == 0) return 0;
    if (pos >= n) return n;
    size_t p = pos;
    if (text[p - 1] != '\n') {
        const uint8_t *nl = (const uint8_t *)memchr(text + p, '\n', n - p);
        if (!nl) return n;
        p = (size_t)(nl - text) + 1;
    }
    while (p < n) {
        if (text[p] != '\t' && text[p] != '#') return p;
        const uint8_t *nl = (const uint8_t *)memchr(text + p, '\n', n - p);
        if (!nl) return n;
        p = (size_t)(nl - text) + 1;
    }
    return n;
}

typedef struct {
    const uint8_t *text; size_t n, lo, hi;  /* shard [lo,hi) of text[0..n) */
    kxo_row *rows; size_t nrows, cap;
    uint64_t *vfirst;                       /* [65536] first anchor of the shard per vendor, ~0 = none */
    uint64_t trunc;                         /* offset where the scan stops (ErrTooLong), ~0 = never */
} kxo_shard_job;

static void *shard_worker(void *arg) {
    kxo_shard_job *j = (kxo_shard_job *)arg;
    uint8_t *dev_seen = (uint8_t *)calloc(65536 / 8, 1);
    size_t pos = j->lo, ls, le;
    int cur_valid = 0, rc;
    uint32_t cur_v = 0;
    uint64_t cur_anchor = 0;
    j->nrows = 0; j->trunc = ~0ull;
    memset(j->vfirst, 0xff, 65536 * sizeof(uint64_t));
    while ((rc = kxo_next_line(j->text, j->hi, &pos, &ls, &le)) == 1) {
        size_t len = le - ls;
        const uint8_t *l = j->text + ls;
        if (len >= 1 && l[0] == '#') continue;
        if (len >= 1 && l[0] == '\t') {
            uint32_t d;
            if (cur_valid && parse_hex4(l + 1, len - 1, &d) && !(dev_seen[d >> 3] & (1u << (d & 7)))) {
                dev_seen[d >> 3] |= (uint8_t)(1u << (d & 7));
                if (j->nrows == j->cap) { j->cap = j->cap ? j->cap * 2 : 4096; j->rows = (kxo_row *)realloc(j->rows, j->cap * sizeof(kxo_row)); }
                j->rows[j->nrows].key = (cur_v << 16) | d; j->rows[j->nrows].line_off = ls; j->rows[j->nrows].anchor_off = cur_anchor;
                j->nrows++;
            }
            continue;
        }
        cur_valid = 0;
        uint32_t v;
        if (parse_hex4(l, len, &v) && j->vfirst[v] == ~0ull) {
            j->vfirst[v] = ls;
            cur_valid = 1; cur_v = v; cur_anchor = ls;
            memset(dev_seen, 0, 65536 / 8);
        }
    }
    if (rc == -1) j->trunc = pos;
    free(dev_seen);
    return NULL;
}

/* rows_out (may be NULL) receives up to cap rows in file order; returns the row count */
size_t kxo_table_build_mt(const uint8_t *text, size_t n, int threads, kxo_row *rows_out, size_t cap) {
    if (threads < 1) threads = 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    kxo_shard_job *jobs = (kxo_shard_job *)calloc((size_t)threads, sizeof(kxo_shard_job));
    size_t cut = 0;
    for (int t = 0; t < threads; t++) {
        size_t next = t + 1 == threads ? n : kxo_next_top(text, n, (size_t)((unsigned __int128)n * (unsigned)(t + 1) / (unsigned)threads));
        if (next < cut) next = cut;
        jobs[t].text = text; jobs[t].n = n; jobs[t].lo = cut; jobs[t].hi = next;
        jobs[t].vfirst = (uint64_t *)malloc(65536 * sizeof(uint64_t));
        cut = next;
        pthread_create(&th[t], NULL, shard_worker, &jobs[t]);
    }
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
    uint64_t *gfirst = (uint64_t *)malloc(65536 * sizeof(uint64_t));
    memset(gfirst, 0xff, 65536 * sizeof(uint64_t));
    uint64_t trunc = ~0ull;
    for (int t = 0; t < threads; t++) {
        for (uint32_t v = 0; v < 65536; v++) if (jobs[t].vfirst[v] < gfirst[v]) gfirst[v] = jobs[t].vfirst[v];
        if (jobs[t].trunc < trunc) trunc = jobs[t].trunc;
    }
    size_t nr = 0;
    for (int t = 0; t < threads; t++) {
        for (size_t i = 0; i < jobs[t].nrows; i++) {
            const kxo_row *r = &jobs[t].rows[i];
            /* a top-level line is a valid anchor only in front of the cut-off, a row only in front of it too */
            if (r->anchor_off == gfirst[r->key >> 16] && r->line_off < trunc) {
                /* field by field, like kxo_table_build: a struct copy would carry the uninitialised padding after key */
                if (rows_out && nr < cap) { rows_out[nr].key = r->key; rows_out[nr].line_off = r->line_off; rows_out[nr].anchor_off = r->anchor_off; }
                nr++;
            }
        }
        free(jobs[t].rows); free(jobs[t].vfirst);
    }
    free(gfirst); free(th); free(jobs);
    return nr;
}

typedef struct { const kxo_row *rows; size_t nr; const uint32_t *keys; size_t lo, hi; int64_t *line_off; } kxo_probe_job;
static void *probe_worker(void *arg) {
    kxo_probe_job *j = (kxo_probe_job *)arg;
    for (size_t i = j->lo; i < j->hi; i++) {
        kxo_row k; k.key = j->keys[i];
        const kxo_row *r = (const kxo_row *)bsearch(&k, j->rows, j->nr, sizeof(kxo_row), row_cmp);
        if (j->line_off) j->line_off[i] = r ? (int64_t)r->line_off : -1;
    }
    return NULL;
}

/* parse on `threads` threads + parallel probes; returns total seconds, *parse_s = parse + merge */
double kxo_bench_parse_mt(const uint8_t *text, size_t n, int threads, const uint32_t *keys, size_t nkeys,
                          int64_t *line_off, double *parse_s) {
    if (threads < 1) threads = 1;
    double t0 = now_s();
    size_t cap = 1u << 16;
    kxo_row *rows = (kxo_row *)malloc(cap * sizeof(kxo_row));
    size_t nr = kxo_table_build_mt(text, n, threads, rows, cap);
    if (nr > cap) { cap = nr; rows = (kxo_row *)realloc(rows, cap * sizeof(kxo_row)); nr = kxo_table_build_mt(text, n, threads, rows, cap); }
    double t1 = now_s();
    qsort(rows, nr, sizeof(kxo_row), row_cmp);
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    kxo_probe_job *pj = (kxo_probe_job *)calloc((size_t)threads, sizeof(kxo_probe_job));
    for (int t = 0; t < threads; t++) {
        pj[t].rows = rows; pj[t].nr = nr; pj[t].keys = keys; pj[t].line_off = line_off;
        pj[t].lo = nkeys * (size_t)t / (size_t)threads; pj[t].hi = nkeys * (size_t)(t + 1) / (size_t)threads;
        pthread_create(&th[t], NULL, probe_worker, &pj[t]);
    }
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
    double t2 = now_s();
    free(th); free(pj); free(rows);
    if (parse_s) *parse_s = t1 - t0;
    return t2 - t0;
}

/* ------------------------------------------------------------------------- */
/* SURVEY 8(f) row 4: the rest of the pci.ids model.  The reference scans the   */
/* subsystem lines and the class section and ignores them (device_plugin.go:    */
/* 229-237); what they MEAN is stated by the file itself (utils/pci.ids:23-27,  */
/* :38195-38200):                                                               */
/*     vendor  vendor_name                                                      */
/*     \t device  device_name                                                   */
/*     \t\t subvendor subdevice  subsystem_name                                 */
/*     C class  class_name / \t subclass  name / \t\t prog-if  name             */
/* Restated with the reference's own matching rules carried one level down:     */
/* raw byte prefixes, first occurrence wins at every level, a block ends at the */
/* first line that is neither a comment nor indented, bufio line semantics.     */
/* Rows (key, offset of the line) in file order:                                */
/*   kind 0 vendor    key = v                                                   */
/*   kind 1 subsystem key = v<<48 | d<<32 | sv<<16 | sd                         */
/*   kind 2 class     key = 1<<24 | c<<16 ; subclass 2<<24 | c<<16 | s<<8 ;     */
/*                    prog-if 3<<24 | c<<16 | s<<8 | p                          */
/* ------------------------------------------------------------------------- */
typedef struct kxo_row64 { uint64_t key; uint64_t line_off; } kxo_row64;

static int parse_hex2(const uint8_t *s, size_t len, uint32_t *v) {
    if (len < 2 || !is_lhex(s[0]) || !is_lhex(s[1])) return 0;
    *v = (uint32_t)(hexval(s[0]) * 16 + hexval(s[1]));
    return 1;
}

size_t kxo_full_build(const uint8_t *text, size_t n, int kind, kxo_row64 *rows, size_t cap) {
    uint8_t *vendor_seen = (uint8_t *)calloc(65536, 1), *class_seen = (uint8_t *)calloc(256, 1);
    uint8_t *dev_seen = (uint8_t *)calloc(65536 / 8, 1), *sub_seen = (uint8_t *)calloc(256 / 8, 1);
    /* (subvendor, subdevice) / prog-if seen under the current device / subclass line: generation-stamped set */
    size_t scap = 1u << 16;
    uint64_t *skeys = (uint64_t *)calloc(scap, sizeof(uint64_t));
    uint32_t *sgen = (uint32_t *)calloc(scap, sizeof(uint32_t)), gen = 0;
    size_t pos = 0, ls, le, nrows = 0;
    int vblock = 0, cblock = 0, dev_ok = 0, sub_ok = 0;
    uint32_t cur_v = 0, cur_d = 0, cur_c = 0, cur_s = 0;
#define KXO_EMIT(k) do { if (nrows < cap) { rows[nrows].key = (k); rows[nrows].line_off = ls; } nrows++; } while (0)
    while (kxo_next_line(text, n, &pos, &ls, &le) == 1) {
        size_t len = le - ls;
        const uint8_t *l = text + ls;
        if (len >= 1 && l[0] == '#') continue;
        if (len >= 2 && l[0] == '\t' && l[1] == '\t') {
            uint64_t key;
            uint32_t a, b;
            if (vblock && dev_ok && parse_hex4(l + 2, len - 2, &a) && len >= 11 && l[6] == ' ' && parse_hex4(l + 7, len - 7, &b))
                key = ((uint64_t)cur_v << 48) | ((uint64_t)cur_d << 32) | ((uint64_t)a << 16) | b;
            else if (cblock && sub_ok && parse_hex2(l + 2, len - 2, &a))
                key = (3ull << 24) | ((uint64_t)cur_c << 16) | ((uint64_t)cur_s << 8) | a;
            else
                continue;
            size_t h = (size_t)((key * 0x9E3779B97F4A7C15ull) >> 40) & (scap - 1);
            int dup = 0;
            while (sgen[h] == gen) { if (skeys[h] == key) { dup = 1; break; } h = (h + 1) & (scap - 1); }
            if (dup) continue;
            sgen[h] = gen; skeys[h] = key;
            if ((vblock && kind == 1) || (cblock && kind == 2)) KXO_EMIT(key);
            continue;
        }
        if (len >= 1 && l[0] == '\t') {
            uint32_t d;
            dev_ok = sub_ok = 0;
            gen++;  /* a new device / subclass line: its second-level set starts empty */
            if (gen == 0) { memset(sgen, 0, scap * sizeof(uint32_t)); gen = 1; }
            if (vblock && parse_hex4(l + 1, len - 1, &d)) {
                if (!(dev_seen[d >> 3] & (1u << (d & 7)))) { dev_seen[d >> 3] |= (uint8_t)(1u << (d & 7)); dev_ok = 1; cur_d = d; }
            } else if (cblock && parse_hex2(l + 1, len - 1, &d)) {
                if (!(sub_seen[d >> 3] & (1u << (d & 7)))) {
                    sub_seen[d >> 3] |= (uint8_t)(1u << (d & 7)); sub_ok = 1; cur_s = d;
                    if (kind == 2) KXO_EMIT((2ull << 24) | ((uint64_t)cur_c << 16) | ((uint64_t)d << 8));
                }
            }
            continue;
        }
        /* top-level line: ends any block; may start a vendor block or a class block */
        vblock = cblock = dev_ok = sub_ok = 0;
        uint32_t v;
        if (len >= 4 && l[0] == 'C' && l[1] == ' ' && parse_hex2(l + 2, len - 2, &v)) {
            if (!class_seen[v]) {
                class_seen[v] = 1; cblock = 1; cur_c = v;
                memset(sub_seen, 0, 256 / 8);
                if (kind == 2) KXO_EMIT((1ull << 24) | ((uint64_t)v << 16));
            }
        } else if (parse_hex4(l, len, &v) && !vendor_seen[v]) {
            vendor_seen[v] = 1; vblock = 1; cur_v = v;
            memset(dev_seen, 0, 65536 / 8);
            if (kind == 0) KXO_EMIT((uint64_t)v);
        }
    }
#undef KXO_EMIT
    free(vendor_seen); free(class_seen); free(dev_seen); free(sub_seen); free(skeys); free(sgen);
    return nrows;
}
