"""GPU parity tests of the pci.ids path (K1-K4) through the C ABI, against the oracle."""
import hashlib

import numpy as np
import pytest

import pyref
from test_oracle import EDGE_TEXTS

pytestmark = pytest.mark.gpu


def table_as_dict(kx, tab):
    keys, offs, rows = kx.table_export(tab)
    names, _, _ = kx.names(tab, rows)
    return keys, offs, rows, names


def check_text(kx, oracle, text, extra_keys=()):
    """Full-table and per-key parity of one text against the oracle."""
    tab = kx.pciids_load(text)
    try:
        keys, offs, rows, names = table_as_dict(kx, tab)
        orows = oracle.table_build(text)
        assert np.array_equal(keys, orows["key"])
        assert np.array_equal(offs, orows["line_off"])
        for k, o, nm in zip(keys[:200], offs[:200], names[:200]):
            assert nm == oracle.row_name(text, int(o))
        q = np.array(list(keys[:64]) + list(extra_keys), dtype=np.uint32)
        if len(q):
            r = kx.lookup(tab, q)
            gn, _, _ = kx.names(tab, r)
            line_of_row = dict(zip(rows.tolist(), offs.tolist()))
            for k, row, nm in zip(q, r, gn):
                ooff, oname = oracle.device_name(text, int(k))
                assert (line_of_row[int(row)] if row >= 0 else -1) == ooff, hex(int(k))
                assert nm == (oname or b"")
    finally:
        tab.free()


def test_cfg2_full_pci_ids(kx, oracle, pci_text, oracle_rows, golden, workloads):
    """BASELINE.json configs[1]: full utils/pci.ids parse + 1024 synthetic lookups, bit-exact."""
    tab = kx.pciids_load(pci_text)
    keys, offs, rows, names = table_as_dict(kx, tab)
    assert tab.rows == golden["rows"]
    assert np.array_equal(keys, oracle_rows["key"]) and np.array_equal(offs, oracle_rows["line_off"])
    dump = b"".join(b"%04x:%04x\t%s\n" % (k >> 16, k & 0xFFFF, nm) for k, nm in zip(keys, names))
    assert hashlib.sha256(dump).hexdigest() == golden["dump_sha256"]
    q = workloads.cfg2_queries(oracle_rows["key"])
    r = kx.lookup(tab, q)
    assert int((r >= 0).sum()) == 768
    ooffs, onames = oracle.lookup_many(pci_text, q)
    line_of_row = dict(zip(rows.tolist(), offs.tolist()))
    got = np.array([line_of_row[x] if x >= 0 else -1 for x in r.tolist()], dtype=np.int64)
    assert np.array_equal(got, ooffs)
    gn, _, _ = kx.names(tab, r)
    assert gn == [n or b"" for n in onames]
    for k, want in golden["spots"].items():
        row = kx.lookup(tab, np.array([int(k, 16)], np.uint32))
        nm = kx.names(tab, row)[0][0]
        assert nm.decode() == (want["name"] or "")
    tab.free()


@pytest.mark.parametrize("text", EDGE_TEXTS)
def test_edge_texts(kx, oracle, text):
    check_text(kx, oracle, text, extra_keys=[0x10de2330, 0x10de0001, 0x10de0002, 0x10df0001, 0, 0xffffffff])


def test_ragged_sizes_around_tile_boundaries(kx, oracle, pci_text):
    """Tile = 16 KiB, TMA stage has 16-byte halos: cut the text at awkward lengths."""
    for n in [1, 5, 15, 16, 17, 16383, 16384, 16385, 16399, 16400, 16401, 32767, 32768, 32769, 49152 + 7, 100001]:
        check_text(kx, oracle, pci_text[:n])


def test_key_ffffffff_and_illegal_vendor(kx, oracle):
    text = b"ffff  Illegal Vendor ID\n\tffff  all ones\n\t0000  zeros\n0000  zero vendor\n\t0000  z\n"
    check_text(kx, oracle, text, extra_keys=[0xffffffff, 0xffff0000, 0, 0x0000ffff])


def test_duplicate_vendor_blocks_first_wins(kx, oracle, pci_text):
    """x3 replication: every key has three occurrences, the first wins; a vendor whose device
    only appears under a LATER anchor must miss."""
    text = pci_text[:200000]
    text = text[:text.rfind(b"\n") + 1]
    check_text(kx, oracle, text * 3)
    tricky = b"10de  first\n\t0001  a\n10df  x\n10de  again\n\t0002  hidden\n" * 50
    check_text(kx, oracle, tricky, extra_keys=[0x10de0002, 0x10de0001])


def test_long_block_needs_tile_lookback(kx, oracle):
    """A vendor block spanning many 16 KiB tiles: device lines far from their vendor line
    resolve through the decoupled look-back carry."""
    lines = [b"abcd  Big vendor\n"]
    for d in range(20000):
        lines.append(b"\t%04x  Device number %d\n" % (d, d))
        if d % 7 == 0:
            lines.append(b"\t\t1234 %04x  subsystem\n" % d)
        if d % 13 == 0:
            lines.append(b"# comment\n")
    lines.append(b"abce  Next\n\t0001  n\n")
    text = b"".join(lines)
    assert len(text) > 30 * 16384
    check_text(kx, oracle, text, extra_keys=[0xabcd0000, 0xabcd4e1f, 0xabce0001, 0xabcd4e20])


def test_short_lines_in_huge_block(kx, oracle):
    """> 2048 device lines of one 64 KiB super-chunk governed by an EARLIER super-chunk: the v3
    kernel's parking buffer overflows and the library falls back to the v2 kernel."""
    lines = [b"abcd  Big\n"] + [b"\t%04x  x\n" % (d & 0xffff) for d in range(40000)] + [b"abce  N\n\t0001  n\n"]
    text = b"".join(lines)
    assert len(text) > 5 * 65536
    check_text(kx, oracle, text, extra_keys=[0xabcd0000, 0xabcd9c3f, 0xabcdffff, 0xabce0001])
    # every line a bare newline / tiny: more line starts than the per-warp list holds (multi-window path)
    text = b"10de  NV\n" + b"\n".join(b"\t%04x" % d for d in range(3000)) + b"\n\n\n\n" * 3000 + b"\t0001  late\n"
    check_text(kx, oracle, text, extra_keys=[0x10de0000, 0x10de0bb7, 0x10de0001])


def test_too_long_line(kx, oracle):
    ok_line = b"#" + b"x" * 65534
    bad_line = b"#" + b"x" * 65535
    for mid in (ok_line, bad_line):
        text = b"10de  NV\n\t0001  a\n" + mid + b"\n\t0002  b\n10df  v\n\t0003  c\n"
        check_text(kx, oracle, text, extra_keys=[0x10de0001, 0x10de0002, 0x10df0003])
    # unterminated, too long final line
    text = b"10de  NV\n\t0001  a\n10df  v\n\t0003  " + b"y" * 70000
    check_text(kx, oracle, text, extra_keys=[0x10de0001, 0x10df0003])
    # long but legal device name (slow path of the sanitiser)
    text = b"10de  NV\n\t0001  " + b"Ab.c " * 2000 + b"\n\t0002  z\n"
    check_text(kx, oracle, text, extra_keys=[0x10de0001, 0x10de0002])


def test_unicode_and_crlf_names(kx, oracle):
    text = (b"10de  NV\r\n\t0001  Wi-Fi\xc2\xae 5 \xc2\xa0\r\n\t0002  d\xc4\xb1g \xc5\xbf\n\t0003   \n\t0004\n"
            b"\t0005  a\tb \x0b c \n\t0006  \xe2\x80\x83em\xe3\x80\x80\n\t0007  \xff\xfe ok\n")
    check_text(kx, oracle, text, extra_keys=[0x10de0000 + i for i in range(1, 9)])


def test_random_pciids_shaped_texts(kx, oracle):
    """Seeded random texts with the pci.ids grammar plus noise (blank lines, class section,
    duplicate vendors, upper-case hex, short lines)."""
    rng = np.random.default_rng(2024)
    for trial in range(12):
        lines = []
        for _ in range(int(rng.integers(5, 400))):
            r = rng.random()
            v = int(rng.integers(0, 40)) * 0x0101
            if r < 0.2:
                lines.append(b"%04x  Vendor %d\n" % (v, v))
            elif r < 0.7:
                lines.append(b"\t%04x  Dev.%d / x\n" % (int(rng.integers(0, 60)), int(rng.integers(0, 1000))))
            elif r < 0.8:
                lines.append(b"\t\t%04x %04x  Sub\n" % (v, v))
            elif r < 0.85:
                lines.append(b"# c\n")
            elif r < 0.88:
                lines.append(b"\n")
            elif r < 0.91:
                lines.append(b"C %02x  Class\n" % int(rng.integers(0, 255)))
            elif r < 0.94:
                lines.append(b"\t%04X  UPPER\n" % int(rng.integers(0xa000, 0xffff)))
            elif r < 0.97:
                lines.append(b"\t12\n")
            else:
                lines.append(b"%04x\n" % v)
        text = b"".join(lines)
        if trial % 3 == 0:
            text = text.rstrip(b"\n")
        keys = [(int(rng.integers(0, 40)) * 0x0101 << 16) | int(rng.integers(0, 60)) for _ in range(40)]
        check_text(kx, oracle, text, extra_keys=keys)


def test_x1000_first_occurrence_wins(kx, oracle, pci_text, oracle_rows, workloads):
    """BASELINE.json configs[3] at full size on one GPU: 1.458 GB text, 2^20 keys; the table must
    equal the oracle's table of the SAME 1.458 GB buffer (kxo_table_build, one pass, ~0.5 s) --
    which in turn equals the single-copy table (first occurrence wins) -- and every lookup must
    agree with it."""
    n, copies = len(pci_text), 1000
    big = np.tile(np.frombuffer(pci_text, np.uint8), copies)
    obig = oracle.table_build(big)
    assert np.array_equal(obig["key"], oracle_rows["key"]) and np.array_equal(obig["line_off"], oracle_rows["line_off"])
    del big
    d_one = kx.dev_alloc(n)
    kx.upload(d_one, np.frombuffer(pci_text, np.uint8))
    d_big = kx.dev_alloc(n * copies)
    kx.replicate(d_big, d_one, n, copies)
    tab = kx.pciids_load_device(d_big, n * copies)
    keys, offs, rows = kx.table_export(tab)
    assert np.array_equal(keys, obig["key"]) and np.array_equal(offs, obig["line_off"])
    q = workloads.cfg4_queries(oracle_rows["key"])
    r = kx.lookup(tab, q)
    # oracle via the single-copy table (identical by the property above)
    order = np.argsort(oracle_rows["key"])
    sk = oracle_rows["key"][order]
    pos = np.searchsorted(sk, q)
    pos[pos >= len(sk)] = 0
    hit = sk[pos] == q
    want = np.where(hit, oracle_rows["line_off"][order][pos].astype(np.int64), -1)
    line_of_row = np.full(tab.rows + 1, -1, np.int64)
    line_of_row[rows] = offs.astype(np.int64)
    got = np.where(r >= 0, line_of_row[np.maximum(r, 0)], -1)
    assert np.array_equal(got, want)
    assert int(hit.sum()) == int((r >= 0).sum()) == 786432
    tab.free()
    kx.dev_free(d_big)
    kx.dev_free(d_one)


def test_names_nospace_and_empty(kx, pci_text):
    import ctypes as C
    tab = kx.pciids_load(pci_text)
    rows = kx.lookup(tab, np.array([0x10de2330, 0x10de2901], np.uint32))
    assert rows[0] >= 0 and rows[1] == -1
    names, blob, offs = kx.names(tab, rows)
    assert names == [b"GH100_H100_SXM5_80GB", b""]
    offs2 = np.empty(3, np.uint32)
    need = C.c_size_t(0)
    out = np.empty(4, np.uint8)
    rc = kx.L.kxpu_names(kx.ctx, tab.handle, rows.ctypes.data, 2, out.ctypes.data, 4, offs2.ctypes.data, C.byref(need))
    assert rc == -4 and need.value == 20
    assert kx.lookup(tab, np.empty(0, np.uint32)).size == 0
    tab.free()


def test_repeated_loads_are_deterministic(kx, pci_text, oracle_rows):
    """The parse kernel hands work between warps through mbarriers, shared-memory status words
    and atomics; run it many times on a text that spans thousands of super-chunks and demand
    the identical table every time (scheduling differs from run to run)."""
    n, copies = len(pci_text), 120
    d_one = kx.dev_alloc(n)
    kx.upload(d_one, np.frombuffer(pci_text, np.uint8))
    d_big = kx.dev_alloc(n * copies)
    kx.replicate(d_big, d_one, n, copies)
    for it in range(30):
        tab = kx.pciids_load_device(d_big, n * copies - (it % 7) * 1001)  # ragged ends too
        keys, offs, rows = kx.table_export(tab)
        if (it % 7) == 0:
            assert np.array_equal(keys, oracle_rows["key"]) and np.array_equal(offs, oracle_rows["line_off"]), it
        else:
            assert len(keys) == len(oracle_rows) and np.array_equal(offs, oracle_rows["line_off"]), it
        tab.free()
    kx.dev_free(d_big)
    kx.dev_free(d_one)


def _big_random_text(rng, n_lines, vendors, dup_prob):
    """pci.ids-shaped text with blocks long enough to cross many 2 KiB chunks / 16 KiB ranges and
    vendor ids that repeat (only the first block of an id may produce hits)."""
    lines, seen = [], []
    while len(lines) < n_lines:
        v = int(rng.choice(seen)) if seen and rng.random() < dup_prob else int(rng.integers(0, vendors))
        seen.append(v)
        lines.append(b"%04x  Vendor %d\n" % (v, v))
        for _ in range(int(rng.integers(0, 1500)) if rng.random() < 0.3 else int(rng.integers(0, 12))):
            d = int(rng.integers(0, 0x10000))
            lines.append(b"\t%04x  Device %d of %d\n" % (d, d, v))
            if rng.random() < 0.3:
                lines.append(b"\t\t%04x %04x  Subsystem\n" % (v, d))
            if rng.random() < 0.02:
                lines.append(b"# comment\n")
    return b"".join(lines)


def test_big_random_texts_many_ranges(kx, oracle):
    """Texts of 0.3-2 MB: carries across chunks and ranges, alive and dead blocks interleaved,
    blocks starting right before / after range boundaries."""
    rng = np.random.default_rng(77)
    for trial, (n_lines, vendors, dup) in enumerate([(12000, 300, 0.3), (40000, 50, 0.6), (60000, 4000, 0.05)]):
        text = _big_random_text(rng, n_lines, vendors, dup)
        if trial == 1:
            text = b"\t0001  orphan before any vendor line\n" + text
        keys = [int(rng.integers(0, vendors)) << 16 | int(rng.integers(0, 0x10000)) for _ in range(64)]
        check_text(kx, oracle, text, extra_keys=keys)


def test_block_boundaries_at_range_edges(kx, oracle):
    """A vendor line placed exactly at / around every 2 KiB chunk and 16 KiB range boundary, the
    block before it alive, the block after it a repeat of an earlier id (dead)."""
    for edge in (2048, 16384, 16384 * 3, 16384 * 8):
        for delta in (-9, -1, 0, 1, 2):
            pad_lines = []
            size = len(b"1111  first\n")
            d = 0
            while size + 14 < edge + delta:
                pad_lines.append(b"\t%04x  pad %03d\n" % (d & 0xffff, d % 1000))
                size += 14
                d += 1
            filler = b"#" + b"x" * max(0, edge + delta - size - 2) + b"\n" if edge + delta - size >= 2 else b""
            text = (b"1111  first\n" + b"".join(pad_lines) + filler + b"2222  second\n\t0001  two-one\n" +
                    b"1111  again\n\t0fff  hidden\n" + b"\t%04x  tail\n" % 7 * 900 + b"3333  third\n\t0003  t\n")
            check_text(kx, oracle, text, extra_keys=[0x11110000, 0x11110fff, 0x22220001, 0x33330003, 0x11110007])


def test_structural_byte_fuzz(kx, oracle):
    """Random byte soup weighted towards the bytes the parser branches on (newline, tab, '#', hex
    digits, CR, VT, NUL, high bytes): every window / chunk / range code path sees odd neighbours."""
    rng = np.random.default_rng(99)
    alphabet = np.frombuffer(b"\n\n\n\n\t\t\t##0123456789abcdefABCDEF  \r\x0b\x00\xff\x80xyz", dtype=np.uint8)
    for trial in range(60):
        n = int(rng.integers(1, 40000))
        body = alphabet[rng.integers(0, len(alphabet), n)].tobytes()
        if trial % 2 == 0:
            # sprinkle well-formed vendor / device lines so that hits exist
            pieces = [body[i:i + 257] for i in range(0, len(body), 257)]
            body = b"".join(p + b"\n%04x  V\n\t%04x  D\n" % (int(rng.integers(0, 6)), int(rng.integers(0, 6))) for p in pieces)
        keys = [(int(rng.integers(0, 6)) << 16) | int(rng.integers(0, 6)) for _ in range(16)]
        check_text(kx, oracle, body, extra_keys=keys)


def test_join_device_equals_load_then_lookup(kx, pci_text, oracle_rows, workloads):
    """kxpu_pciids_join_device == kxpu_pciids_load_device + kxpu_lookup_device (also when the
    table has to grow and the join is replayed)."""
    for text in (pci_text, b"abcd  Big\n" + b"".join(b"\t%04x  x\n" % d for d in range(40000))):
        buf = np.frombuffer(text, np.uint8)
        d_text = kx.dev_alloc(len(buf))
        kx.upload(d_text, buf)
        t0 = kx.pciids_load_device(d_text, len(buf))
        keys, _, _ = kx.table_export(t0)
        q = workloads.make_queries(keys, 4096, 11)
        d_q, d_r = kx.dev_alloc(q.nbytes), kx.dev_alloc(q.nbytes)
        kx.upload(d_q, q)
        kx.lookup_device(t0, d_q, len(q), d_r)
        want = kx.download(d_r, q.nbytes, np.int32)
        kx.upload(d_r, np.full(len(q), -7, np.int32))
        t1 = kx.pciids_join_device(d_text, len(buf), d_q, len(q), d_r)
        got = kx.download(d_r, q.nbytes, np.int32)
        k1, o1, r1 = kx.table_export(t1)
        k0, o0, r0 = kx.table_export(t0)
        assert t1.rows == t0.rows and np.array_equal(k0, k1) and np.array_equal(o0, o1)
        # row handles belong to their table: compare the lines they stand for
        line0 = dict(zip(r0.tolist(), o0.tolist()))
        line1 = dict(zip(r1.tolist(), o1.tolist()))
        assert [line0.get(x, -1) for x in want.tolist()] == [line1.get(x, -1) for x in got.tolist()]
        assert (want >= 0).any() and (got != -7).all()
        for t in (t0, t1):
            t.free()
        for d in (d_text, d_q, d_r):
            kx.dev_free(d)


@pytest.mark.parametrize("rch", [1, 2, 3, 4, 5, 7, 8])
def test_every_range_length(rch, oracle, pci_text, monkeypatch):
    """The parse kernel cuts the text into ranges of 1..8 chunks depending on its size
    (KXPU_RCH forces one): the prefetch ring, the carry and the resolve pass must agree for all."""
    import kxpu_b200 as K
    monkeypatch.setenv("KXPU_RCH", str(rch))
    k = K.Kxpu(0)
    try:
        rng = np.random.default_rng(rch)
        check_text(k, oracle, pci_text[:400003])
        check_text(k, oracle, pci_text[:pci_text.rfind(b"\n", 0, 120000) + 1] * 5)
        check_text(k, oracle, _big_random_text(rng, 9000, 120, 0.4), extra_keys=[0x00010001, 0x00630000])
        for n in (2047, 2048, 2049, 2048 * rch, 2048 * rch + 1, 2048 * rch * 3 - 1):
            check_text(k, oracle, pci_text[:n])
    finally:
        k.close()


def test_name_lengths_around_the_finalize_windows(kx, oracle):
    """The finalize looks at a 128-byte window per row (fast path), stages up to ~1 KB for longer lines
    (warp path) and reads even longer ones serially: names of every length around those limits, at
    every 16-byte phase of the line start, with trailing CR / blanks / non-ASCII bytes."""
    rng = np.random.default_rng(3)
    alphabet = np.frombuffer(b"abcXYZ019 /._-[]()\t", np.uint8)
    parts, keys = [b"1234  Vendor\n"], []
    d = 0
    for ln in list(range(0, 20)) + list(range(100, 135)) + list(range(980, 1040)) + [2000, 5000]:
        for pad in (0, 3, 7, 13):
            name = alphabet[rng.integers(0, len(alphabet), ln)].tobytes()
            tail = [b"", b"\r", b"  ", b" \xc2\xa0"][(ln + pad) % 4]
            parts.append(b"#" + b"x" * pad + b"\n")  # shifts the 16-byte phase of the next line
            parts.append(b"\t%04x  " % d + name + tail + b"\n")
            keys.append(0x12340000 | d)
            d += 1
    text = b"".join(parts)
    tab = kx.pciids_load(text)
    try:
        r = kx.lookup(tab, np.array(keys, np.uint32))
        assert (r >= 0).all()
        names, _, _ = kx.names(tab, r)
        for k, nm in zip(keys, names):
            assert nm == (oracle.device_name(text, k)[1] or b""), hex(k)
    finally:
        tab.free()


def test_host_join_one_round_trip(kx, oracle, pci_text, oracle_rows, workloads):
    """kxpu_pciids_join (host text + host keys, one call): same table and row handles as load + lookup,
    on the small-text kernel (pci.ids) and on a text that is too large for it."""
    for text in (pci_text, pci_text * 8):
        q = workloads.make_queries(oracle_rows["key"], 3000, 5)
        tab, rows = kx.pciids_join(text, q)
        keys, offs, tr = kx.table_export(tab)
        want = oracle.table_build(text)
        assert np.array_equal(keys, want["key"]) and np.array_equal(offs, want["line_off"])
        line_of_row = np.full(tab.rows + 1, -1, np.int64)
        line_of_row[tr] = offs.astype(np.int64)
        got = np.where(rows >= 0, line_of_row[np.maximum(rows, 0)], -1)
        order = np.argsort(want["key"])
        sk = want["key"][order]
        pos = np.searchsorted(sk, q)
        pos[pos >= len(sk)] = 0
        exp = np.where(sk[pos] == q, want["line_off"][order][pos].astype(np.int64), -1)
        assert np.array_equal(got, exp)
        assert np.array_equal(rows, kx.lookup(tab, q))
        tab.free()
    tab, rows = kx.pciids_join(b"", np.array([1, 2], np.uint32))
    assert tab.rows == 0 and (rows == -1).all()
    tab.free()


def test_zero_copy_join_from_pinned_host_buffers(kx, oracle, pci_text, oracle_rows, workloads):
    """kxpu_pciids_join with text, keys and rows in mapped pinned host memory: the small-text kernel pulls the text
    over PCIe itself (no copy is enqueued) and writes row handles and counters to host memory.  Same results as
    the copying path for the real file, ragged sizes around chunk boundaries, edge texts, a text whose table has to
    grow (retry) and a text with a >= 64 KiB line (second attempt leaves the small-text kernel)."""
    rng = np.random.default_rng(11)
    texts = [pci_text] + [pci_text[:n] for n in (1, 15, 16, 17, 2047, 2048, 2049, 2064, 4096, 4097, 300001)] + list(EDGE_TEXTS)
    texts.append(_big_random_text(rng, 60000, 200, 0.2))                     # > 32 k keys: the 2^16 table grows (retry)
    texts.append(b"10de  NVIDIA\n\t2330  H100\n" + b"x" * 70000 + b"\n\t2331  Other\n10df  Next\n\t0001  Dev\n")  # ErrTooLong cut-off
    for text in texts:
        if len(text) == 0:
            continue
        want = oracle.table_build(text)
        q = workloads.make_queries(want["key"] if len(want["key"]) else np.array([0x10de2330], np.uint32), 777, 5)
        h_text, p1 = kx.pinned(len(text))
        h_text[:] = np.frombuffer(text, np.uint8)
        h_q, p2 = kx.pinned(len(q) * 4, np.uint32)
        h_q[:] = q
        h_r, p3 = kx.pinned(len(q) * 4, np.int32)
        h_r[:] = -7
        try:
            tab, rows = kx.pciids_join(h_text, h_q, rows_out=h_r)
            keys, offs, _ = kx.table_export(tab)
            assert np.array_equal(keys, want["key"]) and np.array_equal(offs, want["line_off"]), len(text)
            assert np.array_equal(rows, kx.lookup(tab, q)), len(text)
            ref_tab, ref_rows = kx.pciids_join(bytes(text), q)          # pageable buffers: the copying path
            assert tab.rows == ref_tab.rows
            names, _, _ = kx.names(tab, rows[:200])
            ref_names, _, _ = kx.names(ref_tab, ref_rows[:200])
            assert names == ref_names
            tab.free()
            ref_tab.free()
        finally:
            for p in (p1, p2, p3):
                kx.pinned_free(p)


def test_small_texts_through_the_big_text_kernels(oracle, pci_text, monkeypatch):
    """Small texts normally take the cooperative one-launch kernel; KXPU_NO_SMALL=1 sends them through
    parse_kernel_v5 + resolve + select_finalize, which must agree (ragged sizes, edge texts, real file)."""
    import kxpu_b200 as K
    monkeypatch.setenv("KXPU_NO_SMALL", "1")
    k = K.Kxpu(0)
    try:
        check_text(k, oracle, pci_text)
        for text in EDGE_TEXTS:
            check_text(k, oracle, text)
        for n in (1, 5, 2047, 2048, 2049, 4096, 300001):
            check_text(k, oracle, pci_text[:n])
        rng = np.random.default_rng(8)
        check_text(k, oracle, _big_random_text(rng, 6000, 80, 0.4), extra_keys=[0x00010001, 0x00630000])
        # every chunk of the device lines is a range head with ~340 lines: resolve_chunks_kernel folds its list in passes
        text = b"10de  NV\n" + b"\n".join(b"\t%04x" % d for d in range(3000)) + b"\n\n\n\n" * 3000 + b"\t0001  late\n"
        check_text(k, oracle, text, extra_keys=[0x10de0000, 0x10de0bb7, 0x10de0001])
    finally:
        k.close()
