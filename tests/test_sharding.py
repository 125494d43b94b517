"""N > 1 path: shard planning (CPU, Python planner == kxpu_plan_shards), the shard/merge protocol over
gloo with world_size 2 (CPU), the sharded load + join through the C ABI with several contexts on ONE
GPU (kxpu_ctx_create_multi: the peer-memory exchange runs for real, every box can test it), and the
one-process-per-rank path (CUDA IPC / NCCL) when two GPUs are visible."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def shard_candidates(text, base):
    """What one rank contributes (pure Python restatement of the parse kernel's fold rule): for every
    key the smallest (line, anchor) over ALL blocks of the shard, and per vendor the first anchor."""
    cand, vfirst = {}, {}
    cur = None  # (vendor or None, anchor offset)
    pos = 0
    for line in text.split(b"\n"):
        off = pos
        pos += len(line) + 1
        if off >= len(text):
            break
        if line.endswith(b"\r"):
            line = line[:-1]
        if line.startswith(b"#"):
            continue
        hexok = lambda s: len(s) == 4 and all(c in b"0123456789abcdef" for c in s)
        if line.startswith(b"\t"):
            if cur and cur[0] is not None and hexok(line[1:5]):
                k = (cur[0] << 16) | int(line[1:5], 16)
                v = (base + off, cur[1])
                if k not in cand or v < cand[k]:
                    cand[k] = v
            continue
        v = int(line[:4], 16) if hexok(line[:4]) else None
        cur = (v, base + off)
        if v is not None and v not in vfirst:
            vfirst[v] = base + off
    return cand, vfirst


def merge(parts):
    cand, vfirst = {}, {}
    for c, vf in parts:
        for k, v in c.items():
            if k not in cand or v < cand[k]:
                cand[k] = v
        for v, o in vf.items():
            vfirst[v] = min(o, vfirst.get(v, o))
    rows = sorted((line, k) for k, (line, anchor) in cand.items() if vfirst.get(k >> 16) == anchor)
    return np.array([k for _, k in rows], np.uint32), np.array([l for l, _ in rows], np.uint64)


def test_plan_shards_cuts_at_vendor_lines(pci_text):
    from kxpu_b200.sharding import plan_shards
    for n in (1, 2, 3, 4, 8):
        sh = plan_shards(pci_text, n)
        assert sh[0][0] == 0 and sh[-1][1] == len(pci_text)
        for (a, b), (c, d) in zip(sh, sh[1:]):
            assert b == c
        for a, _ in sh[1:]:
            assert pci_text[a - 1:a] == b"\n" and pci_text[a:a + 1] not in (b"\t", b"#")
    assert plan_shards(b"", 4) == [(0, 0)] * 4
    assert plan_shards(b"\tonly\n\tdevice lines\n", 2) == [(0, 20), (20, 20)]


def test_c_abi_planner_equals_python_planner(pci_text):
    import kxpu_b200 as K
    from kxpu_b200.sharding import plan_shards
    texts = [pci_text, pci_text[:300001], b"", b"\tonly\n\tdevice lines\n", b"a\n#c\n\tb\nc", b"1234  v\n" * 9,
             b"no newline at all", b"\n\n\n", pci_text[1000:200000] * 3]
    for t in texts:
        for n in (1, 2, 3, 4, 7, 8, 16):
            assert K.plan_shards(t, n) == plan_shards(t, n), (len(t), n)


def test_shard_merge_equals_whole_text(oracle, pci_text):
    from kxpu_b200.sharding import plan_shards
    text = pci_text[:300000]
    text = text[:text.rfind(b"\n") + 1] * 2
    want = oracle.table_build(text)
    for n in (1, 2, 5):
        parts = [shard_candidates(text[a:b], a) for a, b in plan_shards(text, n)]
        k, o = merge(parts)
        assert np.array_equal(k, want["key"]) and np.array_equal(o, want["line_off"])


def _gloo_worker(rank, world, port, text, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    import kxpu_b200  # noqa: F401
    from kxpu_b200.sharding import plan_shards
    a, b = plan_shards(text, world)[rank]
    mine = shard_candidates(text[a:b], a)
    parts = [None] * world
    dist.all_gather_object(parts, mine)  # the one exchange of the path
    k, o = merge(parts)
    q.put((rank, k.tobytes(), o.tobytes()))
    dist.destroy_process_group()


def test_world_size_2_gloo(oracle, pci_text):
    """One process per rank over gloo: both ranks end with the table of the whole text."""
    import torch.multiprocessing as mp
    text = pci_text[:200000]
    text = text[:text.rfind(b"\n") + 1] + b"10de  dup\n\t2330  not the first\n" + pci_text[300000:400000]
    want = oracle.table_build(text)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, text, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, kb, ob in got:
        assert np.array_equal(np.frombuffer(kb, np.uint32), want["key"])
        assert np.array_equal(np.frombuffer(ob, np.uint64), want["line_off"])


def _aligned_upload(kx, data):
    d = kx.dev_alloc(max(len(data), 16))
    if len(data):
        kx.upload(d, np.frombuffer(data, np.uint8))
    return d


def _check_multi(oracle, text, nranks, q=None, ordinals=None):
    """Sharded load (+ join) of `text` over `nranks` contexts of one process == oracle on the whole text."""
    import kxpu_b200 as K
    want = oracle.table_build(text)
    m = K.KxpuMulti(ordinals or [0] * nranks)
    bufs = []
    try:
        for rep in range(3):  # both exchange buffers and their clearing one epoch ahead
            shards = []
            nq = 0 if q is None else len(q)
            per = (nq + nranks - 1) // nranks if nq else 0
            for r, (a, b) in enumerate(K.plan_shards(text, nranks)):
                kx = m.ctxs[r]
                d = _aligned_upload(kx, text[a:b])
                sh = dict(d_text=d, n=b - a, global_base=a)
                bufs.append((kx, d))
                if nq:
                    lo, hi = min(r * per, nq), min((r + 1) * per, nq)
                    dq = _aligned_upload(kx, q[lo:hi].tobytes())
                    dr = kx.dev_alloc(max(nq * 4, 16))
                    kx.upload(dr, np.full(nq, -7, np.int32))
                    bufs += [(kx, dq), (kx, dr)]
                    sh.update(d_keys=dq, nq=hi - lo, key_offset=lo, d_rows_all=dr)
                shards.append(sh)
            tabs = m.pciids_join(shards, nq)
            first = None
            for r, t in enumerate(tabs):
                kx = m.ctxs[r]
                keys, offs, rows = kx.table_export(t)
                assert np.array_equal(keys, want["key"]) and np.array_equal(offs, want["line_off"]), (nranks, r, rep)
                names, _, _ = kx.names(t, rows[:200])
                for nm, o in zip(names, offs[:200]):
                    assert nm == oracle.row_name(text, int(o))
                if nq:
                    got = kx.download(shards[r]["d_rows_all"], nq * 4, np.int32)
                    line_of_row = np.full(t.rows + 1, -1, np.int64)
                    line_of_row[rows] = offs.astype(np.int64)
                    got_line = np.where(got >= 0, line_of_row[np.maximum(got, 0)], -1)
                    order = np.argsort(want["key"])
                    sk = want["key"][order]
                    pos = np.searchsorted(sk, q)
                    pos[pos >= max(len(sk), 1)] = 0
                    hit = (sk[pos] == q) if len(sk) else np.zeros(nq, bool)
                    exp = np.where(hit, want["line_off"][order][pos].astype(np.int64), -1) if len(sk) else np.full(nq, -1)
                    assert np.array_equal(got_line, exp), (nranks, r, rep)
                    # row handles are global: identical on every rank
                    if first is None:
                        first = got
                    assert np.array_equal(first, got)
            for t in tabs:
                t.free()
            for kx, d in bufs:
                kx.dev_free(d)
            bufs = []
    finally:
        m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nranks", [1, 2, 3, 8])
def test_sharded_load_and_join_on_one_gpu(nranks, oracle, pci_text, workloads, oracle_rows):
    """kxpu_ctx_create_multi with the same ordinal repeated: phase A (vendor_first all-reduce),
    phase B (winners-only push), the merge and the fused join + gather of hits all run, on any box."""
    q = workloads.make_queries(oracle_rows["key"], 5000, 17)
    _check_multi(oracle, pci_text, nranks, q)
    # first occurrence wins ACROSS shards: later shards hold only losers / hold earlier vendors' duplicates
    _check_multi(oracle, pci_text * 3, nranks, q)
    cut = pci_text.find(b"\n", 1400000) + 1
    _check_multi(oracle, pci_text[700000:cut] + pci_text, nranks, q[:1000])
    _check_multi(oracle, b"10de  NV\n\t0001  a\n10df  x\n\t0002  b\n" * 3, nranks,
                 np.array([0x10de0001, 0x10df0002, 0x10de0002, 5], np.uint32))
    _check_multi(oracle, b"", nranks)
    _check_multi(oracle, b"\tonly\n\tdevice lines\n", nranks)


@pytest.mark.gpu
def test_sharded_too_long_line_and_growth(oracle):
    """A >= 64 KiB line in one shard cuts every later shard off (bufio.ErrTooLong, global minimum of
    the shards' cut-offs); a text with more keys than the default table grows on every rank alike."""
    head = b"1111  one\n\t0001  a\n2222  two\n\t0002  b\n"
    long_line = b"3333  " + b"x" * 70000 + b"\n\t0003  hidden\n"
    tail = b"4444  four\n\t0004  also hidden\n" * 50
    q = np.array([0x11110001, 0x22220002, 0x33330003, 0x44440004], np.uint32)
    for nr in (2, 4):
        _check_multi(oracle, head * 200 + long_line + tail, nr, q)
    big = b"".join(b"%04x  V\n" % v + b"".join(b"\t%04x  d%d\n" % (d, d) for d in range(0, 2500, 7)) for v in range(0x100, 0x100 + 140))
    _check_multi(oracle, big, 3, np.array([0x01000000, 0x01010007, 0x018b09bd, 0x01000001], np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("no_p2p", ["0", "1"])
def test_two_gpu_process_per_rank(no_p2p):
    """One process per rank under torchrun: CUDA-IPC peer memory, and the NCCL transport (KXPU_NO_P2P=1)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs; the exchange itself is covered on one GPU above")
    env = dict(os.environ, KXPU_NO_P2P=no_p2p) if no_p2p == "1" else dict(os.environ)
    env.pop("KXPU_NO_P2P", None) if no_p2p == "0" else None
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29731", os.path.join(ROOT, "scripts", "multi_rank_check.py")],
                       capture_output=True, text=True, timeout=600, env=env)
    assert "MULTI_RANK_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
