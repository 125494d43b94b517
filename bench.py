#!/usr/bin/env python3
"""bench.py -- BASELINE.json metric "pci.ids parse GB/s; device lookups/sec" on B200.

Workload (config.workload): BASELINE.json configs[3] -- utils/pci.ids replicated x1000
(1 458 186 000 B of text) + a 2^20-key (vendor,device) join, first occurrence wins.
One step = parse the text into the (vendor,device) table and join the 2^20 keys against it:
  N = 1   one kxpu_pciids_join_device call (parse + resolve + finalize + join, one host round trip);
  N > 1   STRONG scaling (default): the SAME 1.458 GB text is cut into N shards at vendor lines
          (kxpu_plan_shards), the SAME 2^20 keys into N slices; one kxpu_pciids_join_sharded call per
          step: parse the shard, all-reduce(min) of the first anchors over NVSwitch peer memory, winners
          published per rank and pulled + inserted by every rank, probe of the key slice with the hits
          stored into every rank.
          A WEAK-scaling measurement (every rank its own x1000 shard of one logical x(1000*N) text and
          its own 2^20 keys) rides in the same line under "weak_scaling" (--scaling weak makes it the
          headline instead).

  value      text bytes consumed per second by the whole job, inputs resident in HBM,
             device-timed (CUDA events on the library's stream), max over ranks.
  e2e        same metric through the host side: pinned host text -> H2D, kernels, D2H of the row
             handles, every step (N = 1: kxpu_pciids_load + kxpu_lookup on host buffers).
  roofline   parse kernel: text bytes / mean kernel time vs the measured HBM copy bandwidth.
  parity     outside the timed region every rank's table and join result are compared with the
             oracle's table of the whole text (kxo_table_build on the 1.458 GB buffer, rank 0) and
             with each other ("parity_checked").
  aux        the other rows of the hot path, each with its own roofline: cfg2 (the real 1.4 MB pci.ids once +
             1024 keys: device time with inputs in HBM, and wall clock of ONE kxpu_pciids_join call on pinned
             host buffers -- zero-copy ingest, no cudaMemcpy), cfg3 classify, cfg5 CDI emit (JSON / YAML).
  cpu_best   the honest CPU comparator: single-pass build + binary-search join on 1 / physical / all threads.
  --impl reference   the reference's own algorithm (getDeviceName: one linear rescan of the
             text per key, pkg/device_plugin/device_plugin.go:208-275) restated in C
             (oracle/, Go toolchain absent), all host threads, bounded sample per step.
  --dump-outputs DIR   after the timed steps, rank 0 writes what the last timed step returned as
             float64 .npy files (same inputs on every run, so two builds compare file for file):
             table_key / table_line_off   the table in file order (kxpu_table_export),
             join_line_off                per key, the line offset of the row it hit (-1 = miss).
             Row handles are opaque numbers, so the join is written as the line each handle stands for.

The tree may be read-only: bench.py uses the libraries build() made and writes nothing there.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True  # no __pycache__ in the tree
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

COPIES = 1000
NQ = 1 << 20
METRIC = "pci.ids parse GB/s (x1000 text + 2^20-key join); device lookups/s reported beside it"


def workload_config(n_text):
    """Identical in both arms (ours / reference) and for every N: the job is the same job."""
    return {"workload": "cfg4: pci.ids x1000 (1 458 186 000 B) + 2^20-key join, first occurrence wins",
            "text_bytes": int(n_text), "keys": NQ,
            "l2": "input (1.458 GB) larger than L2 (126 MB); no flush needed"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(name="parse_kernel_traffic.json"):
    """dram bytes per launch of a kernel from the committed ncu capture, if any."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", name)))
        return d.get("dram_bytes_per_launch")
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.samples, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "window": "warm-up + settle steps + timed region, 100 ms period"}


try:
    ALL_CPUS = os.sched_getaffinity(0)  # before any NUMA binding: the CPU legs run on every core of the box
except Exception:
    ALL_CPUS = None


def host_threads():
    if ALL_CPUS is not None:
        return len(ALL_CPUS)
    return os.cpu_count() or 1


def use_all_cpus():
    """Undo the NUMA binding of this rank for the CPU comparators (they are threads of this process)."""
    if ALL_CPUS is not None:
        try:
            os.sched_setaffinity(0, ALL_CPUS)
        except Exception:
            pass


def bind_to_gpu_numa_node(gpu_index):
    """Run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA node its GPU hangs
    off: without it 8 ranks pin 1.46 GB each on whatever node the launcher started them on and half
    of the H2D traffic crosses the socket link.  Returns a short description for the JSON line."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if len(bus) > 12 and bus.startswith("0000"):
            bus = bus[4:]  # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return "numa_node -1 (single node)"
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = set(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed]
        if not cpus:
            return "node %d has no allowed cpu" % node
        os.sched_setaffinity(0, cpus)
        return "node %d (%d cpus)" % (node, len(cpus))
    except Exception as e:  # noqa: BLE001
        return "unbound (%s)" % type(e).__name__


def reference_sample(text_x, present_keys, n_keys, threads, seed):
    """One bounded sample of the reference algorithm on the x1000 text."""
    from kxpu_b200 import workloads as W
    from oracle import oracle as O
    keys = W.make_queries(present_keys, n_keys, seed)
    dt, scanned, _ = O.bench_scan(text_x, keys, threads)
    return dt, scanned, n_keys


def run_reference(args, rank, out_fd):
    """--impl reference: rank 0 alone times the CPU path; other ranks exit 0."""
    if rank != 0:
        return
    import kxpu_b200  # noqa: F401  (workloads only; no GPU context is created on this arm)
    from kxpu_b200 import workloads as W
    from oracle import oracle as O
    text = W.load_pci_ids()
    text_x = np.tile(np.frombuffer(text, np.uint8), COPIES)
    present = O.table_build(text)["key"]
    threads = host_threads()
    n_keys = max(threads * 4, 32)  # 1/8 of them miss on the vendor and rescan all 1.458 GB
    for w in range(args.warmup):
        reference_sample(text_x, present, max(threads, 8), threads, 100 + w)
    tot_t, tot_b, tot_k = 0.0, 0, 0
    for s in range(args.steps):
        dt, scanned, nk = reference_sample(text_x, present, n_keys, threads, 200 + s)
        tot_t += dt; tot_b += scanned; tot_k += nk
    scan_gbs = tot_b / tot_t / 1e9
    job_s = tot_t / tot_k * NQ  # time the reference needs for the whole job: one getDeviceName per key
    gbs = len(text) * COPIES / job_s / 1e9  # same meaning as the GPU arm's value: job text bytes / job time
    line = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": tot_t / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(len(text) * COPIES),
        "sample_keys_per_step": n_keys,
        "lookups_per_s": tot_k / tot_t,
        "scan_gbs": scan_gbs,  # text bytes the scanners consumed per second (the reference re-reads the text per key)
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "port", "scan_gbs": scan_gbs,
                         "sample": "%d of the 2^20 cfg4 keys per step (same hit/miss mix); each key is one literal "
                                   "getDeviceName rescan of the x1000 text (C restatement of the Go reference; Go "
                                   "toolchain absent); value = job text bytes / (sample time x 2^20 / sample keys); "
                                   "scan_gbs = bytes the scanners actually consumed per second" % n_keys},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_line(out_fd, line)


def emit_line(fd, obj):
    os.write(fd, (json.dumps(obj) + "\n").encode())


def expected_lines(orows, q):
    """line offset the oracle's table gives for every key (-1 = miss)."""
    order = np.argsort(orows["key"])
    sk = orows["key"][order]
    pos = np.searchsorted(sk, q)
    pos[pos >= len(sk)] = 0
    hit = sk[pos] == q
    return np.where(hit, orows["line_off"][order][pos].astype(np.int64), -1)


def main():
    # Libraries (NCCL's version banner, for one) print to stdout; the contract is ONE JSON line on
    # stdout, so everything else is sent to stderr and the line is written to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"], help="headline measurement at N > 1")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true")
    ap.add_argument("--no-second-mode", action="store_true", help="N > 1: measure only --scaling, not the other mode beside it")
    ap.add_argument("--settle-ms", type=float, default=400.0,
                    help="untimed extra warm-up (clock settling + nvidia-smi samples); the step count is reported in the line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, real_stdout)
        return

    import kxpu_b200 as K
    from kxpu_b200 import workloads as W
    B = K.binding

    numa = bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    kx = K.Kxpu(local_rank)  # raises without a B200: there is no CPU fallback
    text = W.load_pci_ids()
    n1 = len(text)
    n = n1 * COPIES

    # the whole logical text in pinned host memory (source of the e2e copies and of the shard plan)
    h_text, h_ptr = kx.pinned(n)
    h_text.reshape(COPIES, n1)[:] = np.frombuffer(text, np.uint8)

    def max_over_ranks(x):
        if dist is None:
            return float(x)
        import torch
        v = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        return float(v.item())

    def barrier():
        kx.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    if world > 1:
        import torch
        uid = torch.zeros(B.COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.from_numpy(kx.comm_unique_id()))
        dist.broadcast(uid, 0)
        kx.comm_init(world, rank, uid.cpu().numpy())

    # present keys (for the query mix): the same on every rank, from the product's own table of one copy
    t1 = kx.pciids_load(np.frombuffer(text, np.uint8))
    present, _, _ = kx.table_export(t1)
    t1.free()
    keys = W.make_queries(present, NQ, 2)  # ONE logical key array (cfg4, seed 2)

    # ---------------------------------------------------------------- workloads
    def make_strong():
        """The same 1.458 GB text cut into `world` shards, the same keys into `world` slices."""
        a, b = K.plan_shards(h_text, world)[rank]
        per = NQ // world
        lo, hi = rank * per, (rank + 1) * per if rank + 1 < world else NQ
        d_text = kx.dev_alloc(max(b - a, 16))
        kx.upload(d_text, h_text[a:b])
        d_keys = kx.dev_alloc((hi - lo) * 4)
        kx.upload(d_keys, keys[lo:hi])
        d_rows = kx.dev_alloc(NQ * 4)
        w = dict(kind="strong", d_text=d_text, n=b - a, base=a, d_keys=d_keys, nq=hi - lo, key_off=lo, d_rows=d_rows,
                 h_src=h_text[a:b], h_keys=keys[lo:hi], job_bytes=n, h_rows=np.empty(NQ, np.int32))
        if world == 1:
            w["step"] = lambda: kx.pciids_join_device(d_text, n, d_keys, NQ, d_rows)
        else:
            w["step"] = lambda: kx.pciids_join_sharded(d_text, b - a, a, d_keys, hi - lo, lo, NQ, d_rows)
        w["load"] = (lambda: kx.pciids_load_device(d_text, n)) if world == 1 else (lambda: kx.pciids_load_sharded(d_text, b - a, a))
        return w

    def make_weak():
        """Every rank its own x1000 shard of one logical x(1000*world) text and its own 2^20 keys."""
        d_text = kx.dev_alloc(n)
        kx.upload(d_text, h_text)
        my_keys = W.make_queries(present, NQ, 2 + rank)
        d_keys = kx.dev_alloc(NQ * 4)
        kx.upload(d_keys, my_keys)
        d_rows = kx.dev_alloc(NQ * 4)

        def step():
            t = kx.pciids_load_sharded(d_text, n, rank * n)
            kx.lookup_device(t, d_keys, NQ, d_rows)
            return t
        return dict(kind="weak", d_text=d_text, n=n, base=rank * n, d_keys=d_keys, nq=NQ, key_off=0, d_rows=d_rows,
                    h_src=h_text, h_keys=my_keys, job_bytes=world * n, step=step, h_rows=np.empty(NQ, np.int32),
                    load=lambda: kx.pciids_load_sharded(d_text, n, rank * n))

    def free_workload(w):
        for k in ("d_text", "d_keys", "d_rows"):
            kx.dev_free(w[k])

    def step_result(t, d_rows):
        """The table of a step in file order, the row handles of all NQ keys and the line offset each
        handle stands for (-1 = miss)."""
        tk, to, tr = kx.table_export(t)
        got = kx.download(d_rows, NQ * 4, np.int32)
        line_of_row = np.full(t.rows + 1, -1, np.int64)
        line_of_row[tr] = to.astype(np.int64)
        return tk, to, got, np.where(got >= 0, line_of_row[np.maximum(got, 0)], -1)

    def measure(w, steps, warmup, settle_ms, sampler=None, keep_outputs=False):
        """Device-timed K steps (max over ranks) + per-kernel device times from separate passes.
        keep_outputs: also return what the last timed step computed (read after the timer stops)."""
        for _ in range(warmup):
            w["step"]().free()
        kx.sync()
        t0 = time.time()
        w["step"]().free()
        kx.sync()
        one = max(time.time() - t0, 1e-5)
        settle = int(max_over_ranks(min(settle_ms * 1e-3 / one, 5000)))  # same count on all ranks
        for _ in range(settle):
            w["step"]().free()
        barrier()
        launches0 = kx.launch_count()
        kx.set_stage_timing(False)  # the per-stage events are for the separate per-kernel passes below
        kx.timer_begin()
        t_wall = time.time()
        for _ in range(steps - 1):
            w["step"]().free()
        last = w["step"]()
        ms_total = kx.timer_end()
        kx.set_stage_timing(True)
        barrier()
        wall_ms = (time.time() - t_wall) * 1e3
        outputs = None
        if keep_outputs:
            tk, to, _, got_line = step_result(last, w["d_rows"])
            outputs = {"table_key": tk, "table_line_off": to, "join_line_off": got_line}
        last.free()
        launches = kx.launch_count() - launches0
        clocks = sampler.stop() if sampler is not None else None
        km = {k: [] for k in ("parse", "parse_resolve", "finalize", "merge", "lookup")}
        for _ in range(min(steps, 10)):
            t = w["load"]()  # the load half of the step (N > 1: collective), then the join of this rank's keys
            tm = kx.timings()
            km["parse"].append(tm[B.T_PARSE]); km["parse_resolve"].append(tm[B.T_RESOLVE]); km["finalize"].append(tm[B.T_FINALIZE])
            km["merge"].append(tm[B.T_MERGE])
            kx.lookup_device(t, w["d_keys"], w["nq"], w["d_rows"])
            km["lookup"].append(kx.timings()[B.T_LOOKUP])
            t.free()
        ms_step = max_over_ranks(ms_total) / steps
        return dict(ms_per_step=ms_step, value=w["job_bytes"] / (ms_step * 1e-3) / 1e9, wall_ms_per_step=wall_ms / steps,
                    launches=int(launches), settle_steps=settle, clocks=clocks,
                    kernel_ms={k: float(np.mean(v)) for k, v in km.items()}, outputs=outputs)

    def measure_e2e(w, steps):
        """The same step from HOST buffers: pinned text (shard) -> H2D, kernels, D2H of the row handles."""
        ms = []
        for i in range(1 + steps):
            barrier()
            t0 = time.time()
            if world == 1:
                t = kx.pciids_load(w["h_src"])
                rows = kx.lookup(t, w["h_keys"])
            else:
                kx.upload(w["d_text"], w["h_src"])
                kx.upload(w["d_keys"], w["h_keys"])
                t = w["step"]()
                rows = kx.download(w["d_rows"], NQ * 4, np.int32)
            barrier()
            if i > 0:
                ms.append((time.time() - t0) * 1e3)
            t.free()
        e2e_step = max_over_ranks(float(np.mean(ms)))
        h2d = int(len(w["h_src"]) + 4 * len(w["h_keys"]))
        return dict(value=w["job_bytes"] / (e2e_step * 1e-3) / 1e9, unit="GB/s", h2d_bytes_per_step=h2d,
                    d2h_bytes_per_step=int(4 * NQ), ms_per_step=e2e_step, rows=rows)

    def check_parity(w):
        """Every rank: table hash + join result vs the oracle's table of the WHOLE text (rank 0 builds it
        with kxo_table_build on the 1.458 GB buffer, outside every timed region)."""
        t = w["step"]()
        tk, to, got, got_line = step_result(t, w["d_rows"])
        t.free()
        ok, detail = True, {}
        if w["kind"] == "strong":
            if rank == 0:
                from oracle import oracle as O
                t0 = time.time()
                orows = O.table_build(h_text)
                detail["oracle_s"] = time.time() - t0
                ok = bool(np.array_equal(tk, orows["key"]) and np.array_equal(to, orows["line_off"]))
                ok = ok and bool(np.array_equal(got_line, expected_lines(orows, keys)))
                detail["rows"] = int(len(orows)); detail["hits"] = int((got >= 0).sum())
        else:  # weak: the logical text is x(1000*world); first occurrence wins -> the single-copy table; own keys
            from oracle import oracle as O
            orows = O.table_build(text)
            ok = bool(np.array_equal(tk, orows["key"]) and np.array_equal(to, orows["line_off"]))
            ok = ok and bool(np.array_equal(got_line, expected_lines(orows, w["h_keys"])))
        if dist is not None:
            import torch
            hv = int(np.bitwise_xor.reduce(tk.astype(np.uint64) * np.uint64(31) + to)) & 0x7FFFFFFFFFFFFFFF
            if w["kind"] == "strong":
                hv ^= int(np.bitwise_xor.reduce(got.astype(np.int64).view(np.uint64) * np.arange(1, NQ + 1, dtype=np.uint64))) & 0x7FFFFFFFFFFFFFFF
            h = torch.tensor([hv, 1 if ok else 0], dtype=torch.int64, device="cuda")
            hs = [torch.zeros_like(h) for _ in range(world)]
            dist.all_gather(hs, h)
            ok = all(int(x[0].item()) == int(hs[0][0].item()) for x in hs) and all(int(x[1].item()) == 1 for x in hs)
            detail["identical_on_all_ranks"] = all(int(x[0].item()) == int(hs[0][0].item()) for x in hs)
        return ok, detail

    # ---------------------------------------------------------------- headline + second measurement
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    modes = [args.scaling] + ([("weak" if args.scaling == "strong" else "strong")] if world > 1 and not args.no_second_mode else [])
    results = {}
    for i, mode in enumerate(modes):
        w = make_strong() if mode == "strong" else make_weak()
        r = measure(w, args.steps, args.warmup, args.settle_ms, sampler if (i == 0 and rank == 0) else None,
                    keep_outputs=bool(args.dump_outputs) and i == 0 and rank == 0)
        r["e2e"] = measure_e2e(w, args.e2e_steps)
        r["e2e"].pop("rows")
        ok, detail = check_parity(w)
        r["parity_checked"], r["parity"] = ok, detail
        # the join alone (kernel time, and through the host-buffer ABI)
        t = w["load"]()
        look, lk_ms = [], []
        for j in range(6):
            kx.lookup_device(t, w["d_keys"], w["nq"], w["d_rows"])
            look.append(kx.timings()[B.T_LOOKUP])
            barrier()
            t0 = time.time()
            kx.lookup(t, w["h_keys"])
            if j > 0:
                lk_ms.append((time.time() - t0) * 1e3)
        t.free()
        r["lookup_kernel_ms"], r["lookup_host_ms"], r["nq_rank"] = float(np.mean(look[1:])), float(np.mean(lk_ms)), w["nq"]
        r["shard_bytes"] = int(w["n"])
        results[mode] = r
        if i + 1 < len(modes) or world > 1:
            free_workload(w)
        else:
            results["_w"] = w
    head = results[args.scaling]
    if head["outputs"] is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in head["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a.astype(np.float64))

    line = None
    if rank == 0:
        peak, peak_src = measured_peak()
        pk = head["kernel_ms"]["parse"]
        shard_bytes = head["shard_bytes"]
        achieved = shard_bytes / (pk * 1e-3) / 1e9
        km = dict(head["kernel_ms"])
        stages = {k: v for k, v in km.items()}
        limiting = max(stages, key=lambda k: stages[k])
        line = {
            "metric": METRIC, "value": head["value"], "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "settle_steps": head["settle_steps"], "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(n),
            "parallelism": ("1 GPU" if world == 1 else
                            "%s: text cut at vendor lines into %d shards, keys into %d slices; peer-memory exchange over NVSwitch"
                            % (args.scaling, world, world)),
            "shard_bytes_rank0": shard_bytes,
            "lookups_per_s": world * head["nq_rank"] / (head["lookup_kernel_ms"] * 1e-3),
            "lookups_per_s_e2e": world * head["nq_rank"] / (head["lookup_host_ms"] * 1e-3),
            "lookups_note": "kernel alone on rank 0's slice; keys + rows (8 B/key) are L2 resident after the first pass, "
                            "the table (2.6 MB) always is: a throughput figure, not an HBM roofline",
            "kernel_ms": km, "limiting_stage": limiting,
            "kernel_ms_note": "device time per stage on rank 0 from separate passes with per-stage CUDA events; "
                              "merge = wait for phase A .. insert of the winners (contains the finalize of the winners and the waits for the slowest rank)",
            "wall_ms_per_step": head["wall_ms_per_step"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic() if world == 1 else None, "peak_source": peak_src,
                         "kernel": "kxparse5::parse_kernel_v5", "algorithmic_bytes_per_launch": shard_bytes},
            "e2e": dict(head["e2e"], numa=numa,
                        note="PCIe bound: every rank copies its shard from pinned host memory each step "
                             "(Gen5 x16 ~ 55-57 GB/s per GPU in practice, ~64 GB/s nominal)"),
            "parity_checked": bool(head["parity_checked"]), "parity": head["parity"],
            "gpu_launches": head["launches"],
            "clocks": head["clocks"],
        }
        other = [m for m in modes if m != args.scaling]
        if other:
            o = results[other[0]]
            line[other[0] + "_scaling"] = {
                "value": o["value"], "unit": "GB/s", "ms_per_step": o["ms_per_step"], "kernel_ms": o["kernel_ms"],
                "job_bytes": int(n * world if other[0] == "weak" else n), "e2e": o["e2e"], "gpu_launches": o["launches"],
                "parity_checked": bool(o["parity_checked"]), "settle_steps": o["settle_steps"],
                "note": ("every rank parses its own x1000 shard (1.458 GB) of one logical x(1000*N) text and joins its own 2^20 keys"
                         if other[0] == "weak" else "the fixed 1.458 GB text over N shards, 2^20 keys over N slices")}
    if world == 1:
        w = results["_w"]
        if rank == 0 and not args.no_aux:
            line["aux"] = aux_configs(kx, K, W, text, present, peak)
        if rank == 0 and not args.no_cpu_baseline:
            from oracle import oracle as O
            use_all_cpus()
            threads = host_threads()
            nk = max(threads * 16, 64)  # ~10 s wall on all host cores
            dt, scanned, _ = reference_sample(h_text, present, nk, threads, 300)
            line["cpu_baseline"] = {
                "value": n / (dt / nk * NQ) / 1e9, "unit": "GB/s", "cores": threads, "kind": "port",
                "lookups_per_s": nk / dt, "scan_gbs": scanned / dt / 1e9,
                "sample": "%d of the 2^20 cfg4 keys (same mix), literal getDeviceName rescans of the x1000 text "
                          "(C restatement of the Go reference; Go toolchain absent), %.1f s wall on all host threads; value = job "
                          "text bytes / (sample time x 2^20 / sample keys); scan_gbs = bytes the scanners consumed "
                          "per second (the reference re-reads the text for every key)" % (nk, dt)}
            best = []
            for th in sorted({1, max(1, threads // 2), threads}):  # one core, one thread per physical core, every hardware thread
                dtb, parse_s, offs = O.bench_parse_mt(h_text, keys, th)
                best.append({"cores": th, "parse_gbs": n / parse_s / 1e9, "job_gbs": n / dtb / 1e9, "job_s": dtb})
            top = max(best, key=lambda r: r["job_gbs"])
            line["cpu_best"] = {"runs": best, "job_gbs_all_cores": top["job_gbs"], "cores": top["cores"],
                                "note": "honest best CPU on the SAME job: single pass per thread over vendor-line shards "
                                        "(dead blocks skipped like on the GPU), first anchors min-merged, 2^20 binary-search "
                                        "probes on all threads; host memory only, no PCIe -- compare with e2e.value"}
        free_workload(w)
    if rank == 0:
        emit_line(real_stdout, line)
    kx.pinned_free(h_ptr)
    if dist is not None:
        kx.comm_destroy()
        dist.destroy_process_group()
    kx.close()


def aux_configs(kx, K, W, text, present, peak):
    """The other rows of the hot path (SURVEY.md 8(d) cfg2 / cfg3 / cfg5) through the host-buffer ABI; device
    time of their kernels from the library's CUDA events; each with its own roofline.  Not part of `value`."""
    B = K.binding
    recs = W.cfg3_records(present)
    devs = W.cfg5_devices()
    cls_ms, emit_j_ms, emit_y_ms = [], [], []
    for _ in range(5):
        res = kx.classify(recs)
        cls_ms.append(kx.timings()[B.T_CLASSIFY])
        j = kx.cdi_emit(B.FMT_JSON, devs)
        emit_j_ms.append(kx.timings()[B.T_EMIT])
        y = kx.cdi_emit(B.FMT_YAML, devs)
        emit_y_ms.append(kx.timings()[B.T_EMIT])
    # configs[1] (cfg2): the real utils/pci.ids once + 1024 lookups -- latency, not bandwidth.
    #   device: text and keys resident in HBM, kxpu_pciids_join_device = ONE cooperative kernel (parse, fold, names,
    #           join), device time of that kernel;
    #   e2e:    ONE kxpu_pciids_join call on pinned host buffers, wall clock: zero-copy ingest -- the same kernel pulls
    #           the text over PCIe in its first phase and writes row handles + counters to host memory, nothing is
    #           copied by the host (its device time is reported as kernel_us_inside_e2e_call).
    q2v = W.cfg2_queries(present)
    one, p_one = kx.pinned(len(text))            # the host program reads /usr/pci.ids into a pinned buffer
    one[:] = np.frombuffer(text, np.uint8)
    q2, p_q2 = kx.pinned(len(q2v) * 4, np.uint32)
    q2[:] = q2v
    r2, p_r2 = kx.pinned(len(q2v) * 4, np.int32)
    d_one, d_q2, d_r2 = kx.dev_alloc(len(text)), kx.dev_alloc(len(q2v) * 4), kx.dev_alloc(len(q2v) * 4)
    kx.upload(d_one, text)
    kx.upload(d_q2, q2v)
    c2_dev, c2_e2e, c2_kin = [], [], []
    for i in range(10):
        t = kx.pciids_join_device(d_one, len(text), d_q2, len(q2v), d_r2)
        tm = kx.timings()
        t.free()
        if i > 2:
            c2_dev.append((tm[B.T_PARSE] + tm[B.T_RESOLVE] + tm[B.T_FINALIZE] + tm[B.T_LOOKUP]) * 1e3)
    for i in range(8):
        t, rows2 = kx.pciids_join(one, q2, rows_out=r2)
        tm = kx.timings()
        t.free()
        if i > 2:
            c2_kin.append((tm[B.T_PARSE] + tm[B.T_RESOLVE] + tm[B.T_FINALIZE] + tm[B.T_LOOKUP]) * 1e3)
    kx.set_stage_timing(False)  # the wall-clock figure is taken as a C / cgo host would see it: no per-stage events,
    call = kx.pciids_join_call(one, q2, r2)  # arguments marshalled once (numpy / ctypes cost ~7 us per call otherwise)
    for i in range(16):
        t0 = time.perf_counter()
        h = call()
        dt = (time.perf_counter() - t0) * 1e6
        kx.table_free_handle(h)
        if i > 2:
            c2_e2e.append(dt)
    rows2 = r2
    kx.set_stage_timing(True)
    for d in (d_one, d_q2, d_r2):
        kx.dev_free(d)
    hits2 = int((rows2 >= 0).sum())
    for p in (p_one, p_q2, p_r2):
        kx.pinned_free(p)

    def roof(alg_bytes, ms, kernel):
        a = alg_bytes / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak, "kernel": kernel,
                "algorithmic_bytes_per_launch": int(alg_bytes), "traffic": None}
    cm, jm, ym = float(np.min(cls_ms[1:])), float(np.min(emit_j_ms[1:])), float(np.min(emit_y_ms[1:]))
    return {
        "cfg2_pci_ids_once": {"text_bytes": len(text), "lookups": int(len(q2v)), "hits": hits2,
                              "device_us_parse_resolve_finalize_join": float(np.min(c2_dev)),
                              "e2e_us_host_text_to_rows": float(np.min(c2_e2e)),
                              "kernel_us_inside_e2e_call": float(np.min(c2_kin)),
                              "h2d_bytes": int(len(text) + 4 * len(q2v)), "d2h_bytes": int(4 * len(q2v)),
                              "host_buffers": "pinned, read / written by the kernel itself (zero-copy), no cudaMemcpy",
                              "note": "device: inputs in HBM, one cooperative kernel (three grid barriers); e2e: wall clock "
                                      "around the bare kxpu_pciids_join C call (arguments marshalled once, as a C / cgo "
                                      "host calls it).  1.4 MB is launch / latency bound: far below the roofline by "
                                      "construction"},
        "cfg3_classify": {"records": len(recs), "accepted": int(res["n_accepted"]), "kernel_ms": cm,
                          "records_per_s": len(recs) / (cm * 1e-3),
                          "roofline": roof(len(recs) * 68, cm, "classify kernels (64 B record read + 4 B busIndex write)")},
        "cfg5_cdi_json": {"devices": len(devs), "bytes": len(j), "kernel_ms": jm,
                          "roofline": roof(len(j) + 32 * len(devs), jm, "kxemit (output bytes + 32 B record read)")},
        "cfg5_cdi_yaml": {"devices": len(devs), "bytes": len(y), "kernel_ms": ym,
                          "roofline": roof(len(y) + 32 * len(devs), ym, "kxemit (output bytes + 32 B record read)")},
    }


if __name__ == "__main__":
    main()
