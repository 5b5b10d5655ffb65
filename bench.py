#!/usr/bin/env python
"""bench.py -- the measurement contract.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload all|q6|sum|q1|bruteforce|ivf|dropin]
                    [--dump-outputs DIR]

The default run covers ALL FIVE BASELINE.json configs in one JSON line.  The headline (top-level keys) is config 2, TPC-H Q6
(3-predicate filter + SUM, fp64) over SF100 synthetic lineitem columns (600 037 902 rows, 28 B/row = 16.8 GB) on one B200; the other
configs are under "workloads": sum (config 1), q1 (config 3), bruteforce (config 4), ivf (config 5), plus "dropin" (what one
8192-row block costs through the C-ABI from host pointers).  Every workload carries

  value        whole-job throughput, inputs RESIDENT in HBM when the timed region starts (CUDA events, max over ranks).  A step is
               ONE pass of the hot path: kernel -> partial record in device memory -> (N > 1: NCCL all_gather on the same stream ->
               merge kernel) -> asynchronous D2H of the final record.  Nothing synchronises inside the timed region.
  e2e          the same metric through the C-ABI call with HOST buffers (pinned; a pageable figure is reported next to it):
               H2D copies inside the timed region
  roofline     algorithmic bytes (or flop) per launch / CUDA-event duration of the dominant kernel, against MEASURED_PEAKS.json
  cpu_baseline the oracle port (C restatement of the Go operator chain) on the host cores, bounded sample, median of 5
  parity       GPU result vs the oracle on the same rows / queries, computed in this run
  --impl reference   times that CPU implementation alone (rank 0), same metric / config / unit
  --dump-outputs DIR writes what the last timed step of each workload returned to its caller as DIR/<workload>_<name>.npy (rank 0), so that
                     two builds can be compared output for output: the inputs are seeded, identical from run to run

Multi-GPU (one process per GPU, torchrun): q6 and sum are WEAK scaling (every rank owns an SF100-sized / 10 M-row disjoint block range),
q1 is STRONG scaling of ONE SF100 table (shard.block_range, BASELINE config 3), bruteforce shards the 1 M rows, ivf shards the
10 M-row index (config 5) over the ranks.  The exchange (MergeGroup / MergeTop) stays on the device.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SF100_ROWS = 600_037_902
WORKLOADS = {
    "q6": dict(name="tpch_q6_sf100_fp64", metric="scan+filter+agg rows/sec (TPC-H Q6, fp64)", bytes_per_row=28.0, rows=SF100_ROWS, unit="rows/s", dtype="f64", scaling="weak"),
    "q1": dict(name="tpch_q1_sf100_fp64_packed_keys", metric="scan+filter+group-agg rows/sec (TPC-H Q1, fp64)", bytes_per_row=38.0, rows=SF100_ROWS, unit="rows/s", dtype="f64", scaling="strong"),
    "sum": dict(name="int64_sum_10m_rows", metric="int64 SUM rows/sec", bytes_per_row=8.0, rows=10_000_000, unit="rows/s", dtype="int64", scaling="weak"),
    "bruteforce": dict(name="bruteforce_l2_top10_1Mx768_10k_queries", metric="ANN top-k qps (768-d, brute-force L2 top-10)", bytes_per_row=None, rows=1_000_000, unit="queries/s", dtype="f32", scaling="strong"),
    "ivf": dict(name="ivfflat_l2_top10_10Mx768_nlist1024_nprobe32_10k_queries", metric="ANN top-k qps (768-d, IVF-flat nlist=1024 nprobe=32 top-10)", bytes_per_row=None, rows=10_000_000, unit="queries/s", dtype="f32", scaling="strong"),
    "dropin": dict(name="xcall_go_arith_int64_block8192_host_pointers", metric="rows/sec of one 8192-row block through XCall from host pointers", bytes_per_row=24.0, rows=8192, unit="rows/s", dtype="int64", scaling="weak"),
}
ALL = ["q6", "sum", "q1", "bruteforce", "ivf", "dropin"]
CPU_SAMPLE_ROWS = 1 << 25


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def mem_available():
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                return int(ln.split()[1]) * 1024
    except Exception:
        pass
    return 0


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md recipe); one process per bench run, sliced per workload"""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def window(self, t_begin, t_end):
        """samples whose timestamp lies in [t_begin, t_end] (wall clock)"""
        import datetime
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        sm, mx, reasons = [], [], set()
        for ln in list(self.lines):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if ts < t_begin - 0.02 or ts > t_end + 0.02:
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    out = {"hbm": (6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"), "bf16": (1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s)")}
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            out["hbm"] = (float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)")
            out["bf16"] = (float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst: the kernel is timed alone)")
        except Exception:
            pass
    return out


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set full` capture of
    this workload at this size (profiles/ncu_traffic.json, written by tools/summarize_ncu.py from the .ncu-rep); None if no capture"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = d.get(key)
        return (float(e["bytes_per_launch"]), e.get("source")) if e else (None, None)
    except Exception:
        return None, None


DUMP_ARRAY_BYTES = 8 << 20     # per array: every workload together stays far below 64 MB


def dump_outputs(out_dir, arrays):
    """name -> array, written as out_dir/<name>.npy in float32 (float32 arrays) or float64.  64-bit integers that float64 cannot hold
    exactly become [..., (high 32 bits, low 32 bits)].  An array above DUMP_ARRAY_BYTES keeps a fixed, seeded sample of its rows, whose
    indices go to <name>_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype.kind in "iub" and a.dtype.itemsize == 8 and a.size and (int(a.max()) >= 2 ** 53 or int(a.min()) <= -2 ** 53):
            w = a.view(np.uint64)
            a = np.stack([w >> np.uint64(32), w & np.uint64(0xFFFFFFFF)], axis=-1)
        a = a if a.dtype == np.float32 else a.astype(np.float64)
        if a.nbytes > DUMP_ARRAY_BYTES:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], max(1, DUMP_ARRAY_BYTES * a.shape[0] // a.nbytes), replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def median_time(fn, reps=5, warm=1):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), ts


# =====================================================================================================================
# CPU legs: the oracle port on the host cores (cpu_baseline of our arm, and the whole --impl reference arm)
# =====================================================================================================================
class CpuData:
    """host copies of the sample the CPU leg runs on.  `src` = None: generated by the oracle's own C generators (the --impl reference
    arm must not load the GPU library); else a dict of numpy arrays downloaded from the GPU's own buffers"""
    pass


def cpu_q6(cols, n, threads, reps=5):
    import oracle_lib as O
    from matrixone_b200 import datagen
    P = datagen.q6_params()
    res = {}
    def fn():
        res["r"] = O.q6(cols, n, P, nthreads=threads)
    sec, ts = median_time(fn, reps)
    return n / sec, sec, res["r"]


def cpu_q1(cols, n, threads, reps=5):
    import oracle_lib as O
    from matrixone_b200 import datagen
    res = {}
    def fn():
        res["r"] = O.q1(cols, n, datagen.Q1_CUTOFF, nthreads=threads)
    sec, ts = median_time(fn, reps)
    return n / sec, sec, res["r"]


def cpu_sum(col, n, threads, reps=5):
    import oracle_lib as O
    s = np.zeros(1, dtype=np.int64); nul = np.zeros(1, dtype=np.uint8)
    def fn():
        O.go().og_sum_int64_mt(O.p(col), None, n, threads, O.p(s), O.p(nul))
    sec, ts = median_time(fn, reps)
    return n / sec, sec, int(s[0])


def cpu_bruteforce(ds, qs, threads, reps=3):
    """GoBruteForceIndex.Search on the FULL dataset (per-query work must not shrink), queries spread over the host threads"""
    import oracle_lib as O
    res = {}
    def fn():
        res["r"] = O.bruteforce(ds, qs, 10, 0, threads)
    sec, ts = median_time(fn, reps, warm=0)
    return qs.shape[0] / sec, sec, res["r"]


def cpu_ivf(ents, assign, cents, qs, threads, reps=3):
    """IvfflatSearchIndex.Search (findCentroids + scan of the nprobe probed lists + heap), nlist 1024, nprobe 32, top-10"""
    import oracle_lib as O
    nq, k = qs.shape[0], 10
    keys = np.zeros(nq * k, dtype=np.int64); dists = np.zeros(nq * k)
    def fn():
        O.go().og_ivf_search_f32(O.p(ents), O.p(assign), ents.shape[0], ents.shape[1], O.p(cents), cents.shape[0], O.p(qs), nq, 32, k, 0, 0, threads, O.p(keys), O.p(dists))
    sec, ts = median_time(fn, reps, warm=0)
    return nq / sec, sec, (keys, dists)


def cpu_dropin(threads, reps=200):
    """the Go loop of one 8192-row int64 `a + b` batch with overflow check (opBinaryFixedFixedToFixedWithErrorCheck), one core"""
    import oracle_lib as O
    n = 8192
    a = O.gen_int64(1, 0, n, 1); b = O.gen_int64(2, 0, n, 1); r = np.zeros(n, dtype=np.int64)
    rn = np.zeros(n // 64, dtype=np.uint64); err = np.zeros(1, dtype=np.int64)
    def fn():
        O.go().og_arith(0, 23, O.p(r), O.p(a), O.p(b), n, 0, 0, None, None, O.p(rn), 0, O.p(err))
    for _ in range(20):
        fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    sec = (time.perf_counter() - t0) / reps
    return n / sec, sec, None


def cpu_leg_generated(workload, threads, steps, warmup, full_ivf=True):
    """--impl reference arm: data from the oracle's C generators (first-touched by the worker pool), then the timed passes"""
    import oracle_lib as O
    from matrixone_b200 import datagen
    if workload in ("q6", "q1"):
        n = CPU_SAMPLE_ROWS
        cols = O.gen_lineitem(10, 0, n, threads)
        value, sec, _ = (cpu_q6 if workload == "q6" else cpu_q1)(cols, n, threads, reps=max(5, steps))
        return value, sec, "first %d rows of the SF100 table per step; oracle/oracle_go.c operator chain (filter conjunct by conjunct + Shrink, projection, aggexec fill) on a persistent pool of %d pinned pthreads over 8192-row blocks; median of %d passes" % (n, threads, max(5, steps))
    if workload == "sum":
        n = WORKLOADS["sum"]["rows"]
        col = O.gen_int64(1, 0, n, threads)
        value, sec, _ = cpu_sum(col, n, threads, reps=max(5, steps))
        return value, sec, "all %d rows per step; oracle/oracle_go.c og_sum_int64_mt on %d pinned pthreads; median of %d passes" % (n, threads, max(5, steps))
    if workload == "bruteforce":
        n, dim = WORKLOADS["bruteforce"]["rows"], 768
        ds = O.gen_vectors_f32(20, 0, n, dim, threads)
        qs = O.gen_vectors_f32(21, 0, threads, dim, threads)
        value, sec, _ = cpu_bruteforce(ds, qs, threads, reps=min(3, max(1, steps)))
        return value, sec, "full 1 M x 768 dataset, %d queries per step (one per host thread); oracle/oracle_go.c GoBruteForceIndex.Search (metric.L2DistanceSq + FastMaxHeap)" % threads
    if workload == "ivf":
        dim, nlist = 768, 1024
        n = WORKLOADS["ivf"]["rows"]
        if not full_ivf or mem_available() < 1.6 * n * dim * 4:
            n = n // 8
        cents = O.gen_vectors_f32(30, 0, nlist, dim, threads) * np.float32(4.0)
        ents, assign = O.gen_vectors_f32(31, 0, n, dim, threads, cents, 1.0, True)   # the generating component: a valid list assignment
        qs = O.gen_vectors_f32(32, 0, 8 * threads, dim, threads, cents, 1.0)
        value, sec, _ = cpu_ivf(ents, assign, cents, qs, threads, reps=min(3, max(1, steps)))
        return value, sec, "%d x 768 index (nlist 1024, nprobe 32, top-10), %d queries per step over %d host threads; oracle/oracle_go.c og_ivf_search_f32 (IvfflatSearchIndex.Search)" % (n, 8 * threads, threads)
    if workload == "dropin":
        value, sec, _ = cpu_dropin(threads)
        return value, sec, "one 8192-row int64 a+b batch with overflow check per step, 1 core; oracle/oracle_go.c og_arith (opBinaryFixedFixedToFixedWithErrorCheck)"
    raise SystemExit("unknown workload " + workload)


def run_reference_arm(args):
    if env_int("RANK", 0) != 0:
        return 0
    threads = os.cpu_count() or 1
    names = ALL if args.workload == "all" else [args.workload]
    lines = {}
    for w in names:
        wl = WORKLOADS[w]
        try:
            value, sec, sample = cpu_leg_generated(w, threads, args.steps, args.warmup)
            cores = 1 if w == "dropin" else threads
            lines[w] = {"impl": "reference", "metric": wl["metric"], "value": value, "unit": wl["unit"], "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic",
                        "config": {"workload": wl["name"]},
                        "cpu_baseline": {"value": value, "unit": wl["unit"], "cores": cores, "kind": "port", "sample": sample},
                        "e2e": {"value": value, "unit": wl["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        except Exception as ex:
            lines[w] = {"impl": "reference", "metric": wl["metric"], "error": str(ex)[:200]}
    head = lines[names[0]]
    if len(names) > 1:
        head = dict(head)
        head["workloads"] = {w: lines[w] for w in names[1:]}
    print(json.dumps(head))
    return 0


# =====================================================================================================================
# our arm
# =====================================================================================================================
class Env:
    def __init__(self, args):
        self.args = args
        self.rank, self.world, self.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        os.environ.setdefault("MO_B200_DEVICE", str(self.local))
        from matrixone_b200 import capi, datagen, ops, shard
        from matrixone_b200.vector import DeviceBuffer, PinnedArray
        self.capi, self.datagen, self.ops, self.shard, self.DeviceBuffer, self.PinnedArray = capi, datagen, ops, shard, DeviceBuffer, PinnedArray
        self.lib = capi.load_library()
        capi.check(self.lib.MoB200_Init(self.local), self.lib)
        for kv in args.tune:
            name, _, val = kv.partition("=")
            self.lib.MoB200_SetTuning(name.encode(), int(val))
        self.dist = self.torch = None
        if self.world > 1:
            import torch
            import torch.distributed as dist
            self.torch, self.dist = torch, dist
            torch.cuda.set_device(self.local)
            import datetime
            # a collective mismatch should fail in minutes, not after the default 10-minute watchdog
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local), timeout=datetime.timedelta(seconds=env_int("MO_B200_NCCL_TIMEOUT_S", 180)))
            # ONE stream for the library's kernels and torch's NCCL calls: the whole step (kernel -> all_gather -> merge kernel -> D2H)
            # is stream-ordered on the device, the host never waits inside a step
            self.stream = torch.cuda.Stream()
            torch.cuda.set_stream(self.stream)
            capi.check(self.lib.MoB200_SetStream(self.stream.cuda_stream), self.lib)
        self.peaks = measured_peaks()
        self.sampler = ClockSampler(self.local)
        if self.rank == 0:
            self.sampler.start()
        self.W = max(3, args.warmup)
        self.K = max(1, args.steps)

    def check(self, rc):
        return self.capi.check(rc, self.lib)

    def sync(self):
        self.check(self.lib.MoB200_Sync())
        if self.torch is not None:
            self.torch.cuda.synchronize()

    def barrier_sync(self):
        self.sync()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        self.torch.cuda.synchronize()
        return float(t.item())

    def dev_bytes(self, nbytes):
        """device scratch both the library (raw pointer) and NCCL (torch tensor) can use: (ptr, keepalive)"""
        if self.torch is not None:
            t = self.torch.zeros(max(nbytes, 8), dtype=self.torch.uint8, device="cuda")
            return t.data_ptr(), t
        b = self.DeviceBuffer(max(nbytes, 8), self.lib)
        self.check(self.lib.MoB200_Memset(b.ptr, 0, max(nbytes, 8)))
        return b.ptr, b

    def timed(self, step, K=None, W=None, outputs=None):
        """W warm-up steps, then EXACTLY K steps between CUDA events on the library stream, barrier + synchronise on both sides.
        outputs() is called right after the K-th step has completed: what the last timed step returned, as {name: array}"""
        K = K or self.K
        W = self.W if W is None else W
        for _ in range(W):
            step()
        self.sync()
        if self.rank == 0:
            time.sleep(0.12)      # nvidia-smi needs ~100 ms between samples; keep the idle gap out of the window below
        self.barrier_sync()       # AFTER the sleep: the other ranks wait here, not inside their timed region
        t_region0 = time.time()
        launches0 = self.lib.MoB200_KernelLaunchCount()
        self.check(self.lib.MoB200_TimerStart())
        t_wall0 = time.perf_counter()
        for _ in range(K):
            step()
        ms = C.c_float()
        self.check(self.lib.MoB200_TimerStop(C.byref(ms)))
        self.barrier_sync()
        wall_ms = (time.perf_counter() - t_wall0) * 1e3
        out = outputs() if outputs is not None else {}
        t_region1 = time.time()
        launches = self.lib.MoB200_KernelLaunchCount() - launches0
        total_ms = self.max_over_ranks(max(ms.value, 0.0))
        clocks = None
        if total_ms < 250.0:
            # a short region holds too few 20 ms nvidia-smi samples: keep stepping (untimed) under the sampler.  The number of extra steps is
            # derived from the rank-maximum time, i.e. identical on every rank: the steps contain collectives
            extra = min(20000, int(400.0 / max(total_ms / K, 1e-3)) + 1)
            for _ in range(extra):
                step()
            self.barrier_sync()
            t_region1 = time.time()
        if self.rank == 0:
            clocks = self.sampler.window(t_region0, t_region1)
        if self.dist is not None:
            self.barrier_sync()
        return {"total_ms": total_ms, "ms_per_step": total_ms / K, "launches": int(launches), "wall_ms": wall_ms, "clocks": clocks, "steps": K, "warmup": W,
                "outputs": out}

    def kernel_ms(self, step, reps=5):
        """CUDA-event duration of the dominant kernel: mean over `reps` single steps (MoB200_LastKernelMs synchronises on the kernel's
        end event, so this runs right after the timed region, not inside it)"""
        out = []
        kms = C.c_float()
        for _ in range(reps):
            for _ in range(3):      # back to back, like the timed region: the measured launch is the last of the burst (clocks and caches in steady state)
                step()
            self.check(self.lib.MoB200_LastKernelMs(C.byref(kms)))
            out.append(kms.value)
        self.sync()
        return statistics.mean(out)


def rel_err(a, b):
    a, b = float(a), float(b)
    if a == b:
        return 0.0
    return abs(a - b) / max(abs(a), abs(b), 1e-300)


def pageable_like(pinned_cols):
    return {k: np.array(v, copy=True) for k, v in pinned_cols.items()}


# ---------------------------------------------------------------------------------------------------------- Q6 (headline)
def run_q6(env, n=None):
    lib, ops, capi, DeviceBuffer = env.lib, env.ops, env.capi, env.DeviceBuffer
    wl = WORKLOADS["q6"]
    n = n or env.args.rows or wl["rows"]
    world, rank = env.world, env.rank
    row0 = rank * n                          # this rank's disjoint block range of the N x SF100 table (weak scaling)
    names = ["shipdate", "quantity", "extendedprice", "discount"]
    bufs = {k: DeviceBuffer((4 if k == "shipdate" else 8) * n, lib) for k in names}
    env.check(lib.MoB200_GenLineitem(10, row0, n, bufs["shipdate"].ptr, bufs["quantity"].ptr, bufs["extendedprice"].ptr, bufs["discount"].ptr, None, None, None))
    P = env.datagen.q6_params()
    part_ptr, part_keep = env.dev_bytes(16)
    gath_ptr, gath_keep = env.dev_bytes(16 * world)
    fin_ptr, fin_keep = env.dev_bytes(16)
    host = env.PinnedArray((2,), np.float64, lib)

    def step():
        ops.q6_filter_sum_device(bufs["shipdate"], bufs["discount"], bufs["quantity"], bufs["extendedprice"], n, *P, out_ptr=part_ptr)
        if env.dist is not None:
            env.dist.all_gather_into_tensor(gath_keep[:16 * world], part_keep[:16])
            ops.q6_merge_device(gath_ptr, world, fin_ptr)                       # MergeGroup on the device, rank order
            env.check(lib.MoB200_DownloadAsync(host.ptr, fin_ptr, 16))
        else:
            env.check(lib.MoB200_DownloadAsync(host.ptr, part_ptr, 16))

    t = env.timed(step, outputs=lambda: {"q6_revenue": host.array[:1].copy(), "q6_rows": host.array.view(np.int64)[1:2].copy()})
    final = (float(host.array[0]), int(host.array.view(np.int64)[1]))
    # cross-check of the device seam against the synchronous API + the host-side merge (shard.py; covered by the gloo CPU test)
    sres = ops.q6_filter_sum(bufs["shipdate"], bufs["discount"], bufs["quantity"], bufs["extendedprice"], n, *P)
    seam_ok = None
    if env.dist is not None:
        tt = env.torch.tensor(np.frombuffer(env.shard.pack_q6(sres[0], sres[1]), dtype=np.uint8).copy(), device="cuda")
        gg = env.torch.zeros(16 * world, dtype=env.torch.uint8, device="cuda")
        env.dist.all_gather_into_tensor(gg, tt)
        env.torch.cuda.synchronize()
        hs, hc, _ = env.shard.merge_q6(gg.cpu().numpy().tobytes(), world)
        seam_ok = (hs == final[0] and hc == final[1])
    else:
        seam_ok = (sres[0] == final[0] and sres[1] == final[1])
    kern_ms = env.kernel_ms(lambda: ops.q6_filter_sum_device(bufs["shipdate"], bufs["discount"], bufs["quantity"], bufs["extendedprice"], n, *P, out_ptr=part_ptr))
    value = n * world * t["steps"] / (t["total_ms"] * 1e-3)

    # ---- e2e: host (pinned) columns through the synchronous C-ABI call, H2D inside the timed region
    e2e = None
    if not env.args.no_e2e:
        e2e = e2e_columns(env, bufs, n, {"shipdate": np.int32}, lambda cols, m: ops.q6_filter_sum(cols["shipdate"], cols["discount"], cols["quantity"], cols["extendedprice"], m, *P),
                          lambda res: env.shard.pack_q6(res[0], res[1]), 16, wl["bytes_per_row"], world_units=world)

    out = {"value": value, "units_per_step": n * world, "timing": t, "kernel_ms": kern_ms, "alg_bytes": wl["bytes_per_row"] * n, "kernel": "q6_kernel",
           "e2e": e2e, "result": {"sum": final[0], "rows": final[1]}, "rows_per_gpu": n, "device_seam_matches_host_merge": bool(seam_ok),
           "parallelism": ("block-range shards x%d (weak: every rank scans its own SF100-sized range), NCCL all_gather + merge kernel on one stream" % world) if world > 1 else "1 GPU"}
    # ---- cpu baseline + parity on the first CPU_SAMPLE_ROWS rows of rank 0
    if rank == 0 and not env.args.no_cpu:
        m = min(n, CPU_SAMPLE_ROWS)
        threads = os.cpu_count() or 1
        import oracle_lib as O
        cols = O.gen_lineitem(10, row0, m, threads, names)     # bit-identical to the GPU's rows (tests), first-touched by the worker pool
        v, sec, cres = cpu_q6(cols, m, threads)
        gres = ops.q6_filter_sum(bufs["shipdate"], bufs["discount"], bufs["quantity"], bufs["extendedprice"], m, *P)
        out["cpu_baseline"] = {"value": v, "unit": "rows/s", "cores": threads, "kind": "port",
                               "sample": "first %d rows (the same rows from the oracle's C twin of the generator, NUMA-local first touch), median of 5 passes after 1 warm-up; oracle/oracle_go.c operator chain on a persistent pool of %d pinned pthreads" % (m, threads)}
        out["parity"] = {"sample_rows": m, "oracle_sum": cres[0], "gpu_sum": gres[0], "rel_err": rel_err(cres[0], gres[0]), "rows_equal": cres[1] == gres[1],
                         "tolerance": 1e-5, "ok": bool(rel_err(cres[0], gres[0]) <= 1e-5 and cres[1] == gres[1])}
    for b in bufs.values():
        b.free()
    host.free()
    return out


def e2e_columns(env, bufs, n, dtypes, call, pack, rec_bytes, bytes_per_row, world_units=1, total_units=None):
    """the synchronous drop-in call on HOST columns: pinned (MoB200_HostAlloc) and pageable (plain numpy) copies of the GPU's own rows"""
    lib, capi = env.lib, env.capi
    try:
        need = sum(b.nbytes for b in bufs.values())
        avail = mem_available()
        n_e2e = n
        if avail and need * env.world * 2.6 > avail:
            n_e2e = max(1 << 20, int(n * (avail / (need * env.world * 2.6))) // 8192 * 8192)
        pinned = {}
        for k, b in bufs.items():
            dt = np.dtype(dtypes.get(k, np.float64))
            pa = env.PinnedArray((n_e2e,), dt, lib)
            env.check(lib.MoB200_Download(pa.ptr, b.ptr, n_e2e * dt.itemsize))
            pinned[k] = pa
        hcols = {k: pa.array for k, pa in pinned.items()}

        def exchange(res):
            if env.dist is None:
                return
            tt = env.torch.tensor(np.frombuffer(pack(res), dtype=np.uint8).copy(), device="cuda")
            gg = env.torch.zeros(rec_bytes * env.world, dtype=env.torch.uint8, device="cuda")
            env.dist.all_gather_into_tensor(gg, tt)
            gg.cpu()

        def run(cols, ke):
            exchange(call(cols, n_e2e))
            env.barrier_sync()
            t0 = time.perf_counter()
            for _ in range(ke):
                exchange(call(cols, n_e2e))
            env.barrier_sync()
            return env.max_over_ranks(time.perf_counter() - t0) / ke

        ke = min(env.K, 5)
        sec = run(hcols, ke)
        units = (total_units if total_units is not None else n_e2e * world_units)
        e2e = {"value": units / sec, "unit": "rows/s", "h2d_bytes_per_step": int(bytes_per_row * n_e2e), "d2h_bytes_per_step": rec_bytes, "steps": ke, "rows_per_gpu": n_e2e,
               "host_memory": "pinned (MoB200_HostAlloc)", "timer": "wall clock around the C-ABI calls, max over ranks"}
        if env.world == 1 and not env.args.no_pageable:
            m = min(n_e2e, 1 << 27)      # pageable arm on a 134 M-row prefix: what MatrixOne's mpool / Go-heap vectors cost without a pinned allocator
            pg = {k: np.array(v[:m], copy=True) for k, v in hcols.items()}
            call(pg, m)
            t0 = time.perf_counter()
            call(pg, m); call(pg, m)
            e2e["pageable"] = {"value": m * 2 / (time.perf_counter() - t0), "unit": "rows/s", "rows": m, "host_memory": "pageable (numpy / malloc)"}
        for pa in pinned.values():
            pa.free()
        return e2e
    except Exception as ex:  # report, never fake
        return {"value": None, "unit": "rows/s", "error": str(ex)[:200]}


# ---------------------------------------------------------------------------------------------------------- SUM (config 1)
def run_sum(env):
    lib, ops, capi, DeviceBuffer = env.lib, env.ops, env.capi, env.DeviceBuffer
    wl = WORKLOADS["sum"]
    n = env.args.rows or wl["rows"]
    world, rank = env.world, env.rank
    R = 4    # rotate over 4 distinct columns (320 MB > the 126 MB L2): every timed launch reads HBM, not L2
    cols = []
    for r in range(R):
        b = DeviceBuffer(8 * n, lib)
        env.check(lib.MoB200_GenInt64(1 + r, ((rank * n) // 64) * 64, n, b.ptr, None, 0))
        cols.append(b)
    part_ptr, part_keep = env.dev_bytes(24)
    gath_ptr, gath_keep = env.dev_bytes(24 * world)
    fin_ptr, fin_keep = env.dev_bytes(24)
    host = env.PinnedArray((3,), np.uint64, lib)
    it = [0]
    from matrixone_b200.vector import Vector
    fid = capi.XCALL_AGG(capi.AGG_SUM, capi.T_INT64)
    err = (C.c_uint8 * 256)()
    pre = []
    for c in cols:      # XCall argument blocks marshalled once, as a cgo caller holds them: the timed step is the bare C-ABI call
        arr = (capi.XCallArgs * 2)(Vector(data_ptr=part_ptr, data_nbytes=24, length=1).fill_raw_ptr_len(), Vector(data_ptr=c.ptr, data_nbytes=8 * n, length=n).fill_raw_ptr_len())
        pre.append((arr, C.cast(arr, C.c_void_p)))

    def step():
        arr, argp = pre[it[0] % R]; it[0] += 1
        rc = lib.XCall(1, fid, err, argp, n)
        if rc:
            raise capi.MoError(rc, "sum")
        if env.dist is not None:
            env.dist.all_gather_into_tensor(gath_keep[:24 * world], part_keep[:24])
            ops.agg_merge_device(capi.AGG_SUM, capi.T_INT64, gath_ptr, world, fin_ptr)
            env.check(lib.MoB200_DownloadAsync(host.ptr, fin_ptr, 24))
        else:
            env.check(lib.MoB200_DownloadAsync(host.ptr, part_ptr, 24))

    t = env.timed(step, outputs=lambda: {"sum_state": host.array.view(np.int64).copy()})
    it[0] = 0
    kern_ms = env.kernel_ms(step, reps=8)
    value = n * world * t["steps"] / (t["total_ms"] * 1e-3)
    e2e = None
    if not env.args.no_e2e:
        pa = env.PinnedArray((n,), np.int64, lib)
        env.check(lib.MoB200_Download(pa.ptr, cols[0].ptr, 8 * n))
        ops.agg_sum(capi.T_INT64, pa.array, None, n)
        env.barrier_sync()
        t0 = time.perf_counter()
        for _ in range(10):
            ops.agg_sum(capi.T_INT64, pa.array, None, n)
        env.barrier_sync()
        sec = env.max_over_ranks(time.perf_counter() - t0) / 10
        e2e = {"value": n * world / sec, "unit": "rows/s", "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 8, "steps": 10, "host_memory": "pinned (MoB200_HostAlloc)",
               "timer": "wall clock around the C-ABI calls, max over ranks"}
        pa.free()
    out = {"value": value, "units_per_step": n * world, "timing": t, "kernel_ms": kern_ms, "alg_bytes": 8.0 * n, "kernel": "agg_kernel<int64, SUM>", "e2e": e2e, "rows_per_gpu": n,
           "l2": "4 distinct 80 MB columns used in rotation (320 MB > the 126 MB L2)",
           "parallelism": ("row-range shards x%d (weak), NCCL all_gather of 24-byte states + merge kernel" % world) if world > 1 else "1 GPU"}
    if rank == 0 and not env.args.no_cpu:
        threads = os.cpu_count() or 1
        import oracle_lib as O
        hcol = O.gen_int64(1, ((rank * n) // 64) * 64, n, threads)
        v, sec, csum = cpu_sum(hcol, n, threads)
        rc, gsum, isnull = ops.agg_sum(capi.T_INT64, cols[0], None, n)
        out["cpu_baseline"] = {"value": v, "unit": "rows/s", "cores": threads, "kind": "port", "sample": "all %d rows, median of 5 passes; oracle/oracle_go.c og_sum_int64_mt on %d pinned pthreads" % (n, threads)}
        out["parity"] = {"sample_rows": n, "oracle_sum": csum, "gpu_sum": gsum, "bit_exact": csum == gsum, "ok": bool(csum == gsum and rc == 0)}
    for b in cols:
        b.free()
    host.free()
    return out


# ---------------------------------------------------------------------------------------------------------- Q1 (config 3)
def run_q1(env):
    lib, ops, capi, DeviceBuffer = env.lib, env.ops, env.capi, env.DeviceBuffer
    wl = WORKLOADS["q1"]
    total = env.args.rows or wl["rows"]
    world, rank = env.world, env.rank
    r0, r1 = env.shard.block_range(rank, world, total)     # STRONG scaling: ONE SF100 table cut into contiguous block ranges
    n = r1 - r0
    names = ["shipdate", "quantity", "extendedprice", "discount", "tax", "returnflag", "linestatus"]
    size = {"shipdate": 4, "returnflag": 1, "linestatus": 1}
    bufs = {k: DeviceBuffer(size.get(k, 8) * max(n, 1), lib) for k in names}
    env.check(lib.MoB200_GenLineitem(10, r0, n, *[bufs[k].ptr for k in ("shipdate", "quantity", "extendedprice", "discount", "tax", "returnflag", "linestatus")]))
    RB = ops.Q1_RESULT_BYTES
    part_ptr, part_keep = env.dev_bytes(RB)
    gath_ptr, gath_keep = env.dev_bytes(RB * world)
    fin_ptr, fin_keep = env.dev_bytes(RB)
    host = env.PinnedArray((RB,), np.uint8, lib)
    cut = env.datagen.Q1_CUTOFF

    def call_dev():
        ops.q1_group_agg_device(bufs["shipdate"], bufs["quantity"], bufs["extendedprice"], bufs["discount"], bufs["tax"], bufs["returnflag"], bufs["linestatus"], n, cut, part_ptr, row_base=r0)

    def step():
        call_dev()
        if env.dist is not None:
            env.dist.all_gather_into_tensor(gath_keep[:RB * world], part_keep[:RB])
            ops.q1_merge_device(gath_ptr, world, fin_ptr)
            env.check(lib.MoB200_DownloadAsync(host.ptr, fin_ptr, RB))
        else:
            env.check(lib.MoB200_DownloadAsync(host.ptr, part_ptr, RB))

    q1_fields = ("returnflag", "linestatus", "first_row", "sum_qty", "sum_base_price", "sum_disc_price", "sum_charge", "avg_qty", "avg_price", "avg_disc",
                 "sum_disc", "count_order")
    t = env.timed(step, outputs=lambda: {"q1_groups": np.array([[g[f] for f in q1_fields] for g in ops.q1_result_from_bytes(host.array.tobytes())], dtype=np.float64)})
    final = ops.q1_result_from_bytes(host.array.tobytes())
    # cross-check: synchronous API + host-side merge (shard.merge_q1) must give the same groups
    sres = ops.q1_group_agg(bufs["shipdate"], bufs["quantity"], bufs["extendedprice"], bufs["discount"], bufs["tax"], bufs["returnflag"], bufs["linestatus"], n, cut)
    if env.dist is not None:
        tt = env.torch.tensor(np.frombuffer(env.shard.pack_q1(sres, r0), dtype=np.uint8).copy(), device="cuda")
        gg = env.torch.zeros(env.shard.Q1_REC_BYTES * world, dtype=env.torch.uint8, device="cuda")
        env.dist.all_gather_into_tensor(gg, tt)
        env.torch.cuda.synchronize()
        hm = env.shard.merge_q1(gg.cpu().numpy().tobytes(), world)
    else:
        hm = sres
    seam_ok = len(hm) == len(final) and all(a["returnflag"] == b["returnflag"] and a["linestatus"] == b["linestatus"] and a["count_order"] == b["count_order"] and
                                            a["sum_charge"] == b["sum_charge"] and a["sum_qty"] == b["sum_qty"] for a, b in zip(hm, final))
    kern_ms = env.kernel_ms(call_dev)
    value = total * t["steps"] / (t["total_ms"] * 1e-3)
    e2e = None
    if not env.args.no_e2e:
        e2e = e2e_columns(env, bufs, n, {"shipdate": np.int32, "returnflag": np.uint8, "linestatus": np.uint8},
                          lambda cols, m: ops.q1_group_agg(cols["shipdate"], cols["quantity"], cols["extendedprice"], cols["discount"], cols["tax"], cols["returnflag"], cols["linestatus"], m, cut),
                          lambda res: env.shard.pack_q1(res, r0), env.shard.Q1_REC_BYTES, wl["bytes_per_row"], total_units=total if n == r1 - r0 else None)
        if e2e.get("rows_per_gpu") not in (None, n) and e2e.get("value"):
            e2e["value"] = e2e["value"] * e2e["rows_per_gpu"] / n      # host memory bounded the copy: throughput on the rows actually moved
            e2e["note"] = "host memory bounded the columns to rows_per_gpu rows per rank"
    out = {"value": value, "units_per_step": total, "timing": t, "kernel_ms": kern_ms, "alg_bytes": wl["bytes_per_row"] * n, "kernel": "q1_staged_kernel (packed uint8 keys, 38 B/row)",
           "e2e": e2e, "result": {"groups": len(final), "count_order": [g["count_order"] for g in final]}, "rows_per_gpu": n, "device_seam_matches_host_merge": bool(seam_ok),
           "parallelism": ("ONE SF100 table in %d contiguous block ranges (strong scaling, shard.block_range), NCCL all_gather of %d-byte partial results + MergeGroup kernel on one stream" % (world, RB)) if world > 1 else "1 GPU"}
    if rank == 0 and not env.args.no_cpu:
        m = min(n, CPU_SAMPLE_ROWS)
        threads = os.cpu_count() or 1
        import oracle_lib as O
        cols = O.gen_lineitem(10, r0, m, threads, names)
        v, sec, cres = cpu_q1(cols, m, threads)
        vw = {k: bufs[k].view(size.get(k, 8) * m) for k in names}      # the first m rows of the resident columns
        gres = ops.q1_group_agg(vw["shipdate"], vw["quantity"], vw["extendedprice"], vw["discount"], vw["tax"], vw["returnflag"], vw["linestatus"], m, cut)
        worst, counts_ok = 0.0, len(cres) == len(gres)
        for a, b in zip(cres, gres):
            counts_ok = counts_ok and a["returnflag"] == b["returnflag"] and a["linestatus"] == b["linestatus"] and a["count_order"] == b["count_order"] and a["first_row"] == b["first_row"]
            for f in ("sum_qty", "sum_base_price", "sum_disc_price", "sum_charge", "avg_qty", "avg_price", "avg_disc"):
                worst = max(worst, rel_err(a[f], b[f]))
        out["cpu_baseline"] = {"value": v, "unit": "rows/s", "cores": threads, "kind": "port",
                               "sample": "first %d rows (the same rows from the oracle's C twin of the generator, NUMA-local first touch), median of 5 passes after 1 warm-up; oracle/oracle_go.c operator chain on a persistent pool of %d pinned pthreads" % (m, threads)}
        out["parity"] = {"sample_rows": m, "groups": len(gres), "keys_counts_first_rows_equal": bool(counts_ok), "max_rel_err": worst, "tolerance": 1e-5, "ok": bool(counts_ok and worst <= 1e-5)}
    for b in bufs.values():
        b.free()
    host.free()
    return out


# ---------------------------------------------------------------------------------------------------------- vector search
def topk_parity(okeys, odists, gkeys, gdists, nq, k):
    """oracle vs GPU top-k for the same queries: distances must be bit-equal position by position; keys equal except inside a run of
    EQUAL distances (the GPU breaks ties by lower row id, FastMaxHeap by arrival order)"""
    ok_ = np.asarray(okeys).reshape(nq, k); od = np.asarray(odists).reshape(nq, k)
    gk = np.asarray(gkeys).reshape(nq, k); gd = np.asarray(gdists).reshape(nq, k)
    dist_equal = bool(np.array_equal(od, gd))
    key_mismatch = ok_ != gk
    tie_only = True
    for q, j in zip(*np.nonzero(key_mismatch)):
        same = (od[q] == od[q, j])
        if same.sum() < 2 or set(ok_[q][same]) != set(gk[q][same]):
            tie_only = False
            break
    return {"queries": int(nq), "distances_bit_equal": dist_equal, "key_mismatches": int(key_mismatch.sum()), "mismatches_are_ties": bool(tie_only),
            "ok": bool(dist_equal and tie_only)}


def search_seam(env, nq, k):
    """device buffers of the MergeTop seam: per-rank (keys, dists) -> all_gather -> merge kernel -> final"""
    T = env.torch
    return {"k": T.empty(nq * k, dtype=T.int64, device="cuda"), "d": T.empty(nq * k, dtype=T.float64, device="cuda"),
            "gk": T.empty(env.world * nq * k, dtype=T.int64, device="cuda"), "gd": T.empty(env.world * nq * k, dtype=T.float64, device="cuda"),
            "ok": T.empty(nq * k, dtype=T.int64, device="cuda"), "od": T.empty(nq * k, dtype=T.float64, device="cuda")}


def run_search(env, which):
    lib, ops, capi, DeviceBuffer = env.lib, env.ops, env.capi, env.DeviceBuffer
    wl = WORKLOADS[which]
    world, rank = env.world, env.rank
    dim, nq, k, nlist, nprobe = 768, env.args.queries, 10, 1024, 32
    total = env.args.rows or wl["rows"]
    n_local = total // world
    ivf = idx = None
    if which == "ivf":
        # BASELINE config 5: entries = mixture of 1024 Gaussians, centroids = the generating means, assignment by argmin L2sq (Productl2);
        # every rank holds the full centroid table and its row slice of every list; per-rank top-k are gathered and merged
        centers = env.datagen.vectors_f32(30, 0, nlist, dim) * np.float32(4.0)
        dcent = DeviceBuffer.from_numpy(centers, lib)
        t_b0 = time.perf_counter()
        # LISTS are sharded (config 5: "lists sharded 8 x B200"): rank r keeps the whole lists l with l % world == r of the ONE 10 M-row table
        ivf = ops.IvfflatSearchIndex.build_list_shard(lambda r0, m, ptr: env.check(lib.MoB200_GenVectorsF32(31, r0, m, dim, ptr, dcent.ptr, nlist, 1.0)),
                                                      total, centers, rank, world, capi.METRIC_L2, lib)
        build_s = time.perf_counter() - t_b0
        dcent.free()
        n_local = ivf.n
        dq = DeviceBuffer(4 * nq * dim, lib)
        env.check(lib.MoB200_GenVectorsF32(32, 0, nq, dim, dq.ptr, ivf.d_cent.ptr, nlist, 1.0))
        search = lambda q, out=None: ivf.search(q, k, nprobe, out=out)
    else:
        ds = DeviceBuffer(4 * n_local * dim, lib)
        env.check(lib.MoB200_GenVectorsF32(20, rank * n_local, n_local, dim, ds.ptr, None, 0, 1.0))
        dq = DeviceBuffer(4 * nq * dim, lib)
        env.check(lib.MoB200_GenVectorsF32(21, 0, nq, dim, dq.ptr, None, 0, 1.0))
        t_b0 = time.perf_counter()
        idx = ops.BruteForceIndex(ds, dim, capi.METRIC_L2, key_base=rank * n_local, lib=lib)
        build_s = time.perf_counter() - t_b0
        search = lambda q, out=None: idx.search(q, k, out=out)

    rec_bytes = nq * k * 16
    if env.dist is not None:
        S = search_seam(env, nq, k)
        hk = env.PinnedArray((nq * k,), np.int64, lib); hd = env.PinnedArray((nq * k,), np.float64, lib)

        def step():
            search(dq, out=(S["k"].data_ptr(), S["d"].data_ptr()))
            env.dist.all_gather_into_tensor(S["gk"], S["k"])
            env.dist.all_gather_into_tensor(S["gd"], S["d"])
            ops.topk_merge_device(S["gk"].data_ptr(), S["gd"].data_ptr(), world, nq, k, S["ok"].data_ptr(), S["od"].data_ptr())
            env.check(lib.MoB200_DownloadAsync(hk.ptr, S["ok"].data_ptr(), nq * k * 8))
            env.check(lib.MoB200_DownloadAsync(hd.ptr, S["od"].data_ptr(), nq * k * 8))
    else:
        kd, dd = DeviceBuffer(nq * k * 8, lib), DeviceBuffer(nq * k * 8, lib)
        hk = env.PinnedArray((nq * k,), np.int64, lib); hd = env.PinnedArray((nq * k,), np.float64, lib)

        def step():
            search(dq, out=(kd.ptr, dd.ptr))
            env.check(lib.MoB200_DownloadAsync(hk.ptr, kd.ptr, nq * k * 8))
            env.check(lib.MoB200_DownloadAsync(hd.ptr, dd.ptr, nq * k * 8))

    t = env.timed(step, outputs=lambda: {which + "_keys": hk.array.reshape(nq, k).copy(), which + "_distances": hd.array.reshape(nq, k).copy()})
    kms = C.c_float()
    env.check(lib.MoB200_LastKernelMs(C.byref(kms)))    # the candidate pass of the last timed step
    kern_ms = kms.value
    value = nq * t["steps"] / (t["total_ms"] * 1e-3)
    kused = int(lib.MoB200_SetTuning(b"get_tc_kused", 0)) or 3 * dim
    refined, fallbacks = int(lib.MoB200_SetTuning(b"get_tc_refined", 0)), int(lib.MoB200_SetTuning(b"get_tc_fallbacks", 0))
    if which == "ivf":
        pairs = float(nq) * nprobe * (total / float(nlist)) / world    # (query, probed row) pairs this rank scans: its share of the lists
        flop = 2.0 * pairs * kused
        kernel = "tc_candidates_kernel (tcgen05 bf16, K = %d per pair) over (list, query-tile) units" % kused
    else:
        flop = 2.0 * nq * n_local * kused
        kernel = "tc_candidates_kernel (tcgen05 bf16, K = %d per pair)" % kused

    # ---- e2e: queries from host memory, keys + distances back to host, through the synchronous call (+ the exchange at N > 1)
    e2e = None
    if not env.args.no_e2e:
        qhost = dq.to_numpy(np.float32)
        def e2e_step():
            r = search(qhost)
            if env.dist is not None:
                tk = env.torch.from_numpy(r[0]).cuda(); td = env.torch.from_numpy(r[1]).cuda()
                env.dist.all_gather_into_tensor(S["gk"], tk); env.dist.all_gather_into_tensor(S["gd"], td)
                ops.topk_merge_device(S["gk"].data_ptr(), S["gd"].data_ptr(), world, nq, k, S["ok"].data_ptr(), S["od"].data_ptr())
                S["ok"].cpu(); S["od"].cpu()
        e2e_step()
        env.barrier_sync()
        ke = min(env.K, 5)
        t0 = time.perf_counter()
        for _ in range(ke):
            e2e_step()
        env.barrier_sync()
        sec = env.max_over_ranks(time.perf_counter() - t0) / ke
        e2e = {"value": nq / sec, "unit": "queries/s", "h2d_bytes_per_step": 4 * nq * dim, "d2h_bytes_per_step": rec_bytes, "steps": ke, "host_memory": "pageable (numpy)",
               "note": "index resident (built once, as the reference keeps it in memory); queries from host, keys + distances to host", "timer": "wall clock, max over ranks"}

    out = {"value": value, "units_per_step": nq, "timing": t, "kernel_ms": kern_ms, "alg_flop": flop, "kernel": kernel, "e2e": e2e, "rows_per_gpu": n_local, "rows_total": total,
           "queries": nq, "index_build_s": build_s, "tc_refined_queries": refined, "tc_fallback_queries": fallbacks,
           "parallelism": (("whole LISTS sharded x%d (l %% world == rank; strong: one %d-row index)" if which == "ivf" else "rows sharded x%d (strong: one %d-row index)") % (world, total) + ", NCCL all_gather of per-rank top-k + merge kernel on one stream") if world > 1 else "1 GPU"}

    # ---- cpu baseline + parity: the oracle answers a bounded set of the SAME queries over this rank's FULL shard
    if rank == 0 and not env.args.no_cpu:
        threads = os.cpu_count() or 1
        if which == "bruteforce":
            import oracle_lib as O
            hds = O.gen_vectors_f32(20, rank * n_local, n_local, dim, threads)      # bit-identical to the GPU's rows, pages spread over the NUMA nodes
            hqs = dq.to_numpy(np.float32).reshape(-1, dim)[:threads]
            v, sec, (okeys, odists) = cpu_bruteforce(hds, hqs, threads, reps=1)
            out["cpu_baseline"] = {"value": v, "unit": "queries/s", "cores": threads, "kind": "port",
                                   "sample": "rank 0's full %d x 768 rows, the first %d queries (one per host thread), 1 pass; oracle/oracle_go.c GoBruteForceIndex.Search" % (n_local, hqs.shape[0])}
            gkeys, gdists = idx.search(hqs, k)
            okeys = np.where(okeys >= 0, okeys + rank * n_local, okeys)
        else:
            need = 1.3 * ivf.n * dim * 4
            if mem_available() > need:
                ents = ivf.d_data.to_numpy(np.float32).reshape(ivf.n, dim)                  # list-ordered entries
                assign = np.repeat(np.arange(nlist, dtype=np.int32), np.diff(ivf.offsets))   # their list ids
                cents = ivf.d_cent.to_numpy(np.float32).reshape(nlist, dim)
                hqs = dq.to_numpy(np.float32).reshape(-1, dim)[:8 * threads]
                v, sec, (okeys, odists) = cpu_ivf(ents, assign, cents, hqs, threads, reps=1)
                okeys = np.where(okeys >= 0, ivf.row_ids[np.clip(okeys, 0, ivf.n - 1)], okeys)   # list-ordered position -> primary key
                out["cpu_baseline"] = {"value": v, "unit": "queries/s", "cores": threads, "kind": "port",
                                       "sample": "rank 0's own index (%d x 768, nlist 1024, nprobe 32), the first %d queries over %d host threads, 1 pass; oracle/oracle_go.c og_ivf_search_f32" % (ivf.n, hqs.shape[0], threads)}
                gkeys, gdists = ivf.search(hqs, k, nprobe)
            else:
                okeys = None
                out["cpu_baseline"] = {"value": None, "note": "host memory too small for the %d-row index" % ivf.n}
        if okeys is not None:
            out["parity"] = topk_parity(okeys, odists, gkeys, gdists, hqs.shape[0], k)
            out["parity"]["scope"] = "rank 0's shard, oracle vs GPU through the same C-ABI call"
    hk.free(); hd.free()
    if idx is not None:
        idx.destroy(); ds.free()
    if ivf is not None:
        ivf.destroy()
    dq.free()
    return out


# ---------------------------------------------------------------------------------------------------------- drop-in block cost
def run_dropin(env):
    """What the untouched colexec pipeline pays per 8192-row block when it calls the library from HOST pointers: one XCall of the Go
    elementwise engine's int64 a+b (overflow-checked) = H2D of two 64 KiB columns + a launch + D2H of 64 KiB + a synchronise.
    Reported next to the same call on resident columns and next to the CPU loop, so nobody has to guess."""
    lib, ops, capi, DeviceBuffer = env.lib, env.ops, env.capi, env.DeviceBuffer
    from matrixone_b200.vector import Vector, xcall
    n = 8192
    a = env.datagen.int64_column(1, 0, n)[0]; b = env.datagen.int64_column(2, 0, n)[0]
    fid = capi.XCALL_GO_ARITH(0, capi.T_INT64)
    class GoParams(C.Structure):
        _fields_ = [("div0_null", C.c_int32), ("reserved", C.c_int32), ("err_row", C.c_int64)]
    def mk(host):
        r = np.zeros(n, dtype=np.int64); rn = np.zeros(n // 64, dtype=np.uint64)
        pv = Vector(data=np.frombuffer(bytes(GoParams(0, 0, -1)), dtype=np.uint8).copy(), length=1, const=True)
        if host:
            return [Vector(data=r, nulls=rn, length=n), Vector(data=a, length=n), Vector(data=b, length=n), pv], r
        da, db, dr, dn = DeviceBuffer.from_numpy(a, lib), DeviceBuffer.from_numpy(b, lib), DeviceBuffer(8 * n, lib), DeviceBuffer.from_numpy(rn, lib)
        return [Vector(data_ptr=dr.ptr, data_nbytes=8 * n, nulls_ptr=dn.ptr, length=n), Vector(data_ptr=da.ptr, data_nbytes=8 * n, length=n),
                Vector(data_ptr=db.ptr, data_nbytes=8 * n, length=n), pv], (da, db, dr, dn)
    out, outputs = {}, {}
    for label, host in (("host_pointers", True), ("host_pointers_inputs_pinned_in_column_cache", True), ("resident", False)):
        vecs, keep = mk(host)
        if "pinned" in label:      # MoB200_ColumnPin: the block's input columns are uploaded once, later calls find them on the device
            env.check(lib.MoB200_ColumnCacheConfigure(64 << 20))
            env.check(lib.MoB200_ColumnPin(a.ctypes.data, a.nbytes, 1)); env.check(lib.MoB200_ColumnPin(b.ctypes.data, b.nbytes, 1))
        arr = (capi.XCallArgs * len(vecs))()
        for i, v in enumerate(vecs):
            arr[i] = v.fill_raw_ptr_len()
        err = (C.c_uint8 * 256)()
        call = lambda: lib.XCall(1, fid, err, C.cast(arr, C.c_void_p), n)
        for _ in range(50):
            call()
        env.sync()
        reps = env.K
        t0 = time.perf_counter()
        for _ in range(reps):
            rc = call()
        env.sync()
        sec = (time.perf_counter() - t0) / reps
        out[label] = {"us_per_block": sec * 1e6, "rows_per_s": n / sec, "rc": int(rc)}
        if label == "host_pointers":
            outputs["dropin_sum"] = keep.copy()
        if "pinned" in label:
            env.check(lib.MoB200_ColumnCacheConfigure(0))
        if host:
            ok = bool(np.array_equal(keep, a + b)) and (label == "host_pointers" or ok)
    # one call over 1024 blocks at once from host pointers (the multi-block form of the same entry point: the per-call costs are paid once)
    nb = 1024 * n
    A = env.datagen.int64_column(1, 0, nb)[0]; B = env.datagen.int64_column(2, 0, nb)[0]
    R = np.zeros(nb, dtype=np.int64); RN = np.zeros(nb // 64, dtype=np.uint64)
    pvv = Vector(data=np.frombuffer(bytes(GoParams(0, 0, -1)), dtype=np.uint8).copy(), length=1, const=True)
    bv = [Vector(data=R, nulls=RN, length=nb), Vector(data=A, length=nb), Vector(data=B, length=nb), pvv]
    xcall(fid, bv, nb)
    t0 = time.perf_counter()
    for _ in range(5):
        xcall(fid, bv, nb)
    secb = (time.perf_counter() - t0) / 5
    out["host_pointers_1024_blocks_per_call"] = {"us_per_block": secb * 1e6 / 1024, "rows_per_s": nb / secb, "rc": 0}
    ok = ok and bool(np.array_equal(R, A + B))
    res = {"value": out["host_pointers"]["rows_per_s"], "units_per_step": n, "timing": {"total_ms": out["host_pointers"]["us_per_block"] * 1e-3 * env.K, "ms_per_step": out["host_pointers"]["us_per_block"] * 1e-3, "launches": env.K, "steps": env.K, "warmup": 50, "clocks": None, "wall_ms": None, "outputs": outputs},
           "kernel_ms": None, "kernel": "go_arith_kernel<int64, +>", "blocks": out, "e2e": {"value": out["host_pointers"]["rows_per_s"], "unit": "rows/s", "h2d_bytes_per_step": 16 * n, "d2h_bytes_per_step": 8 * n + n // 8, "host_memory": "pageable (numpy)"},
           "parity": {"bit_exact": ok, "ok": ok}, "parallelism": "1 OS thread, 1 block in flight"}
    if env.rank == 0 and not env.args.no_cpu:
        v, sec, _ = cpu_dropin(1)
        res["cpu_baseline"] = {"value": v, "unit": "rows/s", "cores": 1, "kind": "port", "sample": "the same 8192-row batch, 200 calls; oracle/oracle_go.c og_arith", "us_per_block": sec * 1e6}
        res["verdict"] = ("one block at a time from host pointers is %.1fx SLOWER than the CPU loop: the per-block entry points only pay off on resident columns; "
                          "the fused multi-block entry points (Q6 / Q1 / plan) are the drop-in that wins" % (v / out["host_pointers"]["rows_per_s"])) if v > out["host_pointers"]["rows_per_s"] else "host-pointer block call is faster than the CPU loop"
    return res


# ---------------------------------------------------------------------------------------------------------- line assembly
def finish(env, w, r):
    """raw workload result -> the JSON object of the contract"""
    wl = WORKLOADS[w]
    t = r["timing"]
    line = {"metric": wl["metric"], "value": r["value"], "unit": wl["unit"], "n_gpus": env.world, "steps": t["steps"], "warmup": t["warmup"], "ms_per_step": t["ms_per_step"],
            "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic"}
    cfg = {"workload": wl["name"], "rows_per_gpu": r.get("rows_per_gpu"), "parallelism": r.get("parallelism"),
           "timer": "CUDA events on the library stream (MoB200_TimerStart/Stop) around exactly `steps` steps, barrier + synchronise on both sides, max over ranks",
           "wall_ms_rank0": t.get("wall_ms")}
    if w in ("q6", "q1"):
        cfg["l2"] = "inputs (%.1f GB per GPU) are larger than the 126 MB L2; no flush needed" % (r["alg_bytes"] / 1e9)
    elif w == "sum":
        cfg["l2"] = r["l2"]
    elif w in ("bruteforce", "ivf"):
        cfg["l2"] = "the index (%.1f GB per GPU) is larger than the 126 MB L2; no flush needed" % (4.0 * r["rows_per_gpu"] * 768 / 1e9)
        cfg["queries"] = r["queries"]; cfg["rows_total"] = r["rows_total"]; cfg["index_build_s"] = r["index_build_s"]
    line["config"] = cfg
    if r.get("alg_bytes") is not None and r.get("kernel_ms"):
        peak, src = env.peaks["hbm"]
        ach = r["alg_bytes"] / (r["kernel_ms"] * 1e-3) / 1e9
        traffic, tsrc = ncu_traffic("%s:%d" % (w, r["rows_per_gpu"]))
        line["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "kernel": r["kernel"], "kernel_ms": r["kernel_ms"],
                            "algorithmic_bytes_per_launch": r["alg_bytes"], "peak_source": src, "traffic_source": tsrc,
                            "kernel_ms_source": "mean CUDA-event duration of the kernel (last launch of back-to-back bursts) right after the timed region"}
    elif r.get("alg_flop") is not None and r.get("kernel_ms"):
        peak, src = env.peaks["bf16"]
        ach = r["alg_flop"] / (r["kernel_ms"] * 1e-3) / 1e12
        traffic, tsrc = ncu_traffic("%s:%d:%d" % (w, r["rows_per_gpu"], r["queries"]))
        line["roofline"] = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic, "kernel": r["kernel"], "kernel_ms": r["kernel_ms"],
                            "algorithmic_flop_per_launch": r["alg_flop"], "peak_source": src, "traffic_source": tsrc, "tc_refined_queries": r["tc_refined_queries"],
                            "tc_fallback_queries": r["tc_fallback_queries"], "kernel_ms_source": "CUDA events around the candidate pass of the last timed step",
                            "note": "useful flop only (tiles are padded to 128 queries x 256 rows)" if w == "ivf" else None}
    else:
        line["roofline"] = None
    line["cpu_baseline"] = r.get("cpu_baseline")
    line["e2e"] = r.get("e2e")
    line["parity"] = r.get("parity")
    line["gpu_launches"] = t["launches"]
    line["clocks"] = t.get("clocks")
    for kx in ("result", "device_seam_matches_host_merge", "blocks", "verdict"):
        if kx in r:
            line[kx] = r[kx]
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + ALL)
    ap.add_argument("--rows", type=int, default=0, help="override rows (testing only; the default is the BASELINE config)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--tune", action="append", default=[], metavar="NAME=VALUE",
                    help="kernel-variant knob passed to MoB200_SetTuning (experiments only; the default run uses none)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of each workload returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)

    env = Env(args)
    names = ALL if args.workload == "all" else [args.workload]
    runners = {"q6": run_q6, "sum": run_sum, "q1": run_q1, "bruteforce": lambda e: run_search(e, "bruteforce"), "ivf": lambda e: run_search(e, "ivf"), "dropin": run_dropin}
    lines = {}
    t_all0 = time.time()
    for i, w in enumerate(names):
        if w == "dropin" and env.world > 1:
            continue
        t0 = time.time()
        try:
            r = runners[w](env)
            if args.dump_outputs and env.rank == 0:
                dump_outputs(args.dump_outputs, r["timing"]["outputs"])
            lines[w] = finish(env, w, r)
            lines[w]["bench_seconds"] = time.time() - t0
        except Exception as ex:
            if i == 0:
                raise
            import traceback
            lines[w] = {"metric": WORKLOADS[w]["metric"], "error": "%s: %s" % (type(ex).__name__, str(ex)[:300]), "trace": traceback.format_exc()[-600:]}
    env.sampler.stop()
    if env.rank == 0:
        head = dict(lines[names[0]])
        if len(lines) > 1:
            head["workloads"] = {w: lines[w] for w in names[1:] if w in lines}
        head["bench_seconds_total"] = time.time() - t_all0
        print(json.dumps(head))
    if env.dist is not None:
        env.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    # stdout carries exactly ONE JSON line: library chatter (NCCL version banners, torchrun notices) is sent to stderr by
    # pointing fd 1 at fd 2 for the run and printing the result line to the saved descriptor.
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    _buf = []
    _print = print

    def print(*a, **k):  # noqa: A001  (only the JSON line goes through here)
        _buf.append(" ".join(str(x) for x in a))

    rc = main()
    sys.stdout.flush()
    os.dup2(_real_stdout, 1)
    for line in _buf:
        os.write(1, (line + "\n").encode())
    sys.exit(rc)
