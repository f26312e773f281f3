#!/usr/bin/env python
"""bench.py -- series/sec of the feature-extraction hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--series S] [--len L]
                    [--settings comprehensive|efficient|minimal] [--placement auto|copy|store|multicast|nccl]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (ComprehensiveFCParameters, 783 columns) over one batch of S synthetic
series of length L per GPU (default 1 000 000 x 256 = BASELINE.json configs[2], the configuration the
metric and the north-star target are quoted on).  Weak scaling: every rank owns S series (ids sharded
contiguously, no data-path collective inside the kernels); with N > 1 every rank's finished row blocks are placed
in every rank's copy of the [N*S x F] matrix (tsfresh_b200.distributed.GatheredMatrix: symmetric memory + copy
engines over NVLink while the next block's kernels run; no collective kernel).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (inputs already in HBM, CUDA-event
timed, max over ranks); `e2e` = the same pass through the C-ABI host entry point (tsfx_extract_dense with
pinned HOST buffers: H2D of the values and D2H of the feature matrix inside the timed region); `e2e_long` = from a
long (id, time, value) frame of 20 bytes per row (tsfx_extract_long_alloc, stage (a) included); `e2e_api` =
tsfresh_b200.extract_features(pandas.DataFrame).  `configs` carries the other BASELINE configurations measured in the
same run: config2 (Efficient 100 k x 256, N = 1), config4 (Comprehensive 1 M x 1024 in total, strong scaling),
config5 (roll_time_series 10 k x 4096 -> 1.21 M window views, sharded by parent), minimal (the reduction-only
kernel behind `roofline.minimal`).
`--impl reference` times the CPU path (the oracle port of the reference, all host cores) instead.
`--dump-outputs DIR` writes what the last timed step of the headline pass left in the feature matrix, so that two builds
can be compared output for output (the inputs are seeded).  DUMP_ROWS rows of the [N*S, F] matrix are drawn with a fixed
seed (all rows when there are fewer); every file holds finite values only:
  DIR/features.npy            float64 [rows, F]  the features, 0 where the feature is not finite
  DIR/features_nonfinite.npy  float32 [rows, F]  0 finite, 1 NaN, 2 +inf, 3 -inf (some features are NaN by definition,
                                                 e.g. query_similarity_count without a query)
  DIR/features_rows.npy       float64 [rows]     the row numbers, ascending
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "series/sec extract_features ComprehensiveFCParameters"
DUMP_ROWS = 6144        # x 783 columns x (8 + 4) bytes = 58 MB: the largest plan's dump stays under 64 MB


def settings_by_name(name):
    from tsfresh_b200.settings import ComprehensiveFCParameters, EfficientFCParameters, MinimalFCParameters
    return {"comprehensive": ComprehensiveFCParameters, "efficient": EfficientFCParameters,
            "minimal": MinimalFCParameters}[name]()


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def _cpu_worker(args):
    seed, count, length, name = args
    from oracle.extract import oracle_rows
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((count, length)).astype(np.float32).astype(np.float64)
    t0 = time.perf_counter()
    m = oracle_rows(list(x), settings_by_name(name))
    return m.shape, time.perf_counter() - t0


def usable_cores():
    """host cores this container may actually use: min(affinity mask, cgroup cpu.max quota)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    return max(1, n)


PORT_NOTE = ("oracle port of the reference's per-series loop, one process per usable host core; in the build container "
             "(8 cores) the UNMODIFIED reference's own extract_features(n_jobs=8) -- adapter + MultiprocessingDistributor + "
             "pivot -- runs at 63.8 series/s against 70.5 series/s for this port on the same shape, i.e. the port is 1.11x "
             "FASTER than the real reference, so ratios against it understate the speed-up "
             "(profiles/reference_vs_port_r2.json, profiles/scripts/time_reference_vs_port.py)")


class CpuArm:
    """persistent worker pool for the CPU path (spawned once: imports and pool start-up stay outside the samples)"""

    def __init__(self, length, name, cores=None):
        import multiprocessing as mp
        for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
            os.environ[k] = "1"          # the reference's own advice, docs/text/tsfresh_on_a_cluster.rst:225-231
        self.cores = cores or usable_cores()
        self.length, self.name = length, name
        self.pool = mp.get_context("spawn").Pool(self.cores)
        # warm the workers (imports), calibrate on two series per core using the in-worker time
        self.pool.map(_cpu_worker, [(900 + i, 1, length, name) for i in range(self.cores)])
        res = self.pool.map(_cpu_worker, [(1000 + i, 2, length, name) for i in range(self.cores)])
        self.per_series = max(float(np.median([r[1] for r in res])) / 2.0, 1e-4)
        self.seed = 2000

    def sample(self, target_seconds):
        """every worker gets the same number of series in ONE task (no scheduling imbalance): ~target_seconds of wall"""
        per_core = min(2000, max(8, int(target_seconds / self.per_series)))
        self.seed += 1000
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, [(self.seed + i, per_core, self.length, self.name) for i in range(self.cores)], chunksize=1)
        wall = time.perf_counter() - t0
        busy = float(np.mean([r[1] for r in res]))
        n = per_core * self.cores
        return {"value": n / wall, "unit": "series/s", "cores": self.cores, "kind": "port", "note": PORT_NOTE,
                "pool_overhead_frac": max(0.0, 1.0 - busy / wall),
                "sample": "%d series x len %d (%d per worker process, %d processes), wall %.2f s" % (n, self.length, per_core, self.cores, wall)}

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_baseline(length, name, target_seconds, cores=None):
    """series/s of the CPU path (oracle port of the reference's per-series loop) on all host cores."""
    arm = CpuArm(length, name, cores)
    try:
        return arm.sample(target_seconds)
    finally:
        arm.close()


def run_reference(args):
    """--impl reference: the CPU path on the box's host cores (rank 0 only).  One step = one bounded sample of the
    workload (the same number of series for every worker process, about 6 s of wall clock)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args.len, args.settings)
    per_step = []
    cb = None
    target = min(8.0, max(3.0, 90.0 / max(1, args.steps + args.warmup)))
    try:
        for i in range(args.warmup + args.steps):
            cb = arm.sample(target)
            if i >= args.warmup:
                per_step.append(cb)
    finally:
        arm.close()
    v = float(np.mean([c["value"] for c in per_step])) if per_step else cb["value"]
    cb = dict(cb, value=v, pool_overhead_frac=float(np.mean([c["pool_overhead_frac"] for c in per_step])) if per_step else cb["pool_overhead_frac"])
    n_ref = cb["sample"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "series/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "sample_per_step": n_ref},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "series/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_name(args):
    tag = ""
    if (args.settings, args.series, args.len) == ("comprehensive", 1_000_000, 256):
        tag = " (BASELINE.json configs[2])"
    elif (args.settings, args.len) == ("comprehensive", 1024):
        tag = " (BASELINE.json configs[3] shape)"
    elif (args.settings, args.series, args.len) == ("efficient", 100_000, 256):
        tag = " (BASELINE.json configs[1])"
    return "%sFCParameters on %d series x len %d per GPU%s, synthetic N(0,1) float32" % (
        args.settings.capitalize(), args.series, args.len, tag)


# ----------------------------------------------------------------------------------------------- GPU arm
class Bench:
    """shared state of the GPU arm: process group, stream, context, timing helpers"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from tsfresh_b200 import _lib
        self.torch, self.dist, self._lib = torch, dist, _lib
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.saved_stdout = None
        if self.world > 1:
            # keep stdout to the single JSON line: NCCL prints its version banner with printf on fd 1 when the first
            # communicator is created, so fd 1 points at stderr until the result line is written
            sys.stdout.flush()
            self.saved_stdout = os.dup(1)
            os.dup2(2, 1)
            dist.init_process_group("nccl", device_id=self.dev)
        # a non-default torch stream shared with the library, so torch's CUDA events bracket the library's launches
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        self.ctx = _lib.Context(self.local_rank, stream=self.stream.cuda_stream)
        self.plans = {}

    def plan(self, name):
        from tsfresh_b200.plan import Plan
        if name not in self.plans:
            p = Plan(settings_by_name(name))
            self.plans[name] = (p, self._lib.DevicePlan(self.ctx, p))
        return self.plans[name]

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, after_step=None):
        """W untimed + K timed calls of fn bracketed by barrier + synchronize; CUDA events on the library's stream;
        returns ms per step, max over ranks."""
        torch = self.torch
        for _ in range(warmup):
            fn()
            if after_step:
                after_step()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            fn()
            if after_step:
                after_step()
        e1.record(self.stream)
        self.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item()) / steps

    def wall(self, fn, steps, warmup):
        """host-timed variant for calls that synchronise themselves (host-buffer entry points, the Python API)"""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        t = torch.tensor([dt], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def randn(self, shape, seed):
        gen = self.torch.Generator(device=self.dev)
        gen.manual_seed(seed)
        return self.torch.randn(shape, generator=gen, device=self.dev, dtype=self.torch.float32)


def sharded_pass(B, name, values, S, L, steps, warmup, csr=None, placement="auto", rows_alloc=None, on_timed=None):
    """One configuration, device-resident: every rank extracts its S series (dense [S, L] tensor, or a CSR
    (begin, length) over `values`) and the rows are placed on every rank (tsfresh_b200.distributed.GatheredMatrix).
    on_timed(gm) is called once the timed steps have finished, before anything else writes the matrix.
    Returns (ms per step max over ranks, per-group ms of one extra timed pass over this rank's shard, launches/step, gm)."""
    from tsfresh_b200.distributed import GatheredMatrix, extract_csr_sharded_device, extract_dense_sharded_device
    torch = B.torch
    plan, dp = B.plan(name)
    gm = GatheredMatrix(rows_alloc or S, plan.n_cols, B.dev, mode=placement)      # same shape on every rank
    gm.attach(B.ctx)
    blocks = [1]

    def step():
        if csr is None:
            blocks[0] = extract_dense_sharded_device(dp, values, gm, stream=B.stream, ctx_on_current_stream=True)
        else:
            blocks[0] = extract_csr_sharded_device(dp, values, csr[0], csr[1], gm, stream=B.stream, ctx_on_current_stream=True,
                                                   max_len=L)
        if B.world > 1:
            gm.finish(B.ctx, stream=B.stream, ctx_on_current_stream=True)

    ms = B.timed(step, steps, warmup)
    if on_timed is not None:
        on_timed(gm)
    launches = B.ctx.launch_count() * blocks[0]
    gm.detach(B.ctx)
    # per-group CUDA events: one extra pass over this rank's whole shard with TSFX_FLAG_TIMING
    if csr is None:
        dp.extract_dense_device(values.data_ptr(), S, L, gm.local_ptr(0), timing=True)
    else:
        dp.extract_csr_device(values.data_ptr(), values.numel(), csr[0].data_ptr(), csr[1].data_ptr(), S, gm.local_ptr(0), timing=True,
                              max_len=L)
    torch.cuda.synchronize()
    groups = B.ctx.timings()
    return ms, groups, launches, gm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--series", type=int, default=1_000_000)
    ap.add_argument("--len", type=int, default=256)
    ap.add_argument("--settings", default="comprehensive", choices=["comprehensive", "efficient", "minimal"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline configuration only")
    ap.add_argument("--placement", default="auto", choices=["auto", "copy", "store", "multicast", "nccl"])
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's feature matrix here")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's feature matrix; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    B = Bench(args)
    torch, dist, _lib = B.torch, B.dist, B._lib
    rank, world = B.rank, B.world
    S, L = args.series, args.len
    plan, dp = B.plan(args.settings)
    F = plan.n_cols
    peaks, which = measured_peaks()

    # ---------------- headline: BASELINE.json configs[2] shape per GPU (weak scaling), device resident
    values = B.randn((S, L), 42 + 2 + rank)
    sampler = ClockSampler(B.local_rank)
    if rank == 0:
        sampler.start()
    dump = (lambda gm: dump_outputs(args.dump_outputs, gm)) if args.dump_outputs and rank == 0 else None
    ms_step, group_ms, launches_per_step, gm = sharded_pass(B, args.settings, values, S, L, args.steps, args.warmup,
                                                           placement=args.placement, on_timed=dump)
    clocks = sampler.stop() if rank == 0 else None
    value = world * S / (ms_step / 1e3)
    placement = gm.placement()

    # ---------------- impute of the resident feature matrix (SURVEY 8f row 2): an HBM-bound pass of the framework
    impute_info = None
    if world == 1:
        out_ptr = gm.local_ptr(0)
        B.ctx.impute_device(out_ptr, S, F)                     # warm-up (allocations)
        ims = B.timed(lambda: B.ctx.impute_device(out_ptr, S, F), 3, 0)
        # algorithmic bytes: the statistics sweep reads the matrix once; the replacement sweep only visits the
        # (row slice, column tile) blocks that hold a non-finite value
        impute_info = {"ms": ims, "algorithmic_GB": S * F * 8 / 1e9, "GBps": S * F * 8 / (ims * 1e-3) / 1e9,
                       "bound": "hbm", "kernels": "k_col_stats + k_col_reduce + k_impute_apply (+ one radix sort per NaN column)"}
    del gm
    torch.cuda.empty_cache()

    # ---------------- e2e: host buffers through the C ABI (H2D + kernels + D2H inside the timed region)
    e2e = e2e_long = e2e_api = None
    n_e2e = max(2, min(args.steps, 4))
    if not args.no_e2e:
        hv = torch.empty((S, L), dtype=torch.float32).pin_memory()
        hv.copy_(values.cpu())
        ho = torch.empty((S, F), dtype=torch.float64).pin_memory()
        hv_np, ho_np = hv.numpy(), ho.numpy()
        dt = B.wall(lambda: dp.extract_dense(hv_np, out=ho_np), n_e2e, 2)
        e2e = {"value": world * S / dt, "unit": "series/s", "h2d_bytes_per_step": int(S * L * 4),
               "d2h_bytes_per_step": int(S * F * 8), "ms_per_step": dt * 1e3,
               "call": "tsfx_extract_dense (C ABI, pinned host buffers)"}
        del ho, ho_np
        if world == 1 and not args.no_configs:
            # ---- the north-star boundary: a long (id, time, value) frame, 20 bytes per row, rows ordered by (id, time)
            ids = B.ctx.pinned_array((S * L,), np.int64)
            tms = B.ctx.pinned_array((S * L,), np.int64)
            ids.reshape(S, L)[:] = np.arange(S, dtype=np.int64)[:, None]
            tms.reshape(S, L)[:] = np.arange(L, dtype=np.int64)[None, :]
            vflat = hv_np.reshape(-1)

            def long_call():
                uid, mat = dp.extract_long(ids, tms, vflat)
                assert mat.shape == (S, F)
            dt = B.wall(long_call, n_e2e, 1)
            e2e_long = {"value": S / dt, "unit": "series/s", "ms_per_step": dt * 1e3,
                        "h2d_bytes_per_step": int(S * L * 20), "d2h_bytes_per_step": int(S * F * 8 + S * 8),
                        "call": "tsfx_extract_long_alloc (C ABI): pinned (id int64, time int64, value float32) columns of "
                                "%d rows in (id, time) order -> device CSR -> kernels -> pinned result" % (S * L)}
            # ---- the user-facing call: tsfresh_b200.extract_features(DataFrame) on pageable pandas columns
            import pandas as pd
            from tsfresh_b200 import extract_features
            df = pd.DataFrame({"id": np.array(ids), "time": np.array(tms), "value": np.array(vflat)})
            del ids, tms
            fc = settings_by_name(args.settings)

            def api_call():
                X = extract_features(df, column_id="id", column_sort="time", default_fc_parameters=fc,
                                     disable_progressbar=True, device=B.local_rank, n_jobs=1)
                assert X.shape == (S, F)
            dt = B.wall(api_call, max(2, n_e2e - 1), 1)
            e2e_api = {"value": S / dt, "unit": "series/s", "ms_per_step": dt * 1e3,
                       "h2d_bytes_per_step": int(S * L * 20), "d2h_bytes_per_step": int(S * F * 8 + S * 8),
                       "call": "tsfresh_b200.extract_features(pandas.DataFrame of %d rows, column_id, column_sort) -> DataFrame "
                               "[%d x %d]" % (S * L, S, F)}
            del df
        del hv, hv_np
    del values
    torch.cuda.empty_cache()

    # ---------------- the other BASELINE configurations, same JSON line
    configs = {}
    if not args.no_configs and args.settings == "comprehensive" and (S, L) == (1_000_000, 256):
        ksteps, kwarm = max(2, min(args.steps, 3)), 1

        def entry(name, workload, S_rank, L_, ms, groups, scaling, extra=None):
            pl, _ = B.plan(name)
            tot = world * S_rank if scaling == "weak" else None
            d = {"workload": workload, "ms_per_step": ms, "scaling": scaling, "columns": pl.n_cols,
                 "groups_ms": groups}
            if extra:
                d.update(extra)
            return d

        # config 2: EfficientFCParameters, 100 000 x 256 (a single-GPU configuration: N = 1 only)
        if world == 1:
            v2 = B.randn((100_000, 256), 42 + 1)
            ms2, g2, _, gm2 = sharded_pass(B, "efficient", v2, 100_000, 256, ksteps + 2, 2)
            configs["config2"] = entry("efficient", "EfficientFCParameters on 100 000 series x len 256, 1 GPU (BASELINE.json configs[1])",
                                       100_000, 256, ms2, g2, "n/a", {"value": 100_000 / (ms2 / 1e3), "unit": "series/s"})
            del gm2
            try:
                import pandas as pd
                from tsfresh_b200 import extract_features
                h2 = v2.cpu().numpy()
                df2 = pd.DataFrame({"id": np.repeat(np.arange(100_000, dtype=np.int64), 256),
                                    "time": np.tile(np.arange(256, dtype=np.int64), 100_000), "value": h2.reshape(-1)})
                fc2 = settings_by_name("efficient")
                dt2 = B.wall(lambda: extract_features(df2, column_id="id", column_sort="time", default_fc_parameters=fc2,
                                                      disable_progressbar=True, device=B.local_rank, n_jobs=1), 3, 1)
                configs["config2"]["e2e_api"] = {"value": 100_000 / dt2, "unit": "series/s", "ms_per_step": dt2 * 1e3,
                                                 "call": "tsfresh_b200.extract_features(DataFrame of 25.6 M rows)"}
                del df2, h2
            except Exception as e:                        # the bench line must survive a host-side failure here
                configs["config2"]["e2e_api"] = {"error": repr(e)}
            del v2
            torch.cuda.empty_cache()
            # reduction-only plan (class M of SURVEY 8a): the kernel the north star's HBM target is stated for
            vm = B.randn((S, L), 42 + 9)
            msm, gmn, _, gmm = sharded_pass(B, "minimal", vm, S, L, ksteps + 2, 2)
            plm, _ = B.plan("minimal")
            configs["minimal"] = entry("minimal", "MinimalFCParameters on 1 000 000 series x len 256 (class-M reductions + median)",
                                       S, L, msm, gmn, "n/a", {"value": S / (msm / 1e3), "unit": "series/s"})
            del vm, gmm
            torch.cuda.empty_cache()

        # config 4: ComprehensiveFCParameters, 1 000 000 x 1024 in total, STRONG scaling: each rank takes 1 M / N series
        S4 = 1_000_000 // world
        v4 = B.randn((S4, 1024), 42 + 3 + 17 * rank)
        ms4, g4, _, gm4 = sharded_pass(B, "comprehensive", v4, S4, 1024, ksteps, kwarm, placement=args.placement)
        configs["config4"] = entry("comprehensive", "ComprehensiveFCParameters on 1 000 000 series x len 1024 in total, "
                                   "%d series per rank (BASELINE.json configs[3], strong scaling)" % S4, S4, 1024, ms4, g4, "strong",
                                   {"value": world * S4 / (ms4 / 1e3), "unit": "series/s", "placement": gm4.placement()})
        del v4, gm4
        torch.cuda.empty_cache()

        # config 5: roll_time_series(rolling_direction=32, max_timeshift=255, min_timeshift=255) over 10 000 x 4096
        # -> 1.21 M windows of 256 rows as (begin, len) views on the parents' buffer, sharded by parent
        from tsfresh_b200 import _lib as lib5
        from tsfresh_b200.distributed import shard_windows
        P5, L5 = 10_000, 4096
        t0 = time.perf_counter()
        begin5 = (np.arange(P5, dtype=np.int64) * L5)
        wb, wl, wp, we = lib5.roll_windows(begin5, np.full(P5, L5, dtype=np.int32), 32, 255, 255)
        roll_ms = (time.perf_counter() - t0) * 1e3
        lo5, hi5 = shard_windows(wp, P5, world, rank)
        per5 = (len(wb) + world - 1) // world
        n5 = hi5 - lo5
        v5 = B.randn((P5, L5), 42 + 4)                       # every rank holds the (164 MB) parent buffer
        wb_d = torch.from_numpy(wb[lo5:hi5].copy()).to(B.dev)
        wl_d = torch.from_numpy(wl[lo5:hi5].copy()).to(B.dev)
        mx = torch.tensor([n5], device=B.dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        ms5, g5, _, gm5 = sharded_pass(B, "comprehensive", v5.reshape(-1), n5, 256, ksteps, kwarm, csr=(wb_d, wl_d),
                                       placement=args.placement, rows_alloc=int(mx.item()))
        nt = torch.tensor([n5], device=B.dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(nt)
        configs["config5"] = entry("comprehensive", "roll_time_series(rolling_direction=32, max_timeshift=255, min_timeshift=255) over "
                                   "10 000 series x len 4096 -> %d window views x 256 -> ComprehensiveFCParameters "
                                   "(BASELINE.json configs[4]); windows sharded by parent" % len(wb), n5, 256, ms5, g5, "strong",
                                   {"value": int(nt.item()) / (ms5 / 1e3), "unit": "windows/s", "windows": int(len(wb)),
                                    "roll_windows_host_ms": roll_ms, "placement": gm5.placement()})
        del v5, gm5, wb_d, wl_d
        torch.cuda.empty_cache()

    if rank != 0:
        group_ms = {}
    if rank == 0:
        roofline = None
        groups = {}
        tj = None
        for tf in ("traffic_r2.json", "traffic_r1.json"):
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", tf)))
                tj["_file"] = tf
                break
            except Exception:
                tj = None
        same_workload = bool(tj) and (tj["workload"]["series"], tj["workload"]["len"], tj["workload"]["settings"]) == (S, L, args.settings)
        if group_ms:
            # algorithmic bytes per series of one kernel group: the 4*L value bytes it reads plus the 8 bytes per
            # output column it writes (DESIGN.md "Roofline"); whole pass: 4L + 12 + 8F (SURVEY.md section 8d)
            ncols = dict(group_columns(plan))
            clk = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
            for g, ms in group_ms.items():
                by = S * 16 * F if g == "assemble" else S * (4 * L + 8 * ncols.get(g, 0))
                groups[g] = {"ms": ms, "columns": ncols.get(g, 0), "algorithmic_GBps": by / (ms * 1e-3) / 1e9}
                ginst = tj.get("k_" + g, {}).get("inst_executed") if same_workload else None
                if ginst:
                    groups[g]["issue_frac"] = ginst / (ms * 1e-3) / (148 * 4 * clk)
            dom = max(group_ms, key=lambda g: group_ms[g])
            ach = groups[dom]["algorithmic_GBps"]
            traffic, limiter, issue = None, None, None
            if same_workload and ("k_" + dom) in tj:
                kd = tj["k_" + dom]
                traffic = kd["traffic_bytes"] / 1e9
                limiter = "ncu (%s): fp64 pipe %.0f%% active, issue %.0f%% active" % (tj["_file"], kd["fp64_pipe_active_pct"], kd["issue_active_pct"])
                if kd.get("inst_executed"):
                    # supplementary compute roofline: warp instructions per launch from the committed ncu capture of the
                    # same workload; rate measured live; peak = 148 SMs x 4 schedulers x 1 warp instruction per clock
                    a_i = kd["inst_executed"] / (group_ms[dom] * 1e-3)
                    issue = {"bound": "instruction issue", "achieved": a_i / 1e12, "peak": 148 * 4 * clk / 1e12,
                             "unit": "T warp-inst/s", "frac": a_i / (148 * 4 * clk), "warp_inst_per_series": kd["inst_executed"] / S}
            roofline = {"kernel": "k_" + dom, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"],
                        "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)" if which == "measured" else "fallback 6650 GB/s",
                        "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "traffic_unit": "GB per launch (ncu dram read+write)",
                        "algorithmic_GB_per_launch": S * (4 * L + 8 * ncols.get(dom, 0)) / 1e9,
                        "limiter": limiter or "the dominant kernel is instruction-issue bound, not HBM bound (DESIGN.md section 4)",
                        "compute_roofline": issue,
                        "whole_pass_GBps": S * (4 * L + 12 + 8 * F) / (ms_step * 1e-3) / 1e9,
                        "groups": groups}
            if impute_info:
                impute_info["frac_of_hbm_peak"] = impute_info["GBps"] / peaks["hbm_gbs"]
                roofline["impute"] = impute_info
            if "minimal" in configs:
                # the reduction-only (class M) kernel: the kernel the north star's ">= 60 % of the HBM-read roofline" is about
                gm_ = configs["minimal"]["groups_ms"]
                plm, _ = B.plan("minimal")
                kname = "moments" if "moments" in gm_ else "basic"
                if kname in gm_:
                    cols_m = group_columns(plm).get("basic", 0)
                    bym = S * (4 * L + 8 * cols_m)
                    roofline["minimal"] = {"kernel": "k_" + kname, "bound": "hbm", "ms": gm_[kname],
                                           "achieved": bym / (gm_[kname] * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                           "frac": bym / (gm_[kname] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                           "read_only_frac": S * 4 * L / (gm_[kname] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                           "algorithmic_GB_per_launch": bym / 1e9, "columns": cols_m,
                                           "note": "class-M reductions of MinimalFCParameters at 1 M x 256; the median column is a sort (k_sorted), listed in configs.minimal.groups_ms"}
        cb = None
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_baseline(L, args.settings, args.cpu_seconds)
        line = {
            "metric": METRIC, "value": value, "unit": "series/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args), "columns": F, "global_series": world * S,
                       "l2": "inputs (%.2f GB) + outputs (%.2f GB) per step exceed the 126 MB L2" % (S * L * 4 / 1e9, S * F * 8 / 1e9),
                       "parallelism": "ids sharded contiguously over %d rank(s)%s" % (world, "" if world == 1 else
                                      "; every rank's rows placed on every rank per row block by %s (tsfresh_b200.distributed.GatheredMatrix)" % placement)},
            "clocks": clocks, "e2e": e2e, "e2e_long": e2e_long, "e2e_api": e2e_api,
            "gpu_launches": int(launches_per_step * args.steps),
            "roofline": roofline, "cpu_baseline": cb, "configs": configs,
        }
        if B.saved_stdout is not None:
            sys.stdout.flush()
            try:
                import ctypes
                ctypes.CDLL(None).fflush(None)       # whatever C code buffered for "stdout" leaves through stderr too
            except Exception:
                pass
            os.dup2(B.saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        if B.saved_stdout is not None and rank != 0:
            os.dup2(B.saved_stdout, 1)
        dist.destroy_process_group()


def dump_outputs(directory, gm):
    """DUMP_ROWS rows of gm.full (all rows when there are fewer), drawn with a fixed seed -> directory/*.npy"""
    import torch
    n = gm.full.shape[0]
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    sample = gm.full.index_select(0, torch.from_numpy(rows).to(gm.full.device)).cpu().numpy()
    code = np.zeros(sample.shape, np.float32)
    code[np.isnan(sample)] = 1
    code[sample == np.inf] = 2
    code[sample == -np.inf] = 3
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "features.npy"), np.where(code == 0, sample, 0.0))
    np.save(os.path.join(directory, "features_nonfinite.npy"), code)
    np.save(os.path.join(directory, "features_rows.npy"), rows.astype(np.float64))


def group_columns(plan):
    """number of output columns each kernel group writes (mirrors group_of() in csrc/tsfx_api.cu)."""
    from tsfresh_b200.plan import CALC
    G = {"sorted": ["SYMMETRY_LOOKING", "HAS_DUPLICATE", "MEDIAN", "PERCENTAGE_OF_REOCCURRING_VALUES_TO_ALL_VALUES",
                    "PERCENTAGE_OF_REOCCURRING_DATAPOINTS_TO_ALL_DATAPOINTS", "SUM_OF_REOCCURRING_VALUES",
                    "SUM_OF_REOCCURRING_DATA_POINTS", "RATIO_VALUE_NUMBER_TO_TIME_SERIES_LENGTH", "QUANTILE",
                    "MEAN_N_ABSOLUTE_MAX", "CHANGE_QUANTILES", "FRIEDRICH_COEFFICIENTS", "MAX_LANGEVIN_FIXED_POINT"],
         "spectral": ["FFT_COEFFICIENT", "FFT_AGGREGATED", "SPKT_WELCH_DENSITY", "FOURIER_ENTROPY", "CWT_COEFFICIENTS"],
         "la": ["AR_COEFFICIENT", "AUGMENTED_DICKEY_FULLER"],
         "entropy": ["SAMPLE_ENTROPY", "APPROXIMATE_ENTROPY"],
         "seq": ["LEMPEL_ZIV_COMPLEXITY", "PERMUTATION_ENTROPY"], "peaks": ["NUMBER_CWT_PEAKS"]}
    rev = {}
    for g, names in G.items():
        for n in names:
            rev[CALC["TSFX_" + n]] = g
    out = {}
    for c in plan.descs["calc"]:
        g = rev.get(int(c), "basic")
        out[g] = out.get(g, 0) + 1
    return out


if __name__ == "__main__":
    main()
