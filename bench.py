#!/usr/bin/env python
"""bench.py -- contract benchmark of the legate.sparse_b200 hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank/GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

Metric (BASELINE.json): CSR SpMV GFLOP/s and fraction of the HBM roofline.  Workload at N=1:
BASELINE.json configs[1] -- the 5-point Laplacian of examples/pde.py on a 3162 x 3162 interior grid
(N = 9,998,244 rows, nnz = 49,978,572), fp64 values, int32 indices, one SpMV per step.  At N>1 the grid
grows along y (3162 x 3162*N; weak scaling, 1-D row blocks) and every step includes the x halo exchange.

One JSON line on stdout (rank 0).  `value` = device-resident SpMV throughput (CUDA events, max over ranks);
`e2e` = the same metric through the public API with host (pinned) x and y, H2D + D2H inside the timed region;
`roofline` = algorithmic bytes / measured kernel time vs MEASURED_PEAKS.json; `cpu_baseline` = the CPU
oracle (OpenMP restatement of the reference's spmv_omp.cc) on this box's host cores.
`--impl reference` times that CPU implementation alone (the reference itself needs legate.core/Legion and
cannot be built here, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N1 = 3162  # interior grid edge: (nx-2) with nx = 3164 (SURVEY 8: L5)
# --dump-outputs: y has 10M fp64 rows per GPU (80 MB), so a fixed, seeded sample of 2^22 rows over all ranks is written
# (32 MB); the same arguments give the same rows, so two builds can be compared output for output
DUMP_ROWS = 1 << 22
DUMP_SEED = 20240
METRIC = "csr_spmv_gflops"
WORKLOAD = "5-pt Laplacian (examples/pde.py operator) 3162x3162 interior grid per GPU, fp64 CSR SpMV, int32 indices"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def alg_bytes(nrows, ncols, nnz, sv=8, si=4, sp=4):
    """SURVEY 8(d): B = nnz*(sv+si) + (nrows+1)*sp + ncols*sv + nrows*sv."""
    return nnz * (sv + si) + (nrows + 1) * sp + ncols * sv + nrows * sv


# ----------------------------------------------------------------------------------------------------------
# host-side Laplacian assembly (numpy) for the CPU arms -- same operator as gallery.laplacian_5pt
# ----------------------------------------------------------------------------------------------------------
def laplacian_host(n1, n2):
    N = n1 * n2
    i = np.arange(N, dtype=np.int64)
    a = float((n1 + 1) ** 2)
    g = float((n2 + 1) ** 2)
    c = -2 * a - 2 * g
    cols = np.stack([i - n1, i - 1, i, i + 1, i + n1], axis=1)
    vals = np.tile(np.array([g, a, c, a, g]), (N, 1))
    valid = np.ones((N, 5), dtype=bool)
    valid[:, 0] = i >= n1
    valid[:, 1] = (i % n1) != 0
    valid[:, 3] = (i % n1) != n1 - 1
    valid[:, 4] = i < N - n1
    indptr = np.zeros(N + 1, dtype=np.int32)
    np.cumsum(valid.sum(axis=1), out=indptr[1:])
    return indptr, cols[valid].astype(np.int32), vals[valid], N


def cpu_arm(budget_s, indptr=None, indices=None, data=None, min_reps=20, max_reps=400, warmups=10):
    """The CPU implementation of the path on this box's host cores: the OpenMP oracle (reference spmv_omp.cc:36-45
    restated) on the L5 matrix.  ONE routine for both `cpu_baseline` and `--impl reference`, so the two agree:
    arrays first-touched in parallel (pages spread over the NUMA nodes), thread count calibrated by the median of
    3 timed products per candidate (after 2 warm-ups each), >= 10 warm-ups, then the MEDIAN of >= 20 timed products
    (bounded by `budget_s`).  Returns GFLOP/s, ms, reps, threads, candidates tried."""
    from oracle import oracle as orc

    orc.build()
    if indptr is None:
        indptr, indices, data, _ = laplacian_host(N1, N1)
    n = indptr.shape[0] - 1
    ncpu = os.cpu_count() or 1
    orc.set_num_threads(ncpu)
    indptr, indices, data = (orc.first_touch_copy(a) for a in (indptr, indices, data))
    x = orc.first_touch_copy(np.random.default_rng(0).random(n))
    y = orc.first_touch_copy(np.zeros(n))

    def timed():
        t = time.perf_counter()
        orc.spmv(indptr, indices, data, x, omp=True, out=y)
        return time.perf_counter() - t

    cands = sorted({max(1, ncpu), max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, 8)}, reverse=True)
    tried = {}
    for c in cands:
        orc.set_num_threads(c)
        timed(); timed()
        tried[c] = float(np.median([timed() for _ in range(3)]))
    best = min(tried, key=tried.get)
    orc.set_num_threads(best)
    for _ in range(warmups):
        timed()
    times, t0 = [], time.perf_counter()
    while len(times) < max_reps and (len(times) < min_reps or time.perf_counter() - t0 < budget_s):
        times.append(timed())
    nnz = int(indptr[-1])
    med = float(np.median(times))
    return {"gflops": 2.0 * nnz / med / 1e9, "ms": med * 1e3, "reps": len(times), "threads": best,
            "nnz": nnz, "rows": n, "calibration_ms": {str(k): v * 1e3 for k, v in tried.items()},
            "min_ms": float(min(times)) * 1e3, "max_ms": float(max(times)) * 1e3}


# ----------------------------------------------------------------------------------------------------------
# clocks sampler (NVML; nvidia-smi fallback)
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting",
               0x10: "sync_boost"}

    def __init__(self, index):
        self.index = index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self._h = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self._h is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------------
# reference arm: CPU implementation of the path on this box's host cores
# ----------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    try:
        from oracle import oracle as orc

        orc.build()
    except Exception as exc:
        print(json.dumps({"impl": "reference", "unavailable": f"CPU oracle could not be built: {exc}"}), flush=True)
        return 0
    # one shard of the workload = the bounded sample; K = args.steps timed products (bounded to ~2 minutes),
    # value from the MEDIAN product time (a single slow outlier -- page migration, a noisy neighbour -- must not
    # decide the line the GPU arm is divided by)
    steps = int(max(20, min(args.steps, 4000)))
    r = cpu_arm(budget_s=120.0, min_reps=20, max_reps=steps, warmups=max(args.warmup, 10))
    gf, n, nnz, threads = r["gflops"], r["rows"], r["nnz"], r["threads"]
    sample = (f"{r['reps']} SpMVs of one 3162x3162-grid shard ({n} rows, {nnz} nnz), OpenMP dynamic,128, {threads} threads "
              f"(calibrated over {sorted(int(k) for k in r['calibration_ms'])}), median {r['ms']:.2f} ms "
              f"[min {r['min_ms']:.2f}, max {r['max_ms']:.2f}], arrays first-touched in parallel")
    line = {
        "impl": "reference", "metric": METRIC, "value": gf, "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": r["reps"], "warmup": max(args.warmup, 10), "ms_per_step": r["ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rows": n, "nnz": nnz,
                   "note": "reference's CPU leaf task (spmv_omp.cc) restated in oracle/oracle.c; the reference "
                           "itself needs legate.core/Legion and cannot be built here"},
        "cpu_baseline": {"value": gf, "unit": "GFLOP/s", "cores": threads, "kind": "port", "sample": sample,
                         "calibration_ms": r["calibration_ms"]},
        "e2e": {"value": gf, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def _events(torch, n):
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]


def _time_launches(torch, fn, reps, warm=3):
    """median / min device time (ms) of `fn` over `reps` launches, CUDA events on the current stream."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = _events(torch, reps)
    for s, e in ev:
        s.record()
        fn()
        e.record()
    torch.cuda.synchronize()
    ts = sorted(s.elapsed_time(e) for s, e in ev)
    return ts[len(ts) // 2], ts[0]


def run_gpu(args):
    import torch

    import legate.sparse_b200 as sparse  # noqa: F401
    from legate.sparse_b200 import _ops, gallery
    from legate.sparse_b200 import dist as bd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; legate.sparse_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        bd.init_process_group("nccl")
    import torch.distributed as dist

    n1, n2 = N1, N1 * world
    Nglob = n1 * n2
    plan = bd.RowBlockPlan(Nglob, world)
    lo, hi = plan.rows(rank)
    local = gallery.laplacian_5pt(n1, n2, np.float64, row_lo=lo, row_hi=hi)
    nnz_local = local.nnz
    A = bd.dist_csr_array(local, (Nglob, Nglob), rank=rank, nranks=world)
    x_full = A.new_full_vector(np.float64)
    xl = A.local_view(x_full)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    xl.copy_(torch.rand(xl.shape[0], dtype=torch.float64, device="cuda", generator=g))
    y = torch.empty(hi - lo, dtype=torch.float64, device="cuda")
    Al = A.local
    spmv_plan = Al._get_plan()
    xin = x_full[: Al.shape[1]]

    graphed = world > 1 and os.environ.get("B2S_BENCH_GRAPH", "1") != "0"

    def step():
        # one product of this rank's shard INCLUDING the x halo exchange.  At N>1 the exchange is fused into the SpMV
        # launch (push + in-kernel wait, device-side epochs) and the step is replayed from a CUDA graph.
        if graphed:
            A.dot_graphed(x_full, y)
        else:
            A.dot(x_full, out=y)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    fused_info = A._fused.get((id(Al), x_full.data_ptr())) if world > 1 else None
    exchange_path = "none" if world == 1 else (f"fused-{fused_info['mode']}" if fused_info else f"nccl-{A.exchange_mode}")

    # ---- correctness of the timed path at N>1: the same product with the halo exchanged by NCCL send/recv and the
    # plain (un-fused) kernel on the same shard must agree; a timeout inside a fused wait raises here
    verified = None
    if world > 1 and os.environ.get("B2S_BENCH_NOVERIFY", "0") != "1":
        y_ref = torch.empty_like(y)
        A.exchange(x_full)                       # NCCL p2p (or all-gather) into the same buffer: same values
        _ops.spmv(Al.indptr, Al.indices, Al.data, xin, y_ref, Al.shape, plan=spmv_plan)
        step()
        torch.cuda.synchronize()
        A.check_peer()
        err = float((y - y_ref).abs().max())
        scale = float(y_ref.abs().max())
        verified = bool(err <= 1e-12 * scale)
        vt = torch.tensor([1 if verified else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(vt, op=dist.ReduceOp.MIN)
        verified = bool(int(vt[0]))
        if not verified:
            raise SystemExit(f"bench.py: rank {rank}: fused-exchange product differs from the NCCL-exchanged one "
                             f"(max err {err:.3e}, scale {scale:.3e})")

    sampler = ClockSampler(local_rank)
    kern_ev = _events(torch, args.steps)
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    barrier()
    t_start.record()
    for s, e in kern_ev:
        s.record()
        step()
        e.record()
    t_end.record()
    barrier()
    clocks = sampler.stop()
    dump = {}
    if args.dump_outputs:   # y of the last timed step, as the caller of the product receives it
        k = min(hi - lo, DUMP_ROWS // world)
        rows = np.sort(np.random.default_rng(DUMP_SEED + rank).choice(hi - lo, size=k, replace=False))
        dump["y" if world == 1 else f"y_rank{rank}"] = y[torch.from_numpy(rows).to(y.device)].cpu().numpy()
    elapsed_ms = t_start.elapsed_time(t_end)
    kern_ms = float(np.mean([s.elapsed_time(e) for s, e in kern_ev]))
    bare_ms = kern_ms
    if world > 1:
        # for reference only: the bare kernel without any exchange (not what `value` / `roofline` are computed from)
        bare_ms, _ = _time_launches(torch, lambda: _ops.spmv(Al.indptr, Al.indices, Al.data, xin, y, Al.shape, plan=spmv_plan), 50)
    stats = torch.tensor([elapsed_ms, kern_ms, bare_ms], dtype=torch.float64, device="cuda")
    nnz_t = torch.tensor([nnz_local], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(nnz_t, op=dist.ReduceOp.SUM)
    elapsed_ms, kern_ms, bare_ms = float(stats[0]), float(stats[1]), float(stats[2])
    nnz_glob = int(nnz_t[0])
    ms_per_step = elapsed_ms / args.steps
    value = 2.0 * nnz_glob / (ms_per_step * 1e-3) / 1e9

    # ---- e2e: public API, host (pinned) vectors in and out, every step -----------------------------------
    x_host = torch.empty(Al.shape[1] if world == 1 else xl.shape[0], dtype=torch.float64).pin_memory()
    x_host.copy_(xl.cpu() if world > 1 else xin.cpu())
    y_host = torch.empty(hi - lo, dtype=torch.float64).pin_memory()
    xh_np, yh_np = x_host.numpy(), y_host.numpy()

    def e2e_step():
        if world == 1:
            Al.dot(xh_np, out=yh_np)  # H2D x, kernel, D2H y -- the call a user makes
        else:
            xl.copy_(x_host, non_blocking=True)
            step()
            y_host.copy_(y, non_blocking=False)

    e2e_steps = max(3, min(args.steps, 50))
    for _ in range(10):      # warm-up: copy streams / events of the pipeline are created on the first calls
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_gf = 2.0 * nnz_glob * e2e_steps / float(e2e_t[0]) / 1e9
    assert np.isfinite(yh_np).all()
    if world == 1:   # the host-vector product equals the device-resident one bit for bit (same tiles, same kernel)
        assert np.array_equal(yh_np, y.cpu().numpy()), "e2e (host vectors) result differs from the device-resident product"

    peak, peak_src = measured_peak()
    B = alg_bytes(hi - lo, Al.shape[1] if world == 1 else (hi - lo) + A.recv_elems, nnz_local)
    # roofline of the dominant kernel = the SpMV launch.  At N>1 that launch contains the exchange, so the step time is
    # the kernel time (per-launch events around the graph replay); max over ranks.
    achieved = B / (kern_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "spmv_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None

    # ---- the other hot-path rows (all ranks take part at N>1) ------------------------------------------------
    extras = {}
    if not args.no_extras:
        if world == 1:
            extras = other_rows_of_the_path(torch, gallery, peak, args)
        else:
            del local
            extras = sharded_rows_of_the_path(torch, dist, bd, gallery, peak, rank, world, args)

    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)

    if rank != 0:
        return 0

    # ---- CPU baseline on rank 0 (N=1 only; bounded sample) ------------------------------------------------
    cpu = None
    extra = {}
    if world == 1 and not args.no_cpu:
        ip, ix, dv = (t.cpu().numpy() for t in (Al.indptr, Al.indices, Al.data))
        try:
            r = cpu_arm(args.cpu_budget, ip, ix, dv)
            cpu = {"value": r["gflops"], "unit": "GFLOP/s", "cores": r["threads"], "kind": "port",
                   "sample": f"{r['reps']} full SpMVs of the same matrix ({r['rows']} rows, {r['nnz']} nnz), "
                             f"median {r['ms']:.2f} ms [min {r['min_ms']:.2f}, max {r['max_ms']:.2f}], OpenMP oracle "
                             f"(reference spmv_omp.cc restated), same routine as --impl reference",
                   "calibration_ms": r["calibration_ms"]}
        except Exception as exc:  # the GPU numbers above must survive a broken host toolchain
            cpu = {"value": None, "unit": "GFLOP/s", "cores": 0, "kind": "port", "sample": f"unavailable: {exc}"}
        try:  # scipy (the reference tests' oracle): single-threaded csr_matvec, for context
            import scipy.sparse as sp

            S = sp.csr_array((dv, ix, ip), shape=Al.shape)
            xs = xin.cpu().numpy()
            S @ xs
            ts = []
            for _ in range(3):
                t = time.perf_counter(); S @ xs; ts.append(time.perf_counter() - t)
            extra["scipy_gflops_1thread"] = 2.0 * nnz_local / min(ts) / 1e9
            extra["host_cpu_count"] = os.cpu_count()
        except Exception as exc:  # pragma: no cover
            extra["scipy_error"] = str(exc)

    launches_per_step = 1 if (world == 1 or (fused_info and fused_info["mode"] == "halo") or not fused_info) else \
        1 + sum(1 for b in fused_info["blocks"].values() if b is not None)
    line = {
        "metric": METRIC, "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_rows": Nglob, "global_nnz": nnz_glob, "rows_per_gpu": hi - lo,
                   "index_bytes": 4, "indptr_bytes": 4, "partition": f"1-D row blocks x{world}",
                   "x_exchange": A.exchange_mode, "exchange_path": exchange_path, "halo_elems_per_rank": A.recv_elems,
                   "exchange_fused_into_spmv_launch": bool(fused_info),
                   "exchange_overlapped_with_interior_tiles": bool(fused_info and fused_info["mode"] == "halo"),
                   "step_replayed_from_cuda_graph": bool(graphed),
                   "result_verified_against_nccl_exchange": verified,
                   "l2": "inputs larger than L2 (matrix stream 600 MB + x/y 160 MB per step vs 126 MB L2); no flush",
                   "tile_config": int(spmv_plan.config), "kernel_flavor": ("short-rows" if spmv_plan.short_rows else
                                                                           "uniform-rows" if spmv_plan.uniform else "generic"),
                   "x_lines_per_warp_gather": spmv_plan.lines_per_warp},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": B,
                     "kernel": spmv_plan.kernel_name, "kernel_ms": kern_ms,
                     "timing": "mean of per-launch CUDA events inside the timed region, max over ranks"
                               + ("; the launch includes the fused halo exchange" if world > 1 else ""),
                     "bare_kernel_ms_no_exchange": bare_ms},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_gf, "unit": "GFLOP/s", "h2d_bytes_per_step": int(x_host.numel() * 8) * world,
                "d2h_bytes_per_step": int(y_host.numel() * 8) * world, "steps": e2e_steps,
                "api": "csr_array.dot(x_host, out=y_host)" if world == 1 else "shard copy-in + dist_csr_array.dot + copy-out"},
        "clocks": clocks,
        "gpu_launches": args.steps * world * launches_per_step,
    }
    if extras:
        line["extras"] = extras
    line.update(extra)
    print(json.dumps(line), flush=True)
    return 0


def _r32_case(torch, gallery, _ops, peak, dtype, reps=20):
    """BASELINE config 4 (R32: 10M x 10M, 32 uniformly random columns per row) on one GPU: the product, its HBM
    roofline fraction, and -- measured in the same run -- the gather ceiling of this access pattern (b2s_probe_gather:
    320 M independent reads of the same vector, nothing else), since random columns are bound by the L1 tag stage
    (one lookup per distinct 128-byte line per cycle per SM), not by HBM."""
    from legate.sparse_b200 import _lib
    from legate.sparse_b200.runtime import ptr, runtime, vt_code

    n = 10_000_000
    A = gallery.random_fixed(n, n, 32, dtype)
    tdt = torch.float32 if np.dtype(dtype) == np.float32 else torch.float64
    x = torch.rand(n, dtype=tdt, device="cuda")
    y = torch.empty(n, dtype=tdt, device="cuda")
    plan = A._get_plan()
    med, mn = _time_launches(torch, lambda: _ops.spmv(A.indptr, A.indices, A.data, x, y, A.shape, plan=plan), reps)
    sv = np.dtype(dtype).itemsize
    B = alg_bytes(n, n, A.nnz, sv=sv)
    scratch = torch.zeros(4, dtype=tdt, device="cuda")
    probe = lambda: _lib.check(_lib.lib.b2s_probe_gather(vt_code(tdt), n, A.nnz, ptr(x), ptr(scratch), runtime.stream_ptr()))
    g_med, g_min = _time_launches(torch, probe, 10)
    # the product cannot be faster than its gathers, and streams the matrix through the same L2 on top
    stream_ms = (A.nnz * (sv + 4) + n * (4 + sv)) / (peak * 1e9) * 1e3
    out = {"rows": n, "nnz": A.nnz, "ms": med, "min_ms": mn, "gflops": 2.0 * A.nnz / (med * 1e-3) / 1e9,
           "algorithmic_bytes": B, "frac_of_hbm_peak": B / (med * 1e-3) / 1e9 / peak,
           "gather_ceiling_ms": g_med, "gather_ceiling_ggather_per_s": A.nnz / (g_med * 1e-3) / 1e9,
           "frac_of_gather_ceiling": g_med / med, "matrix_stream_ms_at_hbm_peak": stream_ms,
           "lines_per_warp": plan.lines_per_warp, "kernel": plan.kernel_name,
           "limiter": "L1TEX tag stage: one distinct 128-byte line per cycle per SM (see profiles/ and DESIGN.md 3.2)"}
    # the public call (csr_array.dot) column-splits by itself when x exceeds L2 and the columns are scattered (fp64: x =
    # 80 MB -> two column blocks, each gathering from a 40 MB slice); `ms` above stays the unsplit kernel
    if A._wants_col_split(plan):
        A.dot(x, out=y)
        y_ref = torch.empty_like(y)
        _ops.spmv(A.indptr, A.indices, A.data, x, y_ref, A.shape, plan=plan)
        err = float((y - y_ref).abs().max() / y_ref.abs().max())
        cs_med, cs_min = _time_launches(torch, lambda: A.dot(x, out=y), reps)
        out["col_split"] = {"blocks": len(A._col_split()), "ms": cs_med, "min_ms": cs_min,
                            "gflops": 2.0 * A.nnz / (cs_med * 1e-3) / 1e9, "frac_of_gather_ceiling": g_med / cs_med,
                            "max_rel_diff_vs_unsplit": err, "kernel": A._col_split()[0][1].kernel_name}
    del A, x, y
    torch.cuda.empty_cache()
    return out


def _spgemm_rmat_case(torch, gallery, peak, args):
    """BASELINE config 5: C = A @ A for an R-MAT graph (a,b,c,d = .57,.19,.19,.05), scale 22, edge factor 16, fp64.
    nnz(C) is hundreds of GB, so the product runs through the row-chunked driver (csr.spgemm_chunked): chunks of
    <= 1.5e9 products, each through the two-pass SpGEMM, reduced to (nnz, checksum) and dropped.  scipy on the host:
    a BOUNDED SAMPLE -- 4096 random rows of A times A -- scaled by the share of products (scipy's full product would
    take hours and ~1 TB).  B = nnz_A*12 + products*12 (B rows streamed per A entry) + nnz_C*12 + indptrs (SURVEY 8d)."""
    from legate.sparse_b200.csr import spgemm_chunked

    scale = int(os.environ.get("B2S_BENCH_RMAT_SCALE", "22"))
    ef = 16
    A = gallery.rmat(scale, ef, seed=42)
    n = A.shape[0]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, st = spgemm_chunked(A, A, max_products=int(1.5e9), keep=False)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    byts = A.nnz * 12 + st["products"] * 12 + st["nnz"] * 12 + 3 * 8 * (n + 1)
    out = {"scale": scale, "edge_factor": ef, "rows": n, "nnz_a": A.nnz, "products": st["products"], "nnz_c": st["nnz"],
           "chunks": st["chunks"], "max_chunk_nnz": st["max_chunk_nnz"], "ms": dt * 1e3,
           "gflops": 2.0 * st["products"] / dt / 1e9, "model_bytes": byts, "B_over_t_frac": byts / dt / 1e9 / peak,
           "checksum": st["checksum"], "c_bytes_if_kept": st["nnz"] * 12}
    if not args.no_cpu:
        import scipy.sparse as sp

        S = sp.csr_array((A.data.cpu().numpy(), A.indices.cpu().numpy(), A.indptr.cpu().numpy()), shape=A.shape)
        rows = np.sort(np.random.default_rng(3).choice(n, size=min(4096, n), replace=False))
        lens = np.diff(S.indptr)
        sample_products = int(lens[S.indices[np.concatenate([np.arange(S.indptr[r], S.indptr[r + 1]) for r in rows])]].sum())
        Ssub = S[rows]
        t0 = time.perf_counter()
        Csub = Ssub @ S
        ts = time.perf_counter() - t0
        out.update({"scipy_sample_rows": int(rows.shape[0]), "scipy_sample_products": sample_products,
                    "scipy_sample_ms": ts * 1e3, "scipy_sample_nnz_c": int(Csub.nnz),
                    "scipy_ms_extrapolated_by_products": ts * 1e3 * st["products"] / max(sample_products, 1),
                    "speedup_vs_scipy_extrapolated": (ts * st["products"] / max(sample_products, 1)) / dt})
        del S, Ssub, Csub
    del A
    torch.cuda.empty_cache()
    return out


def other_rows_of_the_path(torch, gallery, peak, args):
    """The other hot-path rows of SURVEY 8 at N=1, so one bench line records them all (bounded: ~1 minute).
    R32: BASELINE config 4 (the north-star shape) fp32 and fp64 with the measured gather ceiling.
    CG: examples/pde.py -nx 4096 -ny 4096 -throughput -max_iter 300 (BASELINE config 3) next to scipy's cg on the host.
    SpGEMM: examples/spgemm_microbenchmark.py shape (banded, 11 nnz/row) at n = 1M.  SpMM: dot_microbenchmark -op spmm."""
    from legate.sparse_b200 import _ops, linalg

    only = [v for v in os.environ.get("B2S_BENCH_EXTRAS", "").split(",") if v]   # development: run a subset
    want = lambda name: not only or name in only
    out = {}
    for key, dt in (("r32_fp32", np.float32), ("r32_fp64", np.float64)):
        if not want("r32"):
            continue
        try:
            out[key] = _r32_case(torch, gallery, _ops, peak, dt)
        except Exception as exc:  # pragma: no cover
            out[key + "_error"] = repr(exc)
    try:
        if not want("cg"):
            raise KeyError("skipped")
        A = gallery.laplacian_5pt(4094, 4094, np.float64)
        b = torch.ones(A.shape[0], dtype=torch.float64, device="cuda")
        linalg.cg(A, b, tol=1e-10, maxiter=30)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        x, iters = linalg.cg(A, b, tol=1e-10, maxiter=300)
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e)
        N, nnz = A.shape[0], A.nnz
        fused_bytes = nnz * 12 + N * 20 + 9 * 8 * N
        res = float(torch.linalg.vector_norm(b - (A @ x)))
        out["cg_pde4096"] = {"iters": iters, "it_per_s": iters / (ms * 1e-3), "us_per_iter": ms / iters * 1e3,
                             "model_bytes_per_iter": fused_bytes, "final_true_residual": res,
                             "frac_of_hbm_peak": fused_bytes * iters / (ms * 1e-3) / 1e9 / peak}
        if not args.no_cpu:
            # scipy on the host: same system, absolute tolerance like the reference (rtol=0, atol=tol), bounded k
            import scipy.sparse as sp
            import scipy.sparse.linalg as spla

            k = 20
            S = sp.csr_array((A.data.cpu().numpy(), A.indices.cpu().numpy(), A.indptr.cpu().numpy()), shape=A.shape)
            bh = np.ones(N)
            t0 = time.perf_counter()
            xs, _info = spla.cg(S, bh, rtol=0.0, atol=1e-10, maxiter=k)
            dt_s = time.perf_counter() - t0
            xg, it_g = linalg.cg(A, b, tol=1e-10, maxiter=k)
            rs = float(np.linalg.norm(bh - S @ xs))
            rg = float(torch.linalg.vector_norm(b - (A @ xg)))
            out["cg_scipy"] = {"iters": k, "it_per_s": k / dt_s, "host_threads": 1, "host_cpu_count": os.cpu_count(),
                               "residual_after_k": rs, "gpu_residual_after_k": rg, "gpu_iters": it_g,
                               "residual_rel_diff": abs(rs - rg) / max(rs, 1e-300),
                               "x_rel_diff": float(np.linalg.norm(xs - xg.cpu().numpy()) / max(np.linalg.norm(xs), 1e-300)),
                               "speedup_it_per_s": (iters / (ms * 1e-3)) / (k / dt_s)}
            del S
        del A, b, x
        torch.cuda.empty_cache()
    except KeyError:
        pass
    except Exception as exc:  # pragma: no cover
        out["cg_error"] = repr(exc)
    try:
        if not want("spgemm_banded"):
            raise KeyError("skipped")
        B = gallery.banded(1_000_000, 11, np.float64)
        C = B @ B
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            C = B @ B
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        info = C.spgemm_info
        out["spgemm_banded1m"] = {"ms": min(ts) * 1e3, "products": info["products"], "nnz_c": info["nnz"],
                                  "gflops": 2 * info["products"] / min(ts) / 1e9}
        del B, C
    except KeyError:
        pass
    except Exception as exc:  # pragma: no cover
        out["spgemm_error"] = repr(exc)
    try:
        if not want("gmg"):
            raise KeyError("skipped")
        # GMG-preconditioned CG (SURVEY 8f row 1): the reference's own benchmark shape (results/summit/legate_gpu_gmg.out:
        # examples/gmg.py -n 4500 -m 200, defaults 2 levels / injection / weighted Jacobi; 37.5 it/s on one V100)
        import re
        import subprocess

        r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "gmg.py"), "-n", "4500", "-l", "2", "-g",
                            "injection", "-m", "200"], capture_output=True, text=True, timeout=300, cwd=os.path.join(ROOT, "examples"))
        m = re.search(r"Iterations / sec: ([0-9.]+)", r.stdout)
        it = re.search(r"after (\d+) iterations, \|b - Ax\| = ([0-9.eE+-]+)", r.stdout)
        if m:
            out["gmg_n4500"] = {"it_per_s": float(m.group(1)), "iters": int(it.group(1)) if it else None,
                                "final_residual": float(it.group(2)) if it else None, "levels": 2, "gridop": "injection",
                                "reference_v100_it_per_s": 37.5}
        else:
            out["gmg_error"] = (r.stdout + r.stderr)[-400:]
    except KeyError:
        pass
    except Exception as exc:  # pragma: no cover
        out["gmg_error"] = repr(exc)
    try:
        if not want("spgemm_rmat"):
            raise KeyError("skipped")
        out["spgemm_rmat"] = _spgemm_rmat_case(torch, gallery, peak, args)
    except KeyError:
        pass
    except Exception as exc:  # pragma: no cover
        out["spgemm_rmat_error"] = repr(exc)
    try:
        if not want("spmm"):
            raise KeyError("skipped")
        # SpMM (SURVEY 8f row 4): examples/dot_microbenchmark.py -op spmm -k 32 shape at n = 4M, fp64
        n, k = 4_000_000, 32
        B = gallery.banded(n, 11, np.float64)
        X = torch.rand((n, k), dtype=torch.float64, device="cuda")
        Y = torch.empty((n, k), dtype=torch.float64, device="cuda")
        t_ms, _ = _time_launches(torch, lambda: B.dot(X, out=Y), 20)
        t = t_ms * 1e-3
        byts = B.nnz * 12 + 4 * (n + 1) + 2 * n * k * 8
        out["spmm_banded4m_k32"] = {"us": t * 1e6, "gflops": 2 * B.nnz * k / t / 1e9, "algorithmic_bytes": byts,
                                    "frac_of_hbm_peak": byts / t / 1e9 / peak}
        del B, X, Y
    except KeyError:
        pass
    except Exception as exc:  # pragma: no cover
        out["spmm_error"] = repr(exc)
    return out


def sharded_rows_of_the_path(torch, dist, bd, gallery, peak, rank, world, args):
    """N>1 extras (every rank takes part; rank 0 reports).
    r32_strong: BASELINE config 4 / the north-star scaling test -- ONE 10M x 10M, 32-per-row random matrix row-sharded
        over the N GPUs; x all-gathered by b2s_peer_push (NVLink remote stores) while the own-column block is
        multiplied, one accumulating launch per source rank waiting in-kernel for its slice.
    r32_weak: the same with 10M rows PER GPU (10M*N columns): config 4 as literally written ("weak-scale 1/2/4/8").
    cg_pde4096_strong: BASELINE config 3 -- pde.py 4096^2 CG (300 iterations) row-sharded over the N GPUs, halo fused
        into the SpMV launch, scalars all-reduced by the NVLink peer kernel, iteration replayed from a CUDA graph."""
    out = {}
    barrier = lambda: (dist.barrier(), torch.cuda.synchronize())

    def r32_case(weak):
        n = 10_000_000 * (world if weak else 1)
        rp = bd.RowBlockPlan(n, world)
        lo, hi = rp.rows(rank)
        local = gallery.random_fixed(hi - lo, n, 32, np.float32, seed=1234 + rank)
        R = bd.dist_csr_array(local, (n, n), rank=rank, nranks=world)
        xf = R.new_full_vector(np.float32)
        R.local_view(xf).copy_(torch.rand(hi - lo, dtype=torch.float32, device="cuda"))
        yl = torch.empty(hi - lo, dtype=torch.float32, device="cuda")
        for _ in range(3):
            R.dot_graphed(xf, yl)
        barrier()
        # verify against the NCCL all-gather + un-blocked kernel on the same shard
        yref = torch.empty_like(yl)
        R.exchange(xf)
        _ops_spmv(local, xf, yref)
        R.dot_graphed(xf, yl)
        torch.cuda.synchronize()
        R.check_peer()
        err = float((yl - yref).abs().max()) / max(float(yref.abs().max()), 1e-30)
        ok = torch.tensor([1 if err <= 5e-6 else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        steps = 50
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            R.dot_graphed(xf, yl)
        e.record()
        barrier()
        t = torch.tensor([s.elapsed_time(e) / steps], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        info = R._fused.get((id(R.local), xf.data_ptr()))
        nnz = 32 * n
        blocks = None
        if info and info["mode"] == "blocks":
            blocks = {"count": sum(1 for b in info["blocks"].values() if b is not None),
                      "kernel": next(b._get_plan().kernel_name for b in info["blocks"].values() if b is not None)}
        res = {"global_rows": n, "global_nnz": nnz, "n_gpus": world, "ms_per_step": ms,
               "gflops": 2.0 * nnz / (ms * 1e-3) / 1e9, "verified_vs_nccl_allgather": bool(int(ok[0])),
               "max_rel_err": err, "exchange_path": f"fused-{info['mode']}" if info else f"nccl-{R.exchange_mode}",
               "column_blocks": blocks,
               "collective": ("all-gather of x by remote stores (b2s_peer_push, many CTAs per destination), one accumulating "
                              "launch per source-rank column block, each waiting in-kernel for its own slice"
                              if info and info["mode"] == "blocks" else
                              "all-gather of x by remote stores (b2s_peer_push, many CTAs per destination) + arrival wait, "
                              "then the product of the unsplit shard" if info else "NCCL all-gather"),
               "nvlink_bytes_in_per_gpu_per_step": int((n - (hi - lo)) * 4),
               "nvlink_ms_at_770GBs": (n - (hi - lo)) * 4 / 770e9 * 1e3,
               "frac_of_hbm_peak_aggregate": alg_bytes(n, n, nnz, sv=4) / (ms * 1e-3) / 1e9 / (peak * world)}
        barrier()
        R.close()
        del R, local, xf, yl, yref
        torch.cuda.empty_cache()
        return res

    for key, weak in (("r32_strong", False), ("r32_weak", True)):
        try:
            out[key] = r32_case(weak)
        except Exception as exc:  # pragma: no cover
            out[key + "_error"] = repr(exc)
    try:
        g1 = 4094
        N = g1 * g1
        rp = bd.RowBlockPlan(N, world)
        lo, hi = rp.rows(rank)
        local = gallery.laplacian_5pt(g1, g1, np.float64, row_lo=lo, row_hi=hi)
        Ad = bd.dist_csr_array(local, (N, N), rank=rank, nranks=world)
        b = torch.ones(hi - lo, dtype=torch.float64, device="cuda")
        bd.cg(Ad, b, tol=1e-10, maxiter=30)
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        xl, iters = bd.cg(Ad, b, tol=1e-10, maxiter=300)
        e.record()
        barrier()
        t = torch.tensor([s.elapsed_time(e)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
        # true residual of the returned iterate, all-reduced
        xfull = Ad.new_full_vector(np.float64)
        Ad.local_view(xfull).copy_(xl)
        r = b - Ad.dot(xfull)
        rr = torch.dot(r, r).reshape(1)
        dist.all_reduce(rr)
        out["cg_pde4096_strong"] = {"n_gpus": world, "iters": iters, "it_per_s": iters / (ms * 1e-3),
                                    "us_per_iter": ms / iters * 1e3, "final_true_residual": float(rr[0]) ** 0.5,
                                    "exchange_fused": bool(Ad._fused)}
        barrier()
        Ad.close()
    except Exception as exc:  # pragma: no cover
        out["cg_strong_error"] = repr(exc)
    return out


def _ops_spmv(A, x_full, out):
    from legate.sparse_b200 import _ops

    _ops.spmv(A.indptr, A.indices, A.data, x_full[: A.shape[1]], out, A.shape, plan=A._get_plan())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU-baseline sampling (rank 0, N=1)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the CG / SpGEMM side measurements at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write y of the last step (a fixed, seeded sample of its rows, float64) "
                         "to DIR/y.npy (DIR/y_rank<r>.npy per rank at N>1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU product; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
