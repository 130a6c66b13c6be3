#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 sparse hot path.

Metric (BASELINE.json): SpMV effective GFLOP/s (2*nnz/t) + achieved HBM GB/s, fp64 CrsMatrix.
Workload at N=1 (BASELINE.json configs[1]): 10M x 10M, ~60 nnz/row, 27-point Laplacian family ->
`lap27(171,171,171) x 2 dof/node`: 10,000,422 rows, 54 entries per interior row (SURVEY.md 8d (ii-a)).
N>1 (configs[4], weak scaling): each rank owns a 10M-row block of the N*10M-row matrix
(grid 171 x 171 x 171N), full x replicated; a step = local SpMV + NCCL all-gather of y into the
next x.  No collective on the data path other than that all-gather.

  python bench.py --gpus N --steps K --warmup W          (our CUDA path; torchrun for N>1)
  python bench.py --impl reference ...                   (the reference's CPU path -- the oracle's
                                                          OpenMP restatement -- on the host cores)
One JSON line on stdout (rank 0).  A "step" is one full SpMV over the whole matrix.
"""
import argparse
import json
import os

import subprocess
import sys


def _affinity_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# Read ONCE, before any OpenMP runtime starts: with OMP_PROC_BIND set, libgomp binds the initial thread to its first place
# (one core) in the first parallel region, after which the affinity mask of this thread shows 2 hardware threads.
_HOST_THREADS = _affinity_threads()


def host_threads():
    """Hardware threads this process may use (its affinity mask at start-up), NOT OMP_NUM_THREADS: torchrun exports
    OMP_NUM_THREADS=1 to every rank, which must not turn the CPU legs into single-core runs."""
    return _HOST_THREADS


_REF_ARM = "reference" in sys.argv and "--impl" in sys.argv
if int(os.environ.get("WORLD_SIZE", "1")) == 1 or (_REF_ARM and int(os.environ.get("RANK", "0")) == 0):
    # reference protocol for the CPU leg (BASELINE.md section 4): the one process that runs a CPU leg owns all host threads.
    # (Never for the GPU ranks under torchrun: every rank's threads would be pinned to the same first cores.)
    os.environ["OMP_NUM_THREADS"] = str(host_threads())
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GRID = 171          # 171^3 nodes x 2 dof = 10,000,422 rows
NDOF = 2
NOISE = 0.5
METRIC = "spmv_fp64_gflops"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons of one GPU DURING the timed region.  A thread reads them through NVML (nvidia-ml-py: the
    library nvidia-smi itself reads) every 2 ms from start() to stop(); mark_begin() / mark_end() bracket the timed region and the
    summary is over the samples taken inside it.  (A 20-step region lasts ~20 ms: nvidia-smi's loop mode, 100 ms at best and 100+ ms
    to start, cannot land a sample in it -- it stays as the fallback when NVML cannot be loaded, started before the warm-up so that it
    is polling by then, and its samples cover warm-up + timed region.)"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []      # nvidia-smi fallback: raw csv lines
        self.samples = []    # NVML: (perf_counter, sm MHz, reasons bitmask)
        self.nvml = None
        self.handle = None
        self.max_mhz = None
        self.t0 = self.t1 = None
        self._stop = False
        self.thread = None

    def _nvml_open(self):
        import pynvml
        pynvml.nvmlInit()
        h = None
        try:  # the device torch calls `idx`, whatever CUDA_VISIBLE_DEVICES did to the numbering
            import torch
            uuid = str(torch.cuda.get_device_properties(self.idx).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            h = None
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
        pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)  # fails here, not in the thread, if unsupported
        self.nvml, self.handle = pynvml, h
        try:
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.max_mhz = None

    def _nvml_loop(self):
        nv, h = self.nvml, self.handle
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop:
            try:
                self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(reasons_fn(h))))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            self._nvml_open()
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def _stop_nvml(self):
        self._stop = True
        self.thread.join(timeout=1.0)
        nv = self.nvml
        inside = [x for x in self.samples if self.t0 is not None and self.t1 is not None and self.t0 <= x[0] <= self.t1]
        window = "timed region"
        if not inside:
            inside, window = list(self.samples), "warm-up + timed region (no sample fell inside the timed region)"
        bits = 0
        for x in inside:
            bits |= x[2]
        names = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown", 0x8), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown", 0x20), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap", 0x4),
                 ("hw_power_brake_slowdown", "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80))
        reasons = sorted(n for n, attr, dflt in names if bits & int(getattr(nv, attr, dflt)))
        sm = [x[1] for x in inside]
        try:
            nv.nvmlShutdown()
        except Exception:
            pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(sm), "window": window, "source": "NVML, 2 ms period"}

    def stop(self):
        if self.nvml is not None and self.thread is not None:
            return self._stop_nvml()
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": "warm-up + timed region", "source": "nvidia-smi -lms 100"}


def ncu_traffic(files=("r02c15_spmv_tile_ncu_key_metrics.csv", "r01_spmv_tile_c2_ncu_key_metrics.csv"), kernel=None):
    """(DRAM bytes per launch, file) of a kernel from the newest committed `ncu --set full` capture of it on the bench workload
    (profiles/*key_metrics*: lines `metric,unit,value`; files holding several kernels separate them by a `Kernel Name` line) --
    a CONSTANT of the repository, not a measurement of this run; (None, None) if absent."""
    for name in files:
        path = os.path.join(ROOT, "profiles", name)
        try:
            vals, active = {}, kernel is None
            for ln in open(path):
                f = ln.strip().split(",")
                if len(f) >= 3 and f[0] == "Kernel Name":
                    active = kernel is None or kernel in ln
                    continue
                if not active or len(f) != 3:
                    continue
                scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(f[1])
                if scale and f[0] not in vals:
                    vals[f[0]] = float(f[2]) * scale
            return int(vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"]), name
        except Exception:
            continue
    return None, None


def alg_bytes(nnz, nrows, ncols, beta_nonzero=False):
    """Compulsory traffic (BASELINE.md section 3): nnz*(8+4) + (rows+1)*4 + cols*8 + rows*8*(1+[beta!=0])."""
    return nnz * 12 + (nrows + 1) * 4 + ncols * 8 + nrows * 8 * (2 if beta_nonzero else 1)


def build_shard(world, rank, grid=GRID):
    """Rows [rank*n/world, (rank+1)*n/world) of lap27(grid, grid, grid*world) x NDOF, rebased row_ptr."""
    from kokkos_kernels_b200 import matgen

    nz = grid * world
    n_total = grid * grid * nz * NDOF
    r0 = (n_total * rank) // world
    r1 = (n_total * (rank + 1)) // world
    t = time.time()
    rp, ci, va = matgen.lap27(grid, grid, nz, ndof=NDOF, row_begin=r0, row_end=r1, noise=NOISE, seed=7)
    log(f"[rank {rank}] generated rows [{r0},{r1}) nnz={len(ci)} in {time.time() - t:.1f}s")
    return rp, ci, va, n_total, r0, r1


def _cpu_spmv(orc):
    """The CPU implementation both timing legs run, all host threads: the reference's OWN host SpMV when oracle/_ref holds it
    (SPMV_Functor of sparse/impl/KokkosSparse_spmv_impl.hpp compiled from the reference tree in place, driven by an OpenMP
    RangePolicy stand-in: kind "reference"), else the oracle's restatement of that loop (kind "port").  Both produce the same
    bits (tests/test_oracle_spmv.py)."""
    if orc.has_ref_spmv_omp():
        return (lambda rp, ci, va, ncols, x, y, threads: orc.ref_spmv_functor_omp(rp, ci, va, x, y, 1.0, 0.0, threads)), "reference", \
            "the reference's own SPMV_Functor (spmv_impl.hpp:86-132 compiled in place, oracle/_ref) under an OpenMP RangePolicy"
    return (lambda rp, ci, va, ncols, x, y, threads: orc.spmv_functor(rp, ci, va, ncols, x, y, 1.0, 0.0, threads)), "port", \
        "oracle O2 (OpenMP functor order, spmv_impl.hpp:110-132)"


def _best_threads(run, rps, cis, vas, ncols, x, y, threads):
    """The thread count the CPU loop is fastest with on this box: all hardware threads, then half, a quarter, ... for as long
    as halving helps (SMT siblings, a second socket or a container CPU quota below the visible thread count make a streaming
    loop slower with more threads): the baseline is the reference at its best, not at a default."""
    best, best_t, tried = threads, None, []
    t = threads
    while t >= 1:
        try:
            run(rps, cis, vas, ncols, x, y, t)
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                run(rps, cis, vas, ncols, x, y, t)
                ts.append(time.perf_counter() - t0)
        except Exception:
            break
        tried.append((t, min(ts)))
        if best_t is None or min(ts) < best_t:
            best, best_t = t, min(ts)
        elif min(ts) > 1.25 * best_t and t < threads:
            break  # clearly past the optimum
        if t == 1:
            break
        t = max(1, t // 2)
    return best, ", ".join(f"{t} threads {ms * 1e3:.1f} ms" for t, ms in tried)


def cpu_leg(rp, ci, va, x, steps, warmup):
    """The reference's host SpMV (see _cpu_spmv) over the WHOLE shard (the same matrix and x the GPU arm multiplies), all host
    threads the box gives this process (affinity mask, not OMP_NUM_THREADS), pages first touched by the threads that stream them
    (the reference protocol: parallel initialisation, 5 warm-up iterations, perf_test/sparse/KokkosSparse_kk_spmv.cpp:121-167).
    Returns (mean ms, min ms, dict): `value` is from the MEAN over `steps` iterations -- the statistic the GPU arm reports."""
    import oracle_lib

    orc = oracle_lib.Oracle()
    run, kind, what = _cpu_spmv(orc)
    threads = host_threads()
    rows = len(rp) - 1
    nnz = int(rp[-1])
    ncols = len(x)
    rps, cis, vas, xs = (orc.first_touch_copy(a, threads) for a in (rp, ci, va, x))
    y = orc.first_touch_copy(np.zeros(rows), threads)
    run(rps, cis, vas, ncols, xs, y, threads)  # first touch of y, page faults
    threads, sweep = _best_threads(run, rps, cis, vas, ncols, xs, y, threads)
    for _ in range(max(warmup, 1)):
        run(rps, cis, vas, ncols, xs, y, threads)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        run(rps, cis, vas, ncols, xs, y, threads)
        ts.append(time.perf_counter() - t0)
    mean, mn = float(np.mean(ts)), float(min(ts))
    gf = 2.0 * nnz / mean / 1e9
    return mean * 1e3, mn * 1e3, {
        "value": round(gf, 3), "unit": "GFLOP/s", "cores": threads, "kind": kind,
        "value_from_min": round(2.0 * nnz / mn / 1e9, 3),
        "sample": f"{what}; the whole shard: {rows} rows, {nnz} nnz, x of {ncols}; {steps} iterations after {max(warmup, 1)} warm-up, "
                  f"mean {mean * 1e3:.2f} ms (reported), min {mn * 1e3:.2f} ms; {alg_bytes(nnz, rows, ncols) / mean / 1e9:.1f} GB/s algorithmic; "
                  f"thread count chosen by a sweep ({sweep}) out of {host_threads()} hardware threads"}


def run_reference(args, emit):
    """--impl reference: the reference's own CPU implementation of the path -- its host SPMV_Functor compiled from the reference
    tree in place (oracle/_ref; falls back to the oracle's restatement of the same loop when that library is absent) -- with all
    host threads, on the configuration the GPU arm runs: at N = 1 the whole configs[1] matrix (same rows, nnz and x); at N > 1
    rank 0's 10M-row block of the N x 10M-row matrix with the full x (a bounded sample of configs[4]: the rate of one block)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from kokkos_kernels_b200 import matgen

    world = max(1, args.gpus)
    rp, ci, va, n_total, r0, r1 = build_shard(world, 0, args.grid)
    x = matgen.fill(n_total, -1.0, 1.0, 1)
    nnz = int(rp[-1])
    ms, ms_min, cpu = cpu_leg(rp, ci, va, x, args.steps, args.warmup)
    gf = cpu["value"]
    out = {
        "impl": "reference", "metric": METRIC, "value": gf, "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4), "ms_per_step_min": round(ms_min, 4),
        "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"spmv fp64 CrsMatrix (int32 offsets/ordinals), lap27({args.grid}x{args.grid}x{args.grid * world}) x {NDOF} dof: "
                               + (f"{n_total} rows, {nnz} nnz ({nnz / n_total:.1f}/row), alpha=1 beta=0, single vector" if world == 1 else
                                  f"bounded sample = rank 0's block of {r1 - r0} rows ({nnz} nnz) of the {n_total}-row matrix, x of {n_total}, "
                                  f"alpha=1 beta=0, single vector"),
                   "baseline_config": "configs[1]" if world == 1 else "configs[4]",
                   "statistic": "mean over the timed steps (min in ms_per_step_min)"},
        "cpu_baseline": cpu,
        "e2e": {"value": gf, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


# ---------------------------------------------------------------------------------------------------------------------
# secondary workloads (N = 1): BASELINE.json configs[2] (SpMM) and configs[3] (SpGEMM), reported inside the one JSON line
# ---------------------------------------------------------------------------------------------------------------------
def secondary_spmm(dev, scale=23, k=16, iters=10):
    """configs[2]: spmv fp32 CrsMatrix, R-MAT scale 23 (Graph500 parameters, edge factor 16, duplicates merged), 16-column
    multivector (LayoutRight), alpha = 1, beta = 0."""
    import torch

    import oracle_lib
    from kokkos_kernels_b200 import matgen, sparse as sp

    t = time.time()
    rp, ci = matgen.rmat(scale, 16)
    n, nnz = len(rp) - 1, len(ci)
    va = matgen.fill(nnz, 0.0, 1.0, 23, dtype=np.float32)
    X = matgen.fill(n * k, -1.0, 1.0, 5, dtype=np.float32).reshape(n, k)
    log(f"[secondary spmm] R-MAT scale {scale}: n={n} nnz={nnz} max row {int(np.diff(rp).max())}, generated in {time.time() - t:.1f}s")
    A = sp.CrsMatrix(torch.from_numpy(rp).to(dev), torch.from_numpy(ci).to(dev), torch.from_numpy(va).to(dev), n)
    Xd = torch.from_numpy(X).to(dev)
    Yd = torch.full((n, k), float("nan"), dtype=torch.float32, device=dev)
    h = sp.SPMVHandle()
    for _ in range(3):
        sp.spmv(h, "N", 1.0, A, Xd, 0.0, Yd)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        sp.spmv(h, "N", 1.0, A, Xd, 0.0, Yd)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    # the same product on LayoutLeft operands (the Kokkos default for a multivector in CudaSpace): relayout + kernel + relayout
    Xl, Yl = Xd.t().contiguous().t(), torch.full((k, n), float("nan"), dtype=torch.float32, device=dev).t()
    hl = sp.SPMVHandle()
    for _ in range(2):
        sp.spmv(hl, "N", 1.0, A, Xl, 0.0, Yl)
    e0.record()
    for _ in range(iters):
        sp.spmv(hl, "N", 1.0, A, Xl, 0.0, Yl)
    e1.record()
    torch.cuda.synchronize()
    ms_left = e0.elapsed_time(e1) / iters
    left_equal = bool(torch.equal(Yl, Yd))
    kernel_left = hl.last_kernel()
    del Xl, Yl, hl
    # parity: sampled rows vs the oracle's multivector loop (O4, spmv_impl.hpp:745-926), component-wise scaled error
    orc = oracle_lib.Oracle()
    Y = Yd.cpu().numpy()
    rows = np.unique(np.concatenate([np.arange(0, 256), np.random.default_rng(0).integers(0, n, 20000), [int(np.argmax(np.diff(rp)))]]))
    worst = 0.0
    for lo in range(0, len(rows), 4096):
        rr = rows[lo:lo + 4096]
        lens = (rp[rr + 1] - rp[rr]).astype(np.int64)
        rps = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
        idx = np.concatenate([np.arange(rp[r], rp[r + 1]) for r in rr]) if lens.sum() else np.zeros(0, dtype=np.int64)
        cis, vas = np.ascontiguousarray(ci[idx]), np.ascontiguousarray(va[idx])
        Yr = np.zeros((len(rr), k), dtype=np.float32)
        orc.spmv_mv(rps, cis, vas, n, X, Yr, 1.0, 0.0, threads=1)
        Ys = np.zeros((len(rr), k), dtype=np.float32)
        orc.spmv_mv(rps, cis, np.abs(vas), n, np.abs(X), Ys, 1.0, 0.0, threads=1)
        worst = max(worst, float(np.max(np.abs(Y[rr] - Yr) / np.maximum(Ys, 1e-30))))
    assert worst <= 1e-4, f"spmm parity {worst}"
    balg = nnz * 8 + (n + 1) * 4 + n * k * 4 * 2
    bgather = nnz * 8 + (n + 1) * 4 + nnz * k * 4 + n * k * 4
    peak, peak_src = peaks()
    # CPU: the oracle's multivector loop on the first rows of the same matrix (bounded sample), all host threads
    threads = host_threads()
    srows = min(n, 1 << 20)
    rps = np.ascontiguousarray(rp[:srows + 1])
    snnz = int(rps[-1])
    Yc = np.zeros((srows, k), dtype=np.float32)
    orc.spmv_mv(rps, ci[:snnz], va[:snnz], n, X, Yc, 1.0, 0.0, threads=threads)
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        orc.spmv_mv(rps, ci[:snnz], va[:snnz], n, X, Yc, 1.0, 0.0, threads=threads)
        ts.append(time.perf_counter() - t0)
    cpu_gf = 2.0 * snnz * k / float(np.mean(ts)) / 1e9
    # end to end: X from pinned host memory, Y back to pinned host memory, every call
    Xh = torch.from_numpy(X).pin_memory()
    Yh = torch.empty((n, k), dtype=torch.float32).pin_memory()
    for _ in range(2):
        Xd.copy_(Xh, non_blocking=True)
        sp.spmv(h, "N", 1.0, A, Xd, 0.0, Yd)
        Yh.copy_(Yd, non_blocking=True)
    torch.cuda.synchronize()
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    q0.record()
    for _ in range(3):
        Xd.copy_(Xh, non_blocking=True)
        sp.spmv(h, "N", 1.0, A, Xd, 0.0, Yd)
        Yh.copy_(Yd, non_blocking=True)
    q1.record()
    torch.cuda.synchronize()
    ems = q0.elapsed_time(q1) / 3
    assert np.array_equal(Yh.numpy()[:1000], Y[:1000])
    return {
        "config": {"workload": f"spmv fp32 CrsMatrix, R-MAT scale {scale} (a,b,c,d = .57,.19,.19,.05, edge factor 16, duplicates merged): "
                               f"{n} rows, {nnz} nnz, max row {int(np.diff(rp).max())}; {k}-column multivector LayoutRight, alpha=1 beta=0",
                   "baseline_config": "configs[2]", "kernel": h.last_kernel(), "parity_max_scaled_err_sampled_rows": worst,
                   "parity_rows_checked": int(len(rows))},
        "metric": "spmm_fp32_gflops", "value": round(2.0 * nnz * k / ms / 1e6, 1), "unit": "GFLOP/s", "ms": round(ms, 4), "dtype": "f32",
        "layout_left": {"ms": round(ms_left, 4), "gflops": round(2.0 * nnz * k / ms_left / 1e6, 1), "kernel": kernel_left,
                        "bits_equal_layout_right": left_equal,
                        "note": "LayoutLeft X and Y (Kokkos' default in CudaSpace): both are relaid out inside the call"},
        "roofline": {"bound": "hbm", "achieved": round(balg / ms / 1e6, 1), "peak": peak, "unit": "GB/s", "frac": round(balg / ms / 1e6 / peak, 4),
                     "algorithmic_bytes_per_launch": balg, "gather_model_bytes": bgather,
                     "frac_gather_model": round(bgather / ms / 1e6 / peak, 4),
                     "traffic": ncu_traffic(("r02c15_spmm_coop_key_metrics.txt", "r02c8_spmm_coop_key_metrics.txt"), "spmm_item_coop_kernel")[0],
                     "traffic_unit": "DRAM bytes of the item kernel per launch, a constant from the committed ncu --set full capture at this size (profiles/r02c*_spmm_coop_key_metrics.txt)",
                     "peak_source": peak_src},
        "cpu_baseline": {"value": round(cpu_gf, 2), "unit": "GFLOP/s", "cores": threads, "kind": "port",
                         "sample": f"oracle O4 (CPU multivector strips, spmv_impl.hpp:745-926, OpenMP over rows), first {srows} rows "
                                   f"({snnz} nnz) of the same matrix, full X, 5 iterations, mean {np.mean(ts) * 1e3:.1f} ms"},
        "e2e": {"value": round(2.0 * nnz * k / ems / 1e6, 1), "unit": "GFLOP/s", "ms": round(ems, 3), "h2d_bytes_per_step": int(n * k * 4),
                "d2h_bytes_per_step": int(n * k * 4), "note": "X pinned host -> device, b200sp_spmm_f32_i32, Y -> pinned host; matrix device-resident"},
    }


def next_rows_bench(dev):
    """Two of the rows either side of the path (SURVEY.md 8f), timed beside the headline at N = 1 so that the driver's record holds
    them: KokkosSparse::spadd on sorted inputs (27.4 M + 27.4 M entries) and the level-set sparse triangular solve (lower triangle of
    lap27(96^3)) with the classic two-stage Gauss-Seidel sweep built on it.  Stand-alone versions with the kernel variants side by
    side: tools/bench_spadd.py, tools/bench_sptrsv.py.  Parity of both is tests/test_gpu_crs_utils.py / test_gpu_sptrsv.py's job;
    here the results are only checked for the obvious (sizes, finiteness)."""
    import scipy.sparse as sps
    import torch

    from kokkos_kernels_b200 import matgen, sparse as sp

    def ev_timed(fn, iters):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    peak, _ = peaks()
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    out = {}
    # ---- spadd, sorted inputs: C = 0.3 A - 1.7 B, B = A's structure with every column moved by one
    g = 64
    rp, ci, va = matgen.lap27(g, g, g, ndof=2, noise=0.5)
    m, n = len(rp) - 1, len(rp)
    A = sp.CrsMatrix(t(rp), t(ci), t(va), n)
    B = sp.CrsMatrix(t(rp), t((ci + 1).astype(np.int32)), t(va[::-1].copy()), n)
    kh = sp.KokkosKernelsHandle()
    kh.create_spadd_handle(True, True)
    crp = torch.zeros(m + 1, dtype=torch.int32, device=dev)
    sym_ms = ev_timed(lambda: sp.spadd_symbolic_views(kh, m, n, A.row_map, A.entries, B.row_map, B.entries, crp), 5)
    nnzc = int(kh.get_spadd_handle().get_c_nnz())
    cci = torch.empty(nnzc, dtype=torch.int32, device=dev)
    cv = torch.empty(nnzc, dtype=torch.float64, device=dev)
    num_ms = ev_timed(lambda: sp.spadd_numeric_views(kh, m, n, A.row_map, A.entries, A.values, 0.3, B.row_map, B.entries, B.values, -1.7,
                                                     crp, cci, cv), 10)
    balg = 12 * (2 * len(ci) + nnzc) + 3 * 4 * (m + 1)
    out["spadd"] = {"workload": f"spadd fp64, sorted rows: A = lap27({g}^3) x 2 dof ({m} rows, {len(ci)} entries), B = A with every column moved by one; nnz(C) = {nnzc}",
                    "symbolic_ms": round(sym_ms, 4), "numeric_ms": round(num_ms, 4), "numeric_alg_GBs": round(balg / num_ms / 1e6, 1),
                    "roofline_frac": round(balg / num_ms / 1e6 / peak, 4), "finite": bool(torch.isfinite(cv).all().item())}
    kh.destroy_spadd_handle()
    del A, B, crp, cci, cv
    # ---- sptrsv: lower triangle of the 27-point operator, and the classic Gauss-Seidel forward sweep on the full operator
    g = 96
    rp, ci, va = matgen.lap27(g, g, g, noise=0.5)
    n = len(rp) - 1
    L = sps.tril(sps.csr_matrix((va, ci, rp), shape=(n, n))).tocsr()
    L.sort_indices()
    lrp, lci, lv = L.indptr.astype(np.int32), L.indices.astype(np.int32), L.data.astype(np.float64)
    b = matgen.fill(n, -1.0, 1.0, 7)
    rpd, cid, vd, bd = t(lrp), t(lci), t(lv), t(b)
    h = sp.SPTRSVHandle(n, True)
    sp.sptrsv_symbolic(h, rpd, cid)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sp.sptrsv_symbolic(h, rpd, cid)
    torch.cuda.synchronize()
    sym_ms = (time.perf_counter() - t0) * 1e3
    xd = torch.full((n,), float("nan"), dtype=torch.float64, device=dev)
    solve_ms = ev_timed(lambda: sp.sptrsv_solve(h, rpd, cid, vd, bd, xd), 10)
    levels = int(h.get_num_levels())
    # residual of the solve, row-scaled: max |L x - b| / (|L| |x| + |b|)
    xh = xd.cpu().numpy()
    res = np.max(np.abs(L @ xh - b) / (abs(L) @ np.abs(xh) + np.abs(b)))
    kg = sp.KokkosKernelsHandle()
    kg.create_gs_handle(sp.GS_TWOSTAGE)
    kg.set_gs_twostage(False, n)
    Ad = sp.CrsMatrix(t(rp), t(ci), t(va), n)
    sp.gauss_seidel_symbolic(kg, n, n, Ad.row_map, Ad.entries, True)
    sp.gauss_seidel_numeric(kg, n, n, Ad.row_map, Ad.entries, Ad.values, True)
    xg = torch.zeros((n, 1), dtype=torch.float64, device=dev)
    gs_ms = ev_timed(lambda: sp.forward_sweep_gauss_seidel_apply(kg, n, n, Ad.row_map, Ad.entries, Ad.values, xg, bd.reshape(n, 1), False, True,
                                                                1.0, 1), 5)
    out["sptrsv"] = {"workload": f"sptrsv fp64, lower triangle of lap27({g}^3): {n} rows, {len(lci)} entries, {levels} levels",
                     "symbolic_ms_wall": round(sym_ms, 3), "solve_ms": round(solve_ms, 4), "us_per_level": round(1e3 * solve_ms / max(1, levels), 3),
                     "launches_per_solve": int(h.get_num_launches()), "row_scaled_residual": float(res),
                     "classic_gauss_seidel_forward_sweep_ms": round(gs_ms, 4),
                     "note": "latency-bound (dependent levels): the time per level is the figure of merit, not GB/s"}
    kg.destroy_gs_handle()
    return out


def secondary_spgemm(dev, n=2_000_000, deg=32, reps=2):
    """configs[3]: spgemm_symbolic + spgemm_numeric fp64, C = A*A, A = 2M x 2M with exactly 32 distinct uniform-random columns
    per row (seed 4), values U(1,50)."""
    import torch

    import oracle_lib
    from kokkos_kernels_b200 import matgen, sparse as sp

    t = time.time()
    rp, ci = matgen.uniform(n, n, deg, 4)
    va = matgen.fill(len(ci), 1.0, 50.0, 4)
    nnz = len(ci)
    products = int(np.sum(np.diff(rp)[ci].astype(np.int64)))
    log(f"[secondary spgemm] A: n={n} nnz={nnz}, {products} products, generated in {time.time() - t:.1f}s")
    A = sp.CrsMatrix(torch.from_numpy(rp).to(dev), torch.from_numpy(ci).to(dev), torch.from_numpy(va).to(dev), n)
    # Protocol of the reference's own driver (perf_test/sparse/KokkosSparse_spgemm.cpp:395-417): row_mapC exists before the
    # symbolic timer starts, the symbolic time ends with a fence; entriesC / valuesC are allocated (uninitialised) inside the
    # numeric timer.  Both wall-clock times are reported; ms_numeric is the device time of the numeric call itself.
    sym, num, num_wall = [], [], []
    C = None
    for rep in range(reps + 1):  # the first repetition warms the allocator pools up
        C = None  # the previous product's arrays go back to torch's caching allocator and are handed out again below
        kh = sp.KokkosKernelsHandle()
        kh.create_spgemm_handle()
        row_mapC = torch.empty(n + 1, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sp.spgemm_symbolic_views(kh, n, n, n, A.row_map, A.entries, False, A.row_map, A.entries, False, row_mapC)
        torch.cuda.synchronize()  # (symbolic is synchronous by contract: it returns nnz(C))
        t_sym = time.perf_counter() - t0
        t1 = time.perf_counter()
        c_nnz = kh.get_spgemm_handle().get_c_nnz()
        entriesC = torch.empty(c_nnz, dtype=torch.int32, device=dev)
        valuesC = torch.empty(c_nnz, dtype=torch.float64, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sp.spgemm_numeric_views(kh, n, n, n, A.row_map, A.entries, A.values, False, A.row_map, A.entries, A.values, False,
                                row_mapC, entriesC, valuesC)
        e1.record()
        torch.cuda.synchronize()
        t_num_wall = time.perf_counter() - t1
        if rep > 0:
            sym.append(t_sym * 1e3)
            num.append(e0.elapsed_time(e1))
            num_wall.append(t_num_wall * 1e3)
        C = sp.CrsMatrix(row_mapC, entriesC, valuesC, n)
        del row_mapC, entriesC, valuesC
        kh.destroy_spgemm_handle()
    c_nnz = C.nnz()
    # parity: blocks of rows vs the oracle (reference SPGEMM_DEBUG + sort), structure AND values bit-exact
    orc = oracle_lib.Oracle()
    rpC = C.row_map.cpu().numpy()
    checked = 0
    for r0 in (0, n // 3, n - 20000):
        r1 = r0 + 20000
        rowlen, ent, val = orc.spgemm_block(r0, r1, rp, ci, va, rp, ci, va, n)
        assert np.array_equal(np.diff(rpC[r0:r1 + 1]), rowlen), "spgemm parity: row_map"
        s0, s1 = int(rpC[r0]), int(rpC[r1])
        assert np.array_equal(C.entries[s0:s1].cpu().numpy(), ent), "spgemm parity: entries"
        assert np.array_equal(C.values[s0:s1].cpu().numpy(), val), "spgemm parity: values"
        checked += r1 - r0
    ms_sym, ms_num = float(np.mean(sym)), float(np.mean(num))
    b_sym = 4 * (2 * nnz) + 4 * (2 * (n + 1)) + 4 * (n + 1)
    b_num = 12 * nnz + 12 * nnz + 4 * (n + 1) + 12 * c_nnz
    b_gather = b_num + 12 * products - 12 * nnz
    peak, peak_src = peaks()
    # CPU: the oracle (reference host path), rows dealt to all host threads, on a block of rows (bounded sample)
    threads = host_threads()
    srows = 100_000
    t0 = time.perf_counter()
    orc.spgemm_block(0, srows, rp, ci, va, rp, ci, va, n, threads=threads)
    t_cpu = time.perf_counter() - t0
    sprod = int(np.sum(np.diff(rp)[ci[:int(rp[srows])]].astype(np.int64)))
    cpu_gf = 2.0 * sprod / t_cpu / 1e9
    # end to end: host CSR in (pinned), C (row_map, entries, values) back to pinned host memory
    e2e = None
    try:
        import psutil

        need = c_nnz * 12 + (n + 1) * 4
        if psutil.virtual_memory().available > 3 * need:
            hA = [torch.from_numpy(a).pin_memory() for a in (rp, ci, va)]
            hC = [torch.empty(n + 1, dtype=torch.int32).pin_memory(), torch.empty(c_nnz, dtype=torch.int32).pin_memory(),
                  torch.empty(c_nnz, dtype=torch.float64).pin_memory()]
            del C
            torch.cuda.empty_cache()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dA = [a.to(dev, non_blocking=True) for a in hA]
            A2 = sp.CrsMatrix(dA[0], dA[1], dA[2], n)
            kh = sp.KokkosKernelsHandle()
            kh.create_spgemm_handle()
            C = sp.spgemm_symbolic(kh, A2, False, A2, False)
            sp.spgemm_numeric(kh, A2, False, A2, False, C)
            hC[0].copy_(C.row_map, non_blocking=True)
            hC[1].copy_(C.entries, non_blocking=True)
            hC[2].copy_(C.values, non_blocking=True)
            torch.cuda.synchronize()
            t_e2e = time.perf_counter() - t0
            assert np.array_equal(hC[0].numpy(), rpC)
            e2e = {"value": round(2.0 * products / t_e2e / 1e9, 2), "unit": "GFLOP/s", "ms": round(t_e2e * 1e3, 2),
                   "h2d_bytes_per_step": int(nnz * 12 + (n + 1) * 4), "d2h_bytes_per_step": int(need),
                   "note": "A (CSR, pinned host) -> device, spgemm_symbolic + spgemm_numeric, C (row_map, entries, values: "
                           f"{need / 1e9:.1f} GB) -> pinned host; one repetition, wall clock"}
            kh.destroy_spgemm_handle()
            del hC
    except Exception as exc:  # the device-timed numbers stand
        e2e = {"value": None, "unit": "GFLOP/s", "note": f"end-to-end leg failed: {type(exc).__name__}: {exc}"}
    return {
        "config": {"workload": f"spgemm_symbolic + spgemm_numeric fp64 C = A*A, A = {n} x {n}, exactly {deg} distinct uniform-random columns "
                               f"per row: nnz(A) = {nnz}, {products} products, nnz(C) = {c_nnz}",
                   "baseline_config": "configs[3]", "parity": f"row_map / entries / values bit-exact on {checked} rows vs the oracle"},
        "metric": "spgemm_fp64_gflops", "value": round(2.0 * products / (ms_num + ms_sym) / 1e6, 2), "unit": "GFLOP/s (symbolic + numeric)",
        "ms_symbolic": round(ms_sym, 3), "ms_numeric": round(ms_num, 3), "ms_numeric_wall_with_allocation": round(float(np.mean(num_wall)), 3),
        "timing": "reference driver protocol (perf_test/sparse/KokkosSparse_spgemm.cpp:395-417): symbolic = wall clock of the view-level call "
                  "incl. its fence, row_mapC allocated before; numeric = CUDA events around the call; the wall-clock numeric time includes the "
                  "allocation of entriesC / valuesC (torch caching allocator, warmed by one repetition)",
        "numeric_gflops": round(2.0 * products / ms_num / 1e6, 2), "dtype": "f64",
        "roofline": {"bound": "hbm", "kernel": "esc_num_kernel<double,256,4,10> (persistent, row pipeline)", "achieved": round(b_num / ms_num / 1e6, 1), "peak": peak,
                     "unit": "GB/s", "frac": round(b_num / ms_num / 1e6 / peak, 4), "algorithmic_bytes_per_launch": b_num,
                     "gather_model_bytes": b_gather, "frac_gather_model": round(b_gather / ms_num / 1e6 / peak, 4),
                     "symbolic_GBs": round(b_sym / ms_sym / 1e6, 1),
                     "traffic": ncu_traffic(("r02c9_esc_key_metrics.txt",), "esc_num_kernel")[0],
                     "traffic_unit": "DRAM bytes of the numeric kernel per launch, a constant from the committed ncu --set full capture at this size (profiles/r02c9_esc_key_metrics.txt)",
                     "peak_source": peak_src},
        "cpu_baseline": {"value": round(cpu_gf, 3), "unit": "GFLOP/s", "cores": threads, "kind": "port",
                         "sample": f"oracle O6 (spgemm_debug symbolic + numeric + row sort, impl_seq.hpp:23-182), rows dealt to {threads} "
                                   f"threads, first {srows} rows ({sprod} products): {t_cpu * 1e3:.0f} ms"},
        "e2e": e2e,
    }


def gpu_local_cpus(dev_index):
    """CPUs of the NUMA node the GPU hangs off (sysfs), intersected with this process's affinity; None if unknown."""
    try:
        import torch

        p = torch.cuda.get_device_properties(dev_index)
        bus = None
        if hasattr(p, "pci_bus_id"):
            bus = f"{getattr(p, 'pci_domain_id', 0):04x}:{p.pci_bus_id:02x}:{getattr(p, 'pci_device_id', 0):02x}.0"
        else:
            import pynvml

            pynvml.nvmlInit()
            hnd = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(p.uuid)).encode()) if hasattr(p, "uuid") else pynvml.nvmlDeviceGetHandleByIndex(dev_index)
            bid = pynvml.nvmlDeviceGetPciInfo(hnd).busId
            bus = (bid.decode() if isinstance(bid, bytes) else bid).lower()[-12:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        return cpus or None
    except Exception:
        return None


class near_gpu:
    """with near_gpu(i): allocations made inside (pinned host buffers are placed by first touch) land on the NUMA node of GPU i."""

    def __init__(self, dev_index):
        # opt-in (B200SP_BENCH_NUMA=1): on the B200 boxes measured, the GPU's own node did not help -- at N = 1 the stream-ordered
        # host-vector step went from 2.00 to 2.73 ms (a node of a sub-NUMA-clustered socket has a fraction of the memory channels),
        # and at N = 8 the bound is the PCIe uplink two GPUs share (~26 GB/s each way per GPU), not the placement
        self.cpus = gpu_local_cpus(dev_index) if os.environ.get("B200SP_BENCH_NUMA") == "1" else None
        self.saved = None

    def __enter__(self):
        if self.cpus:
            try:
                self.saved = os.sched_getaffinity(0)
                os.sched_setaffinity(0, self.cpus)
            except OSError:
                self.saved = None
        return self

    def __exit__(self, *exc):
        if self.saved:
            try:
                os.sched_setaffinity(0, self.saved)
            except OSError:
                pass
        return False


DUMP_ROWS = 3_000_000  # float64 values + their row indices: 48 MB per dump, small enough to keep two runs side by side


def dump_outputs(out_dir, name, v):
    """Writes the device vector v, the result a caller of the timed path receives, to out_dir/<name>.npy as float64.  A longer
    vector than DUMP_ROWS is sampled, the same rows on every run (seed 0); their indices go to out_dir/<name>_rows.npy."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    if v.numel() > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(v.numel(), DUMP_ROWS, replace=False))
        v = v[torch.from_numpy(rows).to(v.device)]
        np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy().astype(np.float64))


def verify_transport(op, x, n_total, world, rank, dev):
    """One step and two chained steps of a row-block operator: every rank's copy of the gathered vector must be bit-identical to
    every other rank's (probes of each block are exchanged over NCCL), and the first result must not change under the steps
    that follow.  All ranks return the same verdict."""
    import torch
    import torch.distributed as dist

    ok = True
    try:
        blk = n_total // world
        a = op.step(x)
        torch.cuda.synchronize()
        dist.barrier()
        keep = a.clone()
        probe = torch.stack([a[q * blk + 5: q * blk + 5 + 4096] for q in range(world)])
        gathered = [torch.empty_like(probe) for _ in range(world)]
        dist.all_gather(gathered, probe)
        ok = ok and all(torch.equal(g, probe) for g in gathered) and bool(torch.isfinite(probe).all())
        x2 = op.step(op.step(a))  # the first of these reads the buffer the step above wrote, the second writes it again
        torch.cuda.synchronize()
        dist.barrier()
        probe = torch.stack([x2[q * blk + 17: q * blk + 17 + 4096] for q in range(world)])
        gathered = [torch.empty_like(probe) for _ in range(world)]
        dist.all_gather(gathered, probe)
        ok = ok and all(torch.equal(g, probe) for g in gathered)
        b = op.step(x)  # same input, same buffer parity as the first step after an even number of steps in between? not
        # necessarily: compare values, not buffers
        torch.cuda.synchronize()
        dist.barrier()
        ok = ok and bool(torch.equal(b, keep))
        if (op.parity & 1) == 1:  # leave the operator at an even number of steps (buffer parity as constructed)
            op.step(x)
            torch.cuda.synchronize()
    except Exception as e:  # a transport that throws is rejected like one that miscompares
        log(f"[rank {rank}] transport check raised {type(e).__name__}: {e}")
        ok = False
    flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return flag.item() >= 1.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--grid", type=int, default=GRID, help="nodes per axis (default 171 -> 10M rows); smaller for dry runs")
    ap.add_argument("--cfg", type=int, default=-1)
    ap.add_argument("--lpr", type=int, default=-1)
    ap.add_argument("--ctas", type=int, default=-1)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step to DIR/<name>.npy (y; x_next for N>1), float64, at most "
                         f"{DUMP_ROWS} seeded sample rows with their indices in DIR/<name>_rows.npy")
    ap.add_argument("--no-secondary", action="store_true", help="N=1: skip the configs[2] / configs[3] workloads")
    ap.add_argument("--collective", default="auto",
                    choices=["auto", "pipelined", "pipelined_mc", "pipelined_sm", "fused", "multicast", "multicast_fwd", "nccl"],
                    help="N>1: how y is all-gathered into the next x.  auto = time every transport on this box during warm-up and "
                         "keep the fastest: pushes of finished pieces behind the compute by copy engines (pipelined), by a small SM "
                         "kernel to the NVSwitch multicast address (pipelined_mc) or to the 7 peers (pipelined_sm), stores from the "
                         "SpMV kernel itself (fused / multicast), or NCCL after it")
    ap.add_argument("--chunks", type=int, default=8)
    ap.add_argument("--push-ctas", type=int, default=32)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    # libraries (NCCL prints its version line) must not pollute stdout: the JSON line is the only thing on it
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    if args.impl == "reference":
        return run_reference(args, emit)

    import torch
    import torch.distributed as dist

    import kokkos_kernels_b200 as kk
    from kokkos_kernels_b200 import matgen, sparse as sp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    assert kk._lib.sparse().b200sp_device_ok() == 1, "not a compute-capability 10.x (B200) device"
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    rp, ci, va, n_total, r0, r1 = build_shard(world, rank, args.grid)
    nrows = r1 - r0
    nnz = len(ci)
    x_host = matgen.fill(n_total, -1.0, 1.0, 1)
    x = torch.from_numpy(x_host).to(dev)
    lib = kk._lib.sparse()

    def timed(fn, reps):
        """device time of `reps` calls of fn, ms per call, MAX over ranks (barrier + synchronize on both sides)"""
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        tt = torch.tensor([a.elapsed_time(b) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return tt.item()

    # multi-GPU: row blocks + all-gather of y behind the compute over NVLink (multigpu.py)
    op = None
    collective = "none"
    mode_ms = {}
    rejected = []
    if world > 1:
        from kokkos_kernels_b200 import multigpu

        cands = ["multicast_fwd", "pipelined_mc", "pipelined_sm", "pipelined", "multicast", "nccl"] if args.collective == "auto" else [args.collective]
        ops = {}
        first = None
        for mode in cands:
            ok = 1.0
            try:
                o = multigpu.RowBlockSpMV(rp, ci, va, n_total, r0, r1, dev, mode=mode, chunks=args.chunks,
                                          tune=(args.cfg, args.lpr, args.ctas), shared=first, push_ctas=args.push_ctas)
            except Exception as e:  # e.g. no multicast mapping: the same on every rank, but agree on it anyway
                log(f"[rank {rank}] collective {mode} unavailable: {type(e).__name__}: {e}")
                o, ok = None, 0.0
            flag = torch.tensor([ok], dtype=torch.float64, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() < 1.0:
                continue
            if first is None:
                first = o
            try:
                for _ in range(3):
                    o.step(x)
                mode_ms[mode] = timed(lambda: o.step(x), 6)
                ops[mode] = o
            except Exception as e:
                log(f"[rank {rank}] collective {mode} failed while timing: {type(e).__name__}: {e}")
                raise
        assert ops, "no all-gather transport is available"
        # fastest first; a transport is only used if every rank's gathered vector verifies (below) -- otherwise the next one
        for cand in sorted(mode_ms, key=mode_ms.get):
            if verify_transport(ops[cand], x, n_total, world, rank, dev):
                collective = cand
                break
            rejected.append(cand)
            log(f"[rank {rank}] collective {cand} REJECTED: the ranks' gathered vectors differ; trying the next transport")
        assert collective != "none", "no all-gather transport produced identical vectors on every rank"
        op = ops[collective]
        for mname in list(ops):
            if mname != collective and ops[mname] is not first:
                del ops[mname]
        if rank == 0:
            log("[collective] ms per step by transport: " + ", ".join(f"{k_} {v_:.3f}" for k_, v_ in mode_ms.items()) + f" -> {collective}"
                + (f" (rejected: {rejected})" if rejected else ""))
        A, h = op.A_full, op.h_full
    else:
        A = sp.CrsMatrix(torch.from_numpy(rp).to(dev), torch.from_numpy(ci).to(dev), torch.from_numpy(va).to(dev), n_total)
        h = sp.SPMVHandle(sp.SPMV_DEFAULT)
        h.tune(args.cfg, args.lpr, args.ctas)
        y = torch.empty(nrows, dtype=torch.float64, device=dev)

    def local_spmv():
        if op is not None:
            op.local_spmv_only(x)
        else:
            sp.spmv(h, "N", 1.0, A, x, 0.0, y)

    def step():
        if op is not None:
            op.step(x)
        else:
            sp.spmv(h, "N", 1.0, A, x, 0.0, y)

    # ---- parity on this rank's shard: sampled rows vs the oracle's Serial path (O1)
    step()
    torch.cuda.synchronize()
    if op is not None:
        x_next, y = op.x_next, op.y
    kernel_name = op.kernel_name() if op is not None else h.last_kernel()
    check = None
    if not args.no_check:
        import oracle_lib

        orc = oracle_lib.Oracle()
        rng = np.random.default_rng(rank)
        b0 = int(rng.integers(0, max(nrows - 200000, 1)))
        b1 = min(b0 + 200000, nrows)
        rps = (rp[b0:b1 + 1] - rp[b0]).astype(np.int32)
        cis, vas = ci[rp[b0]:rp[b1]], va[rp[b0]:rp[b1]]
        yref = np.zeros(b1 - b0)
        orc.spmv_serial(rps, cis, vas, x_host, yref, 1.0, 0.0)
        scale = np.zeros(b1 - b0)
        orc.spmv_serial(rps, cis, np.abs(vas), np.abs(x_host), scale, 1.0, 0.0)
        got = y[b0:b1].cpu().numpy()
        check = float(np.max(np.abs(got - yref) / np.maximum(scale, 1e-300)))
        assert check <= 1e-10, f"parity failure on rank {rank}: {check}"
        if world > 1:
            # every rank's rows must have landed in this rank's copy of the next x: compare a slice of
            # each block with what its owner computed
            torch.cuda.synchronize()
            dist.barrier()
            blk = n_total // world
            probe = torch.stack([x_next[q * blk: q * blk + 4096] for q in range(world)])
            gathered = [torch.empty_like(probe) for _ in range(world)]
            dist.all_gather(gathered, probe)
            for q in range(world):
                assert torch.equal(gathered[q], probe), f"rank {rank}: next-x differs from rank {q}'s copy"
            assert np.array_equal(x_next[r0 + b0: r0 + b1].cpu().numpy(), got), "y landed in the wrong slot"
            # two chained steps (x <- A x twice, the second one reads the buffer the first one wrote): every rank's copy equal
            x2 = op.step(op.step(x))
            torch.cuda.synchronize()
            dist.barrier()
            probe = torch.stack([x2[q * blk + 17: q * blk + 17 + 4096] for q in range(world)])
            gathered = [torch.empty_like(probe) for _ in range(world)]
            dist.all_gather(gathered, probe)
            for q in range(world):
                assert torch.equal(gathered[q], probe), f"rank {rank}: chained next-x differs from rank {q}'s copy"
            assert bool(torch.isfinite(probe).all())

    # ---- timed region (device time, CUDA events on the launching stream, max over ranks)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # before the warm-up: the sampler is running (and the clocks are under load) when the timed region begins
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = lib.b200sp_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    sampler.mark_begin()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    sampler.mark_end()
    if world > 1:
        dist.barrier()
    launches = lib.b200sp_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        if op is None:
            dump_outputs(args.dump_outputs, "y", y)
        else:  # every rank holds the whole gathered vector
            dump_outputs(args.dump_outputs, "x_next", op.x_next)
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    nnz_t = torch.tensor([float(nnz)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(nnz_t, op=dist.ReduceOp.SUM)
    ms_step = t.item() / args.steps
    total_nnz = int(nnz_t.item())
    gflops = 2.0 * total_nnz / (ms_step * 1e-3) / 1e9

    # ---- kernel-only timing for the roofline (SpMV launches alone, same events, this rank)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    k0.record()
    for _ in range(args.steps):
        local_spmv()
    k1.record()
    torch.cuda.synchronize()
    kern_ms = k0.elapsed_time(k1) / args.steps
    balg = alg_bytes(nnz, nrows, n_total)
    peak, peak_src = peaks()
    achieved = balg / (kern_ms * 1e-3) / 1e9
    # the all-gather alone (no compute): its bytes and time "separately and fused" (SURVEY.md section 8d)
    allgather_ms = None
    if op is not None:
        op.allgather_slices()
        allgather_ms = timed(lambda: op.allgather_slices(), 10)

    # ---- end-to-end: host vectors in, host vectors out, every step
    esteps = max(5, min(args.steps, 20))
    e2e_extra = {}
    if world == 1:
        # through the host-vector C-ABI entry: pinned x -> device, SpMV, y -> pinned host
        with near_gpu(local) as ng:  # pinned host vectors on the GPU's own NUMA node
            xh = torch.empty(n_total, dtype=torch.float64).pin_memory()
            yh = torch.empty(nrows, dtype=torch.float64).pin_memory()
            xh.copy_(torch.from_numpy(x_host))
            numa_note = f"; pinned vectors allocated on the GPU's NUMA node ({len(ng.cpus)} local CPUs)" if ng.cpus else ""
        for _ in range(3):
            sp.spmv_hostvec(h, "N", 1.0, A, xh, 0.0, yh)
        torch.cuda.synchronize()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        for _ in range(esteps):
            sp.spmv_hostvec(h, "N", 1.0, A, xh, 0.0, yh)
        q1.record()
        torch.cuda.synchronize()
        e2e_sync_ms = q0.elapsed_time(q1) / esteps
        e2e_ms = e2e_sync_ms
        if not args.no_check and check is not None:
            assert np.array_equal(yh.numpy()[:1000], y[:1000].cpu().numpy())
        e2e_mode, e2e_defer_ms = "stream-ordered completion per call", None
        # the same loop with deferred completion (B200SP_SPMV_OPT_HOSTVEC_DEFER): a call no longer makes the stream wait for its own
        # download, so upload k+1, kernel k+1 and download k overlap; every step still uploads x and downloads y, all downloads are
        # complete (hostvec_flush + synchronize) inside the timed region.  Kept only if it returns the same bits and is faster.
        try:
            y_sync = yh.clone()
            yh.zero_()
            h.hostvec_defer(True)
            for _ in range(3):
                sp.spmv_hostvec(h, "N", 1.0, A, xh, 0.0, yh)
            h.hostvec_flush()
            torch.cuda.synchronize()
            same = bool(torch.equal(yh, y_sync))
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d0.record()
            for _ in range(esteps):
                sp.spmv_hostvec(h, "N", 1.0, A, xh, 0.0, yh)
            h.hostvec_flush()
            d1.record()
            torch.cuda.synchronize()
            same = same and bool(torch.equal(yh, y_sync))
            h.hostvec_defer(False)
            e2e_defer_ms = d0.elapsed_time(d1) / esteps
            if same and e2e_defer_ms < e2e_sync_ms:
                e2e_ms = e2e_defer_ms
                e2e_mode = "deferred completion (hostvec_flush before the closing synchronize)"
            elif not same:
                e2e_mode += "; deferred mode REJECTED: result differs"
        except Exception as exc:  # the stream-ordered number stands
            e2e_mode += f"; deferred mode failed: {type(exc).__name__}"
        h2d, d2h = int(n_total * 8), int(nrows * 8)
        e2e_extra = {"mode": e2e_mode, "ms_per_step_stream_ordered": round(e2e_sync_ms, 4),
                     "ms_per_step_deferred": None if e2e_defer_ms is None else round(e2e_defer_ms, 4),
                     "note": "b200sp_spmv_hostvec_f64_i32: pinned host x -> device, SpMV, y -> pinned host, every step; "
                             "matrix stays device-resident (as a CrsMatrix in CudaSpace does)" + numa_note}
    else:
        # every rank uploads ITS slice of x (n/P values), the all-gather over NVLink completes x on every GPU, local SpMV,
        # every rank downloads its slice of y (RowBlockSpMV.step_host; calls pipelined over the two next-x buffers)
        with near_gpu(local) as ng:  # the pinned slices on the GPU's own NUMA node: 8 ranks share the host's memory channels
            xh = torch.empty(nrows, dtype=torch.float64).pin_memory()
            yh = torch.empty(nrows, dtype=torch.float64).pin_memory()
            xh.copy_(torch.from_numpy(x_host[r0:r1].copy()))
            yh.fill_(float("nan"))
            numa_note = f"pinned buffers allocated on the GPU's NUMA node ({len(ng.cpus)} local CPUs)" if ng.cpus else "pinned buffers with the default placement"
        for _ in range(3):
            op.step_host(xh, yh)
        op.host_flush()
        torch.cuda.synchronize()
        if not args.no_check and check is not None:
            assert np.array_equal(yh.numpy()[b0:b1], got), "end-to-end result differs from the device-resident one"

        def e2e_loop():
            for _ in range(esteps):
                op.step_host(xh, yh)
            op.host_flush()

        e2e_ms = timed(e2e_loop, 1) / esteps
        h2d, d2h = int(n_total * 8), int(n_total * 8)  # all ranks together: every value of x goes up once, of y comes down once
        e2e_extra = {"mode": f"RowBlockSpMV.step_host, all-gather transport {collective}, calls pipelined over two buffers",
                     "note": f"every rank: its {nrows}-value slice of x pinned host -> device, all-gather over NVLink, local SpMV, its slice "
                             "of y -> pinned host, every step; bytes are the totals over all ranks; " + numa_note}
    e2e_gflops = 2.0 * total_nnz / (e2e_ms * 1e-3) / 1e9

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        _, _, cpu = cpu_leg(rp, ci, va, x_host, 10, 3)

    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary and args.grid == GRID:
        del A, x
        if "y" in dir():
            del y
        torch.cuda.empty_cache()
        secondary = []
        for fn in (secondary_spmm, secondary_spgemm):
            try:
                secondary.append(fn(dev))
            except AssertionError:
                raise
            except Exception as exc:
                secondary.append({"config": {"workload": fn.__name__}, "error": f"{type(exc).__name__}: {exc}"})
            torch.cuda.empty_cache()

    next_rows = None
    if secondary is not None:
        try:
            next_rows = next_rows_bench(dev)
            torch.cuda.empty_cache()
        except Exception as exc:  # never let the extra rows cost the headline line
            next_rows = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        out = {
            "metric": METRIC, "value": round(gflops, 2), "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_step, 5), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": f"spmv fp64 CrsMatrix (int32 offsets/ordinals), lap27({args.grid}x{args.grid}x{args.grid * world}) x {NDOF} dof: "
                            f"{n_total} rows, {total_nnz} nnz ({total_nnz / n_total:.1f}/row), alpha=1 beta=0, single vector"
                            + (f", row-partitioned over {world} GPUs, all-gather of y each step ({collective})" if world > 1 else ""),
                "baseline_config": "configs[1]" if world == 1 else "configs[4]",
                "cache": "inputs (matrix %.1f GB per GPU) exceed the 126 MB L2; no flush needed" % (nnz * 12 / 1e9),
                "kernel": kernel_name, "parity_max_scaled_err": check, "collective": collective,
                "statistic": "mean over the timed steps",
            },
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4),
                         "traffic": ncu_traffic()[0] if (world == 1 and args.grid == GRID) else None,
                         "traffic_unit": "DRAM bytes per launch, a CONSTANT read from the committed ncu --set full capture of this kernel on "
                                         f"this workload (profiles/{ncu_traffic()[1]}), not measured by this run",
                         "peak_source": peak_src,
                         "kernel_ms": round(kern_ms, 5), "algorithmic_bytes_per_launch": balg},
            "e2e": dict({"value": round(e2e_gflops, 2), "unit": "GFLOP/s", "h2d_bytes_per_step": h2d,
                         "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_ms, 4)}, **e2e_extra),
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if world > 1:
            recv = (world - 1) * nrows * 8
            out["collective"] = {
                "chosen": collective, "ms_per_step_by_transport": {k_: round(v_, 4) for k_, v_ in mode_ms.items()},
                "rejected_by_verification": rejected,
                "local_kernel_ms": round(kern_ms, 4), "collective_ms": round(max(ms_step - kern_ms, 0.0), 4),
                "collective_ms_note": "exposed communication = step - local SpMV alone (this rank's kernel time)",
                "allgather_alone_ms": None if allgather_ms is None else round(allgather_ms, 4),
                "allgather_bytes_received_per_rank": int(recv),
                "allgather_alone_GBs_per_rank": None if not allgather_ms else round(recv / allgather_ms / 1e6, 1),
            }
        if cpu:
            out["cpu_baseline"] = cpu
        if secondary is not None:
            out["secondary"] = secondary
        if next_rows is not None:
            out["next_rows"] = next_rows
        emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
