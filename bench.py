#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: fp64 CSR SpMV effective HBM GB/s (and fraction of the HBM roofline) at 1/2/4/8
B200, plus CG iterations/s (BASELINE.json configs[3]) as an extra key of the same JSON line.

  python bench.py [--gpus N --steps K --warmup W]          our arm: sm_100a kernels through the cuSPARSE C ABI
  python bench.py --impl reference [...]                    reference arm: the samples' host loop on the CPU cores
  torchrun --nproc-per-node N bench.py --gpus N ...         N>1: row-block shards, x exchanged over NVLink every step
  python bench.py ... --dump-outputs DIR                    also write y of the last timed step to DIR/y.npy (fp64)

A "step" is one y = A*x (alpha=1, beta=0) over the whole matrix.  Workload at N=1 = BASELINE.json configs[1]:
R-MAT 1,000,000 x 1,000,000, 16 non-zeros/row on average, fp64 values, int32 indices (SURVEY.md 8d).  At N>1 the
matrix grows with N (N*1M rows, "weak" scaling): every rank keeps ~16M non-zeros and receives the other ranks' x.
Timing: CUDA events on the launching stream around exactly K steps, barrier + synchronize on both sides, max over
ranks.  No L2 flush: one step streams 212 MB (> 126 MB L2) so val[]/col_ind[] cannot stay resident; x (8 MB) does.

Extra keys of the line (VERDICT r1 "make the measurement contract complete"):
  north_star_10m    the north-star acceptance config (R-MAT 10M x 16, fp64): us, GB/s, fraction of peak, error vs cuSPARSE
  cg_config4        BASELINE.json configs[3]: CG, 5-pt Poisson 8192^2, 200 iterations, row-sharded over the N GPUs: iterations/s
  cusparse_toolkit  the closed library of the CUDA 12.9 toolkit (the one the reference samples link), timed by a C harness
  other_configs     BASELINE.json configs[2] (fp32 SELL 7-pt 256^3) and configs[4] (fp32 CSR x dense, n = 64), N = 1 only
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_REAL_STDOUT = sys.stdout
METRIC = "csr_spmv_fp64_effective_hbm_bandwidth"
UNIT = "GB/s"
ROWS_PER_GPU = 1_000_000
AVG_NNZ = 16
CG_GRID = 8192
ROW_WEIGHT = 2.0       # N>1: work of a row block = nnz + ROW_WEIGHT * rows.  Fitted on the N = 2 runs of round 2 (csr_flat_kernel; weight 8:
                       #      19.7 M nnz / 0.54 M rows in 100.4 us, 12.3 M nnz / 1.46 M rows in 74.5 us -> ~5.1 us per M nnz + ~8 us per M rows;
                       #      round 1's tile kernels paid far more per row: 12)
CG_ITERS = 200
DUMP_LIMIT_BYTES = 64 << 20


def dump_output(out_dir, y):
    """--dump-outputs: y of the last timed step as out_dir/y.npy, fp64, the whole vector.  The inputs come from fixed seeds, so
    two builds run with the same arguments can be compared element by element."""
    import numpy as np
    y = np.ascontiguousarray(y, dtype=np.float64)
    if y.nbytes > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: y is {y.nbytes} bytes, more than --dump-outputs writes ({DUMP_LIMIT_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "y.npy")
    np.save(path, y)
    print(f"[bench] wrote {path} ({y.size} x fp64)", file=sys.stderr, flush=True)


def gather_rows(torch, dist, y_shard, bounds):
    """The row blocks of y (rank r holds rows bounds[r]:bounds[r+1]) joined in row order, on the host of every rank."""
    b = bounds.tolist()
    n = max(hi - lo for lo, hi in zip(b[:-1], b[1:]))
    padded = torch.zeros(max(n, 1), dtype=y_shard.dtype, device=y_shard.device)
    padded[:y_shard.numel()] = y_shard
    parts = [torch.empty_like(padded) for _ in b[:-1]]
    dist.all_gather(parts, padded)
    return torch.cat([p[:hi - lo] for p, lo, hi in zip(parts, b[:-1], b[1:])]).cpu()


def csr_bytes(rows, cols, nnz, vb=8, ib=4):
    # SURVEY.md 8(d): nnz*(val+idx) + (rows+1)*idx + cols*val (x) + rows*val (y), beta = 0
    return nnz * (vb + ib) + (rows + 1) * ib + cols * vb + rows * vb


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_source_sha(kernel="b200::csr_flat_kernel<double>"):
    """Hash of what `kernel` is compiled from: the .cu file under csrc/ that defines it, the device-code header every kernel
    file includes (spmv_common.cuh) and the nvcc flags.  profiles/traffic.json is only quoted when it was captured from THIS
    code; host-side files (the shim, the run-time options) and the other kernels' files do not change the kernel's SASS and do
    not invalidate the capture (checked for the round-2 capture: the SASS of spmv_csr_flat.cu built from the capture's commit
    and from this tree is byte-identical, profiles/README.md)."""
    from cudalibrarysamples_b200 import build as B
    d = os.path.join(ROOT, "cudalibrarysamples_b200", "csrc")
    short = kernel.split("::")[-1].split("<")[0]
    owner = None
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh")) and ("__global__" in open(os.path.join(d, name)).read()) and (" " + short + "(") in open(os.path.join(d, name)).read():
            owner = name
            break
    h = hashlib.sha256()
    for name in ([owner] if owner else []) + ["spmv_common.cuh"]:
        h.update(name.encode())
        h.update(open(os.path.join(d, name), "rb").read())
    h.update(" ".join(B.NVCC_FLAGS).encode())
    return h.hexdigest()[:16]


# ------------------------------------------------------------------------------------------------------------------
# clocks: NVML polled from a thread for the whole run; samples inside the timed window are reported
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.ok, self._stop = [], False, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), sm, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self._stop.set()
        if self.ok and self.t.is_alive():
            self.t.join(1.0)

    def summary(self, t0, t1, probe=None):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        win, where = [s for s in self.samples if t0 <= s[0] <= t1], "timed region"
        if len(win) < 3 and probe is not None:
            win, where = [s for s in self.samples if probe[0] <= s[0] <= probe[1]], "same kernel looped for 1 s right after the timed region (region too short to sample)"
        if not win:
            win, where = self.samples[-5:], "last samples"
        clocks = sorted(s[1] for s in win)
        bits = 0
        for s in win:
            bits |= s[2]
        reasons = [n for b, n in self.REASONS.items() if bits & b and n != "gpu_idle"]
        return {"sm_mhz": clocks[len(clocks) // 2] if clocks else None, "sm_max_mhz": self.max, "reasons": reasons,
                "samples": len(win), "window": where}


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the samples' host verification loop (spmv_csr_op_example.c:307-318) on the host cores
# ------------------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads for the CPU arm, FIXED per box: the CPUs this process may run on, capped by the cgroup CPU quota
    (omp_get_max_threads() counts CPUs outside the quota on some boxes: 128 threads on a 64-CPU allocation ran 20x
    slower in round 1).  No per-run probing: the same count is used by the reference arm and by cpu_baseline."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = int(q) / int(p)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota:
        n = min(n, max(1, int(quota)))
    return max(1, min(n, 64))          # the loop is memory-bound: beyond 64 threads nothing is gained on these hosts


def cpu_times(off, col, val, x, threads, reps):
    """Per-repetition wall times of the oracle's CSR loop; statistic everywhere = MEDIAN."""
    from oracle import oracle as O
    _, times, y = O.time_csr_f64(off, col, val, x, threads, reps=reps)
    ts = sorted(times)
    return ts[len(ts) // 2], times, y


def run_reference_arm(args):
    """The reference's own CPU implementation of the path (the samples' host loop, restated in oracle/spmv_oracle.c),
    all host threads, same metric / unit / config as our arm: at --gpus N the N*1M-row matrix."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    from oracle import oracle as O
    rows = ROWS_PER_GPU * args.gpus
    t_gen = time.time()
    off, col, val = O.rmat_csr(rows, avg_nnz=AVG_NNZ, seed=42, val_seed=43)
    x = O.uniform(44, rows)
    t_gen = time.time() - t_gen
    threads = host_threads()
    nnz = int(col.size)
    steps = args.steps
    for _ in range(max(args.warmup, 3)):
        O.time_csr_f64(off, col, val, x, threads, reps=1)
    med, times, y = cpu_times(off, col, val, x, threads, steps)
    if args.dump_outputs:
        dump_output(args.dump_outputs, y)
    gbs = csr_bytes(rows, rows, nnz) / med / 1e9
    sample = (f"one full y=A*x per step on the {rows}-row R-MAT matrix (nnz={nnz}); OpenMP dynamic row chunks, {threads} threads "
              f"(fixed: allowed CPUs capped by the cgroup quota and 64); {steps} timed steps, MEDIAN reported "
              f"(min {min(times) * 1e3:.2f} ms, max {max(times) * 1e3:.2f} ms); matrix generated on the CPU in {t_gen:.0f} s (not timed)")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(gbs, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(med * 1e3, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus, rows, nnz),
        "cpu_baseline": {"value": round(gbs, 3), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "statistic": "median"},
        "e2e": {"value": round(gbs, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gflops": round(2 * nnz / med / 1e9, 3),
        "reference_arm": "CPU host loop (spmv_csr_op_example.c:307-318 restated, oracle/spmv_oracle.c)",
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


def workload_config(n_gpus, rows, nnz):
    return {
        "workload": f"fp64 CSR SpMV y=A*x, synthetic R-MAT {rows}x{rows}, nnz={nnz} (avg {nnz / max(rows, 1):.2f}/row), "
                    "(a,b,c,d)=(0.57,0.19,0.19,0.05), seed 42, duplicates merged, columns sorted, val,x~U(-1,1), int32 indices",
        "baseline_config": "BASELINE.json configs[1] (R-MAT 1M x 1M avg 16 nnz/row, single B200); N>1 grows the matrix to N*1M rows",
        "rows": rows, "cols": rows, "nnz": nnz, "alpha": 1.0, "beta": 0.0,
        "parallelism": "single GPU" if n_gpus == 1 else f"{n_gpus} row-block shards of A and y (nnz-balanced), x in equal blocks, exchanged over NVLink every step",
        "l2": "no flush: 212 MB streamed per step per GPU > 126 MB L2; x stays L2-resident by design",
    }


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def prebuilt_spmv_call(cs, op, x, y):
    """One cusparseSpMV through the C ABI with the ctypes arguments built once (keeps host overhead ~2 us/step)."""
    api = op.api
    api.cusparseDnVecSetValues(op.vecX, x)
    api.cusparseDnVecSetValues(op.vecY, y)
    one, zero = C.c_double(1.0), C.c_double(0.0)
    fn = api.lib.cusparseSpMV
    argv = (op.handle, C.c_int(cs.CUSPARSE_OPERATION_NON_TRANSPOSE), C.cast(C.pointer(one), C.c_void_p), op.mat, op.vecX,
            C.cast(C.pointer(zero), C.c_void_p), op.vecY, C.c_int(cs.CUDA_R_64F), C.c_int(op.alg),
            C.c_void_p(op.buffer.data_ptr()))

    def call(_keep=(one, zero)):
        st = fn(*argv)
        if st != 0:
            raise RuntimeError(f"cusparseSpMV status {st}")
    return call


def time_steps(torch, fn, steps, dist_on, tail=None):
    """CUDA events on the current stream around `steps` calls of fn; `tail` (optional) makes the current stream wait for
    side streams before the closing event.  Returns (ms, t0, t1) -- max over ranks when distributed."""
    import torch.distributed as dist
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        fn()
    if tail is not None:
        tail()
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    if dist_on:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if dist_on:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, t0, t1


class PipelinedE2E:
    """The user-facing call with HOST buffers, every step: pinned host x -> device, cusparseSpMV through the C ABI, device
    y -> pinned host.  The three legs of consecutive steps overlap (copy streams + two device buffer sets): H2D of step
    k+1 and D2H of step k-1 run while the kernel of step k does; the SpMV itself stays on the handle's stream."""

    def __init__(self, torch, op, hx, rows, cols):
        self.torch, self.op = torch, op
        self.main = torch.cuda.current_stream()
        self.s_in, self.s_out = torch.cuda.Stream(), torch.cuda.Stream()
        self.hx = hx
        self.hy = [torch.empty(rows, dtype=torch.float64).pin_memory() for _ in range(2)]
        self.dx = [torch.empty(cols, dtype=torch.float64, device="cuda") for _ in range(2)]
        self.dy = [torch.empty(rows, dtype=torch.float64, device="cuda") for _ in range(2)]
        ev = lambda: [torch.cuda.Event() for _ in range(2)]
        self.x_ready, self.x_free, self.y_ready, self.y_free = ev(), ev(), ev(), ev()
        for e in self.x_free + self.y_free:
            e.record(self.main)
        self.k = 0

    def step(self):
        torch, i = self.torch, self.k & 1
        with torch.cuda.stream(self.s_in):
            self.s_in.wait_event(self.x_free[i])          # the kernel of step k-2 has finished reading dx[i]
            self.dx[i].copy_(self.hx, non_blocking=True)
            self.x_ready[i].record(self.s_in)
        self.main.wait_event(self.x_ready[i])
        self.main.wait_event(self.y_free[i])               # the D2H of step k-2 has finished reading dy[i]
        self.op(self.dx[i], self.dy[i], 1.0, 0.0)
        self.y_ready[i].record(self.main)
        self.x_free[i].record(self.main)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.y_ready[i])
            self.hy[i].copy_(self.dy[i], non_blocking=True)
            self.y_free[i].record(self.s_out)
        self.k += 1

    def drain(self):
        self.main.wait_stream(self.s_out)
        self.main.wait_stream(self.s_in)

    def last_result(self):
        return self.hy[(self.k - 1) & 1]


def north_star_leg(torch, cs, W, api, peak, steps):
    """R-MAT 10M x 10M, avg 16 nnz/row, fp64: the north-star acceptance config (target >= 0.70 of HBM peak, error < 1e-12)."""
    rows = 10_000_000
    off, col, val = W.rmat_csr(rows, avg_nnz=AVG_NNZ, seed=42, val_seed=43)
    nnz = int(col.numel())
    x = W.uniform(44, rows)
    nbytes = csr_bytes(rows, rows, nnz)
    out = {"workload": f"R-MAT {rows}x{rows}, nnz={nnz}, fp64, same generator as the headline config", "algorithmic_bytes": nbytes}
    ys = {}
    for impl in ("b200", "cusparse"):
        a = api if impl == "b200" else cs.Api("cusparse")
        op = cs.SpMVOperator(a, "csr", rows, rows, dict(off=off, col=col, val=val), preprocess=True)
        y = torch.zeros(rows, dtype=torch.float64, device="cuda")
        call = prebuilt_spmv_call(cs, op, x, y)
        for _ in range(5):
            call()
        ms, _, _ = time_steps(torch, call, steps, False)
        us = ms * 1e3 / steps
        out["ours" if impl == "b200" else "cusparse_torch_bundled"] = {
            "us_per_spmv": round(us, 2), "value": round(nbytes / us / 1e3, 1), "unit": UNIT, "frac_of_peak": round(nbytes / us / 1e3 / peak, 4)}
        ys[impl] = y
        op.close()
    out["rel_err_vs_cusparse"] = float((torch.linalg.norm(ys["b200"] - ys["cusparse"]) / torch.linalg.norm(ys["cusparse"])).item())
    out["target"] = {"frac_of_peak": 0.70, "rel_err": 1e-12}
    return out


def other_configs_leg(torch, cs, W, api, peak):
    """BASELINE.json configs[2] and configs[4] on one GPU, ours and the closed library (torch-bundled copy) on the same buffers:
    fp32 Sliced-ELL SpMV on the 7-pt Laplacian 256^3, and fp32 CSR x dense (2M x 2M, 32 non-zeros per row, n = 64,
    column-major B / C as in spmm_csr_example.c:100-104)."""
    out = {}
    closed = cs.Api("cusparse")

    def timed(fn, steps):
        for _ in range(3):
            fn()
        ms, _, _ = time_steps(torch, fn, steps, False)
        return ms * 1e3 / steps

    # ---- configs[2]: fp32 SELL, 7-pt 3D Laplacian 256^3, slice 32
    nx = 256
    n = nx ** 3
    off, col, val = W.laplace7_csr(nx, torch.float32)
    so, sc, sv = W.csr_to_sell(off, col, val, 32)
    nbytes = W.sell_bytes(n, n, int(sv.numel()), int(so.numel()) - 1, 4)
    arrays = dict(off=so, col=sc, val=sv, slice_size=32, nnz=int(col.numel()))
    x = W.uniform(44, n, torch.float32)
    res, ys = {"workload": f"fp32 Sliced-ELL (slice 32) SpMV, 7-pt Laplacian {nx}^3 ({n} rows, {int(col.numel())} non-zeros)", "algorithmic_bytes": nbytes}, {}
    for name, a in (("ours", api), ("cusparse_torch_bundled", closed)):
        op = cs.SpMVOperator(a, "sell", n, n, arrays)
        y = torch.zeros(n, dtype=torch.float32, device="cuda")
        us = timed(op.prebuilt(x, y, 1.0, 0.0), 50)
        res[name] = {"us_per_spmv": round(us, 2), "value": round(nbytes / us / 1e3, 1), "unit": UNIT, "frac_of_peak": round(nbytes / us / 1e3 / peak, 4)}
        ys[name] = y
        op.close()
    res["rel_err_vs_cusparse"] = float((torch.linalg.norm(ys["ours"].double() - ys["cusparse_torch_bundled"].double()) / torch.linalg.norm(ys["cusparse_torch_bundled"].double())).item())
    out["config3_sell_f32_laplace7_256"] = res
    del off, col, val, so, sc, sv, arrays, x, ys
    torch.cuda.empty_cache()

    # ---- configs[4]: fp32 CSR x dense
    rows, per_row, nn = 2_000_000, 32, 64
    g = torch.Generator(device="cuda").manual_seed(5)
    col = torch.randint(0, rows, (rows, per_row), device="cuda", generator=g, dtype=torch.int32).sort(dim=1).values.reshape(-1).contiguous()
    off = (torch.arange(rows + 1, device="cuda", dtype=torch.int64) * per_row).to(torch.int32)
    val = W.uniform(43, rows * per_row, torch.float32)
    arrays = dict(off=off, col=col, val=val)
    B = W.uniform(46, rows * nn, torch.float32)
    C0 = torch.zeros(rows * nn, dtype=torch.float32, device="cuda")
    nbytes = rows * per_row * 8 + (rows + 1) * 4 + 2 * rows * nn * 4
    res, cs_out = {"workload": f"fp32 CSR x dense, A {rows}x{rows} with {per_row} uniformly random non-zeros per row, B {rows}x{nn} and C column-major, "
                               "alpha=1, beta=0; single GPU (BASELINE.json quotes 8 GPUs: row blocks of A and C with B replicated)",
                   "algorithmic_bytes": nbytes, "flops": 2 * rows * per_row * nn}, {}
    for name, a in (("ours", api), ("cusparse_torch_bundled", closed)):
        ts = []
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            cs_out[name] = cs.spmm(a, rows, rows, arrays, B, C0, 1.0, 0.0, timing=(e0, e1))
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        us = sorted(ts[1:])[1]
        res[name] = {"us_per_spmm": round(us, 1), "gflops": round(res["flops"] / us / 1e3, 1), "value": round(nbytes / us / 1e3, 1), "unit": UNIT,
                     "frac_of_peak": round(nbytes / us / 1e3 / peak, 4)}
    res["rel_err_vs_cusparse"] = float((torch.linalg.norm(cs_out["ours"].double() - cs_out["cusparse_torch_bundled"].double()) / torch.linalg.norm(cs_out["cusparse_torch_bundled"].double())).item())
    out["config5_spmm_f32_2m_n64"] = res
    return out


def spmm_sharded_leg(torch, dist, cs, W, api, rank, world):
    """BASELINE.json configs[4] as it is quoted (8 x B200): A (2M x 2M, 32 per row, fp32) and C in contiguous row blocks, B (2M x 64,
    column-major) replicated on every GPU -- the product shards with no exchange step at all; time = max over ranks."""
    rows_g, per_row, nn = 2_000_000, 32, 64
    rows = rows_g // world
    g = torch.Generator(device="cuda").manual_seed(5 + rank)       # this rank's row block (uniformly random columns: any block looks alike)
    col = torch.randint(0, rows_g, (rows, per_row), device="cuda", generator=g, dtype=torch.int32).sort(dim=1).values.reshape(-1).contiguous()
    off = (torch.arange(rows + 1, device="cuda", dtype=torch.int64) * per_row).to(torch.int32)
    val = W.uniform(43 + rank, rows * per_row, torch.float32)
    B = W.uniform(46, rows_g * nn, torch.float32)
    C0 = torch.zeros(rows * nn, dtype=torch.float32, device="cuda")
    ts = []
    for _ in range(4):
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cs.spmm(api, rows, rows_g, dict(off=off, col=col, val=val), B, C0, 1.0, 0.0, timing=(e0, e1))
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ts.append(float(t.item()) * 1e3)
    us = sorted(ts[1:])[1]
    flops = 2 * rows_g * per_row * nn
    return {"config5_spmm_f32_2m_n64": {"workload": f"fp32 CSR x dense, A 2M x 2M with 32 per row in {world} row blocks, B 2M x 64 column-major replicated, "
                                                    "C in row blocks; no exchange step", "us_per_spmm": round(us, 1), "gflops": round(flops / us / 1e3, 1),
                                        "n_gpus": world, "scaling": "strong"}}


def cg_leg(torch, dist, cs, W, api, rank, world):
    """BASELINE.json configs[3]: CG, fp64, 5-pt Poisson 8192^2 (cg_example.c:71-128 generator), 200 fixed iterations,
    row-sharded over the N GPUs (strong scaling), iterations/s = 200 / max-over-ranks device time."""
    from cudalibrarysamples_b200.cg import make_cg_solver
    from cudalibrarysamples_b200.sharded import ShardedCsr
    n = CG_GRID * CG_GRID
    if n % world:
        return {"skipped": f"{n} rows do not divide by {world} ranks"}
    off, col, val = W.stencil5_csr(CG_GRID)
    nnz = int(col.numel())

    def make_local(r, c, arrays):
        return cs.SpMVOperator(api, "csr", r, c, arrays, preprocess=True)

    sh = ShardedCsr(off, col, val, rank, world, make_local, balance="rows")
    del off, col, val
    torch.cuda.empty_cache()
    ones = torch.ones(n, dtype=torch.float64, device="cuda")
    b = sh.new_y_shard()
    sh.spmv(sh.new_x_shard(ones), b, alpha=0.75, beta=0.0)      # b = 0.75 * A * 1 (cg_example.c:405-418)
    del ones
    solver = make_cg_solver(sh, b)
    solver.run(3)                                               # warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    x, norms = solver.run(CG_ITERS)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    r = b.clone()
    sh.spmv(x, r, alpha=-1.0, beta=1.0)                         # true residual with one more product (cg_example.c:289-300)
    rr = torch.dot(r, r).reshape(1)
    if world > 1:
        dist.all_reduce(rr)
    ms = float(ms.item())
    out = {"metric": "cg_iterations_per_second", "value": round(CG_ITERS / (ms * 1e-3), 2), "unit": "iterations/s",
           "ms_per_iteration": round(ms / CG_ITERS, 4), "iterations": CG_ITERS, "n_gpus": world, "scaling": "strong",
           "config": f"BASELINE.json configs[3]: fp64 CG, 5-pt Poisson {CG_GRID}^2 ({n} rows, nnz={nnz}), unpreconditioned "
                     "(the sample's IC(0)+SpSV preconditioner does not row-shard), x0 = 0, b = 0.75*A*1",
           "exchange": sh.exchange, "driver": solver.describe(),
           "residual_first": float(norms[0]), "residual_last": float(norms[-1]), "true_residual_last": float(rr.sqrt().item())}
    sh.local_op.close()
    return out


def toolkit_cusparse_leg(torch, off, col, val, x, y_ours, steps, warmup, peak):
    """The closed library as the reference samples link it (CUDA 12.9 toolkit's libcusparse), timed from C: inside this
    Python process only the copy torch ships can be loaded (cudalibrarysamples_b200/lib.py)."""
    import numpy as np
    exe = os.path.join(ROOT, "tools", "_bin", "spmv_timer.cusparse")
    if not os.path.exists(exe):
        return {"unavailable": "tools/_bin/spmv_timer.cusparse not built"}
    rows, nnz = int(off.numel()) - 1, int(col.numel())
    with tempfile.TemporaryDirectory(prefix="b200spmv_") as d:
        for name, t in (("off", off), ("col", col), ("val", val), ("x", x)):
            t.cpu().numpy().tofile(os.path.join(d, name + ".bin"))
        env = {k: v for k, v in os.environ.items() if k not in ("B200SPMV_CUSPARSE", "LD_PRELOAD")}
        p = subprocess.run([exe, d, str(rows), str(rows), str(nnz), str(steps), str(max(warmup, 3)), "cusparse"],
                           capture_output=True, text=True, timeout=180, env=env)
        if p.returncode != 0:
            return {"error": (p.stdout + p.stderr)[-400:]}
        res = json.loads(p.stdout.strip().splitlines()[-1])
        y = np.fromfile(os.path.join(d, "y_cusparse.bin"), dtype=np.float64)
    nbytes = csr_bytes(rows, rows, nnz)
    us = res["us_per_spmv"]
    yo = y_ours.cpu().numpy()
    return {"value": round(nbytes / us / 1e3, 3), "unit": UNIT, "us_per_spmv": us, "frac_of_peak": round(nbytes / us / 1e3 / peak, 4),
            "cusparse_version": res["cusparse_version"], "rel_diff_vs_ours": float(np.linalg.norm(yo - y) / np.linalg.norm(y)),
            "what": "closed cusparseSpMV of the CUDA 12.9 toolkit (what the reference samples link), preprocessed, timed by "
                    "tools/spmv_timer.c in its own process on the same matrix (separate process: same box, same loop shape)"}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from cudalibrarysamples_b200 import cusparse_api as cs
    from cudalibrarysamples_b200 import workloads as W
    from cudalibrarysamples_b200.sharded import ShardedCsr

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    dist_on = world > 1
    if dist_on:
        # NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION; the contract is ONE JSON line on stdout
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sampler = ClockSampler(local_rank)
    sampler.start()
    api = cs.Api("b200")
    api.reset_stats()
    peak, peak_src = measured_peak()

    rows = ROWS_PER_GPU * world
    off, col, val = W.rmat_csr(rows, avg_nnz=AVG_NNZ, seed=42, val_seed=43)
    nnz = int(col.numel())
    x = W.uniform(44, rows)
    total_bytes = csr_bytes(rows, rows, nnz)

    if not dist_on:
        op = cs.SpMVOperator(api, "csr", rows, rows, dict(off=off, col=col, val=val), preprocess=True)
        y = torch.zeros(rows, dtype=torch.float64, device="cuda")
        step = prebuilt_spmv_call(cs, op, x, y)
        kernel_bytes = total_bytes
        local = dict(rows=rows, nnz=nnz)
        exchange = None
    else:
        def make_local(r, c, arrays):
            # remote-column panels run with beta = 1: csr_flat_kernel then touches non-empty rows only (no per-row pass),
            # which is what a panel with mostly empty rows wants -- forced on for them, row-statistic choice for the rest
            api.set_option("B200SPMV_FLAT", "on" if arrays.get("role") == "remote" else "auto")
            try:
                return cs.SpMVOperator(api, "csr", r, c, arrays, preprocess=True)
            finally:
                api.set_option("B200SPMV_FLAT", "auto")
        def set_up(exchange_mode, overlap):
            """Shards, operators, the step callables, and the parity check of the sharded product at full size: every rank checks
            its y shard against the closed library run on the same local arrays and the gathered x."""
            sh = ShardedCsr(off, col, val, rank, world, make_local, exchange=exchange_mode, overlap=overlap, row_weight=args.row_weight)   # R-MAT rows read every x block
            xs = sh.new_x_shard(x)
            ys = sh.new_y_shard()
            step = sh.make_step(xs, ys, in_place=True)      # x is constant over the timed loop: published once, exchanged every step
            e2e_inner = sh.make_step(xs, ys, graph=False)   # e2e: a new x arrives from the host every step -> staged + exchanged
            if sh.panels:      # the local product alone = all column panels back to back, no exchange
                def local_call():
                    for c in sh.panel_calls:
                        c()
            else:
                local_call = sh.local_op.prebuilt(sh.x_full, ys, 1.0, 0.0)
            local = dict(rows=sh.rows, nnz=sh.nnz, x_block=sh.x_block)
            step()
            torch.cuda.synchronize()
            dist.barrier()
            capi = cs.Api("cusparse")
            cop = cs.SpMVOperator(capi, "csr", sh.rows, sh.cols_padded, dict(off=sh.off, col=sh.col, val=sh.val), preprocess=True)
            yc = torch.zeros_like(ys)
            cop(sh.x_full, yc, 1.0, 0.0)
            torch.cuda.synchronize()
            shard_rel = (torch.linalg.norm(ys - yc) / torch.linalg.norm(yc)).reshape(1)
            dist.all_reduce(shard_rel, op=dist.ReduceOp.MAX)
            local["max_rel_diff_vs_cusparse_over_ranks"] = float(shard_rel.item())
            assert local["max_rel_diff_vs_cusparse_over_ranks"] < 1e-12
            cop.close()
            return sh, xs, ys, step, e2e_inner, local_call, local

        # The column-panel step (N >= 4) has only ever run at N = 2 (forced); if its set-up or its parity check raises -- the same
        # Python error on every rank, the code path is rank-symmetric -- the run falls back to the plain step that was measured at
        # N = 2 (exchange, then one local product), then to the NCCL all-gather of round 1, and SAYS SO in the JSON line.
        attempts = [(args.exchange, True), (args.exchange, False), ("allgather", False)]
        if world < int(os.environ.get("B200SPMV_PANELS_FROM", "4")):
            attempts = attempts[1:]                         # no panels at this N anyway
        fallback_notes = []
        for k, (mode, overlap) in enumerate(attempts):
            try:
                sh, xs, ys, step, e2e_inner, local_call, local = set_up(mode, overlap)
                break
            except Exception as e:  # pragma: no cover (GPU boxes only)
                if k == len(attempts) - 1:
                    raise
                fallback_notes.append(f"exchange={mode} overlap={overlap}: {e!r}")
                print(f"[bench] rank {rank}: {fallback_notes[-1]} -- falling back", file=sys.stderr, flush=True)
                torch.cuda.synchronize()
                dist.barrier()
        if fallback_notes:
            local["fallback_from"] = fallback_notes
        del off, col, val
        torch.cuda.empty_cache()
        args._panels = sh.panels
        args._npanels = len(sh.panel_ops) if sh.panels else 1
        exchange = sh.describe_exchange()
        kernel_bytes = csr_bytes(sh.rows, sh.cols_padded, sh.nnz)

    for _ in range(max(args.warmup, 3)):
        step()
    ms_total, t0, t1 = time_steps(torch, step, args.steps, dist_on)
    ms_step = ms_total / args.steps
    y_last = None
    if args.dump_outputs:                          # later legs reuse the buffers: keep what the last timed step wrote
        y_last = gather_rows(torch, dist, ys, sh.bounds) if dist_on else y.cpu()
    value = total_bytes / (ms_step * 1e-3) / 1e9

    # dominant kernel alone (no exchange in the loop): average launch duration over the same K launches
    if dist_on:
        for _ in range(3):
            local_call()
        ms_k, _, _ = time_steps(torch, local_call, args.steps, False)
        kern_ms = ms_k / args.steps
        # every rank's local product alone, and the exchange alone (what the overlap has to hide)
        allk = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(allk, torch.tensor([kern_ms * 1e3], dtype=torch.float64, device="cuda"))
        local["local_product_us_per_rank"] = [round(float(t.item()), 2) for t in allk]
        local["rows_per_rank"] = [int(b - a) for a, b in zip(sh.bounds.tolist()[:-1], sh.bounds.tolist()[1:])]
        if sh.panels:
            # a diagnostic, not the metric: a host-side error in it (the same on every rank: the code path is rank-symmetric)
            # must not cost the run its JSON line
            try:
                def xonly():
                    for w in sh._start_exchange(xs):       # one wait per panel
                        w()
                for _ in range(3):
                    xonly()
                ms_x, _, _ = time_steps(torch, xonly, args.steps, True)
                local["exchange_alone_us"] = round(ms_x / args.steps * 1e3, 2)
            except (TypeError, AttributeError, ValueError, KeyError, IndexError) as e:  # pragma: no cover
                local["exchange_alone_us"] = None
                local["exchange_alone_error"] = repr(e)
        kern_ms = max(float(t.item()) for t in allk) * 1e-3
    else:
        kern_ms = ms_step
    achieved = kernel_bytes / (kern_ms * 1e-3) / 1e9
    stats_hot = api.stats()
    kname = api.last_csr_kernel()                  # the main kernel of the timed launches (before the other legs run theirs)

    # clocks: if the timed region was too short for NVML's sampling period, loop the same step for ~1 s and sample that
    probe = None
    if (t1 - t0) < 0.25:
        p0 = time.perf_counter()
        while time.perf_counter() - p0 < 1.0:
            for _ in range(50):
                step()
            torch.cuda.synchronize()
        probe = (p0, time.perf_counter())
    clocks = sampler.summary(t0, t1, probe)
    sampler.stop()

    # ---- e2e: the user-facing call with HOST buffers; x goes up and y comes back every step (A stays resident, as in
    #      cg_example.c:327-362 where the matrix is uploaded once and only vectors move) ----
    e2e = None
    if not dist_on:
        hx = x.cpu().pin_memory()
        pipe = PipelinedE2E(torch, op, hx, rows, rows)
        for _ in range(4):
            pipe.step()
        pipe.drain()
        ms_e, _, _ = time_steps(torch, pipe.step, args.steps, False, tail=pipe.drain)
        e2e = {"value": round(total_bytes / (ms_e / args.steps * 1e-3) / 1e9, 3), "unit": UNIT,
               "h2d_bytes_per_step": rows * 8, "d2h_bytes_per_step": rows * 8, "ms_per_step": round(ms_e / args.steps, 4),
               "what": "every step: pinned host x -> device, cusparseSpMV through the C ABI, device y -> pinned host; A resident; "
                       "the copies of neighbouring steps overlap the kernel (two device buffer sets, two copy streams)"}
        assert torch.equal(pipe.last_result(), y.cpu()), "e2e result differs from the device-resident result"
    else:
        hx = xs.cpu().pin_memory()
        hy = torch.empty(max(sh.rows, 1), dtype=torch.float64).pin_memory()[:sh.rows]

        def e2e_step():
            xs.copy_(hx, non_blocking=True)
            e2e_inner()
            hy.copy_(ys, non_blocking=True)
        for _ in range(3):
            e2e_step()
        ms_e, _, _ = time_steps(torch, e2e_step, args.steps, True)
        e2e = {"value": round(total_bytes / (ms_e / args.steps * 1e-3) / 1e9, 3), "unit": UNIT,
               "h2d_bytes_per_step": sh.x_block * 8 * world, "d2h_bytes_per_step": rows * 8,
               "ms_per_step": round(ms_e / args.steps, 4),
               "what": "per rank: pinned host x shard -> device, x exchange + cusparseSpMV, device y shard -> pinned host"}

    # ---- closed cusparseSpMV (csrmv_v3_kernel, sm_100 SASS) on the same device buffers: the on-box bar to beat ----
    closed = toolkit = None
    if not dist_on and not args.no_cusparse:
        step = prebuilt_spmv_call(cs, op, x, y)
        step()
        try:
            capi = cs.Api("cusparse")
            cop = cs.SpMVOperator(capi, "csr", rows, rows, dict(off=off, col=col, val=val), preprocess=True)
            y2 = torch.zeros_like(y)
            cstep = prebuilt_spmv_call(cs, cop, x, y2)
            for _ in range(max(args.warmup, 3)):
                cstep()
            ms_c, _, _ = time_steps(torch, cstep, args.steps, False)
            rel = float((torch.linalg.norm(y - y2) / torch.linalg.norm(y2)).item())
            closed = {"value": round(total_bytes / (ms_c / args.steps * 1e-3) / 1e9, 3), "unit": UNIT,
                      "ms_per_step": round(ms_c / args.steps, 4), "frac_of_peak": round(total_bytes / (ms_c / args.steps * 1e-3) / 1e9 / peak, 4),
                      "rel_diff_vs_ours": rel, "what": "closed libcusparse.so.12 cusparseSpMV (the copy torch ships; preprocessed), same buffers, same loop"}
            cop.close()
        except Exception as e:  # pragma: no cover
            closed = {"error": repr(e)}
        try:
            toolkit = toolkit_cusparse_leg(torch, off, col, val, x, y, args.steps, args.warmup, peak)
        except Exception as e:  # pragma: no cover
            toolkit = {"error": repr(e)}

    # ---- cpu_baseline: the oracle port on this box's host cores, rank 0, N=1 only, bounded sample ----
    cpu = None
    if not dist_on and not args.no_cpu:
        h_off, h_col, h_val, h_x = (t.cpu().numpy() for t in (off, col, val, x))
        threads = host_threads()
        med, times, ref = cpu_times(h_off, h_col, h_val, h_x, threads, 21)
        gbs = csr_bytes(rows, rows, nnz) / med / 1e9
        # correctness of the measured result against the oracle, at full size
        rel = float(np.linalg.norm(y.cpu().numpy() - ref) / np.linalg.norm(ref))
        assert rel < 1e-12, f"GPU result differs from the CPU oracle: {rel}"
        # SURVEY.md 8(d) also asks for the loop "single-threaded exactly as written" (spmv_csr_op_example.c:307-318): 5 repetitions, median
        med1, times1, _ = cpu_times(h_off, h_col, h_val, h_x, 1, 5)
        cpu = {"value": round(gbs, 3), "unit": UNIT, "cores": threads, "kind": "port", "statistic": "median",
               "sample": f"the full {rows}-row matrix, 21 repetitions, median ({med * 1e3:.2f} ms; min {min(times) * 1e3:.2f}); OpenMP dynamic row chunks",
               "single_thread": {"value": round(csr_bytes(rows, rows, nnz) / med1 / 1e9, 3), "unit": UNIT, "cores": 1,
                                 "ms_per_step": round(med1 * 1e3, 2), "sample": "the same matrix, the row loop as the sample writes it, 5 repetitions, median"},
               "gpu_vs_oracle_rel_err": rel}

    # ---- extra legs: north-star size, CG ----
    north = cg = None
    if not dist_on:
        op.close()
        del off, col, val, x, y
        torch.cuda.empty_cache()
        if not args.no_extra:
            try:
                north = north_star_leg(torch, cs, W, api, peak, max(20, args.steps // 4))
            except Exception as e:  # pragma: no cover
                north = {"error": repr(e)}
            torch.cuda.empty_cache()
    else:
        sh.close()
        del sh, xs, ys
        torch.cuda.empty_cache()
    if not args.no_extra:
        try:
            cg = cg_leg(torch, dist, cs, W, api, rank, world)
        except Exception as e:  # pragma: no cover
            cg = {"error": repr(e)}
    others = None
    if dist_on and not args.no_extra and 2_000_000 % world == 0:
        torch.cuda.empty_cache()
        try:
            others = spmm_sharded_leg(torch, dist, cs, W, api, rank, world)
        except Exception as e:  # pragma: no cover
            others = {"error": repr(e)}
    if not dist_on and not args.no_extra:
        torch.cuda.empty_cache()
        try:
            others = other_configs_leg(torch, cs, W, api, peak)
        except Exception as e:  # pragma: no cover
            others = {"error": repr(e)}

    if rank == 0:
        launches = {"b200::csr_flat_kernel<double>": 2, "b200::csr_seg_kernel<double>": 2, "b200::csr_tile_kernel<double>": 2,
                    "b200::csr_rowwise_kernel<double>": 2}.get(kname, 1) * (getattr(args, "_npanels", 1) if dist_on else 1)
        if dist_on and isinstance(exchange, str) and exchange.startswith("x shards in symmetric memory"):
            launches += 1          # the device-side barrier kernel of the p2p exchange (csrc/peer_sync.cu); the peer copies are copy-engine work
        line = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms_step, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(world, rows, nnz),
            "gflops": round(2 * nnz / (ms_step * 1e-3) / 1e9, 3),
            "frac_of_hbm_peak": round(value / (peak * world), 4),
            "roofline": {"bound": "hbm", "achieved": round(achieved, 3), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                         "traffic": None, "kernel": kname, "kernel_avg_us": round(kern_ms * 1e3, 3),
                         "algorithmic_bytes_per_launch": kernel_bytes, "peak_source": peak_src,
                         "per_rank": local},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches * args.steps, "clocks": clocks,
            "cusparse_same_box": closed, "cusparse_toolkit": toolkit, "north_star_10m": north, "cg_config4": cg, "other_configs": others,
            "exchange": exchange, "forwarded_calls_in_timed_region": stats_hot["forwarded"], "impl": "b200",
        }
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(prof):
            try:
                t = json.load(open(prof))
                if t.get("kernel") == kname and t.get("source_sha") == kernel_source_sha(kname) and world == 1:
                    line["roofline"]["traffic"] = t.get("dram_bytes_per_launch")
                    line["roofline"]["traffic_source"] = t.get("ncu_report")
                else:
                    line["roofline"]["traffic_note"] = ("profiles/traffic.json was captured from other kernel sources / another kernel / "
                                                        "another shard size: not quoted")
            except Exception:
                pass
        if y_last is not None:
            dump_output(args.dump_outputs, y_last.numpy())
        print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()


def main():
    # The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, torchrun hints) also write to fd 1, so
    # everything but our line is re-routed to stderr.
    global _REAL_STDOUT
    # Watchdog: a distributed hang must not wedge the GPU box -- dump every thread's stack and exit after the limit.
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("BENCH_WATCHDOG_S", "900" if "--impl" in sys.argv and "reference" in sys.argv else "420")), exit=True)
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--exchange", default="auto", help="N>1: how x is exchanged (auto | allgather | p2p)")
    ap.add_argument("--row-weight", type=float, default=ROW_WEIGHT, help="N>1: work model of the row partition: nnz + w * rows")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-cusparse", action="store_true", help="skip the closed-library comparison legs")
    ap.add_argument("--no-extra", action="store_true", help="skip the north-star and CG legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write y of the last timed step to DIR/y.npy (fp64) for comparing builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
