"""Helper of tests/test_bench_dry_run.py (not a test module): runs bench.run_ours -- the REAL function, the multi-GPU branch --
in one rank of a gloo process group on CPU tensors.  Only the device layer is replaced:

  torch.cuda.*            no-op streams / events (events read time.perf_counter), is_available() -> True
  device="cuda" factories the same factories on the CPU;  Tensor.pin_memory -> identity
  dist.init_process_group gloo instead of nccl
  workload generators     the CPU oracle's generators at a size a CPU handles (bench.ROWS_PER_GPU / CG_GRID shrunk)
  cusparse_api operators  an oracle-backed operator with the same interface (prebuilt / __call__ / close; no `handle`, so no
                          CUDA-graph capture is attempted) -- for the b200 library and for the closed library alike

Everything else is bench.py / sharded.py / cg.py as shipped: shard set-up with column panels (B200SPMV_PANELS_FROM=2), the
staged attempts, the timing loops, the exchange-alone diagnostic, the e2e loop, the CG leg, the assembly of the JSON line."""
import contextlib
import os
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(rank, world, port, out_path, fail_first_attempt):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                      B200SPMV_PANELS_FROM="2")
    import numpy as np
    import torch
    import torch.distributed as dist

    import bench
    from cudalibrarysamples_b200 import cusparse_api as cs
    from cudalibrarysamples_b200 import sharded
    from cudalibrarysamples_b200 import workloads as W
    from oracle import oracle as O

    # ---- torch.cuda: no device
    class Stream:
        cuda_stream = 0

        def wait_event(self, e):
            pass

        def wait_stream(self, s):
            pass

        def synchronize(self):
            pass

    class Event:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, stream=None):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    torch.cuda.is_available = lambda: True
    torch.cuda.set_device = lambda d: None
    torch.cuda.synchronize = lambda *a: None
    torch.cuda.empty_cache = lambda: None
    torch.cuda.current_stream = lambda *a: Stream()
    torch.cuda.Stream = Stream
    torch.cuda.Event = Event
    torch.cuda.stream = lambda s: contextlib.nullcontext()
    torch.Tensor.pin_memory = lambda self, *a, **k: self
    for name in ("tensor", "zeros", "empty", "ones", "full", "arange"):
        real = getattr(torch, name)

        def on_cpu(*a, _real=real, **k):
            if k.get("device") is not None and str(k["device"]).startswith("cuda"):
                k["device"] = "cpu"
            return _real(*a, **k)
        setattr(torch, name, on_cpu)
    real_init = dist.init_process_group
    dist.init_process_group = lambda backend, **k: real_init("gloo", rank=rank, world_size=world)

    # ---- workloads: the oracle's generators, small
    bench.ROWS_PER_GPU = 1500
    bench.CG_GRID = 32
    bench.CG_ITERS = 5
    W.rmat_csr = lambda rows, avg_nnz=16, seed=42, val_seed=43, **k: tuple(torch.from_numpy(a) for a in O.rmat_csr(rows, avg_nnz=avg_nnz, seed=seed, val_seed=val_seed))
    W.uniform = lambda seed, n, dtype=torch.float64: torch.from_numpy(O.uniform(seed, n)).to(dtype)
    W.stencil5_csr = lambda grid: tuple(torch.from_numpy(a) for a in O.gen_stencil5(grid))

    # ---- the C-ABI operators: oracle-backed, same interface (descriptor handles are plain objects; the fake library's
    #      cusparseSpMV finds the operator by its matrix descriptor and the vectors by theirs, as the shim's side tables do)
    mats, vecs = {}, {}

    class Operator:
        built = 0

        def __init__(self, api, fmt, rows, cols, arrays, base=0, preprocess=True, **k):
            assert fmt == "csr"
            Operator.built += 1
            if fail_first_attempt and Operator.built == 1:
                raise TypeError("injected failure of the first set-up attempt")
            self.api, self.rows, self.cols = api, rows, cols
            self.off, self.col, self.val = (arrays[n].numpy() for n in ("off", "col", "val"))
            # (multi-GPU: no attribute named `handle`, so sharded.py does not try to capture CUDA graphs)
            self.mat, self.vecX, self.vecY, self.alg = object(), object(), object(), 0
            if world == 1:
                self.handle = None                       # prebuilt_spmv_call passes it through to the (fake) library
            self.buffer = torch.zeros(16, dtype=torch.uint8)
            mats[id(self.mat)] = self

        def __call__(self, x, y, alpha=1.0, beta=0.0):
            if self.rows:
                y.copy_(torch.from_numpy(O.spmv_csr(self.off, self.col, self.val, x.numpy(), y.numpy(), alpha, beta)))
            return y

        def prebuilt(self, x, y, alpha=1.0, beta=0.0):
            return lambda: self(x, y, alpha, beta)

        def close(self):
            pass

    cs.SpMVOperator = Operator

    def fake_spmv(handle, op, alpha, mat, vec_x, beta, vec_y, ctype, alg, buf):
        import ctypes as C
        o = mats[id(mat)]
        a = C.cast(alpha, C.POINTER(C.c_double))[0]
        b = C.cast(beta, C.POINTER(C.c_double))[0]
        o(vecs[id(vec_x)], vecs[id(vec_y)], a, b)
        return 0

    class Api:
        def __init__(self, impl="b200"):
            self.impl = impl
            self.lib = types.SimpleNamespace(cusparseSpMV=fake_spmv)

        def cusparseDnVecSetValues(self, d, values):
            vecs[id(d)] = values

        def set_option(self, k, v):
            pass

        def reset_stats(self):
            pass

        def stats(self):
            return dict(native=0, forwarded=0, analyze=0)

        def last_csr_kernel(self):
            return "b200::csr_flat_kernel<double>"
    cs.Api = Api

    # one process: the single-GPU branch (headline line: timing loop, pipelined e2e, cpu_baseline against the oracle at full size);
    # its extra legs need the real library or 10 M rows and sit in try / except blocks of their own: skipped here
    args = types.SimpleNamespace(gpus=world, steps=3, warmup=1, exchange="auto", row_weight=2.0, no_cpu=world > 1, no_cusparse=True,
                                 no_extra=world == 1, dump_outputs=os.path.join(os.path.dirname(out_path), "outputs"))
    bench._REAL_STDOUT = open(out_path, "w") if rank == 0 else open(os.devnull, "w")
    bench.run_ours(args)
    bench._REAL_STDOUT.close()


if __name__ == "__main__":
    main(int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), sys.argv[4], sys.argv[5] == "1")
