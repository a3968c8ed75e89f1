"""CPU, gloo: bench.run_ours -- the real multi-GPU branch of bench.py -- executed end to end at world 2, 4 and 8 with only the
device layer replaced (tests/bench_dry_run_worker.py): column panels, staged set-up, timing loops, exchange-alone diagnostic,
e2e loop, CG leg, JSON line.  Round 2 lost its N >= 4 runs to a one-line host bug in exactly this code; it fails here now."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "bench_dry_run_worker.py")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def dry_run(world, tmp_path, fail_first=False):
    port, out = _free_port(), str(tmp_path / "line.json")
    env = {k: v for k, v in os.environ.items() if not k.startswith("B200SPMV_")}
    procs = [subprocess.Popen([sys.executable, WORKER, str(r), str(world), str(port), out, "1" if fail_first else "0"], env=env,
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(world)]
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=300)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            pytest.fail("bench dry run timed out")
        logs.append(o)
    assert all(p.returncode == 0 for p in procs), "\n".join(l[-3000:] for l in logs)
    check_dumped_y(world, str(tmp_path / "outputs" / "y.npy"))
    return json.loads(open(out).read().strip().splitlines()[-1])


def check_dumped_y(world, path):
    """--dump-outputs: y of the last timed step, all rows in row order, equals y = A*x of the workload the worker generates."""
    from oracle import oracle as O
    rows = 1500 * world
    off, col, val = O.rmat_csr(rows, avg_nnz=16, seed=42, val_seed=43)
    want = O.spmv_csr(off, col, val, O.uniform(44, rows))
    y = np.load(path)
    assert y.dtype == np.float64 and y.shape == (rows,)
    assert np.linalg.norm(y - want) <= 1e-12 * np.linalg.norm(want)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_bench_multi_gpu_branch_runs_end_to_end(world, tmp_path):
    line = dry_run(world, tmp_path)
    assert line["n_gpus"] == world and line["metric"] == "csr_spmv_fp64_effective_hbm_bandwidth" and line["scaling"] == "weak"
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["steps"] == 3 and line["warmup"] == 3
    per = line["roofline"]["per_rank"]
    assert per["max_rel_diff_vs_cusparse_over_ranks"] < 1e-12                       # panels summed against the whole local product
    assert len(per["local_product_us_per_rank"]) == world and sum(per["rows_per_rank"]) == 1500 * world
    assert "exchange_alone_us" in per and per["exchange_alone_us"] is not None      # the diagnostic that crashed in round 2
    assert "fallback_from" not in per
    assert "column panel" in line["exchange"] or "panel" in line["exchange"]
    assert line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 1500 * world * 8
    assert line["gpu_launches"] > 0 and line["config"]["rows"] == 1500 * world
    cg = line["cg_config4"]
    assert cg["iterations"] == 5 and cg["n_gpus"] == world and cg["residual_last"] < cg["residual_first"]


def test_bench_falls_back_and_says_so(tmp_path):
    line = dry_run(4, tmp_path, fail_first=True)
    per = line["roofline"]["per_rank"]
    assert len(per["fallback_from"]) == 1 and "injected failure" in per["fallback_from"][0]
    assert "panel" not in line["exchange"]                                           # the plain step ran
    assert per["max_rel_diff_vs_cusparse_over_ranks"] < 1e-12 and line["value"] > 0


def test_bench_single_gpu_branch_runs_end_to_end(tmp_path):
    """N = 1: the headline line -- timing loop through the prebuilt C-ABI call, the pipelined e2e loop (its result compared with the
    device-resident one), cpu_baseline with the GPU result checked against the oracle, the single-thread baseline, the roofline block."""
    line = dry_run(1, tmp_path)
    assert line["n_gpus"] == 1 and line["value"] > 0 and line["config"]["rows"] == 1500 and line["exchange"] is None
    assert line["e2e"]["h2d_bytes_per_step"] == 1500 * 8 and line["e2e"]["d2h_bytes_per_step"] == 1500 * 8 and line["e2e"]["value"] > 0
    cpu = line["cpu_baseline"]
    assert cpu["kind"] == "port" and cpu["gpu_vs_oracle_rel_err"] < 1e-12 and cpu["value"] > 0
    assert cpu["single_thread"]["cores"] == 1 and cpu["single_thread"]["value"] > 0
    r = line["roofline"]
    assert r["bound"] == "hbm" and r["kernel"] == "b200::csr_flat_kernel<double>" and 0 < r["frac"] and r["algorithmic_bytes_per_launch"] > 0
    assert r["traffic"] is not None or "traffic_note" in r
    assert line["gpu_launches"] == 2 * 3 and line["forwarded_calls_in_timed_region"] == 0
