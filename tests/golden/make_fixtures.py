#!/usr/bin/env python
"""Generates the committed fixtures of tests/golden/.

  toy_4x4.mtx            the reference's 4x4 toy matrix (spmv_csr_example.c:45-52) written by OUR writer
  rmat_300.mtx           a small R-MAT (oracle generator) with empty rows, written by our writer
  sym_lower_5.mtx        a `symmetric` file holding the lower triangle only
  test_real.mtx          a verbatim copy of the reference's own cuSOLVERSp2cuDSS/test_real.mtx (data, 1 KB; not generated)
  reference_mtx.json     what test_real.mtx parses to (sizes, nnz, row counts, a checksum of the values); the CPU test
                         re-reads the stored copy and checks it against this record

Not written by this script: cg_example.cusparse.out and bicgstab_example.cusparse.out, the stdout of the reference's cg /
bicgstab samples linked against the closed cuSPARSE of CUDA 12.9 (oracle/_ref/*.cusparse, `make -C oracle ref`), run on
one B200; tests/test_parity_gpu.py compares the shim-linked samples' convergence with them.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from cudalibrarysamples_b200.mtx import read_matrix_market, write_matrix_market  # noqa: E402
from oracle import oracle as O  # noqa: E402

T = O.TOY
write_matrix_market(os.path.join(HERE, "toy_4x4.mtx"), 4, 4, T["csr_off"], T["csr_col"], T["val"], "spmv_csr_example.c:45-52")
off, col, val = O.rmat_csr(300, avg_nnz=5, seed=11, val_seed=12)
write_matrix_market(os.path.join(HERE, "rmat_300.mtx"), 300, 300, off, col, val, "oracle.rmat_csr(300, avg_nnz=5, seed=11, val_seed=12)")
with open(os.path.join(HERE, "sym_lower_5.mtx"), "w") as f:
    f.write("%%MatrixMarket matrix coordinate real symmetric\n% lower triangle of a 5x5 SPD stencil\n5 5 9\n")
    for i in range(5):
        f.write(f"{i + 1} {i + 1} 4.0\n")
        if i:
            f.write(f"{i + 1} {i} -1.0\n")
ref = os.path.join(HERE, "test_real.mtx")
if os.path.exists(ref):
    n, m, off, col, val = read_matrix_market(ref)
    json.dump(dict(source="cuSOLVERSp2cuDSS/test_real.mtx", rows=n, cols=m, nnz=int(col.size), row_counts=np.diff(off).tolist(),
                   col_sum=int(col.astype(np.int64).sum()), val_sum=float(val.sum()),
                   y_for_x_ones=O.spmv_csr(off, col, val, np.ones(m)).tolist()),
              open(os.path.join(HERE, "reference_mtx.json"), "w"), indent=1)
print("fixtures written")
