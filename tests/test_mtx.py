"""CPU: Matrix Market ingestion (cudalibrarysamples_b200/mtx.py), mirror of cuDSS/simple_matrix_market/matrix_market_reader.h."""
import json
import os

import numpy as np
import pytest

from cudalibrarysamples_b200.mtx import MtxReaderError, read_matrix_market, write_matrix_market
from oracle import oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_toy_fixture_round_trips_to_the_reference_arrays():
    n, m, off, col, val = read_matrix_market(os.path.join(G, "toy_4x4.mtx"), dtype=np.float32)
    T = O.TOY
    assert (n, m) == (4, 4)
    assert np.array_equal(off, T["csr_off"]) and np.array_equal(col, T["csr_col"]) and np.array_equal(val, T["val"])
    assert np.array_equal(O.spmv_csr(off, col, val, T["x"]), T["y_result"])        # {19, 8, 51, 52}


def test_rmat_fixture_with_empty_rows():
    n, m, off, col, val = read_matrix_market(os.path.join(G, "rmat_300.mtx"))
    o2, c2, v2 = O.rmat_csr(300, avg_nnz=5, seed=11, val_seed=12)
    assert np.array_equal(off, o2) and np.array_equal(col, c2) and np.array_equal(val, v2)
    assert (np.diff(off) == 0).any()


def test_symmetric_expansion():
    n, m, off, col, val = read_matrix_market(os.path.join(G, "sym_lower_5.mtx"))
    dense = np.zeros((5, 5))
    for i in range(5):
        dense[i, col[off[i]:off[i + 1]]] = val[off[i]:off[i + 1]]
    assert np.array_equal(dense, dense.T) and dense[0, 1] == -1 and col.size == 13
    n, m, off, col, val = read_matrix_market(os.path.join(G, "sym_lower_5.mtx"), expand_symmetric=False)
    assert col.size == 9                                          # as stored, like the reference reader


def test_reference_file_parses_to_the_recorded_summary():
    """test_real.mtx is a stored copy of the reference's cuSOLVERSp2cuDSS/test_real.mtx (rec["source"])."""
    rec = json.load(open(os.path.join(G, "reference_mtx.json")))
    n, m, off, col, val = read_matrix_market(os.path.join(G, "test_real.mtx"))
    assert (n, m, int(col.size)) == (rec["rows"], rec["cols"], rec["nnz"])
    assert np.diff(off).tolist() == rec["row_counts"] and int(col.astype(np.int64).sum()) == rec["col_sum"]
    assert np.allclose(O.spmv_csr(off, col, val, np.ones(m)), rec["y_for_x_ones"], rtol=0, atol=1e-13)


def test_reader_errors_mirror_the_reference_status_codes(tmp_path):
    p = tmp_path / "bad.mtx"
    p.write_text("%%MatrixMarket matrix array real general\n2 2\n1\n2\n3\n4\n")
    with pytest.raises(MtxReaderError) as e:
        read_matrix_market(str(p))
    assert e.value.status == "MtxReaderErrorInvalidFormatInHeader"
    p.write_text("%%MatrixMarket matrix coordinate real general\n2 2 3\n1 1 1.0\n2 2 1.0\n")
    with pytest.raises(MtxReaderError) as e:
        read_matrix_market(str(p))
    assert e.value.status == "MtxReaderErrorWrongNnz"
    p.write_text("%%MatrixMarket matrix coordinate real general\n2 2 1\n3 1 1.0\n")
    with pytest.raises(MtxReaderError) as e:
        read_matrix_market(str(p))
    assert e.value.status == "MtxReaderErrorOutOfBoundRowIndex"
    with pytest.raises(MtxReaderError) as e:
        read_matrix_market(str(tmp_path / "missing.mtx"))
    assert e.value.status == "MtxReaderErrorFileNotFound"


def test_writer_reader_round_trip(tmp_path):
    off, col, val = O.rmat_csr(120, avg_nnz=7, seed=5, val_seed=6)
    p = str(tmp_path / "a.mtx")
    write_matrix_market(p, 120, 120, off, col, val)
    n, m, o2, c2, v2 = read_matrix_market(p)
    assert np.array_equal(off, o2) and np.array_equal(col, c2) and np.array_equal(val, v2)
