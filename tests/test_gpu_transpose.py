"""CSR -> CSC twin: bit-exact against SMatrix::transpose (reference src/util/Smatrix.h:155-185)."""
import numpy as np
import pytest

from fmwr_b200 import _lib as L
from fmwr_b200 import synth

pytestmark = pytest.mark.gpu


def test_transpose_kat(gpu_ctx):
    # src/test/SMatrix.cpp:10-16
    M = np.array([[1, 0, 0, 0], [0, 3, 4, 0], [0, 0, 5, 6], [0, 8, 0, 1]], np.float32)
    rowptr = [0]; col = []; val = []
    for r in M:
        nz = np.nonzero(r)[0]; col += list(nz); val += list(r[nz]); rowptr.append(len(col))
    d = L.Data.from_csr32(gpu_ctx, 4, 4, rowptr, col, val)
    d.transpose()
    cp, cr, cv = d.get_csc()
    assert list(cp) == [0, 1, 3, 5, 7] and list(cr) == [0, 1, 3, 1, 2, 2, 3] and list(cv) == [1, 3, 8, 4, 5, 6, 1]


@pytest.mark.parametrize("n,p,m,empty", [(1000, 300, 9, False), (5000, 70, 30, True), (300, 5000, 4, True), (1, 1, 1, False)])
def test_transpose_random(gpu_ctx, port, n, p, m, empty):
    rowptr, col, val = synth.random_csr(n, p, m, seed=n + p, empty_rows=empty)
    d = L.Data.from_csr32(gpu_ctx, n, p, rowptr, col, val)
    d.transpose()
    got = d.get_csc()
    want = port.transpose(n, p, rowptr, col, val)
    for a, b in zip(got, want):
        assert a.dtype == b.dtype and (a == b).all()


def test_transpose_matches_restatement_on_full_rows(gpu_ctx, port):
    # every row non-empty, against the restatement's counting sort, which equals SMatrix::transpose's O(n*p) output
    # bit for bit (tests/test_golden.py, tests/test_oracle_pinning.py)
    rowptr, col, val = synth.random_csr(400, 120, 7, seed=12, empty_rows=False)
    d = L.Data.from_csr32(gpu_ctx, 400, 120, rowptr, col, val)
    d.transpose()
    got = d.get_csc()
    want = port.transpose(400, 120, rowptr, col, val)
    for a, b in zip(got, want):
        assert a.shape == b.shape and (a == b).all()


def test_transpose_roundtrip_large(gpu_ctx):
    # size-independent property at a size the oracle would take long on: transpose twice == identity
    ds_rowptr, ds_col, ds_val, p = synth.fields_csr(300_000, synth.criteo_fields(39 * 5000), None, 1, 5)
    n = 300_000
    d = L.Data.from_csr32(gpu_ctx, n, p, ds_rowptr, ds_col, ds_val)
    d.transpose()
    cp, cr, cv = d.get_csc()
    assert cp[-1] == ds_col.size and np.all(np.diff(cp.astype(np.int64)) >= 0)
    # rows ascending inside every column
    seg = np.repeat(np.arange(p), np.diff(cp.astype(np.int64)))
    order_ok = (np.diff(cr.astype(np.int64)) > 0) | (np.diff(seg) > 0)
    assert order_ok.all()
    d2 = L.Data.from_csr32(gpu_ctx, p, n, cp, cr, cv)
    d2.transpose()
    rp, rc, rv = d2.get_csc()
    assert (rp == ds_rowptr).all() and (rc == ds_col).all() and (rv == ds_val).all()


def test_r_list_ingest_matches_csr32(gpu_ctx):
    rowptr, col, val = synth.random_csr(2000, 100, 12, seed=3, empty_rows=True)
    rs = np.diff(rowptr.astype(np.int64)).astype(np.int32)
    d = L.Data.from_r_lists(gpu_ctx, 2000, 100, rs, col.astype(np.int32), val.astype(np.float64), np.arange(2000, dtype=np.float64))
    r2, c2, v2, y2 = d.get_csr()
    assert (r2 == rowptr).all() and (c2 == col).all() and (v2 == val).all() and (y2 == np.arange(2000)).all()
    with pytest.raises(L.FmwrError) as e:
        L.Data.from_r_lists(gpu_ctx, 3, 100, np.array([1, 1, 5], np.int32), col[:3].astype(np.int32), val[:3].astype(np.float64))
    assert "row_size is not correct" in str(e.value)     # same message as SMatrix::assign (Smatrix.h:52)
