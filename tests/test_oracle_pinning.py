"""Pins the plain-C restatement (oracle/fm_oracle.c) against the reference's own headers compiled unmodified
(oracle/_ref) -- function by function, on seeded random inputs and the reference's two hand-derivable KATs.
Where the reference build is absent, `ref` replays a snapshot of the RESTATEMENT's own answers to these calls
(tests/pinning_snapshot.py): there these tests hold the restatement to its recorded behaviour, and tests/test_golden.py
holds it to reference-generated vectors."""
import numpy as np
import pytest

from oracle import oracle as O
from fmwr_b200 import synth
from tests.pinning_snapshot import same
from tests.util import relerr


def csr_of(M):
    rowptr = [0]; col = []; val = []
    for r in np.asarray(M, np.float32):
        nz = np.nonzero(r)[0]; col += list(nz); val += list(r[nz]); rowptr.append(len(col))
    return np.array(rowptr, np.uint32), np.array(col, np.uint32), np.array(val, np.float32)


def test_kat_forward_both(port, ref):
    # src/test/model.cpp:12-34
    X = [[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [1, 0, 0, 0], [0, 0, 1, 0], [1, 0, 0, 1], [2, 0, 0, 0], [0, 0, 0, 1]]
    rowptr, col, val = csr_of(X)
    w = np.full(4, 0.1); v = np.full((4, 3), 0.2)
    want = np.array([.1, .1, .1, .1, .1, .32, .2, .1])
    for orc in (port, ref):
        got = orc.predict(O.make_cfg(k=3), 8, 4, rowptr, col, val, 0.0, w, v, 0)
        assert relerr(got, want) < 1e-15
        sig = orc.predict(O.make_cfg(k=3, solver=O.SGD), 8, 4, rowptr, col, val, 0.0, w, v, 1)
        assert abs(sig[0] - 0.5249791875) < 1e-9 and abs(sig[5] - 0.5793242521) < 1e-9 and abs(sig[6] - 0.5498339973) < 1e-9
        pn = orc.predict(O.make_cfg(k=3, solver=O.ALS), 8, 4, rowptr, col, val, 0.0, w, v, 1)
        assert abs(pn[0] - 0.5398278371) < 1e-9 and abs(pn[5] - 0.6255158326) < 1e-9 and abs(pn[6] - 0.5792597086) < 1e-9


def test_kat_transpose_both(port, ref):
    # src/test/SMatrix.cpp:10-16
    rowptr, col, val = csr_of([[1, 0, 0, 0], [0, 3, 4, 0], [0, 0, 5, 6], [0, 8, 0, 1]])
    for tp, ti, tv in (port.transpose(4, 4, rowptr, col, val), ref.transpose(4, 4, rowptr, col, val, 1), ref.transpose(4, 4, rowptr, col, val, 0)):
        assert list(tp) == [0, 1, 3, 5, 7] and list(ti) == [0, 1, 3, 1, 2, 2, 3] and list(tv) == [1, 3, 8, 4, 5, 6, 1]


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_forward_and_rowwise_pinned(port, ref, seed):
    rng = np.random.default_rng(seed)
    n, p, k = 300, 50, 1 + seed * 3
    rowptr, col, val = synth.random_csr(n, p, 9, seed=seed)
    w = rng.normal(0, 0.2, p); v = rng.normal(0, 0.2, (p, k))
    for solver in (O.SGD, O.ALS):
        for link in (0, 1):
            c = O.make_cfg(solver=solver, k=k)
            a = port.predict(c, n, p, rowptr, col, val, 0.3, w, v, link)
            b = ref.predict(c, n, p, rowptr, col, val, 0.3, w, v, link)
            assert relerr(a, b) < 1e-14
    a = port.predict_rows(O.make_cfg(k=k), n, p, rowptr, col, val, 0.3, w, v)
    b = ref.predict_rows(O.make_cfg(k=k), n, p, rowptr, col, val, 0.3, w, v)
    assert same(a[0], b[0]) and same(a[1], b[1])


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
@pytest.mark.parametrize("task", [O.CLASSIFICATION, O.REGRESSION])
def test_row_solvers_pinned_bitwise(port, ref, solver, task):
    rng = np.random.default_rng(7)
    n, p, k = 250, 40, 3
    rowptr, col, val = synth.random_csr(n, p, 6, seed=5)
    y = (np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == O.CLASSIFICATION else rng.normal(0, 1, n)).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    for regs in ({}, dict(l1_w=0.02, l1_v=0.01), dict(l2_w=0.01, l2_v=0.02, l2_w0=0.05)):
        for step_size, metric in ((-1, O.LL), (37, O.LL if task == O.CLASSIFICATION else O.RMSE), (50, O.AUC if task == O.CLASSIFICATION else O.MAE)):
            c = O.make_cfg(task=task, solver=solver, k=k, max_iter=3 * (n - 1) + 4, min_target=float(y.min()), max_target=float(y.max()),
                           step_size=step_size, metric=metric, convergence=1e-3, **regs)
            a = port.train(c, n, p, rowptr, col, val, y, 0.2, w, v, max_rec=60)
            b = ref.train(c, n, p, rowptr, col, val, y, 0.2, w, v, max_rec=60)
            assert a[0] == b[0] and same(a[1], b[1]) and same(a[2], b[2])
            assert a[3]["n_rec"] == b[3]["n_rec"] and a[3]["convergent"] == b[3]["convergent"]
            # AUC: the reference sorts by |score| with the unstable std::sort (src/core/Evaluation.h:65); rows with tied
            # |score| of opposite class land in an implementation-defined order, so ties move the area slightly
            tol = 1e-2 if metric == O.AUC else 1e-13
            assert same(a[3]["rec_index"], b[3]["rec_index"]) and relerr(a[3]["eval_train"], b[3]["eval_train"]) < tol


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
@pytest.mark.parametrize("k,max_nnz", [(4, 70), (128, 45), (32, 100)])
def test_row_solvers_pinned_on_ragged_empty_and_wide_rows(port, ref, solver, k, max_nnz):
    # the shapes tests/test_gpu_exact.py::test_exact_row_shapes_and_layouts holds the CUDA kernel to: rows from empty to
    # 100 non-zeros (the reference's TDAP position refresh, F6, reads z_w[0 .. nnz) there), k up to 128
    rng = np.random.default_rng(11)
    n, p = 90, 300
    rowptr, col, val = synth.random_csr(n, p, max_nnz, seed=21, empty_rows=True)
    assert (np.diff(rowptr.astype(np.int64)) == 0).any()
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.05, p); v = rng.normal(0, 0.05, (p, k))
    c = O.make_cfg(solver=solver, k=k, max_iter=2 * (n - 1) + 7, l1_w=0.001, l2_w=0.001, l2_v=0.002)
    a = port.train(c, n, p, rowptr, col, val, y, 0.1, w, v)
    b = ref.train(c, n, p, rowptr, col, val, y, 0.1, w, v)
    assert a[0] == b[0] and same(a[1], b[1]) and same(a[2], b[2])
    assert np.isfinite(a[2]).all()


def test_random_step_stream_pinned(port, ref):
    rng = np.random.default_rng(8)
    n, p, k = 200, 30, 2
    rowptr, col, val = synth.random_csr(n, p, 5, seed=6)
    y = rng.normal(0, 1, n).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    rands = rng.integers(0, 2**31 - 1, 4000).astype(np.int32)
    c = O.make_cfg(task=O.REGRESSION, solver=O.FTRL, k=k, max_iter=500, random_step=4, min_target=float(y.min()), max_target=float(y.max()))
    port.set_streams(None, None, rands); ref.set_streams(None, None, rands)
    a = port.train(c, n, p, rowptr, col, val, y, 0.0, w, v)
    b = ref.train(c, n, p, rowptr, col, val, y, 0.0, w, v)
    assert port.stream_pos() == ref.stream_pos()
    port.set_streams(None, None, None); ref.set_streams(None, None, None)
    assert a[0] == b[0] and same(a[1], b[1]) and same(a[2], b[2])


@pytest.mark.parametrize("solver", [O.ALS, O.MCMC])
@pytest.mark.parametrize("task", [O.CLASSIFICATION, O.REGRESSION])
@pytest.mark.parametrize("enable_v", [0, 1])
def test_coordinate_solvers_pinned(port, ref, solver, task, enable_v):
    rng = np.random.default_rng(9)
    n, p, k = 350, 45, 3
    rowptr, col, val = synth.random_csr(n, p, 6, seed=7)
    y = (np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == O.CLASSIFICATION else rng.normal(0, 1, n)).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    normals = rng.standard_normal(50000); gammas = rng.gamma(40.0, 1.0, 2000); rands = rng.integers(0, 2**31 - 1, 500000).astype(np.int32)
    c = O.make_cfg(task=task, solver=solver, k=k, max_iter=5, enable_v=enable_v, l2_w0=0.1, min_target=float(y.min()), max_target=float(y.max()),
                   step_size=1, metric=O.LL if task == O.CLASSIFICATION else O.RMSE)
    port.set_streams(normals, gammas, rands); ref.set_streams(normals, gammas, rands)
    a = port.train(c, n, p, rowptr, col, val, y, 0.1, w, v, max_rec=10)
    b = ref.train(c, n, p, rowptr, col, val, y, 0.1, w, v, use_ref_transpose=1, max_rec=10)
    assert port.stream_pos() == ref.stream_pos() and port.stream_pos()["overrun"] == 0
    port.set_streams(None, None, None); ref.set_streams(None, None, None)
    assert relerr(a[0], b[0]) < 1e-10 and relerr(a[1], b[1]) < 1e-10 and relerr(a[2], b[2]) < 1e-10
    assert relerr(a[3]["eval_train"], b[3]["eval_train"]) < 1e-10
    if not enable_v:
        assert np.array_equal(a[2], v)          # F1: as shipped, V never moves


def test_tables_samplers_metrics_pinned(port, ref):
    rng = np.random.default_rng(10)
    xs = np.concatenate([np.linspace(-7, 7, 4001), rng.normal(0, 2, 1000), [0.0, 5.2003145584, -5.2003145584, -3.0, 5.0]])
    assert relerr([port.pnorm(x) for x in xs], [ref.pnorm(x) for x in xs]) < 1e-12
    assert relerr([port.dpnorm(x) for x in xs], [ref.dpnorm(x) for x in xs]) < 1e-9
    rands = rng.integers(0, 2**31 - 1, 200000).astype(np.int32)
    port.set_streams(None, None, rands); ref.set_streams(None, None, rands)
    a = [port.trnorm_left(x) for x in xs[::7]] + [port.trnorm_right(x) for x in xs[::7]] + [port.random_select(9) for _ in range(50)]
    b = [ref.trnorm_left(x) for x in xs[::7]] + [ref.trnorm_right(x) for x in xs[::7]] + [ref.random_select(9) for _ in range(50)]
    assert a == b and port.stream_pos() == ref.stream_pos()
    port.set_streams(None, None, None); ref.set_streams(None, None, None)
    n = 500
    yh = rng.random(n); ycls = np.where(rng.random(n) < 0.4, 1.0, -1.0); yreg = rng.normal(0, 1, n)
    for m in (O.LL, O.AUC, O.ACC):
        assert port.evaluate(O.CLASSIFICATION, m, yh, ycls) == ref.evaluate(O.CLASSIFICATION, m, yh, ycls)
    for m in (O.RMSE, O.MAE):
        assert port.evaluate(O.REGRESSION, m, yh, yreg) == ref.evaluate(O.REGRESSION, m, yh, yreg)


def test_transpose_and_scales_pinned(port, ref):
    for seed, (n, p, m) in enumerate([(300, 80, 6), (50, 400, 3), (1000, 20, 10)]):
        rowptr, col, val = synth.random_csr(n, p, m, seed=seed)
        a = port.transpose(n, p, rowptr, col, val)
        b = ref.transpose(n, p, rowptr, col, val, use_ref=1)          # the reference's own O(n*p) transpose
        assert all(same(x, y) for x, y in zip(a, b))
        a = port.scales(n, p, rowptr, col, val, np.arange(0, p, 3))
        b = ref.scales(n, p, rowptr, col, val, np.arange(0, p, 3))
        assert same(a[0], b[0]) and same(a[1], b[1]) and same(a[2], b[2], equal_nan=True)
