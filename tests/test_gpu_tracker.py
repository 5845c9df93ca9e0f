"""The tracker's schedule and trace (reference src/core/Tracker.h): which samples or sweeps are recorded, where the convergence
rule stops training, how the MAX_REC storage limit and an empty epoch leave the trace.  Exact mode and ALS/MCMC are held to the
plain-C restatement (port); minibatch mode, which the reference does not have, to a Python restatement of its crossing rule.

convergence = 1e30 passes every guarded test: the rule is applied from the third record on, so an SGD/FTRL/TDAP run stops at its
fifth record.  convergence = -1 passes none."""
import numpy as np
import pytest

from oracle import oracle as O
from fmwr_b200 import _lib as L
from fmwr_b200 import synth
from tests.util import relerr

pytestmark = pytest.mark.gpu

N, P, K = 100, 40, 3
CONVERGENCE = [-1.0, 1e30]


def _data(task=L.CLASSIFICATION, seed=0):
    rng = np.random.default_rng(seed)
    rowptr, col, val = synth.random_csr(N, P, 8, seed=seed + 1)
    y = (np.where(rng.random(N) < 0.5, 1.0, -1.0) if task == L.CLASSIFICATION else rng.normal(0, 1, N)).astype(np.float32)
    init = (0.1, rng.normal(0, 0.1, P), rng.normal(0, 0.1, (P, K)))
    return dict(n=N, p=P, rowptr=rowptr, col=col, val=val, y=y, init=init, task=task)


def _cfgs(ds, solver, mode, step, max_iter, convergence, prec=L.F64, batch=1, random_step=1):
    y = ds["y"]
    cls = ds["task"] == L.CLASSIFICATION
    mc = L.ModelCfg(task=ds["task"], keep_w0=1, keep_w1=1, k=K)
    sc = L.SolverCfg(solver=solver, max_iter=max_iter, random_step=random_step, learn_rate=0.05, alpha_w=0.1, alpha_v=0.1,
                     beta_w=1.0, beta_v=1.0, gamma=1e-4, min_target=float(y.min()), max_target=float(y.max()), mode=mode,
                     batch_size=batch, precision=prec, compat=L.COMPAT_REFERENCE, enable_v=1, step_size=step,
                     metric=L.LL if cls else L.RMSE, convergence=convergence, seed=3)
    return mc, sc


def _train(ctx, ds, mc, sc, prec=L.F64, tr=None, data=None):
    d = data if data is not None else L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], ds["y"])
    m = L.Model(ctx, mc, ds["p"], prec)
    m.set(*ds["init"])
    tr = tr or L.TraceBuf(200)
    L.train_dev(ctx, m, d, sc, tr)
    m.close()
    if data is None:
        d.close()
    return tr.result()


def _port(port, ds, solver, step, max_iter, convergence, max_rec=200):
    y = ds["y"]
    cls = ds["task"] == L.CLASSIFICATION
    cfg = O.make_cfg(task=O.CLASSIFICATION if cls else O.REGRESSION, solver=solver, k=K, max_iter=max_iter, learn_rate=0.05,
                     enable_v=1, min_target=float(y.min()), max_target=float(y.max()), step_size=step,
                     metric=O.LL if cls else O.RMSE, convergence=convergence)
    w0, w, v = ds["init"]
    return port.train(cfg, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y, w0, w, v, max_rec=max_rec)[3]


def _minibatch_schedule(n_rows, row0, batch, step, max_iter, convergence):
    """minibatch mode's records: after every batch whose end crosses the next multiple of step (and after the last batch);
    (record indices, convergent, samples done)"""
    n_batches = -(-(n_rows - row0) // batch)
    it, next_track, recs, conv_times = 0, 0, [], 0
    while it < max_iter:
        for b in range(n_batches):
            if it >= max_iter:
                break
            rb = row0 + b * batch
            it += min(batch, n_rows - rb, max_iter - it)
            if step > 0 and (it > next_track or it >= max_iter):
                next_track = (it // step + 1) * step
                recs.append(it - 1)
                conv_times = conv_times + 1 if (convergence > 0 and len(recs) >= 3) else 0
                if conv_times >= 3:
                    return recs, True, it
    return recs, False, it


MAX_ITER = 60


@pytest.mark.parametrize("step", [1, 7, MAX_ITER - 1])
@pytest.mark.parametrize("convergence", CONVERGENCE)
def test_exact_schedule_matches_port(gpu_ctx, port, step, convergence):
    ds = _data()
    mc, sc = _cfgs(ds, L.FTRL, L.MODE_EXACT, step, MAX_ITER, convergence)
    got = _train(gpu_ctx, ds, mc, sc)
    want = _port(port, ds, O.FTRL, step, MAX_ITER, convergence)
    assert got["n_rec"] == want["n_rec"] and np.array_equal(got["rec_index"], want["rec_index"])
    assert got["convergent"] == want["convergent"] and got["iters_done"] == want["iters_done"]
    assert relerr(got["eval_train"], want["eval_train"]) < 1e-9
    if convergence > 0 and step < MAX_ITER - 1:
        assert got["n_rec"] == 5 and got["convergent"] and got["iters_done"] == step * 4 + 1
    else:
        assert not got["convergent"] and got["iters_done"] == MAX_ITER


MB_SHAPES = [(1, 1, 30), (16, 40, 250), (64, 10, 400), (10, 1000, 120)]     # (batch_size, step_size, max_iter)


@pytest.mark.parametrize("batch,step,max_iter", MB_SHAPES)
@pytest.mark.parametrize("convergence", CONVERGENCE)
def test_minibatch_schedule(gpu_ctx, batch, step, max_iter, convergence):
    ds = _data()
    mc, sc = _cfgs(ds, L.FTRL, L.MODE_MINIBATCH, step, max_iter, convergence, batch=batch)
    got = _train(gpu_ctx, ds, mc, sc)
    recs, convergent, done = _minibatch_schedule(N, 1, batch, step, max_iter, convergence)
    assert got["n_rec"] == len(recs) and np.array_equal(got["rec_index"], recs)
    assert got["convergent"] == convergent and got["iters_done"] == done


def test_minibatch_random_step_scores_the_full_data(gpu_ctx):
    """random_step > 1 trains on the visited rows, gathered in visit order, and the tracker scores the full training data"""
    ds = _data()
    batch, step, max_iter = 16, 40, 250
    mc, sc = _cfgs(ds, L.FTRL, L.MODE_MINIBATCH, step, max_iter, -1.0, batch=batch, random_step=3)
    d = L.Data.from_csr32(gpu_ctx, N, P, ds["rowptr"], ds["col"], ds["val"], ds["y"])
    got = _train(gpu_ctx, ds, mc, sc, tr=L.TraceBuf(200, P, K, snapshots=True), data=d)
    recs, convergent, done = _minibatch_schedule(max_iter, 0, batch, step, max_iter, -1.0)
    assert got["n_rec"] == len(recs) and np.array_equal(got["rec_index"], recs)
    assert got["convergent"] == convergent and got["iters_done"] == done
    m = L.Model(gpu_ctx, mc, P, L.F64)
    for r in range(got["n_rec"]):
        m.set(got["snap_w0"][r], got["snap_w"][r], got["snap_v"][r])
        L.predict_dev(gpu_ctx, m, d, L.LINK_LOGISTIC, sc.min_target, sc.max_target)
        assert L.evaluate_dev(gpu_ctx, d, mc.task, sc.metric) == got["eval_train"][r], r
    m.close(); d.close()


@pytest.mark.parametrize("solver,task,prec", [(L.ALS, L.REGRESSION, L.F64), (L.MCMC, L.REGRESSION, L.F64),
                                              (L.MCMC, L.CLASSIFICATION, L.F32)])
@pytest.mark.parametrize("step", [1, 3])
def test_als_mcmc_schedule_matches_port(gpu_ctx, port, solver, task, prec, step):
    """a record at the start of every step-th sweep and of the last one; ALS/MCMC never converge (fp32 MCMC classification
    runs on the fp64 shadow)"""
    ds = _data(task, seed=4)
    sweeps = 7
    mc, sc = _cfgs(ds, solver, L.MODE_EXACT, step, sweeps, 1e30, prec=prec)
    got = _train(gpu_ctx, ds, mc, sc, prec=prec)
    want = _port(port, ds, O.ALS if solver == L.ALS else O.MCMC, step, sweeps, 1e30)
    assert got["n_rec"] == want["n_rec"] and np.array_equal(got["rec_index"], want["rec_index"])
    assert not got["convergent"] and got["iters_done"] == sweeps


def test_storage_limit(gpu_ctx, port):
    """records past max_rec still count for the schedule but are not stored: n_rec reads max_rec"""
    ds = _data()
    mc, sc = _cfgs(ds, L.FTRL, L.MODE_EXACT, 7, MAX_ITER, -1.0)
    got = _train(gpu_ctx, ds, mc, sc, tr=L.TraceBuf(3))
    want = _port(port, ds, O.FTRL, 7, MAX_ITER, -1.0)
    assert want["n_rec"] > 3 and got["n_rec"] == 3 and np.array_equal(got["rec_index"], want["rec_index"][:3])
    assert got["iters_done"] == MAX_ITER
    mc, sc = _cfgs(ds, L.FTRL, L.MODE_MINIBATCH, 10, 150, -1.0, batch=64)
    got = _train(gpu_ctx, ds, mc, sc, tr=L.TraceBuf(2))
    recs, _, done = _minibatch_schedule(N, 1, 64, 10, 150, -1.0)
    assert len(recs) > 2 and got["n_rec"] == 2 and np.array_equal(got["rec_index"], recs[:2]) and got["iters_done"] == done


@pytest.mark.parametrize("mode", [L.MODE_EXACT, L.MODE_MINIBATCH])
def test_empty_epoch_clears_a_used_trace(gpu_ctx, mode):
    """one row under COMPAT_SKIP_ROW0: the epoch is empty and the trace of an earlier call must not show through"""
    ds = _data()
    tr = L.TraceBuf(200)
    mc, sc = _cfgs(ds, L.FTRL, mode, 1, MAX_ITER, 1e30, batch=1)
    before = _train(gpu_ctx, ds, mc, sc, tr=tr)
    assert before["n_rec"] > 0 and before["convergent"] and before["iters_done"] > 0
    one = dict(ds, n=1, rowptr=np.array([0, 2], np.uint32), col=np.array([0, 1], np.uint32), val=np.ones(2, np.float32),
               y=np.ones(1, np.float32))
    after = _train(gpu_ctx, one, mc, sc, tr=tr)
    assert (after["n_rec"], after["convergent"], after["iters_done"]) == (0, False, 0)
