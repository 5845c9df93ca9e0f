"""MCMC posterior mean (fmwr_train_posterior_dev / api.fm_posterior): the average of the predict.FM predictions of the draws
after a burn-in, formed on the device while the sampler runs.  References use existing calls only: the tracker's per-sweep
snapshots (step_size = 1) are draws 0 .. S-1, the returned model is draw S, and fmwr_predict_dev with the MCMC link scores each
of them.  Tolerances: 1e-12 relative for fp64, 1e-5 (the prediction tolerance) for fp32.  That the chain itself is untouched is
checked bit for bit on the column-parallel coordinate passes, the ones that sum without atomics."""
import warnings

import numpy as np
import pytest

from fmwr_b200 import _lib as L
from fmwr_b200 import api as A
from fmwr_b200 import synth
from tests.util import relerr

S, BURN, K = 8, 3, 4


def _fields(n, fields, seed, drop_every=0):
    rowptr, col, val, p = synth.fields_csr(n, fields, None, 1, seed)
    if drop_every:
        # field-structured but some rows miss a field: few phases, rows no longer implicit (row-major unfused passes)
        keep = np.ones(col.size, bool)
        keep[np.arange(0, col.size, drop_every)] = False
        cnt = np.add.reduceat(keep.astype(np.int64), rowptr[:-1].astype(np.int64))
        rowptr, col, val = np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint32), col[keep], val[keep]
    return dict(n=n, p=p, rowptr=rowptr, col=col, val=val)


def _layout(name):
    """(training set, eval set of the same width from another seed): the layouts of test_als_matches_oracle"""
    if name == "fields":
        return _fields(3000, [40, 25, 8], 5), _fields(700, [40, 25, 8], 15)               # dense fused passes
    if name == "fields_odd":
        return _fields(3001, [40, 2500, 8], 6), _fields(900, [40, 2500, 8], 16)           # permuted rows; fp32 runs on the fp64 shadow
    if name == "fields_sparse":
        return _fields(2000, [30, 20, 10], 7, 7), _fields(500, [30, 20, 10], 17, 7)       # row-major passes
    tr = synth.random_csr(600, 70, 6, seed=5, empty_rows=True)                          # general CSR, many small phases
    ev = synth.random_csr(300, 70, 6, seed=25, empty_rows=True)
    return (dict(n=600, p=70, rowptr=tr[0], col=tr[1], val=tr[2]), dict(n=300, p=70, rowptr=ev[0], col=ev[1], val=ev[2]))


def _data(ctx, ds, y=None):
    return L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y)


def _solver(task, y, sweeps=S, step_size=1, seed=7):
    return L.SolverCfg(solver=L.MCMC, max_iter=sweeps, random_step=1, min_target=float(np.min(y)), max_target=float(np.max(y)),
                       mode=L.MODE_EXACT, precision=L.F64, compat=L.COMPAT_REFERENCE, enable_v=1, step_size=step_size,
                       metric=L.LL if task == L.CLASSIFICATION else L.RMSE, convergence=1e-4, seed=seed)


def _labels(task, n, rng):
    return (np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == L.CLASSIFICATION else rng.normal(0, 1, n)).astype(np.float32)


def _link(task):
    return L.LINK_PROBIT_TABLE if task == L.CLASSIFICATION else L.LINK_CLAMP


def _case(ctx, task, prec, layout):
    rng = np.random.default_rng(11)
    ds, es = _layout(layout)
    y = _labels(task, ds["n"], rng)
    init = (0.1, rng.normal(0, 0.1, ds["p"]), rng.normal(0, 0.1, (ds["p"], K)))
    sc = _solver(task, y)
    sc.precision = prec
    return _data(ctx, ds, y), _data(ctx, es), L.ModelCfg(task=task, keep_w0=1, keep_w1=1, k=K, l2_w0=0.1), init, sc


def _chain(ctx, mc, init, d, sc, prec, post=None):
    """S sweeps from init, every draw but the last snapshotted by the tracker: (final model, trace)"""
    m = L.Model(ctx, mc, d.shape()[1], prec)
    m.set(*init)
    tr = L.TraceBuf(S + 2, m.p, K, snapshots=True)
    if post is None:
        L.train_dev(ctx, m, d, sc, tr)
    else:
        L.train_posterior_dev(ctx, m, d, sc, BURN, post, tr)
    out = m.get(), tr.result()
    m.close()
    assert list(out[1]["rec_index"]) == list(range(S))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["fields", "fields_odd", "fields_sparse", "ragged"])
@pytest.mark.parametrize("prec", [L.F64, L.F32])
@pytest.mark.parametrize("task", [L.CLASSIFICATION, L.REGRESSION])
def test_posterior_equals_mean_of_tracked_draws(gpu_ctx, task, prec, layout):
    """the call's own tracker snapshots are draws 0 .. S-1 and its returned model is draw S: predicting each averaged one and
    summing on the host in draw order gives the mean the call left on the training and on the eval handle.  (The default
    coordinate passes sum their statistics with atomics, so two calls are two chains that differ in the last bits: the reference
    comes from the same call; test_posterior_leaves_the_chain_untouched compares against a plain call bit for bit.)"""
    ctx = gpu_ctx
    d, e, mc, init, sc = _case(ctx, task, prec, layout)
    final, t = _chain(ctx, mc, init, d, sc, prec, post=[e])
    got_d, got_e = L.predict_fetch(ctx, d), L.predict_fetch(ctx, e)
    mr = L.Model(ctx, mc, d.shape()[1], prec)
    acc_d, acc_e = np.zeros(d.shape()[0]), np.zeros(e.shape()[0])
    for draw in range(BURN + 1, S + 1):
        mr.set(*(final if draw == S else (t["snap_w0"][draw], t["snap_w"][draw], t["snap_v"][draw])))
        for dd, acc in ((d, acc_d), (e, acc_e)):
            L.predict_dev(ctx, mr, dd, _link(task), sc.min_target, sc.max_target)
            acc += L.predict_fetch(ctx, dd)
    ref_d, ref_e = acc_d / (S - BURN), acc_e / (S - BURN)
    tol = 1e-12 if prec == L.F64 else 1e-5
    assert relerr(got_d, ref_d) <= tol and relerr(got_e, ref_e) <= tol, (relerr(got_d, ref_d), relerr(got_e, ref_e))
    assert np.std(got_d) > 0 and np.std(got_e) > 0
    for h in (mr, d, e):
        h.close()


@pytest.fixture
def column_kernels():
    """the column-parallel coordinate passes: no atomics, so a chain is reproducible bit for bit from its arguments"""
    import os
    os.environ["FMWR_ALS_COLUMN"] = "1"
    yield
    del os.environ["FMWR_ALS_COLUMN"]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["fields", "fields_odd", "fields_sparse", "ragged"])
@pytest.mark.parametrize("prec", [L.F64, L.F32])
@pytest.mark.parametrize("task", [L.CLASSIFICATION, L.REGRESSION])
def test_posterior_leaves_the_chain_untouched(gpu_ctx, column_kernels, task, prec, layout):
    """final model and trace (scores, every snapshotted draw) bit-identical to fmwr_train_dev with the same arguments,
    including the fp64 shadow an fp32 handle runs on (fields_odd, classification)"""
    ctx = gpu_ctx
    d, e, mc, init, sc = _case(ctx, task, prec, layout)
    final, t = _chain(ctx, mc, init, d, sc, prec)
    final2, t2 = _chain(ctx, mc, init, d, sc, prec, post=[e])
    assert final2[0] == final[0] and np.array_equal(final2[1], final[1]) and np.array_equal(final2[2], final[2])
    for key in ("eval_train", "rec_index", "snap_w0", "snap_w", "snap_v"):
        assert np.array_equal(t2[key], t[key]), key
    assert t2["n_rec"] == t["n_rec"] and t2["iters_done"] == t["iters_done"]
    d.close(); e.close()


@pytest.mark.gpu
def test_burn_in_edges(gpu_ctx):
    ctx = gpu_ctx
    rng = np.random.default_rng(12)
    ds, es = _layout("fields")
    n, p = ds["n"], ds["p"]
    y = _labels(L.REGRESSION, n, rng)
    mc = L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=K)
    sc = _solver(L.REGRESSION, y, step_size=-1)
    w, v = rng.normal(0, 0.1, p), rng.normal(0, 0.1, (p, K))
    d, e = _data(ctx, ds, y), _data(ctx, es)
    # burn_in = S - 1: the mean is the last draw alone
    m = L.Model(ctx, mc, p, L.F64)
    m.set(0.0, w, v)
    L.train_posterior_dev(ctx, m, d, sc, S - 1, [e])
    got_d, got_e = L.predict_fetch(ctx, d), L.predict_fetch(ctx, e)
    rmse = L.evaluate_dev(ctx, d, L.REGRESSION, L.RMSE)          # scores the mean the handle holds
    assert abs(rmse - float(np.sqrt(np.mean((got_d - y.astype(np.float64)) ** 2)))) <= 1e-12 * max(1.0, rmse)
    L.predict_dev(ctx, m, e, L.LINK_CLAMP, sc.min_target, sc.max_target)
    assert np.array_equal(got_e, L.predict_fetch(ctx, e))
    L.predict_dev(ctx, m, d, L.LINK_CLAMP, sc.min_target, sc.max_target)
    assert relerr(got_d, L.predict_fetch(ctx, d)) <= 1e-12
    # burn_in = 0: every draw 1 .. S, no eval set, no trace
    m.set(0.0, w, v)
    L.train_posterior_dev(ctx, m, d, sc, 0)
    all_d = L.predict_fetch(ctx, d)
    assert all_d.shape == (n,) and np.all(np.isfinite(all_d)) and not np.array_equal(all_d, got_d)
    for h in (m, d, e):
        h.close()


@pytest.mark.gpu
def test_abi_argument_errors_leave_the_model_untouched(gpu_ctx):
    ctx = gpu_ctx
    rng = np.random.default_rng(13)
    ds, es = _layout("fields")
    p = ds["p"]
    y = _labels(L.REGRESSION, ds["n"], rng)
    mc = L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=K)
    w, v = rng.normal(0, 0.1, p), rng.normal(0, 0.1, (p, K))
    d, e, e2 = _data(ctx, ds, y), _data(ctx, es), _data(ctx, _fields(300, [40, 25, 8], 18))
    narrow = _data(ctx, _fields(300, [40, 25, 7], 19))
    m = L.Model(ctx, mc, p, L.F64)
    m.set(0.25, w, v)
    before = m.get()
    sc = _solver(L.REGRESSION, y, step_size=-1)
    als = _solver(L.REGRESSION, y, step_size=-1)
    als.solver = L.ALS
    cases = [(als, BURN, [e], L.FmwrError, 1, "needs the MCMC solver"), (sc, -1, [e], L.FmwrError, 1, "burn_in"),
             (sc, S, [e], L.FmwrError, 1, "burn_in"), (sc, BURN, [None], L.FmwrError, 1, "null"),
             (sc, BURN, [e, d], L.FmwrError, 1, "training data"), (sc, BURN, [e, e2, e], L.FmwrError, 1, "twice"),
             (sc, BURN, [e, narrow], L.FmwrError, 3, "number of input's features is not correct")]
    for cfg, burn, evals, exc, code, msg in cases:
        with pytest.raises(exc) as ei:
            L.train_posterior_dev(ctx, m, d, cfg, burn, evals)
        assert ei.value.code == code and msg in ei.value.msg, (code, ei.value.code, ei.value.msg)
        after = m.get()
        assert after[0] == before[0] and np.array_equal(after[1], before[1]) and np.array_equal(after[2], before[2])
    for h in (m, d, e, e2, narrow):
        h.close()


# ---- host API -------------------------------------------------------------------------------------------------------
def _host_data(seed, n, p=12):
    rng = np.random.default_rng(seed)
    x = rng.normal(0, 1, (n, p)) * (rng.random((n, p)) < 0.5)
    y = x @ rng.normal(0, 1, p) + 0.3 * rng.normal(0, 1, n)
    return A.fm_matrix(x, y)


def _mcmc_control(max_iter=S, step_size=-1, solver=None):
    return [A.model_control("REGRESSION", factor_number=3), A.solver_control(max_iter=max_iter, solver=solver or A.MCMC_solver()),
            A.track_control(step_size=step_size, evaluate_metric="RMSE")]


def test_fm_posterior_argument_errors():
    data, new = _host_data(1, 50), _host_data(2, 20)
    with pytest.raises(ValueError, match="needs the MCMC solver"):
        A.fm_posterior(data, [new], burn_in=1, control=_mcmc_control(solver=A.ALS_solver()))
    with pytest.raises(ValueError, match="needs the MCMC solver"):
        A.fm_posterior(data, [new], burn_in=1, control=[A.model_control("REGRESSION")])    # fm.train's default solver is TDAP
    for burn in (-1, S, S + 5, 1.5):
        with pytest.raises(ValueError, match="burn_in"):
            A.fm_posterior(data, [new], burn_in=burn, control=_mcmc_control())
    with pytest.raises(ValueError, match="fm.matrix"):
        A.fm_posterior(data, [dict(new)], burn_in=1, control=_mcmc_control())
    with pytest.raises(ValueError, match="training data"):
        A.fm_posterior(data, [data], burn_in=1, control=_mcmc_control())
    with pytest.raises(ValueError, match="twice"):
        A.fm_posterior(data, [new, new], burn_in=1, control=_mcmc_control())
    with pytest.raises(ValueError, match="there are no labels"):
        A.fm_posterior(A.fm_matrix(np.eye(3)), burn_in=1, control=_mcmc_control())


@pytest.mark.gpu
def test_fm_posterior_shape_error():
    data = _host_data(1, 50)
    with pytest.raises(L.FmwrError) as ei:
        A.fm_posterior(data, [_host_data(2, 20, p=11)], burn_in=1, control=_mcmc_control())
    assert ei.value.code == 3


@pytest.mark.gpu
def test_fm_posterior_equals_public_composition(gpu_ctx, column_kernels):
    """on the reproducible column passes: the fit is fm_train's, and the newdata mean composes predict and fm_select"""
    data, new = _host_data(3, 400), _host_data(4, 150)
    saved = A.options()["FM.enable_v"]
    A.options(**{"FM.enable_v": True})
    try:
        fit = A.fm_train(data, True, _mcmc_control())
        post = A.fm_posterior(data, [new], burn_in=BURN, normalize=True, control=_mcmc_control())
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            tracked = A.fm_train(data, True, _mcmc_control(step_size=1))
        ref = np.zeros(new.nrow())
        for i in range(BURN + 1, S):
            ref += A.predict(A.fm_select(tracked, best_iter=i), new)
        ref += A.predict(tracked, new)
        ref /= S - BURN
    finally:
        A.options(**{"FM.enable_v": saved})
    for key in ("w0", "w", "v"):
        assert np.array_equal(post["fit"]["Model"][key], fit["Model"][key]), key
        assert np.array_equal(tracked["Model"][key], fit["Model"][key]), key
    assert np.array_equal(post["fit"]["Scales"]["mean"], fit["Scales"]["mean"])
    assert post["train"].shape == (data.nrow(),) and len(post["newdata"]) == 1
    assert relerr(post["newdata"][0], ref) <= 1e-12, relerr(post["newdata"][0], ref)


@pytest.mark.gpu
def test_posterior_mean_beats_the_last_draw(gpu_ctx):
    """the planted-model shape of test_mcmc_native_rng_posterior_mean, scored on held-out rows of the same planted model"""
    ctx = gpu_ctx
    rng = np.random.default_rng(4)
    fields, k, sweeps, burn = [60, 40], 4, 80, 30
    tr, te = _fields(6000, fields, 11), _fields(3000, fields, 21)
    for ds in (tr, te):
        ds["val"] = np.ones_like(ds["val"])
        score = synth.planted_scores_fast(ds["rowptr"], ds["col"], ds["val"], ds["p"], k=4, seed=12, scale=0.5)
        ds["y"] = (score + 0.1 * rng.standard_normal(ds["n"])).astype(np.float32)
    p = tr["p"]
    d, e = _data(ctx, tr, tr["y"]), _data(ctx, te)
    m = L.Model(ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=k), p, L.F32)
    m.set(0.0, np.zeros(p), rng.normal(0, 0.1, (p, k)))
    sc = _solver(L.REGRESSION, tr["y"], sweeps=sweeps, step_size=-1, seed=1)
    sc.precision = L.F32
    L.train_posterior_dev(ctx, m, d, sc, burn, [e])
    mean = L.predict_fetch(ctx, e)
    L.predict_dev(ctx, m, e, L.LINK_CLAMP, sc.min_target, sc.max_target)
    last = L.predict_fetch(ctx, e)
    rmse_mean = float(np.sqrt(np.mean((mean - te["y"]) ** 2)))
    rmse_last = float(np.sqrt(np.mean((last - te["y"]) ** 2)))
    print("held-out RMSE: posterior mean of %d draws %.5f, last draw %.5f, sd(y) %.3f" % (sweeps - burn, rmse_mean, rmse_last, float(np.std(te["y"]))))
    assert rmse_mean <= rmse_last and rmse_mean < 0.2 * float(np.std(te["y"]))
    for h in (m, d, e):
        h.close()
