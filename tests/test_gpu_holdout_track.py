"""Held-out tracking (fmwr_train_holdout_dev / api.fm_train_holdout): at every tracker record, every held-out set is scored on the
device with the record's model, the best record on the first set can be restored into the model, and a patience rule can stop
training.  References use existing calls only: with a trace that keeps snapshots, record r's model is snap_*[r]; loaded with
fmwr_model_set into a model of the precision the loop trains (fp64 for the fp64 shadow of an fp32 ALS/MCMC handle) and scored
with fmwr_predict_dev + fmwr_evaluate_dev, it gives the call's held-out scores bit for bit (same parameters, kernel and metric).

Not tested: the refusal of a context with a communicator and world > 1 (FMWR_ERR_UNSUPPORTED), which needs several GPUs."""
import ctypes as C

import numpy as np
import pytest

from fmwr_b200 import _lib as L
from fmwr_b200 import api as A
from fmwr_b200 import synth
from tests.test_gpu_mcmc_posterior import _layout

K = 4
METRICS = [(L.CLASSIFICATION, L.LL), (L.CLASSIFICATION, L.AUC), (L.CLASSIFICATION, L.ACC), (L.REGRESSION, L.RMSE),
           (L.REGRESSION, L.MAE)]
ONLINE = (L.SGD, L.FTRL, L.TDAP)


def _csr(n, p, seed, empty_rows=False):
    rowptr, col, val = synth.random_csr(n, p, 10, seed=seed, empty_rows=empty_rows)
    return dict(n=n, p=p, rowptr=rowptr, col=col, val=val)


def _labels(task, n, rng):
    return (np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == L.CLASSIFICATION else rng.normal(0, 1, n)).astype(np.float32)


class Case:
    """training data, two labelled held-out sets (the second with empty rows), model config, initial model, solver config and
    the precision the training loop runs in"""

    def __init__(self, ctx, solver, prec, task, metric, ds, es, seed, mode=L.MODE_EXACT, random_step=1, loop_prec=None):
        rng = np.random.default_rng(seed)
        p = ds["p"]
        es2 = _csr(400, p, seed + 1, empty_rows=True)
        y = _labels(task, ds["n"], rng)
        self.ctx, self.solver, self.prec, self.p = ctx, solver, prec, p
        self.loop_prec = prec if loop_prec is None else loop_prec
        self.d = L.Data.from_csr32(ctx, ds["n"], p, ds["rowptr"], ds["col"], ds["val"], y)
        self.evals = [L.Data.from_csr32(ctx, e["n"], p, e["rowptr"], e["col"], e["val"], _labels(task, e["n"], rng)) for e in (es, es2)]
        self.mc = L.ModelCfg(task=task, keep_w0=1, keep_w1=1, k=K, l2_w0=0.01, l1_w1=0.001, l2_w1=0.001, l2_v=0.001)
        self.init = (0.1, rng.normal(0, 0.1, p), rng.normal(0, 0.1, (p, K)))
        als = solver in (L.ALS, L.MCMC)
        self.sc = L.SolverCfg(solver=solver, max_iter=8 if als else (2 * ds["n"] if mode == L.MODE_MINIBATCH else 2 * (ds["n"] - 1) + 5),
                              random_step=random_step, learn_rate=0.05, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0, gamma=1e-4,
                              min_target=float(np.min(y)), max_target=float(np.max(y)), mode=mode, batch_size=64, precision=prec,
                              compat=L.COMPAT_REFERENCE, enable_v=1, step_size=1 if als else (400 if mode == L.MODE_MINIBATCH else 150),
                              metric=metric, convergence=-1.0, seed=7)

    def run(self, holdout=True, select=0, patience=0, max_rec=64):
        m = L.Model(self.ctx, self.mc, self.p, self.prec)
        m.set(*self.init)
        tr = L.TraceBuf(max_rec, self.p, K, snapshots=True)
        scores, best = None, None
        if holdout:
            scores, best = L.train_holdout_dev(self.ctx, m, self.d, self.sc, tr, self.evals, select, patience)
        else:
            L.train_dev(self.ctx, m, self.d, self.sc, tr)
        model = m.get()
        state = m.get_state() if self.solver in ONLINE else None
        m.close()
        return model, state, tr.result(), scores, best

    def rescore(self, t):
        """scores of every snapshot on every held-out set, through fmwr_predict_dev + fmwr_evaluate_dev"""
        if self.mc.task == L.REGRESSION:
            link = L.LINK_CLAMP
        else:
            link = L.LINK_PROBIT_TABLE if self.solver in (L.ALS, L.MCMC) else L.LINK_LOGISTIC
        mr = L.Model(self.ctx, self.mc, self.p, self.loop_prec)
        out = np.zeros((len(self.evals), t["n_rec"]))
        for r in range(t["n_rec"]):
            mr.set(t["snap_w0"][r], t["snap_w"][r], t["snap_v"][r])
            for i, e in enumerate(self.evals):
                L.predict_dev(self.ctx, mr, e, link, self.sc.min_target, self.sc.max_target)
                out[i, r] = L.evaluate_dev(self.ctx, e, self.mc.task, self.sc.metric)
        mr.close()
        return out

    def close(self):
        for h in [self.d] + self.evals:
            h.close()


def _online_case(ctx, solver, prec, task, metric, mode=L.MODE_EXACT, random_step=1):
    n = 3000 if mode == L.MODE_MINIBATCH else 1200
    return Case(ctx, solver, prec, task, metric, _csr(n, 300, 1), _csr(500, 300, 2), solver + task + metric, mode, random_step)


def _als_case(ctx, solver, prec, task, metric, layout):
    ds, es = _layout(layout)
    # the precision policy of train_als.cu: fp32 MCMC classification and data with a column of at most two non-zeros
    # (fields_odd) run on an fp64 shadow, which is what the tracker scores and snapshots
    cnt = np.bincount(ds["col"].astype(np.int64), minlength=ds["p"])
    thin = cnt[cnt > 0].min() <= 2
    shadow = prec == L.F32 and ((solver == L.MCMC and task == L.CLASSIFICATION) or thin)
    return Case(ctx, solver, prec, task, metric, ds, es, 31 + solver + task + metric, loop_prec=L.F64 if shadow else prec)


def _same_model(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


def _snapshot(t, r):
    return t["snap_w0"][r], t["snap_w"][r], t["snap_v"][r]


def _better(s, best, have, cls):
    return not np.isnan(s) and (not have or (s > best if cls else s < best))


def _argbest(scores0, cls):
    best, at = None, -1
    for r, s in enumerate(scores0):
        if _better(s, best, at >= 0, cls):
            best, at = s, r
    return at


def _patience_stop(scores0, cls, patience):
    best, have, since = None, False, 0
    for r, s in enumerate(scores0):
        if _better(s, best, have, cls):
            best, have, since = s, True, 0
        else:
            since += 1
        if since >= patience:
            return r
    return None


@pytest.fixture
def column_kernels(monkeypatch):
    """the column-parallel ALS/MCMC coordinate passes: no atomics, so a run is reproducible bit for bit from its arguments"""
    monkeypatch.setenv("FMWR_ALS_COLUMN", "1")


EXACT_CASES = [(s, p, pipe) + METRICS[i % 5] for i, (s, p, pipe) in
               enumerate((s, p, pipe) for s in ONLINE for p in (L.F64, L.F32) for pipe in ("0", "2"))]
MB_CASES = [(p, rs) + METRICS[(i + 2) % 5] for i, (p, rs) in enumerate((p, rs) for p in (L.F32, L.F64) for rs in (1, 3))]
ALS_CASES = [(s, lay, p) + METRICS[i % 5] for i, (s, lay, p) in
             enumerate((s, lay, p) for s in (L.ALS, L.MCMC) for lay in ("fields", "fields_odd", "fields_sparse", "ragged")
                       for p in (L.F64, L.F32))]


def _check_rescored(c):
    _, _, t, scores, best = c.run()
    assert t["n_rec"] >= 8 and scores.shape == (2, t["n_rec"])
    ref = c.rescore(t)
    assert np.array_equal(scores, ref), (scores, ref)
    assert np.std(scores[0]) > 0
    assert best == _argbest(scores[0], c.mc.task == L.CLASSIFICATION)
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver,prec,pipe,task,metric", EXACT_CASES)
def test_exact_scores_equal_rescored_snapshots(gpu_ctx, monkeypatch, solver, prec, pipe, task, metric):
    """FMWR_EXACT_PIPE: 0 = the CTA-wide kernel, 2 = the pipelined kernel"""
    monkeypatch.setenv("FMWR_EXACT_PIPE", pipe)
    _check_rescored(_online_case(gpu_ctx, solver, prec, task, metric))


@pytest.mark.gpu
@pytest.mark.parametrize("prec,random_step,task,metric", MB_CASES)
def test_minibatch_scores_equal_rescored_snapshots(gpu_ctx, prec, random_step, task, metric):
    _check_rescored(_online_case(gpu_ctx, L.FTRL, prec, task, metric, L.MODE_MINIBATCH, random_step))


@pytest.mark.gpu
@pytest.mark.parametrize("solver,layout,prec,task,metric", ALS_CASES)
def test_als_mcmc_scores_equal_rescored_snapshots(gpu_ctx, solver, layout, prec, task, metric):
    """every layout's default passes (atomics included): the snapshots come from the same call"""
    _check_rescored(_als_case(gpu_ctx, solver, prec, task, metric, layout))


def _assert_untouched(plain, tracked):
    model, state, t = plain[:3]
    model2, state2, t2 = tracked[:3]
    assert _same_model(model2, model)
    if state is not None:
        assert state2["solver"] == state["solver"]
        for key in ("scal", "sw", "sv"):
            assert np.array_equal(state2[key], state[key]), key
    for key in ("eval_train", "rec_index", "snap_w0", "snap_w", "snap_v"):
        assert np.array_equal(t2[key], t[key]), key
    assert (t2["n_rec"], t2["convergent"], t2["iters_done"]) == (t["n_rec"], t["convergent"], t["iters_done"])


@pytest.mark.gpu
@pytest.mark.parametrize("solver,prec,mode", [(L.FTRL, L.F64, L.MODE_EXACT), (L.SGD, L.F32, L.MODE_EXACT), (L.TDAP, L.F64, L.MODE_EXACT),
                                              (L.FTRL, L.F32, L.MODE_MINIBATCH), (L.SGD, L.F64, L.MODE_MINIBATCH)])
def test_online_training_untouched(gpu_ctx, solver, prec, mode):
    """select_best = 0, patience = 0: model, optimizer state and trace are fmwr_train_dev's bit for bit"""
    c = _online_case(gpu_ctx, solver, prec, L.CLASSIFICATION, L.AUC, mode)
    c.sc.convergence = 1e-4                              # the train-score convergence rule keeps its meaning
    _assert_untouched(c.run(holdout=False), c.run())
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["fields", "fields_odd", "fields_sparse", "ragged"])
@pytest.mark.parametrize("prec", [L.F64, L.F32])
@pytest.mark.parametrize("solver,task,metric", [(L.ALS, L.REGRESSION, L.RMSE), (L.MCMC, L.CLASSIFICATION, L.LL)])
def test_als_mcmc_training_untouched(gpu_ctx, column_kernels, solver, task, metric, prec, layout):
    c = _als_case(gpu_ctx, solver, prec, task, metric, layout)
    _assert_untouched(c.run(holdout=False), c.run())
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("solver,layout", [(L.ALS, "fields"), (L.MCMC, "fields"), (L.ALS, "fields_sparse"), (L.MCMC, "fields_sparse")])
def test_als_mcmc_atomic_passes_within_their_noise(gpu_ctx, solver, layout):
    """the fused (fields) and row-major (fields_sparse) passes sum their statistics with atomics, so two runs of even the plain
    call differ in the last bits: these are compared to a tolerance, fp64 (the bit-identity is checked above on the column
    passes)"""
    c = _als_case(gpu_ctx, solver, L.F64, L.REGRESSION, L.RMSE, layout)
    plain, tracked = c.run(holdout=False), c.run()
    for a, b in zip(plain[0], tracked[0]):
        assert np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.maximum(1.0, np.abs(np.asarray(a)))) <= 1e-9
    assert np.allclose(plain[2]["eval_train"], tracked[2]["eval_train"], rtol=1e-9, atol=0)
    assert plain[2]["iters_done"] == tracked[2]["iters_done"] and plain[2]["n_rec"] == tracked[2]["n_rec"]
    c.close()


BEST_CASES = [("exact", L.FTRL, L.F64, L.CLASSIFICATION, L.AUC, None), ("exact", L.SGD, L.F32, L.REGRESSION, L.RMSE, None),
              ("minibatch", L.FTRL, L.F32, L.CLASSIFICATION, L.LL, None), ("als", L.ALS, L.F64, L.REGRESSION, L.MAE, "fields"),
              ("als", L.MCMC, L.F32, L.CLASSIFICATION, L.ACC, "fields_odd")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,solver,prec,task,metric,layout", BEST_CASES)
def test_select_best_restores_the_best_snapshot(gpu_ctx, kind, solver, prec, task, metric, layout):
    """(w0, w, V) equal snapshot best_rec: bit for bit in fp64, and in fp32 because f32 -> f64 -> f32 is exact; on the fp64
    shadow (fields_odd, fp32 handle) w and V are the fp32 rounding of the f64 snapshot and w0 (an f64 scalar in both) is equal.
    The optimizer state is the plain run's (w0, its slot 0, aside)."""
    if kind == "als":
        c = _als_case(gpu_ctx, solver, prec, task, metric, layout)
    else:
        c = _online_case(gpu_ctx, solver, prec, task, metric, L.MODE_MINIBATCH if kind == "minibatch" else L.MODE_EXACT)
    plain = c.run(holdout=False)
    model, state, t, scores, best = c.run(select=1)
    assert best == _argbest(scores[0], task == L.CLASSIFICATION) and 0 <= best < t["n_rec"]
    w0, w, v = _snapshot(t, best)
    if c.loop_prec != prec:
        w, v = w.astype(np.float32).astype(np.float64), v.astype(np.float32).astype(np.float64)
    assert _same_model(model, (w0, w, v))
    if state is not None:
        assert np.array_equal(state["scal"][1:], plain[1]["scal"][1:])
        assert np.array_equal(state["sw"], plain[1]["sw"]) and np.array_equal(state["sv"], plain[1]["sv"])
    if kind != "als":                                    # the default ALS/MCMC passes sum with atomics: no second run to compare
        for key in ("eval_train", "rec_index", "snap_w", "snap_v"):
            assert np.array_equal(t[key], plain[2][key]), key
    c.close()


PATIENCE_CASES = [("exact", L.SGD, L.F64, L.CLASSIFICATION, L.LL), ("minibatch", L.FTRL, L.F32, L.REGRESSION, L.RMSE),
                  ("als", L.ALS, L.F64, L.REGRESSION, L.RMSE)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,solver,prec,task,metric", PATIENCE_CASES)
def test_patience_stops_at_the_predicted_record(gpu_ctx, column_kernels, kind, solver, prec, task, metric):
    """the stop record is predicted from a full-length run's eval[0] curve; the held-out labels are independent of the training
    labels, so the curve stops improving early.  ALS decides the stop at the start of a sweep and does not run that sweep:
    iters_done is the record's sweep index there, the record's sample index + 1 for the online solvers."""
    if kind == "als":
        c = _als_case(gpu_ctx, solver, prec, task, metric, "fields")
    else:
        c = _online_case(gpu_ctx, solver, prec, task, metric, L.MODE_MINIBATCH if kind == "minibatch" else L.MODE_EXACT)
    cls = task == L.CLASSIFICATION
    _, _, full, full_scores, _ = c.run()
    for patience in (1, 2):
        stop = _patience_stop(full_scores[0], cls, patience)
        assert stop is not None and stop < full["n_rec"] - 1, (patience, full_scores[0])
        for select in (0, 1):
            model, _, t, scores, best = c.run(select=select, patience=patience)
            assert t["n_rec"] == stop + 1 and not t["convergent"]
            assert np.array_equal(scores, full_scores[:, :stop + 1])
            at = int(full["rec_index"][stop])
            assert t["iters_done"] == (at if kind == "als" else at + 1) and t["iters_done"] < c.sc.max_iter
            assert best == _argbest(full_scores[0][:stop + 1], cls)
            assert _same_model(model, _snapshot(full, best if select else stop)), (patience, select)
    c.close()


def _raw_call(ctx, m, d, sc, trace, evals, scores, select=0, patience=0, n_eval=None):
    arr = (C.c_void_p * max(len(evals), 1))(*[e.h if e is not None else None for e in evals]) if evals is not None else None
    n = len(evals) if n_eval is None else n_eval
    return L.lib().fmwr_train_holdout_dev(ctx.h, m.h, d.h, C.byref(sc), C.byref(trace.c) if trace is not None else None, arr,
                                          C.c_int32(n), L.ptr(scores), C.c_int32(select), C.c_int32(patience), None)


@pytest.mark.gpu
def test_argument_errors_leave_the_model_untouched(gpu_ctx):
    ctx = gpu_ctx
    c = _online_case(ctx, L.FTRL, L.F64, L.CLASSIFICATION, L.LL)
    d, (e, e2) = c.d, c.evals
    ds = _csr(200, 300, 9)
    unlabelled = L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"])
    nw = _csr(200, 299, 10)
    narrow = L.Data.from_csr32(ctx, nw["n"], nw["p"], nw["rowptr"], nw["col"], nw["val"], np.ones(200, np.float32))
    m = L.Model(ctx, c.mc, c.p, L.F64)
    m.set(*c.init)
    before = m.get()
    tr = L.TraceBuf(64, c.p, K, snapshots=True)
    scores = np.zeros((3, 64))
    no_step = L.SolverCfg.from_buffer_copy(c.sc)
    no_step.step_size = 0
    cases = [(dict(trace=None), 1, "needs a trace"), (dict(sc=no_step), 1, "step_size > 0"),
             (dict(evals=[]), 1, "at least one eval set"), (dict(evals=None, n_eval=1), 1, "at least one eval set"),
             (dict(scores=None), 1, "null eval_scores"), (dict(evals=[e, None]), 1, "null eval data"),
             (dict(evals=[e, unlabelled]), 1, "no labels"), (dict(evals=[e, d]), 1, "training data"),
             (dict(evals=[e, e2, e]), 1, "twice"), (dict(patience=-1), 1, "patience"),
             (dict(evals=[e, narrow]), 3, "number of input's features is not correct")]
    for kw, code, msg in cases:
        args = dict(sc=c.sc, trace=tr, evals=[e, e2], scores=scores, select=1, patience=0)
        args.update(kw)
        rc = _raw_call(ctx, m, d, **args)
        err = L.lib().fmwr_last_error().decode()
        assert rc == code and msg in err, (kw, rc, err)
        assert _same_model(m.get(), before), kw
    for h in (m, unlabelled, narrow):
        h.close()
    c.close()


# ---- host API -------------------------------------------------------------------------------------------------------
def _host_data(seed, n, p=10, labels01=True):
    rng = np.random.default_rng(seed)
    x = rng.normal(0, 1, (n, p)) * (rng.random((n, p)) < 0.6) * np.linspace(0.5, 20.0, p)   # column scales z-scoring changes
    y = (x @ np.random.default_rng(99).normal(0, 1, p) + 3.0 * rng.normal(0, 1, n) > 0).astype(np.float64)
    return A.fm_matrix(x, y if labels01 else 2 * y - 1)


def _control(step_size=40, metric="AUC"):
    return [A.model_control("CLASSIFICATION", factor_number=3), A.solver_control(max_iter=700, solver=A.FTRL_solver()),
            A.track_control(step_size=step_size, evaluate_metric=metric)]


def test_fm_train_holdout_argument_errors():
    """raised before any GPU work"""
    data, new = _host_data(1, 60), _host_data(2, 30)
    with pytest.raises(ValueError, match="step_size > 0"):
        A.fm_train_holdout(data, new, control=_control(step_size=-1))
    with pytest.raises(ValueError, match="step_size > 0"):
        A.fm_train_holdout(data, new, control=_control(step_size=0))
    with pytest.raises(ValueError, match="fm.matrix"):
        A.fm_train_holdout(data, [dict(new)], control=_control())
    with pytest.raises(ValueError, match="fm.matrix"):
        A.fm_train_holdout(data, [], control=_control())
    with pytest.raises(ValueError, match="no labels in newdata"):
        A.fm_train_holdout(data, A.fm_matrix(np.eye(10)), control=_control())
    with pytest.raises(ValueError, match="training data"):
        A.fm_train_holdout(data, data, control=_control())
    with pytest.raises(ValueError, match="twice"):
        A.fm_train_holdout(data, [new, new], control=_control())
    with pytest.raises(ValueError, match="select"):
        A.fm_train_holdout(data, new, control=_control(), select="first")
    with pytest.raises(ValueError, match="patience"):
        A.fm_train_holdout(data, new, control=_control(), patience=-1)
    # a trace without model snapshots (snapshots=False) cannot be tracked or selected from
    fit = A.FM(Model={}, Scales={}, Trace={"trace": [np.arange(3.0)], "evaluation.train": np.zeros(3)})
    with pytest.raises(ValueError, match="no model snapshots"):
        A.fm_track(fit, new)
    with pytest.raises(ValueError, match="no model snapshots"):
        A.fm_select(fit, best_iter=1)


@pytest.mark.gpu
def test_fm_train_holdout_equals_the_track_and_select_workflow(gpu_ctx):
    data, new, new2 = _host_data(3, 300), _host_data(4, 200), _host_data(5, 150)
    fit = A.fm_train(data, True, _control())
    tk, tk2 = A.fm_track(fit, new), A.fm_track(fit, new2)
    ho = A.fm_train_holdout(data, [new, new2], True, _control(), select="best")
    tr = ho["Trace"]
    assert np.array_equal(tr["evaluation.test"][0], tk["test"]) and np.array_equal(tr["evaluation.test"][1], tk2["test"])
    assert np.array_equal(tr["trace"][0], fit["Trace"]["trace"][0]) and np.array_equal(tr["evaluation.train"], fit["Trace"]["evaluation.train"])
    assert len(tk["test"]) >= 10 and np.std(tk["test"]) > 0
    best = tr["best.index"]
    assert best == int(np.argmax(tk["test"]))                                   # AUC: higher is better, first arg-best
    sel = A.fm_select(fit, best_iter=best)
    for key in ("w0", "w", "v"):
        assert np.array_equal(ho["Model"][key], sel["Model"][key]), key
    assert np.array_equal(ho["Scales"]["mean"], fit["Scales"]["mean"])
    # last model by default; 0/1 and -1/+1 labels score alike; no snapshots: the curves only, and track / select refuse
    last = A.fm_train_holdout(data, [_host_data(4, 200, labels01=False)], True, _control(), snapshots=False)
    for key in ("w0", "w", "v"):
        assert np.array_equal(last["Model"][key], fit["Model"][key]), key
    assert np.array_equal(last["Trace"]["evaluation.test"][0], tk["test"]) and last["Trace"]["best.index"] == best
    assert len(last["Trace"]["trace"]) == 1
    with pytest.raises(ValueError, match="no model snapshots"):
        A.fm_track(last, new)
    with pytest.raises(ValueError, match="no model snapshots"):
        A.fm_select(last, best_iter=best)
    # newdata is z-scored with the training scales: scoring it unscaled gives another curve
    raw = A.fm_track(fit, new, normalize=False)
    assert not np.array_equal(raw["test"], tk["test"])
