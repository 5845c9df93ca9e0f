"""Host-side mirror of FMwR's R interface on top of the C ABI (include/fmwr_b200.h).

The reference's host language is R, which this image does not have; this module restates the R layer
(R/fm_matrix.R, fm_control.R, fm_solver_control.R, fm_track_control.R, fm_train.R, fm_predict.R,
fm_update.R, fm_track.R, fm_select.R, fm_set_threads.R) and the list (un)packing of src/FM.cpp with the
same names (dots become underscores), argument meaning, defaults, coercions and error messages, so the
parity tests read like the reference's own examples.  All numerics go through libfmwr_b200.so.

Engine options ride on `options()` exactly as the survey proposes for R (`options(FM.mode=...)`), so the
function signatures stay drop-in:
    FM.mode      "exact" (batch = 1, reference order; default) | "minibatch"
    FM.batch     minibatch rows (default 65536)
    FM.precision "auto" (default): f64 wherever the result is held to the reference's -- exact mode (batch = 1), ALS, MCMC -- and f32 in
                 the throughput (minibatch) mode | "f32" | "f64".  The reference computes in fp64 throughout; f32 is an explicit
                 throughput opt-in (parameters within 1e-4 for SGD / FTRL, looser for TDAP: tests/test_gpu_exact.py)
    FM.cache     True (default): the device copy of an fm.matrix lives in a slot of that object, so fm.train -> predict -> fm.update ->
                 fm.track upload X once (SURVEY 8f-3); False: upload per call like the reference's deep copy (src/FM.cpp:31-34)
    FM.compat    "reference" (default; reproduces SURVEY F5/F6/F7) | "fixed"
    FM.enable_v  ALS/MCMC: run the V block the shipped update_all comments out (default False = as shipped)
    FM.device    CUDA ordinal (default 0)
    FM.seed      seed of the V initialisation / native MCMC RNG (stands in for set.seed())
"""
import contextlib
import warnings

import numpy as np

from . import _lib as L

_OPTIONS = {"FM.threads": 1, "FM.mode": "exact", "FM.batch": 65536, "FM.precision": "auto", "FM.cache": True, "FM.compat": "reference",
            "FM.enable_v": False, "FM.device": 0, "FM.seed": 1,
            # engine extension (SURVEY 8f-4): keep the optimizer state (FTRL z/n, TDAP u/nu/delta/h, SGD-L1 q) in the FM object
            # and continue from it in fm.update; False = the reference's behaviour (state dropped, FTRL_Learner.h:48-56)
            "FM.keep_state": False}
_CTX = {}


def options(**kw):
    """options(FM.mode="minibatch") is spelled options(**{"FM.mode": "minibatch"}) or options(FM_mode=...)"""
    for k, v in kw.items():
        key = k.replace("_", ".", 1) if k.startswith("FM_") else k
        if key not in _OPTIONS:
            raise KeyError("unknown option " + key)
        _OPTIONS[key] = v
    return dict(_OPTIONS)


def get_option(name, default=None):
    return _OPTIONS.get(name, default)


def fm_set_threads(nthreads=None):
    """R/fm_set_threads.R:8-17 (kept for signature compatibility; the engine ignores the thread count)"""
    if nthreads is None:
        nthreads = 1
    _OPTIONS["FM.threads"] = int(nthreads)


def fm_get_threads():
    return _OPTIONS["FM.threads"]


def _ctx():
    dev = int(_OPTIONS["FM.device"])
    if dev not in _CTX:
        _CTX[dev] = L.Context(dev)
    return _CTX[dev]


# ---------------------------------------------------------------------------------------------- fm.matrix
class FmMatrix(dict):
    """class "fm.matrix": list(features = list(value, col_idx, row_size, dim, size; attr feature_names, transposed), labels)"""

    def nrow(self):
        return int(self["features"]["dim"][0])

    def ncol(self):
        return int(self["features"]["dim"][1])


def fm_matrix(x, y=None, feature_names=None):
    """R/fm_matrix.R:13-93 -- dense matrix / scipy sparse -> row-compressed lists with 0-based ascending col_idx"""
    try:
        import scipy.sparse as sp
    except Exception:  # pragma: no cover
        sp = None
    if sp is not None and sp.issparse(x):
        m = x.tocsr()
        m.sort_indices()
        m.sum_duplicates()
        value = np.asarray(m.data, np.float64)
        col_idx = np.asarray(m.indices, np.int32)
        row_size = np.diff(m.indptr).astype(np.int32)
        dim = (int(m.shape[0]), int(m.shape[1]))
    else:
        a = np.asarray(x, np.float64)
        if a.ndim != 2:
            raise ValueError("x must be a matrix")
        if np.isnan(a).any():
            raise ValueError("NAs in x")
        mask = a != 0
        row_size = mask.sum(1).astype(np.int32)
        rr, cc = np.nonzero(mask)
        value = a[rr, cc].astype(np.float64)
        col_idx = cc.astype(np.int32)
        dim = a.shape
    if feature_names is None:
        feature_names = ["V%d" % (i + 1) for i in range(dim[1])]
    if len(feature_names) != dim[1]:
        raise ValueError("feature_names has the wrong length")
    feats = dict(value=value, col_idx=col_idx, row_size=row_size, dim=(int(dim[0]), int(dim[1])), size=int(value.size),
                 feature_names=list(feature_names), transposed=False)
    labels = None
    if y is not None:
        labels = np.asarray(y, np.float64).reshape(-1)
        if labels.size != dim[0]:
            raise ValueError("the length of y is not equal to the number of rows of x")
    return FmMatrix(features=feats, labels=labels)


# ---------------------------------------------------------------------------------------------- controls
class Control(dict):
    def __init__(self, cls, **kw):
        super().__init__(**kw)
        self.cls = cls


def control_assign(defaults, assign):
    """R/control_tools.R:1-37: type-coerce by the default's class, warn on unknown names"""
    out = dict(defaults)
    n_known = 0
    for name, val in assign.items():
        if name in out:
            d = out[name]
            if isinstance(d, bool):
                if not isinstance(val, (bool, np.bool_)):
                    raise TypeError("is.logical(%s) is not TRUE" % name)
                val = bool(val)
            elif isinstance(d, int):
                iv = int(val)
                if iv != val:
                    iv = max(d, iv)
                    warnings.warn("%s is not integer, it will be set as %d" % (name, iv))
                val = iv
            out[name] = val
            n_known += 1
    if n_known != len(assign):
        warnings.warn("some arguments are unknown...")
    return out


MODEL_DEFAULT = {"keep.w0": True, "L2.w0": 0.0, "keep.w1": True, "L1.w1": 0.0, "L2.w1": 0.0, "factor.number": 2,
                 "v.init_mean": 0.0, "v.init_stdev": 0.01, "L1.v": 0.0, "L2.v": 0.0}


def _dots(kw):
    """keep_w0 -> keep.w0, L2_w0 -> L2.w0, factor_number -> factor.number, v_init_mean -> v.init_mean"""
    out = {}
    for k, v in kw.items():
        out[k if "." in k else k.replace("_", ".", 1)] = v
    return out


def model_control(task="CLASSIFICATION", **kw):
    """R/fm_control.R:43-66"""
    if task not in ("CLASSIFICATION", "REGRESSION", "RANK"):
        raise ValueError("'arg' should be one of \"CLASSIFICATION\", \"REGRESSION\", \"RANK\"")
    return Control("model.control", task=task, **{"hyper.params": control_assign(MODEL_DEFAULT, _dots(kw))})


def _solver(name, defaults, kw):
    s = Control("solver", **control_assign(defaults, kw))
    s.solver = name
    return s


def MCMC_solver(**kw):
    """R/fm_solver_control.R:36-62 (all six values are overwritten in C++, SURVEY F2)"""
    return _solver("MCMC", dict(alpha_0=1.0, gamma_0=1.0, beta_0=1.0, mu_0=0.0, alpha=1.0, w0_mean_0=1.0), kw)


def ALS_solver(**kw):
    """R/fm_solver_control.R:64-88"""
    return _solver("ALS", dict(alpha_0=1.0, gamma_0=1.0, beta_0=1.0, mu_0=0.0, alpha=1.0, w0_mean_0=1.0), kw)


def SGD_solver(**kw):
    """R/fm_solver_control.R:91-107"""
    return _solver("SGD", dict(learn_rate=0.01, random_step=1), kw)


def FTRL_solver(**kw):
    """R/fm_solver_control.R:109-131"""
    return _solver("FTRL", dict(alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0, random_step=1), kw)


def TDAP_solver(**kw):
    """R/fm_solver_control.R:134-155"""
    return _solver("TDAP", dict(gamma=1e-4, alpha_w=0.1, alpha_v=0.1, random_step=1), kw)


def solver_control(max_iter=10000, solver=None):
    """R/fm_solver_control.R:22-33: MCMC/ALS sweeps are clamped to 100"""
    if solver is None:
        solver = TDAP_solver()
    if solver.solver in ("MCMC", "ALS") and max_iter > 100:
        warnings.warn("the maximum number of iteratorions for MCMC/ALS solver is 100, so max_iter will be set to 100")
        max_iter = min(max_iter, 100)
    return Control("solver.control", nthreads=fm_get_threads(), max_iter=int(max_iter), solver=solver)


def track_control(step_size=-1, evaluate_metric="LL", convergence=1e-4):
    """R/fm_track_control.R:20-26"""
    if evaluate_metric not in ("AUC", "ACC", "LL", "RMSE", "MAE"):
        raise ValueError("evaluate.metric %in% c(\"AUC\", \"ACC\", \"LL\", \"RMSE\", \"MAE\") is not TRUE")
    return Control("track.control", max_iter=1, step_size=int(step_size), **{"evaluate.metric": evaluate_metric},
                   convergence=float(convergence))


# ---------------------------------------------------------------------------------------------- FM() glue
class FM(dict):
    """class "FM": list(Model = list(w0, w, v) + attrs, Scales, Trace)"""


def _precision(solver_name=None):
    """FM.precision; "auto" = fp64 where parity with the reference is the point (exact mode, ALS, MCMC, predict), fp32 in throughput mode"""
    opt = str(_OPTIONS["FM.precision"]).lower()
    if opt in ("f64", "double", "fp64"):
        return L.F64
    if opt in ("f32", "float", "fp32"):
        return L.F32
    if solver_name in ("SGD", "FTRL", "TDAP") and _OPTIONS["FM.mode"] == "minibatch":
        return L.F32
    return L.F64


def _acquire(ctx, feats, labels, normalized):
    """device handle of an fm.matrix: uploaded once and parked in a slot of the features list (the external-pointer slot of the R
    glue, INTEGRATION.md); labels are replaced in place when they changed; the values go back to the uploaded ones unless this
    call rescales them itself (fmwr_data_scales / normalize always start from the uploaded values)"""
    n, p = feats["dim"]
    key = (id(feats["value"]), id(feats["col_idx"]), id(feats["row_size"]), int(n), int(p), int(np.asarray(feats["value"]).size), id(ctx))
    slot = feats.get("_handle") if _OPTIONS["FM.cache"] else None
    if slot is not None and slot["key"] == key and slot["data"].h:
        d = slot["data"]
        if labels is not None and slot["labels_id"] != id(labels):
            d.set_labels(labels)
            slot["labels_id"] = id(labels)
            slot["labels_ref"] = labels
        if not normalized:
            d.restore_values()
        return d, True
    d = L.Data.from_r_lists(ctx, n, p, feats["row_size"], feats["col_idx"], feats["value"], labels)
    if _OPTIONS["FM.cache"]:
        # labels_ref keeps the array alive so its id() cannot be recycled by another array
        feats["_handle"] = dict(key=key, data=d, labels_id=id(labels) if labels is not None else None, labels_ref=labels)
        return d, True
    return d, False


def _compat():
    return L.COMPAT_REFERENCE if _OPTIONS["FM.compat"] == "reference" else 0


def _model_cfg(mc):
    hp = mc["hyper.params"]
    return L.ModelCfg(task=L.TASKS[mc["task"]], keep_w0=int(hp["keep.w0"]), keep_w1=int(hp["keep.w1"]), k=int(hp["factor.number"]),
                      l2_w0=float(hp["L2.w0"]), l1_w1=float(hp["L1.w1"]), l2_w1=float(hp["L2.w1"]), l1_v=float(hp["L1.v"]),
                      l2_v=float(hp["L2.v"]))


def _FM(data, normalize0, fm_controls, solver_controls, track_controls, model_list, streams=None, posterior=None, holdout=None):
    """body of FM() (reference src/FM.cpp:7-174) on top of the C ABI.  posterior (fm_posterior): dict(burn_in, newdata) in, and
    the device means out as posterior["train"] and posterior["newdata_mean"].  holdout (fm_train_holdout): dict(newdata, labels,
    select_best, patience, snapshots) in; the trace gains "evaluation.test" and "best.index"."""
    ctx = _ctx()
    feats = data["features"]
    n, p = feats["dim"]
    labels = data["labels"]
    normalize0 = np.atleast_1d(np.asarray(normalize0, np.int64))
    d, parked = _acquire(ctx, feats, labels, normalize0[0] > -1)
    evals = []                                                            # (handle, parked) of posterior / holdout["newdata"]
    try:
        scales = {}
        if normalize0[0] > -1:                                            # FM.cpp:36-38
            mean, sd = d.scales(normalize0.astype(np.int32))
            scales["mean"], scales["std"] = mean, sd
        scales["model.vars"] = list(feats["feature_names"])
        mc = _model_cfg(fm_controls)
        hp = fm_controls["hyper.params"]
        k = mc.k
        prec = _precision(solver_controls["solver"].solver)
        m = L.Model(ctx, mc, p, prec)
        try:
            # Model::init (src/core/Model.h:63-72): w = 0, V ~ rnorm(mean, sd) filled factor-major (f outer, feature inner)
            rng = np.random.default_rng(int(_OPTIONS["FM.seed"]))
            v = (hp["v.init_mean"] + hp["v.init_stdev"] * rng.standard_normal((k, p))).T.copy() if k > 0 else np.zeros((p, 0))
            w0, w = 0.0, np.zeros(p)
            lo, hi = float(np.min(labels)), float(np.max(labels))
            if model_list is not None:                                     # warm start == fm.update (FM.cpp:66-72, :91-96)
                md = model_list["Model"]
                w0, w = float(md["w0"]), np.asarray(md["w"], np.float64)
                v = np.asarray(md["v"], np.float64).T.copy()               # stored k x p like R
                tr = model_list["Scales"]["target.range"]
                lo, hi = min(lo, tr[0]), max(hi, tr[1])
            m.set(w0, w, v)
            s = solver_controls["solver"]
            name = s.solver
            warm = 0
            if (model_list is not None and _OPTIONS["FM.keep_state"] and model_list.get("State") is not None
                    and model_list["State"]["solver"] == L.SOLVERS[name] and name in ("SGD", "FTRL", "TDAP")):
                m.set_state(model_list["State"])
                warm = 1
            sc = L.SolverCfg(solver=L.SOLVERS[name], max_iter=int(solver_controls["max_iter"]), random_step=int(s.get("random_step", 1)),
                             learn_rate=float(s.get("learn_rate", 0.01)), alpha_w=float(s.get("alpha_w", 0.1)),
                             alpha_v=float(s.get("alpha_v", 0.1)), beta_w=float(s.get("beta_w", 1.0)), beta_v=float(s.get("beta_v", 1.0)),
                             gamma=float(s.get("gamma", 1e-4)), min_target=lo, max_target=hi,
                             mode=L.MODE_MINIBATCH if _OPTIONS["FM.mode"] == "minibatch" else L.MODE_EXACT,
                             batch_size=int(_OPTIONS["FM.batch"]), precision=prec, compat=_compat(),
                             enable_v=int(bool(_OPTIONS["FM.enable_v"])), step_size=int(track_controls["step_size"]),
                             metric=L.METRICS[track_controls["evaluate.metric"]], convergence=float(track_controls["convergence"]),
                             seed=int(_OPTIONS["FM.seed"]), warm_state=warm)
            keep = []
            if streams:
                for fld, cnt, dt in (("normals", "n_normals", np.float64), ("gammas", "n_gammas", np.float64), ("rands", "n_rands", np.int32)):
                    if streams.get(fld) is not None:
                        a = np.ascontiguousarray(streams[fld], dt)
                        keep.append(a)
                        setattr(sc, fld, L.ptr(a)); setattr(sc, cnt, a.size)
            trace = None
            if sc.step_size > 0:
                from math import ceil
                nrec = min(10001, int(ceil((sc.max_iter - 0.5) / sc.step_size)) + 2)
                trace = L.TraceBuf(nrec, p, k, snapshots=holdout is None or holdout["snapshots"])
            if holdout is not None:
                for nd, nd_labels in zip(holdout["newdata"], holdout["labels"]):   # z-scored with the training scales as fm.track does
                    evals.append(_acquire(ctx, nd["features"], nd_labels, normalize0[0] > -1))
                    if normalize0[0] > -1:
                        evals[-1][0].normalize(scales["mean"], scales["std"])
                test, best = L.train_holdout_dev(ctx, m, d, sc, trace, [e for e, _ in evals], holdout["select_best"],
                                                 holdout["patience"], keep=keep)
            elif posterior is None:
                L.train_dev(ctx, m, d, sc, trace, keep=keep)
            else:
                for nd in posterior["newdata"]:                           # checked and z-scored as predict does it
                    evals.append(_acquire(ctx, nd["features"], None, normalize0[0] > -1))
                    if normalize0[0] > -1:
                        evals[-1][0].normalize(scales["mean"], scales["std"])
                L.train_posterior_dev(ctx, m, d, sc, posterior["burn_in"], [e for e, _ in evals], trace, keep=keep)
                posterior["train"] = L.predict_fetch(ctx, d)
                posterior["newdata_mean"] = [L.predict_fetch(ctx, e) for e, _ in evals]
            gw0, gw, gv = m.get()
            state = m.get_state() if (_OPTIONS["FM.keep_state"] and name in ("SGD", "FTRL", "TDAP")) else None
        finally:
            m.close()
    finally:
        if not parked:
            d.close()
        for e, e_parked in evals:
            if not e_parked:
                e.close()
    model = dict(w0=gw0, w=gw, v=gv.T.copy())                              # v returned k x p like Model::save_model
    model["model.control"] = fm_controls
    model["solver.control"] = solver_controls
    model["track.control"] = track_controls
    res = FM(Model=model, Scales=scales)
    if state is not None:
        res["State"] = state
    if trace is not None:
        t = trace.result()
        model["convergence"] = t["convergent"]
        snaps = ([dict(w0=t["snap_w0"][i], w=t["snap_w"][i], v=t["snap_v"][i].T.copy()) for i in range(len(t["rec_index"]))]
                 if "snap_w0" in t else [])
        res["Trace"] = {"trace": [t["rec_index"].astype(np.float64)] + snaps, "evaluation.train": t["eval_train"]}
        if holdout is not None:
            res["Trace"]["evaluation.test"] = [row for row in test]
            res["Trace"]["best.index"] = best
    else:
        model["convergence"] = False
    scales["target.range"] = (lo, hi)
    return res


def fm_train(data, normalize=True, control=None, _streams=None):
    """R/fm_train.R:70-127"""
    data, norm, ctl = _train_setup(data, normalize, control)
    return _FM(data, norm - 1, ctl["model"], ctl["solver"], ctl["track"], None, streams=_streams)


def _train_setup(data, normalize, control):
    """argument checks and controls of fm.train (R/fm_train.R:70-125): (data with recoded labels, 1-based columns to normalize
    or [-1], controls)"""
    if data.get("labels") is None:
        raise ValueError("there are no labels in data")
    ncol = data.ncol()
    if isinstance(normalize, (bool, np.bool_)):
        norm = np.arange(1, ncol + 1) if normalize else np.array([-1])
    else:
        norm = np.asarray(normalize)
        if not np.issubdtype(norm.dtype, np.integer):
            raise ValueError("normalize should be a logical value or an integer vector")
        if np.any(norm < 1) or np.any(norm > ncol):
            raise ValueError("the columns to be normalized is out of range")
    ctl = {"model": model_control(), "solver": solver_control(max_iter=max(10000, 2 * data.nrow())), "track": track_control()}
    if control is not None:
        for c in control:
            if not isinstance(c, Control) or not c.cls.endswith(".control"):
                raise ValueError("control list is wrong")
            ctl[c.cls.split(".")[0]] = c
    ctl["model"]["nthreads"] = fm_get_threads()
    ctl["solver"]["nthreads"] = fm_get_threads()
    ctl["track"]["max_iter"] = ctl["solver"]["max_iter"]
    if ctl["solver"]["solver"].solver in ("MCMC", "ALS") and ctl["track"]["step_size"] > 1:
        warnings.warn("the step_size will be set to 1 for MCMC/ALS solver")
        ctl["track"]["step_size"] = 1
    if ctl["model"]["task"] == "CLASSIFICATION":
        u = np.unique(data["labels"])
        if u.size != 2:
            raise ValueError("target should have two levels")
        if np.array_equal(u, [0, 1]):
            data = FmMatrix(features=data["features"], labels=np.where(data["labels"] < 1, -1.0, 1.0))
        elif not np.array_equal(u, [-1, 1]):
            raise ValueError("target should be c(0, 1) or c(-1, 1)")
    return data, norm, ctl


def _check_newdata(newdata, data, need_labels):
    """the newdata list of fm_posterior / fm_train_holdout: fm.matrix objects (labelled where they are scored) without NAs,
    none of them the training data, each listed once"""
    for i, nd in enumerate(newdata):
        if not isinstance(nd, FmMatrix):
            raise ValueError("newdata must be fm.matrix objects")
        if need_labels and nd.get("labels") is None:
            raise ValueError("there are no labels in newdata")
        if np.isnan(nd["features"]["value"]).any():
            raise ValueError("there are NAs in newdata")
        if nd["features"] is data["features"]:
            raise ValueError("newdata is the training data")
        if any(nd["features"] is o["features"] for o in newdata[:i]):
            raise ValueError("the same newdata appears twice")


def fm_posterior(data, newdata=(), burn_in=0, normalize=True, control=None):
    """Engine extension: the MCMC posterior mean libFM predicts with.  Trains exactly as fm_train(data, normalize, control) and
    also averages, on the device, the predict.FM prediction of draws burn_in+1 .. max_iter (draw t = the model after sweep t)
    on data and on every newdata (fm.matrix objects of the same width, z-scored with the training scales as predict does).
    Returns dict(fit=<what fm_train returns>, train=<mean on data>, newdata=[<mean per newdata>])."""
    if isinstance(newdata, FmMatrix):
        newdata = [newdata]
    newdata = list(newdata)
    data, norm, ctl = _train_setup(data, normalize, control)
    if ctl["solver"]["solver"].solver != "MCMC":
        raise ValueError("posterior averaging needs the MCMC solver")
    max_iter = int(ctl["solver"]["max_iter"])
    if int(burn_in) != burn_in or not 0 <= burn_in < max_iter:
        raise ValueError("burn_in must be an integer in [0, max_iter) = [0, %d)" % max_iter)
    _check_newdata(newdata, data, need_labels=False)
    post = dict(burn_in=int(burn_in), newdata=newdata)
    fit = _FM(data, norm - 1, ctl["model"], ctl["solver"], ctl["track"], None, posterior=post)
    return dict(fit=fit, train=post["train"], newdata=post["newdata_mean"])


def fm_train_holdout(data, newdata, normalize=True, control=None, select="last", patience=0, snapshots=True):
    """Engine extension of the fm.train -> fm.track -> fm.select workflow: trains exactly as fm_train(data, normalize, control)
    and, at every tracker record (step_size > 0 in track.control), also scores every newdata (labelled fm.matrix objects of the
    same width, labels 0/1 recoded and values z-scored with the training scales as fm_track does) on the device.
    Trace gains "evaluation.test" (one array per newdata, what fm_track would return as "test") and "best.index" (the first
    record with the best score on newdata[0]: highest for classification, lowest for regression; -1 if all were NaN).
    select="best" puts that record's model in Model (fm_select(fit, best_iter=best.index)); patience > 0 also stops training
    after that many records in a row without an improvement on newdata[0].  snapshots=False keeps no per-record model on the
    host (the trace is then the index, the train and test curves and best.index; fm_track and fm_select refuse such a fit)."""
    if isinstance(newdata, FmMatrix):
        newdata = [newdata]
    if not isinstance(newdata, (list, tuple)) or not newdata:
        raise ValueError("newdata must be a fm.matrix object or a non-empty list of them")
    newdata = list(newdata)
    if select not in ("last", "best"):
        raise ValueError("select must be \"last\" or \"best\"")
    if int(patience) != patience or patience < 0:
        raise ValueError("patience must be an integer >= 0")
    data, norm, ctl = _train_setup(data, normalize, control)
    if ctl["track"]["step_size"] <= 0:
        raise ValueError("held-out tracking needs step_size > 0 in track.control")
    _check_newdata(newdata, data, need_labels=True)
    cls = ctl["model"]["task"] == "CLASSIFICATION"
    labels = []
    for nd in newdata:
        y = np.asarray(nd["labels"], np.float64)
        if cls and np.array_equal(np.unique(y), [0, 1]):                 # as fm_track recodes them
            y = np.where(y < 1, -1.0, 1.0)
        labels.append(y)
    ho = dict(newdata=newdata, labels=labels, select_best=int(select == "best"), patience=int(patience), snapshots=bool(snapshots))
    return _FM(data, norm - 1, ctl["model"], ctl["solver"], ctl["track"], None, holdout=ho)


def _require_snapshots(obj):
    t = obj["Trace"]["trace"]
    if len(t) - 1 != len(t[0]):
        raise ValueError("the trace keeps no model snapshots (fm_train_holdout(..., snapshots=False)): "
                         "its held-out scores are Trace$evaluation.test and its best record Trace$best.index")


def _link_for(model):
    task = model["model.control"]["task"]
    if task == "CLASSIFICATION":
        name = model["solver.control"]["solver"].solver
        return L.LINK_PROBIT_TABLE if name in ("MCMC", "ALS") else L.LINK_LOGISTIC      # Model::predict_prob, Model.h:163-180
    return L.LINK_CLAMP


@contextlib.contextmanager
def _on_device(obj, newdata, normalize):
    """the prologue of predict (R/fm_predict.R:12-34, src/FM.cpp:177-203): newdata checks and warnings, newdata's parked device
    handle z-scored with the model's Scales, and the model on the device; yields (ctx, model handle, data handle)"""
    if newdata is None:
        raise ValueError("newdata is null")
    if not isinstance(newdata, FmMatrix):
        raise ValueError("newdata must be a fm.matrix object")
    if np.isnan(newdata["features"]["value"]).any():
        raise ValueError("there are NAs in newdata")
    has_mean = obj["Scales"].get("mean") is not None
    if normalize and not has_mean:
        raise ValueError("can not normalize newdata because all the variables have not been normalized in FM model")
    if not normalize and has_mean:
        warnings.warn("some variables in FM model are normalized, but those in newdata will not")
    ctx = _ctx()
    feats = newdata["features"]
    n, p = feats["dim"]
    model = obj["Model"]
    d, parked = _acquire(ctx, feats, None, bool(normalize))
    try:
        if normalize:
            d.normalize(obj["Scales"]["mean"], obj["Scales"]["std"])
        m = L.Model(ctx, _model_cfg(model["model.control"]), p, _precision())
        try:
            m.set(float(model["w0"]), np.asarray(model["w"]), np.asarray(model["v"]).T.copy())
            yield ctx, m, d
        finally:
            m.close()
    finally:
        if not parked:
            d.close()


def predict(obj, newdata=None, normalize=True):
    """R/fm_predict.R:12-34 + FMPredict (src/FM.cpp:177-214)"""
    with _on_device(obj, newdata, normalize) as (ctx, m, d):
        lo, hi = obj["Scales"]["target.range"]
        L.predict_dev(ctx, m, d, _link_for(obj["Model"]), lo, hi)
        return L.predict_fetch(ctx, d)


def fm_contrib(obj, newdata, normalize=True):
    """Engine extension (xgboost's predcontrib, LightGBM's pred_contrib): the exact per-feature Shapley values of the raw score,
    phi_j = [keep.w1] w_j x_j + 1/2 x_j sum_f v_jf (S_f - x_j v_jf) for every stored entry of newdata, computed on the device.
    Checks, warnings and z-scoring are predict's, on the same parked handle.  Returns dict(bias=[keep.w0] w0,
    contrib=<scipy.sparse.csr_matrix n x p with newdata's pattern>, score=<raw scores>) with bias + contrib.sum(1) == score.
    The contributions are on the margin scale (the links are not additive) and of the values the model sees, z-scored when
    normalize is on; an explicitly stored zero gets 0."""
    import scipy.sparse as sp
    with _on_device(obj, newdata, normalize) as (ctx, m, d):
        L.contrib_dev(ctx, m, d)
        phi = L.contrib_fetch(ctx, d)
        score = L.predict_fetch(ctx, d)
    feats = newdata["features"]
    indptr = np.concatenate([[0], np.cumsum(np.asarray(feats["row_size"], np.int64))])
    contrib = sp.csr_matrix((phi, np.asarray(feats["col_idx"], np.int32), indptr), shape=tuple(feats["dim"]))
    model = obj["Model"]
    bias = float(model["w0"]) if model["model.control"]["hyper.params"]["keep.w0"] else 0.0
    return dict(bias=bias, contrib=contrib, score=score)


def fm_update(obj, data, normalize=None, control=None):
    """R/fm_update.R:18-135: warm start of (w0, w, V) on new data with the stored controls; traces are spliced"""
    if not isinstance(obj, FM):
        raise ValueError("object must be a FM object")
    if data.get("labels") is None:
        raise ValueError("there are no labels in data")
    if list(data["features"]["feature_names"]) != list(obj["Scales"]["model.vars"]):
        raise ValueError("the features of data are not the same as those in FM model")
    model = obj["Model"]
    ctl = {"model": model["model.control"], "solver": model["solver.control"], "track": model["track.control"]}
    if control is not None:
        for c in control:
            if c.cls == "model.control":
                raise ValueError("model.control can not be changed in fm.update")
            ctl[c.cls.split(".")[0]] = c
    was_normalized = obj["Scales"].get("mean") is not None
    if normalize is None:
        normalize = was_normalized
    if normalize != was_normalized:
        raise ValueError("normalization of data must be the same as in the FM model")
    ncol = data.ncol()
    norm = np.arange(1, ncol + 1) if normalize else np.array([-1])
    if ctl["model"]["task"] == "CLASSIFICATION":
        u = np.unique(data["labels"])
        if np.array_equal(u, [0, 1]):
            data = FmMatrix(features=data["features"], labels=np.where(data["labels"] < 1, -1.0, 1.0))
    new = _FM(data, norm - 1, ctl["model"], ctl["solver"], ctl["track"], obj)
    if "Trace" in obj and "Trace" in new:                                   # R/fm_update.R:125-133
        old_t, new_t = obj["Trace"], new["Trace"]
        off = old_t["trace"][0][-1] + 1 if len(old_t["trace"][0]) else 0
        idx = np.concatenate([old_t["trace"][0], new_t["trace"][0] + off])
        new["Trace"] = {"trace": [idx] + old_t["trace"][1:] + new_t["trace"][1:],
                        "evaluation.train": np.concatenate([old_t["evaluation.train"], new_t["evaluation.train"]])}
    return new


def fm_track(obj, newdata, normalize=True, evaluate_metric=None):
    """R/fm_track.R:27 + FMTrack / Tracker::report (src/FM.cpp:218-258, src/core/Tracker.h:70-94):
    score every recorded snapshot on new data"""
    if "Trace" not in obj:
        raise ValueError("there is no trace in FM model, please set step_size > 0 in track.control")
    _require_snapshots(obj)
    if newdata.get("labels") is None:
        raise ValueError("there are no labels in newdata")
    model = obj["Model"]
    metric = evaluate_metric or model["track.control"]["evaluate.metric"]
    feats = newdata["features"]
    n, p = feats["dim"]
    labels = np.asarray(newdata["labels"], np.float64)
    if model["model.control"]["task"] == "CLASSIFICATION" and np.array_equal(np.unique(labels), [0, 1]):
        labels = np.where(labels < 1, -1.0, 1.0)
    do_norm = bool(normalize and obj["Scales"].get("mean") is not None)
    ctx = _ctx()
    # Tracker::report (src/core/Tracker.h:70-94) on the parked device copy of newdata: per snapshot a forward + the metric
    d, parked = _acquire(ctx, feats, labels, do_norm)
    snaps = obj["Trace"]["trace"][1:]
    out = np.zeros(len(snaps))
    try:
        if do_norm:
            d.normalize(obj["Scales"]["mean"], obj["Scales"]["std"])        # SMatrix::normalize, src/util/Smatrix.h:144-150
        mc = _model_cfg(model["model.control"])
        lo, hi = obj["Scales"]["target.range"]
        m = L.Model(ctx, mc, p, _precision())
        try:
            for i, sn in enumerate(snaps):
                m.set(float(sn["w0"]), np.asarray(sn["w"], np.float64), np.asarray(sn["v"], np.float64).T.copy())
                L.predict_dev(ctx, m, d, _link_for(model), lo, hi)
                out[i] = L.evaluate_dev(ctx, d, mc.task, L.METRICS[metric])
        finally:
            m.close()
    finally:
        if not parked:
            d.close()
    return dict(index=obj["Trace"]["trace"][0], train=obj["Trace"]["evaluation.train"], test=out, metric=metric)


def fm_select(obj, best_iter=None, track=None, higher_is_better=None):
    """R/fm_select.R:58-61: swap a recorded snapshot in as the model"""
    if "Trace" not in obj:
        raise ValueError("there is no trace in FM model")
    _require_snapshots(obj)
    if best_iter is None:
        if track is None:
            raise ValueError("either best_iter or the result of fm.track is needed")
        if higher_is_better is None:
            higher_is_better = track["metric"] in ("LL", "AUC", "ACC")
        best_iter = int(np.argmax(track["test"]) if higher_is_better else np.argmin(track["test"]))
    snap = obj["Trace"]["trace"][1 + int(best_iter)]
    new = FM(obj)
    new["Model"] = dict(obj["Model"])
    new["Model"].update(w0=snap["w0"], w=snap["w"], v=snap["v"])
    return new
