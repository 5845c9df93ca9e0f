"""MCMC attribute groups on the device (fmwr_solver_cfg::attr_group): the engine against the fp64 restatement of the grouped
sampler (tests/mcmc_groups_ref.py) with the same injected streams on every coordinate-pass layout, a one-group map unchanged,
the posterior / held-out wrappers on the same chain, the argument checks, and the host mirror's features$attr_group."""
import numpy as np
import pytest

from fmwr_b200 import _lib as L
from fmwr_b200 import api as A
from tests import mcmc_groups_cases as G
from tests.util import relerr

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("group_map", G.MAPS)
@pytest.mark.parametrize("task", [L.CLASSIFICATION, L.REGRESSION])
@pytest.mark.parametrize("enable_v", [0, 1])
@pytest.mark.parametrize("layout", G.LAYOUTS + ["fields_column"])
def test_grouped_mcmc_matches_restatement(gpu_ctx, port, monkeypatch, layout, enable_v, task, group_map):
    """fields: fused dense passes; fields_odd: permuted rows, fp32 on the fp64 shadow; fields_sparse: row-major passes;
    ragged: column-parallel kernels; fields_column: the fields data forced onto the column-parallel kernels"""
    if layout == "fields_column":
        monkeypatch.setenv("FMWR_ALS_COLUMN", "1")
    ds, fields = G.layout("fields" if layout == "fields_column" else layout)
    y, w0, w, v = G.problem(task, ds)
    grp, ng = G.group_map(group_map, ds["p"], fields)
    strm = G.streams(ds["p"], ng)
    t64 = 1e-6 if layout == "fields_odd" else 1e-8
    for compat in (L.COMPAT_REFERENCE, 0):
        for prec, tol in ((L.F64, t64), (L.F32, 1e-4)):
            init = (w0, w, v) if prec == L.F64 else (float(np.float32(w0)), w.astype(np.float32).astype(np.float64),
                                                     v.astype(np.float32).astype(np.float64))
            r = G.reference_run(port, task, ds, y, init, enable_v, compat, strm, grp, ng)
            g = G.engine_run(gpu_ctx, task, ds, y, init, enable_v, compat, prec, strm, grp, ng)
            errs = (relerr(g[0], r[0]), relerr(g[1], r[1]), relerr(g[2], r[2]))
            assert max(errs) < tol, (compat, prec, errs)


def test_one_group_map_is_unchanged(gpu_ctx, monkeypatch):
    """on the column-parallel passes, which sum without atomics and so repeat a chain bit for bit"""
    monkeypatch.setenv("FMWR_ALS_COLUMN", "1")
    ds, _ = G.layout("fields")
    for task in (L.CLASSIFICATION, L.REGRESSION):
        y, *init = G.problem(task, ds)
        strm = G.streams(ds["p"], 1)
        plain = G.engine_run(gpu_ctx, task, ds, y, init, 1, L.COMPAT_REFERENCE, L.F64, strm, None, 0)
        one = G.engine_run(gpu_ctx, task, ds, y, init, 1, L.COMPAT_REFERENCE, L.F64, strm, np.zeros(ds["p"], np.int32), 1)
        assert plain[0] == one[0] and np.array_equal(plain[1], one[1]) and np.array_equal(plain[2], one[2])


def test_wrappers_run_the_grouped_chain(gpu_ctx, monkeypatch):
    """fmwr_train_posterior_dev and fmwr_train_holdout_dev (select last, patience 0) leave the model of fmwr_train_dev"""
    monkeypatch.setenv("FMWR_ALS_COLUMN", "1")
    ctx = gpu_ctx
    ds, fields = G.layout("fields")
    y, w0, w, v = G.problem(L.REGRESSION, ds)
    grp, ng = G.group_map("scattered", ds["p"], fields)
    strm = G.streams(ds["p"], ng)
    d = L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y)
    e = L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y)
    m = L.Model(ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=G.K, l2_w0=0.1), ds["p"], L.F64)
    out = {}
    try:
        for how in ("train", "posterior", "holdout"):
            m.set(w0, w, v)
            sc, keep = G.engine_cfg(L.REGRESSION, y, 1, L.COMPAT_REFERENCE, L.F64, strm, grp, ng, step_size=1)
            tr = L.TraceBuf(G.SWEEPS + 2)
            if how == "train":
                L.train_dev(ctx, m, d, sc, tr, keep=keep)
            elif how == "posterior":
                L.train_posterior_dev(ctx, m, d, sc, 1, [e], tr, keep=keep)
            else:
                L.train_holdout_dev(ctx, m, d, sc, tr, [e], select_best=0, patience=0, keep=keep)
            out[how] = m.get()
    finally:
        m.close(); d.close(); e.close()
    assert float(np.max(np.abs(out["train"][2] - v))) > 1e-3
    for how in ("posterior", "holdout"):
        assert out[how][0] == out["train"][0] and np.array_equal(out[how][1], out["train"][1]) and np.array_equal(out[how][2], out["train"][2]), how


def test_bad_grouping_is_rejected_and_leaves_the_model(gpu_ctx):
    ctx = gpu_ctx
    ds, fields = G.layout("fields")
    p = ds["p"]
    y, w0, w, v = G.problem(L.REGRESSION, ds)
    good, ng = G.group_map("fields", p, fields)
    d = L.Data.from_csr32(ctx, ds["n"], p, ds["rowptr"], ds["col"], ds["val"], y)
    e = L.Data.from_csr32(ctx, ds["n"], p, ds["rowptr"], ds["col"], ds["val"], y)
    m = L.Model(ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=G.K), p, L.F64)
    m.set(w0, w, v)
    before = m.get()
    high, neg = good.copy(), good.copy()
    high[5] = ng
    neg[7] = -1
    cases = [(high, ng, L.MCMC, "out of range"), (neg, ng, L.MCMC, "out of range"),
             (good, 0, L.MCMC, "n_groups must be"), (np.zeros(p, np.int32), -1, L.MCMC, "n_groups must be"),
             (np.zeros(p, np.int32), 65537, L.MCMC, "n_groups must be"), (np.zeros(p, np.int32), p + 1, L.MCMC, "n_groups must be"),
             (None, 2, L.MCMC, "needs an attr_group map"), (good, ng, L.ALS, "need the MCMC solver"),
             (good, ng, L.FTRL, "need the MCMC solver")]
    try:
        for grp, n_groups, solver, msg in cases:
            sc, keep = G.engine_cfg(L.REGRESSION, y, 1, L.COMPAT_REFERENCE, L.F64, None, grp, n_groups, step_size=1)
            sc.solver = solver
            for call in ("train", "posterior", "holdout"):
                if call != "train" and solver != L.MCMC:
                    continue
                with pytest.raises(L.FmwrError) as ei:
                    if call == "train":
                        L.train_dev(ctx, m, d, sc, keep=keep)
                    elif call == "posterior":
                        L.train_posterior_dev(ctx, m, d, sc, 1, [e], keep=keep)
                    else:
                        L.train_holdout_dev(ctx, m, d, sc, L.TraceBuf(8), [e], keep=keep)
                assert ei.value.code == 1, (call, msg, ei.value.code)
                assert msg in ei.value.msg, (call, msg, ei.value.msg)
                after = m.get()
                assert after[0] == before[0] and np.array_equal(after[1], before[1]) and np.array_equal(after[2], before[2])
    finally:
        m.close(); d.close(); e.close()


def _host_problem():
    ds, fields = G.layout("fields")
    n, p = ds["n"], ds["p"]
    import scipy.sparse as sp
    X = sp.csr_matrix((ds["val"].astype(np.float64), ds["col"].astype(np.int64), ds["rowptr"].astype(np.int64)), shape=(n, p))
    y = np.random.default_rng(8).normal(0, 1, n)
    data = A.fm_matrix(X, y)
    grp, ng = G.group_map("fields", p, fields)
    return data, grp, ng


def _control(solver, max_iter=G.SWEEPS):
    return [A.model_control("REGRESSION", factor_number=G.K), A.solver_control(max_iter=max_iter, solver=solver),
            A.track_control(step_size=-1, evaluate_metric="RMSE")]


def test_host_mirror_passes_the_map(gpu_ctx, monkeypatch):
    monkeypatch.setenv("FMWR_ALS_COLUMN", "1")            # bit-for-bit comparisons: the passes that sum without atomics
    data, grp, ng = _host_problem()
    n, p = data.nrow(), data.ncol()
    saved = A.options()["FM.enable_v"]
    A.options(**{"FM.enable_v": True})
    try:
        strm = dict(zip(("normals", "gammas"), G.streams(p, ng)[:2]))
        plain = A.fm_train(data, False, _control(A.MCMC_solver()), _streams=strm)
        data["features"]["attr_group"] = grp
        fit = A.fm_train(data, False, _control(A.MCMC_solver()), _streams=strm)
        post = A.fm_posterior(data, [], burn_in=1, normalize=False, control=_control(A.MCMC_solver()))
        post_plain = A.fm_train(data, False, _control(A.MCMC_solver()))
        sgd = A.fm_train(data, False, _control(A.SGD_solver(), max_iter=2 * n))
        del data["features"]["attr_group"]
        sgd_plain = A.fm_train(data, False, _control(A.SGD_solver(), max_iter=2 * n))
    finally:
        A.options(**{"FM.enable_v": saved})
    # the same run through the C ABI: fm_train's initial model (Model::init with FM.seed), its target range and its precision
    rng = np.random.default_rng(int(A.get_option("FM.seed")))
    hp = A.model_control("REGRESSION", factor_number=G.K)["hyper.params"]
    v = (hp["v.init_mean"] + hp["v.init_stdev"] * rng.standard_normal((G.K, p))).T.copy()
    d = L.Data.from_r_lists(gpu_ctx, n, p, data["features"]["row_size"], data["features"]["col_idx"], data["features"]["value"], data["labels"])
    m = L.Model(gpu_ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=G.K), p, L.F64)
    try:
        m.set(0.0, np.zeros(p), v)
        sc, keep = G.engine_cfg(L.REGRESSION, data["labels"], 1, L.COMPAT_REFERENCE, L.F64, (strm["normals"], strm["gammas"], np.zeros(1)),
                                grp, ng)
        sc.rands = None; sc.n_rands = 0                                    # fm_train passes no rand() stream
        L.train_dev(gpu_ctx, m, d, sc, keep=keep)
        abi = m.get()
    finally:
        m.close(); d.close()
    assert fit["Model"]["w0"] == abi[0] and np.array_equal(fit["Model"]["w"], abi[1]) and np.array_equal(fit["Model"]["v"], abi[2].T)
    assert relerr(fit["Model"]["w"], plain["Model"]["w"]) > 1e-3            # the map reached the sampler
    for key in ("w0", "w", "v"):                                          # fm_posterior reads the map from the same place
        assert np.array_equal(post["fit"]["Model"][key], post_plain["Model"][key]), key
        assert np.array_equal(sgd["Model"][key], sgd_plain["Model"][key]), key
