"""Shared cases of the MCMC attribute-group tests: the data layouts of test_als_matches_oracle, two group maps per layout,
injected streams long enough for the grouped draw order, one engine run (fmwr_train_dev) with a map, and the runs of the two
fp64 restatements (the C one of the shipped one-group sampler, the numpy one of the grouped sampler)."""
import numpy as np

from fmwr_b200 import _lib as L
from fmwr_b200 import synth

LAYOUTS = ["fields", "fields_odd", "fields_sparse", "ragged"]
MAPS = ["fields", "scattered"]
K, SWEEPS = 4, 4


def layout(name):
    """(dataset dict, field sizes or None) -- the shapes test_als_matches_oracle uses"""
    if name == "fields":
        fields = [40, 25, 8]
        rowptr, col, val, p = synth.fields_csr(3000, fields, None, 1, 5)
        return dict(n=3000, p=p, rowptr=rowptr, col=col, val=val), fields
    if name == "fields_odd":
        fields = [40, 2500, 8]
        rowptr, col, val, p = synth.fields_csr(3001, fields, None, 1, 6)
        return dict(n=3001, p=p, rowptr=rowptr, col=col, val=val), fields
    if name == "fields_sparse":
        fields = [30, 20, 10]
        rowptr, col, val, p = synth.fields_csr(2000, fields, None, 1, 7)
        keep = np.ones(col.size, bool)
        keep[np.arange(0, col.size, 7)] = False
        cnt = np.add.reduceat(keep.astype(np.int64), rowptr[:-1].astype(np.int64))
        return dict(n=2000, p=p, rowptr=np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint32), col=col[keep], val=val[keep]), fields
    rowptr, col, val = synth.random_csr(600, 70, 6, seed=5, empty_rows=True)
    return dict(n=600, p=70, rowptr=rowptr, col=col, val=val), None


def group_map(kind, p, fields):
    """(attr_group int32[p], n_groups): "fields" = one group per field (three equal column ranges without fields);
    "scattered" = a seeded random map over five groups of which group 2 stays empty"""
    if kind == "fields":
        if fields is None:
            return (np.arange(p) * 3 // p).astype(np.int32), 3
        return np.repeat(np.arange(len(fields)), fields).astype(np.int32), len(fields)
    g = np.random.default_rng(17).choice(np.array([0, 1, 3, 4]), p).astype(np.int32)
    return g, 5


def problem(task, ds, seed=3):
    """labels and initial parameters (w0, w, V)"""
    rng = np.random.default_rng(seed)
    n, p = ds["n"], ds["p"]
    y = (np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == L.CLASSIFICATION else rng.normal(0, 1, n)).astype(np.float32)
    return y, 0.1, rng.normal(0, 0.1, p), rng.normal(0, 0.1, (p, K))


def streams(p, n_groups, sweeps=SWEEPS, k=K, seed=9):
    """standard normals, unit-scale gammas and rand() ints for `sweeps` grouped sweeps (with room to spare)"""
    rng = np.random.default_rng(seed)
    normals = rng.standard_normal(sweeps * (1 + n_groups + p + k * (n_groups + p)) + 64)
    gammas = rng.gamma(30.0, 1.0, sweeps * (1 + n_groups * (1 + k)) + 64)
    rands = rng.integers(0, 2**31 - 1, 400000).astype(np.int32)
    return normals, gammas, rands


def engine_cfg(task, y, enable_v, compat, prec, strm, attr_group, n_groups, sweeps=SWEEPS, step_size=-1):
    """(SolverCfg, arrays it points to)"""
    sc = L.SolverCfg(solver=L.MCMC, max_iter=sweeps, random_step=1, min_target=float(np.min(y)), max_target=float(np.max(y)),
                     mode=L.MODE_EXACT, precision=prec, compat=compat, enable_v=enable_v, step_size=step_size, metric=L.RMSE,
                     convergence=1e-4, seed=1)
    keep = []
    if strm is not None:
        nrm, gam, rnd = (np.ascontiguousarray(strm[0], np.float64), np.ascontiguousarray(strm[1], np.float64),
                         np.ascontiguousarray(strm[2], np.int32))
        keep += [nrm, gam, rnd]
        sc.normals = L.ptr(nrm); sc.n_normals = nrm.size
        sc.gammas = L.ptr(gam); sc.n_gammas = gam.size
        sc.rands = L.ptr(rnd); sc.n_rands = rnd.size
    if attr_group is not None:
        g = np.ascontiguousarray(attr_group, np.int32)
        keep.append(g)
        sc.attr_group = L.ptr(g)
    sc.n_groups = n_groups
    return sc, keep


def engine_run(ctx, task, ds, y, init, enable_v, compat, prec, strm, attr_group, n_groups, sweeps=SWEEPS):
    """fmwr_train_dev on a fresh data handle; returns (w0, w, V)"""
    w0, w, v = init
    d = L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y)
    m = L.Model(ctx, L.ModelCfg(task=task, keep_w0=1, keep_w1=1, k=K, l2_w0=0.1), ds["p"], prec)
    try:
        m.set(w0, w, v)
        sc, keep = engine_cfg(task, y, enable_v, compat, prec, strm, attr_group, n_groups, sweeps)
        L.train_dev(ctx, m, d, sc, keep=keep)
        return m.get()
    finally:
        m.close(); d.close()


def oracle_run(port, task, ds, y, init, enable_v, strm, sweeps=SWEEPS):
    """the C restatement of the shipped (one-group) sampler with the same streams; returns (w0, w, V)"""
    from oracle import oracle as O
    w0, w, v = init
    cfg = O.make_cfg(task=task, solver=O.MCMC, k=K, max_iter=sweeps, enable_v=enable_v, l2_w0=0.1,
                     min_target=float(np.min(y)), max_target=float(np.max(y)))
    port.set_streams(*strm)
    try:
        rw0, rw, rv, _ = port.train(cfg, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y, w0, w, v)
        assert port.stream_pos()["overrun"] == 0
    finally:
        port.set_streams(None, None, None)
    return rw0, rw, rv


def reference_run(port, task, ds, y, init, enable_v, compat, strm, attr_group, n_groups, sweeps=SWEEPS):
    """the fp64 restatement of the grouped sampler (tests/mcmc_groups_ref.py) with the same streams and map (None: one
    group); returns (w0, w, V)"""
    from tests import mcmc_groups_ref
    w0, w, v = init
    return mcmc_groups_ref.train(port, task, ds["n"], ds["p"], K, ds["rowptr"], ds["col"], ds["val"], y, w0, w, v, sweeps, enable_v, 0.1,
                                 strm, attr_group, n_groups, compat)
