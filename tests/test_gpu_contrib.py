"""Per-feature contributions of the FM score (fmwr_contrib_dev / fmwr_contrib_fetch / api.fm_contrib).

phi_j = [k1] w_j x_j + 1/2 x_j sum_f v_jf (S_f - x_j v_jf) is checked three ways: against Shapley values enumerated over every
subset of small rows (which checks the closed form itself), against a numpy fp64 restatement of the closed form per entry, and
through the efficiency identity phi_0 + sum_j phi_j = the raw score of the existing forward.  Tolerances are the forward's:
1e-12 for fp64, 1e-5 relative with a max(1, |ref|) denominator for fp32."""
import math
import warnings

import numpy as np
import pytest

from fmwr_b200 import _lib as L
from fmwr_b200 import api as A
from fmwr_b200 import synth
from tests.util import relerr


def _tol(prec):
    return 1e-5 if prec == L.F32 else 1e-12


def _stored(a, prec):
    """the parameters as a handle of this precision stores them"""
    a = np.asarray(a, np.float64)
    return a.astype(np.float32).astype(np.float64) if prec == L.F32 else a


def _closed_form(n, rowptr, col, val, w, v, k1=1):
    """numpy fp64 restatement of phi_j"""
    col = np.asarray(col, np.int64)
    x = np.asarray(val, np.float32).astype(np.float64)
    rows = np.repeat(np.arange(n), np.diff(np.asarray(rowptr, np.int64)))
    vj = v[col]
    S = np.zeros((n, v.shape[1]))
    np.add.at(S, rows, vj * x[:, None])
    return k1 * w[col] * x + 0.5 * x * (np.einsum("ij,ij->i", vj, S[rows]) - x * (vj * vj).sum(1))


def _contrib(ctx, prec, n, p, rowptr, col, val, w0, w, v, k0=1, k1=1):
    """(phi, score left in the handle, predict_dev(LINK_NONE) on the same handle afterwards)"""
    d = L.Data.from_csr32(ctx, n, p, rowptr, col, val)
    m = L.Model(ctx, L.ModelCfg(task=L.CLASSIFICATION, keep_w0=k0, keep_w1=k1, k=v.shape[1]), p, prec)
    m.set(w0, w, v)
    L.contrib_dev(ctx, m, d)
    phi = L.contrib_fetch(ctx, d)
    score = L.predict_fetch(ctx, d)
    L.predict_dev(ctx, m, d, L.LINK_NONE)
    pred = L.predict_fetch(ctx, d)
    m.close(); d.close()
    return phi, score, pred


def _check(ctx, prec, n, p, rowptr, col, val, w0, w, v, k0=1, k1=1):
    phi, score, pred = _contrib(ctx, prec, n, p, rowptr, col, val, w0, w, v, k0, k1)
    rowptr = np.asarray(rowptr, np.int64)
    assert phi.shape == (int(rowptr[-1]),) and score.shape == (n,)
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    sums = k0 * float(_stored([w0], prec)[0]) + np.bincount(rows, weights=phi, minlength=n)
    assert relerr(sums, pred) < _tol(prec)
    assert relerr(score, pred) < _tol(prec)
    want = _closed_form(n, rowptr, col, val, _stored(w, prec), _stored(v, prec), k1)
    assert relerr(phi, want) < _tol(prec)
    return phi


def _rows(lengths, p, seed):
    """CSR with the given row lengths, ascending unique columns, values in [-1.5, 1.5]"""
    rng = np.random.default_rng(seed)
    col = [np.sort(rng.choice(p, size=m, replace=False)) for m in lengths]
    rowptr = np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint32)
    col = np.concatenate(col).astype(np.uint32) if col else np.zeros(0, np.uint32)
    return rowptr, col, rng.uniform(-1.5, 1.5, col.size).astype(np.float32)


@pytest.mark.gpu
def test_contrib_known_answers(gpu_ctx):
    # the pattern of the reference's scratch test (src/test/model.cpp:12-34): w = 0.1, v = 0.2, k = 3
    rowptr = [0, 2, 3]
    col = [0, 3, 0]
    val = [1.0, 1.0, 2.0]
    w, v = np.full(4, 0.1), np.full((4, 3), 0.2)
    for prec, tol in ((L.F32, 1e-6), (L.F64, 1e-14)):
        phi, score, _ = _contrib(gpu_ctx, prec, 2, 4, rowptr, col, val, 0.0, w, v)
        assert np.max(np.abs(phi - [0.16, 0.16, 0.2])) < tol
        assert np.max(np.abs(score - [0.32, 0.2])) < tol


def _shapley(c, x, w0, w, v, k0, k1):
    """Shapley values of v(T) = the FM score of the row restricted to the entries in T, by enumeration of every subset"""
    m = len(c)
    A_ = v[c] * x[:, None]
    G = A_ @ A_.T
    lin = k1 * w[c] * x
    masks = np.arange(1 << m)
    M = ((masks[:, None] >> np.arange(m)) & 1).astype(np.float64)
    val = k0 * w0 + M @ lin + 0.5 * (np.einsum("ti,ij,tj->t", M, G, M) - M @ np.diag(G))
    size = M.sum(1).astype(int)
    wt = np.array([math.factorial(s) * math.factorial(m - s - 1) / math.factorial(m) for s in range(m)])
    phi = np.zeros(m)
    for j in range(m):
        without = masks[(masks >> j) & 1 == 0]
        phi[j] = np.sum(wt[size[without]] * (val[without | (1 << j)] - val[without]))
    return phi


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 3, 8])
def test_contrib_equals_brute_force_shapley(gpu_ctx, k):
    rng = np.random.default_rng(40 + k)
    p = 40
    lengths = [m for m in range(1, 11) for _ in range(3)]
    rowptr, col, val = _rows(lengths, p, seed=k)
    w, v, w0 = rng.normal(0, 0.5, p), rng.normal(0, 0.4, (p, k)), 0.3
    phi, _, _ = _contrib(gpu_ctx, L.F64, len(lengths), p, rowptr, col, val, w0, w, v)
    for r in range(len(lengths)):
        b, e = int(rowptr[r]), int(rowptr[r + 1])
        want = _shapley(col[b:e].astype(np.int64), val[b:e].astype(np.float64), w0, w, v, 1, 1)
        assert np.all(np.abs(phi[b:e] - want) <= 1e-12 * np.maximum(1.0, np.abs(want))), r


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1, 2, 3, 8, 10, 29, 30, 32, 33, 64, 100, 128, 200])
@pytest.mark.parametrize("prec", [L.F32, L.F64])
def test_contrib_matches_the_forward(gpu_ctx, k, prec):
    # the ragged CSR (with empty rows) of test_forward_random_ragged
    rng = np.random.default_rng(k + 7)
    n, p = 700, 300
    rowptr, col, val = synth.random_csr(n, p, 45, seed=k, empty_rows=True)
    w = rng.normal(0, 0.3, p); v = rng.normal(0, 0.2, (p, k)); w0 = 0.25
    _check(gpu_ctx, prec, n, p, rowptr, col, val, w0, w, v)


# (precision, k, row lengths): the team layouts of forward_launch's dispatch and both paths of the batched gathers
LAYOUTS = {
    "short_lpr8": (L.F32, 32, [1, 2, 5, 0, 7, 3, 4, 16, 8, 12]),             # one row per 8-lane group; 4 and 16: full batches only
    "short_lpr1": (L.F32, 3, [1, 9, 4, 0, 30, 8, 2]),                         # one lane per row
    "short_f64_lpr4": (L.F64, 8, [3, 1, 8, 0, 12, 5]),
    "long_half_warp": (L.F32, 32, [48, 40, 17, 0, 63, 33, 8, 96]),            # two 8-lane sub-groups per row; 8 entries per batch
    "long_half_warp_f64": (L.F64, 3, [130, 96, 70, 0, 150, 65, 1, 128]),     # 2-lane groups: long past 64 entries a row
    "k64_lpr16": (L.F32, 64, [48, 40, 17, 0, 63, 33, 8, 96]),                 # one row per 16-lane group
    "warp_ch1": (L.F32, 128, [48, 40, 17, 0, 63, 33, 1, 96]),                 # one row per warp, 8 entries per batch
    "warp_ch2": (L.F32, 256, [48, 40, 17, 0, 63, 33, 1, 96]),
    "warp_ch4_f64": (L.F64, 256, [48, 40, 17, 0, 63, 33, 1, 96]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_contrib_team_layouts(gpu_ctx, layout):
    prec, k, lengths = LAYOUTS[layout]
    lengths = lengths * 40
    p = 500
    rng = np.random.default_rng(len(layout))
    rowptr, col, val = _rows(lengths, p, seed=k)
    w = rng.normal(0, 0.3, p); v = rng.normal(0, 0.2, (p, k)); w0 = -0.1
    _check(gpu_ctx, prec, len(lengths), p, rowptr, col, val, w0, w, v)


@pytest.mark.gpu
def test_contrib_criteo_shape(gpu_ctx):
    ds = synth.make_dataset("criteo", 20000, p=39 * 2000)
    rng = np.random.default_rng(0)
    k = 32
    w = rng.normal(0, 0.1, ds["p"]); v = rng.normal(0, 0.05, (ds["p"], k))
    _check(gpu_ctx, L.F32, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], 0.2, w, v)


@pytest.mark.gpu
@pytest.mark.parametrize("k0,k1", [(0, 0), (0, 1), (1, 0)])
def test_contrib_keep_flags(gpu_ctx, k0, k1):
    rng = np.random.default_rng(3)
    n, p, k = 200, 80, 8
    rowptr, col, val = synth.random_csr(n, p, 10, seed=9)
    w = rng.normal(0, 0.3, p); v = rng.normal(0, 0.2, (p, k)); w0 = -0.4
    _check(gpu_ctx, L.F64, n, p, rowptr, col, val, w0, w, v, k0, k1)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [L.F32, L.F64])
def test_contrib_explicit_zeros_and_empty_handles(gpu_ctx, prec):
    rng = np.random.default_rng(5)
    n, p, k = 300, 60, 8
    rowptr, col, val = synth.random_csr(n, p, 20, seed=6, empty_rows=True)
    zero = np.arange(0, col.size, 3)
    val[zero] = 0.0
    w = rng.normal(0, 0.3, p); v = rng.normal(0, 0.2, (p, k))
    phi = _check(gpu_ctx, prec, n, p, rowptr, col, val, 0.5, w, v)
    assert np.all(phi[zero] == 0.0)
    # no rows
    phi, score, pred = _contrib(gpu_ctx, prec, 0, p, [0], [], [], 0.5, w, v)
    assert phi.size == 0 and score.size == 0 and pred.size == 0
    # rows but no entries: every score is w0
    phi, score, pred = _contrib(gpu_ctx, prec, 7, p, np.zeros(8), [], [], 0.5, w, v)
    assert phi.size == 0 and np.all(score == 0.5) and np.all(pred == 0.5)


@pytest.mark.gpu
def test_contrib_errors_leave_the_handle_untouched(gpu_ctx):
    lib = L.lib()
    rowptr, col, val = synth.random_csr(10, 20, 3, seed=1)
    d = L.Data.from_csr32(gpu_ctx, 10, 20, rowptr, col, val)
    m = L.Model(gpu_ctx, L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=2), 20, L.F64)
    m.set(0.1, np.full(20, 0.2), np.full((20, 2), 0.1))
    wide = L.Model(gpu_ctx, L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=2), 21, L.F64)
    L.predict_dev(gpu_ctx, m, d, L.LINK_LOGISTIC)
    before = L.predict_fetch(gpu_ctx, d)
    with pytest.raises(L.FmwrError) as e:                          # fetch before any fmwr_contrib_dev on this handle
        L.contrib_fetch(gpu_ctx, d)
    assert e.value.code == 1
    with pytest.raises(L.FmwrError) as e:                          # width mismatch: the predict message
        L.contrib_dev(gpu_ctx, wide, d)
    assert e.value.code == 3 and "features is not correct" in str(e.value)
    assert lib.fmwr_contrib_dev(None, m.h, d.h) == 1
    assert lib.fmwr_contrib_dev(gpu_ctx.h, None, d.h) == 1
    assert lib.fmwr_contrib_dev(gpu_ctx.h, m.h, None) == 1
    assert lib.fmwr_contrib_fetch(None, d.h, L.ptr(np.zeros(d.shape()[2]))) == 1
    assert lib.fmwr_contrib_fetch(gpu_ctx.h, None, L.ptr(np.zeros(d.shape()[2]))) == 1
    with pytest.raises(L.FmwrError) as e:                          # still nothing computed, and the forward result kept
        L.contrib_fetch(gpu_ctx, d)
    assert e.value.code == 1
    assert np.array_equal(L.predict_fetch(gpu_ctx, d), before)
    L.contrib_dev(gpu_ctx, m, d)
    assert lib.fmwr_contrib_fetch(gpu_ctx.h, d.h, None) == 1
    assert L.contrib_fetch(gpu_ctx, d).size == d.shape()[2]
    wide.close(); m.close(); d.close()


# ---- host API -------------------------------------------------------------------------------------------------------
def _host_data(seed, n, p=10, task="CLASSIFICATION"):
    rng = np.random.default_rng(seed)
    x = rng.normal(0, 1, (n, p)) * (rng.random((n, p)) < 0.6) * np.linspace(0.5, 20.0, p)   # column scales z-scoring changes
    s = x @ np.random.default_rng(99).normal(0, 0.1, p) + 0.3 * rng.normal(0, 1, n)
    return A.fm_matrix(x, (s > 0).astype(np.float64) if task == "CLASSIFICATION" else s)


def test_fm_contrib_argument_errors():
    """predict's checks, raised before any GPU work"""
    fit = A.FM(Model={}, Scales={"mean": None})
    new = _host_data(1, 20)
    with pytest.raises(ValueError, match="newdata is null"):
        A.fm_contrib(fit, None)
    with pytest.raises(ValueError, match="fm.matrix"):
        A.fm_contrib(fit, dict(new))
    bad = A.fm_matrix(np.eye(3))
    bad["features"]["value"][0] = np.nan
    with pytest.raises(ValueError, match="NAs"):
        A.fm_contrib(fit, bad)
    with pytest.raises(ValueError, match="can not normalize"):
        A.fm_contrib(fit, new, normalize=True)


def _row_sums(r):
    return r["bias"] + np.asarray(r["contrib"].sum(1)).ravel()


@pytest.mark.gpu
def test_fm_contrib_classification_sgd(gpu_ctx):
    data, new = _host_data(3, 300), _host_data(4, 200)
    ctl = [A.model_control("CLASSIFICATION", factor_number=3), A.solver_control(max_iter=700, solver=A.SGD_solver()), A.track_control()]
    fit = A.fm_train(data, True, ctl)
    ctx = A._ctx()
    before = A.predict(fit, new)
    r = A.fm_contrib(fit, new)
    h2d = ctx.transfer_bytes()[0]
    r2 = A.fm_contrib(fit, new)
    p, k = new.ncol(), 3
    assert ctx.transfer_bytes()[0] - h2d == 8 + 8 * p + 8 * p * k          # the model only: X stays parked
    assert np.array_equal(r2["contrib"].data, r["contrib"].data) and np.array_equal(r2["score"], r["score"])
    assert np.array_equal(A.predict(fit, new), before)
    assert np.max(np.abs(_row_sums(r) - np.log(before / (1.0 - before)))) < 1e-9
    assert np.max(np.abs(_row_sums(r) - r["score"])) < 1e-12
    assert r["bias"] == fit["Model"]["w0"] and np.std(r["contrib"].data) > 0
    feats = new["features"]
    c = r["contrib"]
    assert c.shape == tuple(feats["dim"])
    assert np.array_equal(c.indptr, np.concatenate([[0], np.cumsum(feats["row_size"])]))
    assert np.array_equal(c.indices, feats["col_idx"])
    # unscaled newdata against a normalised model: predict's warning, and the contributions of the raw values
    with warnings.catch_warnings(record=True) as wr:
        warnings.simplefilter("always")
        raw = A.fm_contrib(fit, new, normalize=False)
    assert any("will not" in str(x.message) for x in wr)
    assert not np.allclose(raw["contrib"].data, r["contrib"].data)


@pytest.mark.gpu
@pytest.mark.parametrize("solver", ["ALS", "MCMC"])
def test_fm_contrib_als_mcmc(gpu_ctx, solver):
    data, new = _host_data(5, 300, task="REGRESSION"), _host_data(6, 150, task="REGRESSION")
    s = A.ALS_solver() if solver == "ALS" else A.MCMC_solver()
    ctl = [A.model_control("REGRESSION", factor_number=4), A.solver_control(max_iter=5, solver=s), A.track_control()]
    fit = A.fm_train(data, True, ctl)
    r = A.fm_contrib(fit, new)
    # predict_dev(LINK_NONE) on the handle fm_contrib z-scored (parked in newdata)
    ctx = A._ctx()
    d = new["features"]["_handle"]["data"]
    md = fit["Model"]
    m = L.Model(ctx, A._model_cfg(md["model.control"]), new.ncol(), L.F64)
    m.set(float(md["w0"]), np.asarray(md["w"]), np.asarray(md["v"]).T.copy())
    L.predict_dev(ctx, m, d, L.LINK_NONE)
    want = L.predict_fetch(ctx, d)
    m.close()
    assert relerr(_row_sums(r), want) < 1e-12 and relerr(r["score"], want) < 1e-12
    assert np.array_equal(r["contrib"].indices, new["features"]["col_idx"])
