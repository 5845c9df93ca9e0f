"""SGDA's numpy restatement on the CPU (tests/sgda_ref.py): its lambda gradients against finite differences of the look-ahead score,
the clamp at zero, the plain simultaneous-form loop it reduces to without lambda steps, and fm_train_sgda's argument checks, which
all fire before a device is needed."""
import numpy as np
import pytest

from fmwr_b200 import api
from tests import sgda_ref as R


def random_csr(n, p, nnz, rng, empty=()):
    rowptr = [0]
    cols, vals = [], []
    for r in range(n):
        c = np.sort(rng.choice(p, size=0 if r in empty else int(rng.integers(1, nnz + 1)), replace=False))
        cols.extend(c.tolist())
        vals.extend(rng.uniform(0.5, 1.5, c.size).astype(np.float32).tolist())
        rowptr.append(len(cols))
    return dict(rowptr=np.array(rowptr, np.uint32), col=np.array(cols, np.uint32), val=np.array(vals, np.float32))


def problem(rng, p=30, k=5, G=4):
    groups = rng.integers(0, G, p)
    state = dict(w0=0.2, w=rng.normal(0, 0.3, p), V=rng.normal(0, 0.3, (p, k)), gw=rng.normal(0, 0.5, p),
                 gv=rng.normal(0, 0.5, (p, k)), lam_w=rng.uniform(0, 0.5, G), lam_v=rng.uniform(0, 0.5, (G, k)))
    return groups, state


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("k1", [1, 0])
def test_lambda_gradients_match_finite_differences(seed, k1):
    rng = np.random.default_rng(seed)
    groups, st = problem(rng)
    cols = np.sort(rng.choice(30, 12, replace=False))
    x = rng.uniform(0.5, 1.5, cols.size)
    assert np.unique(groups[cols]).size > 1
    lr = 0.05

    def p1(lw, lv):
        return R.lookahead(st["w0"], st["w"], st["V"], st["gw"], st["gv"], lw, lv, groups, cols, x, lr, 1, k1)[0]

    _, dw, dv = R.lookahead(st["w0"], st["w"], st["V"], st["gw"], st["gv"], st["lam_w"], st["lam_v"], groups, cols, x, lr, 1, k1)
    h = 1e-4
    for g in range(st["lam_w"].size):
        lp, lm = st["lam_w"].copy(), st["lam_w"].copy()
        lp[g] += h; lm[g] -= h
        fd = (p1(lp, st["lam_v"]) - p1(lm, st["lam_v"])) / (2 * h)
        assert abs(fd - dw[g]) <= 1e-6 * max(abs(fd), 1e-3), (g, fd, dw[g])
        for f in range(st["lam_v"].shape[1]):
            vp, vm = st["lam_v"].copy(), st["lam_v"].copy()
            vp[g, f] += h; vm[g, f] -= h
            fd = (p1(st["lam_w"], vp) - p1(st["lam_w"], vm)) / (2 * h)
            assert abs(fd - dv[g, f]) <= 1e-6 * max(abs(fd), 1e-3), (g, f, fd, dv[g, f])
    absent = np.setdiff1d(np.arange(st["lam_w"].size), groups[cols])
    assert np.all(dw[absent] == 0) and np.all(dv[absent] == 0)


def data(rng, n, p, task, empty=()):
    ds = random_csr(n, p, 6, rng, empty)
    ds["y"] = (np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == R.CLASSIFICATION else rng.normal(0, 1, n)).astype(np.float32)
    return ds


def test_lambda_clamped_at_zero():
    rng = np.random.default_rng(5)
    p, k, G = 20, 3, 3
    tr, va = data(rng, 40, p, R.REGRESSION), data(rng, 15, p, R.REGRESSION)
    groups = rng.integers(0, G, p)
    w, V = rng.normal(0, 0.5, p), rng.normal(0, 0.5, (p, k))
    # from lambda = 0 every step that points below zero is clamped: some rates stay exactly 0, the rest moved up
    out = R.sgda(tr, va, R.REGRESSION, 0.0, w, V, np.zeros(G), np.zeros((G, k)), groups, 0.05, 4 * 39)
    lam = np.concatenate([out[3], out[4].ravel()])
    assert np.all(lam >= 0) and np.any(lam == 0) and np.any(lam > 0)


def plain_loop(tr, task, w0, w, V, lam_w, lam_v, groups, lr, iters):
    """the simultaneous-form step with fixed rates, written out entry by entry"""
    w, V = w.copy(), V.copy()
    n = len(tr["rowptr"]) - 1
    lo, hi = float(tr["y"].min()), float(tr["y"].max())
    for t in range(iters):
        r = t % (n - 1) + 1
        b, e = int(tr["rowptr"][r]), int(tr["rowptr"][r + 1])
        cols, x = tr["col"][b:e].astype(int), tr["val"][b:e].astype(float)
        S = np.array([sum(V[c, f] * xi for c, xi in zip(cols, x)) for f in range(V.shape[1])])
        p = w0 + sum(w[c] * xi for c, xi in zip(cols, x))
        p += 0.5 * sum(S[f] ** 2 - sum((V[c, f] * xi) ** 2 for c, xi in zip(cols, x)) for f in range(V.shape[1]))
        m = R.grad_mult(task, p, float(tr["y"][r]), lo, hi)
        Vold = V.copy()
        for c, xi in zip(cols, x):
            g = groups[c]
            w[c] -= lr * (m * xi + lam_w[g] * w[c])
            for f in range(V.shape[1]):
                V[c, f] -= lr * (m * (S[f] * xi - Vold[c, f] * xi * xi) + lam_v[g, f] * Vold[c, f])
        w0 -= lr * m
    return w0, w, V


@pytest.mark.parametrize("task", [R.CLASSIFICATION, R.REGRESSION])
def test_without_lambda_steps_equals_plain_loop(task):
    rng = np.random.default_rng(7)
    p, k, G = 25, 4, 3
    tr, va = data(rng, 30, p, task, empty=(4,)), data(rng, 10, p, task)
    groups = rng.integers(0, G, p)
    w, V = rng.normal(0, 0.2, p), rng.normal(0, 0.2, (p, k))
    lw, lv = rng.uniform(0, 0.1, G), rng.uniform(0, 0.1, (G, k))
    iters = 3 * 29 + 5
    got = R.sgda(tr, va, task, 0.1, w, V, lw, lv, groups, 0.05, iters, lambda_step=False)
    want = plain_loop(tr, task, 0.1, w, V, lw, lv, groups, 0.05, iters)
    assert abs(got[0] - want[0]) < 1e-12
    assert np.allclose(got[1], want[1], rtol=0, atol=1e-12) and np.allclose(got[2], want[2], rtol=0, atol=1e-12)
    assert np.array_equal(got[3], lw) and np.array_equal(got[4], lv)
    moved = R.sgda(tr, va, task, 0.1, w, V, lw, lv, groups, 0.05, iters)
    assert not np.array_equal(moved[3], lw)


def fm_data(rng, n=20, p=6, labels=True, groups=None):
    x = rng.uniform(0, 1, (n, p)) * (rng.random((n, p)) < 0.6)
    y = np.where(rng.random(n) < 0.5, 1.0, 0.0) if labels else None
    d = api.fm_matrix(x, y)
    if groups is not None:
        d["features"]["attr_group"] = np.asarray(groups)
    return d


def test_fm_train_sgda_argument_errors_before_the_device():
    rng = np.random.default_rng(0)
    tr, va = fm_data(rng), fm_data(rng)
    sgd = api.solver_control(solver=api.SGD_solver())
    with pytest.raises(ValueError, match="fm.matrix"):
        api.fm_train_sgda(tr, {"features": va["features"]}, control=[sgd])
    with pytest.raises(ValueError, match="SGD solver"):
        api.fm_train_sgda(tr, va, control=[api.solver_control(solver=api.FTRL_solver())])
    with pytest.raises(ValueError, match="SGD solver"):
        api.fm_train_sgda(tr, va)                                    # the default solver is TDAP
    with pytest.raises(ValueError, match="L1"):
        api.fm_train_sgda(tr, va, control=[sgd, api.model_control(L1_w1=0.1)])
    with pytest.raises(ValueError, match="L1"):
        api.fm_train_sgda(tr, va, control=[sgd, api.model_control(L1_v=0.1)])
    with pytest.raises(ValueError, match="no labels in newdata"):
        api.fm_train_sgda(tr, fm_data(rng, labels=False), control=[sgd])
    with pytest.raises(ValueError, match="training data"):
        api.fm_train_sgda(tr, tr, control=[sgd])
    with pytest.raises(ValueError, match="columns"):
        api.fm_train_sgda(tr, fm_data(rng, p=7), control=[sgd])
    with pytest.raises(ValueError, match="attr_group"):
        api.fm_train_sgda(fm_data(rng, groups=[0, 1, -1, 0, 1, 0]), va, control=[sgd])
    with pytest.raises(ValueError, match="attr_group"):
        api.fm_train_sgda(fm_data(rng, groups=[0, 1]), va, control=[sgd])
    with pytest.raises(ValueError, match="no labels in data"):
        api.fm_train_sgda(fm_data(rng, labels=False), va, control=[sgd])
    old = api.get_option("FM.mode")
    try:
        api.options(**{"FM.mode": "minibatch"})
        with pytest.raises(ValueError, match="exact mode"):
            api.fm_train_sgda(tr, va, control=[sgd])
    finally:
        api.options(**{"FM.mode": old})
