"""SGDA on the device (fmwr_train_sgda_dev, csrc/train_sgda.cu) against its fp64 numpy restatement (tests/sgda_ref.py).

Every case runs more than two passes over the training rows, so lambda steps run and the validation set wraps.  The data has
rows longer than one round of the kernel's slots (and than its staged ring), empty rows in both sets, and validation sets smaller
and larger than the training set."""
import ctypes

import numpy as np
import pytest

from fmwr_b200 import _lib as L
from fmwr_b200 import api
from tests import sgda_ref as R
from tests.util import relerr

pytestmark = pytest.mark.gpu

P, FIELDS = 600, 6                      # features 100 f .. 100 f + 99 form field f


def make_set(rng, n, task, long_row, empty_row, nnz=24):
    rowptr, cols, vals = [0], [], []
    for r in range(n):
        size = 0 if r == empty_row else (500 if r == long_row else int(rng.integers(1, nnz + 1)))
        c = np.sort(rng.choice(P, size=size, replace=False))
        cols.extend(c.tolist())
        vals.extend((rng.uniform(0.5, 1.5, size) * (0.05 if r == long_row else 1.0)).tolist())   # keeps the long row's score bounded
        rowptr.append(len(cols))
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == R.CLASSIFICATION else rng.normal(0, 1, n)
    return dict(rowptr=np.array(rowptr, np.uint32), col=np.array(cols, np.uint32), val=np.array(vals, np.float32),
                y=y.astype(np.float32))


def group_map(kind, rng):
    if kind == "one":
        return None, 1
    if kind == "field":
        return (np.arange(P) // (P // FIELDS)).astype(np.int32), FIELDS
    return rng.integers(0, 5, P).astype(np.int32), 5                # scattered


def engine(ctx, prec, tr, va, task, k, w0, w, V, lam_w, lam_v, grp, lr, max_iter, k0=1, k1=1, compat=L.COMPAT_REFERENCE,
           visit=None, step_size=-1, convergence=1e-4, metric=L.LL, random_step=1):
    d = L.Data.from_csr32(ctx, len(tr["rowptr"]) - 1, P, tr["rowptr"], tr["col"], tr["val"], tr["y"])
    dv = L.Data.from_csr32(ctx, len(va["rowptr"]) - 1, P, va["rowptr"], va["col"], va["val"], va["y"])
    m = L.Model(ctx, L.ModelCfg(task=task, keep_w0=k0, keep_w1=k1, k=k), P, prec)
    m.set(w0, w, V)
    sc = L.SolverCfg(solver=L.SGD, max_iter=max_iter, random_step=random_step, learn_rate=lr, min_target=float(tr["y"].min()),
                     max_target=float(tr["y"].max()), mode=L.MODE_EXACT, precision=prec, compat=compat, step_size=step_size,
                     metric=metric, convergence=convergence)
    keep = []
    if grp is not None:
        keep.append(grp)
        sc.attr_group = L.ptr(grp); sc.n_groups = int(grp.max()) + 1
    if visit is not None:
        vo = np.ascontiguousarray(visit, np.uint32)
        keep.append(vo)
        sc.visit_order = L.ptr(vo); sc.n_visit = vo.size
    lw, lv = np.array(lam_w, np.float64), np.array(lam_v, np.float64)
    tr_buf = L.TraceBuf(100) if step_size > 0 else None
    L.train_sgda_dev(ctx, m, d, sc, dv, lw, lv, tr_buf, keep=keep)
    gw0, gw, gv = m.get()
    solver, _ = m.state_info()
    m.close(); d.close(); dv.close()
    return dict(w0=gw0, w=gw, V=gv, lam_w=lw, lam_v=lv, solver=solver, trace=tr_buf.result() if tr_buf else None)


def reference(tr, va, task, w0, w, V, lam_w, lam_v, grp, lr, iters, **kw):
    G = lam_w.size
    groups = grp if grp is not None else np.zeros(P, np.int64)
    assert groups.max() < G
    out = R.sgda(tr, va, task, w0, w, V, lam_w, lam_v, groups, lr, iters, **kw)
    return dict(zip(("w0", "w", "V", "lam_w", "lam_v"), out))


def worst(a, b):
    return max(relerr(a[key], b[key]) for key in ("w0", "w", "V", "lam_w", "lam_v"))


def setup(task, k, gkind, seed, n=70, n_val=31, lam0=0.02):
    rng = np.random.default_rng(seed)
    tr = make_set(rng, n, task, long_row=3, empty_row=5)
    va = make_set(rng, n_val, task, long_row=2, empty_row=1)
    grp, G = group_map(gkind, rng)
    w = rng.normal(0, 0.1, P); V = rng.normal(0, 0.1, (P, k))
    lam_w = np.full(G, lam0) if lam0 else np.zeros(G)
    lam_v = np.full((G, k), lam0) if lam0 else np.zeros((G, k))
    return tr, va, grp, w, V, lam_w, lam_v


LR = 0.05


# k -> fp64 layout: 2: LPR 1, 4: 2, 8: 4, 16: 8, 32: 16, 64: 32, 128: LPR 32 and CH 2
@pytest.mark.parametrize("task", [R.CLASSIFICATION, R.REGRESSION])
@pytest.mark.parametrize("k", [2, 4, 8, 16, 32, 64, 128])
@pytest.mark.parametrize("gkind", ["one", "field", "scattered"])
def test_fp64_matches_reference(gpu_ctx, task, k, gkind):
    tr, va, grp, w, V, lam_w, lam_v = setup(task, k, gkind, seed=k)
    iters = int(3.4 * 69)
    got = engine(gpu_ctx, L.F64, tr, va, task, k, 0.1, w, V, lam_w, lam_v, grp, LR, iters)
    want = reference(tr, va, task, 0.1, w, V, lam_w, lam_v, grp, LR, iters)
    assert all(np.all(np.isfinite(want[key])) for key in want)
    assert worst(got, want) < 1e-8, worst(got, want)
    frozen = reference(tr, va, task, 0.1, w, V, lam_w, lam_v, grp, LR, iters, lambda_step=False)
    assert worst(got, frozen) > 1e-5                                    # negative control: the lambda steps matter
    assert got["solver"] == 0


VARIANTS = {
    "f5_off": dict(compat=0),
    "keep_w0_off": dict(k0=0),
    "keep_w1_off": dict(k1=0),
    "lambda0_zero": dict(lam0=0.0),
    "n_val_larger": dict(n=40, n_val=90),
    "random_step": dict(random_step=3),
    "tracker_mid_pass": dict(step_size=47),
    "converges": dict(step_size=30, convergence=1e30),            # the rule holds from the third record: stops at sample 120
}


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("task", [R.CLASSIFICATION, R.REGRESSION])
def test_fp64_variants(gpu_ctx, variant, task):
    opt = dict(VARIANTS[variant])
    n, n_val, lam0 = opt.pop("n", 70), opt.pop("n_val", 31), opt.pop("lam0", 0.02)
    tr, va, grp, w, V, lam_w, lam_v = setup(task, 8, "field", seed=11, n=n, n_val=n_val, lam0=lam0)
    passes = 3.5 if variant != "n_val_larger" else 4.5                  # n_val > n still wraps
    iters = int(passes * (n - 1))
    visit = None
    if opt.pop("random_step", 1) > 1:
        rng = np.random.default_rng(4)
        visit = np.concatenate([np.cumsum(rng.integers(1, 4, 40)) for _ in range(2)])   # random_step = 3 strides, two sweeps
        visit = visit[visit < n].astype(np.uint32)
    kw = {key: opt[key] for key in ("k0", "k1", "compat") if key in opt}
    got = engine(gpu_ctx, L.F64, tr, va, task, 8, 0.1, w, V, lam_w, lam_v, grp, LR, iters, visit=visit,
                 step_size=opt.get("step_size", -1), convergence=opt.get("convergence", 1e-4), **kw)
    done = iters
    if got["trace"] is not None:
        done = got["trace"]["iters_done"]
        if variant == "converges":
            assert got["trace"]["convergent"] and done < iters
        else:
            assert done == iters and got["trace"]["n_rec"] > 3
    ref_kw = dict(k0=kw.get("k0", 1), k1=kw.get("k1", 1), skip_row0=kw.get("compat", L.COMPAT_REFERENCE) & L.COMPAT_SKIP_ROW0 != 0,
                  order=visit)
    want = reference(tr, va, task, 0.1, w, V, lam_w, lam_v, grp, LR, done, **ref_kw)
    assert worst(got, want) < 1e-8, worst(got, want)
    if variant == "keep_w1_off":
        assert np.array_equal(got["lam_w"], lam_w)
    frozen = reference(tr, va, task, 0.1, w, V, lam_w, lam_v, grp, LR, done, lambda_step=False, **ref_kw)
    assert worst(got, frozen) > 1e-5


def random_step_order(seed, step, n, max_iter):
    """the visit sequence of random_step > 1 (train_exact.cu: visit_order_host) from glibc rand() after srand(seed)"""
    libc = ctypes.CDLL(None)
    libc.srand(seed)
    draw = lambda: int((libc.rand() / 2147483648.0) * step + 1)     # noqa: E731
    order = []
    while len(order) < max_iter:
        i = draw()
        while i < n and len(order) < max_iter:
            order.append(i)
            i += draw()
    return np.array(order, np.uint32)


@pytest.mark.parametrize("task", [R.CLASSIFICATION, R.REGRESSION])
def test_fp64_random_step_sequence(gpu_ctx, task):
    """random_step > 1 without an explicit order: the sweeps are cut at max_iter, and T0 is the first sweep"""
    tr, va, grp, w, V, lam_w, lam_v = setup(task, 8, "scattered", seed=13)
    n, step, iters = 70, 3, 180
    ctypes.CDLL(None).srand(77)
    got = engine(gpu_ctx, L.F64, tr, va, task, 8, 0.1, w, V, lam_w, lam_v, grp, LR, iters, random_step=step)
    order = random_step_order(77, step, n, iters)
    t0 = int(np.argmax(np.diff(order.astype(np.int64)) <= 0)) + 1
    assert 20 < t0 < 60 and order.size == iters                       # a sweep of ~n/2 rows, then more sweeps
    want = reference(tr, va, task, 0.1, w, V, lam_w, lam_v, grp, LR, iters, order=order, t0=t0)
    assert worst(got, want) < 1e-8, worst(got, want)
    assert not np.array_equal(got["lam_w"], lam_w) and not np.array_equal(got["lam_v"], lam_v)
    frozen = reference(tr, va, task, 0.1, w, V, lam_w, lam_v, grp, LR, iters, order=order, t0=t0, lambda_step=False)
    assert worst(got, frozen) > 1e-5


def test_host_mirror_random_step_moves_the_rates(gpu_ctx):
    rng = np.random.default_rng(14)
    n, p = 120, 30
    x = rng.uniform(0, 2, (n, p)) * (rng.random((n, p)) < 0.3)
    xv = rng.uniform(0, 2, (40, p)) * (rng.random((40, p)) < 0.3)
    data = api.fm_matrix(x, rng.normal(0, 1, n))
    valid = api.fm_matrix(xv, rng.normal(0, 1, 40))
    ctl = [api.model_control(task="REGRESSION", factor_number=4, L2_w1=0.01, L2_v=0.01),
           api.solver_control(max_iter=600, solver=api.SGD_solver(learn_rate=0.05, random_step=3))]
    fit = api.fm_train_sgda(data, valid, control=ctl)
    assert not np.array_equal(fit["Model"]["reg"]["w"], [0.01]) and not np.all(fit["Model"]["reg"]["v"] == 0.01)


@pytest.mark.parametrize("k", [4, 16, 128])
@pytest.mark.parametrize("task", [R.CLASSIFICATION, R.REGRESSION])
def test_fp32_within_tolerance(gpu_ctx, task, k):
    # lr = 0.02: at 0.05 the k = 128 regression run is so ill-conditioned that a one-ulp fp32 perturbation of the initial model
    # alone moves the fp64 reference by 2.6e-5, which says nothing about the kernel (at 0.02: 1e-7)
    lr = 0.02
    tr, va, grp, w, V, lam_w, lam_v = setup(task, k, "field", seed=20 + k)
    w, V = w.astype(np.float32).astype(np.float64), V.astype(np.float32).astype(np.float64)
    iters = int(3.4 * 69)
    got = engine(gpu_ctx, L.F32, tr, va, task, k, 0.1, w, V, lam_w, lam_v, grp, lr, iters)
    want = reference(tr, va, task, 0.1, w, V, lam_w, lam_v, grp, lr, iters)
    par = max(relerr(got[key], want[key]) for key in ("w0", "w", "V"))
    lam = max(relerr(got[key], want[key]) for key in ("lam_w", "lam_v"))
    print("fp32 SGDA k=%d task=%d: parameters %.3g, lambdas %.3g" % (k, task, par, lam))
    assert par < 1e-4
    assert lam < 1e-4


@pytest.mark.parametrize("prec", [L.F32, L.F64])
def test_repeatable(gpu_ctx, prec):
    tr, va, grp, w, V, lam_w, lam_v = setup(R.CLASSIFICATION, 16, "scattered", seed=3)
    runs = [engine(gpu_ctx, prec, tr, va, R.CLASSIFICATION, 16, 0.1, w, V, lam_w, lam_v, grp, LR, 250, step_size=60)
            for _ in range(2)]
    for key in ("w0", "w", "V", "lam_w", "lam_v"):
        assert np.array_equal(runs[0][key], runs[1][key]), key


def test_state_after_call_and_sgd_still_refuses_groups(gpu_ctx):
    tr, va, grp, w, V, lam_w, lam_v = setup(R.CLASSIFICATION, 4, "field", seed=8)
    d = L.Data.from_csr32(gpu_ctx, len(tr["rowptr"]) - 1, P, tr["rowptr"], tr["col"], tr["val"], tr["y"])
    dv = L.Data.from_csr32(gpu_ctx, len(va["rowptr"]) - 1, P, va["rowptr"], va["col"], va["val"], va["y"])
    m = L.Model(gpu_ctx, L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=4), P, L.F64)
    m.set(0.0, w, V)
    sc = L.SolverCfg(solver=L.SGD, max_iter=50, random_step=1, learn_rate=LR, min_target=-1, max_target=1, mode=L.MODE_EXACT,
                     precision=L.F64, compat=L.COMPAT_REFERENCE, step_size=-1)
    L.train_dev(gpu_ctx, m, d, sc)                                      # plain SGD first: its state (none without L1)
    sc.attr_group = L.ptr(grp); sc.n_groups = FIELDS
    L.train_sgda_dev(gpu_ctx, m, d, sc, dv, lam_w, lam_v)
    assert m.state_info()[0] == 0
    with pytest.raises(L.FmwrError, match="attribute groups need the MCMC solver") as e:
        L.train_dev(gpu_ctx, m, d, sc)
    assert e.value.code == 1
    m.close(); d.close(); dv.close()


def test_argument_errors_leave_model_and_lambdas(gpu_ctx):
    tr, va, grp, w, V, lam_w, lam_v = setup(R.REGRESSION, 4, "field", seed=9)
    n, nv = len(tr["rowptr"]) - 1, len(va["rowptr"]) - 1
    d = L.Data.from_csr32(gpu_ctx, n, P, tr["rowptr"], tr["col"], tr["val"], tr["y"])
    dv = L.Data.from_csr32(gpu_ctx, nv, P, va["rowptr"], va["col"], va["val"], va["y"])
    unlabelled = L.Data.from_csr32(gpu_ctx, nv, P, va["rowptr"], va["col"], va["val"])
    empty = L.Data.from_csr32(gpu_ctx, 0, P, np.zeros(1, np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.float32),
                              np.zeros(0, np.float32))
    narrow = L.Data.from_csr32(gpu_ctx, 1, P - 1, np.array([0, 1], np.uint32), np.array([0], np.uint32),
                               np.array([1], np.float32), np.array([1], np.float32))

    def base(**kw):
        sc = L.SolverCfg(solver=L.SGD, max_iter=200, random_step=1, learn_rate=LR, min_target=-3, max_target=3,
                         mode=L.MODE_EXACT, precision=L.F64, compat=L.COMPAT_REFERENCE, step_size=-1)
        sc.attr_group = L.ptr(grp); sc.n_groups = FIELDS
        for key, val in kw.items():
            setattr(sc, key, val)
        return sc

    bad_grp = grp.copy(); bad_grp[7] = FIELDS
    neg, nan = lam_v.copy(), lam_w.copy()
    neg[1, 2] = -1e-3; nan[0] = np.nan
    cases = [  # (code, cfg, model regs, valid, lambda_w, lambda_v)
        (1, base(solver=L.FTRL), {}, dv, lam_w, lam_v),
        (1, base(mode=L.MODE_MINIBATCH), {}, dv, lam_w, lam_v),
        (1, base(warm_state=1), {}, dv, lam_w, lam_v),
        (1, base(), dict(l1_w1=0.1), dv, lam_w, lam_v),
        (1, base(), dict(l1_v=0.1), dv, lam_w, lam_v),
        (1, base(), {}, None, lam_w, lam_v),
        (1, base(), {}, unlabelled, lam_w, lam_v),
        (1, base(), {}, d, lam_w, lam_v),
        (1, base(), {}, empty, lam_w, lam_v),
        (1, base(), {}, dv, None, lam_v),
        (1, base(), {}, dv, lam_w, None),
        (1, base(), {}, dv, nan, lam_v),
        (1, base(), {}, dv, lam_w, neg),
        (1, base(attr_group=L.ptr(bad_grp)), {}, dv, lam_w, lam_v),
        (1, base(n_groups=0), {}, dv, lam_w, lam_v),
        (3, base(), {}, narrow, lam_w, lam_v),
    ]
    for code, sc, regs, valid, lw, lv in cases:
        m = L.Model(gpu_ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=4, **regs), P, L.F64)
        m.set(0.25, w, V)
        before = m.get()
        lw_in = None if lw is None else lw.copy()
        lv_in = None if lv is None else lv.copy()
        with pytest.raises(L.FmwrError) as e:
            L.train_sgda_dev(gpu_ctx, m, d, sc, valid, lw_in, lv_in)
        assert e.value.code == code, (code, str(e.value))
        after = m.get()
        assert after[0] == before[0] and np.array_equal(after[1], before[1]) and np.array_equal(after[2], before[2])
        if lw is not None:
            assert lw_in.tobytes() == lw.tobytes()
        if lv is not None:
            assert lv_in.tobytes() == lv.tobytes()
        m.close()
    for h in (d, dv, unlabelled, empty, narrow):
        h.close()


def test_host_mirror_matches_abi(gpu_ctx):
    rng = np.random.default_rng(12)
    n, nv, p, k = 120, 50, 40, 4
    x = rng.uniform(0, 3, (n, p)) * (rng.random((n, p)) < 0.3)
    xv = rng.uniform(0, 3, (nv, p)) * (rng.random((nv, p)) < 0.3)
    beta = rng.normal(0, 1, p)
    y = (x @ beta > np.median(x @ beta)).astype(float)
    yv = (xv @ beta > np.median(x @ beta)).astype(float)
    data, valid = api.fm_matrix(x, y), api.fm_matrix(xv, yv)
    groups = (np.arange(p) // 10).astype(np.int32)
    data["features"]["attr_group"] = groups
    ctl = [api.model_control(factor_number=k, L2_w1=0.01, L2_v=0.02), api.solver_control(max_iter=400, solver=api.SGD_solver(learn_rate=0.05))]
    fit = api.fm_train_sgda(data, valid, normalize=True, control=ctl)
    # the same run spelled out on the ABI: z-score both sets with the training scales, the model as fm.train initialises it
    ctx = gpu_ctx
    feats = data["features"]
    d = L.Data.from_r_lists(ctx, n, p, feats["row_size"], feats["col_idx"], feats["value"], np.where(y < 1, -1.0, 1.0))
    mean, sd = d.scales(np.arange(p, dtype=np.int32))
    vf = valid["features"]
    dv = L.Data.from_r_lists(ctx, nv, p, vf["row_size"], vf["col_idx"], vf["value"], np.where(yv < 1, -1.0, 1.0))
    dv.normalize(mean, sd)
    m = L.Model(ctx, L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w1=0.01, l2_v=0.02), p, L.F64)
    rs = np.random.default_rng(int(api.get_option("FM.seed")))
    m.set(0.0, np.zeros(p), (0.0 + 0.01 * rs.standard_normal((k, p))).T.copy())
    sc = L.SolverCfg(solver=L.SGD, max_iter=400, random_step=1, learn_rate=0.05, min_target=-1.0, max_target=1.0, mode=L.MODE_EXACT,
                     precision=L.F64, compat=L.COMPAT_REFERENCE, step_size=-1, metric=L.LL, convergence=1e-4, seed=1)
    sc.attr_group = L.ptr(groups); sc.n_groups = 4
    lw, lv = np.full(4, 0.01), np.full((4, k), 0.02)
    L.train_sgda_dev(ctx, m, d, sc, dv, lw, lv, keep=[groups])
    w0, w, v = m.get()
    m.close(); d.close(); dv.close()
    md = fit["Model"]
    assert md["w0"] == w0 and np.array_equal(md["w"], w) and np.array_equal(md["v"], v.T)
    assert np.array_equal(md["reg"]["w"], lw) and np.array_equal(md["reg"]["v"], lv.T)
    assert not np.array_equal(lw, np.full(4, 0.01))
    pred = api.predict(fit, valid)
    assert pred.shape == (nv,) and np.all(np.isfinite(pred))
