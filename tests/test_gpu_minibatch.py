"""Throughput (minibatch) mode: (a) batch = 1 reproduces the exact mode (same per-coordinate arithmetic), (b) statistical parity with the
oracle's batch = 1 run on the same data (loss / AUC), (c) determinism and the truncated-last-batch path."""
import numpy as np
import pytest

from oracle import oracle as O
from fmwr_b200 import _lib as L
from fmwr_b200 import synth
from tests import minibatch_cases as MC
from tests.util import relerr

pytestmark = pytest.mark.gpu

SOLV = {O.SGD: L.SGD, O.FTRL: L.FTRL, O.TDAP: L.TDAP}


def mb_train(ctx, prec, ds, y, task, solver, k, w0, w, v, max_iter, batch, mode=L.MODE_MINIBATCH, regs=None, compat=L.COMPAT_REFERENCE, **sk):
    regs = regs or {}
    d = L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y)
    mc = L.ModelCfg(task=task, keep_w0=1, keep_w1=1, k=k, l2_w0=regs.get("l2_w0", 0), l1_w1=regs.get("l1_w", 0),
                    l2_w1=regs.get("l2_w", 0), l1_v=regs.get("l1_v", 0), l2_v=regs.get("l2_v", 0))
    m = L.Model(ctx, mc, ds["p"], prec)
    m.set(w0, w, v)
    sc = L.SolverCfg(solver=solver, max_iter=max_iter, random_step=1, learn_rate=sk.get("learn_rate", 0.01),
                     alpha_w=sk.get("alpha_w", 0.1), alpha_v=sk.get("alpha_v", 0.1), beta_w=1.0, beta_v=1.0,
                     gamma=1e-4, min_target=float(np.min(y)), max_target=float(np.max(y)), mode=mode, batch_size=batch,
                     precision=prec, compat=compat, step_size=-1)
    tr = L.TraceBuf(10)
    L.train_dev(ctx, m, d, sc, tr)
    out = m.get()
    # train-set probabilities / scores for the statistical checks
    L.predict_dev(ctx, m, d, L.LINK_LOGISTIC if task == L.CLASSIFICATION else L.LINK_NONE)
    pred = L.predict_fetch(ctx, d)
    m.close(); d.close()
    return out, pred, tr.result()


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
@pytest.mark.parametrize("regs", [dict(), dict(l1_w=0.01, l1_v=0.01), dict(l2_w=0.01, l2_v=0.02, l2_w0=0.01)])
def test_batch1_equals_exact_mode(gpu_ctx, solver, regs):
    rng = np.random.default_rng(1)
    rowptr, col, val = synth.random_csr(300, 50, 7, seed=2)
    ds = dict(n=300, p=50, rowptr=rowptr, col=col, val=val)
    y = np.where(rng.random(300) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, 50); v = rng.normal(0, 0.1, (50, 4))
    iters = 2 * 299 + 5
    # F6 is an exact-mode-only quirk: compare with it off on both sides
    compat = L.COMPAT_SKIP_ROW0
    for prec in (L.F32, L.F64):
        a, _, ta = mb_train(gpu_ctx, prec, ds, y, L.CLASSIFICATION, SOLV[solver], 4, 0.2, w, v, iters, 1, regs=regs, compat=compat)
        b, _, tb = mb_train(gpu_ctx, prec, ds, y, L.CLASSIFICATION, SOLV[solver], 4, 0.2, w, v, iters, 1, mode=L.MODE_EXACT, regs=regs, compat=compat)
        assert ta["iters_done"] == tb["iters_done"] == iters
        # same arithmetic per coordinate; only the reduction tree of S_f differs between the two kernels
        tol = 1e-10 if prec == L.F64 else (2e-2 if solver == O.TDAP else 1e-4)
        assert relerr(a[0], b[0]) < tol and relerr(a[1], b[1]) < tol and relerr(a[2], b[2]) < tol


@pytest.mark.parametrize("solver,batch", [(O.FTRL, 256), (O.FTRL, 400), (O.TDAP, 256), (O.SGD, 64), (O.SGD, 400)])
def test_minibatch_statistical_parity(gpu_ctx, port, solver, batch):
    # Criteo-shaped classification; the comparison run is batch = 1 for the same number of samples (the oracle for
    # SGD / FTRL; for TDAP the engine's own exact mode with F6 off, because the reference's z_w[position] bug makes
    # its TDAP diverge on 39-wide rows).  Parity is statistical: train log-loss within 3 % and AUC within 0.02, for
    # batches small enough that an epoch still has >= 100 optimizer steps (bench.py keeps that ratio: 10M rows / 65536).
    ds = synth.make_dataset("criteo", 40000, p=39 * 300)
    n, p, k = ds["n"], ds["p"], 8
    rng = np.random.default_rng(3)
    y = ds["y"]
    w = np.zeros(p); v = rng.normal(0, 0.01, (p, k))
    iters = 2 * (n - 1)
    regs = dict(l2_w=1e-4) if solver == O.SGD else {}
    if solver == O.TDAP:
        compat = L.COMPAT_SKIP_ROW0
        _, rp, _ = mb_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, L.TDAP, k, 0.0, w, v, iters, 1, mode=L.MODE_EXACT, compat=compat)
    else:
        compat = L.COMPAT_REFERENCE
        cfg = O.make_cfg(solver=solver, k=k, max_iter=iters, **regs)
        rw0, rw, rv, _ = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, 0.0, w, v)
        rp = port.predict(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], rw0, rw, rv, 1)
    _, gp, tr = mb_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.0, w, v, iters, batch, regs=regs, compat=compat)
    assert tr["iters_done"] == iters

    def ll(pr):
        return float(-np.mean(np.log(np.clip(np.where(y > 0, pr, 1 - pr), 1e-12, 1.0))))
    ll_r, ll_g = ll(rp), ll(gp)
    auc_r = port.evaluate(O.CLASSIFICATION, O.AUC, rp, y)
    auc_g = port.evaluate(O.CLASSIFICATION, O.AUC, gp, y)
    assert ll_r < 0.68                                             # the comparison run learned something
    assert abs(ll_g - ll_r) / ll_r < (0.15 if solver == O.TDAP else 0.03), (ll_g, ll_r)
    assert abs(auc_g - auc_r) < 0.02, (auc_g, auc_r)


def test_minibatch_deterministic_and_truncated_tail(gpu_ctx):
    ds = synth.make_dataset("criteo", 5000, p=39 * 100)
    rng = np.random.default_rng(4)
    k = 32
    w = np.zeros(ds["p"]); v = rng.normal(0, 0.01, (ds["p"], k))
    iters = 4999 + 1234                      # one full epoch + a truncated second one ending mid-batch
    a, pa, ta = mb_train(gpu_ctx, L.F32, ds, ds["y"], L.CLASSIFICATION, L.FTRL, k, 0.0, w, v, iters, 512)
    b, pb, tb = mb_train(gpu_ctx, L.F32, ds, ds["y"], L.CLASSIFICATION, L.FTRL, k, 0.0, w, v, iters, 512)
    assert ta["iters_done"] == iters
    assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert np.isfinite(a[2]).all() and np.isfinite(pa).all()
    # the second epoch stops 210 rows into its third batch: only those rows are applied.  The fp64 reference of the batch step
    # on the same inputs (tests/minibatch_cases.py: truncated_tail_case) holds the run to that; applying the whole third batch
    # moves the result by > 1 (tests/test_minibatch_reference.py)
    c = MC.truncated_tail_case()
    assert c["max_iter"] == iters and c["B"] == 512 and np.array_equal(c["v"], v.astype(np.float32).astype(np.float64))
    want = MC.reference(c)
    err = max(relerr(a[0], want["w0"]), relerr(a[1], want["w"]), relerr(a[2], want["v"]))
    print("truncated tail against the reference: max relerr %.3g (tolerance %.1g)" % (err, c["tol"]))
    assert err <= c["tol"], err


def test_minibatch_hot_feature_segments(gpu_ctx, port):
    # a tiny field (4 ids) makes segments thousands of rows long: exercises the long-segment path
    rowptr, col, val, p = synth.fields_csr(20000, [4, 3000, 3000], None, 1, 9)
    score = synth.planted_scores_fast(rowptr, col, val, p, seed=10)
    y = synth.labels_from_scores(score, "classification", seed=11)
    ds = dict(n=20000, p=p, rowptr=rowptr, col=col, val=val)
    rng = np.random.default_rng(5)
    k = 8
    w = np.zeros(p); v = rng.normal(0, 0.01, (p, k))
    iters = 19999
    cfg = O.make_cfg(solver=O.FTRL, k=k, max_iter=iters)
    rw0, rw, rv, _ = port.train(cfg, 20000, p, rowptr, col, val, y, 0.0, w, v)
    rp = port.predict(cfg, 20000, p, rowptr, col, val, rw0, rw, rv, 1)
    _, gp, _ = mb_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, L.FTRL, k, 0.0, w, v, iters, 2048)
    ll_r = -port.evaluate(O.CLASSIFICATION, O.LL, rp, y) / 20000
    ll_g = -port.evaluate(O.CLASSIFICATION, O.LL, gp, y) / 20000
    assert abs(ll_g - ll_r) / ll_r < 0.05, (ll_g, ll_r)


@pytest.mark.parametrize("solver,regs", [(O.FTRL, dict(l1_w1=1e-3, l2_w1=1e-3, l2_v=1e-3)), (O.TDAP, dict(l1_w1=1e-3, l2_v=1e-3)),
                                         (O.SGD, dict(l1_w1=1e-3, l1_v=1e-4))])
@pytest.mark.parametrize("mode", [L.MODE_MINIBATCH, L.MODE_EXACT])
def test_warm_state_continues_the_optimizer(gpu_ctx, solver, regs, mode):
    """SURVEY 8f-4: two calls of one epoch with warm_state = one call of two epochs, bit for bit -- also when the state
    travels through host arrays into a fresh model handle (what the R glue does between fm.train and fm.update).
    Without warm_state the second call restarts the state (the reference's fm.update) and ends elsewhere."""
    ctx = gpu_ctx
    rowptr, col, val, p = synth.fields_csr(3000, [40] * 6, None, 1, 5)
    n = rowptr.size - 1
    score = synth.planted_scores_fast(rowptr, col, val, p, seed=6)
    y = synth.labels_from_scores(score, "classification", seed=7)
    rng = np.random.default_rng(8)
    k = 8
    w = rng.normal(0, 0.05, p); v = rng.normal(0, 0.05, (p, k)); w0 = 0.05
    d = L.Data.from_csr32(ctx, n, p, rowptr, col, val, y)
    mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, **regs)
    epoch = n - 1

    def cfg(iters, warm):
        return L.SolverCfg(solver=solver, max_iter=iters, random_step=1, learn_rate=0.01, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0,
                           gamma=1e-4, min_target=-1.0, max_target=1.0, mode=mode, batch_size=256, precision=L.F64,
                           compat=L.COMPAT_REFERENCE, step_size=-1, warm_state=warm)

    def fresh():
        m = L.Model(ctx, mc, p, L.F64)
        m.set(w0, w, v)
        return m

    m = fresh(); L.train_dev(ctx, m, d, cfg(2 * epoch, 0)); both = m.get(); m.close()
    m = fresh(); L.train_dev(ctx, m, d, cfg(epoch, 0)); L.train_dev(ctx, m, d, cfg(epoch, 1)); warm = m.get()
    assert m.state_info()[0] == solver
    m.close()
    m = fresh(); L.train_dev(ctx, m, d, cfg(epoch, 0)); half = m.get(); st = m.get_state(); m.close()
    m2 = L.Model(ctx, mc, p, L.F64); m2.set(*half); m2.set_state(st); L.train_dev(ctx, m2, d, cfg(epoch, 1)); moved = m2.get(); m2.close()
    m = fresh(); L.train_dev(ctx, m, d, cfg(epoch, 0)); L.train_dev(ctx, m, d, cfg(epoch, 0)); cold = m.get(); m.close()
    for a, b in ((both, warm), (both, moved)):
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert not np.array_equal(both[2], cold[2])
    d.close()


@pytest.mark.parametrize("group_entries,pinned,random_step",
                         [(None, False, 1), ("1000000", False, 1), ("250000", False, 1), ("1000000", True, 1), (None, True, 1), ("1000000", True, 3)])
@pytest.mark.parametrize("solver", [O.FTRL, O.SGD])
def test_one_shot_train_equals_handle_path(gpu_ctx, monkeypatch, solver, group_entries, pinned, random_step):
    """fmwr_train (host fm.matrix lists in, host model out; the values upload on the copy stream while the per-batch CSC is
    sorted, and every batch waits only for its own chunk) must give the parameters of the handle path bit for bit --
    also over two epochs, when the second pass finds every value in place.  random_step > 1 gathers the visited rows up front,
    so there the one-shot call must upload every value before training."""
    import ctypes as C
    ctx = gpu_ctx
    lib = L.lib()
    # the one-shot path builds the per-batch CSC row group by row group behind the column upload: one group, ~9 groups of
    # several batches, and one batch per group (43 groups) must all give the one-piece structure
    # pinned: with page-locked caller buffers every third value chunk goes up as raw f64 and is narrowed on the device by its
    # first reader (mixed upload); the rounding is the same conversion either way, so the result stays bit-identical
    monkeypatch.setenv("FMWR_VAL_CHUNK", "1500000")            # several column / value chunks (and group boundaries inside them)
    if group_entries:
        monkeypatch.setenv("FMWR_GROUP_ENTRIES", group_entries)
    n, fields, k = 700_000, [997] * 13, 8               # 9.1M entries: several upload chunks' worth is not needed for the check
    rowptr, col, val, p = synth.fields_csr(n, fields, None, 1, 21)
    score = synth.planted_scores_fast(rowptr, col, val, p, seed=22)
    y = synth.labels_from_scores(score, "classification", seed=23)
    rng = np.random.default_rng(24)
    w = rng.normal(0, 0.02, p); v = rng.normal(0, 0.02, (p, k)); w0 = 0.01
    mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l1_w1=1e-4, l2_w1=1e-3, l2_v=1e-3)
    for iters in (n - 1, 2 * (n - 1) - 12345):
        sc = L.SolverCfg(solver=solver, max_iter=iters, random_step=random_step, learn_rate=0.01, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0,
                         min_target=-1.0, max_target=1.0, mode=L.MODE_MINIBATCH, batch_size=16384, precision=L.F32,
                         compat=L.COMPAT_REFERENCE, step_size=-1)
        d = L.Data.from_csr32(ctx, n, p, rowptr, col, val, y)
        m = L.Model(ctx, mc, p, L.F32); m.set(w0, w, v)
        C.CDLL(None).srand(5)                              # random_step > 1: both calls draw the same visit sequence from rand()
        L.train_dev(ctx, m, d, sc)
        a = m.get(); m.close(); d.close()
        # the library reuses freed device blocks: leave other values in the blocks of this size, so that a value the one-shot
        # call never uploads shows up as a difference instead of as the handle path's leftover
        L.Data.from_csr32(ctx, n, p, rowptr, col, val + 1.0, y).close()
        rs = np.diff(rowptr.astype(np.int64)).astype(np.int32)
        ci = col.astype(np.int32); v64 = val.astype(np.float64); y64 = y.astype(np.float64)
        bw0 = C.c_double(w0); bw = w.copy(); bv = v.copy()
        if pinned:
            for arr in (ci, v64):
                L.check(lib.fmwr_host_pin(L.ptr(arr), C.c_int64(arr.nbytes)))
        try:
            C.CDLL(None).srand(5)
            L.check(lib.fmwr_train(C.byref(mc), C.byref(sc), C.c_int64(n), C.c_int64(p), C.c_int64(ci.size), L.ptr(rs), L.ptr(ci), L.ptr(v64),
                                   L.ptr(y64), C.byref(bw0), L.ptr(bw), L.ptr(bv), None))
        finally:
            if pinned:
                for arr in (ci, v64):
                    lib.fmwr_host_unpin(L.ptr(arr))
        assert a[0] == bw0.value and np.array_equal(a[1], bw) and np.array_equal(a[2], bv)


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL])
def test_minibatch_ragged_rows_with_empty_rows_and_wide_rows(gpu_ctx, solver):
    """edge cases of the data: empty rows (score = w0 only, no segment), rows wider than one gather chunk (> 64 non-zeros),
    a batch size that does not divide the row count, k that needs padding -- batch = 1 must still equal the exact mode,
    and a larger batch must be deterministic and finite"""
    rng = np.random.default_rng(11)
    n, p, k = 500, 400, 5
    rowptr, col, val = synth.random_csr(n, p, 30, seed=12, empty_rows=True)
    # make a few rows very wide
    counts = np.diff(rowptr.astype(np.int64))
    assert (counts == 0).any()
    wide = [3, 250, 499]
    rows = []
    for r in range(n):
        if r in wide:
            c = np.sort(rng.choice(p, 150, replace=False)).astype(np.uint32)
            rows.append((c, rng.uniform(0.5, 1.5, c.size).astype(np.float32)))
        else:
            rows.append((col[rowptr[r]:rowptr[r + 1]], val[rowptr[r]:rowptr[r + 1]]))
    rowptr2 = np.concatenate([[0], np.cumsum([c.size for c, _ in rows])]).astype(np.uint32)
    col2 = np.concatenate([c for c, _ in rows]).astype(np.uint32)
    val2 = np.concatenate([x for _, x in rows]).astype(np.float32)
    ds = dict(n=n, p=p, rowptr=rowptr2, col=col2, val=val2)
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.05, p); v = rng.normal(0, 0.05, (p, k))
    iters = 2 * (n - 1) + 3
    regs = dict(l2_w=0.01, l2_v=0.01)
    a, _, _ = mb_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.1, w, v, iters, 1, regs=regs, compat=L.COMPAT_SKIP_ROW0)
    b, _, _ = mb_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.1, w, v, iters, 1, mode=L.MODE_EXACT, regs=regs, compat=L.COMPAT_SKIP_ROW0)
    assert relerr(a[0], b[0]) < 1e-10 and relerr(a[1], b[1]) < 1e-10 and relerr(a[2], b[2]) < 1e-10
    c1, p1, _ = mb_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.1, w, v, iters, 37, regs=regs)
    c2, p2, _ = mb_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.1, w, v, iters, 37, regs=regs)
    assert c1[0] == c2[0] and np.array_equal(c1[1], c2[1]) and np.array_equal(c1[2], c2[2])
    assert np.isfinite(c1[2]).all() and np.isfinite(p1).all() and np.array_equal(p1, p2)


@pytest.mark.parametrize("solver,regs", [(O.FTRL, dict(l1_w=1e-3, l2_w=1e-3, l2_v=1e-3)), (O.SGD, dict(l2_w=1e-3, l2_v=1e-3)),
                                          (O.SGD, dict(l1_w=1e-3, l1_v=1e-3)), (O.TDAP, dict(l1_w=1e-3, l2_v=1e-3))])
@pytest.mark.parametrize("k", [32, 30, 8, 3])
def test_dense_update_kernel_equals_gather_kernel(gpu_ctx, solver, regs, k, monkeypatch):
    """mb_update_tma_kernel (parameter ranges staged by bulk copies, csrc/update_tma.cuh) against mb_update_kernel (per-segment
    gathers) on the same batches: same per-segment arithmetic and entry order, so the models agree to rounding of the
    compiler's FMA choices.  Fields of 300 ids with batch 1024 make most tiles dense; a 40 000-id field and a skewed one
    add sparse tiles (fallback path) and long segments to the same launch."""
    n = 6000
    fields = [300] * 8 + [40_000, 2000]
    rowptr, col, val, p = synth.fields_csr(n, fields, [0] * 9 + [1], 1, 11)
    ds = dict(n=n, p=p, rowptr=rowptr, col=col, val=val)
    rng = np.random.default_rng(5)
    y = np.where(rng.random(n) < 0.4, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    iters = 2 * (n - 1)
    for batch in (1024, 777):
        monkeypatch.delenv("FMWR_K2_GATHER", raising=False)
        a, _, _ = mb_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.1, w, v, iters, batch, regs=regs)
        monkeypatch.setenv("FMWR_K2_GATHER", "1")
        b, _, _ = mb_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.1, w, v, iters, batch, regs=regs)
        monkeypatch.delenv("FMWR_K2_GATHER", raising=False)
        tol = 1e-3 if solver == O.TDAP else 1e-5
        assert relerr(a[0], b[0]) < tol and relerr(a[1], b[1]) < tol and relerr(a[2], b[2]) < tol
        assert np.isfinite(a[2]).all()


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
def test_minibatch_parity_in_the_benchmark_regime(gpu_ctx, port, solver):
    """The regime bench.py measures, scaled down: a batch touches each id of a field 2.56 times (batch 256 over 100-id fields;
    the bench: 65 536 over 25 641) and an epoch has 150 optimizer steps (the bench: 153).  Two epochs of the throughput mode
    against two epochs of batch = 1 in the reference's order (the oracle for SGD / FTRL; the engine's own exact mode with F6
    off for TDAP, whose reference diverges on 39-wide rows): train log-loss within 3 %, AUC within 0.02."""
    n, fid, B, k = 150 * 256, 100, 256, 8
    ds = synth.make_dataset("criteo", n, p=39 * fid)
    p = ds["p"]
    y = ds["y"]
    rng = np.random.default_rng(13)
    w = np.zeros(p); v = rng.normal(0, 0.01, (p, k))
    iters = 2 * (n - 1)
    regs = dict(l2_w=1e-4) if solver == O.SGD else dict(l1_w=1e-3, l2_w=1e-3, l2_v=1e-3)
    if solver == O.TDAP:
        compat = L.COMPAT_SKIP_ROW0
        _, rp, _ = mb_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, L.TDAP, k, 0.0, w, v, iters, 1, mode=L.MODE_EXACT, regs=regs, compat=compat)
    else:
        compat = L.COMPAT_REFERENCE
        cfg = O.make_cfg(solver=solver, k=k, max_iter=iters, **regs)
        rw0, rw, rv, _ = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, 0.0, w, v)
        rp = port.predict(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], rw0, rw, rv, 1)
    _, gp, tr = mb_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, 0.0, w, v, iters, B, regs=regs, compat=compat)
    assert tr["iters_done"] == iters

    def ll(pr):
        return float(-np.mean(np.log(np.clip(np.where(y > 0, pr, 1 - pr), 1e-12, 1.0))))
    ll_r, ll_g = ll(rp), ll(gp)
    auc_r = port.evaluate(O.CLASSIFICATION, O.AUC, rp, y)
    auc_g = port.evaluate(O.CLASSIFICATION, O.AUC, gp, y)
    print("bench-regime parity solver=%d: LL batch=1 %.5f minibatch %.5f (%.2f %%), AUC %.4f vs %.4f" % (solver, ll_r, ll_g, 100 * (ll_g - ll_r) / ll_r, auc_r, auc_g))
    assert ll_r < 0.69
    assert abs(ll_g - ll_r) / ll_r < 0.03, (ll_g, ll_r)
    assert abs(auc_g - auc_r) < 0.02, (auc_g, auc_r)


def test_throughput_mode_follows_a_strided_visit_sequence(gpu_ctx):
    """random_step > 1 (reference random_select, src/util/Random.h:126-132; scan loops SGD_Learner.h:84-88): the throughput mode
    batches consecutive VISITS.  With an explicit visit sequence and batch = 1 it equals the exact mode on the same sequence;
    with the engine's own rand()-driven strides and a real batch it trains and reports the visits it made."""
    rng = np.random.default_rng(21)
    rowptr, col, val = synth.random_csr(500, 60, 7, seed=22)
    n, p, k = 500, 60, 4
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    visit = []
    while len(visit) < 1300:                                # three passes of strides 1..4, ascending inside a pass
        i = int(rng.integers(1, 5))
        while i < n and len(visit) < 1300:
            visit.append(i); i += int(rng.integers(1, 5))
    visit = np.array(visit, np.uint32)

    def run(mode, batch, visit_order=None, random_step=1, max_iter=1300):
        d = L.Data.from_csr32(gpu_ctx, n, p, rowptr, col, val, y)
        m = L.Model(gpu_ctx, L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w1=0.01, l2_v=0.01), p, L.F64)
        m.set(0.1, w, v)
        sc = L.SolverCfg(solver=L.FTRL, max_iter=max_iter, random_step=random_step, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0, min_target=-1.0,
                         max_target=1.0, mode=mode, batch_size=batch, precision=L.F64, compat=L.COMPAT_SKIP_ROW0, step_size=-1)
        keep = None
        if visit_order is not None:
            keep = np.ascontiguousarray(visit_order, np.uint32)
            sc.visit_order = L.ptr(keep); sc.n_visit = keep.size
        tr = L.TraceBuf(4)
        L.train_dev(gpu_ctx, m, d, sc, tr, keep=(keep,))
        out = m.get()
        m.close(); d.close()
        return out, tr.result()

    a, ta = run(L.MODE_MINIBATCH, 1, visit)
    b, tb = run(L.MODE_EXACT, 1, visit)
    assert ta["iters_done"] == tb["iters_done"] == 1300
    assert relerr(a[0], b[0]) < 1e-10 and relerr(a[1], b[1]) < 1e-10 and relerr(a[2], b[2]) < 1e-10
    c, tc = run(L.MODE_MINIBATCH, 64, None, random_step=3, max_iter=900)
    assert tc["iters_done"] == 900 and np.isfinite(c[2]).all() and float(np.max(np.abs(c[2] - v))) > 1e-3


@pytest.mark.parametrize("bad", ["range", "order"])
def test_one_shot_train_rejects_a_bad_matrix(gpu_ctx, bad):
    """The one-shot path uploads the column ids in chunks and validates them group by group while it builds the per-batch CSC
    (data.cu: minibatch_build_grouped): a column out of range or a row that is not ascending must still come back as the
    reference's shape error (src/util/Smatrix.h:52 family), not as a crash in the kernels that follow."""
    import ctypes as C
    lib = L.lib()
    n, fields, k = 60_000, [97] * 7, 4
    rowptr, col, val, p = synth.fields_csr(n, fields, None, 1, 5)
    col = col.copy()
    if bad == "range":
        col[rowptr[41_000] + 3] = p + 5
    else:
        j = rowptr[17_000]
        col[j], col[j + 1] = col[j + 1], col[j]
    y = np.where(np.arange(n) % 2 == 0, 1.0, -1.0)
    mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w1=1e-3, l2_v=1e-3)
    sc = L.SolverCfg(solver=L.FTRL, max_iter=n - 1, random_step=1, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0, min_target=-1.0, max_target=1.0,
                     mode=L.MODE_MINIBATCH, batch_size=4096, precision=L.F32, compat=L.COMPAT_REFERENCE, step_size=-1)
    rs = np.diff(rowptr.astype(np.int64)).astype(np.int32)
    ci = col.astype(np.int32); v64 = val.astype(np.float64)
    w0 = C.c_double(0.0); w = np.zeros(p); v = np.zeros((p, k))
    rc = lib.fmwr_train(C.byref(mc), C.byref(sc), C.c_int64(n), C.c_int64(p), C.c_int64(ci.size), L.ptr(rs), L.ptr(ci), L.ptr(v64), L.ptr(y),
                        C.byref(w0), L.ptr(w), L.ptr(v), None)
    assert rc == L.ERR_SHAPE if hasattr(L, "ERR_SHAPE") else rc != 0
    msg = lib.fmwr_last_error().decode()
    assert ("out of range" in msg) if bad == "range" else ("ascending" in msg)
    # and the library is still usable afterwards
    col2 = synth.fields_csr(n, fields, None, 1, 5)[1]
    ci2 = col2.astype(np.int32)
    L.check(lib.fmwr_train(C.byref(mc), C.byref(sc), C.c_int64(n), C.c_int64(p), C.c_int64(ci2.size), L.ptr(rs), L.ptr(ci2), L.ptr(v64), L.ptr(y),
                           C.byref(w0), L.ptr(w), L.ptr(v), None))
    assert np.isfinite(w).all() and np.abs(w).sum() > 0      # (V starts at zero and an all-zero V has a zero gradient)
