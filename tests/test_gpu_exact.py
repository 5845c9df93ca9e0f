"""Exact (batch = 1) SGD / FTRL / TDAP parity against the oracle after N epochs
(reference src/solver/{SGD,FTRL,TDAP}_Learner.h).  Tolerance: 1e-4 relative on parameters
(north star); the fp64 instantiation is held to 1e-9."""
import numpy as np
import pytest

from oracle import oracle as O
from fmwr_b200 import _lib as L
from fmwr_b200 import synth
from tests.util import relerr

pytestmark = pytest.mark.gpu

SOLV = {O.SGD: L.SGD, O.FTRL: L.FTRL, O.TDAP: L.TDAP}


def gpu_train(ctx, prec, ds, y, task, solver, k, w0, w, v, max_iter, regs=None, step_size=-1, metric=L.LL, compat=L.COMPAT_REFERENCE,
              visit=None, random_step=1, k0=1, k1=1, **sk):
    regs = regs or {}
    d = L.Data.from_csr32(ctx, ds["n"], ds["p"], ds["rowptr"], ds["col"], ds["val"], y)
    mc = L.ModelCfg(task=task, keep_w0=k0, keep_w1=k1, k=k, l2_w0=regs.get("l2_w0", 0), l1_w1=regs.get("l1_w", 0),
                    l2_w1=regs.get("l2_w", 0), l1_v=regs.get("l1_v", 0), l2_v=regs.get("l2_v", 0))
    m = L.Model(ctx, mc, ds["p"], prec)
    m.set(w0, w, v)
    sc = L.SolverCfg(solver=solver, max_iter=max_iter, random_step=random_step, learn_rate=sk.get("learn_rate", 0.01),
                     alpha_w=sk.get("alpha_w", 0.1), alpha_v=sk.get("alpha_v", 0.1), beta_w=sk.get("beta_w", 1.0),
                     beta_v=sk.get("beta_v", 1.0), gamma=sk.get("gamma", 1e-4), min_target=float(np.min(y)),
                     max_target=float(np.max(y)), mode=L.MODE_EXACT, precision=prec, compat=compat,
                     step_size=step_size, metric=metric, convergence=sk.get("convergence", 1e-4))
    keep = None
    if visit is not None:
        keep = np.ascontiguousarray(visit, np.uint32)
        sc.visit_order = L.ptr(keep); sc.n_visit = keep.size
    tr = L.TraceBuf(200)
    L.train_dev(ctx, m, d, sc, tr, keep=(keep,))
    out = m.get()
    m.close(); d.close()
    return out, tr.result()


def small(n=400, p=60, seed=3, nnz=8):
    rowptr, col, val = synth.random_csr(n, p, nnz, seed=seed)
    return dict(n=n, p=p, rowptr=rowptr, col=col, val=val)


REGS = [dict(), dict(l1_w=0.01, l1_v=0.01, l2_w=0.001), dict(l2_w=0.01, l2_v=0.02, l2_w0=0.01)]


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
@pytest.mark.parametrize("task", [O.CLASSIFICATION, O.REGRESSION])
@pytest.mark.parametrize("regs", REGS)
def test_exact_matches_oracle_fp64(gpu_ctx, port, solver, task, regs):
    rng = np.random.default_rng(1)
    ds = small()
    n, p, k = ds["n"], ds["p"], 4
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == O.CLASSIFICATION else rng.normal(0, 1, n)
    y = y.astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k)); w0 = 0.3
    iters = 3 * (n - 1) + 11                                 # N epochs == N*(n-1) updates (F4/F5), plus a ragged tail
    cfg = O.make_cfg(task=task, solver=solver, k=k, max_iter=iters, min_target=float(y.min()), max_target=float(y.max()), **regs)
    rw0, rw, rv, _ = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, w0, w, v)
    (gw0, gw, gv), tr = gpu_train(gpu_ctx, L.F64, ds, y, task, SOLV[solver], k, w0, w, v, iters, regs)
    assert tr["iters_done"] == iters
    assert relerr(gw0, rw0) < 1e-9 and relerr(gw, rw) < 1e-9 and relerr(gv, rv) < 1e-9


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
def test_exact_fp32_within_north_star_tolerance(gpu_ctx, port, solver):
    rng = np.random.default_rng(2)
    ds = synth.make_dataset("c1", 3000)                      # C1-shaped (10 fields x 1000 ids, real-valued x), regression
    n, p, k = ds["n"], ds["p"], 8
    y = ds["y"]
    w = np.zeros(p); v = rng.normal(0, 0.01, (p, k)); w0 = 0.0
    iters = 2 * (n - 1)
    cfg = O.make_cfg(task=O.REGRESSION, solver=solver, k=k, max_iter=iters, l2_w=0.001, l2_v=0.001,
                     min_target=float(y.min()), max_target=float(y.max()))
    rw0, rw, rv, _ = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, w0, w, v)
    (gw0, gw, gv), _ = gpu_train(gpu_ctx, L.F32, ds, y, L.REGRESSION, SOLV[solver], k, w0, w, v, iters, dict(l2_w=0.001, l2_v=0.001))
    # north star: batch=1 SGD / FTRL parameters within 1e-4.  TDAP is not on that list: theta = -(nu - h)/delta has no
    # beta in the denominator and cancels two running sums, so fp32 STORAGE of nu and h costs ~1e-2; its tight parity
    # is asserted with the fp64 instantiation (test_exact_matches_oracle_fp64) and here only loosely.
    tol = 5e-2 if solver == O.TDAP else 1e-4
    assert relerr(gw0, rw0) < tol and relerr(gw, rw) < tol and relerr(gv, rv) < tol


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL])
def test_exact_wide_rows_and_large_k(gpu_ctx, port, solver):
    # rows wider than the CTA's slot count and k that needs several 16-byte chunks per lane
    rng = np.random.default_rng(4)
    n, p, k = 60, 400, 40
    rowptr, col, val = synth.random_csr(n, p, 150, seed=8)
    ds = dict(n=n, p=p, rowptr=rowptr, col=col, val=val)
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.05, p); v = rng.normal(0, 0.05, (p, k)); w0 = 0.0
    iters = 2 * (n - 1)
    cfg = O.make_cfg(solver=solver, k=k, max_iter=iters)
    rw0, rw, rv, _ = port.train(cfg, n, p, rowptr, col, val, y, w0, w, v)
    (gw0, gw, gv), _ = gpu_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, SOLV[solver], k, w0, w, v, iters)
    assert relerr(gw0, rw0) < 1e-9 and relerr(gw, rw) < 1e-9 and relerr(gv, rv) < 1e-9


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
@pytest.mark.parametrize("k,max_nnz,prec", [(4, 70, "f64"), (128, 45, "f64"), (32, 100, "f32"), (128, 45, "f32")])
def test_exact_row_shapes_and_layouts(gpu_ctx, port, solver, k, max_nnz, prec):
    # ragged rows from empty to wider than the shared-memory ring (64) and than the factor warps' slot count
    # (56 at k=32 fp32, 14 at k=128 fp32, 7 at k=128 fp64): every gather/update path of the kernel -- registers kept,
    # second round from global memory, the linear warp's two-per-lane and looped forms, TDAP's position refresh (F6)
    rng = np.random.default_rng(11)
    n, p = 90, 300
    rowptr, col, val = synth.random_csr(n, p, max_nnz, seed=21, empty_rows=True)
    ds = dict(n=n, p=p, rowptr=rowptr, col=col, val=val)
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.05, p); v = rng.normal(0, 0.05, (p, k)); w0 = 0.1
    iters = 2 * (n - 1) + 7
    regs = dict(l1_w=0.001, l2_w=0.001, l2_v=0.002)
    cfg = O.make_cfg(solver=solver, k=k, max_iter=iters, **regs)
    rw0, rw, rv, _ = port.train(cfg, n, p, rowptr, col, val, y, w0, w, v)
    (gw0, gw, gv), _ = gpu_train(gpu_ctx, L.F64 if prec == "f64" else L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, w0, w, v, iters, regs)
    tol = 1e-9 if prec == "f64" else (5e-2 if solver == O.TDAP else 1e-4)
    assert relerr(gw0, rw0) < tol and relerr(gw, rw) < tol and relerr(gv, rv) < tol


def test_exact_tracker_and_convergence(gpu_ctx, port):
    rng = np.random.default_rng(5)
    ds = small(n=300, p=40, seed=6)
    n, p, k = ds["n"], ds["p"], 3
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = np.zeros(p); v = rng.normal(0, 0.01, (p, k))
    iters = 1500
    for metric in (O.LL, O.AUC, O.ACC):
        cfg = O.make_cfg(solver=O.FTRL, k=k, max_iter=iters, step_size=100, metric=metric, convergence=1e-3)
        rw0, rw, rv, rt = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, 0.0, w, v, max_rec=100)
        (gw0, gw, gv), gt = gpu_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, L.FTRL, k, 0.0, w, v, iters, step_size=100,
                                      metric=metric, convergence=1e-3)
        assert gt["n_rec"] == rt["n_rec"] and (gt["rec_index"] == rt["rec_index"]).all()
        assert gt["convergent"] == rt["convergent"] and gt["iters_done"] == rt["iters_done"]
        assert relerr(gt["eval_train"], rt["eval_train"]) < 1e-9
        assert relerr(gv, rv) < 1e-9


def test_exact_explicit_visit_order_random_step(gpu_ctx, port):
    # random_step > 1: both sides consume the same injected rand() stream (reference src/util/Random.h:126-132)
    rng = np.random.default_rng(6)
    ds = small(n=500, p=50, seed=7)
    n, p, k = ds["n"], ds["p"], 4
    y = rng.normal(0, 1, n).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    rands = rng.integers(0, 2**31 - 1, 5000).astype(np.int32)
    step, iters = 5, 700
    # the visit sequence the reference derives from that stream
    u = rands / (2.0**31)
    sel = (u * step + 1).astype(np.uint32)
    order = []; q = 0
    while len(order) < iters:
        i = sel[q]; q += 1
        while i < n and len(order) < iters:
            order.append(i); i += sel[q]; q += 1
    cfg = O.make_cfg(task=O.REGRESSION, solver=O.SGD, k=k, max_iter=iters, random_step=step, min_target=float(y.min()),
                     max_target=float(y.max()))
    port.set_streams(None, None, rands)
    rw0, rw, rv, _ = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, 0.1, w, v)
    port.set_streams(None, None, None)
    (gw0, gw, gv), _ = gpu_train(gpu_ctx, L.F64, ds, y, L.REGRESSION, L.SGD, k, 0.1, w, v, iters, visit=order, random_step=step)
    assert relerr(gw0, rw0) < 1e-9 and relerr(gw, rw) < 1e-9 and relerr(gv, rv) < 1e-9


def test_exact_keep_flags(gpu_ctx, port):
    rng = np.random.default_rng(8)
    ds = small(n=200, p=30, seed=9)
    n, p, k = ds["n"], ds["p"], 2
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    for k0, k1 in ((0, 1), (1, 0)):
        cfg = O.make_cfg(solver=O.SGD, k=k, max_iter=300, k0=k0, k1=k1)
        rw0, rw, rv, _ = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, 0.2, w, v)
        (gw0, gw, gv), _ = gpu_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, L.SGD, k, 0.2, w, v, 300, k0=k0, k1=k1)
        assert relerr(gw0, rw0) < 1e-9 and relerr(gw, rw) < 1e-9 and relerr(gv, rv) < 1e-9


def test_exact_fixed_mode_visits_row0(gpu_ctx):
    # compat=0 ("fixed"): the scan includes row 0, which the reference never trains on (F5)
    ds = small(n=5, p=10, seed=1, nnz=3)
    y = np.ones(5, np.float32)
    w = np.zeros(10); v = np.zeros((10, 2))
    (w0a, wa, _), _ = gpu_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, L.SGD, 2, 0.0, w, v, 1, compat=0)
    (w0b, wb, _), _ = gpu_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, L.SGD, 2, 0.0, w, v, 1, compat=L.COMPAT_REFERENCE)
    r0 = ds["col"][ds["rowptr"][0]:ds["rowptr"][1]]
    r1 = ds["col"][ds["rowptr"][1]:ds["rowptr"][2]]
    assert np.count_nonzero(wa) == len(r0) and np.all(wa[r0] != 0)
    assert np.count_nonzero(wb) == len(r1) and np.all(wb[r1] != 0)


def test_exact_tdap_single_nnz_rows_no_fma_residue(gpu_ctx, port):
    # rows with one non-zero make S_f*x - v*x*x exactly 0 in the reference; a fused multiply-add would leave a
    # residue whose sign TDAP amplifies to +-alpha (see coord.cuh: fm_grad)
    rng = np.random.default_rng(9)
    n, p, k = 300, 20, 4
    rowptr, col, val = synth.random_csr(n, p, 2, seed=10)
    ds = dict(n=n, p=p, rowptr=rowptr, col=col, val=val)
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    for prec, tol in ((L.F64, 1e-9), (L.F32, 1e-3)):
        cfg = O.make_cfg(solver=O.TDAP, k=k, max_iter=2 * (n - 1))
        rw0, rw, rv, _ = port.train(cfg, n, p, rowptr, col, val, y, 0.3, w, v)
        (gw0, gw, gv), _ = gpu_train(gpu_ctx, prec, ds, y, L.CLASSIFICATION, L.TDAP, k, 0.3, w, v, 2 * (n - 1))
        assert relerr(gw0, rw0) < tol and relerr(gw, rw) < tol and relerr(gv, rv) < tol


def test_configs0_in_full_against_the_restatement(gpu_ctx, port):
    """BASELINE configs[0] at its full size: fm.train SGD.solver, k=8, L2, 100k x 10k regression (10 nnz/row, real-valued x).
    Exact mode over all 99 999 updates of an epoch, two epochs, against the plain-C restatement of the reference's
    SGD_Learner (oracle/fm_oracle.c; reference src/solver/SGD_Learner.h:86-177), every parameter: fp32 within the north
    star's 1e-4, fp64 within 1e-9.  The restatement is held to the reference by tests/test_golden.py and
    tests/test_oracle_pinning.py."""
    ds = synth.make_dataset("c1", 100_000)
    n, p, k = ds["n"], ds["p"], 8
    y = ds["y"]
    rng = np.random.default_rng(20240603)
    w = np.zeros(p); v = rng.normal(0, 0.01, (p, k)); w0 = 0.0
    iters = 2 * (n - 1)
    regs = dict(l2_w=0.001, l2_v=0.001)
    cfg = O.make_cfg(task=O.REGRESSION, solver=O.SGD, k=k, max_iter=iters, min_target=float(y.min()), max_target=float(y.max()), **regs)
    rw0, rw, rv, _ = port.train(cfg, n, p, ds["rowptr"], ds["col"], ds["val"], y, w0, w, v)
    assert float(np.max(np.abs(rv - v))) > 1e-3              # the run trained
    for prec, tol in ((L.F64, 1e-9), (L.F32, 1e-4)):
        (gw0, gw, gv), tr = gpu_train(gpu_ctx, prec, ds, y, L.REGRESSION, L.SGD, k, w0, w, v, iters, regs)
        assert tr["iters_done"] == iters
        assert relerr(gw0, rw0) < tol and relerr(gw, rw) < tol and relerr(gv, rv) < tol


# ---- the pipelined kernel (train_exact_pipe.cuh): several samples in flight, serial semantics through column-hazard tracking.
# FMWR_EXACT_PIPE: 0 = CTA-wide kernel only, 2 = pipelined wherever it can run, unset = the engine's choice per solver / precision.
HAZARD_SHAPES = [
    # (n, p, max nnz, k): what the shape stresses
    (3000, 40, 12, 8),        # every sample shares columns with its neighbours: the pipeline degrades to the serial order
    (6000, 2500, 30, 32),     # dependencies at every distance inside the ring, many table sets holding two live columns
    (1500, 6000, 150, 32),    # rows longer than the ring and the stage: chunked path, columns hashed from global memory
    (4000, 300, 45, 4),       # 16 entries per round (k = 4): many lanes of a warp in the same table set
]


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL, O.TDAP])
@pytest.mark.parametrize("shape", HAZARD_SHAPES)
def test_pipelined_exact_kernel_keeps_the_serial_order(gpu_ctx, port, monkeypatch, solver, shape):
    """fp64, so a single stale read (a hazard the tracker missed) shows at 1e-3 while the two kernels' different summation
    orders stay below 1e-9; then the oracle itself on the smaller shapes."""
    n, p, max_nnz, k = shape
    rng = np.random.default_rng(n + k)
    rowptr, col, val = synth.random_csr(n, p, max_nnz, seed=n, empty_rows=True)
    ds = dict(n=n, p=p, rowptr=rowptr, col=col, val=val)
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k)); w0 = 0.1
    regs = dict(l1_w=0.001, l2_w=0.001, l2_v=0.001)
    iters = 2 * (n - 1) + 7
    out = {}
    for pipe in ("0", "2"):
        monkeypatch.setenv("FMWR_EXACT_PIPE", pipe)
        out[pipe], _ = gpu_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, SOLV[solver], k, w0, w, v, iters, regs=regs)
    tol = 1e-9 if solver != O.TDAP else 1e-6        # TDAP amplifies rounding (DESIGN.md section 4)
    assert abs(out["0"][0] - out["2"][0]) < tol * max(1.0, abs(out["0"][0]))
    assert relerr(out["2"][1], out["0"][1]) < tol and relerr(out["2"][2], out["0"][2]) < tol
    if n * max_nnz <= 200_000:
        cfg = O.make_cfg(task=O.CLASSIFICATION, solver=solver, k=k, max_iter=iters, min_target=-1.0, max_target=1.0, **regs)
        rw0, rw, rv = port.train(cfg, n, p, rowptr, col, val, y, w0, w, v)[:3]
        assert abs(out["2"][0] - rw0) < 1e-8 * max(1.0, abs(rw0)) if solver != O.TDAP else True
        assert relerr(out["2"][1], rw) < (1e-8 if solver != O.TDAP else 1e-5)
        assert relerr(out["2"][2], rv) < (1e-8 if solver != O.TDAP else 1e-5)


@pytest.mark.parametrize("solver", [O.SGD, O.FTRL])
def test_pipelined_exact_kernel_fp32_and_visit_orders(gpu_ctx, monkeypatch, solver):
    """fp32 instantiation, an explicit visit order with repeats (the same row twice in a row is the sharpest hazard), the
    tracker's launch segmentation (step_size) and a launch shorter than the pipeline's depth."""
    n, p, k = 2000, 900, 32
    rng = np.random.default_rng(5)
    rowptr, col, val = synth.random_csr(n, p, 40, seed=11, empty_rows=True)
    ds = dict(n=n, p=p, rowptr=rowptr, col=col, val=val)
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k)); w0 = 0.0
    visit = rng.integers(0, n, 5000).astype(np.uint32)
    visit[100:140] = 7                                  # forty visits of one row
    visit[200:260:2] = 9                                # every other visit
    for kw in (dict(visit=visit, max_iter=5000), dict(max_iter=3), dict(max_iter=2 * n, step_size=37)):
        out = {}
        for pipe in ("0", "2"):
            monkeypatch.setenv("FMWR_EXACT_PIPE", pipe)
            mi = kw["max_iter"]
            out[pipe], tr = gpu_train(gpu_ctx, L.F32, ds, y, L.CLASSIFICATION, SOLV[solver], k, w0, w, v, mi, regs=dict(l2_w=0.001, l2_v=0.001),
                                      visit=kw.get("visit"), step_size=kw.get("step_size", -1))
        assert abs(out["0"][0] - out["2"][0]) < 2e-5
        assert relerr(out["2"][1], out["0"][1]) < 2e-5 and relerr(out["2"][2], out["0"][2]) < 2e-5


def test_hazard_tracking_is_what_keeps_the_order(gpu_ctx, monkeypatch):
    """The same pipeline with the dependency waits switched off (FMWR_EXACT_NOHAZARD=1, a test-only switch) must NOT reproduce
    the serial result on data whose neighbouring samples share columns: the stress tests above are sensitive to a missed hazard."""
    n, p, max_nnz, k = HAZARD_SHAPES[0]
    rng = np.random.default_rng(2)
    rowptr, col, val = synth.random_csr(n, p, max_nnz, seed=n)
    ds = dict(n=n, p=p, rowptr=rowptr, col=col, val=val)
    y = np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k)); w0 = 0.1
    out = {}
    for name, env in (("serial", {"FMWR_EXACT_PIPE": "0"}), ("tracked", {"FMWR_EXACT_PIPE": "2"}), ("untracked", {"FMWR_EXACT_PIPE": "2", "FMWR_EXACT_NOHAZARD": "1"})):
        monkeypatch.delenv("FMWR_EXACT_NOHAZARD", raising=False)
        for kk, vv in env.items():
            monkeypatch.setenv(kk, vv)
        out[name], _ = gpu_train(gpu_ctx, L.F64, ds, y, L.CLASSIFICATION, L.SGD, k, w0, w, v, 2 * (n - 1), regs=dict(l2_w=0.001, l2_v=0.001), learn_rate=0.05)
    assert relerr(out["tracked"][2], out["serial"][2]) < 1e-9
    assert relerr(out["untracked"][2], out["serial"][2]) > 1e-6
