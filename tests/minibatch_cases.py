"""Inputs of the throughput-mode reference tests (tests/test_gpu_minibatch_reference.py), shared with their CPU negative
controls (tests/test_minibatch_reference.py) so that both speak about the same data and tolerances.

case(name) returns a dict:
  data   n, p, rowptr, col, val, y (the CSR the engine uploads)
  model  task, k, keep_w0 / keep_w1, precision ("f32" / "f64"), w0, w, v, state (None: the solver starts from zero)
  solver solver, hyper-parameters, B, max_iter, compat, visit_order, step_size
  tol    the asserted max relerr of every parameter and state array, and `env` (FMWR_K2_GATHER) where a case forces a kernel
"""
import numpy as np

from fmwr_b200 import synth
from tests import minibatch_ref as R

CLASSIFICATION, REGRESSION = R.CLASSIFICATION, R.REGRESSION
SGD, FTRL, TDAP = R.SGD, R.FTRL, R.TDAP
SOLVER_NAMES = {"sgd": SGD, "ftrl": FTRL, "tdap": TDAP}
COMPAT_SKIP_ROW0, COMPAT_REFERENCE = 1, 15

REGS = {SGD: dict(l1_w=1e-3, l1_v=1e-3, l2_w0=1e-2), FTRL: dict(l1_w=1e-3, l2_w=1e-3, l1_v=1e-4, l2_v=1e-3),
        TDAP: dict(l1_w=1e-3, l2_v=1e-3)}

# asserted tolerances (max relerr); the measured maxima on a B200 are in the docstrings of the GPU tests
TOL_F64_STEP = 1e-11
TOL_F64_TRAJ = 1e-9
TOL_F32_STEP = 1e-5              # SGD / FTRL / TDAP: MUFU exp / sqrt / rcp are <= 2 ulp
TOL_F32_HOT = 1e-4               # fp32 segments of ~2 000 entries: the sum of G rounds once per entry
TOL_F32_TAIL_TRAJ = 1e-5         # the fp32 FTRL run of test_minibatch_deterministic_and_truncated_tail (measured on a B200: 5.8e-8)

# kernel paths of K1 / K2 by (precision, k, fields): the TMA cases mix 300-id fields (dense tiles at B = 1024) with a 40 000-id
# field (its tiles span more rows than a stage holds: the sparse fallback) in one launch
WIDE = [300] * 8 + [40_000]               # 9 non-zeros per row: the stream K1 at fp32 k = 32
NARROW = [300] * 4 + [40_000]             # 5 non-zeros per row: the team K1
PATHS = {
    "f32-k1-tma-lpr1": ("f32", 1, WIDE),
    "f32-k5-tma-lpr2": ("f32", 5, WIDE),
    "f32-k16-tma-lpr4": ("f32", 16, WIDE),
    "f32-k32-teamK1-tma": ("f32", 32, NARROW),
    "f32-k32-streamK1-tma": ("f32", 32, WIDE),
    "f32-k48-gather-lpr16": ("f32", 48, WIDE),
    "f32-k100-gather-lpr32": ("f32", 100, WIDE),
    "f32-k200-gather-ch2": ("f32", 200, WIDE),
    "f64-k2-gather-lpr1": ("f64", 2, WIDE),
    "f64-k8-gather-lpr4": ("f64", 8, WIDE),
    "f64-k16-gather-lpr8": ("f64", 16, WIDE),
    "f64-k64-gather-lpr32": ("f64", 64, WIDE),
    "f64-k100-gather-ch2": ("f64", 100, WIDE),
}
TMA_PATHS = [k for k in PATHS if "tma" in k]


def random_state(rng, solver, task, regs, p, k):
    """non-trivial optimizer state: positive n / u / delta, non-zero z / nu / h / q and scal[1..7]"""
    ns = R.n_state(solver, task, regs.get("l1_w", 0.0), regs.get("l1_v", 0.0))
    sw = np.zeros((ns, p)); sv = np.zeros((ns, p, k))
    scal = np.concatenate([[0.0], rng.uniform(0.5, 2.0, 7) * np.where(rng.random(7) < 0.5, -1.0, 1.0)])
    if solver == FTRL:
        sw[0] = rng.normal(0, 0.5, p); sw[1] = rng.uniform(0.5, 2.0, p)
        sv[0] = rng.normal(0, 0.5, (p, k)); sv[1] = rng.uniform(0.5, 2.0, (p, k))
        scal[2] = abs(scal[2])                                   # n0 >= 0
    elif solver == TDAP:
        for a, shp in ((sw, (p,)), (sv, (p, k))):
            a[0] = rng.uniform(0.5, 2.0, shp); a[1] = rng.normal(0, 0.5, shp)
            a[2] = rng.uniform(5.0, 15.0, shp); a[3] = rng.normal(0, 0.5, shp)
        scal[1] = abs(scal[1]); scal[3] = abs(scal[3]) + 5.0     # u0 >= 0, delta0 > 0
    elif ns:
        sw[0] = rng.normal(0, 0.01, p); sv[0] = rng.normal(0, 0.01, (p, k))
        scal[1] = abs(scal[1]) * 0.01; scal[2] = abs(scal[2]) * 0.01   # u_w, u_v >= 0
    return dict(solver=solver, scal=scal, sw=sw, sv=sv)


def _labels(rng, n, task):
    if task == CLASSIFICATION:
        return np.where(rng.random(n) < 0.5, 1.0, -1.0).astype(np.float32)
    return rng.uniform(-0.3, 0.3, n).astype(np.float32)


def _base(name, rowptr, col, val, p, *, solver, task=CLASSIFICATION, k=8, prec="f64", B, max_iter=None, epochs=None,
          warm=False, seed=0, compat=COMPAT_REFERENCE, wscale=0.1, regs=None, tol=None, **kw):
    rng = np.random.default_rng(seed)
    n = rowptr.size - 1
    regs = dict(REGS[solver] if regs is None else regs)
    y = kw.pop("y", None)
    y = _labels(rng, n, task) if y is None else y
    w = rng.normal(0, wscale, p); v = rng.normal(0, wscale, (p, k)); w0 = float(rng.normal(0, wscale))
    state = random_state(rng, solver, task, regs, p, k) if warm else None
    row0 = 1 if compat & COMPAT_SKIP_ROW0 else 0
    if max_iter is None:
        max_iter = (epochs or 1) * (n - row0)
    if tol is None:
        if prec == "f64":
            tol = TOL_F64_STEP if warm and max_iter <= B else TOL_F64_TRAJ
        else:
            tol = TOL_F32_STEP
    c = dict(name=name, n=n, p=p, rowptr=rowptr, col=col, val=val, y=y, solver=solver, task=task, k=k, prec=prec, B=B,
             max_iter=max_iter, compat=compat, w0=w0, w=w, v=v, state=state, regs=regs, tol=tol, k0=1, k1=1, lr=0.01,
             alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0, gamma=1e-4, lo=float(np.min(y)), hi=float(np.max(y)),
             visit_order=None, step_size=-1, env={})
    c.update(kw)
    if prec == "f32":                                            # what an fp32 model holds after set / set_state
        c["w"] = c["w"].astype(np.float32).astype(np.float64); c["v"] = c["v"].astype(np.float32).astype(np.float64)
        if state is not None:
            state["sw"] = state["sw"].astype(np.float32).astype(np.float64)
            state["sv"] = state["sv"].astype(np.float32).astype(np.float64)
    return c


def _with_rows(n, p, rows):
    rowptr = np.concatenate([[0], np.cumsum([len(c) for c, _ in rows])]).astype(np.uint32)
    col = np.concatenate([np.asarray(c, np.uint32) for c, _ in rows] + [np.zeros(0, np.uint32)])
    val = np.concatenate([np.asarray(x, np.float32) for _, x in rows] + [np.zeros(0, np.float32)])
    return rowptr, col, val


def step_case(solver_name, path, gather=False):
    """one batch of 1024 rows from a random model and random optimizer state"""
    prec, k, fields = PATHS[path]
    solver = SOLVER_NAMES[solver_name]
    rowptr, col, val, p = synth.fields_csr(1025, fields, None, 1, 31)
    c = _base("step-%s-%s%s" % (solver_name, path, "-gatherenv" if gather else ""), rowptr, col, val, p, solver=solver, k=k,
              prec=prec, B=1024, max_iter=1024, warm=True, seed=32 + k)
    if gather:
        c["env"] = {"FMWR_K2_GATHER": "1"}
    return c


def bench_case(solver_name):
    """the benchmark's batch: 65 537 rows x 39 fields of 25 641 ids, k = 32, fp32, B = 65 536 with row 0 skipped (TDAP: the same
    batch : field ratio at 8 192 rows over 39 fields of 3 205 ids)"""
    solver = SOLVER_NAMES[solver_name]
    B, fid = (8192, 3205) if solver == TDAP else (65536, 25641)
    rowptr, col, val, p = synth.fields_csr(B + 1, [fid] * 39, None, 0, 41)
    return _base("bench-%s" % solver_name, rowptr, col, val, p, solver=solver, k=32, prec="f32", B=B, max_iter=B, warm=True,
                 seed=42, wscale=0.02)


def trajectory_case(name):
    """fp64 runs over two or more epochs"""
    if name == "traj-ftrl-tail":
        # B = 300 does not divide the 1 999-row epoch; the third epoch stops 150 rows into its first batch, and column p - 1
        # occurs only in rows 151 .. 300 (the cut part of that batch)
        n, p = 2000, 120
        rowptr, col, val = synth.random_csr(n, p - 1, 12, seed=51, empty_rows=True)
        rows = [(col[rowptr[r]:rowptr[r + 1]], val[rowptr[r]:rowptr[r + 1]]) for r in range(n)]
        for r in range(151, 301, 7):
            rows[r] = (np.append(rows[r][0], p - 1), np.append(rows[r][1], 0.9))
        return _base(name, *_with_rows(n, p, rows), p, solver=FTRL, k=6, B=300, max_iter=2 * (n - 1) + 150, seed=52)
    if name == "traj-sgd-onebatch-compat0":
        rowptr, col, val = synth.random_csr(2000, 150, 10, seed=53)
        return _base(name, rowptr, col, val, 150, solver=SGD, k=4, B=5000, epochs=3, compat=0, seed=54,
                     regs=dict(l2_w=1e-2, l2_v=2e-2, l2_w0=1e-2), lr=0.05)
    if name == "traj-tdap-skiprow0":
        rowptr, col, val = synth.random_csr(1500, 200, 9, seed=55)
        return _base(name, rowptr, col, val, 200, solver=TDAP, k=5, B=256, epochs=2, compat=COMPAT_SKIP_ROW0, seed=56)
    if name == "traj-ftrl-visit-order":
        rng = np.random.default_rng(57)
        rowptr, col, val = synth.random_csr(500, 60, 7, seed=58)
        visit = []
        while len(visit) < 1300:
            i = int(rng.integers(1, 5))
            while i < 500 and len(visit) < 1300:
                visit.append(i); i += int(rng.integers(1, 5))
        return _base(name, rowptr, col, val, 60, solver=FTRL, k=4, B=64, max_iter=1300, seed=59,
                     visit_order=np.array(visit, np.uint32))
    if name in ("traj-ftrl-nokeep", "traj-tdap-nokeep", "traj-sgd-nokeep"):
        solver = SOLVER_NAMES[name.split("-")[1]]
        rowptr, col, val = synth.random_csr(800, 90, 8, seed=60)
        return _base(name, rowptr, col, val, 90, solver=solver, k=4, B=100, epochs=2, seed=61, k0=0, k1=0)
    if name in ("traj-sgd-regression-clamp", "traj-ftrl-regression-clamp"):
        # labels in [-0.3, 0.3] and a model whose scores reach well past them: many multipliers come from the clamp
        solver = SOLVER_NAMES[name.split("-")[1]]
        rowptr, col, val = synth.random_csr(1200, 100, 10, seed=62)
        regs = dict(l1_w=1e-3, l1_v=1e-3) if solver == SGD else dict(l2_w=1e-3, l2_v=1e-3)
        return _base(name, rowptr, col, val, 100, solver=solver, task=REGRESSION, k=6, B=128, epochs=2, seed=63, wscale=0.4,
                     regs=regs)
    raise KeyError(name)


TRAJECTORIES = ["traj-ftrl-tail", "traj-sgd-onebatch-compat0", "traj-tdap-skiprow0", "traj-ftrl-visit-order", "traj-ftrl-nokeep",
                "traj-tdap-nokeep", "traj-sgd-nokeep", "traj-sgd-regression-clamp", "traj-ftrl-regression-clamp"]


def edge_case(name):
    """data edges, fp64 over two epochs unless the name says otherwise"""
    if name in ("edge-empty-rows-ftrl", "edge-empty-rows-sgd"):
        rowptr, col, val = synth.random_csr(1000, 80, 6, seed=70, empty_rows=True)
        assert (np.diff(rowptr.astype(np.int64)) == 0).sum() > 50
        solver = FTRL if name.endswith("ftrl") else SGD
        return _base(name, rowptr, col, val, 80, solver=solver, k=4, B=50, epochs=2, seed=71)
    if name == "edge-stored-zeros":
        # columns 0 .. 9 are stored only as 0.0: they take a step (FTRL refreshes theta from its state) without a gradient
        rng = np.random.default_rng(72)
        rowptr, col, val = synth.random_csr(900, 100, 8, seed=73)
        val = val.copy()
        val[col < 10] = 0.0
        val[rng.random(val.size) < 0.1] = 0.0
        return _base(name, rowptr, col, val, 100, solver=FTRL, k=4, B=64, epochs=2, seed=74)
    if name == "edge-tdap-one-nnz-rows":
        # half the rows hold one non-zero: their v-gradient is exactly 0 per entry (fresh state, TDAP)
        rng = np.random.default_rng(75)
        rows = []
        for r in range(1200):
            m = 1 if r % 2 else int(rng.integers(2, 6))
            c = np.sort(rng.choice(70, m, replace=False))
            rows.append((c, rng.uniform(-1.5, 1.5, m)))
        return _base(name, *_with_rows(1200, 70, rows), 70, solver=TDAP, k=4, B=40, epochs=2, seed=76)
    if name == "edge-wide-rows":
        rng = np.random.default_rng(77)
        rowptr, col, val = synth.random_csr(600, 400, 20, seed=78)
        rows = [(col[rowptr[r]:rowptr[r + 1]], val[rowptr[r]:rowptr[r + 1]]) for r in range(600)]
        for r in range(0, 600, 9):
            c = np.sort(rng.choice(400, 150, replace=False))
            rows[r] = (c, rng.uniform(0.5, 1.5, 150))
        return _base(name, *_with_rows(600, 400, rows), 400, solver=FTRL, k=5, B=70, epochs=2, seed=79)
    if name in ("edge-hot-feature", "edge-hot-feature-f32"):
        # a 4-id field: segments of ~2 000 entries at B = 8192
        rowptr, col, val, p = synth.fields_csr(16385, [4, 3000, 3000], None, 1, 80)
        if name.endswith("f32"):
            return _base(name, rowptr, col, val, p, solver=FTRL, k=16, prec="f32", B=8192, max_iter=8192, warm=True, seed=81,
                         tol=TOL_F32_HOT)
        return _base(name, rowptr, col, val, p, solver=FTRL, k=8, B=8192, epochs=2, seed=81)
    if name in ("edge-graph-chunk", "edge-plain-launches"):
        # 2 250 batches per epoch: the epoch crosses a CUDA-graph chunk (2 048 batches); step_size > 0 runs plain launches
        rowptr, col, val = synth.random_csr(4501, 300, 6, seed=82)
        c = _base(name, rowptr, col, val, 300, solver=FTRL, k=2, B=2, epochs=2, seed=83)
        if name == "edge-plain-launches":
            c["step_size"] = 1000
        return c
    raise KeyError(name)


EDGES = ["edge-empty-rows-ftrl", "edge-empty-rows-sgd", "edge-stored-zeros", "edge-tdap-one-nnz-rows", "edge-wide-rows",
         "edge-hot-feature", "edge-hot-feature-f32", "edge-graph-chunk", "edge-plain-launches"]


def truncated_tail_case():
    """the data of test_minibatch_deterministic_and_truncated_tail: one epoch and 1 234 rows of the next, fp32 FTRL k = 32, B = 512"""
    ds = synth.make_dataset("criteo", 5000, p=39 * 100)
    rng = np.random.default_rng(4)
    k = 32
    w = np.zeros(ds["p"]); v = rng.normal(0, 0.01, (ds["p"], k))
    c = _base("truncated-tail", ds["rowptr"], ds["col"], ds["val"], ds["p"], solver=FTRL, k=k, prec="f32", B=512,
              max_iter=4999 + 1234, y=ds["y"], regs={}, tol=TOL_F32_TAIL_TRAJ)
    c.update(w0=0.0, w=w, v=v.astype(np.float32).astype(np.float64))
    return c


def case(name):
    if name.startswith("step-"):
        parts = name.split("-")
        gather = name.endswith("-gatherenv")
        path = "-".join(parts[2:-1] if gather else parts[2:])
        return step_case(parts[1], path, gather)
    if name.startswith("bench-"):
        return bench_case(name.split("-")[1])
    if name.startswith("traj-"):
        return trajectory_case(name)
    if name.startswith("edge-"):
        return edge_case(name)
    if name == "truncated-tail":
        return truncated_tail_case()
    raise KeyError(name)


def reference(c, mutate=None):
    """the reference run of case c"""
    r = c["regs"]
    return R.train(c["solver"], c["task"], c["n"], c["p"], c["rowptr"], c["col"], c["val"], c["y"], c["w0"], c["w"], c["v"],
                   B=c["B"], max_iter=c["max_iter"], skip_row0=bool(c["compat"] & COMPAT_SKIP_ROW0), visit_order=c["visit_order"],
                   k0=c["k0"], k1=c["k1"], lr=c["lr"], alpha_w=c["alpha_w"], alpha_v=c["alpha_v"], beta_w=c["beta_w"],
                   beta_v=c["beta_v"], gamma=c["gamma"], l2_w0=r.get("l2_w0", 0.0), l1_w=r.get("l1_w", 0.0),
                   l2_w=r.get("l2_w", 0.0), l1_v=r.get("l1_v", 0.0), l2_v=r.get("l2_v", 0.0), lo=c["lo"], hi=c["hi"],
                   state=c["state"], f32_params=c["prec"] == "f32", mutate=mutate)
