"""The fp64 reference of the throughput-mode step (tests/minibatch_ref.py), checked on the CPU:

(a) at batch = 1 it is the exact mode: it equals the plain-C restatement (the `port` oracle) to 1e-13 for SGD (L2, cumulative L1,
    L1-as-L2 regression), FTRL and TDAP in both tasks, on data with empty rows, over two epochs and a few rows;
(b) negative controls: on the inputs of the GPU tests (tests/minibatch_cases.py), each deliberate deviation from the defined
    batch step moves the result by at least 10x the tolerance that the matching GPU test asserts, so those tolerances would
    catch it."""
import numpy as np
import pytest

from oracle import oracle as O
from fmwr_b200 import synth
from tests import minibatch_cases as MC
from tests import minibatch_ref as R
from tests.util import relerr

BATCH1_CASES = [(O.SGD, O.CLASSIFICATION, dict(l2_w=0.01, l2_v=0.02, l2_w0=0.01)), (O.SGD, O.CLASSIFICATION, dict(l1_w=0.01, l1_v=0.01)),
                (O.SGD, O.REGRESSION, dict(l1_w=0.01, l1_v=0.01)), (O.FTRL, O.CLASSIFICATION, dict(l1_w=0.01, l2_w=0.01, l1_v=0.01, l2_v=0.02)),
                (O.FTRL, O.REGRESSION, dict(l2_w=0.01)), (O.TDAP, O.CLASSIFICATION, dict(l1_w=0.001, l2_v=0.01)), (O.TDAP, O.REGRESSION, dict())]


@pytest.mark.parametrize("solver,task,regs", BATCH1_CASES, ids=["sgd-l2", "sgd-l1", "sgd-regression-l1-as-l2", "ftrl", "ftrl-regression",
                                                                "tdap", "tdap-regression"])
def test_reference_at_batch1_equals_port(port, solver, task, regs):
    rng = np.random.default_rng(1)
    n, p, k = 300, 50, 4
    if solver == O.TDAP:
        # columns 0 .. m-1 in every row (position == column): the port's F6 (TDAP z_w indexed by position) cannot act
        rp, cc, vv = [0], [], []
        for _ in range(n):
            m = int(rng.integers(0, 8)); cc += list(range(m)); vv += list(rng.uniform(-1.5, 1.5, m)); rp.append(len(cc))
        rowptr, col, val = np.array(rp, np.uint32), np.array(cc, np.uint32), np.array(vv, np.float32)
    else:
        rowptr, col, val = synth.random_csr(n, p, 7, seed=2, empty_rows=True)
    assert (np.diff(rowptr.astype(np.int64)) == 0).any()
    y = (np.where(rng.random(n) < 0.5, 1.0, -1.0) if task == O.CLASSIFICATION else rng.normal(0, 1, n)).astype(np.float32)
    lo, hi = float(y.min()), float(y.max())
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.1, (p, k))
    iters = 2 * (n - 1) + 5
    cfg = O.make_cfg(solver=solver, task=task, k=k, max_iter=iters, min_target=lo, max_target=hi, **regs)
    rw0, rw, rv, _ = port.train(cfg, n, p, rowptr, col, val, y, 0.2, w, v)
    got = R.train(solver, task, n, p, rowptr, col, val, y, 0.2, w, v, B=1, max_iter=iters, lo=lo, hi=hi, **regs)
    assert relerr(got["w0"], rw0) <= 1e-13 and relerr(got["w"], rw) <= 1e-13 and relerr(got["v"], rv) <= 1e-13
    assert np.abs(got["v"] - v).max() > 1e-3                     # it trained


# each mutation against the GPU cases that exercise what it breaks
NEGATIVE = [
    ("drop_entry", "step-ftrl-f32-k32-streamK1-tma"), ("drop_entry", "step-tdap-f32-k16-tma-lpr4"), ("drop_entry", "step-sgd-f64-k8-gather-lpr4"),
    ("drop_entry", "traj-ftrl-tail"),
    ("no_vb", "step-ftrl-f32-k32-streamK1-tma"), ("no_vb", "step-sgd-f32-k5-tma-lpr2"), ("no_vb", "step-tdap-f32-k16-tma-lpr4"),
    ("no_vb", "traj-sgd-onebatch-compat0"),
    ("intercept_form", "step-ftrl-f32-k32-streamK1-tma"), ("intercept_form", "step-sgd-f32-k32-streamK1-tma"),
    ("intercept_form", "step-tdap-f32-k16-tma-lpr4"), ("intercept_form", "edge-empty-rows-sgd"),
    ("drop_last_row", "step-ftrl-f32-k32-streamK1-tma"), ("drop_last_row", "step-sgd-f32-k1-tma-lpr1"), ("drop_last_row", "traj-sgd-onebatch-compat0"),
    ("skip_zero_touch", "edge-stored-zeros"),
    ("apply_tail", "traj-ftrl-tail"), ("apply_tail", "truncated-tail"),
    ("drop_entry", "edge-hot-feature-f32"), ("no_vb", "edge-hot-feature-f32"), ("intercept_form", "edge-hot-feature-f32"),
]


@pytest.mark.parametrize("mutation,case", NEGATIVE, ids=["%s-%s" % mc for mc in NEGATIVE])
def test_mutated_step_exceeds_the_gpu_tolerance(mutation, case):
    c = MC.case(case)
    good = MC.reference(c)
    bad = MC.reference(c, mutate=mutation)
    moved = R.max_relerr(bad, good)
    assert moved >= 10 * c["tol"], "%s on %s moves the result by %.3g only (tolerance %.1g)" % (mutation, case, moved, c["tol"])


def test_cut_column_is_untouched_in_the_last_epoch():
    """traj-ftrl-tail: the column that only the cut rows hold keeps its value from the end of the second epoch"""
    c = MC.case("traj-ftrl-tail")
    full = MC.reference(c)
    two = MC.reference(dict(c, max_iter=2 * (c["n"] - 1)))
    assert np.array_equal(full["v"][-1], two["v"][-1]) and np.array_equal(full["sv"][:, -1], two["sv"][:, -1])
    assert not np.array_equal(MC.reference(c, mutate="apply_tail")["v"][-1], two["v"][-1])
