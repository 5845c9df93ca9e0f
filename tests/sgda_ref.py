"""fp64 numpy restatement of SGDA (fmwr_train_sgda_dev, include/fmwr_b200.h): SGD in exact mode that takes, from the second pass
over the training visit sequence on, one gradient step on the per-group L2 rates after every training step, on one validation row.

Data sets are dicts with rowptr, col, val (the CSR arrays of the device handle) and y.  The visit sequence is the explicit
`order` when given (cycled), else the scan of rows skip_row0 .. n-1 (F5); lambda steps start at sample t0, by default one pass of
that sequence.  lambda_step=False leaves the rates alone (the negative control)."""
import numpy as np

CLASSIFICATION, REGRESSION = 10, 20


def grad_mult(task, p, y, lo, hi):
    """calculate_grad_mult of SGD (regression: the score clamped to [lo, hi])"""
    if task == REGRESSION:
        return -(y - min(hi, max(lo, p)))
    return -y * (1.0 - 1.0 / (1.0 + np.exp(-y * p)))


def row(ds, r):
    b, e = int(ds["rowptr"][r]), int(ds["rowptr"][r + 1])
    return np.asarray(ds["col"][b:e], np.int64), np.asarray(ds["val"][b:e], np.float64)


def lookahead(w0, w, V, gw, gv, lam_w, lam_v, groups, cols, x, lr, k0=1, k1=1):
    """The validation row's look-ahead score p' and its gradients d p' / d lam_w [G] and d p' / d lam_v [G, k]"""
    g = groups[cols]
    wp = w[cols] - lr * (gw[cols] + lam_w[g] * w[cols])
    vp = V[cols] - lr * (gv[cols] + lam_v[g] * V[cols])
    vx = vp * x[:, None]
    Sp = vx.sum(0)
    p1 = (w0 if k0 else 0.0) + (float(wp @ x) if k1 else 0.0) + 0.5 * float(Sp @ Sp - (vx * vx).sum())
    dw = np.zeros(lam_w.shape)
    dv = np.zeros(lam_v.shape)
    if k1:
        np.add.at(dw, g, -lr * x * w[cols])
    np.add.at(dv, g, -lr * x[:, None] * V[cols] * (Sp[None, :] - x[:, None] * vp))
    return p1, dw, dv


def sgda(train, valid, task, w0, w, V, lam_w, lam_v, groups, lr, max_iter, order=None, skip_row0=True, k0=1, k1=1, reg_w0=0.0,
         lo=None, hi=None, lambda_step=True, t0=None):
    """Returns (w0, w, V, lam_w, lam_v) after max_iter samples"""
    w = np.array(w, np.float64)
    V = np.array(V, np.float64)
    lam_w = np.array(lam_w, np.float64)
    lam_v = np.array(lam_v, np.float64)
    groups = np.asarray(groups, np.int64)
    gw = np.zeros_like(w)
    gv = np.zeros_like(V)
    n = len(train["rowptr"]) - 1
    nval = len(valid["rowptr"]) - 1
    lo = float(np.min(train["y"])) if lo is None else lo
    hi = float(np.max(train["y"])) if hi is None else hi
    period = len(order) if order is not None else n - int(skip_row0)
    t0 = period if t0 is None else t0
    for t in range(max_iter):
        q = t % period
        r = int(order[q]) if order is not None else q + int(skip_row0)
        cols, x = row(train, r)
        vx = V[cols] * x[:, None]
        S = vx.sum(0)
        p = (w0 if k0 else 0.0) + (float(w[cols] @ x) if k1 else 0.0) + 0.5 * float(S @ S - (vx * vx).sum())
        m = grad_mult(task, p, float(train["y"][r]), lo, hi)
        g = groups[cols]
        if k1:
            gw[cols] = m * x
            w[cols] = w[cols] - lr * (gw[cols] + lam_w[g] * w[cols])
        gv[cols] = m * (S[None, :] * x[:, None] - V[cols] * x[:, None] ** 2)
        V[cols] = V[cols] - lr * (gv[cols] + lam_v[g] * V[cols])
        if k0:
            w0 -= lr * (m + reg_w0 * w0)
        if lambda_step and t >= t0:
            u = (t - t0) % nval
            cols, x = row(valid, u)
            p1, dw, dv = lookahead(w0, w, V, gw, gv, lam_w, lam_v, groups, cols, x, lr, k0, k1)
            m1 = grad_mult(task, p1, float(valid["y"][u]), lo, hi)
            present = np.unique(groups[cols])
            if k1:
                lam_w[present] = np.maximum(0.0, lam_w[present] - lr * m1 * dw[present])
            lam_v[present] = np.maximum(0.0, lam_v[present] - lr * m1 * dv[present])
    return w0, w, V, lam_w, lam_v
