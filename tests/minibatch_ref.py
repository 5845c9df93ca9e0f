"""fp64 numpy / scipy reference of one epoch loop of the throughput (minibatch) mode, vectorised per batch.

It restates the step that fmwr_b200/csrc/train_minibatch.cu defines (header, train_minibatch_t, mb_intercept, seg_finish) with
the per-coordinate optimizer steps of coord.cuh:

  batches   rows [row0 + b*B, ...) with row0 = 1 under COMPAT_SKIP_ROW0; the last batch of an epoch is short; max_iter counts rows
            and cuts the batch in which it runs out.  With an explicit visit order the visited rows (order[:max_iter]) are taken
            in visit order, row 0 is not skipped and there is one pass over them.
  K1        frozen parameters: score_r = [k0] w0 + [k1] sum w x + 1/2 sum_f (S_rf^2 - sum v^2 x^2), m_r = grad_mult(score_r).
  K2        every column with a stored entry in the batch (a stored 0.0 included) takes ONE optimizer step with
            G_w = sum_r m_r x_rc and G_v,f = sum_r m_r (S_rf x_rc - v_cf x_rc x_rc), the v-part formed per entry in that order.
  intercept SGD: the batch mean of m; FTRL / TDAP: the summed m, on the f64 scalar block.

Optimizer state uses the layout of Model.get_state(): sw[n_state][p], sv[n_state][p][k], scal[8] (scal[0] = w0).
  SGD with cumulative L1 (classification): sw/sv[0] = q, scal[1..2] = u_w, u_v.  Other SGD: no arrays.
  FTRL: [0] = z, [1] = n; scal[1] = z0, scal[2] = n0.
  TDAP: [0] = u, [1] = nu, [2] = delta, [3] = h; scal[1..5] = u0, nu0, delta0, h0, z0.

`mutate` names one deliberate deviation from the definition (MUTATIONS); the tests use them as negative controls that show
how far a subtly wrong step lands from the right one.
"""
import numpy as np
import scipy.sparse as sp

CLASSIFICATION, REGRESSION = 10, 20
SGD, FTRL, TDAP = 300, 500, 600

MUTATIONS = (
    "drop_entry",         # drop the last entry of every segment that has more than one
    "no_vb",              # G_v without its -v x^2 part
    "intercept_form",     # FTRL / TDAP intercept from the batch mean, SGD from the batch sum
    "drop_last_row",      # the last row of every batch takes no part in the step
    "skip_zero_touch",    # a column whose batch entries are all stored zeros takes no step
    "apply_tail",         # the batch cut by max_iter is applied in full
)


def n_state(solver, task, l1_w=0.0, l1_v=0.0):
    if solver == SGD:
        return 1 if (l1_w > 0 or l1_v > 0) and task == CLASSIFICATION else 0
    return 2 if solver == FTRL else 4


def _f32(x):
    return float(np.float32(x))


def train(solver, task, n, p, rowptr, col, val, y, w0, w, v, *, B, max_iter, skip_row0=True, visit_order=None, k0=1, k1=1,
          lr=0.01, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0, gamma=1e-4, l2_w0=0.0, l1_w=0.0, l2_w=0.0, l1_v=0.0,
          l2_v=0.0, lo=-1.0, hi=1.0, state=None, f32_params=False, mutate=None):
    """returns dict(w0, w, v, scal, sw, sv) after max_iter rows of the throughput mode.

    state: optional dict(sw, sv, scal) to start from (warm state); zeros otherwise.
    f32_params: round the hyper-parameters to fp32, as an fp32 model's kernels receive them (the inputs w, v, state are the
    caller's to round)."""
    assert mutate is None or mutate in MUTATIONS, mutate
    rowptr = np.asarray(rowptr, np.int64)
    col = np.asarray(col, np.int64)
    val = np.asarray(val, np.float64)
    y = np.asarray(y, np.float64)
    if visit_order is not None:
        order = np.asarray(visit_order, np.int64)[:max_iter]
        cnt = rowptr[order + 1] - rowptr[order]
        idx = np.concatenate([np.arange(rowptr[r], rowptr[r + 1]) for r in order]) if cnt.sum() else np.zeros(0, np.int64)
        rowptr = np.concatenate([[0], np.cumsum(cnt)])
        col, val, y = col[idx], val[idx], y[order]
        n = order.size
        skip_row0 = False
        max_iter = n
    k = v.shape[1]
    w = np.array(w, np.float64, copy=True)
    v = np.array(v, np.float64, copy=True).reshape(p, k)
    ns = n_state(solver, task, l1_w, l1_v)
    if state is None:
        sw = np.zeros((ns, p)); sv = np.zeros((ns, p, k)); sc = np.zeros(8)
    else:
        sw = np.array(state["sw"], np.float64, copy=True).reshape(ns, p)
        sv = np.array(state["sv"], np.float64, copy=True).reshape(ns, p, k)
        sc = np.array(state["scal"], np.float64, copy=True)
    sc[0] = w0
    rnd = _f32 if f32_params else float
    lr, alpha_w, alpha_v, beta_w, beta_v = rnd(lr), rnd(alpha_w), rnd(alpha_v), rnd(beta_w), rnd(beta_v)
    l1_w, l2_w, l1_v, l2_v, l2_w0 = rnd(l1_w), rnd(l2_w), rnd(l1_v), rnd(l2_v), rnd(l2_w0)
    eg = rnd(np.exp(-gamma))
    l1 = False
    if solver == SGD:
        # SGD_Learner::init: any L1 > 0 selects the L1 rates; L1 proper only for classification, else they act as L2 rates
        l1 = (l1_w > 0 or l1_v > 0) and task == CLASSIFICATION
        rw, rv = (l1_w, l1_v) if (l1_w > 0 or l1_v > 0) else (l2_w, l2_v)
        uw, uv = (sc[1], sc[2]) if (l1 and state is not None) else (0.0, 0.0)
    row0 = 1 if skip_row0 else 0
    it = 0
    if n - row0 <= 0:
        return dict(w0=sc[0], w=w, v=v, scal=sc, sw=sw, sv=sv)
    while it < max_iter:
        for rb in range(row0, n, B):
            if it >= max_iter:
                break
            rows = min(B, n - rb, max_iter - it)
            used = min(B, n - rb) if mutate == "apply_tail" else rows
            inc = used - 1 if mutate == "drop_last_row" else used       # rows whose entries and multipliers take part
            e0, e1 = rowptr[rb], rowptr[rb + inc]
            rl = np.repeat(np.arange(inc), np.diff(rowptr[rb:rb + inc + 1]))
            c, x = col[e0:e1], val[e0:e1]
            Xb = sp.csr_matrix((x, c, rowptr[rb:rb + inc + 1] - e0), shape=(inc, p))
            S = np.asarray(Xb @ v)
            score = 0.5 * (S * S - np.asarray(Xb.multiply(Xb) @ (v * v))).sum(1)
            if k1:
                score = np.asarray(Xb @ w).ravel() + score
            if k0:
                score = sc[0] + score
            yb = y[rb:rb + inc]
            if task == REGRESSION:
                m = -(yb - np.clip(score, lo, hi))
            else:
                m = -yb * (1.0 - 1.0 / (1.0 + np.exp(-yb * score)))
            gsum = float(m.sum())
            # segments: the batch's entries sorted by (column, row)
            o = np.argsort(c, kind="stable")
            c, x, rl = c[o], x[o], rl[o]
            keep = np.ones(c.size, bool)
            if mutate == "drop_entry":
                last = np.ones(c.size, bool); last[:-1] = c[1:] != c[:-1]
                prev = np.zeros(c.size, bool); prev[1:] = c[1:] == c[:-1]
                keep = ~(last & prev)                    # a segment's last entry, unless it is also its first
            if mutate == "skip_zero_touch":
                nz = np.unique(c[x != 0.0])
                keep &= np.isin(c, nz)
            c, x, rl = c[keep], x[keep], rl[keep]
            touched, start = np.unique(c, return_index=True)
            mx = m[rl] * x
            if touched.size:
                Gw = np.add.reduceat(mx, start)
                ve = v[c] * x[:, None] * x[:, None]
                ge = m[rl, None] * (S[rl] * x[:, None] - (0.0 if mutate == "no_vb" else ve))
                Gv = np.add.reduceat(ge, start, axis=0)
                th_w, th_v = w[touched], v[touched]
            if solver == SGD:
                if l1:
                    uw += used * lr * rw; uv += used * lr * rv

                def sgd(th, g, reg, u, q):
                    th = th - lr * g
                    if not l1:
                        return th - lr * reg * th, q
                    old = th
                    pos = np.maximum(0.0, old - (u + q)); neg = np.minimum(0.0, old + (u - q))
                    th = np.where(old > 0, pos, np.where(old < 0, neg, old))
                    return th, q + th - old
                if touched.size:
                    if k1:
                        q = sw[0, touched] if l1 else None
                        w[touched], q = sgd(th_w, Gw, rw, uw, q)
                        if l1:
                            sw[0, touched] = q
                    q = sv[0, touched] if l1 else None
                    v[touched], q = sgd(th_v, Gv, rv, uv, q)
                    if l1:
                        sv[0, touched] = q
                if k0:
                    g0 = gsum if mutate == "intercept_form" else gsum / used
                    sc[0] -= lr * (g0 + l2_w0 * sc[0])
            elif solver == FTRL:
                def ftrl(th, g, z, nn, a, b, l1_, l2_):
                    n2 = nn + g * g
                    sig = (np.sqrt(n2) - np.sqrt(nn)) / a
                    z = z + g - sig * th
                    r = -(z - np.where(z < 0, -1.0, 1.0) * l1_) / ((b + np.sqrt(n2)) / a + l2_)
                    return np.where(np.abs(z) <= l1_, 0.0, r), z, n2
                if touched.size:
                    if k1:
                        w[touched], sw[0, touched], sw[1, touched] = ftrl(th_w, Gw, sw[0, touched], sw[1, touched], alpha_w, beta_w, l1_w, l2_w)
                    v[touched], sv[0, touched], sv[1, touched] = ftrl(th_v, Gv, sv[0, touched], sv[1, touched], alpha_v, beta_v, l1_v, l2_v)
                if k0:
                    g0 = gsum / used if mutate == "intercept_form" else gsum
                    old = sc[2]; sc[2] += g0 * g0
                    sc[1] += g0 - (np.sqrt(sc[2]) - np.sqrt(old)) / alpha_w * sc[0]
                sc[0] = -sc[1] * alpha_w / (beta_w + np.sqrt(sc[2]))
            else:
                def tdap(th, g, u, nu, dl, h, a, l1_, l2_):
                    u2 = u + g * g; nu = nu + g
                    sig = (np.sqrt(u2) - np.sqrt(u)) / a
                    dl = eg * (dl + sig); h = eg * (h + sig * th)
                    z = nu - h
                    with np.errstate(invalid="ignore", divide="ignore"):
                        r = -(z - np.where(z < 0, -1.0, 1.0) * l1_) / (dl + l2_)
                    return np.where(np.abs(z) <= l1_, 0.0, r), u2, nu, dl, h
                if touched.size:
                    if k1:
                        w[touched], *st = tdap(th_w, Gw, *[sw[i, touched] for i in range(4)], alpha_w, l1_w, l2_w)
                        for i in range(4):
                            sw[i, touched] = st[i]
                    v[touched], *st = tdap(th_v, Gv, *[sv[i, touched] for i in range(4)], alpha_v, l1_v, l2_v)
                    for i in range(4):
                        sv[i, touched] = st[i]
                if k0:
                    g0 = gsum / used if mutate == "intercept_form" else gsum
                    old = sc[1]; sc[1] += g0 * g0; sc[2] += g0
                    sig = (np.sqrt(sc[1]) - np.sqrt(old)) / alpha_w
                    sc[3] = eg * (sc[3] + sig); sc[4] = eg * (sc[4] + sig * sc[0]); sc[5] = sc[2] - sc[4]
                with np.errstate(invalid="ignore", divide="ignore"):
                    sc[0] = -sc[5] / sc[3]
            it += rows
    if solver == SGD and l1:
        sc[1], sc[2] = uw, uv
    return dict(w0=sc[0], w=w, v=v, scal=sc, sw=sw, sv=sv)


def max_relerr(a, b):
    """max over w0, w, v, scal and every state array of max |a - b| / max(1, |b|) (NaN == NaN)"""
    worst = 0.0
    for key in ("w", "v", "scal", "sw", "sv"):
        x = np.asarray(a[key], np.float64); r = np.asarray(b[key], np.float64)
        assert x.shape == r.shape, (key, x.shape, r.shape)
        if x.size == 0:
            continue
        both_nan = np.isnan(x) & np.isnan(r)
        d = np.where(both_nan, 0.0, np.abs(x - r) / np.maximum(1.0, np.abs(r)))
        worst = max(worst, float(np.max(np.where(np.isnan(d), np.inf, d))))
    return worst
