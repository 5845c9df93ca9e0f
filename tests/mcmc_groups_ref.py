"""TEST INFRASTRUCTURE ONLY -- fp64 numpy restatement of the grouped MCMC sampler (fmwr_solver_cfg::attr_group).

The reference ships one attribute group, so the multi-group rules are this project's (include/fmwr_b200.h, at the attr_group
field) and no reference code exists for them.  This module states them once, in the operation order of the plain-C
restatement's MCMC loop (oracle/fm_oracle.c: learn_mcmc_als, exact Gauss-Seidel in feature order), with injected streams:

  per sweep  e = predict (the oracle's own predict_batch) -> e -= y, or the truncated-normal draw of classification (the oracle's
             trnorm_left / trnorm_right on its injected rand() stream) -> alpha -> w0 -> lambda_w[0..G-1] -> mu_w[0..G-1] -> w pass
             -> lambda_v (f outer, g inner) -> mu_v (same order) -> V pass on local copies of e and q

  lambda[g] ~ Gamma((alpha_0 + p_g + 1) / 2, scale 2 / (sum_{i in I_g} (x_i - mu[g])^2 + (beta_0 (mu[g] - mu_0)^2 + gamma_0)))
  mu[g]     ~ N((s_g + beta_0 mu_0) / (p_g + beta_0), variance 1 / ((p_g + beta_0) lambda[g]))

with s_g = sum_{i in I_g} x_i, or (FMWR_COMPAT_MCMC_VMU_IDX, V only) v_gf added p_g times; the coordinate step of feature i uses
group attr_group[i]'s pair, and FMWR_COMPAT_MCMC_W_SD draws w with the variance as s.d.  Constants as MCMC_ALS_Learner::init
forces them (alpha_0 = gamma_0 = beta_0 = 1, mu_0 = 0).  With one group and compat = FMWR_COMPAT_REFERENCE this is the shipped
sampler, and tests/test_mcmc_groups_reference.py holds it to the C restatement there.
"""
import math

import numpy as np

from oracle import oracle as O

COMPAT_MCMC_W_SD, COMPAT_MCMC_VMU_IDX = 4, 8


def _seq(a):
    """sum in index order (the C loops' order)"""
    s = 0.0
    for x in a.tolist():
        s += x
    return s


def _bad(x):
    return math.isnan(x) or math.isinf(x)


class _Stream:
    def __init__(self, a, what):
        self.a, self.i, self.what = (np.asarray(a, np.float64) if a is not None else np.zeros(0)), 0, what

    def next(self):
        if self.i >= self.a.size:
            raise ValueError("injected %s stream exhausted" % self.what)
        self.i += 1
        return float(self.a[self.i - 1])


def train(port, task, n, p, k, rowptr, col, val, y, w0, w, v, sweeps, enable_v, l2_w0, streams, attr_group=None, n_groups=1,
          compat=15):
    """returns (w0, w [p], V [p][k]) after `sweeps` grouped MCMC sweeps; streams = (normals, gammas, rands)"""
    alpha_0 = gamma_0 = beta_0 = 1.0
    mu_0 = 0.0
    normals, gammas, rands = streams
    nz, gz = _Stream(normals, "normal"), _Stream(gammas, "gamma")
    rowptr = np.ascontiguousarray(rowptr, np.uint32); col = np.ascontiguousarray(col, np.uint32); val = np.ascontiguousarray(val, np.float32)
    y = np.asarray(y, np.float32)
    w = np.array(w, np.float64); v = np.array(v, np.float64).reshape(p, k)
    G = int(n_groups) if attr_group is not None else 1
    grp = np.asarray(attr_group, np.int64) if attr_group is not None else np.zeros(p, np.int64)
    members = [np.nonzero(grp == g)[0] for g in range(G)]
    cnt = np.array([m.size for m in members], np.float64)
    cfg = O.make_cfg(task=task, solver=O.MCMC, k=k, max_iter=1, enable_v=enable_v, l2_w0=l2_w0)
    tp, ti, tv = port.transpose(n, p, rowptr, col, val, 0)
    cols = [(ti[tp[i]:tp[i + 1]].astype(np.int64), tv[tp[i]:tp[i + 1]].astype(np.float64),
             (tv[tp[i]:tp[i + 1]] * tv[tp[i]:tp[i + 1]]).astype(np.float64)) for i in range(p)]   # x*x of a float x is a float
    alpha = 1.0
    w_lam, w_mu = np.zeros(G), np.zeros(G)
    v_lam, v_mu = np.zeros((k, G)), np.zeros((k, G))

    def draw_lambda(x, lam, mu):
        """lambda[g] for g = 0..G-1 over the column x (w, or factor f of V)"""
        for g in range(G):
            xs = x[members[g]]
            gg = _seq((xs - mu[g]) * (xs - mu[g])) + (beta_0 * (mu[g] - mu_0) * (mu[g] - mu_0) + gamma_0)
            nl = 2.0 / gg * gz.next()
            if not _bad(nl):
                lam[g] = nl

    def draw_mu(x, lam, mu, from_row):
        """mu[g] for g = 0..G-1; from_row: the sum is x[g] added p_g times"""
        for g in range(G):
            if from_row:
                s = 0.0
                for _ in range(int(cnt[g])):
                    s += x[g]
            else:
                s = _seq(x[members[g]])
            m = (s + beta_0 * mu_0) / (cnt[g] + beta_0)
            nm = m + math.sqrt(1.0 / ((cnt[g] + beta_0) * lam[g])) * nz.next()
            if not _bad(nm):
                mu[g] = nm

    port.set_streams(None, None, rands)          # the truncated-normal draws consume the oracle's rand() stream
    try:
        for _ in range(sweeps):
            err = port.predict(cfg, n, p, rowptr, col, val, w0, w, v, 0)
            if task == O.REGRESSION:
                err -= y.astype(np.float64)
            else:
                for i in range(n):
                    e = float(err[i])
                    err[i] -= port.trnorm_left(e) if y[i] >= 0.0 else port.trnorm_right(e)
            gamma_n = gamma_0
            for e in err.tolist():
                gamma_n += e * e
            a = 2.0 / gamma_n * gz.next()
            if not _bad(a):
                alpha = a
            e_sum = 0.0
            for e in err.tolist():
                e_sum += e - w0
            var = 1.0 / (l2_w0 + alpha * n)
            nw = -(alpha * e_sum - 0.0 * l2_w0) * var + math.sqrt(var) * nz.next()
            if _bad(nw):
                nw = w0
            err -= w0 - nw
            w0 = nw
            draw_lambda(w, w_lam, w_mu)
            draw_mu(w, w_lam, w_mu, False)
            for i in range(p):
                r, x, xx = cols[i]
                old = w[i]
                lam, mu = w_lam[grp[i]], w_mu[grp[i]]
                var = 1.0 / (lam + alpha * _seq(x * x))
                mean = -var * (alpha * _seq(err[r] * x - old * x * x) - mu * lam)
                if _bad(var):                     # (a normal is drawn only for a finite variance, as in the C loop)
                    nv = 0.0
                else:
                    nv = mean + (var if compat & COMPAT_MCMC_W_SD else math.sqrt(var)) * nz.next()
                upd = True
                if _bad(nv):
                    nv, upd = old, False
                w[i] = nv
                if upd:
                    err[r] -= x * (old - nv)
            if enable_v and k > 0:
                for f in range(k):                # lambda_v: f outer, g inner; then mu_v in the same order
                    draw_lambda(v[:, f], v_lam[f], v_mu[f])
                for f in range(k):
                    draw_mu(v[:, f], v_lam[f], v_mu[f], bool(compat & COMPAT_MCMC_VMU_IDX))
                e2 = err.copy()
                for f in range(k):
                    vq = np.zeros(n)
                    for i in range(p):
                        r, x, _ = cols[i]
                        vq[r] += x * v[i, f]
                    for i in range(p):
                        r, x, xx = cols[i]
                        old = v[i, f]
                        lam, mu = v_lam[f, grp[i]], v_mu[f, grp[i]]
                        h = x * vq[r] - xx * old
                        mean, var = _seq(h * e2[r]), _seq(h * h)
                        mean -= old * var
                        var = 1.0 / (lam + alpha * var)
                        mean = -var * (alpha * mean - mu * lam)
                        nv = 0.0 if _bad(var) else mean + math.sqrt(var) * nz.next()
                        upd = True
                        if _bad(nv):
                            nv, upd = old, False
                        v[i, f] = nv
                        if upd:
                            d = old - nv
                            vq[r] -= x * d
                            e2[r] -= h * d
    finally:
        port.set_streams(None, None, None)
    return w0, w, v
