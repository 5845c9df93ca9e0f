"""Cost and effect of MCMC attribute groups (fmwr_solver_cfg::attr_group).

Cost: the configs[3] workload bench.py builds (20M ratings x 3 one-hot fields [138493, 26744, 2048], skew [0, 1, 0]), k = 64,
fp32, V block on.  S sweeps of fmwr_train_dev with no map and with groups = the three fields, alternating within every repeat,
each from the same initial model; medians, the grouped overhead, and the card name and power limit read in the same run.

Effect: planted data whose three fields' linear effects (and factors) differ in scale by 100x; held-out RMSE of the posterior
mean (fm_posterior) with one group and with groups = fields, same seed and controls.  Reported as measured.

    python profiles/tools/mcmc_groups_cost.py [--sweeps 10] [--repeats 6] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from fmwr_b200 import _lib as L  # noqa: E402
from fmwr_b200 import api as A  # noqa: E402
from fmwr_b200 import synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    return q.stdout.strip()


def cost(say, S, repeats):
    ctx = L.Context(0)
    na = 20_000_000
    fields, skew, k = [138493, 26744, 2048], [0, 1, 0], 64
    pa = sum(fields)
    da = L.Data.synth(ctx, na, fields, skew, 0, 3, 0.3, 20240601)
    m = L.Model(ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=k), pa, L.F32)
    grp = np.ascontiguousarray(np.repeat(np.arange(3), fields), np.int32)

    def cfg(grouped):
        sc = L.SolverCfg(solver=L.MCMC, max_iter=S, random_step=1, min_target=0.5, max_target=5.0, mode=L.MODE_EXACT,
                         precision=L.F32, compat=L.COMPAT_REFERENCE, enable_v=1, step_size=-1, seed=5)
        if grouped:
            sc.attr_group = L.ptr(grp); sc.n_groups = 3
        return sc

    cfgs = {"one group": cfg(False), "3 groups": cfg(True)}
    times = {name: [] for name in cfgs}
    for rep in range(repeats + 1):                       # repeat 0 warms both paths up and is not counted
        for name, sc in cfgs.items():
            m.init_random(0.0, 0.01, 20240603)
            ctx.sync()
            ctx.timer_start()
            L.train_dev(ctx, m, da, sc)
            ms = ctx.timer_stop_ms()
            model = m.get()
            assert np.isfinite(model[0]) and all(np.all(np.isfinite(a)) for a in model[1:])
            if rep > 0:
                times[name].append(ms)
    say("card (name, power limit, max SM clock): %s" % card())
    say("cost: configs[3], %d ratings x 3 one-hot fields %s skew %s, k=%d, fp32, enable_v=1; %d MCMC sweeps per run; "
        "median of %d alternating repeats, each from the same initial model and seed" % (na, fields, skew, k, S, repeats))
    base = statistics.median(times["one group"])
    for name, t in times.items():
        med = statistics.median(t)
        say("  %-10s %9.2f ms  (%7.2f ms/sweep)  range %.2f .. %.2f ms  overhead %+6.2f %%" % (
            name, med, med / S, min(t), max(t), 100.0 * (med - base) / base))
    m.close(); da.close(); ctx.close()


def effect(say):
    fields, scales, k = [3000, 600, 40], [1.0, 0.1, 0.01], 4
    n_tr, n_te = 150_000, 50_000
    p = sum(fields)
    rng = np.random.default_rng(71)
    grp = np.repeat(np.arange(3), fields).astype(np.int32)
    sd = np.asarray(scales)[grp]
    w_star = rng.normal(0, 1, p) * sd
    v_star = rng.normal(0, 0.5, (p, k)) * np.sqrt(sd)[:, None]

    def make(n, seed):
        rowptr, col, val, _ = synth.fields_csr(n, fields, [0, 1, 0], 0, seed)
        c = col.reshape(n, 3).astype(np.int64)
        xv = v_star[c].sum(1)
        y = 3.0 + w_star[c].sum(1) + 0.5 * np.sum(xv * xv - np.sum(v_star[c] ** 2, 1), 1) + 0.1 * rng.standard_normal(n)
        import scipy.sparse as sp
        X = sp.csr_matrix((val.astype(np.float64), col.astype(np.int64), rowptr.astype(np.int64)), shape=(n, p))
        return A.fm_matrix(X, y), y

    tr, _ = make(n_tr, 72)
    te, y_te = make(n_te, 73)
    saved = A.options()["FM.enable_v"]
    A.options(**{"FM.enable_v": True})
    sweeps, burn = 60, 20
    ctl = [A.model_control("REGRESSION", factor_number=k), A.solver_control(max_iter=sweeps, solver=A.MCMC_solver()),
           A.track_control(step_size=-1, evaluate_metric="RMSE")]
    saved_compat = A.options()["FM.compat"]
    say("effect: planted data, 3 one-hot fields %s whose effects have s.d. %s (w) and %s (V entries); %d training / %d held-out "
        "rows, k=%d, noise s.d. 0.1; fm_posterior, %d sweeps, burn_in %d, fp64" % (
            fields, scales, [round(0.5 * float(np.sqrt(s)), 4) for s in scales], n_tr, n_te, k, sweeps, burn))
    try:
        # FM.compat "reference" keeps the F7 readings (w drawn with the variance as s.d., mu_v from v(f, attr_group[i]));
        # "none" draws as documented without them
        for compat in ("reference", "none"):
            A.options(**{"FM.compat": compat})
            out = {}
            for name, g in (("one group", None), ("groups = fields", grp)):
                tr["features"].pop("attr_group", None)
                if g is not None:
                    tr["features"]["attr_group"] = g
                post = A.fm_posterior(tr, [te], burn_in=burn, normalize=False, control=ctl)
                out[name] = float(np.sqrt(np.mean((post["newdata"][0] - y_te) ** 2)))
            say("  FM.compat=%-9s held-out RMSE of the posterior mean: one group %.5f, groups = fields %.5f (%+.2f %%)" % (
                compat, out["one group"], out["groups = fields"], 100.0 * (out["groups = fields"] - out["one group"]) / out["one group"]))
    finally:
        A.options(**{"FM.enable_v": saved, "FM.compat": saved_compat})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    cost(say, args.sweeps, args.repeats)
    effect(say)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
