"""Cost and value of SGDA (fmwr_train_sgda_dev): adaptive-regularization SGD against exact-mode SGD.

Speed, per training sample, fp32 and fp64, on two workloads:
  * configs[0]: 100k x 10 fields of 1000 ids (10 nnz/row, real values), k = 8, regression (bench.py run_c1's matrix); the
    validation set is the next 20k rows of the same synthetic matrix;
  * a 10^6-row prefix of configs[1]: Criteo-shaped 39 one-hot fields, p = 999 999, k = 32, classification; validation = the next
    10^5 rows.
SGDA takes no lambda step in its first pass (T0 = n - 1 samples with the F5 scan), so it is timed over one pass and over two
passes from the same initial model: the first pass gives its cost without lambda steps, the difference of the two its cost per
sample with one (a training row's step and a validation row's look-ahead and lambda step).  SGD is timed over one pass on the
pipelined exact kernel (the default) and on the CTA-wide one (FMWR_EXACT_PIPE=0).  Every time is a host clock around work that ends
in a device synchronise, after one warm-up of each variant; variants alternate within every repeat; medians and ranges are given.

Quality: seeded planted regression data -- 5 signal fields with a planted FM (k = 4) and 5 noise fields of ids that do not enter
the label, 200 ids each, one id per field per row, N(0, 0.5^2) label noise -- 8 000 training rows, 4 000 validation rows, 8 000
test rows.  After the same number of samples (12 passes), the validation and test RMSE of SGDA from lambda = 0 (one group per
field), SGD with L2 = 0 and SGD over a fixed L2 grid (the same rate for w and V) that runs past the grid's best point.

    python profiles/tools/sgda_cost.py [--repeats 3] [--out FILE]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from fmwr_b200 import _lib as L  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    return q.stdout.strip()


def solver_cfg(prec, iters, lo, hi, lr):
    return L.SolverCfg(solver=L.SGD, max_iter=iters, random_step=1, learn_rate=lr, min_target=lo, max_target=hi, mode=L.MODE_EXACT,
                       precision=prec, compat=L.COMPAT_REFERENCE, step_size=-1)


def speed(ctx, say, name, d, dv, n, p, k, task, grp, G, repeats):
    _, _, _, y = d.get_csr()
    lo, hi = float(y.min()), float(y.max())
    mc = L.ModelCfg(task=task, keep_w0=1, keep_w1=1, k=k, l2_w1=1e-3, l2_v=1e-3)
    T0 = n - 1
    for prec, pname in ((L.F32, "fp32"), (L.F64, "fp64")):
        def run(kind):
            m = L.Model(ctx, mc, p, prec)
            m.init_random(0.0, 0.01, 20240603)
            ctx.sync()
            t0 = time.perf_counter()
            if kind.startswith("sgda"):
                sc = solver_cfg(prec, T0 * (2 if kind == "sgda2" else 1), lo, hi, 0.01)
                sc.attr_group = L.ptr(grp); sc.n_groups = G
                L.train_sgda_dev(ctx, m, d, sc, dv, np.full(G, 1e-3), np.full((G, k), 1e-3), keep=[grp])
            else:
                if kind == "sgd_cta":
                    os.environ["FMWR_EXACT_PIPE"] = "0"
                L.train_dev(ctx, m, d, solver_cfg(prec, T0, lo, hi, 0.01))
                os.environ.pop("FMWR_EXACT_PIPE", None)
            ctx.sync()
            dt = time.perf_counter() - t0
            m.close()
            return dt
        kinds = ("sgd_pipe", "sgd_cta", "sgda1", "sgda2")
        for kd in kinds:
            run(kd)                                                          # warm-up
        times = {kd: [] for kd in kinds}
        for _ in range(repeats):
            for kd in kinds:
                times[kd].append(run(kd))
        per = {kd: [t * 1e6 / T0 for t in times[kd]] for kd in kinds}
        per["sgda_lambda"] = [(b - a) * 1e6 / T0 for a, b in zip(times["sgda1"], times["sgda2"])]
        med = {kd: statistics.median(v) for kd, v in per.items()}
        say("%s %s (us per sample, median [min .. max] of %d):" % (name, pname, repeats))
        for kd, label in (("sgd_pipe", "SGD, pipelined exact kernel"), ("sgd_cta", "SGD, CTA-wide exact kernel"),
                          ("sgda1", "SGDA first pass (no lambda step)"), ("sgda_lambda", "SGDA sample with a lambda step")):
            say("  %-34s %7.3f  [%.3f .. %.3f]" % (label, med[kd], min(per[kd]), max(per[kd])))
        say("  SGDA with a lambda step / CTA-wide SGD = %.2fx, / pipelined SGD = %.2fx"
            % (med["sgda_lambda"] / med["sgd_cta"], med["sgda_lambda"] / med["sgd_pipe"]))


def planted(rng, n, Vt, wt, F=10, ids=200, noise=0.5):
    cols = np.stack([f * ids + rng.integers(0, ids, n) for f in range(F)], 1)
    x = np.ones((n, F), np.float32)
    sig = cols[:, :F // 2]
    S = Vt[sig].sum(1)
    y = wt[sig].sum(1) + 0.5 * ((S * S).sum(1) - (Vt[sig] ** 2).sum((1, 2))) + rng.normal(0, noise, n)
    rowptr = np.arange(n + 1, dtype=np.uint32) * F
    return rowptr, cols.reshape(-1).astype(np.uint32), x.reshape(-1), y.astype(np.float32)


def quality(ctx, say):
    rng = np.random.default_rng(20240605)
    F, ids, k = 10, 200, 4
    p = F * ids
    wt = np.zeros(p); wt[:p // 2] = rng.normal(0, 0.5, p // 2)
    Vt = np.zeros((p, k)); Vt[:p // 2] = rng.normal(0, 0.4, (p // 2, k))
    sets = {}
    for name, n in (("train", 8000), ("valid", 4000), ("test", 8000)):
        rp, c, x, y = planted(rng, n, Vt, wt, F, ids)
        sets[name] = (L.Data.from_csr32(ctx, n, p, rp, c, x, y), y)
    d, y = sets["train"]
    lo, hi = float(y.min()), float(y.max())
    grp = (np.arange(p) // ids).astype(np.int32)
    iters = 12 * 7999
    lr, kf = 0.02, 8
    say("quality: planted FM regression, 5 signal + 5 noise fields x %d ids, k_true = %d, noise sd 0.5; 8000 train / 4000 valid / "
        "8000 test rows; k = %d, lr = %g, fp64, %d samples (12 passes), same initial model" % (ids, k, kf, lr, iters))

    def rmse(m, which):
        dd = sets[which][0]
        L.predict_dev(ctx, m, dd, L.LINK_CLAMP, lo, hi)
        return L.evaluate_dev(ctx, dd, L.REGRESSION, L.RMSE)

    def fit(l2, adaptive):
        m = L.Model(ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=kf, l2_w1=l2, l2_v=l2), p, L.F64)
        r = np.random.default_rng(1)
        m.set(0.0, np.zeros(p), r.normal(0, 0.1, (p, kf)))
        sc = solver_cfg(L.F64, iters, lo, hi, lr)
        lw = lv = None
        if adaptive:
            sc.attr_group = L.ptr(grp); sc.n_groups = F
            lw, lv = np.full(F, l2), np.full((F, kf), l2)
            L.train_sgda_dev(ctx, m, d, sc, sets["valid"][0], lw, lv, keep=[grp])
        else:
            L.train_dev(ctx, m, d, sc)
        out = (rmse(m, "valid"), rmse(m, "test"), lw, lv)
        m.close()
        return out

    va, te, lw, lv = fit(0.0, True)
    say("  %-26s valid RMSE %.4f  test RMSE %.4f" % ("SGDA from lambda = 0", va, te))
    say("    learned lambda_w by field: " + " ".join("%.3g" % v for v in lw))
    say("    learned mean lambda_v by field: " + " ".join("%.3g" % v for v in lv.mean(1)))
    for l2 in (0.0, 1e-3, 1e-2, 3e-2, 1e-1, 3e-1, 1.0, 3.0):
        va, te, _, _ = fit(l2, False)
        say("  %-26s valid RMSE %.4f  test RMSE %.4f" % ("SGD L2 = %g" % l2, va, te))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-speed", action="store_true")
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    ctx = L.Context(0)
    say("card (name, power limit, max SM clock): " + card())
    if not args.skip_speed:
        n0, f0 = 100_000, [1000] * 10
        d0 = L.Data.synth(ctx, n0, f0, None, 1, 2, 0.1, 20240601)
        v0 = L.Data.synth_rows(ctx, n0, 20_000, f0, None, 1, 2, 0.1, 20240601)
        g0 = (np.arange(sum(f0)) // 1000).astype(np.int32)
        speed(ctx, say, "configs[0] 100000 x 10 fields, k=8, regression, groups = fields", d0, v0, n0, sum(f0), 8, L.REGRESSION,
              g0, 10, args.repeats)
        d0.close(); v0.close()
        n1, F = 1_000_000, 39
        f1 = [1_000_000 // F] * F
        d1 = L.Data.synth(ctx, n1, f1, None, 0, 1, 0.1, 20240601)
        v1 = L.Data.synth_rows(ctx, n1, 100_000, f1, None, 0, 1, 0.1, 20240601)
        g1 = (np.arange(sum(f1)) // f1[0]).astype(np.int32)
        speed(ctx, say, "configs[1] prefix 1000000 x 39 fields, k=32, classification, groups = fields", d1, v1, n1, sum(f1), 32,
              L.CLASSIFICATION, g1, F, args.repeats)
        d1.close(); v1.close()
    quality(ctx, say)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
