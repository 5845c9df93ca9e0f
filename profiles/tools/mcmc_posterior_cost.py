"""Cost of the MCMC posterior mean (fmwr_train_posterior_dev) on the configs[3] workload bench.py builds: 20M ratings x 3 one-hot
fields [138493, 26744, 2048] (skew [0, 1, 0]), k = 64, fp32, V block on.

Times S sweeps three ways, alternating within every repeat, each from the same initial model:
  plain      fmwr_train_dev
  post       fmwr_train_posterior_dev, burn_in = 0, no eval set
  post+eval  the same with one eval set of 2M rows (synth_rows from row 20M)
and reports the medians, the overhead over the plain sweeps, the time of one predict of the eval set (what each draw should cost
it), and the card name and power limit read in the same run.  The fused coordinate passes sum their statistics with atomics, so
two runs of one chain differ in the last bits: each variant's largest relative difference from the first plain run's final model
is reported, the plain line giving the run-to-run size of it (tests/test_gpu_mcmc_posterior.py compares the chains bit for bit on
the column-parallel passes, which sum without atomics).

    python profiles/tools/mcmc_posterior_cost.py [--sweeps 10] [--repeats 6] [--out FILE]
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


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    S = args.sweeps
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    ctx = L.Context(0)
    na, n_eval = 20_000_000, 2_000_000
    fields, skew, k = [138493, 26744, 2048], [0, 1, 0], 64
    pa = sum(fields)
    da = L.Data.synth(ctx, na, fields, skew, 0, 3, 0.3, 20240601)
    ev = L.Data.synth_rows(ctx, na, n_eval, fields, skew, 0, 0, 0.3, 20240601)
    m = L.Model(ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=k), pa, L.F32)
    sc = L.SolverCfg(solver=L.MCMC, max_iter=S, random_step=1, min_target=0.5, max_target=5.0, mode=L.MODE_EXACT, precision=L.F32,
                     compat=L.COMPAT_REFERENCE, enable_v=1, step_size=-1, seed=5)
    runs = {
        "plain": lambda: L.train_dev(ctx, m, da, sc),
        "post": lambda: L.train_posterior_dev(ctx, m, da, sc, 0),
        "post+eval": lambda: L.train_posterior_dev(ctx, m, da, sc, 0, [ev]),
    }

    def timed(name):
        m.init_random(0.0, 0.01, 20240603)
        ctx.sync()
        ctx.timer_start()
        runs[name]()
        ms = ctx.timer_stop_ms()
        return ms, m.get()

    def rel(a, b):
        return max(abs(a[0] - b[0]) / max(1.0, abs(b[0])), float(np.max(np.abs(a[1] - b[1]) / np.maximum(1.0, np.abs(b[1])))),
                   float(np.max(np.abs(a[2] - b[2]) / np.maximum(1.0, np.abs(b[2])))))

    times = {name: [] for name in runs}
    diff = {name: 0.0 for name in runs}
    ref = None
    for rep in range(args.repeats + 1):                  # repeat 0 warms every path up and is not counted
        for name in runs:
            ms, model = timed(name)
            assert all(np.all(np.isfinite(a)) for a in model[1:]) and np.isfinite(model[0])
            if ref is None:
                ref = model
            else:
                diff[name] = max(diff[name], rel(model, ref))
            if rep > 0:
                times[name].append(ms)
    # one predict of the eval set (raw scores), the forward each averaged draw adds per eval set
    for _ in range(3):
        L.predict_dev(ctx, m, ev)
    ctx.sync()
    pred = []
    for _ in range(args.repeats):
        ctx.timer_start()
        L.predict_dev(ctx, m, ev)
        pred.append(ctx.timer_stop_ms())
    mean_all = L.predict_fetch(ctx, da)                  # the last post+eval run's posterior mean on the training rows
    assert np.all(np.isfinite(mean_all))

    say("card (name, power limit, max SM clock): %s" % card())
    say("workload: configs[3], %d ratings x 3 one-hot fields %s skew %s, k=%d, fp32, enable_v=1; %d MCMC sweeps per run, burn_in 0 "
        "(%d averaged draws); eval set %d rows (synth_rows from row %d)" % (na, fields, skew, k, S, S, n_eval, na))
    say("median of %d alternating repeats, each from the same initial model and seed" % args.repeats)
    base = statistics.median(times["plain"])
    for name in runs:
        t = times[name]
        med = statistics.median(t)
        say("  %-10s %9.2f ms  (%7.2f ms/sweep)  range %.2f .. %.2f ms  overhead %+6.2f %%  final model vs first plain run: max rel diff %.2e" % (
            name, med, med / S, min(t), max(t), 100.0 * (med - base) / base, diff[name]))
    pm = statistics.median(pred)
    extra = statistics.median(times["post+eval"]) - statistics.median(times["post"])
    say("  predict of the eval set: %.3f ms (median of %d); eval-set cost per draw: %.3f ms (= %.2f predicts)" % (
        pm, len(pred), extra / S, extra / S / pm))
    say("  training-row accumulation by bytes: %d B/row/draw x %d rows x %d draws = %.2f GB, plus one forward of the training rows "
        "for the last draw" % (20, na, S, 20.0 * na * S / 1e9))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    m.close(); ev.close(); da.close(); ctx.close()


if __name__ == "__main__":
    main()
