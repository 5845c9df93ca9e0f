"""Cost of the per-feature contributions (fmwr_contrib_dev) against predict (fmwr_predict_dev, FMWR_LINK_NONE) on the same handle.

Two workloads:
  configs[1]  the matrix bench.py builds: 10M rows x 39 one-hot fields of 25641 ids (p = 999999), fp32, k = 32,
              V ~ N(0, 0.01) as bench.py initialises it; predict runs the stream kernel there, contributions the team kernel
  configs[0]  its shape: 100k rows x 10 fields of 1000 ids, values ~ U(0.5, 1.5), fp64, k = 8
Inside every repeat the two calls alternate, each after fmwr_flush_l2 and timed with CUDA events on the engine's stream; the
medians are reported with the rows/s of each, their ratio, the fraction of 6539 GB/s (the measured copy peak, DESIGN section 3)
by the byte model below, and the card name, power limit and max SM clock read in the same run.

Bytes per row of m entries (SURVEY section 8d, parameters of e bytes): predict 4 + m(8 + e(1 + k)) + 4; contributions add 8m
(phi, f64) and 8 (the score, f64).  The efficiency identity (row sums of phi plus w0 against predict) is checked on every
workload before timing.

    python profiles/tools/contrib_cost.py [--repeats 15] [--out FILE]
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

PEAK_GBS = 6539.0


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    return q.stdout.strip()


def workload(ctx, name):
    if name == "configs[1]":
        F, k, prec = 39, 32, L.F32
        field = 1_000_000 // F
        n, fields, value_mode, label_mode = 10_000_000, [field] * F, 0, 1
    else:
        F, k, prec = 10, 8, L.F64
        n, fields, value_mode, label_mode = 100_000, [1000] * F, 1, 2
    d = L.Data.synth(ctx, n, fields, None, value_mode, label_mode, 0.1, 20240601)
    m = L.Model(ctx, L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k), sum(fields), prec)
    m.init_random(0.0, 0.01, 20240603)
    return d, m, n, F, k, prec


def check_identity(ctx, d, m, n, F):
    """every synthetic row holds one id per field, so phi is [n][F]"""
    L.predict_dev(ctx, m, d, L.LINK_NONE)
    pred = L.predict_fetch(ctx, d)
    L.contrib_dev(ctx, m, d)
    phi = L.contrib_fetch(ctx, d)
    assert phi.size == n * F
    sums = m.get()[0] + phi.reshape(n, F).sum(1)
    return float(np.max(np.abs(sums - pred) / np.maximum(1.0, np.abs(pred))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    ctx = L.Context(0)
    say("card (name, power limit, max SM clock): %s" % card())
    say("median of %d repeats; predict (LINK_NONE) and contributions alternate inside each repeat, each after an L2 flush" % args.repeats)
    for name in ("configs[1]", "configs[0]"):
        d, m, n, F, k, prec = workload(ctx, name)
        e = 4 if prec == L.F32 else 8
        err = check_identity(ctx, d, m, n, F)
        runs = {"predict": lambda: L.predict_dev(ctx, m, d, L.LINK_NONE), "contrib": lambda: L.contrib_dev(ctx, m, d)}
        for f in runs.values():                     # warm-up
            f()
        times = {key: [] for key in runs}
        for _ in range(args.repeats):
            for key, f in runs.items():
                ctx.flush_l2()
                ctx.sync()
                ctx.timer_start()
                f()
                times[key].append(ctx.timer_stop_ms())
        b_pred = 4 + F * (8 + e * (1 + k)) + 4
        b_con = b_pred + 8 * F + 8
        say("%s: %d rows x %d entries, k=%d, %s; max |w0 + sum phi - predict| / max(1, |predict|) = %.2e" % (
            name, n, F, k, "fp32" if prec == L.F32 else "fp64", err))
        med = {}
        for key, b in (("predict", b_pred), ("contrib", b_con)):
            t = times[key]
            med[key] = statistics.median(t)
            say("  %-8s %8.3f ms  range %.3f .. %.3f  %6.3f G rows/s  %5d B/row  %.2f of %.0f GB/s" % (
                key, med[key], min(t), max(t), n / med[key] / 1e6, b, n * b / (med[key] * 1e-3) / 1e9 / PEAK_GBS, PEAK_GBS))
        say("  contrib / predict = %.2f" % (med["contrib"] / med["predict"]))
        m.close(); d.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
