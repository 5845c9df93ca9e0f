"""Cost of held-out tracking (fmwr_train_holdout_dev) on the configs[1] workload bench.py builds: 10M Criteo-shaped rows x 39
one-hot fields (999 999 features), k = 32, fp32, one FTRL minibatch epoch (batch 65536), L1+L2 as in bench.py.  The held-out
set is 1M rows of the same synthetic matrix past the training rows (fmwr_data_synth_rows from row 10M), and the tracker records
every 10^6 samples (step_size = 10^6, metric LL).

Times one epoch four ways, alternating within every repeat, each from the same initial model:
  (a) plain      fmwr_train_dev, no tracker
  (b) tracker    fmwr_train_dev with a scores-only trace (no snapshots)
  (c) holdout    fmwr_train_holdout_dev with a scores-only trace and the held-out set
  (d) snapshots  today's workflow: fmwr_train_dev with host snapshots, then per snapshot fmwr_model_set + predict + evaluate on
                 the held-out set (fm.track)
Every time is a host clock around work that ends in a device synchronise.  Reports medians, the per-record cost over (b), and
the host bytes each variant holds for its trace; checks that (c) and (d) give the same held-out curve; prints the card name and
power limit read in the same run.

    python profiles/tools/holdout_track_cost.py [--repeats 3] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--eval-rows", type=int, default=1_000_000)
    ap.add_argument("--step", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    ctx = L.Context(0)
    n, F, k, B = args.rows, 39, 32, 65536
    field = 1_000_000 // F
    p = field * F
    fields = [field] * F
    d = L.Data.synth(ctx, n, fields, None, 0, 1, 0.1, 20240601)
    ev = L.Data.synth_rows(ctx, n, args.eval_rows, fields, None, 0, 1, 0.1, 20240601)
    mcfg = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=1e-3, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
    m = L.Model(ctx, mcfg, p, L.F32)
    sc = L.SolverCfg(solver=L.FTRL, max_iter=n - 1, random_step=1, learn_rate=0.01, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0,
                     gamma=1e-4, min_target=-1.0, max_target=1.0, mode=L.MODE_MINIBATCH, batch_size=B, precision=L.F32,
                     compat=L.COMPAT_REFERENCE, step_size=-1, metric=L.LL, convergence=-1.0)
    st = L.SolverCfg.from_buffer_copy(sc)
    st.step_size = args.step
    nrec = int(np.ceil((sc.max_iter - 0.5) / args.step)) + 2
    d.minibatch_info(B)                                   # the per-batch CSC, built once like bench.py does before timing
    out = {}

    def plain():
        L.train_dev(ctx, m, d, sc)

    def tracker():
        tr = L.TraceBuf(nrec)
        L.train_dev(ctx, m, d, st, tr)
        out["b"] = tr.result()
        return tr.eval_train.nbytes + tr.rec_index.nbytes

    def holdout():
        tr = L.TraceBuf(nrec)
        scores, best = L.train_holdout_dev(ctx, m, d, st, tr, [ev])
        out["c"] = (tr.result(), scores[0], best)
        return tr.eval_train.nbytes + tr.rec_index.nbytes + scores.nbytes

    def snapshots():
        tr = L.TraceBuf(nrec, p, k, snapshots=True)
        L.train_dev(ctx, m, d, st, tr)
        t = tr.result()
        mr = L.Model(ctx, mcfg, p, L.F32)
        test = np.zeros(t["n_rec"])
        for r in range(t["n_rec"]):
            mr.set(t["snap_w0"][r], t["snap_w"][r], t["snap_v"][r])
            L.predict_dev(ctx, mr, ev, L.LINK_LOGISTIC, sc.min_target, sc.max_target)
            test[r] = L.evaluate_dev(ctx, ev, mcfg.task, L.LL)
        mr.close()
        out["d"] = (t, test)
        return sum(a.nbytes for a in (tr.eval_train, tr.rec_index, tr.snap_w0, tr.snap_w, tr.snap_v))

    runs = {"(a) plain": plain, "(b) tracker": tracker, "(c) holdout": holdout, "(d) snapshots": snapshots}
    times = {name: [] for name in runs}
    host = {}
    for rep in range(args.repeats + 1):                  # repeat 0 warms every path up and is not counted
        for name, fn in runs.items():
            m.init_random(0.0, 0.01, 20240603)
            ctx.sync()
            t0 = time.perf_counter()
            host[name] = fn() or 0
            ctx.sync()
            if rep > 0:
                times[name].append((time.perf_counter() - t0) * 1e3)
    tb, (tc, test_c, best_c), (td, test_d) = out["b"], out["c"], out["d"]
    assert np.array_equal(tc["eval_train"], tb["eval_train"]) and np.array_equal(tc["rec_index"], td["rec_index"])
    assert np.array_equal(test_c, test_d), (test_c, test_d)
    n_rec = tc["n_rec"]

    say("card (name, power limit, max SM clock): %s" % card())
    say("workload: configs[1], %d rows x %d one-hot fields (p=%d), k=%d, fp32, FTRL minibatch (batch %d), one epoch of %d samples; "
        "held-out set %d rows (synth_rows from row %d); tracker step %d samples -> %d records, metric LL" % (
            n, F, p, k, B, sc.max_iter, args.eval_rows, n, args.step, n_rec))
    say("median of %d alternating repeats, host clock around work ending in a device synchronise, same initial model each run" % args.repeats)
    med = {name: statistics.median(t) for name, t in times.items()}
    for name, t in times.items():
        say("  %-14s %9.1f ms/epoch  range %.1f .. %.1f ms  host bytes held for the trace: %d (%.1f MB)" % (
            name, med[name], min(t), max(t), host[name], host[name] / 1e6))
    base = med["(b) tracker"]
    say("  per record over (b): tracker itself %.2f ms (b - a), held-out scoring %.2f ms (c - b), snapshot workflow %.2f ms (d - b)" % (
        (med["(b) tracker"] - med["(a) plain"]) / n_rec, (med["(c) holdout"] - base) / n_rec, (med["(d) snapshots"] - base) / n_rec))
    say("  held-out LL per record, (c) == (d) bit for bit: %s; best record %d" % (" ".join("%.6g" % x for x in test_c), best_c))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    m.close(); ev.close(); d.close(); ctx.close()


if __name__ == "__main__":
    main()
