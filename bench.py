#!/usr/bin/env python
"""bench.py -- headline benchmark of the FM hot path (BASELINE.json configs[1]).

A "step" is one FTRL-Proximal training epoch (minibatch throughput mode) over the Criteo-shaped
synthetic matrix (10M rows x 39 nnz, 1M features, k=32, binary logloss, L1+L2); `value` is samples/s with
the data resident in HBM.  The same run also times predict.FM over the same rows (`predict`), the
end-to-end call through the C ABI with HOST buffers (`e2e`), the reference's CPU path on a bounded sample
(`cpu_baseline`) and reports the dominant kernel's achieved HBM bandwidth (`roofline`).

Roofline accounting (DESIGN.md section 6): `roofline.frac` of the update kernel is COMPULSORY bytes per launch -- counted from
the real per-batch structure (segments x (record + offset + theta/state rows and w scalars, read and write) + entries x 8 B)
-- over the CUDA-event launch time over the measured HBM peak.  SURVEY 8(d)'s per-sample model (every gather at full width,
no cache credit) is kept as a labelled second figure without a fraction: a 65 536-row batch touches a coordinate ~2.6 times
and updates it once, so that model overstates the bytes this kernel has to move.  Kernels whose committed ncu DRAM traffic is
below half the per-sample model (predict, K1: V is half L2-resident) report their fraction against the MEASURED traffic.

    python bench.py --gpus N --steps K --warmup W            # engine arm
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU implementation
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also save what the timed path computed, DIR/<name>.npy

For N > 1 launch with torchrun (one rank per GPU); see DESIGN.md section "Multi-GPU".
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# one metric string for both arms (the reference arm runs the reference's batch = 1 CPU loop; `predict` only on the engine arm)
METRIC = "samples/sec per epoch (fm.train FTRL.solver, L1+L2 binary logloss, configs[1]); predict rows/sec in `predict`"

ALG_BYTES = {
    # SURVEY.md section 8(d): fp32 params/state, u32 ids, f32 x, every gather at full width
    "predict": lambda m, k: 8 + m * (12 + 4 * k),
    "sgd": lambda m, k: 8 + m * (8 + 2 * (4 + 4 * k)),
    "ftrl": lambda m, k: 8 + m * (8 + 6 * (4 + 4 * k)),
    "tdap": lambda m, k: 8 + m * (8 + 10 * (4 + 4 * k)),
}


N_ARRAYS = {"sgd": 1, "sgd_l1": 2, "ftrl": 3, "tdap": 5}      # theta + optimizer-state arrays a coordinate step reads and writes


def k2_compulsory_bytes(solver, info, kp):
    """bytes the coordinate-update kernel MUST move per epoch, from the real per-batch CSC: per (batch, feature) segment the
    16-byte record, the 4-byte entry offset, the theta/state rows (kp x 4 B each) and the w scalars, read and written once;
    per entry 8 bytes (row id + value).  The S-cache / multiplier gathers stay in L2 (8 MB per batch) and are not counted."""
    na = N_ARRAYS[solver]
    return info["n_segments"] * (20 + 2 * na * 4 * kp + 2 * na * 4) + info["n_entries"] * 8


def k1_compulsory_bytes(info, n, m, kp):
    """forward of the batches: the CSR rows once (8 B per entry + 4 B row offset + 4 B label) and, per batch, each touched
    feature's factor row and weight once (a perfect cache inside a batch); the S-cache writes stay in L2"""
    return n * (8 * m + 8) + info["n_segments"] * (4 * kp + 4)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(nm)
        if sm:
            top = sorted(sm)[len(sm) // 2:]          # upper half ~ samples under load
            out.update(sm_mhz=float(np.median(top)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def ncu_traffic(kernel, units_per_launch):
    """DRAM bytes per launch from the committed ncu capture (profiles/traffic_r02.json), scaled to this run's launch size"""
    for name in ("traffic_r02.json", "traffic_r01.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))[kernel]
            return int(t["dram_bytes"] * units_per_launch / t["rows_per_launch"])
        except Exception:
            continue
    return None


def parse_profile(txt):
    agg = {}
    for line in txt.strip().split("\n"):
        if not line:
            continue
        tag, n, ms = line.split("\t")
        name = tag.strip("()").split("<")[0]
        a = agg.setdefault(name, [0, 0.0])
        a[0] += int(n); a[1] += float(ms)
    return agg


DUMP_LIMIT = 64 << 20


def fixed_sample(n, m, seed):
    """sorted indices of a seeded sample of m out of n (all n when m >= n): the same for every run with the same n"""
    if m >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, m, replace=False))


def write_outputs(path, arrays):
    """--dump-outputs: each array as <path>/<name>.npy in float64, so two builds can be compared output for output"""
    arrays = {name: np.asarray(a, np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, "outputs to dump take %d bytes, over the %d-byte limit" % (total, DUMP_LIMIT)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------ engine arm
def update_kernel_of(prof):
    """the coordinate-update kernel that ran (dense TMA variant or the gather kernel): the one with the larger total"""
    cands = [(v[1], name) for name, v in prof.items() if name.startswith("mb_update")]
    return max(cands)[1] if cands else None


def forward_kernel_of(prof):
    cands = [(v[1], name) for name, v in prof.items() if "forward" in name]
    return max(cands)[1] if cands else None


def profiled(L, lib, ctx, fn, steps):
    """run fn() `steps` times with a CUDA-event pair around every kernel launch (events pre-created by one untimed pass)"""
    buf = C.create_string_buffer(1 << 16)
    L.check(lib.fmwr_profile_enable(ctx.h, 1))
    fn()
    L.check(lib.fmwr_profile_enable(ctx.h, 1))          # returns the events to the pool, clears the records
    ctx.timer_start()
    for _ in range(steps):
        fn()
    ms = ctx.timer_stop_ms()
    L.check(lib.fmwr_profile_read(ctx.h, buf, C.c_int64(len(buf))))
    prof = parse_profile(buf.value.decode())
    L.check(lib.fmwr_profile_enable(ctx.h, 0))
    return prof, ms


def mb_solver_cfg(L, solver, max_iter, B, mode=None, precision=None):
    return L.SolverCfg(solver=solver, max_iter=max_iter, random_step=1, learn_rate=0.01, alpha_w=0.1, alpha_v=0.1, beta_w=1.0, beta_v=1.0,
                       gamma=1e-4, min_target=-1.0, max_target=1.0, mode=L.MODE_MINIBATCH if mode is None else mode, batch_size=B,
                       precision=L.F32 if precision is None else precision, compat=L.COMPAT_REFERENCE, step_size=-1)


def run_engine(args):
    from fmwr_b200 import _lib as L
    rank, world, local = dist_env()
    if world > 1:
        return run_engine_multi(args, rank, world, local)
    lib = L.lib()
    ctx = L.Context(local)
    peak, peak_src = measured_peak()
    n, F, k, B = args.rows, 39, args.k, args.batch
    kp = (k + 3) // 4 * 4
    field = args.features // F
    p = field * F
    m_nnz = F

    t0 = time.time()
    data = L.Data.synth(ctx, n, [field] * F, None, 0, 1, 0.1, 20240601)
    mcfg = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=1e-3, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
    model = L.Model(ctx, mcfg, p, L.F32)
    model.init_random(0.0, 0.01, 20240603)
    ctx.sync()
    t_gen = time.time() - t0

    epoch = n - 1                       # one reference epoch == n-1 sample updates (SURVEY F4/F5)
    sc = mb_solver_cfg(L, L.FTRL, epoch, B)
    # ---- the per-batch CSC the update kernel works on: built once per (data, batch size), timed on its own ----------
    ctx.sync(); ctx.timer_start()
    info = data.minibatch_info(B)
    prep_cold_ms = ctx.timer_stop_ms()              # first build of the process: includes cudaMalloc of ~12 GB of scratch and outputs
    data.minibatch_info(2 * B)                      # drop it (another batch size) ...
    ctx.sync(); ctx.timer_start()
    info = data.minibatch_info(B)                   # ... and build it again with the allocator warm: what a second fm.train pays
    prep_ms = ctx.timer_stop_ms()
    # ---- FTRL epoch, data resident ------------------------------------------------------------------
    for _ in range(args.warmup):
        L.train_dev(ctx, model, data, sc)
    ctx.sync()
    clocks = ClockSampler(local)
    clocks.start()
    # timed region A: K steps, no per-kernel events -> `value`
    l0 = ctx.launches()
    ctx.timer_start()
    for _ in range(args.steps):
        L.train_dev(ctx, model, data, sc)
    ms_train = ctx.timer_stop_ms()
    l1 = ctx.launches()
    train_sps = epoch * args.steps / (ms_train * 1e-3)
    dump = {}
    if args.dump_outputs:
        # the model the last timed step returns (w0, w, V); w and V as fixed samples of their rows (16 MB of V at any k)
        w0_t, w_t, v_t = model.get()
        w_rows = fixed_sample(p, 1 << 20, 1)
        v_rows = fixed_sample(p, (16 << 20) // (8 * max(k, 1)), 2)
        dump.update(w0=np.array([w0_t]), w_sample=w_t[w_rows], w_sample_rows=w_rows, v_sample=v_t[v_rows], v_sample_rows=v_rows)
        del v_t
    # timed region B: the same K steps with a CUDA-event pair around every kernel launch -> per-kernel durations for the roofline
    prof_train, ms_train_prof = profiled(L, lib, ctx, lambda: L.train_dev(ctx, model, data, sc), args.steps)

    # ---- predict.FM, data resident -------------------------------------------------------------------
    for _ in range(args.warmup):
        L.predict_dev(ctx, model, data, L.LINK_LOGISTIC)
    ctx.timer_start()
    for _ in range(args.steps):
        L.predict_dev(ctx, model, data, L.LINK_LOGISTIC)
    ms_pred = ctx.timer_stop_ms()
    if args.dump_outputs:
        # predict.FM's probabilities from its last timed step, a fixed sample of the rows
        pred_rows = fixed_sample(n, 1 << 20, 3)
        dump.update(predict_sample=L.predict_fetch(ctx, data)[pred_rows], predict_sample_rows=pred_rows)
        write_outputs(args.dump_outputs, dump)
    prof_pred, _ = profiled(L, lib, ctx, lambda: L.predict_dev(ctx, model, data, L.LINK_LOGISTIC), args.steps)
    clk = clocks.stop()
    pred_rps = n * args.steps / (ms_pred * 1e-3)

    # ---- roofline of the dominant kernel (the coordinate-update kernel K2) ---------------------------------
    b_fwd = ALG_BYTES["predict"](m_nnz, k)
    b_ftrl = ALG_BYTES["ftrl"](m_nnz, k)
    nb = max(1, info["n_batches"])
    k2_bytes = k2_compulsory_bytes("ftrl", info, kp)           # per epoch
    k1_bytes = k1_compulsory_bytes(info, n, m_nnz, kp)
    roof = None
    kn = update_kernel_of(prof_train)
    if kn and prof_train[kn][1] > 0:
        launches, ms = prof_train[kn]
        per_launch = k2_bytes * args.steps / launches
        ach = per_launch / (ms / launches * 1e-3) / 1e9
        traffic = ncu_traffic(kn, min(B, n)) if (p, k) == (999999, 32) else None
        roof = {"kernel": kn, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                "traffic": traffic,
                "alg_bytes_per_launch": int(per_launch),
                "model": "compulsory bytes of one batch from its real structure: %d segments x (16 B record + 4 B offset + theta/z/n rows and w scalars read+written) "
                         "+ %d entries x 8 B, per epoch / %d batches; S-cache gathers are L2-resident and not counted" % (info["n_segments"], info["n_entries"], nb),
                "frac_of_traffic": round(traffic / (ms / launches * 1e-3) / 1e9 / peak, 4) if traffic else None,
                "survey_model_bytes_per_launch": int((b_ftrl - b_fwd) * epoch * args.steps / launches),
                "survey_model_note": "SURVEY 8(d) per-sample model (every gather at full width, no cache credit): more than this kernel has to move, "
                                     "because a batch touches a coordinate %.2f times and updates it once -- reported without a fraction" % (info["n_entries"] / max(1, info["n_segments"])),
                "peak_source": peak_src, "launches": launches, "avg_launch_ms": round(ms / launches, 5),
                "share_of_step": round(ms / ms_train_prof, 4), "ms_per_step_with_events": round(ms_train_prof / args.steps, 3)}
    fwd_roof = None
    fk = forward_kernel_of(prof_pred)
    if fk and prof_pred[fk][1] > 0:
        launches, ms = prof_pred[fk]
        traffic = ncu_traffic(fk, n) if (p, k) == (999999, 32) else None
        t_s = ms / launches * 1e-3
        # guard of SURVEY 8(d): measured DRAM bytes below half the per-row model (V is half L2-resident) -> fraction against the measured bytes
        # the per-row model counts every factor-row gather as DRAM traffic; with V (128 MB) about half L2-resident the kernel moves
        # less than half of it, so the fraction is taken against the MEASURED bytes (null until a capture of this kernel is committed)
        use_traffic = traffic is not None and traffic < 0.5 * n * b_fwd
        basis = traffic if use_traffic else (n * b_fwd if traffic is not None else None)
        fwd_roof = {"kernel": fk, "bound": "hbm", "achieved": round(basis / t_s / 1e9, 1) if basis else None, "peak": peak, "unit": "GB/s",
                    "frac": round(basis / t_s / 1e9 / peak, 4) if basis else None, "traffic": traffic,
                    "basis": "measured DRAM bytes (ncu): below half the per-row model because V is half L2-resident" if use_traffic else "SURVEY 8(d) per-row model",
                    "survey_model_gbs": round(n * b_fwd / t_s / 1e9, 1), "alg_bytes_per_row": b_fwd, "avg_launch_ms": round(ms / launches, 4),
                    "gather_ceiling_ms": GATHER_CEILING_MS.get((p, k)),
                    "gather_ceiling_note": "profiles/r02_gather_bench.md: a kernel that does nothing but this launch's 390M random 128-byte row gathers from a 128 MB table "
                                           "(8 loads in flight per lane, 32 warps/SM) takes this long on the same B200"}
    kernels = {name: {"launches": v[0], "ms": round(v[1], 3)} for name, v in prof_train.items()}
    step_bytes = k1_bytes + k2_bytes
    step_gbs = step_bytes / (ms_train / args.steps * 1e-3) / 1e9

    # ---- the other solvers of the north_star (secondary lines) ------------------------------------------------------
    solvers = None
    if not args.no_solvers:
        solvers = run_other_solvers(L, lib, ctx, data, args, peak, n, F, p, k, B, info, kp)
        if not args.no_sweep:
            solvers["batch_sweep"] = run_batch_sweep(L, ctx, data, args, n, F, field, p, k)
        solvers["c1"] = run_c1(L, ctx, args)

    # ---- end to end through the C ABI with host buffers -------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(L, lib, ctx, data, mcfg, mb_solver_cfg(L, L.FTRL, epoch, B), n, p, k, args)

    # ---- CPU baseline (the reference's own C++ where available, else the C port) on a bounded sample ----------------
    cpu = None
    if not args.no_cpu:
        cpu = cpu_baseline_ftrl(L, data, n, p, k, F, seconds=args.cpu_seconds)

    out = {
        "metric": METRIC,
        "value": round(train_sps, 1), "unit": "samples/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_train / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: Criteo-shaped %d rows x %d nnz, %d features, k=%d, FTRL L1+L2 binary logloss" % (n, F, p, k),
                   "rows": n, "nnz_per_row": F, "features": p, "k": k, "batch_size": B, "mode": "minibatch",
                   "l2_flush": "inputs (%.1f GB CSR + %.1f GB params/state) larger than L2" % (n * F * 8 / 1e9, p * (k + 1) * 12 / 1e9),
                   "epoch": "n-1 sample updates (reference scan skips row 0)",
                   "optimizer_steps_per_epoch": info["n_batches"],
                   "quality": "train LL / AUC after one epoch for this and other batch sizes, next to the batch = 1 run: solvers.batch_sweep"},
        "roofline": roof,
        "step_roofline": {"compulsory_bytes_per_step": int(step_bytes), "achieved": round(step_gbs, 1), "unit": "GB/s", "frac": round(step_gbs / peak, 4),
                          "model": "forward (CSR once + each touched factor row once per batch) + update (roofline.model)",
                          "survey_model_bytes_per_sample": b_ftrl},
        "prep_ms": round(prep_ms, 2), "prep_cold_ms": round(prep_cold_ms, 2),
        "prep_note": "per-batch CSC build (hand-written radix sort + segment emit), once per (data, batch size): not inside `value`, inside `e2e`; "
                     "R's default run is 2 epochs (R/fm_train.R:92)",
        "kernels": kernels,
        "predict": {"value": round(pred_rps, 1), "unit": "rows/s", "ms_per_step": round(ms_pred / args.steps, 3),
                    "roofline": fwd_roof},
        "solvers": solvers,
        "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": int(l1 - l0),
        "clocks": clk, "setup_s": round(t_gen, 2),
    }
    print(json.dumps(out), flush=True)
    data.close(); model.close(); ctx.close()


# measured by profiles/tools/gather_bench.cu on this pool's B200 (profiles/r02_gather_bench.md), keyed by (features, k)
GATHER_CEILING_MS = {(999999, 32): 3.85}


def run_other_solvers(L, lib, ctx, data, args, peak, n, F, p, k, B, info, kp):
    """the north_star's other training paths, same timing rules (3 warm-ups, CUDA events, data resident): SGD and TDAP
    minibatch epochs on the configs[1] matrix already on the device; one ALS sweep on configs[2] and one MCMC sweep on
    configs[3] (MovieLens-shaped 20M ratings, 3 one-hot fields).  Minibatch fractions are against the compulsory bytes of the
    epoch (forward + update, see k1_/k2_compulsory_bytes); SURVEY 8(d)'s per-sample model is given without a fraction."""
    out = {}
    steps = args.steps

    def timed(fn):
        for _ in range(3):
            fn()
        ctx.sync(); ctx.timer_start()
        for _ in range(steps):
            fn()
        return ctx.timer_stop_ms() / steps

    for name, solver in (("sgd", L.SGD), ("tdap", L.TDAP)):
        mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=0.0 if name == "sgd" else 1e-3, l2_w1=1e-3,
                        l1_v=0.0, l2_v=1e-3)
        m = L.Model(ctx, mc, p, L.F32)
        m.init_random(0.0, 0.01, 20240603)
        sc = mb_solver_cfg(L, solver, n - 1, B)
        ms = timed(lambda: L.train_dev(ctx, m, data, sc))
        prof, ms_prof = profiled(L, lib, ctx, lambda: L.train_dev(ctx, m, data, sc), 1)
        b = ALG_BYTES[name](F, k)
        sps = (n - 1) / (ms * 1e-3)
        comp = k1_compulsory_bytes(info, n, F, kp) + k2_compulsory_bytes(name, info, kp)
        kn = update_kernel_of(prof)
        k2 = None
        if kn:
            launches, kms = prof[kn]
            per_launch = k2_compulsory_bytes(name, info, kp) / launches
            k2 = {"kernel": kn, "avg_launch_ms": round(kms / launches, 5), "alg_bytes_per_launch": int(per_launch),
                  "frac": round(per_launch / (kms / launches * 1e-3) / 1e9 / peak, 4), "traffic": ncu_traffic(kn + "_" + name, min(B, n)) if (p, k) == (999999, 32) else None}
        out[name] = {"workload": "configs[1] matrix, %s minibatch epoch (batch %d)" % (name.upper(), B), "value": round(sps, 1), "unit": "samples/s",
                     "ms_per_step": round(ms, 3), "compulsory_bytes_per_step": int(comp), "achieved_gbs": round(comp / (ms * 1e-3) / 1e9, 1),
                     "frac": round(comp / (ms * 1e-3) / 1e9 / peak, 4), "update_kernel": k2, "survey_model_bytes_per_sample": b,
                     "kernels": {kk: {"launches": v[0], "ms": round(v[1], 3)} for kk, v in prof.items()}}
        m.close()
    # exact mode (batch = 1, the reference's own sample order and arithmetic): one CTA -- every sample reads w0 written by the
    # previous one; SGD and FTRL run several samples in flight behind a column-hazard tracker (exact_pipe_kernel), TDAP the CTA-wide
    # kernel -- so it is reported in samples/s on a bounded sample of the same matrix, next to the reference's single-thread rate in
    # cpu_baseline; no HBM fraction (one SM, instruction-bound).  `cta_wide_us_per_sample` is the same run with FMWR_EXACT_PIPE=0.
    it = int(min(n - 1, 200_000))
    ex = {}
    for name, solver in (("sgd", L.SGD), ("ftrl", L.FTRL), ("tdap", L.TDAP)):
        mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=1e-3, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
        m = L.Model(ctx, mc, p, L.F32)
        m.init_random(0.0, 0.01, 20240603)
        sc = mb_solver_cfg(L, solver, it, 1, mode=L.MODE_EXACT)
        L.train_dev(ctx, m, data, sc)
        ctx.sync(); ctx.timer_start()
        L.train_dev(ctx, m, data, sc)
        ms = ctx.timer_stop_ms()
        ex[name] = {"value": round(it / (ms * 1e-3), 1), "unit": "samples/s", "us_per_sample": round(ms * 1e3 / it, 3)}
        if solver != L.TDAP:
            os.environ["FMWR_EXACT_PIPE"] = "0"
            L.train_dev(ctx, m, data, sc)
            ctx.sync(); ctx.timer_start()
            L.train_dev(ctx, m, data, sc)
            ex[name]["cta_wide_us_per_sample"] = round(ctx.timer_stop_ms() * 1e3 / it, 3)
            del os.environ["FMWR_EXACT_PIPE"]
        m.close()
    out["exact"] = {"workload": "configs[1] matrix, batch=1 reference-order updates, first %d samples, fp32" % it, **ex}
    if args.rows < 1_000_000:
        return out                                  # reduced smoke runs: skip the 20M-rating sweeps
    na = 20_000_000
    fields = [138493, 26744, 2048]
    pa, Na = sum(fields), 3 * na
    da = L.Data.synth(ctx, na, fields, [0, 1, 0], 0, 3, 0.3, 20240601)
    for name, solver, ka in (("als", L.ALS, 32), ("mcmc", L.MCMC, 64)):
        mc = L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=ka)
        m = L.Model(ctx, mc, pa, L.F32)
        m.init_random(0.0, 0.01, 20240603)
        sc = L.SolverCfg(solver=solver, max_iter=1, random_step=1, min_target=0.5, max_target=5.0, mode=L.MODE_EXACT, precision=L.F32,
                         compat=L.COMPAT_REFERENCE, enable_v=1, step_size=-1, seed=5)
        ms = timed(lambda: L.train_dev(ctx, m, da, sc))
        bfwd = 8 + 3 * (12 + 4 * ka)
        sweep_bytes = na * bfwd + 16 * na + 16 * Na + ka * (32 * Na + 4 * na + 8 * pa) + (8 * na if name == "mcmc" else 0)
        out[name] = {"workload": "configs[%d]: %d ratings x 3 one-hot fields (138493 / 26744 skewed / 2048), k=%d, one %s sweep (w and V blocks)" % (
                         2 if name == "als" else 3, na, ka, name.upper()),
                     "value": round(na / (ms * 1e-3), 1), "unit": "ratings/s", "ms_per_step": round(ms, 3), "alg_bytes_per_sweep": sweep_bytes,
                     "achieved_gbs": round(sweep_bytes / (ms * 1e-3) / 1e9, 1), "frac": round(sweep_bytes / (ms * 1e-3) / 1e9 / peak, 4)}
        m.close()
    da.close()
    return out


def quality(L, ctx, model, data):
    """train-set LL (the reference's sum form, src/core/Evaluation.h:80-89, divided by n here) and AUC of the model"""
    L.predict_dev(ctx, model, data, L.LINK_LOGISTIC)
    nrow = data.shape()[0]
    ll = L.evaluate_dev(ctx, data, L.CLASSIFICATION, L.LL)
    auc = L.evaluate_dev(ctx, data, L.CLASSIFICATION, L.AUC)
    return round(ll / nrow, 6), round(auc, 5)


def run_batch_sweep(L, ctx, data, args, n, F, field, p, k):
    """ties the throughput numbers to model quality: for batch sizes 4096 / 16384 / 65536 the epoch rate on the full matrix
    and the train LL / AUC after ONE epoch over a 10^6-row prefix (same ids per field, so the same touches per coordinate
    per batch as the full matrix), next to the batch = 1 (reference order and arithmetic) epoch over the same prefix"""
    n_pre = int(min(n, args.sweep_rows))
    pre = L.Data.synth(ctx, n_pre, [field] * F, None, 0, 1, 0.1, 20240601)      # rows 0 .. n_pre-1 of the same matrix (hash keyed by row)
    mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=1e-3, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
    out = {"workload": "FTRL L1+L2, one epoch; quality on the first %d rows of the configs[1] matrix (p=%d, k=%d), rate on all %d rows" % (n_pre, p, k, n),
           "ll": "mean train log-loss as the reference sums it (Evaluation.h:80-89) / rows"}
    m = L.Model(ctx, mc, p, L.F32)
    m.init_random(0.0, 0.01, 20240603)
    out["init"] = dict(zip(("ll", "auc"), quality(L, ctx, m, pre)))
    sc = mb_solver_cfg(L, L.FTRL, n_pre - 1, 1, mode=L.MODE_EXACT)
    ctx.sync(); ctx.timer_start()
    L.train_dev(ctx, m, pre, sc)
    ms = ctx.timer_stop_ms()
    ll, auc = quality(L, ctx, m, pre)
    out["exact_batch1"] = {"ll": ll, "auc": auc, "samples_per_s": round((n_pre - 1) / (ms * 1e-3), 1), "optimizer_steps": n_pre - 1}
    m.close()
    for B in (4096, 16384, 65536):
        m = L.Model(ctx, mc, p, L.F32)
        m.init_random(0.0, 0.01, 20240603)
        L.train_dev(ctx, m, pre, mb_solver_cfg(L, L.FTRL, n_pre - 1, B))
        ll, auc = quality(L, ctx, m, pre)
        m.close()
        # rate on the full matrix (its per-batch CSC is rebuilt for this batch size: prep_ms)
        ctx.sync(); ctx.timer_start()
        data.minibatch_info(B)
        prep = ctx.timer_stop_ms()
        mf = L.Model(ctx, mc, p, L.F32)
        mf.init_random(0.0, 0.01, 20240603)
        scf = mb_solver_cfg(L, L.FTRL, n - 1, B)
        L.train_dev(ctx, mf, data, scf)
        ctx.sync(); ctx.timer_start()
        for _ in range(2):
            L.train_dev(ctx, mf, data, scf)
        msf = ctx.timer_stop_ms() / 2
        mf.close()
        out["batch_%d" % B] = {"ll": ll, "auc": auc, "optimizer_steps": -(-(n_pre - 1) // B), "samples_per_s": round((n - 1) / (msf * 1e-3), 1),
                               "ms_per_epoch": round(msf, 3), "prep_ms": round(prep, 2)}
    pre.close()
    data.minibatch_info(args.batch)             # leave the headline batch size cached for the callers that follow
    return out


def run_c1(L, ctx, args):
    """BASELINE configs[0]: fm.train SGD.solver, k=8, L2, 100k x 10k regression, 10 nnz/row -- the case the reference runs on a CPU.
    Exact mode (the reference's order and arithmetic, one persistent CTA), the throughput mode, and the reference's own C++ on
    this box's host, one epoch each.  Says plainly which side wins in exact mode."""
    n, fields, k = 100_000, [1000] * 10, 8
    p = sum(fields)
    d = L.Data.synth(ctx, n, fields, None, 1, 2, 0.1, 20240601)
    mc = L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=0.0, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
    rowptr, col, val, y = d.get_csr()
    lo, hi = float(y.min()), float(y.max())
    out = {"workload": "configs[0]: SGD L2, k=8, %d x %d regression, 10 nnz/row, one epoch (n-1 updates)" % (n, p)}

    def run(mode, prec, B, reps):
        m = L.Model(ctx, mc, p, prec)
        m.init_random(0.0, 0.01, 20240603)
        sc = L.SolverCfg(solver=L.SGD, max_iter=n - 1, random_step=1, learn_rate=0.01, min_target=lo, max_target=hi, mode=mode, batch_size=B,
                         precision=prec, compat=L.COMPAT_REFERENCE, step_size=-1)
        L.train_dev(ctx, m, d, sc)
        ctx.sync(); ctx.timer_start()
        for _ in range(reps):
            L.train_dev(ctx, m, d, sc)
        ms = ctx.timer_stop_ms() / reps
        m.close()
        return {"value": round((n - 1) / (ms * 1e-3), 1), "unit": "samples/s", "ms_per_epoch": round(ms, 3)}

    out["exact_f32"] = run(L.MODE_EXACT, L.F32, 1, 2)
    out["exact_f64"] = run(L.MODE_EXACT, L.F64, 1, 2)
    out["minibatch_f32_b4096"] = run(L.MODE_MINIBATCH, L.F32, 4096, 5)
    if not args.no_cpu:
        O, orc, kind = oracle_for_baseline()
        rng = np.random.default_rng(20240603)
        w = np.zeros(p); v = rng.normal(0, 0.01, (p, k))
        cfg = O.make_cfg(solver=O.SGD, task=O.REGRESSION, k=k, max_iter=n - 1, l2_w=1e-3, l2_v=1e-3, learn_rate=0.01, nthreads=1,
                         min_target=lo, max_target=hi)
        orc.train(cfg, n, p, rowptr, col, val, y, 0.0, w.copy(), v.copy())
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            orc.train(cfg, n, p, rowptr, col, val, y, 0.0, w.copy(), v.copy())
        dt = (time.perf_counter() - t0) / reps
        out["cpu_reference"] = {"value": round((n - 1) / dt, 1), "unit": "samples/s", "cores": 1, "kind": kind, "ms_per_epoch": round(dt * 1e3, 3)}
        g, c = out["exact_f32"]["value"], out["cpu_reference"]["value"]
        out["exact_mode_verdict"] = ("the reference's single-thread CPU loop is %.1fx FASTER than the GPU exact mode on this 4 MB problem (it fits the CPU's cache; "
                                     "the GPU path is one CTA whose samples queue behind the hazard tracker and the w0 chain)" % (c / g)) if c > g else "GPU exact mode is %.1fx the reference CPU" % (g / c)
    d.close()
    return out


def run_e2e(L, lib, ctx, data, mcfg, sc, n, p, k, args):
    """fmwr_train one-shot: host fm.matrix lists in, host (w0, w, V) out, every step"""
    rowptr, col, val, y = data.get_csr()
    row_size = np.diff(rowptr.astype(np.int64)).astype(np.int32)
    col_i = col.view(np.int32)
    val64 = val.astype(np.float64)
    y64 = y.astype(np.float64)
    del rowptr, val
    w0 = C.c_double(0.0)
    w = np.zeros(p)
    rng = np.random.default_rng(20240603)
    v = rng.normal(0.0, 0.01, (p, k))
    pinned = []
    for a in (row_size, col_i, val64, y64, w, v):
        if lib.fmwr_host_pin(L.ptr(a), C.c_int64(a.nbytes)) == 0:
            pinned.append(a)
    # the library narrows the f64 values to f32 on the host (several threads, pinned staging) before they cross PCIe: 4 B per value
    host_narrow = os.environ.get("FMWR_HOST_NARROW", "1") != "0"
    val_bytes = val64.nbytes // 2 if host_narrow else val64.nbytes
    h2d = row_size.nbytes + col_i.nbytes + val_bytes + y64.nbytes + w.nbytes + v.nbytes + 8
    d2h = w.nbytes + v.nbytes + 8
    steps = args.steps

    def one():
        L.check(lib.fmwr_train(C.byref(mcfg), C.byref(sc), C.c_int64(n), C.c_int64(p), C.c_int64(col_i.size), L.ptr(row_size),
                               L.ptr(col_i), L.ptr(val64), L.ptr(y64), C.byref(w0), L.ptr(w), L.ptr(v), None))
    one()                                   # warm-up (creates the default context)
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    # predict one-shot as well
    out = np.zeros(n)
    lib.fmwr_host_pin(L.ptr(out), C.c_int64(out.nbytes))

    def pone():
        L.check(lib.fmwr_predict(C.byref(mcfg), L.F32, C.c_int64(n), C.c_int64(p), C.c_int64(col_i.size), L.ptr(row_size), L.ptr(col_i),
                                 L.ptr(val64), w0, L.ptr(w), L.ptr(v), L.LINK_LOGISTIC, C.c_double(0), C.c_double(0), L.ptr(out)))
    pone()
    t1 = time.perf_counter()
    for _ in range(steps):
        pone()
    dtp = time.perf_counter() - t1
    # the same fm.train on a PARKED fm.matrix (the glue's default, INTEGRATION.md item 4: the device copy lives in a slot of the R
    # object): X is already resident, every step still ships the host model in and out and trains one epoch
    d2 = L.Data.from_r_lists(ctx, n, p, row_size, col_i, val64, y64)
    h0 = ctx.transfer_bytes()

    def parked():
        m2 = L.Model(ctx, mcfg, p, L.F32)
        L.check(lib.fmwr_model_set(m2.h, C.c_double(0.0), L.ptr(w), L.ptr(v)))
        L.train_dev(ctx, m2, d2, sc)
        L.check(lib.fmwr_model_get(m2.h, C.byref(w0), L.ptr(w), L.ptr(v)))          # into the caller's (pinned) buffers, like the one-shot call
        m2.close()
    parked()
    h1 = ctx.transfer_bytes()
    t2 = time.perf_counter()
    for _ in range(steps):
        parked()
    dtk = time.perf_counter() - t2
    h2 = ctx.transfer_bytes()
    d2.close()
    resident = {"value": round((n - 1) * steps / dtk, 1), "unit": "samples/s", "ms_per_step": round(dtk / steps * 1e3, 2),
                "h2d_bytes_per_step": int((h2[0] - h1[0]) / steps), "d2h_bytes_per_step": int((h2[1] - h1[1]) / steps),
                "call": "fm.train on an fm.matrix whose device copy is parked (fmwr_model_set + fmwr_train_dev + fmwr_model_get): second and later calls of an R session"}
    for a in pinned:
        lib.fmwr_host_unpin(L.ptr(a))
    lib.fmwr_host_unpin(L.ptr(out))
    return {"value": round((n - 1) * steps / dt, 1), "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "steps": steps, "ms_per_step": round(dt / steps * 1e3, 2), "call": "fmwr_train (host fm.matrix lists -> host model)",
            "host_bytes_per_step": int(row_size.nbytes + col_i.nbytes + val64.nbytes + y64.nbytes + w.nbytes + v.nbytes + 8),
            "note": "h2d_bytes_per_step = bytes that cross PCIe: the 8-byte values are narrowed to f32 on the host by the library (threads + pinned staging ring) "
                    "while earlier chunks upload; host_bytes_per_step = the caller's buffers" if host_narrow else "values uploaded as f64 and narrowed on the device",
            "parked_matrix": resident,
            "predict": {"value": round(n * steps / dtp, 1), "unit": "rows/s", "ms_per_step": round(dtp / steps * 1e3, 2),
                        "h2d_bytes_per_step": int(row_size.nbytes + col_i.nbytes + val_bytes + w.nbytes + v.nbytes),
                        "d2h_bytes_per_step": int(out.nbytes), "call": "fmwr_predict"}}


# ------------------------------------------------------------------------------------------------ CPU legs
def host_prefix(L, data, rows):
    """first `rows` rows of the device-resident synthetic matrix, on the host"""
    rowptr, col, val, y = data.get_csr()
    e = int(rowptr[rows])
    return rowptr[:rows + 1].copy(), col[:e].copy(), val[:e].copy(), y[:rows].copy()


def oracle_for_baseline():
    from oracle import oracle as O
    if O.available("ref"):
        return O, O.Oracle("ref"), "reference"
    if not O.available("port"):
        O.build("port")
    return O, O.Oracle("port"), "port"


def time_ftrl_cpu(O, orc, rowptr, col, val, y, p, k, rows):
    rng = np.random.default_rng(20240603)
    w = np.zeros(p)
    v = rng.normal(0, 0.01, (p, k))
    cfg = O.make_cfg(solver=O.FTRL, k=k, max_iter=rows - 1, l1_w=1e-3, l2_w=1e-3, l2_v=1e-3, nthreads=1)
    t0 = time.perf_counter()
    orc.train(cfg, rows, p, rowptr[:rows + 1], col[:rowptr[rows]], val[:rowptr[rows]], y[:rows], 0.0, w, v)
    return (rows - 1) / (time.perf_counter() - t0)


def cpu_baseline_ftrl(L, data, n, p, k, F, seconds=15.0):
    O, orc, kind = oracle_for_baseline()
    probe = min(n, 4000)
    cap = min(n, 400_000)
    rowptr, col, val, y = host_prefix(L, data, cap)
    sps = time_ftrl_cpu(O, orc, rowptr, col, val, y, p, k, probe)
    rows = int(max(probe, min(cap, sps * seconds)))
    sps = time_ftrl_cpu(O, orc, rowptr, col, val, y, p, k, rows)
    # predict_batch with every host thread (the reference's only OpenMP row loop, src/core/Model.h:123,138)
    nt = orc.num_threads()
    rng = np.random.default_rng(1)
    w = rng.normal(0, 0.1, p); v = rng.normal(0, 0.01, (p, k))
    cfgp = O.make_cfg(k=k, nthreads=nt)
    t0 = time.perf_counter()
    orc.predict(cfgp, cap, p, rowptr, col, val, 0.0, w, v, 1)
    rps = cap / (time.perf_counter() - t0)
    return {"value": round(sps, 1), "unit": "samples/s", "cores": 1, "kind": kind,
            "sample": "FTRL epoch on the first %d rows of the same synthetic matrix (same p, k, nnz); 1 thread -- the reference has no parallel "
                      "sample loop (todo_list.md:7)" % rows,
            "predict": {"value": round(rps, 1), "unit": "rows/s", "cores": nt, "sample": "predict_prob on the first %d rows, %d OpenMP threads" % (cap, nt)}}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the FTRL epoch, bounded sample per step"""
    rank, world, local = dist_env()
    if rank != 0:
        return
    from fmwr_b200 import synth
    O, orc, kind = oracle_for_baseline()
    F, k = 39, args.k
    field = args.features // F
    p = field * F
    cap = min(args.rows, 200_000)
    rowptr, col, val, _ = synth.fields_csr(cap, [field] * F, None, 0, 20240601)
    score = synth.planted_scores_fast(rowptr, col, val, p, seed=20240602)
    y = synth.labels_from_scores(score, "classification", seed=20240604)
    sps = time_ftrl_cpu(O, orc, rowptr, col, val, y, p, k, min(cap, 4000))
    rows = int(max(4000, min(cap, sps * args.ref_step_seconds)))
    for _ in range(args.warmup):
        time_ftrl_cpu(O, orc, rowptr, col, val, y, p, k, min(rows, 4000))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        time_ftrl_cpu(O, orc, rowptr, col, val, y, p, k, rows)
    dt = time.perf_counter() - t0
    value = (rows - 1) * args.steps / dt
    sample = "each step = one FTRL pass over the first %d rows of the configs[1] matrix (p=%d, k=%d, 39 nnz), 1 thread" % (rows, p, k)
    out = {"impl": "reference", "metric": METRIC,
           "value": round(value, 1), "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic",
           "config": {"workload": "configs[1]: Criteo-shaped %d rows x 39 nnz, %d features, k=%d, FTRL L1+L2 binary logloss" % (args.rows, p, k),
                      "rows": args.rows, "nnz_per_row": 39, "features": p, "k": k},
           "cpu_baseline": {"value": round(value, 1), "unit": "samples/s", "cores": 1, "kind": kind, "sample": sample},
           "e2e": {"value": round(value, 1), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def multi_parity(L, multi, dist, ctx, rank, world, local, fields, k, prec, solver, n_rows, B):
    """driver-side correctness of the feature-parallel path: train an n_rows prefix of the configs[1] matrix on `world` GPUs
    (column slices, in-kernel peer exchange) and on ONE GPU (rank 0, a context without communicator), same initial model and
    batches; returns max |a-b| / max(1,|b|) over (w0, w, V) on rank 0"""
    F = len(fields)
    p = int(sum(fields))
    f0, f1, c0, c1 = multi.field_partition(fields, world)[rank]
    mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=1e-3, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
    sc = mb_solver_cfg(L, solver, 2 * (n_rows - 1), B, precision=prec)
    full = L.Data.synth(ctx, n_rows, fields, None, 0, 1, 0.1, 20240601)
    part = full.slice_columns(c0, c1)
    # identical initial parameters on both sides: the full model's device init, sliced
    m0 = L.Model(ctx, mc, p, prec)
    m0.init_random(0.0, 0.01, 20240603)
    w0_, w_, v_ = m0.get()
    m0.close()
    m = L.Model(ctx, mc, c1 - c0, prec)
    m.set(w0_, w_[c0:c1], v_[c0:c1])
    L.train_dev(ctx, m, part, sc)
    mine = m.get()
    m.close(); part.close()
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    err = None
    if rank == 0:
        gw0, gw, gv = multi.gather_model(parts)
        solo = L.Context(local)                           # no communicator: the single-GPU path
        rowptr, col, val, y = full.get_csr()
        d1 = L.Data.from_csr32(solo, n_rows, p, rowptr, col, val, y)
        m1 = L.Model(solo, mc, p, prec)
        m1.set(w0_, w_, v_)
        L.train_dev(solo, m1, d1, sc)
        sw0, sw, sv = m1.get()
        m1.close(); d1.close(); solo.close()
        err = max(abs(gw0 - sw0) / max(1.0, abs(sw0)), float(np.max(np.abs(gw - sw) / np.maximum(1, np.abs(sw)))),
                  float(np.max(np.abs(gv - sv) / np.maximum(1, np.abs(sv)))))
        moved = float(np.max(np.abs(sv - v_)))
        if not moved > 1e-4:
            err = float("inf")                            # a run that did not train proves nothing
    full.close()
    return err


def multi_parity_als(L, multi, dist, ctx, rank, world, local, solver, n_rows):
    """row-sharded ALS / MCMC against one GPU: every rank must end the sweeps with the model the single-GPU run ends with
    (MCMC: same seed -> same counter-based draws); returns max |a-b| / max(1,|b|) on rank 0"""
    afields, k = [138493, 26744, 2048], 8
    p = sum(afields)
    a0, a1 = multi.row_partition(n_rows, world)[rank]
    mc = L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=k)
    sc = L.SolverCfg(solver=solver, max_iter=2, random_step=1, min_target=0.5, max_target=5.0, mode=L.MODE_EXACT, precision=L.F64,
                     compat=L.COMPAT_REFERENCE, enable_v=1, step_size=-1, seed=7)
    d = L.Data.synth_rows(ctx, a0, a1 - a0, afields, [0, 1, 0], 0, 3, 0.3, 20240601)
    m = L.Model(ctx, mc, p, L.F64)
    m.init_random(0.0, 0.01, 20240603)
    start = m.get()
    L.train_dev(ctx, m, d, sc)
    mine = m.get()
    m.close(); d.close()
    err = None
    if rank == 0:
        solo = L.Context(local)
        d1 = L.Data.synth(solo, n_rows, afields, [0, 1, 0], 0, 3, 0.3, 20240601)
        m1 = L.Model(solo, mc, p, L.F64)
        m1.set(*start)
        L.train_dev(solo, m1, d1, sc)
        sw0, sw, sv = m1.get()
        m1.close(); d1.close(); solo.close()
        err = max(abs(mine[0] - sw0) / max(1.0, abs(sw0)), float(np.max(np.abs(mine[1] - sw) / np.maximum(1, np.abs(sw)))),
                  float(np.max(np.abs(mine[2] - sv) / np.maximum(1, np.abs(sv)))))
        if not float(np.max(np.abs(sv - start[2]))) > 1e-4:
            err = float("inf")
    return err


def run_c5(L, multi, dist, ctx, args, rank, world, timed, peak):
    """BASELINE configs[4]: SGD / TDAP minibatch epochs + predict on 100M rows x 39 nnz, 50M features, k=32, sharded over the box.
    Training is feature-parallel (every rank: all rows, its fields' columns, generated in row chunks on the device);
    predict is row-sharded with the 6.4 GB model replicated.  In this regime a batch touches a feature about once
    (1.28M ids per field against 65 536 rows), so nothing is L2-resident and the compulsory bytes are close to SURVEY 8(d)'s model."""
    n, F, k, B = args.c5_rows, 39, 32, args.batch
    field = args.c5_features // F
    fields = [field] * F
    p = field * F
    f0, f1, c0, c1 = multi.field_partition(fields, world)[rank]
    t0 = time.time()
    parts = []
    chunk = 10_000_000
    for r0 in range(0, n, chunk):
        full = L.Data.synth_rows(ctx, r0, min(chunk, n - r0), fields, None, 0, 1, 0.1, 20240601)
        parts.append(full.slice_columns(c0, c1))
        full.close()
    shard = L.Data.concat_rows(parts) if len(parts) > 1 else parts[0]
    if len(parts) > 1:
        for q in parts:
            q.close()
    ctx.sync()
    t_gen = time.time() - t0
    out = {"workload": "configs[4]: %d rows x 39 nnz, %d features, k=32; training feature-parallel x%d (fields %s), batch %d; predict row-sharded" % (
               n, p, world, [b - a for a, b, _, _ in multi.field_partition(fields, world)], B),
           "setup_s": round(t_gen, 1)}
    ctx.sync(); ctx.timer_start()
    info = shard.minibatch_info(B)
    out["prep_ms"] = round(ctx.timer_stop_ms(), 1)
    for name, solver in (("sgd", L.SGD), ("tdap", L.TDAP)):
        mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=0.0 if name == "sgd" else 1e-3, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
        m = L.Model(ctx, mc, c1 - c0, L.F32)
        m.init_random(0.0, 0.01, 20240603 + c0)
        sc = mb_solver_cfg(L, solver, n - 1, B)
        L.train_dev(ctx, m, shard, sc)
        steps = 2
        ms = timed(lambda: L.train_dev(ctx, m, shard, sc), steps) / steps
        m.close()
        sps = (n - 1) / (ms * 1e-3)
        # compulsory bytes of the whole job: every rank's update bytes from ITS segment counts (all-reduced) + the forward's
        segs = [None] * world
        dist.all_gather_object(segs, info)
        tot = {"n_segments": sum(q["n_segments"] for q in segs), "n_entries": sum(q["n_entries"] for q in segs)}
        comp = k1_compulsory_bytes(tot, n, F, 32) + k2_compulsory_bytes(name, tot, 32)
        out[name] = {"value": round(sps, 1), "unit": "samples/s", "ms_per_step": round(ms, 2), "optimizer_steps_per_epoch": info["n_batches"],
                     "compulsory_bytes_per_step": int(comp), "achieved_gbs": round(comp / (ms * 1e-3) / 1e9, 1),
                     "frac_of_n_gpus_peak": round(comp / (ms * 1e-3) / 1e9 / (peak * world), 4),
                     "survey_model_bytes_per_sample": ALG_BYTES[name](F, k)}
    shard.close()
    # predict: rows sharded, model replicated
    r0, r1 = multi.row_partition(n, world)[rank]
    pd = L.Data.synth_rows(ctx, r0, r1 - r0, fields, None, 0, 0, 0.1, 20240601)
    mc = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k)
    pm = L.Model(ctx, mc, p, L.F32)
    pm.init_random(0.0, 0.01, 20240603)
    for _ in range(2):
        L.predict_dev(ctx, pm, pd, L.LINK_LOGISTIC)
    steps = 3
    ms = timed(lambda: L.predict_dev(ctx, pm, pd, L.LINK_LOGISTIC), steps) / steps
    pd.close(); pm.close()
    b_fwd = ALG_BYTES["predict"](F, k)
    rps = n / (ms * 1e-3)
    out["predict"] = {"value": round(rps, 1), "unit": "rows/s", "ms_per_step": round(ms, 3), "alg_bytes_per_row": b_fwd,
                      "achieved_gbs": round(rps * b_fwd / 1e9, 1), "frac_of_n_gpus_peak": round(rps * b_fwd / 1e9 / (peak * world), 4),
                      "note": "6.4 GB of factor rows per GPU: every gather is a DRAM access, so SURVEY 8(d)'s per-row model is the compulsory traffic here"}
    return out


def run_engine_multi(args, rank, world, local):
    """N > 1 (torchrun, one rank per GPU): minibatch epochs FEATURE-parallel, the per-batch exchange of the rows' partials inside
    our own kernels over CUDA-IPC peer windows (NVLink stores + in-kernel flags; FMWR_BENCH_NCCL=1: one NCCL all-reduce per batch
    instead); predict.FM row-sharded with no collective; ALS / MCMC row-sharded with one statistics exchange per coordinate step.
    Strong scaling: the configs[1] problem is fixed, N grows."""
    import torch
    import torch.distributed as dist
    from fmwr_b200 import _lib as L
    from fmwr_b200 import multi
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("gloo", rank=rank, world_size=world)       # control plane only (id exchange, barriers, max-reduce)
    lib = L.lib()
    ctx = L.Context(local)
    ctx.comm_init(multi.exchange_unique_id(dist, L.Context, rank), rank, world)
    peak, peak_src = measured_peak()
    n, F, k, B = args.rows, 39, args.k, args.batch
    kp = (k + 3) // 4 * 4
    use_peer = os.environ.get("FMWR_BENCH_NCCL", "0") != "1"
    if use_peer:
        multi.open_peer_windows(dist, ctx, rank, world, B, k)      # per-batch exchange inside our kernels (NVLink), no NCCL call
    field = args.features // F
    p = field * F
    fields = [field] * F
    f0, f1, c0, c1 = multi.field_partition(fields, world)[rank]

    full = L.Data.synth(ctx, n, fields, None, 0, 1, 0.1, 20240601)
    data = full.slice_columns(c0, c1)
    full.close()
    mcfg = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=1e-3, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
    model = L.Model(ctx, mcfg, c1 - c0, L.F32)
    model.init_random(0.0, 0.01, 20240603 + c0)
    epoch = n - 1
    sc = mb_solver_cfg(L, L.FTRL, epoch, B)

    def timed(fn, steps):
        ctx.sync(); dist.barrier()
        ctx.timer_start()
        for _ in range(steps):
            fn()
        ms = ctx.timer_stop_ms()
        ctx.sync(); dist.barrier()
        t = torch.tensor([ms], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                      # device time, max over ranks
        return float(t[0])

    info = data.minibatch_info(B)
    for _ in range(args.warmup):
        L.train_dev(ctx, model, data, sc)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = ctx.launches()
    ms_train = timed(lambda: L.train_dev(ctx, model, data, sc), args.steps)
    l1 = ctx.launches()
    train_sps = epoch * args.steps / (ms_train * 1e-3)
    # per-kernel events on rank 0's stream (second pass)
    buf = C.create_string_buffer(1 << 16)
    L.check(lib.fmwr_profile_enable(ctx.h, 1))
    L.train_dev(ctx, model, data, sc)
    L.check(lib.fmwr_profile_enable(ctx.h, 1))
    ms_prof = timed(lambda: L.train_dev(ctx, model, data, sc), args.steps)
    L.check(lib.fmwr_profile_read(ctx.h, buf, C.c_int64(len(buf))))
    prof = parse_profile(buf.value.decode())
    L.check(lib.fmwr_profile_enable(ctx.h, 0))
    model.close()
    infos = [None] * world
    dist.all_gather_object(infos, info)
    tot = {"n_segments": sum(q["n_segments"] for q in infos), "n_entries": sum(q["n_entries"] for q in infos)}

    # SGD epoch on the same column slices (the solver the north_star's scaling target names)
    sgd = None
    if not args.no_solvers:
        mc_s = L.ModelCfg(task=L.CLASSIFICATION, keep_w0=1, keep_w1=1, k=k, l2_w0=0.0, l1_w1=0.0, l2_w1=1e-3, l1_v=0.0, l2_v=1e-3)
        ms_ = L.Model(ctx, mc_s, c1 - c0, L.F32)
        ms_.init_random(0.0, 0.01, 20240603 + c0)
        sc_s = mb_solver_cfg(L, L.SGD, epoch, B)
        for _ in range(args.warmup):
            L.train_dev(ctx, ms_, data, sc_s)
        steps_s = max(1, min(args.steps, 5))
        ms_sgd = timed(lambda: L.train_dev(ctx, ms_, data, sc_s), steps_s) / steps_s
        ms_.close()
        comp = k1_compulsory_bytes(tot, n, F, kp) + k2_compulsory_bytes("sgd", tot, kp)
        sgd = {"workload": "configs[1] matrix, SGD minibatch epoch (batch %d), feature-parallel x%d" % (B, world),
               "value": round(epoch / (ms_sgd * 1e-3), 1), "unit": "samples/s", "ms_per_step": round(ms_sgd, 3),
               "compulsory_bytes_per_step": int(comp), "frac_of_n_gpus_peak": round(comp / (ms_sgd * 1e-3) / 1e9 / (peak * world), 4)}
    data.close()

    # correctness carried in the line: N GPUs against one GPU on a prefix, same batches
    parity = None
    if not args.no_parity:
        e64 = multi_parity(L, multi, dist, ctx, rank, world, local, fields, k, L.F64, L.FTRL, args.parity_rows, 8192)
        e32 = multi_parity(L, multi, dist, ctx, rank, world, local, fields, k, L.F32, L.FTRL, args.parity_rows, 8192)
        es = multi_parity(L, multi, dist, ctx, rank, world, local, fields, k, L.F64, L.SGD, args.parity_rows, 8192)
        ea = multi_parity_als(L, multi, dist, ctx, rank, world, local, L.ALS, args.parity_rows)
        em = multi_parity_als(L, multi, dist, ctx, rank, world, local, L.MCMC, args.parity_rows)
        if rank == 0:
            parity = {"multi_vs_single_max_rel_err": e64, "ftrl_f32": e32, "sgd_f64": es, "als_f64": ea, "mcmc_f64": em,
                      "rows": args.parity_rows, "batch": 8192, "epochs": 2,
                      "what": "max |a-b|/max(1,|b|) over (w0, w, V): FTRL fp64 (headline key), FTRL fp32 (the benchmarked precision; the S_f sums are "
                              "split by shard, so fp32 differs by rounding), SGD fp64 -- %d GPUs (in-kernel peer exchange) against one GPU; "
                              "als_f64 / mcmc_f64: two sweeps (w and V blocks) row-sharded against one GPU on a MovieLens-shaped prefix" % world,
                      "asserted": "fp64 < 1e-8 (ALS / MCMC < 1e-6: their statistics are summed in a different order), fp32 < 5e-3"}
        ok = [parity is None or (parity["multi_vs_single_max_rel_err"] < 1e-8 and parity["sgd_f64"] < 1e-8 and parity["ftrl_f32"] < 5e-3
                                 and parity["als_f64"] < 1e-6 and parity["mcmc_f64"] < 1e-6)]
        dist.broadcast_object_list(ok, src=0)
        if not ok[0]:
            if rank == 0:
                print(json.dumps({"error": "multi-GPU parity check failed", "parity": parity}), flush=True)
            ctx.comm_destroy(); ctx.close()
            dist.barrier(); dist.destroy_process_group()
            sys.exit(3)

    # predict.FM: rows sharded, full model replicated
    r0, r1 = multi.row_partition(n, world)[rank]
    pdata = L.Data.synth_rows(ctx, r0, r1 - r0, fields, None, 0, 0, 0.1, 20240601)
    pmodel = L.Model(ctx, mcfg, p, L.F32)
    pmodel.init_random(0.0, 0.01, 20240603)
    for _ in range(args.warmup):
        L.predict_dev(ctx, pmodel, pdata, L.LINK_LOGISTIC)
    ms_pred = timed(lambda: L.predict_dev(ctx, pmodel, pdata, L.LINK_LOGISTIC), args.steps)
    pred_rps = n * args.steps / (ms_pred * 1e-3)
    pdata.close(); pmodel.close()

    # ALS / MCMC sweeps, rows sharded (SURVEY 8e): configs[2] / configs[3] split into `world` row ranges, one exchange of the
    # field's statistics per coordinate step (peer windows, else one NCCL all-reduce); every rank ends the sweep with the same model
    als = {}
    if not args.no_solvers and args.rows >= 1_000_000:
        na, afields = 20_000_000, [138493, 26744, 2048]
        a0, a1 = multi.row_partition(na, world)[rank]
        ad = L.Data.synth_rows(ctx, a0, a1 - a0, afields, [0, 1, 0], 0, 3, 0.3, 20240601)
        pa_, Na_ = sum(afields), 3 * na
        for name, solver, ka in (("als", L.ALS, 32), ("mcmc", L.MCMC, 64)):
            am = L.Model(ctx, L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=ka), pa_, L.F32)
            am.init_random(0.0, 0.01, 20240603)
            asc = L.SolverCfg(solver=solver, max_iter=1, random_step=1, min_target=0.5, max_target=5.0, mode=L.MODE_EXACT, precision=L.F32,
                              compat=L.COMPAT_REFERENCE, enable_v=1, step_size=-1, seed=5)
            for _ in range(args.warmup):
                L.train_dev(ctx, am, ad, asc)
            steps_a = max(1, min(args.steps, 5))
            ms_a = timed(lambda: L.train_dev(ctx, am, ad, asc), steps_a) / steps_a
            sweep_bytes = na * (8 + 3 * (12 + 4 * ka)) + 16 * na + 16 * Na_ + ka * (32 * Na_ + 4 * na + 8 * pa_) + (8 * na if name == "mcmc" else 0)
            als[name] = {"workload": "configs[%d]: 20000000 ratings x 3 one-hot fields, k=%d, one %s sweep, rows sharded over %d GPUs "
                                     "(statistics of 2 x |field| f32 exchanged per coordinate step through the peer windows)" % (2 if name == "als" else 3, ka, name.upper(), world),
                         "value": round(na / (ms_a * 1e-3), 1), "unit": "ratings/s", "ms_per_step": round(ms_a, 3),
                         "frac_of_n_gpus_peak": round(sweep_bytes / (ms_a * 1e-3) / 1e9 / (peak * world), 4)}
            am.close()
        ad.close()

    c5 = None
    if (world == 8 and not args.no_c5) or os.environ.get("FMWR_BENCH_C5") == "1":
        c5 = run_c5(L, multi, dist, ctx, args, rank, world, timed, peak)
    clk = clocks.stop() if rank == 0 else None

    if rank == 0:
        b_fwd, b_ftrl = ALG_BYTES["predict"](F, k), ALG_BYTES["ftrl"](F, k)
        roof = None
        kn = update_kernel_of(prof)
        if kn and prof[kn][1] > 0:
            launches, ms = prof[kn]
            per_launch = k2_compulsory_bytes("ftrl", info, kp) * (args.steps) / launches     # rank 0's own segments
            ach = per_launch / (ms / launches * 1e-3) / 1e9
            roof = {"kernel": kn, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                    "traffic": None, "alg_bytes_per_launch": int(per_launch), "peak_source": peak_src, "launches": launches, "avg_launch_ms": round(ms / launches, 5),
                    "note": "rank 0 only: %d of %d fields; compulsory bytes from its real segment counts" % (f1 - f0, F), "share_of_step": round(ms / ms_prof, 4)}
        step_bytes = k1_compulsory_bytes(tot, n, F, kp) + k2_compulsory_bytes("ftrl", tot, kp)
        solvers = dict(als)
        if sgd:
            solvers["sgd"] = sgd
        if c5:
            solvers["c5"] = c5
        out = {
            "metric": METRIC,
            "value": round(train_sps, 1), "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_train / args.steps, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: Criteo-shaped %d rows x %d nnz, %d features, k=%d, FTRL L1+L2 binary logloss" % (n, F, p, k),
                       "rows": n, "nnz_per_row": F, "features": p, "k": k, "batch_size": B, "mode": "minibatch",
                       "parallelism": "feature-parallel x%d (fields split %s), per minibatch one exchange of rows x (k+4) f32 partials %s; predict row-sharded" % (
                           world, [b - a for a, b, _, _ in multi.field_partition(fields, world)],
                           "inside the forward/exchange/update kernels (peer-memory stores over NVLink + in-kernel flags)" if use_peer else "by NCCL all-reduce"),
                       "l2_flush": "inputs larger than L2"},
            "roofline": roof,
            "step_roofline": {"compulsory_bytes_per_step": int(step_bytes), "achieved": round(step_bytes / (ms_train / args.steps * 1e-3) / 1e9, 1), "unit": "GB/s",
                              "frac_of_n_gpus_peak": round(step_bytes / (ms_train / args.steps * 1e-3) / 1e9 / (peak * world), 4),
                              "survey_model_bytes_per_sample": b_ftrl},
            "parity": parity,
            "multi_vs_single_max_rel_err": parity["multi_vs_single_max_rel_err"] if parity else None,
            "kernels": {name: {"launches": v[0], "ms": round(v[1], 3)} for name, v in prof.items()},
            "predict": {"value": round(pred_rps, 1), "unit": "rows/s", "ms_per_step": round(ms_pred / args.steps, 3),
                        "roofline": {"bound": "hbm", "survey_model_gbs": round(pred_rps * b_fwd / 1e9, 1), "unit": "GB/s",
                                     "note": "per-row model, no cache credit (V is L2-resident per GPU at this size): see the N=1 line for the fraction by measured DRAM bytes"}},
            "solvers": solvers or None,
            "cpu_baseline": None,
            "e2e": None,
            "gpu_launches": int(l1 - l0),
            "clocks": clk,
        }
        print(json.dumps(out), flush=True)
    ctx.comm_destroy()
    ctx.close()
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the headline FTRL epoch and predict.FM, of the SGD / TDAP / ALS / MCMC lines and of e2e; the "
                         "exact-mode (one run per solver), batch-sweep (two epochs per batch size) and configs[0] (2, 2, 5 and 3 runs) "
                         "lines time fixed counts, and the secondary lines of a multi-GPU run at most 5")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--features", type=int, default=1_000_000)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-solvers", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--sweep-rows", type=int, default=1_000_000)
    ap.add_argument("--parity-rows", type=int, default=200_000)
    ap.add_argument("--c5-rows", type=int, default=100_000_000)
    ap.add_argument("--c5-features", type=int, default=50_000_000)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--ref-step-seconds", type=float, default=4.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the model after the last timed training step and the last timed predict.FM output (fixed samples of "
                         "the large arrays) to DIR/<name>.npy; single-GPU engine runs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "engine" or dist_env()[1] > 1):
        ap.error("--dump-outputs is for single-GPU engine runs")
    if args.warmup < 3 and args.impl == "engine":
        args.warmup = max(args.warmup, 3) if os.environ.get("FMWR_BENCH_STRICT", "1") == "1" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
