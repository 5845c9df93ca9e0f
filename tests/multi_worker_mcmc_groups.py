"""torchrun worker for tests/test_gpu_multi_mcmc_groups.py: grouped MCMC (fmwr_solver_cfg::attr_group) on ROW-sharded data must
give every rank the parameters of the single-GPU run on the whole data.  The group priors are drawn on every rank from its
replicated model; with injected normal / gamma streams both runs make the same draws."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch.distributed as dist
    from fmwr_b200 import _lib as L
    from fmwr_b200 import multi, synth
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ctx = L.Context(local)
    ctx.comm_init(multi.exchange_unique_id(dist, L.Context, rank), rank, world)
    fields = [700, 260, 24]
    n, k = 24000, 8
    rowptr, col, val, p = synth.fields_csr(n, fields, [0, 1, 0], 0, 41)
    y = synth.labels_from_scores(synth.planted_scores_fast(rowptr, col, val, p, seed=42), "regression", seed=43)
    rng = np.random.default_rng(44)
    w = np.zeros(p); v = rng.normal(0, 0.05, (p, k)); w0 = 0.0
    grp = np.ascontiguousarray(np.repeat(np.arange(len(fields)), fields), np.int32)
    G = len(fields)
    r0, r1 = multi.row_partition(n, world)[rank]
    sweeps = 3
    normals = np.ascontiguousarray(rng.normal(size=sweeps * (1 + G + (k + 1) * (p + G)) + 64), np.float64)
    gammas = np.ascontiguousarray(rng.gamma(5.0, size=sweeps * (1 + G * (1 + k)) + 64), np.float64)
    ok = True
    for exchange in ("nccl", "peer"):
        if exchange == "peer":
            multi.open_peer_windows(dist, ctx, rank, world, 4096, k)
        mc = L.ModelCfg(task=L.REGRESSION, keep_w0=1, keep_w1=1, k=k)
        sc = L.SolverCfg(solver=L.MCMC, max_iter=sweeps, random_step=1, min_target=float(y.min()), max_target=float(y.max()),
                         mode=L.MODE_EXACT, precision=L.F64, compat=L.COMPAT_REFERENCE, enable_v=1, step_size=-1, seed=7)
        sc.normals = L.ptr(normals); sc.n_normals = normals.size
        sc.gammas = L.ptr(gammas); sc.n_gammas = gammas.size
        sc.attr_group = L.ptr(grp); sc.n_groups = G
        e0, e1 = int(rowptr[r0]), int(rowptr[r1])
        shard = L.Data.from_csr32(ctx, r1 - r0, p, (rowptr[r0:r1 + 1] - rowptr[r0]).astype(np.uint32), col[e0:e1], val[e0:e1], y[r0:r1])
        m = L.Model(ctx, mc, p, L.F64)
        m.set(w0, w, v)
        L.train_dev(ctx, m, shard, sc)
        mine = m.get()
        m.close(); shard.close()
        parts = [None] * world
        dist.all_gather_object(parts, mine)
        if rank == 0:
            solo = L.Context(local)
            d1 = L.Data.from_csr32(solo, n, p, rowptr, col, val, y)
            m1 = L.Model(solo, mc, p, L.F64)
            m1.set(w0, w, v)
            L.train_dev(solo, m1, d1, sc)
            sw0, sw, sv = m1.get()
            m1.close(); d1.close(); solo.close()
            gw0, gw, gv = parts[0]
            err = max(abs(gw0 - sw0), float(np.max(np.abs(gw - sw) / np.maximum(1, np.abs(sw)))),
                      float(np.max(np.abs(gv - sv) / np.maximum(1, np.abs(sv)))))
            moved = float(np.max(np.abs(sv - v)))
            same = all(q[0] == parts[0][0] and np.array_equal(q[1], parts[0][1]) and np.array_equal(q[2], parts[0][2]) for q in parts[1:])
            print("exchange=%s row-sharded grouped MCMC world=%d max rel err vs single GPU = %.3e (moved %.3e) replicas identical=%s" % (
                exchange, world, err, moved, same), flush=True)
            ok = ok and err < 1e-8 and moved > 1e-3 and same
    flag = [ok]
    dist.broadcast_object_list(flag, src=0)
    ctx.comm_destroy(); ctx.close()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MULTI_GROUPS_OK" if flag[0] else "MULTI_GROUPS_FAIL", flush=True)
    sys.exit(0 if flag[0] else 1)


if __name__ == "__main__":
    main()
