"""Many directions per LSQR launch against one conic operator: k single calls against one multi call.

For each config and k in --ks, forward and reverse are timed three ways, alternating from round to round:
  (a) k single calls (conic_forward / conic_reverse), device time summed over the calls;
  (b) one multi call (conic_forward_multi / conic_reverse_multi);
  (c) reverse only, without PSD cones: the lock-step batch (ConicBatch) holding k copies of the problem.
Device time is the library's CUDA-event bracket of the LSQR launch(es) (ctx.last_kernel_ms); each arm keeps the best
of its rounds.

Algorithmic bytes per iteration, with the matrix streamed once for all k directions:
    bytes = 2 (12 nnz(M) + 4 (N + 1)) + 88 N k
(12 bytes per nonzero of val + colind and 4 bytes per row pointer for M and M', 88 bytes per entry and direction of the
vectors one iteration reads and writes), reported as a share of the project's measured 6541.8 GB/s (DESIGN §4.5).
The largest relative 2-norm difference from (a) over the first 8 directions is reported as max_rel_vs_a.

Configs: 4 (as named, 500 fixed iterations), 4c (conditioned, converged at the default tolerances), 4x (scaled 200x,
50 fixed iterations), 4xb (scaled 200x, stage-structured, 50 fixed iterations), 5 (max-cut PSD, 50 fixed iterations).
Prints one JSON line per (config, k, mode) after a first line with the GPU's name and power limit."""
import argparse
import json
import os
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench_data  # noqa: E402
import diffopt_b200  # noqa: E402
from bench_exp_cone import gpu_info  # noqa: E402
from bench_lsqr_drivers import config5_data  # noqa: E402

HBM_GBS = 6541.8
KEEP = 8  # directions whose outputs are compared between the arms (host memory on the scaled configs)


def fixed(iters):
    return dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)


DEFAULT = dict(atol=1.4901161193847656e-08, btol=1.4901161193847656e-08, conlim=1 / 1.4901161193847656e-08, maxiter=None)


def model_of(ctx, d, tol, setup=True):
    cm = diffopt_b200.submodule("conic")
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"], d.get("cone_params"))
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    model.tolerances = dict(tol)
    if setup:
        model.vp()
    return model


def rel_max(a, b):
    return float(max(np.linalg.norm(a[j] - b[j]) / max(np.linalg.norm(b[j]), 1e-300) for j in range(len(b))))


def bench_config(ctx, name, d, tol, ks, rounds, batch_max_k):
    cm = diffopt_b200.submodule("conic")
    model = model_of(ctx, d, tol)
    m, n = d["A"].shape
    N = n + m + 1
    nnzM = 2 * 2 * d["A"].nnz + 2 * n + 2 * m  # A, A', c, b, the unit blocks (order of magnitude: dominated by A)
    psd = any(int(t) == cm.CONE_PSD for t in d["cone_types"])
    rng = np.random.default_rng(17)
    kmax = max(ks)
    seeds = rng.normal(size=(kmax, n))
    # sparse dA directions with uniformly random positions: 20 nonzeros per row on the named sizes, 0.2 on the scaled ones
    nnz = int(m * (20 if n <= 100_000 else 0.2))
    dAs = [sp.csc_matrix((rng.normal(size=nnz), (rng.integers(0, m, nnz), rng.integers(0, n, nnz))), shape=(m, n))
           for _ in range(kmax)]
    dbs, dcs = rng.normal(size=(kmax, m)), rng.normal(size=(kmax, n))
    batch = {}
    for k in ks:
        def singles_rev():
            ms, out, itn = 0.0, [], 0
            for j in range(k):
                model.reverse_differentiate(seeds[j])
                ms += model.last_stats["kernel_ms"]
                itn += model.last_stats["itn"]
                if j < KEEP:
                    out.append(model.back_grad_cache["g"].copy())
            return ms, np.array(out), itn

        def multi_rev():
            r = model.reverse_differentiate_multi(seeds[:k])
            return ctx.last_kernel_ms, r["g"][:KEEP].copy(), int(r["stats"][:, 1].sum())

        def singles_fwd():
            ms, out, itn = 0.0, [], 0
            for j in range(k):
                model.forward_differentiate(dAs[j], dbs[j], dcs[j])
                ms += model.last_stats["kernel_ms"]
                itn += model.last_stats["itn"]
                if j < KEEP:
                    out.append(model.forward_variable_primal().copy())
            return ms, np.array(out), itn

        def multi_fwd():
            f = model.forward_differentiate_multi(dAs[:k], dbs[:k], dcs[:k])
            return ctx.last_kernel_ms, f["dx"][:KEEP].copy(), int(f["stats"][:, 1].sum())

        arms = {("reverse", "a_single"): singles_rev, ("reverse", "b_multi"): multi_rev,
                ("forward", "a_single"): singles_fwd, ("forward", "b_multi"): multi_fwd}
        if not psd and k <= batch_max_k:
            if k not in batch:
                b = cm.ConicBatch(ctx, [model_of(ctx, d, tol, setup=False) for _ in range(k)], ctas_per_problem=1)
                b.tolerances = dict(tol)
                batch[k] = b

            def batch_rev():
                out = batch[k].reverse_differentiate(seeds[:k])
                return batch[k].kernel_ms, np.asarray(out["g"])[:KEEP].copy(), int(np.asarray(out["stats"])[:, 1].sum())
            arms[("reverse", "c_batch")] = batch_rev
        best = {}
        outs = {}
        for rnd in range(rounds + 1):  # round 0 warms every shape up
            order = list(arms) if rnd % 2 == 0 else list(arms)[::-1]
            for key in order:
                ms, out, itn = arms[key]()
                if rnd == 0:
                    continue
                if key not in best or ms < best[key][0]:
                    best[key] = (ms, itn)
                outs[key] = out
        for (mode, arm), (ms, itn) in sorted(best.items()):
            iters = itn / k  # mean iterations per direction
            bytes_it = 2 * (12 * nnzM + 4 * (N + 1)) + 88 * N * k
            rec = dict(config=name, k=k, mode=mode, arm=arm, device_ms=round(ms, 4),
                       us_per_direction_iteration=round(1e3 * ms / max(itn, 1), 3), mean_itn=round(iters, 1),
                       bytes_per_iteration=bytes_it,
                       hbm_share=round(bytes_it * iters / (ms * 1e-3) / (HBM_GBS * 1e9), 4) if ms > 0 else None)
            if arm != "a_single":
                rec["max_rel_vs_a"] = rel_max(outs[(mode, arm)], outs[(mode, "a_single")])
            print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--configs", default="4,4c,4x,4xb,5")
    ap.add_argument("--ks", default="1,4,8,32,64")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--batch-max-k-large", type=int, default=8,
                    help="largest k of the lock-step batch arm on the scaled configs (k copies of a 1e6-row problem)")
    args = ap.parse_args()
    print(json.dumps(gpu_info()), flush=True)
    ctx = diffopt_b200.Context(0)
    ks = [int(k) for k in args.ks.split(",")]
    big = dict(n=1_000_000, n_zero=100_000, n_nonneg=800_000, n_soc=60_000)
    makers = {
        "4": (lambda: bench_data.conic_config4(), fixed(500), 10**9),
        "4c": (lambda: bench_data.conic_config4_conditioned(), DEFAULT, 10**9),
        "4x": (lambda: bench_data.conic_config4(**big), fixed(50), args.batch_max_k_large),
        "4xb": (lambda: bench_data.conic_config4(col_window=2000, **big), fixed(50), args.batch_max_k_large),
        "5": (config5_data, fixed(50), 0),
    }
    for name in args.configs.split(","):
        make, tol, bmax = makers[name]
        bench_config(ctx, name, make(), tol, ks, args.rounds, bmax)


if __name__ == "__main__":
    main()
