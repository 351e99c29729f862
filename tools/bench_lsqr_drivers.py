"""A/B timing of the LSQR drivers: two builds of libdiffopt_b200.so on the same inputs, in one process.

Each library gets its own context (the same override `DIFFOPT_B200_LIB` provides, one per build); every workload runs on
both, alternating the order from round to round, and each round keeps the best of `--reps` runs.  The spread of an arm
is (max - min) / min over its rounds.  All LSQR solves run a fixed number of iterations (atol = btol = conlim = 0), so
both builds do the same work; their outputs are compared at the end (relative 2-norm difference).
Run each pair in both orders: the same build loaded twice reads about 1 % apart on some workloads (the second
context is not the first), so differences of that size are position, not code.

Workloads (device time from the library's CUDA-event bracket):
  config5_reverse_50     max-cut SDP, one 200 x 200 PSD cone (bench_aux config 5): 50 iterations, PSD build
  config5_reverse_3      the same problem after 3 iterations (output parity)
  config5_dpi_apply      the same problem: one Dpi apply (conic_dpi_apply)
  config1_kkt_lsqr       LP config 1: LSQR on the explicit KKT matrix (lsqr_csc), cluster driver
  config4c_reverse       config 4, well-conditioned generator: cluster driver
  config4_mid_reverse    config-4 generator with work in (2^20, 4 * 2^20]: gstream driver
  config4c_mid_reverse_3 the same size on the well-conditioned generator after 3 iterations (output parity)
  config4xb_reverse      config 4 scaled 200x, stage-structured sparsity: streaming driver
  config4b_batch         lock-step batch of 296 config-4 problems
  csr_large_lsqr         explicit CSR operator with work above 4 * 2^20 (lsqr_csc): gstream driver
  config4_conic_apply_M  config 4: one M apply (conic_M_apply)
  config4c_reverse_3     config 4c after 3 iterations (output parity only)

Prints one JSON line per workload after a first line with the GPU's name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench_data  # noqa: E402
import diffopt_b200  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in out.split(","))
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        return dict(gpu="unknown")


def context_for(lib_path):
    capi = diffopt_b200.submodule("_capi")
    capi.LIB_PATH, capi._lib = os.path.abspath(lib_path), None
    return capi.Context(0)


def fixed(iters):
    return dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)


def config5_data():
    """bench_aux.config5's problem (same seed)."""
    from oracle import cones as ocones
    dd, r = 200, 20
    rng = np.random.default_rng(5)
    V = rng.normal(size=(dd, r)); V /= np.linalg.norm(V, axis=1, keepdims=True)
    X = V @ V.T
    Qf, _ = np.linalg.qr(np.hstack([V, rng.normal(size=(dd, dd - r))]))
    W = Qf[:, r:]
    Smat = (W * rng.uniform(0.5, 1.5, size=dd - r)) @ W.T
    k = dd * (dd + 1) // 2
    s = np.concatenate([np.zeros(dd), ocones.vec_symm(X)])
    y = np.concatenate([rng.normal(size=dd), ocones.vec_symm(Smat)])
    iu = [(i * (i + 1) // 2 + i) for i in range(dd)]
    A = sp.vstack([sp.csc_matrix((np.ones(dd), (np.arange(dd), iu)), shape=(dd, k)), -sp.identity(k)]).tocsc()
    x = ocones.vec_symm(X)
    t = rng.normal(size=dd + k)
    return dict(A=A, b=A @ x + s, c=-(A.T @ y), x=x, s=s, y=y, cone_types=[ocones.ZERO, ocones.PSD], cone_dims=[dd, k],
                t=t, seed=rng.normal(size=k))


def conic_model(ctx, d):
    cm = diffopt_b200.submodule("conic")
    model = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"])
    model.set_variable_primal(d["x"]); model.set_constraint_primal(d["s"]); model.set_constraint_dual(d["y"])
    return model


def workloads(args):
    """name -> (setup(ctx) -> state, run(ctx, state) -> (ms, output))."""
    from oracle import qp as oqp
    lsqr = diffopt_b200.submodule("lsqr")
    cm = diffopt_b200.submodule("conic")
    w = {}

    def reverse(d, iters):
        def setup(ctx):
            m = conic_model(ctx, d)
            m.tolerances = fixed(iters)
            return m

        def run(ctx, m):
            m.reverse_differentiate(d["seed"])
            assert m.last_stats["itn"] == iters, m.last_stats
            return m.last_stats["kernel_ms"], m.back_grad_cache["g"].copy()
        return setup, run

    def csc(A, b, iters):
        def run(ctx, _):
            x, st = lsqr.lsqr_csc(ctx, A, b, maxiter=iters, atol=0.0, btol=0.0, conlim=0.0)
            assert st["itn"] == iters, st
            return ctx.last_kernel_ms, x
        return (lambda ctx: None), run

    d5 = config5_data()
    w["config5_reverse_50"] = reverse(d5, 50)
    w["config5_reverse_3"] = reverse(d5, 3)

    def dpi_run(ctx, m):
        out = m.dpi_apply(d5["t"])
        return ctx.last_kernel_ms, out
    w["config5_dpi_apply"] = (lambda ctx: conic_model(ctx, d5), dpi_run)

    d1 = bench_data.lp_config1()
    K = sp.csc_matrix(oqp.create_lhs(d1["z"], d1["lam"], d1["Q"], d1["G"], d1["h"], d1["A"]))
    rhs = np.zeros(K.shape[0]); rhs[:d1["Q"].shape[0]] = d1["seed"]
    w["config1_kkt_lsqr"] = csc(K, rhs, 30)   # (converges -- istop 5 -- after 60)

    d4c = bench_data.conic_config4_conditioned()
    w["config4c_reverse"] = reverse(d4c, 200)
    w["config4c_reverse_3"] = reverse(d4c, 3)

    # work = 2 nnz(A) + n + 2 m = 1.2e6 + 4e4 + 1.2e5 ~ 1.36e6: above 2^20, below the streaming threshold 4 * 2^20
    mid = dict(n=40_000, n_zero=4_000, n_nonneg=32_000, n_soc=2_400)
    w["config4_mid_reverse"] = reverse(bench_data.conic_config4(**mid), 200)
    w["config4c_mid_reverse_3"] = reverse(bench_data.conic_config4_conditioned(**mid), 3)

    if not args.quick:
        w["config4xb_reverse"] = reverse(bench_data.conic_config4(n=1_000_000, n_zero=100_000, n_nonneg=800_000,
                                                                  n_soc=60_000, col_window=2000), 50)

        datas = [bench_data.conic_config4(seed=4000 + k) for k in range(296)]
        seeds = np.stack([d["seed"] for d in datas])

        def batch_setup(ctx):
            b = cm.ConicBatch(ctx, [conic_model(ctx, d) for d in datas], ctas_per_problem=1)
            b.tolerances = fixed(100)
            return b

        def batch_run(ctx, b):
            out = b.reverse_differentiate(seeds)
            return b.kernel_ms, np.asarray(out["g"]).copy()
        w["config4b_batch"] = (batch_setup, batch_run)

    # 2.5e6 x 1e6, 2 random entries per row plus a unit diagonal: nnz ~ 6e6, work = nnz + rows + columns ~ 9.5e6
    rng = np.random.default_rng(11)
    nr, nc = 2_500_000, 1_000_000
    R = sp.random(nr, nc, density=2.0 / nc, random_state=rng, format="csc") + sp.eye(nr, nc, format="csc")
    w["csr_large_lsqr"] = csc(R.tocsc(), rng.normal(size=nr), 30)

    d4 = bench_data.conic_config4()
    t4 = np.random.default_rng(12).normal(size=d4["A"].shape[1] + d4["A"].shape[0] + 1)

    def apply_run(ctx, m):
        out = m.M_apply(t4)
        return ctx.last_kernel_ms, out
    w["config4_conic_apply_M"] = (lambda ctx: conic_model(ctx, d4), apply_run)
    return w


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--libs", nargs=2, required=True, metavar=("A", "B"), help="the two builds of libdiffopt_b200.so")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=2, help="runs per round; the round keeps the fastest")
    ap.add_argument("--quick", action="store_true", help="skip the 4xb and 4b workloads (slow to generate)")
    ap.add_argument("--only", default="", help="comma-separated workload names")
    args = ap.parse_args()
    print(json.dumps(dict(gpu_info(), libs=args.libs)), flush=True)
    ctxs = [context_for(p) for p in args.libs]
    wl = workloads(args)
    if args.only:
        wl = {k: v for k, v in wl.items() if k in args.only.split(",")}
    for name, (setup, run) in wl.items():
        states = [setup(c) for c in ctxs]
        for c, s in zip(ctxs, states):   # warm-up (module load, buffers)
            run(c, s)
        ms = [[], []]
        outs = [None, None]
        for r in range(args.rounds):
            for arm in ((0, 1) if r % 2 == 0 else (1, 0)):
                best = float("inf")
                for _ in range(args.reps):
                    t, outs[arm] = run(ctxs[arm], states[arm])
                    best = min(best, t)
                ms[arm].append(best)
        a, b = (np.array(m) for m in ms)
        diff = float(np.linalg.norm(outs[0] - outs[1]) / max(np.linalg.norm(outs[1]), 1e-300))
        print(json.dumps({"workload": name, "A_ms": a.tolist(), "B_ms": b.tolist(),
                          "A_spread": float((a.max() - a.min()) / a.min()), "B_spread": float((b.max() - b.min()) / b.min()),
                          "B_over_A": float(b.min() / a.min()), "rel_diff_outputs": diff}), flush=True)
        del states


if __name__ == "__main__":
    main()
