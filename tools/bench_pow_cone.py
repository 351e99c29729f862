"""Cost of power cones on the B200.

1. cone_pow_kernel on 10^5 and 10^6 cones (tools/bench/pow_cone_bench.cu, built into a temporary directory): kernel time
   and evaluations of psi per cone (max, mean over the cones that need the root).
2. conic_setup of a problem made of 10^5 / 10^6 power cones (all setup kernels, device events).
3. Time per LSQR iteration of config 4 (n = 5000, Zeros(500) + Nonnegatives(4000) + 300 SOC(10)) against the same
   problem with the 3000 SOC rows replaced by 1000 power cones (500 PowerCone, 500 DualPowerCone) and by 1000
   exponential cones: reverse solves at a fixed iteration count (zero tolerances), default driver selection, the three
   problems alternated.

Prints one JSON line per measurement, with the GPU's name and power limit first."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_exp_cone import gpu_info  # noqa: E402


def kernel_bench(nvcc, sizes):
    src = os.path.join(ROOT, "tools", "bench", "pow_cone_bench.cu")
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "pow_cone_bench")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-o", exe, src], check=True)
        for k in sizes:
            out = subprocess.run([exe, str(k), "20"], capture_output=True, text=True, check=True).stdout.strip()
            print(json.dumps(dict(what="cone_pow_kernel", **json.loads(out))), flush=True)


def setup_bench(ctx, sizes):
    cm = __import__("diffopt_b200").submodule("conic")
    rng = np.random.default_rng(1)
    for k in sizes:
        m = 3 * k
        n = 1000
        A = sp.csc_matrix((rng.standard_normal(m), (np.arange(m), rng.integers(0, n, m))), shape=(m, n))
        types = np.where(np.arange(k) % 2 == 0, cm.CONE_POW, cm.CONE_DUAL_POW)
        model = cm.ConicModel(ctx, A, np.zeros(m), np.zeros(n), types, np.full(k, 3), rng.uniform(0.05, 0.95, k))
        model.set_variable_primal(np.zeros(n)); model.set_constraint_primal(np.zeros(m))
        model.set_constraint_dual(rng.standard_normal(m) * 10.0 ** rng.uniform(-3, 2, m))
        times = []
        for _ in range(5):
            model.gradient_cache = False
            model._gradient_cache()
            times.append(model.setup_ms)
        print(json.dumps(dict(what="conic_setup", cones=k, setup_ms_median=float(np.median(times[1:])))), flush=True)


def lsqr_bench(ctx, iters, reps):
    import bench_data
    cm = __import__("diffopt_b200").submodule("conic")
    base = dict(n=5000, n_zero=500, n_nonneg=4000, n_soc=0, nnz_per_row=10, seed=4)
    cases = {
        "config4_soc": bench_data.conic_config4(),
        "config4_exp": bench_data.conic_exp_problem(n_exp=500, n_dual_exp=500, **base),
        "config4_pow": bench_data.conic_exp_problem(n_exp=0, n_dual_exp=0, n_pow=500, n_dual_pow=500, **base),
    }
    models = {}
    for name, d in cases.items():
        mdl = cm.ConicModel(ctx, d["A"], d["b"], d["c"], d["cone_types"], d["cone_dims"], d.get("cone_params"))
        mdl.set_variable_primal(d["x"]); mdl.set_constraint_primal(d["s"]); mdl.set_constraint_dual(d["y"])
        mdl.tolerances = dict(atol=0.0, btol=0.0, conlim=0.0, maxiter=iters)
        mdl.reverse_differentiate(d["seed"])   # warm-up
        models[name] = (mdl, d)
    res = {k: [] for k in models}
    for _ in range(reps):                      # alternate the problems
        for name, (mdl, d) in models.items():
            mdl.reverse_differentiate(d["seed"])
            assert mdl.last_stats["itn"] == iters
            res[name].append(mdl.last_stats["kernel_ms"] / iters * 1e3)
    for name, (mdl, d) in models.items():
        print(json.dumps(dict(what="lsqr_per_iteration", problem=name, m=mdl.m, nnz=int(d["A"].nnz), iterations=iters,
                              us_per_iter_median=float(np.median(res[name])), us_per_iter_min=float(np.min(res[name])),
                              us_per_iter_max=float(np.max(res[name])))), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--sizes", default="100000,1000000")
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--nvcc", default=os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))
    args = ap.parse_args()
    sizes = [int(s) for s in args.sizes.split(",")]
    print(json.dumps(gpu_info()), flush=True)
    kernel_bench(args.nvcc, sizes)
    import diffopt_b200
    ctx = diffopt_b200.Context(0)
    setup_bench(ctx, sizes)
    lsqr_bench(ctx, args.iters, args.reps)


if __name__ == "__main__":
    main()
