"""Batched LSQR branch for LPs (diffopt_b200_qp_batch_solve_lsqr) on the B200, against the single-instance routes.

Workloads (forward direction: dense dq, dh, db; reverse seed: dense), IterativeSolvers' default tolerances:
  (a) 4096 config-1 LPs (n = 200, m = 100, p = 0, 60 active rows), each with its own seed: G staged in shared memory;
  (b) the same with one G for the batch (DIFFOPT_QP_SHARED_MATRICES);
  (c) 4096 LPs with n = 64, m = 64, p = 16, 40 active rows: several CTAs per SM;
  (d) 512 LPs with n = 400, m = 200, p = 8, 120 active rows: G read from global memory.
Per workload: device time of the call (CUDA events, median of the repetitions, inputs in device memory), solves/s
(a forward and a reverse solve count as two), mean and max iterations per mode, and FP64 FLOP/s from the counted
4 (m + p) n FMAs per solve-iteration (2 FLOP each) against the repository's measured DGEMM rate (35.69 TFLOP/s).
Baselines in the same run: QPModel single calls (lsqr_csc on the host-built KKT CSC) on 64 config-1 instances, and scipy's
lsqr on the CPU on 16 config-1 instances, both extrapolated to 4096 and labelled as such.

Prints one JSON line per measurement, with the GPU's name and power limit first."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_exp_cone import gpu_info  # noqa: E402

DGEMM_TFLOPS = 35.69


def lp_batch(B, n, m, p, n_active, seed0, shared=False):
    """B LPs, instance b drawn from default_rng(seed0 + b) (shared: G, A from seed0 for all); logical arrays."""
    G = np.empty((1 if shared else B, m, n))
    A = np.empty((1 if shared else B, p, n))
    d = {k: np.empty(s) for k, s in dict(h=(B, m), z=(B, n), lam=(B, m), nu=(B, p), dq=(B, n), dh=(B, m), db=(B, p),
                                         seed=(B, n)).items()}
    for b in range(B):
        rng = np.random.default_rng(seed0 + b)
        if b == 0 or not shared:
            G[b] = rng.standard_normal((m, n))
            A[b] = rng.standard_normal((p, n))
        z = rng.standard_normal(n)
        act = rng.permutation(m)[:n_active]
        lam = np.zeros(m)
        lam[act] = rng.uniform(0.5, 1.5, size=act.size)
        slack = -rng.uniform(0.5, 1.5, size=m)
        slack[act] = 0.0
        g = G[0 if shared else b]
        d["z"][b], d["lam"][b], d["h"][b], d["nu"][b] = z, lam, g @ z - slack, rng.standard_normal(p)
        d["dq"][b], d["dh"][b], d["db"][b], d["seed"][b] = (rng.standard_normal(n), rng.standard_normal(m),
                                                            rng.standard_normal(p), rng.standard_normal(n))
    d["G"], d["A"] = G, A
    return d


def run_batch(ctx, qpm, capi, torch, d, n, m, p, shared, reps):
    B = d["z"].shape[0]
    N = n + m + p
    Bm = 1 if shared else B
    cm = lambda X, r: torch.from_numpy(qpm.colmajor(X, r, n, Bm)).cuda() if r else None
    t = lambda v, k: torch.from_numpy(np.ascontiguousarray(v)).cuda() if k else None
    args = [cm(d["G"], m), cm(d["A"], p), t(d["h"], m), t(d["z"], n), t(d["lam"], m), t(d["nu"], p), None, t(d["dq"], n),
            None, t(d["dh"], m), None, t(d["db"], p), t(d["seed"], n)]
    fwd = torch.empty((B, N), dtype=torch.float64, device="cuda")
    rev = torch.empty_like(fwd)
    st = torch.empty((B, 2, 4), dtype=torch.float64, device="cuda")
    from oracle.lsqr import SQRT_EPS
    ms = []
    for r in range(reps + 1):
        rc = ctx.lib.diffopt_b200_qp_batch_solve_lsqr(ctx.h, B, n, m, p, *[capi.ptr(x) for x in args], SQRT_EPS, SQRT_EPS,
                                                      1 / SQRT_EPS, 0, capi.ptr(fwd), capi.ptr(rev), capi.ptr(st),
                                                      capi.DEVICE, capi.QP_SHARED_MATRICES if shared else 0)
        ctx.check(rc)
        if r:  # the first call is the warm-up
            ms.append(ctx.last_kernel_ms)
    s = st.cpu().numpy()
    itn = s[:, :, 1]
    med = float(np.median(ms))
    fma = 4.0 * (m + p) * n * itn.sum()          # counted FMAs of the operator passes over G and A, both modes
    return dict(B=B, n=n, m=m, p=p, shared=shared, device_ms_median=med, device_ms_min=float(min(ms)), reps=reps,
                solves_per_s=2 * B / (med * 1e-3), us_per_instance=med * 1e3 / B,
                itn_fwd_mean=float(itn[:, 0].mean()), itn_fwd_max=int(itn[:, 0].max()),
                itn_rev_mean=float(itn[:, 1].mean()), itn_rev_max=int(itn[:, 1].max()),
                istop_counts={str(int(k)): int(v) for k, v in zip(*np.unique(s[:, :, 0], return_counts=True))},
                fp64_tflops=2 * fma / (med * 1e-3) / 1e12,
                fp64_share_of_dgemm=2 * fma / (med * 1e-3) / 1e12 / DGEMM_TFLOPS), fwd.cpu().numpy(), rev.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch

    import diffopt_b200
    from oracle import qp as oqp
    qpm = diffopt_b200.submodule("qp")
    capi = diffopt_b200.submodule("_capi")
    ctx = diffopt_b200.Context(0)
    lines = [dict(what="device", **gpu_info())]

    def emit(rec):
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    print(json.dumps(lines[0]), flush=True)

    cases = [("a_config1", 4096, (200, 100, 0, 60), False), ("b_config1_shared", 4096, (200, 100, 0, 60), True),
             ("c_64_64_16", 4096, (64, 64, 16, 40), False), ("d_400_200_8_global", 512, (400, 200, 8, 120), False)]
    d1 = None
    for name, B, (n, m, p, na), shared in cases:
        d = lp_batch(B, n, m, p, na, seed0=1, shared=shared)
        rec, fwd, rev = run_batch(ctx, qpm, capi, torch, d, n, m, p, shared, args.reps)
        # spot check against the oracle on the first instance (same default tolerances)
        g = d["G"][0]
        a = d["A"][0]
        Q = np.zeros((n, n))
        of = np.concatenate(oqp.forward(Q, g, d["h"][0], a, d["z"][0], d["lam"][0], d["nu"][0], np.zeros((n, n)),
                                        d["dq"][0], np.zeros((m, n)), d["dh"][0], np.zeros((p, n)), d["db"][0]))
        orv = np.concatenate(oqp.reverse(Q, g, d["h"][0], a, d["z"][0], d["lam"][0], d["nu"][0], d["seed"][0]))
        rec["rel_err_inst0"] = max(np.linalg.norm(fwd[0] - of) / np.linalg.norm(of),
                                   np.linalg.norm(rev[0] - orv) / np.linalg.norm(orv))
        emit(dict(what=name, **rec))
        if name == "a_config1":
            d1, rec1 = d, rec

    # baselines on config 1: QPModel single calls (GPU lsqr_csc, host-built CSC) and scipy lsqr on the CPU
    n, m = 200, 100
    dev_ms, wall = 0.0, 0.0
    K0 = 64
    for b in range(K0 + 1):
        model = qpm.QPModel(ctx, np.zeros((n, n)), np.zeros(n), d1["G"][b], d1["h"][b], np.zeros((0, n)), np.zeros(0))
        model.set_variable_primal(d1["z"][b]); model.set_constraint_dual_le(-d1["lam"][b]); model.set_constraint_dual_eq([])
        t0 = time.perf_counter()
        model.forward_differentiate(dq=d1["dq"][b], dh=d1["dh"][b])
        k1 = ctx.last_kernel_ms
        model.reverse_differentiate(d1["seed"][b])
        k2 = ctx.last_kernel_ms
        t1 = time.perf_counter()
        if b:  # instance 0 is the warm-up
            dev_ms += k1 + k2
            wall += (t1 - t0) * 1e3
    emit(dict(what="baseline_qpmodel_single_calls_config1", instances=K0, device_ms_per_instance=dev_ms / K0,
              wall_ms_per_instance=wall / K0, extrapolated_device_ms_4096=dev_ms / K0 * 4096,
              extrapolated_wall_ms_4096=wall / K0 * 4096,
              batch_speedup_device_time=dev_ms / K0 * 4096 / rec1["device_ms_median"], note="extrapolated from 64 calls"))
    import scipy.sparse.linalg as spla
    from oracle.lsqr import SQRT_EPS
    K1 = 16
    t0 = time.perf_counter()
    for b in range(K1):
        K = oqp.create_lhs(d1["z"][b], d1["lam"][b], np.zeros((n, n)), d1["G"][b], d1["h"][b], np.zeros((0, n)))
        rhs = np.zeros(n + m); rhs[:n] = d1["seed"][b]
        rf = oqp.forward_rhs(d1["z"][b], d1["lam"][b], np.zeros(0), np.zeros((n, n)), d1["dq"][b], np.zeros((m, n)),
                             d1["dh"][b], np.zeros((0, n)), np.zeros(0))
        for M, r in ((K, rhs), (K.T, rf)):
            spla.lsqr(M, r, atol=SQRT_EPS, btol=SQRT_EPS, conlim=1 / SQRT_EPS, iter_lim=n + m)
    cpu_ms = (time.perf_counter() - t0) * 1e3 / K1
    emit(dict(what="baseline_scipy_lsqr_cpu_config1", instances=K1, ms_per_instance=cpu_ms,
              extrapolated_ms_4096=cpu_ms * 4096, batch_speedup=cpu_ms * 4096 / rec1["device_ms_median"],
              note="extrapolated from 16 instances, one host thread per call"))
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
