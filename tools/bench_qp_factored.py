"""k sensitivity directions of one batched QP on the B200: refactorise per direction, or factorise once.

Device-resident batches of 4096 instances (n/m/p = 64/64/16, 32/32/8, 100/50/0; bench_data.qp_batch_fast, 16 / 8 / 10
active rows) and, for k in {1, 8, 64}, two ways to get k forward directions (sparse triplets: 2 symmetric pairs in dQ,
4 entries in dG, 2 in dA, dense dq, dh, db) and k reverse seeds, alternated in the same run:
  (a) k stream-ordered qp_batch_solve_coo calls (DIFFOPT_QP_ASYNC), each one direction and one seed, then synchronize --
      what a caller does without the stored factor;
  (b) qp_batch_factorize + qp_batch_forward_multi(k) + qp_batch_reverse_multi(k) (blocking calls).
Reported per (shape, k): device time between CUDA events on the ctx stream (median of the repetitions), microseconds per
direction (a forward direction and a reverse seed count as one), the algorithmic bytes and flops of (b) with their shares of
the measured HBM bandwidth (6541.8 GB/s) and FP64 DGEMM peak (35.69 TFLOP/s), and the largest relative difference between
(a) and (b) over every (instance, direction).  Flops of (b): the factorisation nred^3/3 plus 4 nred^2 per right-hand side
(two triangular sweeps), per instance.  Bytes of (b): problem data read and factor written once, the factor read by each
multi call, right-hand sides (the assembled forward ones written and read), seeds, triplets and outputs.

Prints one JSON line per measurement, with the GPU's name and power limit first."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_exp_cone import gpu_info  # noqa: E402

HBM_GBS, DGEMM_TFLOPS = 6541.8, 35.69


def triplets(rng, S, rows, n, nnz, sym):
    """nnz entries per slot (sym: nnz/2 symmetric pairs), 0-based offsets, 1-based (I, J)"""
    if sym:
        i = rng.integers(0, rows, (S, nnz // 2))
        j = rng.integers(0, n, (S, nnz // 2))
        v = rng.standard_normal((S, nnz // 2))
        I, J, V = np.concatenate([i, j], 1), np.concatenate([j, i], 1), np.concatenate([v, v], 1) / 2
    else:
        I, J, V = rng.integers(0, rows, (S, nnz)), rng.integers(0, n, (S, nnz)), rng.standard_normal((S, nnz))
    return dict(nnz=nnz, I=I + 1, J=J + 1, V=V)


def oracle_slice(d, trip, dq, dh, db, seeds, B, k, n, m, p, sel, kk):
    """CPU oracle for the instances `sel`, directions 0 .. kk-1"""
    from oracle import qp as oqp
    N = n + m + p
    fwd, rev = np.empty((len(sel), kk, N)), np.empty((len(sel), kk, N))
    for a, b in enumerate(sel):
        for j in range(kk):
            s = b * k + j
            mats = {}
            for key, rows in (("dQ", n), ("dG", m), ("dA", p)):
                M = np.zeros((rows, n))
                t = trip[key]
                if t is not None:
                    np.add.at(M, (t["I"][s] - 1, t["J"][s] - 1), t["V"][s])
                mats[key] = M
            f, r = oqp.batch_forward_reverse(d["Q"][b:b + 1], d["G"][b:b + 1], d["A"][b:b + 1], d["h"][b:b + 1], d["z"][b:b + 1],
                                             d["lam"][b:b + 1], d["nu"][b:b + 1], seeds[b:b + 1, j], mats["dQ"][None], dq[b:b + 1, j],
                                             mats["dG"][None], dh[b:b + 1, j], mats["dA"][None], db[b:b + 1, j])
            fwd[a, j], rev[a, j] = f[0], r[0]
    return dict(sel=sel, kk=kk, fwd=fwd, rev=rev)


def run_shape(ctx, torch, n, m, p, na, B, ks, reps):
    import bench_data
    qpm = __import__("diffopt_b200").submodule("qp")
    capi = __import__("diffopt_b200").submodule("_capi")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.ExternalStream(ctx.stream)
    d = bench_data.qp_batch_fast(B, n, m, p, n_active=na, seed=7)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    Qc, Gc, Ac = T(qpm.colmajor(d["Q"], n, n, B)), T(qpm.colmajor(d["G"], m, n, B)) if m else None, \
        T(qpm.colmajor(d["A"], p, n, B)) if p else None
    h, z, lam, nu = T(d["h"]), T(d["z"]), T(d["lam"]), T(d["nu"])
    ptr = lambda t: None if t is None or t.numel() == 0 else capi.ptr(t)
    ctx.check(ctx.lib.diffopt_b200_qp_batch_setup(ctx.h, B, n, m, p, ptr(Qc), ptr(Gc), ptr(Ac), ptr(h), ptr(z), ptr(lam), ptr(nu),
                                                  capi.DEVICE))
    N = n + m + p
    nred = ((n + 7) // 8) * 8 + na + p
    nt = (nred + 7) // 8
    factor_bytes = 8 * (nt * (nt + 1) // 2 * 64 + 8 * nt + m) + 4 * (m + 1)
    problem_bytes = 8 * (n * n + m * n + p * n + 2 * m + n + p)
    for k in ks:
        rng = np.random.default_rng(k)
        S = B * k
        trip = {"dQ": triplets(rng, S, n, n, 4, True), "dG": triplets(rng, S, m, n, 4, False) if m else None,
                "dA": triplets(rng, S, p, n, 2, False) if p else None}
        dq, dh, db = rng.standard_normal((B, k, n)), rng.standard_normal((B, k, m)), rng.standard_normal((B, k, p))
        seeds = rng.standard_normal((B, k, n))
        keep = []

        def coo(t, sel=None):
            if t is None:
                return None
            I, J, V = (t[x] if sel is None else t[x].reshape(B, k, -1)[:, sel] for x in ("I", "J", "V"))
            slots = S if sel is None else B
            arrs = [T(np.arange(slots + 1, dtype=np.int64) * t["nnz"]), T(I.reshape(-1).astype(np.int64)),
                    T(J.reshape(-1).astype(np.int64)), T(V.reshape(-1))]
            st = capi.CooBatch(*[a.data_ptr() for a in arrs])
            keep.append((arrs, st))
            return capi.C.addressof(st)
        def dev_ptr(a):   # device copy kept alive for the whole measurement
            t = T(a)
            keep.append(t)
            return ptr(t)
        # (b): all k directions of an instance in one call
        b_args = [coo(trip["dQ"]), dev_ptr(dq), coo(trip["dG"]), dev_ptr(dh), coo(trip["dA"]), dev_ptr(db)]
        sd = T(seeds)
        fb, rb = torch.empty((B, k, N), dtype=torch.float64, device=dev), torch.empty((B, k, N), dtype=torch.float64, device=dev)
        # (a): direction j of every instance as its own batch
        a_args = [[coo(trip["dQ"], j), dev_ptr(dq[:, j]), coo(trip["dG"], j), dev_ptr(dh[:, j]), coo(trip["dA"], j), dev_ptr(db[:, j]),
                   dev_ptr(seeds[:, j])] for j in range(k)]
        fa = [torch.empty((B, N), dtype=torch.float64, device=dev) for _ in range(k)]
        ra = [torch.empty((B, N), dtype=torch.float64, device=dev) for _ in range(k)]
        prob = [ptr(Qc), ptr(Gc), ptr(Ac), ptr(h), ptr(z), ptr(lam), ptr(nu)]

        def way_a():
            for j in range(k):
                ctx.check(ctx.lib.diffopt_b200_qp_batch_solve_coo(ctx.h, B, n, m, p, *prob, *a_args[j], ptr(fa[j]), ptr(ra[j]), None,
                                                                  capi.DEVICE, capi.QP_ASYNC))
            assert ctx.lib.diffopt_b200_synchronize(ctx.h) == 0

        def way_b():
            assert ctx.lib.diffopt_b200_qp_batch_factorize(ctx.h, None, capi.DEVICE) == 0
            assert ctx.lib.diffopt_b200_qp_batch_forward_multi(ctx.h, k, *b_args, ptr(fb), capi.DEVICE) == 0
            assert ctx.lib.diffopt_b200_qp_batch_reverse_multi(ctx.h, k, ptr(sd), ptr(rb), capi.DEVICE) == 0

        times = {"a": [], "b": []}
        for rep in range(reps + 2):   # two warm-up rounds
            for name, fn in (("a", way_a), ("b", way_b)):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                e1.synchronize()
                if rep >= 2:
                    times[name].append(e0.elapsed_time(e1))
        fa_s, ra_s = torch.stack(fa, 1), torch.stack(ra, 1)
        rel = lambda x, y: float((torch.linalg.vector_norm(x - y, dim=-1) / torch.linalg.vector_norm(y, dim=-1)).max())
        orc = oracle_slice(d, trip, dq, dh, db, seeds, B, k, n, m, p, [0, 1, B // 2, B - 1], min(k, 2))
        chk = {f"oracle_{w}_{x}": rel(y[orc["sel"]][:, :orc["kk"]].cpu(), torch.from_numpy(orc[x]))
               for w, (yf, yr) in (("a", (fa_s, ra_s)), ("b", (fb, rb))) for x, y in (("fwd", yf), ("rev", yr))}
        ta, tb = float(np.median(times["a"])), float(np.median(times["b"]))
        nnz = sum(t["nnz"] for t in trip.values() if t is not None)
        # factor written once and read by both multi calls; forward: triplets, dq/dh/db, assembled rhs written and read,
        # output; reverse: G once, seeds, output
        bytes_b = (problem_bytes + 3 * factor_bytes + 8 * m * n + k * (24 * nnz + 8 * (n + m + p) + 3 * 8 * N + 8 * n + 8 * N)) * B
        flops_b = (nred ** 3 / 3 + 2 * 4 * nred ** 2 * k) * B
        print(json.dumps(dict(
            what="qp_factored_vs_refactorise", shape=f"{n}/{m}/{p}", active=na, B=B, k=k, reps=reps,
            a_ms=round(ta, 4), b_ms=round(tb, 4), a_us_per_direction=round(1e3 * ta / k, 3), b_us_per_direction=round(1e3 * tb / k, 3),
            speedup=round(ta / tb, 3), b_bytes=int(bytes_b), b_flops=int(flops_b),
            b_hbm_share=round(bytes_b / (tb * 1e-3) / (HBM_GBS * 1e9), 4), b_dgemm_share=round(flops_b / (tb * 1e-3) / (DGEMM_TFLOPS * 1e12), 4),
            factor_mb=round(factor_bytes * B / 1e6, 1),
            max_rel_diff_fwd=rel(fb, fa_s), max_rel_diff_rev=rel(rb, ra_s), **chk)), flush=True)
        del fa, ra, fb, rb, keep
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--ks", default="1,8,64")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shapes", default="64/64/16/16,32/32/8/8,100/50/0/10")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_qp_factored: needs a CUDA device")
    print(json.dumps(dict(what="gpu", **gpu_info())), flush=True)
    ctx = __import__("diffopt_b200").Context(0)
    ks = [int(x) for x in args.ks.split(",")]
    for sh in args.shapes.split(","):
        n, m, p, na = (int(x) for x in sh.split("/"))
        run_shape(ctx, torch, n, m, p, na, args.B, ks, args.reps)


if __name__ == "__main__":
    main()
