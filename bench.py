#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 sensitivity hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (config 2 of BASELINE.json): a batch of 4096 dense random QPs, n=64, m_eq=16,
m_ineq=64 (KKT order N=144).  One *solve* = KKT assembly + one LU factorisation + one forward
(LHS') and one reverse (LHS) sensitivity solve for one instance; one *step* = one pass over the
batch.  With N GPUs the SAME 4096 instances are split into contiguous shards, one per rank (strong
scaling, no data-path collective; `weak` carries the 4096-per-rank companion number, `shared_variant`
the OptNet-shared form with its NCCL all-reduce).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (the tree may be read-only)

N_VAR, M_INEQ, P_EQ = 64, 64, 16
KKT_N = N_VAR + M_INEQ + P_EQ
FLOP_PER_SOLVE = 2 * KKT_N**3 // 3 + 2 * (2 * KKT_N**2)          # 2 073 600 (SURVEY.md §8d)
BYTES_PER_SOLVE = 8 * ((N_VAR**2 + M_INEQ * N_VAR + P_EQ * N_VAR + N_VAR + 2 * M_INEQ + P_EQ) * 2 - M_INEQ
                       + N_VAR + 2 * KKT_N)                        # ~153 KB: inputs + direction + seed + outputs
METRIC = "KKT sensitivity solves/sec (4096xQP n=64)"
FIELDS = ["Q", "G", "A", "h", "z", "lam", "nu", "dQ", "dq", "dG", "dh", "dA", "db", "seed"]
SHAPES = dict(Q=(N_VAR, N_VAR), G=(M_INEQ, N_VAR), A=(P_EQ, N_VAR), dQ=(N_VAR, N_VAR), dG=(M_INEQ, N_VAR),
              dA=(P_EQ, N_VAR))


def host_buffers(B, seed, pinned_alloc=None):
    """Instance-major, column-major-per-instance fp64 buffers exactly as the C ABI takes them."""
    import bench_data
    d = bench_data.qp_batch_fast(B, N_VAR, M_INEQ, P_EQ, seed=seed)
    out = {}
    for k in FIELDS:
        a = d[k]
        if k in SHAPES:
            a = a.transpose(0, 2, 1)
        if pinned_alloc is not None:
            buf = pinned_alloc(a.shape)
            np.copyto(buf, a)
            out[k] = buf
        else:
            out[k] = np.ascontiguousarray(a)
    return out, d


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout=2.0):
        """Block until nvidia-smi has produced its first line (so that the timed region is actually sampled)."""
        t_end = time.perf_counter() + timeout
        while self.proc is not None and not self.rows and time.perf_counter() < t_end:
            time.sleep(0.01)

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def fp64_peaks():
    """Runs tools/fp64_peak (cuBLAS DGEMM 8192^3 + raw DMMA/DFMA issue rates) on this GPU."""
    tool = os.path.join(ROOT, "tools", "fp64_peak")
    try:
        out = subprocess.run([tool], capture_output=True, text=True, timeout=120).stdout.strip().splitlines()[-1]
        return json.loads(out)
    except Exception as e:  # pragma: no cover
        return {"error": str(e)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on host cores (oracle port; Julia/UMFPACK are not in the image)

def _kkt_pattern():
    """CSC index arrays of LHS = [Q G'L A'; G D 0; A 0 0] for dense blocks (identical for every instance): the
    reference holds LHS as a SparseMatrixCSC built once per problem by sparse hcat/vcat (QuadraticProgram.jl:256-282);
    here only the value vector is assembled per instance, never a dense N x N detour."""
    n, m, p = N_VAR, M_INEQ, P_EQ
    N = n + m + p
    mask = np.zeros((N, N), dtype=bool)
    mask[:n, :n] = True; mask[:n, n:n + m] = True; mask[:n, n + m:] = True
    mask[n:n + m, :n] = True; mask[n + m:, :n] = True
    mask[np.arange(n, n + m), np.arange(n, n + m)] = True
    import scipy.sparse as sp
    P = sp.csc_matrix(mask.astype(np.float64))
    P.sort_indices()
    PT = sp.csc_matrix(mask.T.astype(np.float64))
    PT.sort_indices()
    return P.indices.copy(), P.indptr.copy(), PT.indices.copy(), PT.indptr.copy(), mask


_PATTERN = None


def _cpu_chunk(args):
    r"""Per-instance work of one worker.  variant:
    'faithful'    -- what the reference does: LHS assembled once as CSC (_gradient_cache), then one sparse LU factorisation
                     PER differentiate call: `LHS' \ RHS` in forward_differentiate! (:438) and `LHS \ RHS` in
                     reverse_differentiate! (:335);
    'factor_once' -- one sparse LU of LHS serving both solves (what a caching reimplementation would do);
    'dense'       -- LAPACK getrf once + two getrs on the dense 144 x 144 matrix (strongest simple CPU variant)."""
    import scipy.linalg as sla
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    from oracle import qp as oqp
    global _PATTERN
    lo, hi, variant = args
    d = _CPU_DATA
    n = N_VAR
    if _PATTERN is None:
        _PATTERN = _kkt_pattern()
    ind, ptr, indT, ptrT, mask = _PATTERN
    for b in range(lo, hi):
        Kd = oqp.create_lhs(d["z"][b], d["lam"][b], d["Q"][b], d["G"][b], d["h"][b], d["A"][b])
        rf = oqp.forward_rhs(d["z"][b], d["lam"][b], d["nu"][b], d["dQ"][b], d["dq"][b], d["dG"][b], d["dh"][b],
                             d["dA"][b], d["db"][b])
        rb = np.zeros(KKT_N)
        rb[:n] = d["seed"][b]
        if variant == "dense":
            lu = sla.lu_factor(Kd, check_finite=False)
            sla.lu_solve(lu, rf, trans=1, check_finite=False)
            sla.lu_solve(lu, rb, check_finite=False)
            continue
        K = sp.csc_matrix((Kd.T[mask.T], ind, ptr), shape=Kd.shape)       # values in CSC order of the fixed pattern
        if variant == "factor_once":
            lu = spla.splu(K)
            lu.solve(rf, trans="T")
            lu.solve(rb)
        else:
            KT = sp.csc_matrix((Kd[mask], indT, ptrT), shape=Kd.shape)
            spla.splu(KT).solve(rf)      # forward_differentiate!: LHS' \ RHS
            spla.splu(K).solve(rb)       # reverse_differentiate!: LHS \ RHS
    return hi - lo


_CPU_DATA = None


def cpu_reference_rate(d, sample, procs, variant="faithful"):
    """solves/s of the CPU port on `sample` instances using `procs` single-threaded worker processes (fork: the workers
    inherit the inputs, nothing is pickled inside the timed region; BLAS/OpenMP pinned to one thread per worker so the
    pool is not oversubscribed)."""
    import multiprocessing as mp
    global _CPU_DATA
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    _CPU_DATA = {k: v[:sample] for k, v in d.items()}
    bounds = np.linspace(0, sample, procs + 1).astype(int)
    chunks = [(int(bounds[i]), int(bounds[i + 1]), variant) for i in range(procs) if bounds[i + 1] > bounds[i]]
    if procs == 1:
        _cpu_chunk((0, min(4, sample), variant))
        t0 = time.perf_counter()
        _cpu_chunk(chunks[0])
        return sample / (time.perf_counter() - t0)
    with mp.get_context("fork").Pool(procs) as pool:
        pool.map(_cpu_chunk, [(0, min(4, sample), variant)] * procs)  # warm the workers (imports)
        t0 = time.perf_counter()
        pool.map(_cpu_chunk, chunks)
        dt = time.perf_counter() - t0
    return sample / dt


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


CPU_SAMPLE_TXT = ("all {sample} instances of the step; per instance the reference's work: LHS assembled once as CSC, then one "
                  "sparse LU factorisation + solve for forward_differentiate! (LHS') and another for reverse_differentiate! "
                  "(LHS), QuadraticProgram.jl:335,438; SuperLU (scipy) stands in for UMFPACK; {procs} single-threaded worker "
                  "processes (OMP/OPENBLAS/MKL threads = 1)")


def cpu_baseline_block(d, sample, procs):
    rate = cpu_reference_rate(d, sample, procs, "faithful")
    once = cpu_reference_rate(d, sample, procs, "factor_once")
    dense = cpu_reference_rate(d, sample, procs, "dense")
    return {"value": rate, "unit": "solves/s", "cores": procs, "kind": "port",
            "sample": CPU_SAMPLE_TXT.format(sample=sample, procs=procs), "same_config": sample == 4096,
            "variants": {"reference_faithful_two_sparse_lu_per_instance": rate,
                         "factor_once_sparse_lu": once, "dense_lapack_getrf_getrs": dense}}


def run_reference(args, rank, world):
    if rank != 0:
        return
    import bench_data
    procs = host_cores()
    sample = int(os.environ.get("DIFFOPT_BENCH_CPU_SAMPLE", 4096))
    d = bench_data.qp_batch_fast(sample, N_VAR, M_INEQ, P_EQ, seed=2026)
    for _ in range(args.warmup):
        cpu_reference_rate(d, min(sample, 16 * procs), procs)
    dt = 0.0
    done = 0
    steps = args.steps   # each step is the full 4096-instance batch (~0.2 s on 32 cores)
    for _ in range(steps):
        dt += sample / cpu_reference_rate(d, sample, procs)   # times the worker map only, not pool start-up
        done += sample
    val = done / dt
    base = cpu_baseline_block(d, sample, procs)
    base["value"] = val
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "solves/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps * (4096 / sample),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "4096 x dense QP n=64 m_ineq=64 m_eq=16 (KKT N=144), forward + reverse "
                                   "sensitivities (BASELINE.json configs[1]); CPU arm: the reference's algorithm on the "
                                   "host cores of rank 0", "global_batch": 4096},
            "cpu_baseline": base,
            "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(local_rank):
    """Pins this process (and therefore the pinned host buffers it allocates next: first touch) to the CPUs of the NUMA
    node the GPU hangs off.  Without it every rank of a multi-GPU run stages through node 0 (r1: e2e efficiency 0.43 at 8
    GPUs).  Returns a description for the JSON line."""
    try:
        q = subprocess.run(["nvidia-smi", f"--id={local_rank}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = q[-12:] if len(q) >= 12 else q           # 00000000:1b:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": node, "bound": False}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"numa_node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "bound": True, "cpus": len(cpus)}
    except Exception as e:  # pragma: no cover
        return {"bound": False, "why": str(e)[:80]}


DUMP_LIMIT_BYTES = 60_000_000   # array data; the files stay under 64 MB with their .npy headers


def dump_outputs(out_dir, arrays, rank, world):
    """Writes what the timed call returned in its last step, every rank's shard in instance order, as
    out_dir/<name>.npy in float64: the inputs are seeded, so two builds can be compared output for output.  Above
    DUMP_LIMIT_BYTES in all, a fixed seeded sample of instances is kept and their indices go to instance.npy."""
    import torch.distributed as dist
    host = {k: v.cpu().numpy().astype(np.float64) for k, v in arrays.items()}
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, host)
        host = {k: np.concatenate([p[k] for p in parts]) for k in host}
    if rank != 0:
        return
    B = len(host["fwd"])
    row_bytes = sum(v[0].nbytes for v in host.values())
    if B * row_bytes > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_LIMIT_BYTES // (row_bytes + 8), replace=False))
        host = {k: v[keep] for k, v in host.items()}
        host["instance"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def run_b200(args, rank, world, local_rank):
    numa = bind_to_gpu_numa_node(local_rank)
    import torch
    import torch.distributed as dist

    import diffopt_b200
    capi = diffopt_b200.submodule("_capi")
    sharding = diffopt_b200.submodule("sharding")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = diffopt_b200.Context(local_rank)
    lib = ctx.lib
    BT = args.batch                                   # the whole job: 4096 instances
    lo, hi = sharding.shard_range(BT, rank, world)    # strong scaling: this rank's contiguous shard
    B = hi - lo
    N = KKT_N

    # every rank generates the full batch (same seed) and keeps its shard: the job is the SAME 4096 problems at any N
    hb_full, logical_full = host_buffers(BT, seed=2026)
    logical = {k: v[lo:hi] for k, v in logical_full.items()}
    hb = {}
    for k in FIELDS:
        buf = capi.pinned_empty(hb_full[k][lo:hi].shape)
        np.copyto(buf, hb_full[k][lo:hi])
        hb[k] = buf
    db = {k: torch.from_numpy(v).to(dev) for k, v in hb.items()}     # resident inputs (torch = device memory)
    fwd = torch.empty((B, N), dtype=torch.float64, device=dev)
    rev = torch.empty((B, N), dtype=torch.float64, device=dev)
    info = torch.zeros(B, dtype=torch.int32, device=dev)
    fwd_h = capi.pinned_empty((B, N))
    rev_h = capi.pinned_empty((B, N))
    info_h = np.zeros(B, dtype=np.int32)
    in_bytes = sum(v.nbytes for v in hb.values())
    out_bytes = fwd_h.nbytes + rev_h.nbytes + info_h.nbytes

    def dptr(t):
        return capi.vp(t.data_ptr())

    def check(rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} rc={rc}: {lib.diffopt_b200_last_error(ctx.h).decode()}")

    dev_args = [dptr(db[k]) for k in FIELDS] + [dptr(fwd), dptr(rev), dptr(info)]

    def step_device():
        # stream-ordered form of the call (device-resident inputs): batches run back to back on the ctx stream, the
        # status of every queued call is collected by diffopt_b200_synchronize after the timed region
        check(lib.diffopt_b200_qp_batch_solve_async(ctx.h, B, N_VAR, M_INEQ, P_EQ, *dev_args), "qp_batch_solve_async")

    def step_device_blocking():
        check(lib.diffopt_b200_qp_batch_solve(ctx.h, B, N_VAR, M_INEQ, P_EQ, *dev_args, capi.DEVICE), "qp_batch_solve")

    def finish_device():
        check(lib.diffopt_b200_synchronize(ctx.h), "diffopt_b200_synchronize")

    def step_e2e():
        check(lib.diffopt_b200_qp_batch_solve(
            ctx.h, B, N_VAR, M_INEQ, P_EQ, *[capi.ptr(hb[k]) for k in FIELDS], capi.ptr(fwd_h), capi.ptr(rev_h),
            capi.ptr(info_h), capi.HOST), "qp_batch_solve(host)")

    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, finish=None):
        """CUDA events on the library's own stream, barrier + synchronize on both sides, max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kms = 0.0
        barrier()
        e0.record(stream)
        for _ in range(steps):
            fn()
            kms += ctx.last_kernel_ms
        e1.record(stream)
        barrier()
        if finish:
            finish()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, kms / steps

    sampler = ClockSampler(local_rank) if rank == 0 else None   # started early: nvidia-smi needs ~0.2 s to come up
    for _ in range(max(args.warmup, 3)):
        step_device()
    finish_device()
    if sampler:
        sampler.wait_first()
    l0 = ctx.launch_count
    t0 = time.perf_counter()
    ms, _ = timed(step_device, args.steps, finish_device)
    t1 = time.perf_counter()
    launches = ctx.launch_count - l0
    clocks = sampler.stop(t0, t1) if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"fwd": fwd, "rev": rev, "info": info}, rank, world)
    kernel_ms = ms / args.steps   # device time per launch: the timed region holds nothing but the K launches
    # the blocking form of the same call (what the reference-facing API does): a few calls, for the record
    step_device_blocking()
    ms_blocking, call_kernel_ms = timed(step_device_blocking, 5)

    # parity spot-check of what was just timed (oracle as checker only)
    from oracle import qp as oqp
    sl = slice(0, min(8, B))
    of, orv = oqp.batch_forward_reverse(*[logical[k][sl] for k in ["Q", "G", "A", "h", "z", "lam", "nu", "seed",
                                                                   "dQ", "dq", "dG", "dh", "dA", "db"]])
    gf, gr = fwd[sl].cpu().numpy(), rev[sl].cpu().numpy()
    err = max((np.linalg.norm(gf - of, axis=1) / np.linalg.norm(of, axis=1)).max(),
              (np.linalg.norm(gr - orv, axis=1) / np.linalg.norm(orv, axis=1)).max())
    if not err <= 1e-8:
        raise RuntimeError(f"parity check failed inside bench (rank {rank}): rel err {err:.3e}")

    # end-to-end through the C ABI with host (pinned) buffers: H2D + kernel + D2H every step
    for _ in range(2):
        step_e2e()
    e2e_steps = max(2, min(args.steps, 10))
    ms_e2e, _ = timed(step_e2e, e2e_steps)
    e2e_variants = e2e_byte_variants(args, ctx, lib, capi, hb, logical, B, BT, world, timed, check, fwd_h, rev_h, info_h, e2e_steps)

    # weak-scaling companion number (second field): every rank a full 4096-instance batch of its own
    weak = None
    if world > 1:
        dbw = {k: torch.from_numpy(np.ascontiguousarray(hb_full[k])).to(dev) for k in FIELDS}
        fw = torch.empty((BT, N), dtype=torch.float64, device=dev)
        rw = torch.empty((BT, N), dtype=torch.float64, device=dev)
        iw = torch.zeros(BT, dtype=torch.int32, device=dev)
        wargs = [dptr(dbw[k]) for k in FIELDS] + [dptr(fw), dptr(rw), dptr(iw)]

        def step_weak():
            check(lib.diffopt_b200_qp_batch_solve_async(ctx.h, BT, N_VAR, M_INEQ, P_EQ, *wargs), "qp_batch_solve_async")
        for _ in range(3):
            step_weak()
        finish_device()
        wsteps = min(args.steps, 50)
        ms_w, _ = timed(step_weak, wsteps, finish_device)
        weak = {"value": world * BT * wsteps / (ms_w * 1e-3), "unit": "solves/s", "ms_per_step": ms_w / wsteps,
                "batch_per_gpu": BT, "scaling": "weak"}
        del dbw, fw, rw, iw

    shared = shared_variant(args, rank, world, ctx, lib, capi, sharding, dev, db, logical, B, BT, timed, check, dptr)
    aux = active_set_sweep(args, ctx, lib, capi, dev, timed, check, dptr) if world == 1 and not args.no_aux else None
    if aux is not None:
        # second half of the BASELINE.json metric ("sparse solve ms"): config 3, one sparse KKT system with 256 right-hand sides
        import bench_aux
        try:
            aux["other_shapes"] = other_shapes_sweep(ctx, lib, capi, dev, timed, check, dptr)
        except Exception as e:
            aux["other_shapes"] = {"error": str(e)[:300]}
        try:
            aux["sparse_config3"] = bench_aux.config3(ctx, cpu=not args.no_cpu)
        except Exception as e:  # the headline line must survive a failure here
            aux["sparse_config3"] = {"error": str(e)[:300]}
        try:   # ... and its portfolio (arrowhead) variant; CPU time of this one: profiles/r02_bench_aux.jsonl (35 s of SuperLU)
            aux["sparse_config3_portfolio"] = bench_aux.config3(ctx, portfolio=True, cpu=False)
        except Exception as e:
            aux["sparse_config3_portfolio"] = {"error": str(e)[:300]}
        # conic side of the path (configs 4, 5): lock-step batch of config-4 problems (the HBM-meaningful form, SURVEY 8d),
        # config 4 converged on the conditioned generator, the 200 x 200 PSD cone
        for key, fn in (("conic_batch_config4", lambda: bench_aux.run_conic_batch(ctx, B=296, iters=100, emit=False)),
                        ("conic_config4_converged", lambda: bench_aux.run_conic(
                            ctx, "4c", __import__("bench_data").conic_config4_conditioned(), iters=None,
                            cpu_iters=None if not args.no_cpu else 0, emit=False)),
                        ("psd_config5", lambda: bench_aux.config5(ctx, emit=False)),
                        ("dense_single_kkt", lambda: bench_aux.dense_single(ctx, emit=False))):
            try:
                aux[key] = fn()
            except Exception as e:
                aux[key] = {"error": str(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = BT * args.steps / (ms * 1e-3)
    e2e_val = BT * e2e_steps / (ms_e2e * 1e-3)
    peaks = fp64_peaks() if world == 1 else {}
    achieved = B * FLOP_PER_SOLVE / (kernel_ms * 1e-3) / 1e12
    peak = peaks.get("dgemm8192_tflops_sustained")
    prof = _profile_facts()
    hbm_peak = _hbm_peak()
    hbm_ach = B * BYTES_PER_SOLVE / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": (achieved / peak) if peak else None, "traffic": prof.get("dram_bytes_per_launch"),
                "kernel": "qp_kkt_sqd_kernel (KKT assembly + blocked LDL' on DMMA + 2 solves; pivoted-LU fallback kernel "
                          "launched behind it, plus the active-set scan), avg device time per launch %.3f ms over the "
                          "timed region (%d instances per launch on this rank); blocking call: %.3f ms per call (%.3f ms "
                          "of it between the library's own events)" % (kernel_ms, B, ms_blocking / 5, call_kernel_ms),
                "algorithmic_flop_per_solve": FLOP_PER_SOLVE, "algorithmic_bytes_per_solve": BYTES_PER_SOLVE,
                "executed_flop_per_solve_estimate": prof.get("executed_flop_per_solve"),
                "note": "achieved = SURVEY.md 8(d) algorithmic flop (LU of the N=144 KKT + 2x2 triangular solves) / device "
                        "time; the kernel reaches it by eliminating column singletons and factorising the symmetric "
                        "quasi-definite reduced system with LDL' (fewer executed flop, see DESIGN.md), so the binding "
                        "roofline of the reformulated kernel is HBM (hbm_secondary); traffic from profiles/ (ncu capture of "
                        "the same kernel, per 4096-instance launch)",
                "peak_source": "measured in this run: cuBLAS DGEMM 8192^3 sustained 4 s (tools/fp64_peak); "
                               "MEASURED_PEAKS.json has no FP64 entry",
                "fp64_peaks": peaks,
                "hbm_secondary": {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s",
                                  "frac": hbm_ach / hbm_peak, "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)"}}
    line = {"metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "4096 x dense QP n=64 m_ineq=64 m_eq=16 (KKT N=144), forward + reverse "
                                   "sensitivities (BASELINE.json configs[1])",
                       "global_batch": BT, "batch_per_gpu": B,
                       "parallelism": f"4096 instances split into contiguous shards over {world} GPU(s), no collective on "
                                      f"the data path (SURVEY.md 8e)",
                       "l2_policy": "per-rank inputs (%.0f MB/step) %s the 126 MB L2%s" % (
                           B * BYTES_PER_SOLVE / 1e6, "larger than" if B * BYTES_PER_SOLVE > 126e6 else "SMALLER than",
                           "" if B * BYTES_PER_SOLVE > 126e6 else
                           " (strong scaling shrinks the shard); see `weak` for the HBM-streaming number"),
                       "call": "diffopt_b200_qp_batch_solve_async x K + diffopt_b200_synchronize (stream-ordered, "
                               "device-resident inputs); e2e uses the blocking host-buffer call",
                       "host_numa": numa},
            "roofline": roofline, "e2e": {"value": e2e_val, "unit": "solves/s", "h2d_bytes_per_step": in_bytes * world,
                                          "d2h_bytes_per_step": out_bytes * world, "ms_per_step": ms_e2e / e2e_steps},
            "e2e_variants": e2e_variants,
            "gpu_launches": launches, "clocks": clocks, "parity_rel_err": err}
    if weak:
        line["weak"] = weak
    if shared:
        line["shared_variant"] = shared
    if aux:
        line["aux"] = aux
    if world == 1 and not args.no_cpu:
        procs = host_cores()
        sample = int(os.environ.get("DIFFOPT_BENCH_CPU_SAMPLE", 4096))
        line["cpu_baseline"] = cpu_baseline_block({k: logical_full[k][:sample] for k in logical_full}, sample, procs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def e2e_byte_variants(args, ctx, lib, capi, hb, logical, B, BT, world, timed, check, fwd_h, rev_h, info_h, steps):
    """The end-to-end call is PCIe bound (r1: 97 % of the step is the host-to-device copy), so the boundary accepts the
    same problem in fewer bytes (diffopt_b200_qp_batch_solve_ex).  Same metric, host (pinned) buffers, H2D + kernels + D2H
    inside the timed region:
      packed_triangles  Q and dQ as packed lower triangles (both are symmetric: utils.jl:46-69)
      shared_matrices   OptNet layer: Q, G, A and the direction dQ, dG, dA are ONE instance for the whole batch"""
    import diffopt_b200
    qpm = diffopt_b200.submodule("qp")
    out = {}
    pk = {k: capi.pinned_empty((B, N_VAR * (N_VAR + 1) // 2)) for k in ("Q", "dQ")}
    for k in pk:
        np.copyto(pk[k], qpm.pack_lower(logical[k]))

    def args_for(sub):
        return [capi.ptr(sub.get(k, hb[k])) for k in FIELDS]

    def step_packed():
        check(lib.diffopt_b200_qp_batch_solve_ex(ctx.h, B, N_VAR, M_INEQ, P_EQ, *args_for(pk), capi.ptr(fwd_h), capi.ptr(rev_h),
                                                 capi.ptr(info_h), capi.HOST, capi.QP_PACKED_Q), "qp_batch_solve_ex(packed)")
    ref_f, ref_r = fwd_h.copy(), rev_h.copy()      # results of the plain end-to-end call on the same data
    for _ in range(2):
        step_packed()
    if not (np.array_equal(fwd_h, ref_f) and np.array_equal(rev_h, ref_r)):
        raise RuntimeError("packed-triangle end-to-end call differs from the plain call")
    ms, _ = timed(step_packed, steps)
    nb = sum((pk[k] if k in pk else hb[k]).nbytes for k in FIELDS)
    out["packed_triangles"] = {"value": BT * steps / (ms * 1e-3), "unit": "solves/s", "ms_per_step": ms / steps,
                               "h2d_bytes_per_step": nb * world, "check": "bitwise equal to the plain call"}
    sh = {k: capi.pinned_empty(hb[k][:1].shape) for k in ("Q", "G", "A", "dQ", "dG", "dA")}
    for k in sh:
        np.copyto(sh[k], hb[k][:1])

    def step_shared():
        check(lib.diffopt_b200_qp_batch_solve_ex(ctx.h, B, N_VAR, M_INEQ, P_EQ, *args_for(sh), capi.ptr(fwd_h), capi.ptr(rev_h),
                                                 capi.ptr(info_h), capi.HOST, capi.QP_SHARED_MATRICES | capi.QP_SHARED_DIRECTION),
              "qp_batch_solve_ex(shared)")
    for _ in range(2):
        step_shared()
    if info_h.any() or not np.isfinite(fwd_h).all():
        raise RuntimeError("shared-matrix end-to-end call failed")
    ms, _ = timed(step_shared, steps)
    nb = sum((sh[k] if k in sh else hb[k]).nbytes for k in FIELDS)
    out["shared_matrices"] = {"value": BT * steps / (ms * 1e-3), "unit": "solves/s", "ms_per_step": ms / steps,
                              "h2d_bytes_per_step": nb * world,
                              "note": "Q, G, A, dQ, dG, dA of instance 0 serve the whole batch (a different problem set than the "
                                      "headline: the OptNet-shared form); parity of this entry: tests/test_qp_gpu.py"}
    # sparse directions: the reference's own packing (triplets per matrix, src/diff_opt.jl:594-656); the problem data stay
    # dense and per instance.  1 % of the entries of dQ, dG, dA are nonzero (a perturbation of a few coefficients).
    try:
        rng = np.random.default_rng(99)
        keep = {k: rng.random(logical[k].shape) < 0.01 for k in ("dG", "dA")}
        kq = np.triu(rng.random(logical["dQ"].shape) < 0.01)
        keep["dQ"] = kq | kq.transpose(0, 2, 1)
        coo_arrays, structs = {}, {}
        for k in ("dQ", "dG", "dA"):
            b_idx, i_idx, j_idx = np.nonzero(keep[k])
            ptrs = np.zeros(B + 1, dtype=np.int64)
            np.cumsum(np.bincount(b_idx, minlength=B), out=ptrs[1:])
            arrs = (ptrs, (i_idx + 1).astype(np.int64), (j_idx + 1).astype(np.int64), np.ascontiguousarray(logical[k][keep[k]]))
            pinned = []
            for a_ in arrs:
                buf = capi.pinned_empty(a_.shape, a_.dtype)
                np.copyto(buf, a_)
                pinned.append(buf)
            coo_arrays[k] = pinned
            structs[k] = capi.CooBatch(*[x.ctypes.data for x in pinned])
        base = [capi.ptr(hb[k]) for k in ("Q", "G", "A", "h", "z", "lam", "nu")]
        import ctypes

        def step_coo():
            check(lib.diffopt_b200_qp_batch_solve_coo(
                ctx.h, B, N_VAR, M_INEQ, P_EQ, *base, ctypes.addressof(structs["dQ"]), capi.ptr(hb["dq"]),
                ctypes.addressof(structs["dG"]), capi.ptr(hb["dh"]), ctypes.addressof(structs["dA"]), capi.ptr(hb["db"]),
                capi.ptr(hb["seed"]), capi.ptr(fwd_h), capi.ptr(rev_h), capi.ptr(info_h), capi.HOST, 0), "qp_batch_solve_coo")
        for _ in range(2):
            step_coo()
        if info_h.any() or not (np.linalg.norm(rev_h - ref_r, axis=1) <= 1e-10 * np.linalg.norm(ref_r, axis=1)).all():
            raise RuntimeError("sparse-direction end-to-end call failed")
        # forward results against the dense call on the masked direction (a few instances, through the plain entry)
        nchk = 8
        dsub = {k: np.ascontiguousarray((logical[k][:nchk] * keep[k][:nchk]).transpose(0, 2, 1)) for k in ("dQ", "dG", "dA")}
        fchk = np.empty((nchk, KKT_N))
        ichk = np.zeros(nchk, dtype=np.int32)
        got = fwd_h[:nchk].copy()
        check(lib.diffopt_b200_qp_batch_solve(
            ctx.h, nchk, N_VAR, M_INEQ, P_EQ, *[capi.ptr(np.ascontiguousarray(hb[k][:nchk])) for k in ("Q", "G", "A", "h", "z", "lam", "nu")],
            capi.ptr(dsub["dQ"]), capi.ptr(np.ascontiguousarray(hb["dq"][:nchk])), capi.ptr(dsub["dG"]),
            capi.ptr(np.ascontiguousarray(hb["dh"][:nchk])), capi.ptr(dsub["dA"]), capi.ptr(np.ascontiguousarray(hb["db"][:nchk])),
            None, capi.ptr(fchk), None, capi.ptr(ichk), capi.HOST), "qp_batch_solve(check)")
        rel = float((np.linalg.norm(got - fchk, axis=1) / np.linalg.norm(fchk, axis=1)).max())
        if not rel <= 1e-8:
            raise RuntimeError(f"sparse-direction results differ from the dense call: {rel:.3e}")
        ms, _ = timed(step_coo, steps)
        nb = sum(hb[k].nbytes for k in ("Q", "G", "A", "h", "z", "lam", "nu", "dq", "dh", "db", "seed")) + \
            sum(x.nbytes for v in coo_arrays.values() for x in v)
        out["sparse_directions"] = {"value": BT * steps / (ms * 1e-3), "unit": "solves/s", "ms_per_step": ms / steps,
                                    "h2d_bytes_per_step": nb * world, "direction_density": 0.01,
                                    "kernel": "shape-generic LDL' fast path on the right-hand side assembled from the triplets",
                                    "check_rel_diff_vs_dense_call": rel}
    except Exception as e:  # the headline line must survive a failure here
        out["sparse_directions"] = {"error": str(e)[:300]}
    return out


def shared_variant(args, rank, world, ctx, lib, capi, sharding, dev, db, logical, B, BT, timed, check, dptr):
    """OptNet-shared variant of config 2 (SURVEY.md 8d): Q, G, A are ONE instance shared by the 4096 problems (read once,
    L2 resident), only z, lam, nu, h and the seeds vary.  One step = reverse sensitivities of this rank's shard + the
    device-side batch sum of the shared-parameter gradients (dQ, dq, dG, dh, dA, db) + ONE device-resident fp64
    ncclAllReduce of the 9360 sums over the ranks, all stream-ordered inside the timed region."""
    import torch
    import torch.distributed as dist
    if world > 1:
        sharding.nccl_init(ctx, rank, world)
    n, m = N_VAR, M_INEQ
    per = N_VAR * N_VAR + N_VAR + M_INEQ * N_VAR + M_INEQ + P_EQ * N_VAR + P_EQ
    rev = torch.empty((B, KKT_N), dtype=torch.float64, device=dev)
    grads = torch.empty(per, dtype=torch.float64, device=dev)
    # the shared weights and the per-instance solutions: the same job on every rank (same seed), each keeps its shard
    import bench_data
    w = bench_data.qp_batch_shared_fast(BT, N_VAR, M_INEQ, P_EQ, seed=4242)
    lo, hi = sharding.shard_range(BT, rank, world)
    sh = {k: torch.from_numpy(np.ascontiguousarray(w[k].T)).to(dev) for k in ("Q", "G", "A")}     # column-major
    logical = {k: w[k][lo:hi] for k in ("h", "z", "lam", "nu", "seed")}
    db = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in logical.items()}
    null = capi.vp(None)
    flags = capi.QP_SHARED_MATRICES | capi.QP_ASYNC
    gflags = capi.QP_ASYNC | (capi.QP_ALLREDUCE if world > 1 else 0)

    def step():
        check(lib.diffopt_b200_qp_batch_solve_ex(
            ctx.h, B, N_VAR, M_INEQ, P_EQ, dptr(sh["Q"]), dptr(sh["G"]), dptr(sh["A"]), dptr(db["h"]), dptr(db["z"]),
            dptr(db["lam"]), dptr(db["nu"]), null, null, null, null, null, null, dptr(db["seed"]), null, dptr(rev), null,
            capi.DEVICE, flags), "qp_batch_solve_ex(shared)")
        check(lib.diffopt_b200_qp_batch_shared_grads(
            ctx.h, B, N_VAR, M_INEQ, P_EQ, dptr(db["z"]), dptr(db["lam"]), dptr(db["nu"]), dptr(rev), dptr(grads),
            capi.DEVICE, gflags), "qp_batch_shared_grads")

    def finish():
        check(lib.diffopt_b200_synchronize(ctx.h), "diffopt_b200_synchronize")
    for _ in range(3):
        step()
    finish()
    steps = min(args.steps, 100)
    ms, _ = timed(step, steps, finish)
    # post-timing checks (oracle / host arithmetic as checker only).  (1) the reverse solves against the oracle on a few
    # instances.  (2) batch sum + all-reduce: the getters evaluated
    # on the host from this rank's device results, summed over the ranks by torch.distributed as an independent path.
    from oracle import qp as oqp
    r = rev.cpu().numpy()
    z, lam, nu = logical["z"], logical["lam"], logical["nu"]
    serr = 0.0
    for b in range(min(4, B)):
        want_b = np.concatenate(oqp.reverse(w["Q"], w["G"], logical["h"][b], w["A"], z[b], lam[b], nu[b], logical["seed"][b]))
        serr = max(serr, float(np.linalg.norm(r[b] - want_b) / np.linalg.norm(want_b)))
    if not serr <= 1e-8:
        raise RuntimeError(f"shared-variant reverse solve check failed on rank {rank}: {serr:.3e}")
    dQ = 0.5 * (np.einsum("bi,bj->ij", r[:, :n], z) + np.einsum("bi,bj->ij", z, r[:, :n]))
    dG = np.einsum("bi,bj->ij", lam * r[:, n:n + m], z) + np.einsum("bi,bj->ij", lam, r[:, :n])
    dA = np.einsum("bi,bj->ij", r[:, n + m:], z) + np.einsum("bi,bj->ij", nu, r[:, :n])
    loc = np.concatenate([dQ.T.ravel(), r[:, :n].sum(0), dG.T.ravel(), -(lam * r[:, n:n + m]).sum(0), dA.T.ravel(),
                          -r[:, n + m:].sum(0)])
    tot = torch.from_numpy(loc).to(dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    got, want = grads.cpu().numpy(), tot.cpu().numpy()
    cerr = float(np.linalg.norm(got - want) / np.linalg.norm(want))
    if not cerr <= 1e-10:
        raise RuntimeError(f"shared-variant gradient sum / all-reduce check failed on rank {rank}: {cerr:.3e}")
    if world > 1:
        lib.diffopt_b200_nccl_destroy(ctx.h)
    return {"value": BT * steps / (ms * 1e-3), "unit": "solves/s", "ms_per_step": ms / steps, "steps": steps,
            "workload": "config 2, OptNet-shared: Q, G, A one instance for all 4096 problems; reverse sensitivities + "
                        "batch-summed shared-parameter gradients",
            "collective": ("ncclAllReduce(sum, f64, %d values = %d B) on the ctx stream, device resident, once per step"
                           % (per, 8 * per)) if world > 1 else "none (1 GPU): device batch sum only",
            "kernels_per_step": "qp_kkt_sqd_kernel + fallback list kernel + shared_grads_partial + shared_grads_final"
                                + (" + NCCL all-reduce" if world > 1 else ""),
            "allreduced_grads_rel_err_vs_host_sum": cerr, "reverse_rel_err_vs_oracle": serr}


def active_set_sweep(args, ctx, lib, capi, dev, timed, check, dptr):
    """Throughput of the headline call away from the benchmark's fixed 16 active rows (r1 review): 0 / 16 / 32 / 48 active
    inequalities, and interior-point style duals (inactive rows carry lam = 1e-9, active rows slack -1e-9: nothing is an
    exact zero)."""
    import torch

    import bench_data
    out = {}
    B = 4096
    cases = [("active_0", 0, False), ("active_16", 16, False), ("active_32", 32, False), ("active_48", 48, False),
             ("ipm_duals_16_active", 16, True)]
    for name, na, ipm in cases:
        d = bench_data.qp_batch_fast(B, N_VAR, M_INEQ, P_EQ, n_active=na, seed=77 + na)
        if ipm:
            act = d["lam"] > 0
            Gz = np.einsum("bij,bj->bi", d["G"], d["z"])
            d["lam"] = np.where(act, d["lam"], 1e-9)
            d["h"] = Gz - np.where(act, -1e-9, Gz - d["h"])
        t = {k: torch.from_numpy(np.ascontiguousarray(d[k].transpose(0, 2, 1) if k in SHAPES else d[k])).to(dev) for k in FIELDS}
        fo = torch.empty((B, KKT_N), dtype=torch.float64, device=dev)
        ro = torch.empty_like(fo)
        io = torch.zeros(B, dtype=torch.int32, device=dev)
        a = [dptr(t[k]) for k in FIELDS] + [dptr(fo), dptr(ro), dptr(io)]
        for _ in range(3):   # blocking calls first: they let the launch configuration follow the new active-set size
            check(lib.diffopt_b200_qp_batch_solve(ctx.h, B, N_VAR, M_INEQ, P_EQ, *a, capi.DEVICE), "qp_batch_solve")

        def step():
            check(lib.diffopt_b200_qp_batch_solve_async(ctx.h, B, N_VAR, M_INEQ, P_EQ, *a), "qp_batch_solve_async")
        steps = 20
        ms, _ = timed(step, steps, lambda: check(lib.diffopt_b200_synchronize(ctx.h), "synchronize"))
        nfb, hint, kern = ctx.qp_last_stats()
        out[name] = {"solves_per_s": B * steps / (ms * 1e-3), "ms_per_step": ms / steps,
                     "kernel": {0: "generic LU", 1: "pivoted LU", 2: "LDL' fast path"}.get(kern, "?"),
                     "instances_sent_to_pivoted_lu": nfb, "configured_active_rows": hint}
        del t, fo, ro, io
    return out


def other_shapes_sweep(ctx, lib, capi, dev, timed, check, dptr):
    """Batched QPs of shapes other than the headline's (r1 review: the fast kernel was hard-wired to 64/64/16): the
    shape-generic LDL' fast path against the generic pivoted-LU kernel (DIFFOPT_B200_QP_KERNEL=generic) on the same batch,
    forward + reverse sensitivities, device-resident inputs, stream-ordered calls."""
    import torch

    import bench_data
    out = {}
    for n, m, p, na, B in [(100, 50, 0, 10, 4096), (32, 32, 8, 8, 8192), (16, 16, 4, 4, 16384), (50, 100, 10, 20, 4096),
                           (100, 100, 10, 15, 2048),           # N = 210: the pivoted LU keeps its matrix in global memory
                           (N_VAR, M_INEQ, P_EQ, 16, 4096)]:   # last: the headline shape through the shape-generic kernel
        d = bench_data.qp_batch_fast(B, n, m, p, n_active=na, seed=500 + n)
        t = {k: torch.from_numpy(np.ascontiguousarray(d[k].transpose(0, 2, 1) if k in SHAPES else d[k])).to(dev) for k in FIELDS}
        N = n + m + p
        res = {}
        headline = (n, m, p) == (N_VAR, M_INEQ, P_EQ)
        for label, force in (("ldl_fast_path", "ldl_any" if headline else None), ("generic_pivoted_lu", "generic")):
            fo = torch.empty((B, N), dtype=torch.float64, device=dev)
            ro = torch.empty_like(fo)
            io = torch.zeros(B, dtype=torch.int32, device=dev)
            a = [dptr(t[k]) for k in FIELDS] + [dptr(fo), dptr(ro), dptr(io)]
            if force:
                os.environ["DIFFOPT_B200_QP_KERNEL"] = force
            try:
                for _ in range(3):
                    check(lib.diffopt_b200_qp_batch_solve(ctx.h, B, n, m, p, *a, capi.DEVICE), "qp_batch_solve")

                def step():
                    check(lib.diffopt_b200_qp_batch_solve_async(ctx.h, B, n, m, p, *a), "qp_batch_solve_async")
                steps = (3 if n + m + p > 165 else 10) if force == "generic" else 20
                ms, _ = timed(step, steps, lambda: check(lib.diffopt_b200_synchronize(ctx.h), "synchronize"))
            finally:
                os.environ.pop("DIFFOPT_B200_QP_KERNEL", None)
            nfb, hint, kern = ctx.qp_last_stats()
            res[label] = {"solves_per_s": B * steps / (ms * 1e-3), "ms_per_step": ms / steps,
                          "kernel": {0: "generic LU", 1: "pivoted LU", 2: "LDL' fast path"}.get(kern, "?"),
                          "instances_sent_to_pivoted_lu": nfb}
            res[label + "_out"] = (fo.cpu().numpy(), ro.cpu().numpy())
        f0, r0 = res.pop("ldl_fast_path_out")
        f1, r1 = res.pop("generic_pivoted_lu_out")
        rel = lambda x, y: float((np.linalg.norm(x - y, axis=1) / np.linalg.norm(y, axis=1)).max())
        res["max_rel_diff_between_kernels"] = max(rel(f0, f1), rel(r0, r1))
        res["speedup"] = res["ldl_fast_path"]["solves_per_s"] / res["generic_pivoted_lu"]["solves_per_s"]
        bytes_per = 8 * (2 * (n * n + m * n + p * n) + 3 * n + 3 * m + 3 * p + 2 * N)
        res["hbm_gbs_algorithmic"] = bytes_per * res["ldl_fast_path"]["solves_per_s"] / 1e9
        res["batch"] = B
        out[f"n{n}_m{m}_p{p}_active{na}"] = res
        del t
    return out


def _profile_facts():
    """Numbers read off the committed ncu capture of the dominant kernel (profiles/qp_sqd_facts.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "qp_sqd_facts.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def _hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"]
    except Exception:
        return 6650.0  # B200_PROFILING.md fallback


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-aux", action="store_true", help="skip the active-set sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the forward / reverse sensitivities and info codes of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the CPU arm only times the reference's work)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
