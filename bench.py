#!/usr/bin/env python
"""Benchmarks of the hot path (BASELINE.json metric "CDU linear-MPC QP solves/sec & sim-steps/sec at
1/2/4/8 B200 vs host-CPU ref").

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path, headline workload
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU path, same workload
    python bench.py --workload {cdu_closed_loop,horizon_sweep,cstr_qp_1m,nn_10m} ...
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's results

--dump-outputs DIR writes what the timed path returned in its last timed step (rank 0) as DIR/<name>.npy, float64,
64 MB at most: above that, the same seeded sample of batch rows of every array.  The inputs are seeded, so two
builds run with the same arguments can be compared file by file (bench_outputs/ is ignored by git).

Workloads (BASELINE.json configs[...]):
  cdu_closed_loop [2]  default, the headline.  The crude-distillation linear MPC of the reference (252 states,
                       32 inputs, 90 outputs, horizon N = 140 -> 4480 decision variables per QP,
                       cdu_parameters.py:94-102) on the documented synthetic stand-in plant (CDU_Model.mat is not
                       shipped), PRBS set-point / disturbance signals with the reference's statistics
                       (cdu_parameters.py:115-143).  --traj closed-loop trajectory chunks per GPU (the reference's
                       OS processes, lib/linearMPC.py:786-825) advance together; one bench step advances every
                       chunk by --slab simulation steps: target-selector QP -> regulator QP -> plant step
                       (lib/linearMPC.py:845-866).  Weak scaling over GPUs, no collective on the solve path.
  horizon_sweep   [4]  the same generator at --horizon 140/280/560 for a FIXED total of --samples samples over all
                       GPUs (strong scaling); the NCCL all-gather of the generated dataset is inside the timed step.
  cstr_qp_1m      [1]  --batch random CSTR regulator QPs (n = 540) per step through DenseQPRegulator.solve_batch.
  nn_10m          [3]  --batch states per step through RegulatorLayerWithUprev (568-832-832-832-32).

Numbers on the JSON line
  value         the workload's metric, all ranks, inputs resident in HBM, CUDA events, max over ranks, from a CLEAN
                timing pass (no profiling hooks)
  e2e           the same through the reference-facing host API with pinned HOST buffers: host->device copies of the
                step's inputs and device->host copies of its results inside the timed region
  roofline      the dominant kernel, from a separate PROFILED pass over the same inputs (CUDA events recorded by
                the library around each group of launches on the launching stream)
  cpu_baseline  the reference-style CPU path (oracle port) on this host's cores, on a bounded sample
The reference arm (--impl reference) times that CPU path: every step is one bounded sample of the workload.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KKT_TOL = 1e-8
DUMP_BYTES = 64_000_000
WORKLOADS = {
    "cdu_closed_loop": ("cdu_closed_loop_sim_steps_per_s", "sim-steps/s"),
    "horizon_sweep": ("cdu_closed_loop_sim_steps_per_s", "sim-steps/s"),
    "cstr_qp_1m": ("cstr_regulator_qp_solves_per_s", "QP solves/s"),
    "nn_10m": ("cdu_structured_nn_states_per_s", "states/s"),
}
# kept for importers of the round-1 names
METRIC, UNIT = WORKLOADS["cdu_closed_loop"]
NN_HIDDEN = [832, 832, 832]


# ------------------------------------------------------------------------------------------ helpers
def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def dump_outputs(dirname, arrays, seed=0):
    """--dump-outputs: every array (batch axis first; CUDA tensor or NumPy) -> dirname/<name>.npy in float64.  Above
    DUMP_BYTES in all, every array keeps the same seeded, sorted sample of batch rows."""
    rows = next(iter(arrays.values())).shape[0]
    assert all(a.shape[0] == rows for a in arrays.values()), {k: tuple(a.shape) for k, a in arrays.items()}
    row_bytes = sum(8 * int(np.prod(a.shape[1:])) for a in arrays.values())
    keep = min(rows, (DUMP_BYTES - 4096 * len(arrays)) // row_bytes)       # 4 kB per file for the .npy header
    idx = np.arange(rows) if keep == rows else np.sort(np.random.default_rng(seed).choice(rows, keep, replace=False))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if isinstance(a, np.ndarray):
            a = a[idx]
        else:                                    # gather the sample on the device, copy only that
            import torch
            a = a.index_select(0, torch.as_tensor(idx, device=a.device)).cpu().numpy()
        np.save(os.path.join(dirname, name + ".npy"), a.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thr = index, [], None, None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            self.thr.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def _scenarios(traj, steps, seed, gain_norm=None, r_weight=None):
    """PRBS-like set-points / disturbances with the reference's hold statistics, split into `traj`
    contiguous chunks of `steps` rows (lib/linearMPC.py:786-801) -> (traj, steps, .) arrays.
    gain_norm / r_weight: conditioning study of the synthetic stand-in (defaults: plants/cdu.py, R = 0.1 I)."""
    from industrial_nnmpc_2021_b200.plants import get_cdu_problem
    from industrial_nnmpc_2021_b200.plants import cdu as _cdu
    p = get_cdu_problem(Nsim=traj * steps, seed=seed, gain_norm=_cdu.GAIN_NORM if gain_norm is None else gain_norm)
    if r_weight is not None:
        p.R = r_weight * np.eye(p.Nu)
    sp = p.setpoints.reshape(traj, steps, p.Ny)
    ds = p.disturbances.reshape(traj, steps, p.Nd)
    return p, sp, ds


def _sweep_slab(args, world):
    """horizon_sweep: simulation steps per chunk and bench step so that K steps generate --samples in total."""
    per_step = world * args.traj * max(args.steps, 1)
    return max(1, int(-(-int(args.samples) // per_step)))


def _config(args, world=None):
    """The workload description: a function of the command line only, so that both arms (--impl native /
    reference) print the same block for the same flags."""
    world = args.gpus if world is None else world
    wl = args.workload
    if wl in ("cdu_closed_loop", "horizon_sweep"):
        slab = args.slab if wl == "cdu_closed_loop" else _sweep_slab(args, world)
        c = {"workload": ("CDU linear-MPC closed-loop offline data generation (BASELINE.json configs[2]): synthetic CDU "
                          "stand-in 252x32x90, reference tuning, PRBS scenarios") if wl == "cdu_closed_loop" else
                         ("CDU horizon/batch sweep (BASELINE.json configs[4]): closed-loop data generation of a fixed "
                          "number of samples over all GPUs, NVLink all-gather of the dataset inside the timed step"),
             "Nx": 252, "Nu": 32, "Ny": 90, "horizon": args.horizon, "qp_vars": args.horizon * 32,
             "trajectories_per_gpu": args.traj, "concurrent_slots_per_gpu": min(args.traj, args.slots),
             "sim_steps_per_step": slab, "tol_kkt": KKT_TOL,
             "scenario_slabs": f"{args.unique_slabs} distinct PRBS slabs at most, cycled over the steps",
             "precision": args.precision, "gain_norm": args.gain_norm, "R": args.r_weight,
             "shape_note": "65 536 chunks x 16 steps on 16 384 slots is the best point of the builder's own sweep "
                           "(profiles/r01v_bench_shape_sweep.txt); the reference's shape is 149 chunks x 2400 steps. "
                           "Short chunks are conservative on cold starts (1 QP in 16)",
             "l2": "no flush: operators (2 x 161 MB FP64 + 2 x 40 MB fp16 at N = 140) + solver state exceed the 126 MB L2 "
                   "every iteration",
             "parallelism": f"trajectories sharded over {world} GPU(s), no collective on the solve path"}
        if wl == "horizon_sweep":
            c["samples_total"] = int(args.samples)
        return c
    if wl == "cstr_qp_1m":
        return {"workload": "CSTRs batched linear MPC (BASELINE.json configs[1]): random (x0, uprev, setpoint) regulator QPs, "
                            "cold start, through DenseQPRegulator.solve_batch",
                "Nx": 12, "Nu": 6, "horizon": 90, "qp_vars": 540, "batch_per_gpu": args.batch or (1 << 20),
                "x_minus_xs_sigma": [0.02, 0.1, 0.5, 2.0], "tol_kkt": KKT_TOL,
                "l2": "no flush: five B x 540 FP64 state arrays (22 GB at 1 M QPs) stream through every iteration",
                "parallelism": f"samples sharded over {world} GPU(s), no collective"}
    return {"workload": "CDU structured NN batched policy evaluation (BASELINE.json configs[3]): RegulatorLayerWithUprev "
                        "568-832-832-832-32, u = us + f(x,uprev,xs,us) - f(xs,us,xs,us)",
            "Nx": 252, "Nu": 32, "hidden": NN_HIDDEN, "batch_per_gpu": args.batch or 10_000_000,
            "nn_precision": os.environ.get("NNMPC_MLP", "tc"),
            "l2": "no flush: 45 GB of inputs per step",
            "parallelism": f"samples sharded over {world} GPU(s), no collective"}


# ------------------------------------------------------------------------------------------ CPU paths
_W = {}     # per-worker state of the CPU pool


def _cpu_layout():
    cores = os.cpu_count() or 1
    threads = min(cores, 8)
    mem_gb = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES") / 2**30
    workers = max(1, min(cores // threads, int(mem_gb // 6), 32))
    return cores, workers, threads


def _cdu_worker_init(seed0, threads, horizon, counter):
    """One reference-style process (lib/linearMPC.py:803-825): its own operators and trajectory, kept alive across
    the steps of the arm so that only the closed-loop steps are timed."""
    import threadpoolctl
    import scipy.linalg
    from oracle import linear_mpc as om
    from industrial_nnmpc_2021_b200 import condense
    with counter.get_lock():
        wid = counter.value
        counter.value += 1
    _W["limits"] = threadpoolctl.threadpool_limits(limits=threads)
    p, sp, ds = _scenarios(1, 4000, seed0 + 2 * wid)
    Aa, Ba, Qa, Ra, Ma = om.augmented_matrices_for_regulator(p.A, p.B, p.Q, p.R, p.S)
    _, Pf = om.dlqr(Aa, Ba, Qa, Ra, Ma)
    P, tq = condense.condensed_hessian(Aa, Ba, Qa, Ra, Ma, Pf, horizon)   # setup, untimed
    E = np.vstack([np.eye(p.Nu), -np.eye(p.Nu)])
    _W.update(p=p, sp=sp[0], ds=ds[0], P=P, tq=tq, G=scipy.linalg.block_diag(*([E] * horizon)),   # dense tE (:459-460)
              ots=om.TargetSelectorOracle(A=p.A, B=p.B, C=p.C, H=p.H, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs,
                                          ulb=p.ulb, uub=p.uub),
              x=p.xprior.copy(), up=p.uprev.copy(), t=0, horizon=horizon)


def _cdu_worker_step(job):
    """nsteps closed-loop steps of this worker's trajectory, every QP by the cvxopt-like interior point
    (oracle.qp.ipm_qp): dense G and operators re-materialised per call as the reference does
    (lib/linearMPC.py:15-20, :503), or the structure-exploiting diagonal-G variant."""
    nsteps, strong = job
    from oracle import qp as oq
    w = _W
    p, horizon = w["p"], w["horizon"]
    iters, t0 = [], time.time()
    for _ in range(nsteps):
        t = w["t"] % w["sp"].shape[0]
        ysp, d = w["sp"][t][:, None], w["ds"][t][:, None]
        xs, us = w["ots"].solve(ysp, d)
        x0 = np.vstack([w["x"] - xs, w["up"] - us])
        h = np.tile(np.vstack([p.uub - us, -(p.ulb - us)]), (horizon, 1))
        if strong:
            useq, info = oq.ipm_qp(w["P"], w["tq"] @ x0, None, h, diagonal_G=True, rematerialise=False)
        else:
            useq, info = oq.ipm_qp(w["P"], w["tq"] @ x0, w["G"], h)
        iters.append(info["iters"])
        u = useq[:p.Nu] + us
        w["x"] = p.A @ w["x"] + p.B @ u + p.Bd @ d
        w["up"] = u
        w["t"] += 1
    return t0, time.time(), iters


def _worker_ready(_):
    return os.getpid()


class CduCpuPool:
    """The reference CPU path of the CDU workload on every host core: `workers` processes (the reference's
    num_parallel) x `threads` BLAS threads.  A dense interior-point iteration at n = 4480 is ~0.4 TFLOP of
    BLAS-3, so 8 threads per process give the same aggregate throughput as 8 single-thread processes while a
    step (one QP per process) takes ~10 s instead of ~80 s - what keeps W + K reference steps within minutes."""

    def __init__(self, horizon, seed=11):
        import multiprocessing as mp
        self.cores, self.workers, self.threads = _cpu_layout()
        ctx = mp.get_context("spawn")
        self.counter = ctx.Value("i", 0)
        self.pool = ctx.Pool(self.workers, initializer=_cdu_worker_init,
                             initargs=(seed, self.threads, horizon, self.counter))
        self.horizon = horizon
        self.pool.map(_worker_ready, range(self.workers), chunksize=1)      # operators are built (untimed set-up)

    def step(self, nsteps=1, strong=False):
        """-> (sim-steps/s over all workers, seconds per QP, IPM iterations)."""
        res = self.pool.map(_cdu_worker_step, [(nsteps, strong)] * self.workers, chunksize=1)
        span = max(r[1] for r in res) - min(r[0] for r in res)
        return self.workers * nsteps / span, span / nsteps, [i for r in res for i in r[2]]

    def sample(self, nsteps, iters, strong=False):
        return (f"{self.workers} trajectories x {nsteps} closed-loop step(s) (CDU, N={self.horizon}, n={self.horizon * 32}), "
                f"cold-start {'diagonal-G (structure-exploiting)' if strong else 'dense-G (cvxopt-like)'} interior point "
                f"per QP, mean {np.mean(iters):.1f} IPM iterations, {self.workers} processes x {self.threads} BLAS threads")

    def close(self):
        self.pool.close()
        self.pool.join()


def _cstr_cpu_init(threads):
    import threadpoolctl
    from oracle import linear_mpc as om
    from industrial_nnmpc_2021_b200.plants import get_cstrs_problem
    _W["limits"] = threadpoolctl.threadpool_limits(limits=threads)
    p = get_cstrs_problem()
    reg = om.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    _W.update(p=p, reg=reg)


def _cstr_cpu_step(job):
    from oracle import qp as oq
    X0, LB, UB = job
    reg, p = _W["reg"], _W["p"]
    t0 = time.time()
    for i in range(X0.shape[0]):
        h = np.tile(np.concatenate([UB[i], -LB[i]])[:, None], (p.N, 1))
        oq.ipm_qp(reg.P, reg.tq @ X0[i][:, None], reg.G, h)
    return t0, time.time()


def _nn_cpu_rate(weights, ins, threads):
    import threadpoolctl
    from oracle import nn as onn
    with threadpoolctl.threadpool_limits(limits=threads):
        onn.layer_call(weights, [a[:256] for a in ins], True)
        t0 = time.perf_counter()
        onn.layer_call(weights, ins, True)
        return ins[0].shape[0] / (time.perf_counter() - t0)


# ------------------------------------------------------------------------------------------ common GPU plumbing
class Ctx:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (this framework has no CPU fallback)")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.dev = torch.device("cuda", self.local)
        self.f64 = dict(dtype=torch.float64, device=self.dev)
        if self.rank == 0:
            from industrial_nnmpc_2021_b200 import build
            build.build()
        if self.world > 1:
            dist.barrier()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def maxrank(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], **self.f64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def events(self):
        return self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)

    def pinned(self, shape, dtype=None):
        return self.torch.empty(shape, dtype=dtype or self.torch.float64, pin_memory=True).numpy()

    def finish(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def _dgemm_peak(ctx):
    torch = ctx.torch
    a = torch.randn((6144, 6144), **ctx.f64); b = torch.randn((6144, 6144), **ctx.f64)
    for _ in range(3):
        torch.matmul(a, b)
    best = 0.0
    for _ in range(5):
        g0, g1 = ctx.events()
        g0.record(); torch.matmul(a, b); g1.record(); torch.cuda.synchronize()
        best = max(best, 2 * 6144 ** 3 / (g0.elapsed_time(g1) * 1e-3) / 1e12)
    return best


def _int8_peak(ctx):
    """Dense INT8 tensor throughput of this GPU measured with the library GEMM (torch._int_mm -> cuBLASLt), best of
    5, TOP/s; None when the library path is unavailable."""
    torch = ctx.torch
    try:
        a = torch.randint(-100, 100, (8192, 8192), dtype=torch.int8, device=ctx.dev)
        b = torch.randint(-100, 100, (8192, 8192), dtype=torch.int8, device=ctx.dev).t().contiguous().t()
        for _ in range(3):
            torch._int_mm(a, b)
        best = 0.0
        for _ in range(5):
            g0, g1 = ctx.events()
            g0.record(); torch._int_mm(a, b); g1.record(); torch.cuda.synchronize()
            best = max(best, 2 * 8192 ** 3 / (g0.elapsed_time(g1) * 1e-3) / 1e12)
        return best
    except Exception:
        return None


def _base_line(args, ctx, metric, unit, value, ms_step, K, W, scaling="weak", dtype="f64"):
    return {"metric": metric, "value": value, "unit": unit, "n_gpus": ctx.world, "steps": K, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": dtype, "data": "synthetic", "config": _config(args, ctx.world)}


# ------------------------------------------------------------------------------------------ CDU closed loop
def run_cdu(args):
    ctx = Ctx(args)
    torch, world, rank, dev = ctx.torch, ctx.world, ctx.rank, ctx.dev
    from industrial_nnmpc_2021_b200 import _lib
    from industrial_nnmpc_2021_b200 import distributed as nd_
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController, ClosedLoopEngine
    L = _lib.lib()
    sweep = args.workload == "horizon_sweep"
    metric, unit = WORKLOADS[args.workload]
    K, W, B = args.steps, max(args.warmup, 3), args.traj
    Ts = _sweep_slab(args, world) if sweep else args.slab
    Tw = min(Ts, args.warmup_slab) if sweep else Ts          # horizon_sweep: short warm-up steps
    nuniq = min(2 * (W + K), max(1, args.unique_slabs))
    # distinct PRBS scenario slabs kept in memory; further steps cycle through them (bounds host memory).  Trajectories
    # that continue across steps (--traj <= --slots) see one extra set-point jump where the cycle wraps.
    p, sp, ds = _scenarios(B, nuniq * Ts, seed=101 + 2 * rank, gain_norm=args.gain_norm, r_weight=args.r_weight)
    p.N = args.horizon
    t_setup = time.perf_counter()
    ts = LinearMPCController.setup_target_selector(p.A, p.B, p.C, p.H, p.Bd, p.Cd, p.usp, p.Qs, p.Rs, p.ulb, p.uub,
                                                   device=dev)
    solver_kw = {}
    if args.alpha is not None:
        solver_kw["alpha"] = args.alpha
    if args.rho_scale is not None:
        solver_kw["rho_scale"] = args.rho_scale
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub, device=dev, **solver_kw)
    eng = ClosedLoopEngine(reg, ts, p.A, p.B, p.Bd, precision=args.precision, slots=args.slots)
    t_setup = time.perf_counter() - t_setup
    n, nx, nu, ny, ndist = p.N * p.Nu, p.Nx, p.Nu, p.Ny, p.Nd

    def slab_np(i, T=Ts):
        j = i % nuniq
        return sp[:, j * Ts:j * Ts + T], ds[:, j * Ts:j * Ts + T]

    slabs = [tuple(torch.tensor(np.ascontiguousarray(a), **ctx.f64) for a in slab_np(i)) for i in range(min(W + K, nuniq))]

    def out_dev(T):
        return dict(x=torch.empty((B, T, nx), **ctx.f64), uprev=torch.empty((B, T, nu), **ctx.f64),
                    xs=torch.empty((B, T, nx), **ctx.f64), us=torch.empty((B, T, nu), **ctx.f64),
                    u=torch.empty((B, T, nu), **ctx.f64), iters=torch.empty((B, T), dtype=torch.int32, device=dev),
                    kkt=torch.empty((B, T), **ctx.f64))
    out_d = out_dev(Ts)
    out_w = out_d if Tw == Ts else out_dev(Tw)
    state = dict(x=p.xprior, up=p.uprev, hit=False, first=True)

    def dev_step(i, warm=False):
        a, b = slabs[i % len(slabs)]
        if warm and Tw != Ts:
            a, b = a[:, :Tw].contiguous(), b[:, :Tw].contiguous()
        r = eng.run(state["x"], state["up"], a, b, resume=not state["first"], out=out_w if warm else out_d,
                    max_iter=args.max_iter)
        state.update(x=r["x_final"], up=r["uprev_final"], first=False)
        state["hit"] |= bool(r["maxiter_hit"])
        if sweep and world > 1 and not warm:        # configs[4]: the dataset gather is part of the measured step
            full = nd_.gather_chunks({k: r[k] for k in nd_.DATASET_KEYS}, world * B)
            del full
        return r

    # ---- device-resident phase: clean timing pass --------------------------------------------
    for i in range(W):
        dev_step(i, warm=True)
    if sweep and world > 1:
        nd_.gather_chunks({k: out_d[k] for k in nd_.DATASET_KEYS}, world * B)     # NCCL communicator set-up, untimed
    ctx.barrier()
    kkt_acc = torch.zeros((), **ctx.f64)
    it_sum = torch.zeros((), dtype=torch.int64, device=dev)
    it_acc = torch.zeros((), dtype=torch.int32, device=dev)
    st0 = eng.stats()
    launches0 = L.nnmpc_launch_count()
    ev0, ev1 = ctx.events()
    with ClockSampler(ctx.local) as clk:
        ev0.record()
        for i in range(W, W + K):
            r = dev_step(i)
            # validity of the timed work itself (device-side reductions, read after the timing)
            kkt_acc = torch.maximum(kkt_acc, r["kkt"].max())
            it_sum = it_sum + r["iters"].sum(dtype=torch.int64)
            it_acc = torch.maximum(it_acc, r["iters"].max())
        ev1.record()
        ctx.barrier()
    ms_dev = ctx.maxrank(ev0.elapsed_time(ev1))
    launches = L.nnmpc_launch_count() - launches0
    st1 = eng.stats()
    kkt_max, it_sum, it_max = float(kkt_acc), int(it_sum), int(it_acc)
    clocks = clk.summary()
    value = world * B * Ts * K / (ms_dev * 1e-3)
    if args.dump_outputs and rank == 0:          # before the profiled pass reuses the result buffers
        dump_outputs(args.dump_outputs, {k: r[k] for k in ("x", "uprev", "xs", "us", "u", "iters", "kkt",
                                                           "x_final", "uprev_final")})

    # ---- profiled pass: the same kind of steps with the library's CUDA-event spans switched on ----
    Kp = max(1, min(K, args.prof_steps))
    _lib.prof_enable(True)
    _lib.prof_read(reset=True)
    ctx.barrier()
    pv0, pv1 = ctx.events()
    sp0 = eng.stats()
    pv0.record()
    for i in range(W + K, W + K + Kp):
        dev_step(i)
    pv1.record()
    ctx.barrier()
    ms_prof = pv0.elapsed_time(pv1)            # this rank's own clock: shares are per rank
    chans = _lib.prof_readn(4, reset=True)
    _lib.prof_enable(False)
    sp1 = eng.stats()
    (gemm_ms, gemm_flops, gemm_launches), (f64_ms, f64_flops, f64_launches) = chans[0], chans[1]
    (tail_ms, tail_flops, _), rest_ms = chans[2], chans[3][0]
    value_prof = world * B * Ts * Kp / (ctx.maxrank(ms_prof) * 1e-3)

    # ---- end-to-end phase: host buffers through the reference-facing API -----------------------
    if args.no_e2e:          # kernel A/B runs only: a line without "e2e" is not a bench result
        if rank == 0:
            t1 = sp1["tiles_one_term"] - sp0["tiles_one_term"]
            t2 = sp1["tiles_two_terms"] - sp0["tiles_two_terms"]
            nq = max(sp1["qps"] - sp0["qps"], 1)
            print(json.dumps({"ab_run": True, "value": value, "value_profiled": value_prof,
                              "iterations_mean": it_sum / (B * Ts * K), "iterations_max": it_max, "kkt_max": kkt_max,
                              "lp_tflops": gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None,
                              "exact_tflops_fp64eq": f64_flops / (f64_ms * 1e-3) / 1e12 if f64_ms > 0 else None,
                              "one_term_tile_share": t1 / max(t1 + t2, 1),
                              "mma_products_per_iteration": (t1 + 2.0 * t2 + sp1.get("tiles_second_term_delivery", 0)
                                                             - sp0.get("tiles_second_term_delivery", 0)) / max(t1 + t2, 1),
                              "work_per_qp": {k: (sp1[k] - sp0[k]) / nq for k in ("row_iterations", "anchors", "exact_checks")},
                              "shares": {"lp": gemm_ms / ms_prof, "exact": f64_ms / ms_prof, "tail": tail_ms / ms_prof,
                                         "rest": rest_ms / ms_prof}, "clocks": clocks,
                              "env": {k: v for k, v in os.environ.items() if k.startswith("NNMPC_")}}), flush=True)
        ctx.finish()
        return
    out_h = dict(x=ctx.pinned((B, Ts, nx)), uprev=ctx.pinned((B, Ts, nu)), xs=ctx.pinned((B, Ts, nx)),
                 us=ctx.pinned((B, Ts, nu)), u=ctx.pinned((B, Ts, nu)), iters=ctx.pinned((B, Ts), torch.int32),
                 kkt=ctx.pinned((B, Ts)))
    sp_h, ds_h = ctx.pinned((B, Ts, ny)), ctx.pinned((B, Ts, ndist))
    xh, uph = state["x"].cpu().numpy(), state["up"].cpu().numpy()
    e2e_kkt, hit_e2e = 0.0, False
    gat = {k: torch.empty((B, Ts, out_h[k].shape[2]), **ctx.f64) for k in nd_.DATASET_KEYS} if sweep and world > 1 else None
    ctx.barrier()
    We = 1 if sweep else W                    # horizon_sweep: steps are long and already warm
    for i in range(We + K):
        if i == We:
            ctx.barrier()
            ee0, ee1 = ctx.events()
            ee0.record()
            t_e2e = time.perf_counter()
        a, b = slab_np(W + K + Kp + i)
        sp_h[...] = a                                  # this step's inputs staged in pinned host memory
        ds_h[...] = b
        r = eng.run(xh, uph, sp_h, ds_h, resume=True, out=out_h, max_iter=args.max_iter)
        xh, uph = r["x_final"], r["uprev_final"]
        e2e_kkt = max(e2e_kkt, float(out_h["kkt"].max()))      # the device->host result is read every step
        hit_e2e |= bool(r["maxiter_hit"])
        if gat is not None:                            # configs[4]: gather of the generated rows over NVLink
            for k in nd_.DATASET_KEYS:
                gat[k].copy_(torch.from_numpy(out_h[k]), non_blocking=True)
            full = nd_.gather_chunks(gat, world * B)
            del full
    ee1.record()
    ctx.barrier()
    wall_e2e = time.perf_counter() - t_e2e
    ms_e2e = ctx.maxrank(max(ee0.elapsed_time(ee1), 1e3 * wall_e2e))
    e2e_value = world * B * Ts * K / (ms_e2e * 1e-3)
    h2d = (sp_h.nbytes + ds_h.nbytes + xh.nbytes + uph.nbytes) * world
    d2h = (sum(v.nbytes for v in out_h.values()) + xh.nbytes + uph.nbytes) * world

    # ---- dataset gather over NCCL/NVLink, timed alone (weak-scaling runs keep it outside `value`) ----
    gather = None
    if world > 1:
        local_d = {k: out_d[k] for k in nd_.DATASET_KEYS}
        nd_.gather_chunks(local_d, world * B)          # warm-up (NCCL communicator set-up)
        ctx.barrier()
        gv0, gv1 = ctx.events()
        gv0.record()
        full = nd_.gather_chunks(local_d, world * B)
        gv1.record()
        ctx.barrier()
        g_ms = ctx.maxrank(gv0.elapsed_time(gv1))
        g_bytes = sum(v.numel() * v.element_size() for v in full.values())
        # content check: this rank's block of the gathered arrays is its own data, bit for bit
        lo = rank * B
        same = all(bool(torch.equal(full[k][lo:lo + B], out_d[k])) for k in nd_.DATASET_KEYS)
        gather = {"ms": g_ms, "bytes_gathered_per_rank": g_bytes, "algbw_GBs": g_bytes / (g_ms * 1e-3) / 1e9,
                  "inside_value": bool(sweep), "own_block_bit_exact": same,
                  "what": "all_gather_into_tensor of one step's dataset rows (x, uprev, xs, us, u) from every rank"}
        del full

    if kkt_max > KKT_TOL or e2e_kkt > KKT_TOL or state["hit"] or hit_e2e:
        raise SystemExit(f"bench.py: timed solves missed the tolerance (kkt {kkt_max:.2e}/{e2e_kkt:.2e}, "
                         f"maxiter_hit={state['hit'] or hit_e2e}); number rejected")

    # ---- rooflines of the two tensor-core kernels ---------------------------------------------------
    peaks, peak_src = _peaks()
    best = _dgemm_peak(ctx)
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    dgemm_src = ("cuBLAS DGEMM 6144^3 measured in this run (FP64 has no tcgen05 kind; MEASURED_PEAKS.json carries "
                 f"bf16 {peaks.get('bf16_tflops')} TF/s and HBM {peaks.get('hbm_gbs')} GB/s only, {peak_src})")
    per_unit = f"active samples x 2 n^2 (n = {n}: {2 * n * n / 1e6:.2f} MFLOP per sample-iteration)"
    where = f"separate profiled pass of {Kp} step(s) after the clean timing pass"
    if args.precision == "f64":
        roofline = {"bound": "tensor", "kernel": "gemm_f64_kernel<EpiAdmm> (regulator-QP iteration, FP64 DMMA)",
                    "achieved": achieved, "peak": best, "unit": "TFLOP/s", "frac": achieved / best if best else None,
                    "traffic": None, "launches": gemm_launches, "avg_launch_ms": gemm_ms / max(gemm_launches, 1),
                    "share_of_step": gemm_ms / ms_prof, "peak_source": dgemm_src, "flops_per_launch": per_unit,
                    "measured_in": where}
        roofline2 = None
    else:
        lp_peak = float(peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 1590.0)
        f64_ach = f64_flops / (f64_ms * 1e-3) / 1e12 if f64_ms > 0 else 0.0
        rows_per_launch = (gemm_flops / (2.0 * n * n)) / max(gemm_launches, 1)
        # tiles of late-phase rows run with one operator term (LpShape::need2): executed MMA work per algorithmic flop
        t1, t2 = sp1["tiles_one_term"] - sp0["tiles_one_term"], sp1["tiles_two_terms"] - sp0["tiles_two_terms"]
        tc = sp1.get("tiles_second_term_delivery", 0) - sp0.get("tiles_second_term_delivery", 0)
        mma_factor = (t1 + 2.0 * t2 + tc) / max(t1 + t2, 1) if (t1 + t2) else 2.0
        # DRAM bytes per launch: a MODEL, not a per-run measurement - the fp16 operator terms read once per pass
        # (mma_factor x 2 n^2 B) plus the per-row state, with the per-row constant taken from the one `ncu --set full`
        # capture of this kernel: deferred second term (profiles/r02r_ncu_full_lp_gemm.txt) 3.87 GB per launch at 16 384
        # rows, n = 4480 -> 233.8 kB per row vs 46 B x n = 206.1 kB algorithmic (42 B of state + 4 B of pending sums);
        # both terms in every pass (profiles/r02h_ncu_full_lp_gemm.txt) 222 kB per row vs 42 B x n; scaled linearly in n
        deferred = tc > 0
        op_bytes = mma_factor * 2.0 * n * n
        row_model, row_alg = (233.8e3, 46.0) if deferred else (222.0e3, 42.0)
        r_lp = {"bound": "tensor", "kernel": ("lp_gemm_kernel<EpiDelta> + lp_gemm_kernel<EpiAddX> (regulator-QP iteration: tcgen05 kind::f16, fp16 "
                           "increments x first fp16 operator term every pass, second term delivered every 8th pass from the "
                           "pending sums, fp32 TMEM accumulators, FP64 state)") if deferred else
                          ("lp_gemm_kernel<EpiDelta> (regulator-QP iteration: tcgen05 kind::f16, fp16 increments x two-term fp16 "
                           "operator split, fp32 TMEM accumulators, FP64 state)"),
                "mma_products_per_iteration": mma_factor,
                "achieved": achieved, "executed_mma": mma_factor * achieved, "peak": lp_peak, "unit": "TFLOP/s",
                "one_term_tile_share": t1 / max(t1 + t2, 1),
                "frac": achieved / lp_peak, "frac_executed": mma_factor * achieved / lp_peak,
                "traffic": op_bytes + row_model * (n / 4480.0) * rows_per_launch,
                "traffic_kind": "model scaled from one ncu capture (see bench.py), not measured in this run",
                "traffic_algorithmic": op_bytes + row_alg * n * rows_per_launch,
                "rows_per_launch": rows_per_launch,
                "launches": gemm_launches, "avg_launch_ms": gemm_ms / max(gemm_launches, 1),
                "share_of_step": gemm_ms / ms_prof,
                "peak_source": f"dense 16-bit tensor throughput, sustained figure of MEASURED_PEAKS.json ({peak_src}); "
                               "kernel timed inside a long step",
                "flops_per_launch": per_unit + "; the kernel executes up to 2x that in MMA work (T1 and T2 products)",
                "measured_in": where}
        if os.environ.get("NNMPC_EXACT_GEMM", "int8") == "dmma":
            r_64 = {"bound": "tensor", "kernel": "gemm_f64_kernel<EpiAnchor|EpiVerifyMax> (FP64 anchors x = Top w - c and "
                                                 "exact KKT checks P z + q, DMMA, small row lists)",
                    "achieved": f64_ach, "peak": best, "unit": "TFLOP/s", "frac": f64_ach / best if best else None,
                    "traffic": None, "launches": f64_launches, "avg_launch_ms": f64_ms / max(f64_launches, 1),
                    "share_of_step": f64_ms / ms_prof, "peak_source": dgemm_src,
                    "flops_per_launch": "listed samples x 2 n^2", "measured_in": where}
        else:
            # INT8-sliced exact applies: 21 (anchors, 6 levels) / 36 (checks, 8 levels) INT8 products of 2 n^2 ops per row
            n_anch, n_chk = sp1["anchors"] - sp0["anchors"], sp1["exact_checks"] - sp0["exact_checks"]
            int8_ops = 2.0 * n * n * (21.0 * n_anch + 36.0 * n_chk)
            int8_ach = int8_ops / (f64_ms * 1e-3) / 1e12 if f64_ms > 0 else 0.0
            int8_meas = _int8_peak(ctx)
            int8_peak = int8_meas if int8_meas else 2.0 * lp_peak
            r_64 = {"bound": "tensor", "kernel": "oz_gemm2_kernel<.,.,128,OzEpiAnchor|OzEpiVerify> + k_oz_slice (FP64-accurate "
                                                 "anchors x = Top w - c and exact KKT checks P z + q on tcgen05 kind::i8: "
                                                 "error-free base-128 digit planes, exact INT32 accumulation)",
                    "achieved": int8_ach, "fp64_equivalent": f64_ach, "peak": int8_peak, "unit": "TOP/s",
                    "frac": int8_ach / int8_peak, "fp64_equivalent_vs_cublas_dgemm": f64_ach / best if best else None,
                    "cublas_dgemm_tflops": best,
                    "traffic": None, "launches": f64_launches, "avg_launch_ms": f64_ms / max(f64_launches, 1),
                    "share_of_step": f64_ms / ms_prof,
                    "peak_source": ("dense INT8 GEMM 8192^3 through the library (torch._int_mm -> cuBLASLt) measured in this run"
                                    if int8_meas else "2 x the sustained 16-bit dense figure of MEASURED_PEAKS.json (the "
                                    "library INT8 GEMM was not available to measure)"),
                    "flops_per_launch": "listed samples x 2 n^2 FP64-equivalent = x 21 (anchor) or 36 (check) INT8 products; "
                                        "span includes the digit-plane slicing kernel", "measured_in": where}
        roofline, roofline2 = (r_lp, r_64) if gemm_ms >= f64_ms else (r_64, r_lp)

    if rank == 0:
        cpu = cpu_strong = None
        if world == 1 and not args.no_cpu_baseline:
            pool = CduCpuPool(args.horizon)
            rate, spq, iters = pool.step(1)
            cpu = {"value": rate, "unit": unit, "cores": pool.workers * pool.threads, "kind": "port",
                   "sample": pool.sample(1, iters), "seconds_per_qp": spq, "host_cores": pool.cores}
            rate2, spq2, iters2 = pool.step(2, strong=True)
            cpu_strong = {"value": rate2, "unit": unit, "cores": pool.workers * pool.threads, "kind": "port",
                          "sample": pool.sample(2, iters2, strong=True), "seconds_per_qp": spq2,
                          "note": "stronger CPU baseline than the reference's own path: G = [I; -I] never formed"}
            pool.close()
        nq = max(st1["qps"] - st0["qps"], 1)
        line = _base_line(args, ctx, metric, unit, value, ms_dev / K, K, W, scaling="strong" if sweep else "weak")
        line.update({
            "qp_solves_per_s": {"regulator": value, "target_selector": value},
            "iterations": {"mean": it_sum / (B * Ts * K), "max": it_max, "kkt_max": kkt_max},
            "conditioning": {"cond_P": reg.eig_range[1] / reg.eig_range[0], "lambda_min": reg.eig_range[0],
                             "lambda_max": reg.eig_range[1],
                             "active_bound_frac": (st1["qps_with_active_bounds"] - st0["qps_with_active_bounds"]) / nq,
                             "mean_active_bounds_per_qp": (st1["active_bounds"] - st0["active_bounds"]) / nq,
                             "what": "condition number of the condensed Hessian; share of the timed QPs whose optimum has "
                                     ">= 1 active input bound; active bounds per QP (of n); sweep: profiles/r02_conditioning.md"},
            "roofline": roofline, "roofline_second_kernel": roofline2, "cpu_baseline": cpu,
            "cpu_baseline_strong": cpu_strong, "precision": args.precision,
            "solver_work_per_qp": {k: (st1[k] - st0[k]) / nq for k in ("row_iterations", "anchors", "exact_checks")},
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / K, "kkt_max": e2e_kkt, "gather_inside": bool(gat is not None)},
            "profiled_pass": {"steps": Kp, "value": value_prof,
                              "note": "same steps with the library's CUDA-event spans on; `value` comes from the clean pass"},
            "time_breakdown": {"unit": "share of the profiled pass (CUDA events on the launching stream, rank 0)",
                               "iteration_passes": gemm_ms / ms_prof, "exact_anchors_and_checks": f64_ms / ms_prof,
                               "fp64_tail_iterations": tail_ms / ms_prof,
                               "fp64_tail_tflops": tail_flops / (tail_ms * 1e-3) / 1e12 if tail_ms > 0 else None,
                               "plant_target_qbuild_lists": rest_ms / ms_prof,
                               "other": 1.0 - (gemm_ms + f64_ms + tail_ms + rest_ms) / ms_prof},
            "gpu_launches": int(launches), "clocks": clocks, "setup_s": t_setup, "gather": gather,
        })
        print(json.dumps(line), flush=True)
    ctx.finish()


# ------------------------------------------------------------------------------------------ CSTR QPs (configs[1])
def _cstr_batch(p, ts, B, dev, torch, seed):
    """BASELINE.json configs[1] / SURVEY 8(d): set-point and disturbance rows of the CSTR scenario -> target selector ->
    (xs, us); x - xs ~ N(0, sigma^2) with sigma drawn from {0.02, 0.1, 0.5, 2}; uprev ~ U(ulb, uub)."""
    rng = np.random.default_rng(seed)
    YSP = torch.tensor(p.setpoints[rng.integers(0, p.setpoints.shape[0], B)], device=dev)
    D = torch.tensor(p.disturbances[rng.integers(0, p.disturbances.shape[0], B)], device=dev)
    XS, US = ts.solve_batch(YSP, D)
    sigma = torch.tensor(rng.choice([0.02, 0.1, 0.5, 2.0], B), device=dev)[:, None]
    g = torch.Generator(device=dev).manual_seed(seed + 7)
    dx = sigma * torch.randn((B, p.Nx), dtype=torch.float64, device=dev, generator=g)
    ulb, uub = torch.tensor(p.ulb.T, device=dev), torch.tensor(p.uub.T, device=dev)
    uprev = ulb + (uub - ulb) * torch.rand((B, p.Nu), dtype=torch.float64, device=dev, generator=g)
    X0 = torch.cat([dx, uprev - US], dim=1).contiguous()
    return X0, (ulb - US).contiguous(), (uub - US).contiguous()


def run_cstr_qp(args):
    ctx = Ctx(args)
    torch, world, rank, dev = ctx.torch, ctx.world, ctx.rank, ctx.dev
    from industrial_nnmpc_2021_b200 import _lib
    from industrial_nnmpc_2021_b200.plants import get_cstrs_problem
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    L = _lib.lib()
    metric, unit = WORKLOADS["cstr_qp_1m"]
    K, W, B = args.steps, max(args.warmup, 3), args.batch or (1 << 20)
    p = get_cstrs_problem()
    t_setup = time.perf_counter()
    ts = LinearMPCController.setup_target_selector(p.A, p.B, p.C, p.H, p.Bd, p.Cd, p.usp, p.Qs, p.Rs, p.ulb, p.uub, device=dev)
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub, device=dev)
    t_setup = time.perf_counter() - t_setup
    n = p.N * p.Nu
    X0, LB, UB = _cstr_batch(p, ts, B, dev, torch, 2021 + rank)
    mode = dict(precision=args.qp_precision) if args.qp_precision != "lockstep" else {}

    def solve():
        return reg.solve_batch(X0, LB, UB, max_iter=args.max_iter, **mode)

    for _ in range(W):
        U, info = solve()
    ctx.barrier()
    launches0 = L.nnmpc_launch_count()
    ev0, ev1 = ctx.events()
    with ClockSampler(ctx.local) as clk:
        ev0.record()
        for _ in range(K):
            U, info = solve()
        ev1.record()
        ctx.barrier()
    ms_dev = ctx.maxrank(ev0.elapsed_time(ev1))
    launches = L.nnmpc_launch_count() - launches0
    value = world * B * K / (ms_dev * 1e-3)
    kkt_max = float(info["kkt"].max())
    it_mean, it_max = float(info["iters"].double().mean()), int(info["iters"].max())
    Us = U.view(B, p.N, p.Nu)
    active = float(((Us == LB[:, None, :]) | (Us == UB[:, None, :])).any(dim=2).any(dim=1).double().mean())
    if kkt_max > KKT_TOL or info["maxiter_hit"]:
        raise SystemExit(f"bench.py: timed solves missed the tolerance (kkt {kkt_max:.2e}); number rejected")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"U": U, "cost": info["cost"], "kkt": info["kkt"], "iters": info["iters"]})
    # profiled pass
    _lib.prof_enable(True)
    _lib.prof_read(reset=True)
    pv0, pv1 = ctx.events()
    pv0.record(); solve(); pv1.record(); ctx.barrier()
    ms_prof = pv0.elapsed_time(pv1)
    chans = _lib.prof_readn(4, reset=True)
    _lib.prof_enable(False)
    gemm_ms, gemm_flops, gemm_launches = chans[0]
    # e2e: host buffers through solve_batch's NumPy form (nnmpc_qp_solve_host: copies in and out inside the call)
    X0h, LBh, UBh = ctx.pinned(tuple(X0.shape)), ctx.pinned(tuple(LB.shape)), ctx.pinned(tuple(UB.shape))
    X0h[...], LBh[...], UBh[...] = X0.cpu().numpy(), LB.cpu().numpy(), UB.cpu().numpy()
    outh = dict(U=ctx.pinned((B, n)), cost=ctx.pinned((B,)), kkt=ctx.pinned((B,)), iters=ctx.pinned((B,), torch.int32))
    del U, Us
    torch.cuda.empty_cache()
    ctx.barrier()
    for i in range(1 + K):
        if i == 1:
            ctx.barrier()
            t_e2e = time.perf_counter()
        Uh, ih = reg.solve_batch(X0h, LBh, UBh, max_iter=args.max_iter, out=outh, **mode)
        e2e_kkt = float(ih["kkt"].max())
    ctx.barrier()
    ms_e2e = ctx.maxrank(1e3 * (time.perf_counter() - t_e2e))
    e2e_value = world * B * K / (ms_e2e * 1e-3)
    best = _dgemm_peak(ctx)
    peaks, peak_src = _peaks()
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    lowp = bool(chans[1][0] > 0)          # the mixed tiers record their exact applies on channel 1
    peak = float(peaks.get("bf16_tflops_sustained") or 1386.0) if lowp else best
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = _cstr_cpu_baseline(X0, LB, UB, unit)
        line = _base_line(args, ctx, metric, unit, value, ms_dev / K, K, W)
        line.update({
            "iterations": {"mean": it_mean, "max": it_max, "kkt_max": kkt_max, "active_bound_frac": active},
            "roofline": {"bound": "tensor",
                         "kernel": ("lp_gemm_kernel<EpiDelta> (tcgen05 fp16 increments)" if lowp else
                                    "gemm_f64_kernel<EpiAdmm> (regulator-QP iteration, FP64 DMMA mma.sync m8n8k4)"),
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                         "traffic": None, "launches": gemm_launches, "avg_launch_ms": gemm_ms / max(gemm_launches, 1),
                         "share_of_step": gemm_ms / ms_prof,
                         "flops_per_launch": f"active samples x 2 n^2 (n = {n}: {2 * n * n / 1e6:.3f} MFLOP per sample-iteration)",
                         "peak_source": (f"sustained 16-bit dense figure of MEASURED_PEAKS.json ({peak_src})" if lowp else
                                         "cuBLAS DGEMM 6144^3 measured in this run (FP64 has no tcgen05 kind)"),
                         "measured_in": "separate profiled pass of 1 step"},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": (X0h.nbytes + LBh.nbytes + UBh.nbytes) * world,
                    "d2h_bytes_per_step": sum(v.nbytes for v in outh.values()) * world, "ms_per_step": ms_e2e / K,
                    "kkt_max": e2e_kkt},
            "gpu_launches": int(launches), "clocks": clk.summary(), "setup_s": t_setup,
        })
        print(json.dumps(line), flush=True)
    ctx.finish()


def _cstr_cpu_baseline(X0, LB, UB, unit, per_worker=6):
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    workers = min(cores, 64)
    m = workers * per_worker
    X0h, LBh, UBh = X0[:m].cpu().numpy(), LB[:m].cpu().numpy(), UB[:m].cpu().numpy()
    with mp.get_context("spawn").Pool(workers, initializer=_cstr_cpu_init, initargs=(1,)) as pool:
        jobs = [(X0h[w::workers], LBh[w::workers], UBh[w::workers]) for w in range(workers)]
        pool.map(_cstr_cpu_step, [(j[0][:1], j[1][:1], j[2][:1]) for j in jobs], chunksize=1)     # warm the workers
        res = pool.map(_cstr_cpu_step, jobs, chunksize=1)
    span = max(r[1] for r in res) - min(r[0] for r in res)
    return {"value": m / span, "unit": unit, "cores": workers, "kind": "port",
            "sample": f"{m} of the timed QPs, {workers} single-thread processes x {per_worker} QPs, cold-start dense-G "
                      "(cvxopt-like) interior point", "seconds_per_qp": span / per_worker, "host_cores": cores}


# ------------------------------------------------------------------------------------------ structured NN (configs[3])
def _nn_weights(nx, nu, hidden, seed=1):
    rng = np.random.default_rng(seed)
    dims = [2 * nx + 2 * nu] + hidden + [nu]
    ws = []
    for i in range(len(dims) - 1):
        lim = np.sqrt(6.0 / (dims[i] + dims[i + 1]))            # Glorot-uniform (keras.layers.Dense default)
        ws.append(rng.uniform(-lim, lim, (dims[i], dims[i + 1])))
        if i < len(dims) - 2:
            ws.append(0.1 * rng.standard_normal(dims[i + 1]))  # non-zero biases exercise the bias path
    return ws


def run_nn(args):
    ctx = Ctx(args)
    torch, world, rank, dev = ctx.torch, ctx.world, ctx.rank, ctx.dev
    from industrial_nnmpc_2021_b200 import _lib
    from industrial_nnmpc_2021_b200.LinearMPCLayers import RegulatorLayerWithUprev
    from oracle import nn as onn
    L = _lib.lib()
    metric, unit = WORKLOADS["nn_10m"]
    nx, nu = 252, 32
    K, W, B = args.steps, max(args.warmup, 3), args.batch or 10_000_000
    ws = _nn_weights(nx, nu, NN_HIDDEN)
    layer = RegulatorLayerWithUprev(layer_dims=NN_HIDDEN + [nu], device=dev)
    layer.set_weights(ws)
    g = torch.Generator(device=dev).manual_seed(11 + rank)
    x = torch.randn((B, nx), generator=g, **ctx.f64)
    xs = x + 0.3 * torch.randn((B, nx), generator=g, **ctx.f64)
    up = 2.0 * torch.rand((B, nu), generator=g, **ctx.f64) - 1.0
    us = 2.0 * torch.rand((B, nu), generator=g, **ctx.f64) - 1.0
    for _ in range(W):
        out = layer([x, up, xs, us])
    ctx.barrier()
    launches0 = L.nnmpc_launch_count()
    ev0, ev1 = ctx.events()
    with ClockSampler(ctx.local) as clk:
        ev0.record()
        for _ in range(K):
            out = layer([x, up, xs, us])
        ev1.record()
        ctx.barrier()
    ms_dev = ctx.maxrank(ev0.elapsed_time(ev1))
    launches = L.nnmpc_launch_count() - launches0
    value = world * B * K / (ms_dev * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"u": out})
    # validity: a sample of the timed outputs against the NumPy restatement (tolerance of the north star: 1e-5)
    pick = torch.randint(0, B, (512,), device=dev, generator=g)
    ins = [t[pick].cpu().numpy() for t in (x, up, xs, us)]
    err = float(np.max(np.abs(out[pick].cpu().numpy() - onn.layer_call(ws, ins, True))))
    if not err <= 1e-5:
        raise SystemExit(f"bench.py: structured-network outputs differ from the NumPy restatement by {err:.2e} > 1e-5")
    # e2e: 1 M-row blocks from pinned host memory through the NumPy form of the layer call
    Bh = min(B, 1 << 20)
    host = [ctx.pinned((Bh, w_)) for w_ in (nx, nu, nx, nu)]
    for hbuf, t in zip(host, (x, up, xs, us)):
        hbuf[...] = t[:Bh].cpu().numpy()
    nblk = -(-B // Bh)
    ctx.barrier()
    for i in range(1 + K):
        if i == 1:
            ctx.barrier()
            t_e2e = time.perf_counter()
        for _ in range(nblk):
            oh = layer(host)
    ctx.barrier()
    ms_e2e = ctx.maxrank(1e3 * (time.perf_counter() - t_e2e))
    e2e_value = world * nblk * Bh * K / (ms_e2e * 1e-3)
    dims = [2 * nx + 2 * nu] + NN_HIDDEN + [nu]
    flops_state = 2 * sum(2 * dims[i] * dims[i + 1] for i in range(len(dims) - 1))      # both passes f(x,..) and f(xs,..)
    achieved = value / world * flops_state / 1e12
    lowp = layer.precision == "tc"
    peaks, peak_src = _peaks()
    best = _dgemm_peak(ctx)
    int8_meas = _int8_peak(ctx) if lowp else None
    if lowp:            # INT8 tier: 10 digit-plane products per FP64-equivalent flop
        achieved *= 10.0
        peak = int8_meas if int8_meas else 2.0 * float(peaks.get("bf16_tflops_sustained") or 1386.0)
    else:
        peak = best
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            m = 20000
            rate = _nn_cpu_rate(ws, [a[:m] for a in host], cores)
            cpu = {"value": rate, "unit": unit, "cores": cores, "kind": "port",
                   "sample": f"{m} of the timed states through the NumPy restatement of RegulatorLayerWithUprev.call "
                             f"(float64, {cores} BLAS threads)"}
        line = _base_line(args, ctx, metric, unit, value, ms_dev / K, K, W)
        line.update({
            "max_abs_err_vs_numpy": err,
            "roofline": {"bound": "tensor",
                         "kernel": ("oz_gemm2_kernel<0,3,128,OzEpiDense> + k_oz_slice<4> (tcgen05 kind::i8: 4 base-128 digit planes "
                                    "of activations and weights, 10 products, exact INT32 accumulation)" if lowp else
                                    "gemm_f64_kernel<EpiStore|EpiStructOut> (FP64 DMMA, bias + ReLU fused)"),
                         "achieved": achieved, "peak": peak, "unit": "TOP/s" if lowp else "TFLOP/s",
                         "frac": achieved / peak if peak else None, "traffic": None,
                         "fp64_equivalent_tflops": achieved / 10.0 if lowp else achieved, "cublas_dgemm_tflops": best,
                         "flops_per_launch": f"{flops_state / 1e6:.2f} MFLOP per state (both network passes, all layers)"
                                             + (" x 10 INT8 digit-plane products" if lowp else "") + "; whole forward timed "
                                             "(slicing kernels included), achieved = states/s x ops per state",
                         "peak_source": (("dense INT8 GEMM 8192^3 through the library (torch._int_mm) measured in this run"
                                          if int8_meas else f"2 x the sustained 16-bit dense figure of MEASURED_PEAKS.json ({peak_src})")
                                         if lowp else "cuBLAS DGEMM 6144^3 measured in this run")},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": sum(h.nbytes for h in host) * nblk * world,
                    "d2h_bytes_per_step": oh.nbytes * nblk * world, "ms_per_step": ms_e2e / K,
                    "blocks": f"{nblk} blocks of {Bh} states from pinned host memory per step"},
            "gpu_launches": int(launches), "clocks": clk.summary(),
        })
        print(json.dumps(line), flush=True)
    ctx.finish()


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """The reference's CPU implementation of the workload (oracle port; cvxopt / TensorFlow are not installable
    here) on every host core: W untimed + exactly K timed steps, each a bounded sample of the workload."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    metric, unit = WORKLOADS[args.workload]
    K, W = args.steps, args.warmup
    if args.workload in ("cdu_closed_loop", "horizon_sweep"):
        pool = CduCpuPool(args.horizon)
        for _ in range(W):
            pool.step(args.ref_steps)
        t0 = time.perf_counter()
        rates, iters, spq = [], [], []
        for _ in range(K):
            r, s, it = pool.step(args.ref_steps)
            rates.append(r); spq.append(s); iters += it
        wall = time.perf_counter() - t0
        value = pool.workers * args.ref_steps * K / wall
        cpu = {"value": value, "unit": unit, "cores": pool.workers * pool.threads, "kind": "port",
               "sample": "per step: " + pool.sample(args.ref_steps, iters), "seconds_per_qp": float(np.mean(spq)),
               "host_cores": pool.cores}
        pool.close()
        note = ("reference CPU path = oracle port of lib/linearMPC.py simulate_offline with a cvxopt-like dense interior "
                "point (cvxopt itself is not installable here); paper: 35 s/QP, 3.57 steps/s on 149 processes")
    elif args.workload == "cstr_qp_1m":
        import torch
        from industrial_nnmpc_2021_b200.plants import get_cstrs_problem
        from oracle import linear_mpc as om
        p = get_cstrs_problem()
        rng = np.random.default_rng(2021)
        ots = om.TargetSelectorOracle(A=p.A, B=p.B, C=p.C, H=p.H, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs,
                                      ulb=p.ulb, uub=p.uub)
        cores = os.cpu_count() or 1
        m = min(cores, 64) * 6
        rows = []
        for _ in range(m):
            xs, us = ots.solve(p.setpoints[rng.integers(0, p.setpoints.shape[0])][:, None],
                               p.disturbances[rng.integers(0, p.disturbances.shape[0])][:, None])
            dx = rng.choice([0.02, 0.1, 0.5, 2.0]) * rng.standard_normal((p.Nx, 1))
            up = p.ulb + (p.uub - p.ulb) * rng.random((p.Nu, 1))
            rows.append((np.vstack([dx, up - us])[:, 0], (p.ulb - us)[:, 0], (p.uub - us)[:, 0]))
        X0, LB, UB = (torch.tensor(np.asarray([r[i] for r in rows])) for i in range(3))
        vals = [_cstr_cpu_baseline(X0, LB, UB, unit) for _ in range(W + K)][W:]
        value = float(np.mean([v["value"] for v in vals]))
        wall = sum(m / v["value"] for v in vals)
        cpu = dict(vals[-1], value=value)
        note = "reference CPU path = oracle port of DenseQPRegulator.solve with a cvxopt-like dense interior point"
    else:
        from oracle import nn as onn  # noqa: F401
        cores = os.cpu_count() or 1
        ws = _nn_weights(252, 32, NN_HIDDEN)
        rng = np.random.default_rng(11)
        m = 20000
        ins = [rng.standard_normal((m, 252)), rng.uniform(-1, 1, (m, 32)), rng.standard_normal((m, 252)),
               rng.uniform(-1, 1, (m, 32))]
        t0 = None
        vals = []
        for i in range(W + K):
            if i == W:
                t0 = time.perf_counter()
            vals.append(_nn_cpu_rate(ws, ins, cores))
        wall = time.perf_counter() - t0
        value = float(np.mean(vals[W:]))
        cpu = {"value": value, "unit": unit, "cores": cores, "kind": "port",
               "sample": f"per step: {m} states through the NumPy restatement of RegulatorLayerWithUprev.call (float64)"}
        note = "reference path = NumPy restatement of the Keras layer (TensorFlow is not installable here)"
    line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": K,
            "warmup": W, "ms_per_step": 1e3 * wall / max(K, 1), "higher_is_better": True,
            "scaling": "strong" if args.workload == "horizon_sweep" else "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": _config(args), "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "note": note}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="cdu_closed_loop", choices=sorted(WORKLOADS))
    ap.add_argument("--unique-slabs", type=int, default=6,
                    help="distinct scenario slabs generated; steps beyond that cycle through them")
    ap.add_argument("--traj", type=int, default=None,
                    help="closed-loop trajectory chunks per GPU and bench step (the reference's per-process chunks, "
                         "lib/linearMPC.py:786-801); with --slots below it they queue up (continuous batching)")
    ap.add_argument("--slab", type=int, default=16, help="simulation steps every trajectory advances per bench step")
    ap.add_argument("--horizon", type=int, default=140)
    ap.add_argument("--samples", type=float, default=10e6, help="horizon_sweep: samples generated by the K timed steps, all GPUs")
    ap.add_argument("--warmup-slab", type=int, default=2, help="horizon_sweep: simulation steps per warm-up step")
    ap.add_argument("--batch", type=int, default=None, help="cstr_qp_1m / nn_10m: samples per GPU and step")
    ap.add_argument("--ref-steps", type=int, default=1, help="closed-loop steps per worker per reference step")
    ap.add_argument("--slots", type=int, default=16384,
                    help="trajectories advanced concurrently per GPU; with --traj above it the other chunks queue up and "
                         "finished slots take the next one (continuous batching)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="kernel A/B runs: stop after the device-resident passes")
    ap.add_argument("--precision", default="mixed", choices=["mixed", "f64"],
                    help="regulator-QP iteration arithmetic: tcgen05 fp16 increments + FP64 anchors, or all FP64 DMMA")
    ap.add_argument("--qp-precision", default="mixed", choices=["mixed", "f64", "lockstep"],
                    help="cstr_qp_1m: solve_batch through the continuously batched engine (tcgen05 tiers or FP64), or the "
                         "lock-step FP64 solver")
    ap.add_argument("--prof-steps", type=int, default=2, help="steps of the separate profiled pass")
    ap.add_argument("--alpha", type=float, default=None, help="Douglas-Rachford relaxation (solver default 1.8)")
    ap.add_argument("--rho-scale", type=float, default=None, help="multiplier of the default ADMM penalty (solver default 1)")
    ap.add_argument("--gain-norm", type=float, default=None,
                    help="conditioning study: steady-state gain-row norm of the synthetic plant (default plants/cdu.py: 0.7)")
    ap.add_argument("--r-weight", type=float, default=None, help="conditioning study: R = r I (reference tuning: 0.1)")
    ap.add_argument("--max-iter", type=int, default=None,
                    help="per-QP iteration cap (a hit rejects the number); default 3000 (CDU closed loop) / 20000 (cold CSTR QPs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy (float64, seeded row sample, "
                         "64 MB at most)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of this repository's CUDA path, not of --impl reference")
    if args.traj is None:
        args.traj = 16384 if args.workload == "horizon_sweep" else 65536
    if args.max_iter is None:
        args.max_iter = 20000 if args.workload == "cstr_qp_1m" else 3000
    if args.impl == "reference":
        run_reference(args)
    elif args.workload in ("cdu_closed_loop", "horizon_sweep"):
        run_cdu(args)
    elif args.workload == "cstr_qp_1m":
        run_cstr_qp(args)
    else:
        run_nn(args)


if __name__ == "__main__":
    main()
