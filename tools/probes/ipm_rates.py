"""Throughput of the interior-point regulator kernel (csrc/ipm.cu) on strongly unstable plants.

    python tools/probes/ipm_rates.py [--batch 16384] [--reps 3]

Prints one line per shape: card name and power limit (read in the same run), QPs/s, mean / max interior-point
iterations and algorithmic FLOP/s.  The flop count per iteration is the formula of `ipm_flops_per_iteration` below,
from the shapes alone (Riccati factorisation + two right-hand sides + roll-out + adjoint pass).
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))


def unstable_plant(nx, nu, seed, rho):
    rng = np.random.default_rng(seed)
    lam = np.concatenate([[rho, 0.97], rng.uniform(0.3, 0.9, nx - 2)])
    V = rng.standard_normal((nx, nx)) + 2.0 * np.eye(nx)
    return V @ np.diag(lam) @ np.linalg.inv(V), rng.standard_normal((nx, nu))


def ipm_flops_per_iteration(nx, nu, N):
    """Per QP and interior-point iteration (nx = padded augmented state, nu inputs, N stages)."""
    factor = 2 * nx**3 + 2 * nx**2 * nu + 2 * nu**2 * nx + 2 * nu * nx**2 + nu**3 / 3 + 2 * nx * nu**2 + 2 * nx**3 \
        + 2 * nx**2 * nu
    rhs = 2 * nx * nu + 2 * nu**2 + 2 * nx * nu + 2 * nx**2 + 2 * nx * nu + 2 * nx * nu * 2 + 2 * nx**2 + 2 * nx * nu
    rollout = 2 * nx**2 + 2 * nx * nu + 2 * nx * nu
    adjoint = 2 * nu**2 + 4 * nx * nu + 2 * nx**2 + 2 * nx * nu + 2 * nx * nu
    return N * (factor + 2 * rhs + rollout + adjoint)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return out
    except Exception as exc:       # noqa: BLE001
        return f"unknown ({exc})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch
    from industrial_nnmpc_2021_b200.linearMPC import DenseQPRegulator, LinearMPCController
    if not torch.cuda.is_available():
        raise SystemExit("ipm_rates: needs a CUDA device")
    gpu = card()
    shapes = {"cstr_like nxa=18 nu=6 N=90": (12, 6, 90, 1.5, True), "small nxa=6 nu=2 N=30": (6, 2, 30, 2.0, False)}
    for label, (nx, nu, N, rho, rate) in shapes.items():
        A, B = unstable_plant(nx, nu, 7, rho)
        if rate:
            reg = LinearMPCController.setup_regulator(A=A, B=B, Q=np.eye(nx), R=np.eye(nu), S=0.2 * np.eye(nu), N=N,
                                                      ulb=-np.ones((nu, 1)), uub=np.ones((nu, 1)))
        else:
            reg = DenseQPRegulator(A=A, B=B, Q=np.eye(nx), R=0.5 * np.eye(nu), M=np.zeros((nx, nu)), N=N,
                                   ulb=-np.ones((nu, 1)), uub=np.ones((nu, 1)))
        assert reg.solver == "ipm", label
        rng = np.random.default_rng(0)
        D = rng.standard_normal((a.batch, reg.Nx))
        D /= np.abs(D @ reg._S.T).max(axis=1)[:, None]
        X0 = torch.as_tensor(D * np.logspace(-1, np.log10(2.5), a.batch)[:, None], device="cuda")
        reg.solve_batch(X0)                       # warm-up: module load, scratch allocation
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.reps):
            U, info = reg.solve_batch(X0)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / a.reps
        it = info["iters"].double()
        flops = ipm_flops_per_iteration(reg._nxa_ld, nu, N) * float(it.sum())
        print(f"{gpu} | {label} | B={a.batch} | {a.batch / dt:.0f} QPs/s | iterations mean {float(it.mean()):.2f} "
              f"max {int(it.max())} | {flops / dt / 1e9:.1f} GFLOP/s algorithmic | maxiter {info['maxiter_hit']}")


if __name__ == "__main__":
    main()
