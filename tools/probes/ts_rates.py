"""Rate of the batched target selector (nnmpc_ts_solve, device entry point) on the full CDU (252 x 32 x 90, nd = 5)
in its three modes: H empty (box kernel k_target_selector), H empty with output bounds (k_ts_general over Ny + Nu rows)
and H = Hsel, the 4 weighted outputs pinned (reduced k_ts_general, nw = 28 variables, Nu rows).

    python tools/probes/ts_rates.py [--batch 16384] [--reps 20] [--out FILE]

Times whole calls with CUDA events after warm-up and prints one JSON line per mode, with the card's name and power
limit read in the same run.  Set-points: the CDU PRBS scenario for the H-empty modes; for H = Hsel the outputs of
steady states at interior inputs (PRBS set-points mostly cannot be pinned inside the input box)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in q.split(",")]
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from industrial_nnmpc_2021_b200.linearMPC import TargetSelector
    from industrial_nnmpc_2021_b200.plants import get_cdu_problem
    from industrial_nnmpc_2021_b200.plants.cdu import NZ
    name, power = card()
    p = get_cdu_problem(Nsim=100000)
    rng = np.random.default_rng(0)
    B = a.batch
    idx = rng.integers(0, p.setpoints.shape[0], B)
    ysp_prbs, d_prbs = p.setpoints[idx], p.disturbances[idx]
    # reachable pinned set-points: y = C (I-A)^-1 (B u0 + Bd d) at inputs inside 60 % of the box
    u0 = 0.6 * rng.uniform(-1.0, 1.0, (B, p.Nu))
    xs0 = np.linalg.solve(np.eye(p.Nx) - p.A, p.B @ u0.T + p.Bd @ d_prbs.T).T
    ysp_pin = xs0 @ p.C.T
    Hsel = np.hstack([np.zeros((NZ, p.Ny - NZ)), np.eye(NZ)])
    base = dict(A=p.A, B=p.B, C=p.C, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs, ulb=p.ulb, uub=p.uub)
    H0 = np.zeros((0, p.Ny))
    modes = [("box", dict(base, H=H0), ysp_prbs),
             ("output_bounds", dict(base, H=H0, ylb=-1.05 * np.ones((p.Ny, 1)), yub=1.05 * np.ones((p.Ny, 1))), ysp_prbs),
             ("pinned_hsel", dict(base, H=Hsel), ysp_pin)]
    f64 = dict(dtype=torch.float64, device="cuda")
    D = torch.as_tensor(d_prbs, **f64)
    lines = []
    for mode, kw, ysp in modes:
        ts = TargetSelector(**kw)
        Y = torch.as_tensor(ysp, **f64)
        for _ in range(3):
            xs, us, it = ts.solve_batch(Y, D, return_iters=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            ts.solve_batch(Y, D)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.reps
        itn = it.cpu().numpy()
        rec = dict(mode=mode, batch=B, nw=getattr(ts, "nw", p.Nu), ms_per_call=round(ms, 4),
                   samples_per_s=round(B / ms * 1e3), mean_steps=float(np.mean(np.abs(itn))),
                   infeasible=int(np.sum(itn < 0)), card=name, power_limit=power)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        del ts
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
