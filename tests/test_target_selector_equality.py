"""Target selector with pinned outputs (H non-empty) or an integrating plant (I - A singular): the host-side null-space
reduction of TargetSelector (CPU only; the handle is never created, the kernel is tested in
test_gpu_target_selector_equality.py).

No reference artefact pins the H rows of tA / tb: the reference code is not in this tree and no fixture covers H != 0.
The rows are checked against their definition (linearMPC.py:254-267: H C xs = H (ysp - Cd dhat)) and against the
oracle's restatement of the same formulation, solved through a null-space basis
(ts_equality_cases.EqualityTargetOracle)."""
import os
import sys

import numpy as np
import pytest


sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ts_equality_cases as tc        # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools", "probes"))
from ts_dual_active_set import dual_active_set        # noqa: E402


@pytest.fixture(scope="module")
def cdu_full_problem():
    from industrial_nnmpc_2021_b200.plants import get_cdu_problem
    return get_cdu_problem(with_scenarios=False)


def host_ts(kw):
    """The product class's host set-up without a GPU handle."""
    from industrial_nnmpc_2021_b200.linearMPC import TargetSelector
    ts = TargetSelector.__new__(TargetSelector)
    for k, v in kw.items():
        setattr(ts, k, v)
    ts.Nx, ts.Nu = kw["B"].shape
    ts.Ny, ts.Nd, ts.Nz = kw["C"].shape[0], kw["Bd"].shape[1], kw["H"].shape[0]
    ts._setup_fixed_matrices()
    return ts


@pytest.fixture(params=tc.CASES)
def eq_case(request, cstrs_problem, cdu_small_problem, cdu_full_problem):
    kw, YSP, D = tc.case(request.param, cstrs_problem, cdu_small_problem, cdu_full_problem)
    return request.param, kw, YSP, D, host_ts(kw)


def test_sizes_of_the_issue_cases(eq_case):
    name, kw, _, _, ts = eq_case
    nw = {"cstrs_z": 0, "cdu_small_h2": 2, "cdu_hsel": 28, "integrating": 3, "integrating_h": 1}
    assert ts.reduced and ts.nw == nw[name.replace("_ybounds", "")]
    assert np.linalg.matrix_rank(ts.tA) == ts.Nx + ts.Nz
    assert ts.mb == ts.Nu + (ts.Ny if kw["ylb"] is not None else 0)


def test_null_space_basis_keeps_the_equalities(eq_case):
    _, _, _, _, ts = eq_case
    assert np.allclose(ts.Z.T @ ts.Z, np.eye(ts.nw), rtol=0, atol=1e-12)
    rng = np.random.default_rng(0)
    for _ in range(5):
        s = rng.standard_normal((ts.Ny + ts.Nd, 1))
        v = rng.standard_normal((ts.nw, 1))
        w = ts.K @ s + ts.Z @ v
        b = ts.tb @ s
        scale = max(np.abs(b).max(), np.abs(ts.tA).max() * np.abs(w).max())
        assert np.max(np.abs(ts.tA @ w - b)) <= 1e-12 * scale


def test_reduced_objective_differs_by_a_constant(eq_case):
    _, _, YSP, D, ts = eq_case
    rng = np.random.default_rng(1)
    for y, d in zip(YSP[:3], D[:3]):
        s = np.concatenate([y, d])[:, None]
        q = ts._setup_changing_matrices(y[:, None], d[:, None])[0]
        f = ts.Fy @ y[:, None] + ts.Fd @ d[:, None] + ts.f0
        gaps, scale = [], 0.0
        for _ in range(4):
            v = rng.standard_normal((ts.nw, 1))
            w = ts.K @ s + ts.Z @ v
            full = (0.5 * w.T @ ts.P @ w + q.T @ w).item()
            red = (0.5 * v.T @ ts.Hr @ v + f.T @ v).item()
            gaps.append(full - red)
            scale = max(scale, abs(full), abs(red), abs((0.5 * w.T @ ts.P @ w).item()))
        assert np.ptp(gaps) <= 1e-9 * max(scale, 1e-12)


def test_reduced_solution_maps_back_to_the_oracle(eq_case):
    """The reduced QP solved by the NumPy restatement of the kernel's dual active-set method, mapped back through
    (K, Z), equals the oracle's (xs, us)-space solve; infeasible samples are infeasible for both."""
    name, kw, YSP, D, ts = eq_case
    ots = tc.EqualityTargetOracle(**kw)
    solved = 0
    for y, d in zip(YSP, D):
        s = np.concatenate([y, d])
        lo, hi = ts.lo0[:, 0] - ts.R @ s, ts.hi0[:, 0] - ts.R @ s
        f = ts.Fy @ y + ts.Fd @ d + ts.f0[:, 0]
        v, it = dual_active_set(ts.Hinv, ts.Abar, ts.AH, ts.Mbar, f, lo, hi, ts.nw)
        try:
            oxs, ous = ots.solve(y[:, None], d[:, None])
        except ValueError:
            assert v is None, name
            continue
        assert v is not None, (name, it)
        w = ts.K @ s + ts.Z @ v
        xs, us = w[:ts.Nx], np.clip(w[ts.Nx:], kw["ulb"][:, 0], kw["uub"][:, 0])
        assert np.max(np.abs(us - ous[:, 0])) <= 1e-6 * max(1.0, np.abs(ous).max())
        assert np.max(np.abs(xs - oxs[:, 0])) <= 1e-5 * max(1.0, np.abs(oxs).max())
        solved += 1
    assert solved >= 4


def test_refusals():
    # an integrator no input reaches: the row of I - A at it and of B are zero, tA loses a rank
    kw = tc.integrating_plant(with_h=False)
    A, B = np.array(kw["A"]), np.array(kw["B"])
    i = int(np.argmin(np.abs(np.diag(A) - 1.0)))
    A[i, :] = 0.0
    A[i, i] = 1.0
    B[i, :] = 0.0
    with pytest.raises(ValueError, match="rank"):
        host_ts(dict(kw, A=A, B=B, ylb=None, yub=None))
    # no input weight and one weighted output for three free inputs: Z'PZ is singular, the target is not unique
    ny = kw["C"].shape[0]
    with pytest.raises(ValueError, match="not unique"):
        host_ts(dict(kw, Rs=np.zeros((3, 3)), Qs=np.diag([1.0] + [0.0] * (ny - 1)), ylb=None, yub=None))
    # more constraint rows than the kernel holds per sample
    rng = np.random.default_rng(2)
    big = dict(kw, C=rng.standard_normal((160, kw["A"].shape[0])), H=np.zeros((0, 160)), Cd=np.zeros((160, 2)),
               Qs=np.eye(160), ylb=-np.ones((160, 1)), yub=np.ones((160, 1)))
    with pytest.raises(NotImplementedError, match="160"):
        host_ts(big)


@pytest.mark.parametrize("ybounds", [False, True])
def test_invertible_plants_without_h_keep_the_elimination(cstrs_problem, cdu_small_problem, ybounds):
    for p in (cstrs_problem, cdu_small_problem):
        ylb, yub = (-5.0 * np.ones((p.Ny, 1)), 5.0 * np.ones((p.Ny, 1))) if ybounds else (None, None)
        ts = host_ts(tc.ts_kwargs(p, p.H, ylb, yub))
        assert not ts.reduced and hasattr(ts, "Gx") and hasattr(ts, "Ht") and not hasattr(ts, "Z")
        assert hasattr(ts, "Ryd") == ybounds
