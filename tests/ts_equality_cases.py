"""Target-selector problems with pinned outputs (H non-empty) or an integrating plant, shared by
test_target_selector_equality.py (CPU) and test_gpu_target_selector_equality.py (GPU)."""
import numpy as np
import scipy.linalg

from oracle import linear_mpc as om
from oracle import qp as oq

CASES =["cstrs_z", "cdu_small_h2", "cdu_small_h2_ybounds", "cdu_hsel", "cdu_hsel_ybounds", "integrating",
         "integrating_h", "integrating_h_ybounds"]


class EqualityTargetOracle(om.TargetSelectorOracle):
    """The oracle's literal formulation of the target problem (tA, tb, P, G, h of linearMPC.py:229-296), solved by
    eliminating tA w = b through a null-space basis and then the inequality QP of oracle.qp (interior point and
    active-set polish) - the route the oracle takes for output bounds.  The oracle's own input-box route
    (solve_eq_box_qp) cannot reduce a problem with H rows.  An empty null space (as many pinned outputs as inputs)
    leaves the least-squares solution of the equalities.  Raises ValueError when no feasible target exists."""

    def solve(self, ysp, dhats, return_info=False):
        q, h, b = self.changing(ysp, dhats)
        wp = np.linalg.lstsq(self.tA, b, rcond=None)[0]
        Z = scipy.linalg.null_space(self.tA)
        if Z.shape[1]:
            Pr = Z.T @ self.P @ Z
            y, info = oq.solve_general_qp(0.5 * (Pr + Pr.T), Z.T @ (q + self.P @ wp), self.G @ Z, h - self.G @ wp)
        else:
            y, info = np.zeros((0, 1)), {}
        w = wp + Z @ y
        if not np.all(np.isfinite(w)) or not np.max(self.G @ w - h) <= 1e-7 * (1.0 + np.abs(h).max()):
            raise ValueError("EqualityTargetOracle: the target problem is infeasible")
        xs, us = w[:self.Nx], w[self.Nx:]
        return ((xs, us), info) if return_info else (xs, us)


def ts_kwargs(p, H, ylb=None, yub=None):
    return dict(A=p.A, B=p.B, C=p.C, H=H, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs, ulb=p.ulb, uub=p.uub,
                ylb=ylb, yub=yub)


def integrating_plant(with_h, nx=7, nu=3, ny=4, nd=2, seed=11):
    """A with an exact eigenvalue 1 (upper triangular, then a permutation similarity), controllable at it."""
    rng = np.random.default_rng(seed)
    diag = np.concatenate([[1.0], rng.uniform(0.3, 0.9, nx - 1)])
    A = np.triu(0.2 * rng.standard_normal((nx, nx)), 1) + np.diag(diag)
    perm = rng.permutation(nx)
    A = A[np.ix_(perm, perm)]
    B = rng.standard_normal((nx, nu))
    C = rng.standard_normal((ny, nx))
    Bd = rng.standard_normal((nx, nd)) * 0.3
    Cd = np.zeros((ny, nd))
    Cd[0, 0] = 0.5
    H = np.eye(ny)[[0, 2]] if with_h else np.zeros((0, ny))
    return dict(A=A, B=B, C=C, H=H, Bd=Bd, Cd=Cd, usp=0.1 * np.ones((nu, 1)), Rs=1e-3 * np.eye(nu),
                Qs=np.diag(rng.uniform(0.5, 2.0, ny)), ulb=-np.ones((nu, 1)), uub=np.ones((nu, 1)))


def steady_states(kw, n, seed, frac=0.6, dscale=0.3):
    """n steady states (xs0, us0, d) with us0 strictly inside the input box: the set-points ysp = C xs0 + Cd d they
    produce are reachable, whatever rows H pins (with the CDU tuning, set-points drawn at random mostly are not)."""
    A, B, Bd = kw["A"], kw["B"], kw["Bd"]
    nx, nu, nd = B.shape[0], B.shape[1], Bd.shape[1]
    ulb, uub = kw["ulb"][:, 0], kw["uub"][:, 0]
    M = np.hstack([np.eye(nx) - A, -B])
    N = scipy.linalg.null_space(M)
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        d = rng.uniform(-dscale, dscale, nd)
        u0 = 0.5 * (ulb + uub) + frac * 0.5 * (uub - ulb) * rng.uniform(-1.0, 1.0, nu)
        wp = np.linalg.lstsq(M, Bd @ d, rcond=None)[0]
        c = np.linalg.lstsq(N[nx:], u0 - wp[nx:], rcond=1e-10)[0]      # singular at an integrator
        w = wp + N @ c
        if np.all(w[nx:] > ulb + 1e-3) and np.all(w[nx:] < uub - 1e-3):
            out.append((w[:nx], w[nx:], d))
    return out


def case(name, cstrs=None, cdu_small=None, cdu_full=None):
    """(TargetSelector keywords, YSP (n, ny), D (n, nd)) with reachable set-points."""
    from industrial_nnmpc_2021_b200.plants.cdu import NZ
    if name == "cstrs_z":
        p = cstrs
        kw = ts_kwargs(p, np.eye(p.Ny)[list(p.extra["z_indices"])])
    elif name.startswith("cdu_small"):
        p = cdu_small
        kw = ts_kwargs(p, np.eye(p.Ny)[[6, 7]])
    elif name.startswith("cdu_hsel"):
        p = cdu_full
        kw = ts_kwargs(p, np.hstack([np.zeros((NZ, p.Ny - NZ)), np.eye(NZ)]))
    else:
        kw = integrating_plant(with_h=name != "integrating")
        kw.update(ylb=None, yub=None)
    C, Cd = kw["C"], kw["Cd"]
    sts = steady_states(kw, 12, seed=len(name))
    Y0 = np.array([C @ xs + Cd @ d for xs, _, d in sts])
    rng = np.random.default_rng(3)
    # pinned rows get the reachable values; the others a perturbation of them (they only enter the objective)
    YSP = Y0 + 0.2 * rng.standard_normal(Y0.shape) * (np.abs(Y0).max(axis=0) + 1e-3)
    hrows = np.flatnonzero(np.abs(kw["H"]).sum(axis=0))
    YSP[:, hrows] = Y0[:, hrows]
    D = np.array([d for _, _, d in sts])
    if name.endswith("ybounds"):
        span = Y0.max(axis=0) - Y0.min(axis=0)
        ylb, yub = Y0.min(axis=0) - 2.0 * span - 1.0, Y0.max(axis=0) + 2.0 * span + 1.0
        free = [j for j in range(C.shape[0]) if j not in set(hrows)]
        j = free[int(np.argmax(span[free]))]
        yub[j] = np.median(Y0[:, j])              # cuts some optima; a sample the cut makes infeasible is skipped
        kw.update(ylb=ylb[:, None], yub=yub[:, None])
    return kw, YSP, D
