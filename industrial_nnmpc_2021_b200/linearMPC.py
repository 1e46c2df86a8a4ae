"""Drop-in host-side mirror of the hot path of /root/reference/lib/linearMPC.py.

Same class names, constructor keywords, method signatures and return shapes as the reference;
every QP solve and the closed-loop plant recursion run in the sm_100a kernels of
``csrc/libnnmpc.so`` (C ABI in ``include/nnmpc.h``) instead of ``cvxopt``.  Additive batched
entry points (``solve_batch``, ``OfflineSimulator.generate_batch``) expose the data-parallel
form the GPU is built for.  PyTorch is used only to own device memory and streams.

There is no CPU fallback: constructing a solver without the built library / a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os
import sys
import time

import numpy as np
import scipy.linalg

from . import _lib
from . import condense
from .condense import dlqr, dlqe, c2d          # noqa: F401  (re-exported like the reference module)

DEFAULT_TOL = 1e-9        # stop on true KKT residual ||u - clip(u - (Pu+q))||_inf <= tol
DEFAULT_MAX_ITER = 20000
IPM_MAX_ITER = 200        # interior-point regulators (solver == "ipm") when max_iter is left at its default


def _torch():
    import torch
    return torch


def _device_index(device):
    torch = _torch()
    if not torch.cuda.is_available():
        raise _lib.NnmpcError("no CUDA device visible: this package has no CPU fallback")
    idx = None if device is None else torch.device(device).index
    return torch.cuda.current_device() if idx is None else idx


# ------------------------------------------------------------------------------ stability helpers
def _eigval_eigvec_test(X, Y):
    """linearMPC.py:66-77."""
    vals, vecs = np.linalg.eig(X)
    for vec in vecs[:, np.abs(vals) >= 1.0].T:
        if np.linalg.norm(Y @ vec) <= 1e-8:
            return False
    return True


def assert_detectable(A, Cm):
    assert _eigval_eigvec_test(A, Cm)


def assert_stabilizable(A, B):
    assert _eigval_eigvec_test(A.T, B.T)


class LinearPlantSimulator:
    """x+ = Ax + Bu + Bp p with measurement noise (linearMPC.py:87-131).  Host NumPy, as upstream."""

    def __init__(self, *, A, B, C, Bp, Rv, sample_time, x0):
        self.A, self.B, self.C, self.Bp = A, B, C, Bp
        self.Nx, self.Nu, self.Ny = A.shape[0], B.shape[1], C.shape[0]
        self.measurement_noise_std = np.sqrt(np.diag(Rv)[:, np.newaxis])
        self.sample_time = sample_time
        self.x, self.u, self.p = [x0], [], []
        self.v = [self.measurement_noise_std * np.random.randn(self.Ny, 1)]
        self.y = [self.C @ x0 + self.v[-1]]
        self.t = [0.0]

    def step(self, u, p):
        x = self.A @ self.x[-1] + self.B @ u + self.Bp @ p
        v = self.measurement_noise_std * np.random.randn(self.Ny, 1)
        y = self.C @ x + v
        for lst, val in ((self.x, x), (self.u, u), (self.p, p), (self.v, v), (self.y, y)):
            lst.append(val)
        self.t.append(self.t[-1] + self.sample_time)
        return y


class KalmanFilter:
    """Steady-state Kalman filter (linearMPC.py:133-176); online loop only, host NumPy."""

    def __init__(self, *, A, B, C, Qw, Rv, xprior):
        self.A, self.B, self.C, self.Qw, self.Rv = A, B, C, Qw, Rv
        self.L, _ = dlqe(A, C, Qw, Rv)
        self.xhat, self.xhat_pred, self.y, self.uprev = [xprior], [], [], []

    def solve(self, y, uprev):
        pred = self.A @ self.xhat[-1] + self.B @ uprev
        xhat = pred + self.L @ (y - self.C @ pred)
        self.xhat.append(xhat)
        self.xhat_pred.append(pred)
        self.y.append(y)
        self.uprev.append(uprev)
        return xhat


# ------------------------------------------------------------------------------ target selector
class TargetSelector:
    """Steady-state target problem (linearMPC.py:178-319), solved on the GPU.

        min_(xs,us) |us-usp|^2_Rs + |C xs + Cd dhat - ysp|^2_Qs
        s.t. [I-A, -B; HC, 0][xs; us] = [Bd dhat; H(ysp - Cd dhat)],  ulb <= us <= uub

    ``Nu <= 32``.  With ``H`` empty (both reference examples: cstrs_parameters.py:278, cdu_parameters.py:78) and
    ``I - A`` invertible (any A without an eigenvalue at 1, stable or not), ``xs = Gx us + Gd dhat`` and the problem is
    an exactly equivalent ``Nu``-dimensional QP (see csrc/ts.cu): a box QP solved by a primal active-set method, or -
    with output bounds ``ylb <= C xs + Cd dhat <= yub`` (linearMPC.py:242-248, :284-288; ``Ny + Nu <= 160``) - a QP
    over ``Ny + Nu`` two-sided rows solved by a dual active-set method.
    With ``H`` non-empty (chosen outputs reach their set-points exactly) or an integrating plant (``I - A`` singular)
    the equalities are eliminated through a null-space basis instead, ``[xs; us] = K s + Z v`` with ``s = [ysp; dhat]``
    (``reduced`` is True, operators from ``_setup_reduction``), and the same dual active-set method solves over the
    ``Nu - Nz`` entries of ``v``.  ``tA`` must then have full row rank and the reduced Hessian ``Z'PZ`` must be positive
    definite (a unique target); the constructor refuses other problems.
    An infeasible or stalled solve raises ``NnmpcError`` (cvxopt would report a status).
    """

    def __init__(self, *, A, B, C, H, Bd, Cd, usp, Rs, Qs, ulb, uub, ylb=None, yub=None, device=None):
        self.A, self.B, self.C, self.H, self.Bd, self.Cd, self.Rs, self.Qs = A, B, C, H, Bd, Cd, Rs, Qs
        self.Nx, self.Nu = B.shape
        self.Ny, self.Nd, self.Nz = C.shape[0], Bd.shape[1], H.shape[0]
        self.usp = usp
        self.ysp, self.dhats, self.xs, self.us = [], [], [], []
        self.ulb, self.uub, self.ylb, self.yub = ulb, uub, ylb, yub
        if (ylb is None) != (yub is None):
            ylb = yub = self.ylb = self.yub = None      # the reference uses output bounds only when both are given (:242)
        self._setup_fixed_matrices()
        self._dev = _device_index(device)
        self._handle = None
        self._create()

    def _setup_fixed_matrices(self):
        """Reference attribute names (linearMPC.py:229-274) + the reduced operators."""
        nx, nu, ny = self.Nx, self.Nu, self.Ny
        E = np.vstack([np.eye(nu), -np.eye(nu)])
        self.F = np.vstack([np.eye(ny), -np.eye(ny)])
        if self.ylb is not None and self.yub is not None:           # :242-248
            self.G = np.block([[self.F @ self.C, np.zeros((2 * ny, nu))], [np.zeros((2 * nu, nx)), E]])
            self.f = np.vstack([self.yub, -self.ylb])
            self.e = np.vstack([self.uub, -self.ulb])
            self.h = None
        else:
            self.G = np.hstack([np.zeros((2 * nu, nx)), E])
            self.h = np.vstack([self.uub, -self.ulb])
        self.tA = np.block([[np.eye(nx) - self.A, -self.B], [self.H @ self.C, np.zeros((self.Nz, nu))]])
        self.tb = np.block([[np.zeros((nx, ny)), self.Bd], [self.H, -(self.H @ self.Cd)]])
        self.P = scipy.linalg.block_diag(self.C.T @ (self.Qs @ self.C), self.Rs)
        ImA = np.eye(nx) - self.A
        self.reduced = self.Nz != 0 or np.linalg.cond(ImA) > 1e12
        if self.reduced:
            self._setup_reduction()
            return
        self.Gx = np.linalg.solve(ImA, self.B)
        self.Gd = np.linalg.solve(ImA, self.Bd)
        CG = self.C @ self.Gx
        QsCG = self.Qs @ CG
        Ht = CG.T @ QsCG + self.Rs
        self.Ht = 0.5 * (Ht + Ht.T)
        self.Fy = -QsCG.T                                    # d f / d ysp
        self.Fd = QsCG.T @ (self.C @ self.Gd + self.Cd)      # d f / d dhat
        self.f0 = -(self.Rs @ self.usp)
        if self.ylb is not None and self.yub is not None:
            # operators of the dual active-set solve over the rows Abar = [C Gx; I] (csrc/ts.cu, k_ts_general)
            self.Abar = np.vstack([CG, np.eye(nu)])
            cho = scipy.linalg.cho_factor(self.Ht)
            self.Hinv = scipy.linalg.cho_solve(cho, np.eye(nu))
            self.Hinv = 0.5 * (self.Hinv + self.Hinv.T)
            self.AH = scipy.linalg.cho_solve(cho, self.Abar.T).T
            Mb = self.AH @ self.Abar.T
            self.Mbar = 0.5 * (Mb + Mb.T)
            self.Ryd = self.C @ self.Gd + self.Cd

    def _setup_reduction(self):
        """Null-space reduction of ``tA w = tb s`` (w = [xs; us], s = [ysp; dhat]) for ``H`` non-empty or ``I - A``
        singular, where xs cannot be eliminated through (I - A)^-1.

        ``w = K s + Z v`` with ``K = tA^+ tb`` and ``Z`` an orthonormal basis of null(tA) (both from one SVD), so the
        equalities hold for every ``v`` (``nw = Nu - Nz`` entries).  The reference objective becomes
        ``1/2 v'(Z'PZ)v + f'v + const`` with ``f = Fy ysp + Fd dhat + f0``, and the inequalities become the ``mb`` rows
        ``lo0 - R s <= Abar v <= hi0 - R s``: the output rows ``C Zx v`` with offset ``(C Kx + [0 Cd]) s`` when
        output bounds are given, then the input rows ``Zu v`` with offset ``Ku s``.  The GPU kernel (csrc/ts.cu,
        k_ts_general) solves that QP and reconstructs ``xs = Kx s + Zx v``, ``us = Ku s + Zu v``."""
        nx, nu, ny, nd, nz = self.Nx, self.Nu, self.Ny, self.Nd, self.Nz
        U, sv, Vt = np.linalg.svd(self.tA)
        rank = int(np.sum(sv > max(self.tA.shape) * np.finfo(float).eps * sv[0]))
        if rank < nx + nz:
            raise ValueError(f"TargetSelector: tA = [I-A, -B; HC, 0] has rank {rank} < {nx + nz} rows: the target "
                             "equalities are dependent or contradictory (uncontrollable integrator, or H rows that the "
                             "inputs cannot move independently)")
        self.nw = nu - nz
        self.Z = Vt[rank:].T
        self.K = Vt[:rank].T @ ((U.T @ self.tb) / sv[:, None])
        self.Zx, self.Zu, self.Kx, self.Ku = self.Z[:nx], self.Z[nx:], self.K[:nx], self.K[nx:]
        Hr = self.Z.T @ self.P @ self.Z
        self.Hr = 0.5 * (Hr + Hr.T)
        if self.nw:
            ev = np.linalg.eigvalsh(self.Hr)
            if not ev[0] > 1e-12 * ev[-1]:
                raise ValueError(f"TargetSelector: the reduced Hessian Z'PZ is singular (eigenvalues {ev[0]:.3e} .. "
                                 f"{ev[-1]:.3e}): the target is not unique; weight more outputs in Qs or the inputs in Rs")
        # q(s) = [-C'Qs (ysp - Cd dhat); -Rs usp] (linearMPC.py:276-283) = Qsd s + q0
        CQ = self.C.T @ self.Qs
        Qsd = np.vstack([np.hstack([-CQ, CQ @ self.Cd]), np.zeros((nu, ny + nd))])
        q0 = np.vstack([np.zeros((nx, 1)), -(self.Rs @ self.usp)])
        Fs = self.Z.T @ (self.P @ self.K + Qsd)
        self.Fy, self.Fd, self.f0 = Fs[:, :ny], Fs[:, ny:], self.Z.T @ q0
        if self.ylb is not None and self.yub is not None:
            Ry = self.C @ self.Kx + np.hstack([np.zeros((ny, ny)), self.Cd])
            self.Abar = np.vstack([self.C @ self.Zx, self.Zu])
            self.R = np.vstack([Ry, self.Ku])
            self.lo0, self.hi0 = np.vstack([self.ylb, self.ulb]), np.vstack([self.yub, self.uub])
        else:
            self.Abar, self.R, self.lo0, self.hi0 = self.Zu, self.Ku, self.ulb, self.uub
        self.mb = self.Abar.shape[0]
        if self.mb > 160:
            raise NotImplementedError(f"TargetSelector: {self.mb} constraint rows (Ny + Nu with output bounds) exceed "
                                      "the 160 the GPU solver holds per sample")
        if self.nw:
            cho = scipy.linalg.cho_factor(self.Hr)
            self.Hinv = scipy.linalg.cho_solve(cho, np.eye(self.nw))
            self.Hinv = 0.5 * (self.Hinv + self.Hinv.T)
            self.AH = scipy.linalg.cho_solve(cho, self.Abar.T).T
        else:
            self.Hinv, self.AH = np.zeros((0, 0)), np.zeros((self.mb, 0))
        Mb = self.AH @ self.Abar.T
        self.Mbar = 0.5 * (Mb + Mb.T)

    def _create(self):
        L = _lib.lib()
        hnd = C.c_void_p()
        if self.reduced:
            arrs = [_lib.host(a) for a in (self.Hinv, self.Abar, self.AH, self.Mbar, self.Fy, self.Fd, self.f0, self.R,
                                           self.lo0, self.hi0, self.Kx, self.Ku, self.Zx, self.Zu, self.ulb, self.uub)]
            rc = L.nnmpc_ts_create_reduced(C.byref(hnd), self.Nx, self.Nu, self.Ny, self.Nd, self.nw, self.mb,
                                           *[_lib.hptr(a) if a.size else None for a in arrs], self._dev)
            _lib.check(rc, "nnmpc_ts_create_reduced")
            self._handle = hnd
            return
        arrs = [_lib.host(a) for a in (self.Ht, self.Fy, self.Fd if self.Nd else np.zeros((self.Nu, 1)), self.f0,
                                       self.Gx, self.Gd if self.Nd else np.zeros((self.Nx, 1)), self.ulb, self.uub)]
        rc = L.nnmpc_ts_create(C.byref(hnd), self.Nx, self.Nu, self.Ny, self.Nd, *[_lib.hptr(a) for a in arrs],
                               self._dev)
        _lib.check(rc, "nnmpc_ts_create")
        self._handle = hnd
        if self.ylb is not None and self.yub is not None:
            arrs = [_lib.host(a) for a in (self.Hinv, self.Abar, self.AH, self.Mbar,
                                           self.Ryd if self.Nd else np.zeros((self.Ny, 1)), self.ylb, self.yub)]
            _lib.check(L.nnmpc_ts_set_output_bounds(hnd, *[_lib.hptr(a) for a in arrs]), "nnmpc_ts_set_output_bounds")

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _lib.lib().nnmpc_ts_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_handle"] = None
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self._create()

    def _setup_changing_matrices(self, ysp, dhats):
        """linearMPC.py:276-296 (kept for inspection/tests; the GPU path uses Fy, Fd, f0)."""
        q = np.vstack([-(self.C.T @ (self.Qs @ (ysp - self.Cd @ dhats))), -(self.Rs @ self.usp)])
        if self.h is None:                                          # :284-288
            h = np.vstack([self.f - self.F @ (self.Cd @ dhats), self.e])
        else:
            h = self.h
        return q, h, self.tb @ np.vstack([ysp, dhats])

    def solve_batch(self, YSP, D, return_iters=False):
        """(B,Ny),(B,Nd) -> xs (B,Nx), us (B,Nu).  torch CUDA tensors stay on the device;
        NumPy arrays go through the host entry point."""
        L = _lib.lib()
        if isinstance(YSP, np.ndarray):
            YSP, D = _lib.host(YSP), _lib.host(D)
            Bn = YSP.shape[0]
            xs, us = np.empty((Bn, self.Nx)), np.empty((Bn, self.Nu))
            it = np.empty(Bn, dtype=np.int32)
            rc = L.nnmpc_ts_solve_host(self._handle, Bn, _lib.hptr(YSP), _lib.hptr(D), _lib.hptr(xs), _lib.hptr(us),
                                       _lib.hptr(it))
            _lib.check(rc, "nnmpc_ts_solve_host")
        else:
            torch = _torch()
            YSP, D = YSP.contiguous(), D.contiguous()
            Bn, dv = YSP.shape[0], self._dev
            xs = torch.empty((Bn, self.Nx), dtype=torch.float64, device=YSP.device)
            us = torch.empty((Bn, self.Nu), dtype=torch.float64, device=YSP.device)
            it = torch.empty(Bn, dtype=torch.int32, device=YSP.device)
            rc = L.nnmpc_ts_solve(self._handle, Bn, _lib.dptr(YSP, device=dv), self.Ny, _lib.dptr(D, device=dv), self.Nd,
                                  _lib.dptr(xs, device=dv), _lib.dptr(us, device=dv), _lib.dptr_i32(it, dv),
                                  _lib.stream_ptr(dv))
            _lib.check(rc, "nnmpc_ts_solve")     # asynchronous: a failed sample carries a negative entry in `it`
        return (xs, us, it) if return_iters else (xs, us)

    def solve(self, ysp, dhats):
        """(Ny,1),(Nd,1) -> (xs (Nx,1), us (Nu,1))   (linearMPC.py:298-311)."""
        xs, us = self.solve_batch(np.asarray(ysp, float).reshape(1, -1), np.asarray(dhats, float).reshape(1, -1))
        xs, us = xs.reshape(-1, 1), us.reshape(-1, 1)
        self.xs.append(xs)
        self.us.append(us)
        self.ysp.append(ysp)
        self.dhats.append(dhats)
        return xs, us


# ------------------------------------------------------------------------------ regulator
def _is_factorisation_error(exc):
    """A failed Cholesky of the set-up (scipy / NumPy, or torch.linalg on the GPU set-up path)."""
    if isinstance(exc, np.linalg.LinAlgError):
        return True
    torch = sys.modules.get("torch")
    return torch is not None and isinstance(exc, torch.linalg.LinAlgError)


class DenseQPRegulator:
    """Condensed regulator QP (linearMPC.py:321-517) with a batched GPU solver.

    Keeps the reference attributes (``P, tq, G, tA, tB, Pf, Krep, reparameterize, ulb, uub, x0,
    useq``); ``tA``/``tB``/``G`` are built lazily because the reference's dense forms are huge at
    CDU size.  ``solve(x0)`` has the reference signature; ``solve_batch`` is the data-parallel form.

    Solver parameters (additive): ``rho_scale`` multiplies the default ADMM penalty
    ``0.5 sqrt(lambda_min lambda_max)`` which is spread over the variables proportionally to
    ``diag(P)``; ``alpha`` is the over-relaxation.
    """

    def __init__(self, *, A, B, Q, R, M, N, ulb, uub, rho_scale=1.0, alpha=1.8, tol=DEFAULT_TOL,
                 max_iter=DEFAULT_MAX_ITER, device=None):
        self.A, self.B, self.Q, self.R, self.M, self.N = A, B, Q, R, M, int(N)
        self.ulb, self.uub = ulb, uub
        self.Nx, self.Nu = B.shape
        self.tol, self.max_iter, self.alpha, self.rho_scale = tol, max_iter, alpha, rho_scale
        self.Krep, self.Pf = dlqr(A, B, Q, R, M)                       # :356
        self._reparameterize()
        self.P, self.tq = condense.condensed_hessian(self.A, self.B, self.Q, self.R, self.M, self.Pf, self.N)
        self._tA = self._tB = self._G = None
        # operators the GPU solves with: the QP itself on the box path; its exact image in the original inputs
        # (again a box QP) on the re-parameterised path
        if self.reparameterize:
            self._Pu, self._tqu, self._T, self._S = condense.input_space_operators(self.A, self.B, self.Krep, self.N,
                                                                                 self.P, self.tq)
        else:
            self._Pu, self._tqu, self._T, self._S = self.P, self.tq, None, None
        self.x0, self.useq = [], []
        self.last_info = None
        self._dev = _device_index(device)
        self._handle = None
        self._setup_solver()

    def _reparameterize(self):
        """linearMPC.py:366-382: with an open-loop unstable A the reference optimises v in u = Krep x + v.
        ``A, Q, M, P, tq, G`` keep the reference's (v-space) meaning; the GPU solves the equivalent box QP
        in u (``condense.input_space_operators``), or - where that QP is too ill-conditioned - the v-space
        QP by interior point (``solver``), and ``solve`` returns u, as the reference does after mapping
        back (:507-509)."""
        if np.any(np.abs(np.linalg.eigvals(self.A)) >= 1.0):
            self.A, self.Q, self.M = condense.reparameterize(self.A, self.B, self.Q, self.R, self.M, self.Krep)
            self.reparameterize = True
        else:
            self.reparameterize = False

    # lazily built reference attributes
    @property
    def tA(self):
        if self._tA is None:
            self._tA, self._tB = condense.prediction_matrices(self.A, self.B, self.N)
        return self._tA

    @property
    def tB(self):
        if self._tB is None:
            self._tA, self._tB = condense.prediction_matrices(self.A, self.B, self.N)
        return self._tB

    @property
    def tE(self):
        E = np.vstack([np.eye(self.Nu), -np.eye(self.Nu)])
        return scipy.linalg.block_diag(*([E] * self.N))

    @property
    def tK(self):
        """linearMPC.py:462-463 (re-parameterised path only)."""
        return scipy.linalg.block_diag(*([self.Krep] * self.N)) if self.reparameterize else None

    @property
    def G(self):
        """linearMPC.py:476-482: tE, or tE (tK tB_N + I) = tE T on the re-parameterised path."""
        if self._G is None:
            self._G = self.tE @ self._T if self.reparameterize else self.tE
        return self._G

    def _get_h(self, x0):
        """linearMPC.py:484-493."""
        te = np.tile(np.vstack([self.uub, -self.ulb]), (self.N, 1))
        if self.reparameterize:
            return te - self.tE @ (self._S @ np.asarray(x0, float).reshape(-1, 1))
        return te

    def to_v(self, useq, x0):
        """Input sequence(s) (., n) -> the reference's decision variable v = T^-1 (u - S x0) (identity on the box
        path); with it the reference's objective value is 1/2 v'Pv + (tq x0)'v."""
        U, X0 = np.atleast_2d(np.asarray(useq, float)), np.atleast_2d(np.asarray(x0, float))
        if not self.reparameterize:
            return U
        rhs = (U - X0[:, :self._S.shape[1]] @ self._S.T).T
        return scipy.linalg.solve_triangular(self._T, rhs, lower=True, unit_diagonal=True).T

    @property
    def solver(self):
        """Which GPU solver this regulator uses: "dr" - Douglas-Rachford on the (input-space) box QP, or "ipm" - the
        interior-point method on the stagewise v-space QP (``csrc/ipm.cu``), taken by re-parameterised regulators
        whose input-space Hessian the box path cannot use (its factorisation fails, it has non-finite entries, or its
        condition number is 1e10 or more)."""
        return self._solver

    def _setup_solver(self):
        n = self.N * self.Nu
        if n % 2:
            raise NotImplementedError("N*Nu must be even")
        P, tq = self._Pu, self._tqu
        # A strongly unstable plant makes the input-space image of the v-space Hessian ill-conditioned (cond grows
        # like rho^2N) or numerically indefinite; its QP is then solved in v by the interior-point kernel instead.
        if self.reparameterize and not np.all(np.isfinite(P)):
            return self._setup_ipm()
        # One-time dense linear algebra of the set-up (Cholesky of P, (P + D)^-1, extreme eigenvalues).  The reference
        # does its set-up with NumPy/SciPy on the host (:384-395); at n >= 4096 (CDU horizons x1/x2/x4: n = 4480 /
        # 8960 / 17920, 2 n^3 up to 1.2e13 flop) the same LAPACK-style calls run on the GPU through torch.linalg
        # (cuSOLVER, FP64) so that the set-up stays in seconds.  Library code at set-up time only - no solve goes
        # through it.
        try:
            if n >= 4096 and os.environ.get("NNMPC_SETUP", "gpu") != "host":
                self.Kunc, (lmin, lmax), self.rho_vec, Top, Mtq = self._setup_dense_gpu(P, tq)
            else:
                cho = scipy.linalg.cho_factor(P, lower=True)
                self.Kunc = -scipy.linalg.cho_solve(cho, tq)                # unconstrained law u = Kunc x0
                lmin, lmax = condense.extreme_eigs(P, cho)
                self.rho_vec = self._penalty(P, lmin, lmax)
                Minv = scipy.linalg.inv(P + np.diag(self.rho_vec))
                Minv = 0.5 * (Minv + Minv.T)
                Top, Mtq = Minv * self.rho_vec[None, :], Minv @ tq
        except Exception as exc:
            if self.reparameterize and _is_factorisation_error(exc):
                return self._setup_ipm()
            raise
        self.eig_range = (lmin, lmax)
        if self.reparameterize and not lmax / lmin < 1e10:
            del Top, Mtq
            return self._setup_ipm()
        self._solver = "dr"
        self._nxa_ld = (self.Nx + 1) & ~1

        def pad(Mx):
            if self._nxa_ld == self.Nx:
                return _lib.host(Mx)
            out = np.zeros((Mx.shape[0], self._nxa_ld))
            out[:, :self.Nx] = Mx
            return out
        ops = [_lib.host(P), pad(tq), _lib.host(Top), pad(Mtq), pad(self.Kunc)]
        del Top
        L = _lib.lib()
        hnd = C.c_void_p()
        rc = L.nnmpc_qp_create(C.byref(hnd), n, self._nxa_ld, self.Nu, self.N, *[_lib.hptr(a) for a in ops],
                               float(self.alpha), self._dev)
        _lib.check(rc, "nnmpc_qp_create")
        self._handle = hnd
        rho = _lib.host(self.rho_vec)
        _lib.check(L.nnmpc_qp_set_penalty(hnd, _lib.hptr(rho)), "nnmpc_qp_set_penalty")

    def _setup_ipm(self):
        """Interior-point regulator (nnmpc_qp_create_ipm) on the stagewise v-space QP of the re-parameterised plant:
        stage weights ``Q, R, M`` (v-space, as held after ``_reparameterize``), dynamics ``A = A_open + B Krep``,
        terminal weight ``Pf`` and bounds on ``u = Krep x + v``."""
        nxa, nu = self.Nx, self.Nu
        self._nxa_ld = (nxa + 1) & ~1
        if self._nxa_ld > 64 or nu > 32:
            raise NotImplementedError(
                f"re-parameterised regulator with Nxa = {nxa}, Nu = {nu}: the input-space box QP is too ill-conditioned "
                "for the Douglas-Rachford path, and the interior-point solver holds at most Nxa = 64 states (after "
                "padding to an even count) and Nu = 32 inputs")
        if not hasattr(self, "eig_range"):
            self.eig_range = (float("nan"), float("nan"))
        ld = self._nxa_ld

        def pad(Mx, rows, cols):
            out = np.zeros((rows, cols))
            out[:Mx.shape[0], :Mx.shape[1]] = Mx
            return out
        ops = [pad(self.A, ld, ld), pad(self.B, ld, nu), pad(self.Q, ld, ld), _lib.host(self.R), pad(self.M, ld, nu),
               pad(self.Pf, ld, ld), pad(self.Krep, nu, ld)]
        L = _lib.lib()
        hnd = C.c_void_p()
        rc = L.nnmpc_qp_create_ipm(C.byref(hnd), ld, nu, self.N, *[_lib.hptr(a) for a in ops], self._dev)
        _lib.check(rc, "nnmpc_qp_create_ipm")
        self._handle = hnd
        self._solver = "ipm"
        if self.max_iter == DEFAULT_MAX_ITER:      # the Douglas-Rachford budget; an interior point needs tens
            self.max_iter = IPM_MAX_ITER

    def _penalty(self, P, lmin, lmax):
        """ADMM penalty vector: 0.5 sqrt(lmin lmax) (swept on the CDU closed loop, 0.28 .. 1.1, B200 round 1ae) spread
        over the variables proportionally to diag(P)."""
        dP = np.diag(P)
        return 0.5 * np.sqrt(lmin * lmax) * self.rho_scale * dP / np.exp(np.mean(np.log(dP)))

    def _setup_dense_gpu(self, P, tq):
        torch = _torch()
        dev = torch.device("cuda", self._dev)
        with torch.no_grad():
            Pd = torch.as_tensor(P, dtype=torch.float64, device=dev)
            tqd = torch.as_tensor(tq, dtype=torch.float64, device=dev)
            Lc = torch.linalg.cholesky(Pd)
            Kunc = -torch.cholesky_solve(tqd, Lc)
            # extreme eigenvalues: power iteration on P and on P^-1 (two triangular solves per apply)
            g = torch.Generator(device=dev).manual_seed(0)
            v = torch.randn((P.shape[0], 1), dtype=torch.float64, device=dev, generator=g)
            w = v.clone()
            lmax = lmin_inv = 0.0
            ref = (0.0, 0.0)
            for it in range(3000):
                v = Pd @ v
                lmax = float(torch.linalg.vector_norm(v))
                v /= lmax
                w = torch.cholesky_solve(w, Lc)
                lmin_inv = float(torch.linalg.vector_norm(w))
                w /= lmin_inv
                if it % 20 == 19:       # both estimates grow monotonically: stop when 20 more applies add < 1e-5
                    if lmax - ref[0] <= 1e-5 * lmax and lmin_inv - ref[1] <= 1e-5 * lmin_inv:
                        break
                    ref = (lmax, lmin_inv)
            lmin = 1.0 / lmin_inv
            rho = self._penalty(P, lmin, lmax)
            rhod = torch.as_tensor(rho, dtype=torch.float64, device=dev)
            Minv = torch.cholesky_inverse(torch.linalg.cholesky(Pd + torch.diag(rhod)))
            del Pd, Lc
            Minv = 0.5 * (Minv + Minv.T)
            Mtq = (Minv @ tqd).cpu().numpy()
            Top = (Minv * rhod[None, :]).cpu().numpy()
            return Kunc.cpu().numpy(), (lmin, lmax), rho, Top, Mtq

    def __del__(self):
        try:
            if getattr(self, "_qp_engine", None):
                _lib.lib().nnmpc_sim_destroy(self._qp_engine)
                self._qp_engine = None
            if getattr(self, "_handle", None):
                _lib.lib().nnmpc_qp_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_handle"] = None
        d.pop("_qp_engine", None)
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self._setup_solver()

    # ---- batched solve -------------------------------------------------------------------
    def _batch_engine(self, precision, slots):
        """QP-only engine handle (no target selector, no plant) behind ``solve_batch(precision=...)``."""
        eng = getattr(self, "_qp_engine", None)
        L = _lib.lib()
        if eng is None:
            hnd = C.c_void_p()
            rc = L.nnmpc_sim_create(C.byref(hnd), self._handle, None, self._nxa_ld - self.Nu, self.Nu, 0, 0, None, self._dev)
            _lib.check(rc, "nnmpc_sim_create")
            eng = self._qp_engine = hnd
        _lib.check(L.nnmpc_sim_set_precision(eng, _lib.PRECISION[precision]), "nnmpc_sim_set_precision")
        _lib.check(L.nnmpc_sim_set_slots(eng, int(slots)), "nnmpc_sim_set_slots")
        return eng

    def solve_batch(self, X0, LB=None, UB=None, *, warm_state=None, tol=None, max_iter=None, return_info=True,
                    out=None, precision=None, slots=16384):
        """Solve B regulator QPs.

        ``precision`` (CUDA-tensor form): None - the lock-step FP64 solver (supports ``warm_state``); "mixed" / "f64"
        - cold solves through the continuously batched engine (``nnmpc_sim_solve_qps``): ``slots`` QPs iterate
        concurrently, a finished slot takes the next QP, iterations run on the tcgen05 fp16-increment tier with
        INT8-exact anchors and KKT checks ("mixed") or in FP64.

        ``out`` (NumPy form only): dict of preallocated result arrays ``U (B,n), cost (B,), kkt (B,), iters (B,)
        int32`` - e.g. pinned host memory - written in place.

        X0 (B,Nxa); LB, UB (B,Nu) per-sample stage bounds (default: this object's ulb/uub).
        Returns U (B,n) in deviation variables and, with ``return_info``, dict(cost, kkt, iters,
        maxiter_hit).  CUDA tensors in -> CUDA tensors out (no copies); NumPy in -> NumPy out via
        the host entry point.  ``warm_state`` (CUDA (B,n) tensor) carries the solver state between
        calls: pass the same tensor again to warm start.
        """
        L = _lib.lib()
        tol = self.tol if tol is None else tol
        max_iter = self.max_iter if max_iter is None else max_iter
        n = self.N * self.Nu
        if isinstance(X0, np.ndarray) and precision is not None:
            # host buffers through the engine form: copies in, device solve, copies out (into ``out`` when given)
            torch = _torch()
            dev = torch.device("cuda", self._dev)
            up = lambda a: None if a is None else torch.from_numpy(_lib.host(a)).to(dev, non_blocking=True)
            Ud, info = self.solve_batch(up(X0), up(LB), up(UB), tol=tol, max_iter=max_iter, precision=precision, slots=slots)
            if out is None:
                res = (Ud.cpu().numpy(), {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in info.items()})
            else:
                for k, v in (("U", Ud), ("cost", info["cost"]), ("kkt", info["kkt"]), ("iters", info["iters"])):
                    torch.from_numpy(out[k]).copy_(v, non_blocking=True)
                torch.cuda.synchronize(dev)
                res = (out["U"], dict(cost=out["cost"], kkt=out["kkt"], iters=out["iters"], maxiter_hit=info["maxiter_hit"]))
            self.last_info = res[1]
            return res if return_info else res[0]
        if isinstance(X0, np.ndarray):
            Bn = X0.shape[0]
            X0p = np.zeros((Bn, self._nxa_ld))
            X0p[:, :self.Nx] = X0
            LB = np.tile(self.ulb.reshape(1, -1), (Bn, 1)) if LB is None else LB
            UB = np.tile(self.uub.reshape(1, -1), (Bn, 1)) if UB is None else UB
            LB, UB = _lib.host(LB), _lib.host(UB)
            if tuple(LB.shape) != (Bn, self.Nu) or tuple(UB.shape) != (Bn, self.Nu):
                raise ValueError("LB / UB must have shape (B, Nu)")
            if out is None:
                U, cost, kkt = np.empty((Bn, n)), np.empty(Bn), np.empty(Bn)
                iters = np.empty(Bn, dtype=np.int32)
            else:
                U, cost, kkt, iters = out["U"], out["cost"], out["kkt"], out["iters"]
                for a, shp, dt in ((U, (Bn, n), np.float64), (cost, (Bn,), np.float64), (kkt, (Bn,), np.float64),
                                   (iters, (Bn,), np.int32)):
                    if tuple(a.shape) != shp or a.dtype != dt or not a.flags["C_CONTIGUOUS"]:
                        raise ValueError("out arrays must be C-contiguous U (B,n), cost (B,), kkt (B,) float64 and iters (B,) int32")
            rc = L.nnmpc_qp_solve_host(self._handle, Bn, _lib.hptr(X0p), _lib.hptr(LB), _lib.hptr(UB), _lib.hptr(U),
                                       _lib.hptr(cost), _lib.hptr(kkt), _lib.hptr(iters), float(tol), int(max_iter))
            warned = _lib.check(rc, "nnmpc_qp_solve_host")
        else:
            torch = _torch()
            dev = X0.device
            Bn = X0.shape[0]
            if X0.shape[1] != self._nxa_ld:
                X0p = torch.zeros((Bn, self._nxa_ld), dtype=torch.float64, device=dev)
                X0p[:, :self.Nx] = X0
            else:
                X0p = X0.contiguous()
            if LB is None:
                LB = torch.as_tensor(self.ulb.reshape(1, -1), device=dev).repeat(Bn, 1)
            if UB is None:
                UB = torch.as_tensor(self.uub.reshape(1, -1), device=dev).repeat(Bn, 1)
            LB, UB = LB.contiguous(), UB.contiguous()
            if tuple(LB.shape) != (Bn, self.Nu) or tuple(UB.shape) != (Bn, self.Nu):
                raise ValueError("LB / UB must have shape (B, Nu)")
            U = torch.empty((Bn, n), dtype=torch.float64, device=dev)
            cost = torch.empty(Bn, dtype=torch.float64, device=dev)
            kkt = torch.empty(Bn, dtype=torch.float64, device=dev)
            iters = torch.empty(Bn, dtype=torch.int32, device=dev)
            warm = 0
            if warm_state is not None:
                if tuple(warm_state.shape) != (Bn, n) or not warm_state.is_contiguous():
                    raise ValueError("warm_state must be a contiguous (B, n) CUDA tensor")
                warm = 1 if getattr(warm_state, "_nnmpc_valid", False) else 0
            dv = self._dev
            if precision is not None:
                if precision not in _lib.PRECISION:
                    raise ValueError(f"precision must be one of {sorted(_lib.PRECISION)} or None")
                if warm_state is not None:
                    raise ValueError("warm_state is a feature of the lock-step solver (precision=None)")
                eng = self._batch_engine(precision, slots)
                rc = L.nnmpc_sim_solve_qps(eng, Bn, _lib.dptr(X0p, device=dv), _lib.dptr(LB, device=dv),
                                           _lib.dptr(UB, device=dv), _lib.dptr(U, device=dv), _lib.dptr(cost, device=dv),
                                           _lib.dptr(kkt, device=dv), _lib.dptr_i32(iters, dv), float(tol), int(max_iter),
                                           _lib.stream_ptr(dv))
                warned = _lib.check(rc, "nnmpc_sim_solve_qps")
                info = dict(cost=cost, kkt=kkt, iters=iters, maxiter_hit=warned)
                self.last_info = info
                return (U, info) if return_info else U
            rc = L.nnmpc_qp_solve(self._handle, Bn, _lib.dptr(X0p, device=dv), _lib.dptr(LB, device=dv),
                                  _lib.dptr(UB, device=dv), _lib.dptr(U, device=dv), _lib.dptr(warm_state, device=dv),
                                  warm, _lib.dptr(cost, device=dv), _lib.dptr(kkt, device=dv), _lib.dptr_i32(iters, dv),
                                  float(tol), int(max_iter), _lib.stream_ptr(dv))
            warned = _lib.check(rc, "nnmpc_qp_solve")
            if warm_state is not None:
                warm_state._nnmpc_valid = True
        info = dict(cost=cost, kkt=kkt, iters=iters, maxiter_hit=warned)
        self.last_info = info
        return (U, info) if return_info else U

    def solve(self, x0):
        """(Nxa,1) -> useq (N*Nu,1), as linearMPC.py:495-512 (bounds = current self.ulb/self.uub)."""
        x0 = np.asarray(x0, float)
        U = self.solve_batch(x0.reshape(1, -1), self.ulb.reshape(1, -1), self.uub.reshape(1, -1), return_info=False)
        useq = U.reshape(-1, 1)
        self.x0.append(x0)
        self.useq.append(useq)
        return useq


# ------------------------------------------------------------------------------ controller glue
class LinearMPCController:
    """Kalman filter + target selector + regulator (linearMPC.py:519-701)."""

    def __init__(self, *, A, B, C, H, Qwx, Qwd, Rv, xprior, dprior, Rs, Qs, Bd, Cd, usp, uprev, Q, R, S, ulb, uub,
                 N, device=None):
        self.A, self.B, self.C, self.H = A, B, C, H
        self.Qwx, self.Qwd, self.Rv, self.xprior, self.dprior = Qwx, Qwd, Rv, xprior, dprior
        self.Rs, self.Qs, self.Bd, self.Cd, self.usp = Rs, Qs, Bd, Cd, usp
        self.uprev = uprev
        self.useq = np.tile(uprev, (N, 1))
        self.Q, self.R, self.S, self.ulb, self.uub, self.N = Q, R, S, ulb, uub, N
        self.Nx, self.Nu, self.Ny, self.Nd = A.shape[0], B.shape[1], C.shape[0], Bd.shape[1]
        self.filter = LinearMPCController.setup_filter(A=A, B=B, C=C, Bd=Bd, Cd=Cd, Qwx=Qwx, Qwd=Qwd, Rv=Rv,
                                                       xprior=xprior, dprior=dprior)
        self.target_selector = LinearMPCController.setup_target_selector(
            A=A, B=B, C=C, H=H, Bd=Bd, Cd=Cd, usp=usp, Qs=Qs, Rs=Rs, ulb=ulb, uub=uub, device=device)
        self.regulator = LinearMPCController.setup_regulator(A=A, B=B, Q=Q, R=R, S=S, N=N, ulb=ulb, uub=uub,
                                                             device=device)
        _, _, self.Qaug, self.Raug, self.Maug = LinearMPCController.get_augmented_matrices_for_regulator(A, B, Q, R, S)
        self.average_stage_costs = [np.zeros((1, 1))]
        self.computation_times = []

    @staticmethod
    def setup_filter(A, B, C, Bd, Cd, Qwx, Qwd, Rv, xprior, dprior):
        Aaug, Baug, Caug, Qwaug = LinearMPCController.get_augmented_matrices_for_filter(A, B, C, Bd, Cd, Qwx, Qwd)
        return KalmanFilter(A=Aaug, B=Baug, C=Caug, Qw=Qwaug, Rv=Rv, xprior=np.concatenate((xprior, dprior)))

    @staticmethod
    def setup_target_selector(A, B, C, H, Bd, Cd, usp, Qs, Rs, ulb, uub, device=None):
        return TargetSelector(A=A, B=B, C=C, H=H, Bd=Bd, Cd=Cd, usp=usp, Rs=Rs, Qs=Qs, ulb=ulb, uub=uub,
                              device=device)

    @staticmethod
    def setup_regulator(A, B, Q, R, S, N, ulb, uub, device=None, **solver_kwargs):
        Aaug, Baug, Qaug, Raug, Maug = LinearMPCController.get_augmented_matrices_for_regulator(A, B, Q, R, S)
        return DenseQPRegulator(A=Aaug, B=Baug, Q=Qaug, R=Raug, N=N, M=Maug, ulb=ulb, uub=uub, device=device,
                                **solver_kwargs)

    @staticmethod
    def get_augmented_matrices_for_filter(A, B, C, Bd, Cd, Qwx, Qwd):
        """Integrating-disturbance augmentation (linearMPC.py:606-624)."""
        nx, nu, nd = A.shape[0], B.shape[1], Bd.shape[1]
        Aaug = np.block([[A, Bd], [np.zeros((nd, nx)), np.eye(nd)]])
        Baug = np.vstack([B, np.zeros((nd, nu))])
        Caug = np.hstack([C, Cd])
        Qwaug = scipy.linalg.block_diag(Qwx, Qwd)
        assert_detectable(Aaug, Caug)
        return Aaug, Baug, Caug, Qwaug

    @staticmethod
    def get_augmented_matrices_for_regulator(A, B, Q, R, S):
        """Rate-of-change augmentation with state [x; uprev] (linearMPC.py:626-644)."""
        nx, nu = B.shape
        Aaug = np.zeros((nx + nu, nx + nu))
        Aaug[:nx, :nx] = A
        Baug = np.vstack([B, np.eye(nu)])
        Qaug = scipy.linalg.block_diag(Q, S)
        Raug = R + S
        Maug = np.vstack([np.zeros((nx, nu)), -S])
        return Aaug, Baug, Qaug, Raug, Maug

    def control_law(self, ysp, y):
        """Measurement -> control input (linearMPC.py:646-669); times only the regulator solve."""
        xhat, dhat = LinearMPCController.get_state_estimates(self.filter, y, self.uprev, self.Nx)
        xs, us = LinearMPCController.get_target_pair(self.target_selector, ysp, dhat)
        tstart = time.time()
        self.useq = LinearMPCController.get_control_sequence(self.regulator, xhat, self.uprev, xs, us, self.ulb,
                                                             self.uub)
        tend = time.time()
        avg_ell = LinearMPCController.get_updated_average_stage_cost(
            xhat, self.uprev, xs, us, self.useq[0:self.Nu, :], self.Qaug, self.Raug, self.Maug,
            self.average_stage_costs[-1], len(self.average_stage_costs))
        self.average_stage_costs.append(avg_ell)
        self.uprev = self.useq[0:self.Nu, :]
        self.computation_times.append(tend - tstart)
        return self.uprev

    @staticmethod
    def get_state_estimates(filter, y, uprev, Nx):
        return np.split(filter.solve(y, uprev), [Nx])

    @staticmethod
    def get_target_pair(target_selector, ysp, dhat):
        return target_selector.solve(ysp, dhat)

    @staticmethod
    def get_control_sequence(regulator, x, uprev, xs, us, ulb, uub):
        """linearMPC.py:682-689: bounds shifted by us, x0 in deviation variables, us added back."""
        regulator.ulb = ulb - us
        regulator.uub = uub - us
        x0 = np.concatenate((x - xs, uprev - us))
        return regulator.solve(x0) + np.tile(us, (regulator.N, 1))

    @staticmethod
    def get_updated_average_stage_cost(x, uprev, xs, us, u, Qaug, Raug, Maug, average_stage_cost, time_index):
        """Running mean of x'Qx + u'Ru + 2x'Mu in deviation variables (linearMPC.py:691-701)."""
        xa = np.concatenate((x - xs, uprev - us), axis=0)
        du = u - us
        ell = xa.T @ (Qaug @ xa) + du.T @ (Raug @ du) + xa.T @ (Maug @ du) + du.T @ (Maug.T @ xa)
        return (average_stage_cost * (time_index - 1) + ell) / time_index


def online_simulation(plant, controller, *, setpoints=None, disturbances=None, Nsim=None, stdout_filename=None):
    """Sequential closed loop with a plant object (linearMPC.py:703-718)."""
    out = open(stdout_filename, "w") if stdout_filename else None
    measurement = plant.y[0]
    for i, (sp, dist) in enumerate(zip(setpoints[..., np.newaxis], disturbances[..., np.newaxis])):
        if i >= Nsim:
            break
        u = controller.control_law(sp, measurement)
        if out:
            print(f"Simulation Step:{i}\nComputation time:{controller.computation_times[-1]}", file=out)
        measurement = plant.step(u, dist)
    if out:
        out.close()
    return plant


# ------------------------------------------------------------------------------ offline data generation
def _save_training_data(dictionary, filename):
    """H5pyTool.save_training_data (lib/python_utils.py:53-58): one dataset per key.  h5py is
    used when importable; otherwise the same keys go into ``<filename>.npz``."""
    try:
        import h5py
    except ImportError:
        np.savez(filename + ".npz", **dictionary)
        return filename + ".npz"
    with h5py.File(filename, "w") as f:
        for k, v in dictionary.items():
            f.create_dataset(k, data=v)
    return filename


def load_training_data(filename):
    """H5pyTool.load_training_data (lib/python_utils.py:43-50) for either container."""
    npz, h5 = filename + ".npz", filename
    have_npz, have_h5 = os.path.exists(npz), os.path.exists(h5)
    if have_npz and (not have_h5 or os.path.getmtime(npz) >= os.path.getmtime(h5)):    # the newer container wins
        with np.load(npz) as z:
            return {k: np.asarray(z[k]) for k in z.files}
    import h5py
    with h5py.File(filename, "r") as f:
        return {k: np.asarray(f.get(k)) for k in f.keys()}


class ClosedLoopEngine:
    """Owns the nnmpc_sim handle for one (regulator, target selector, plant) triple."""

    def __init__(self, regulator, target_selector, A, B, Bd, precision=None, tail_rows=None, slots=None):
        """``precision``: "f64" (every iteration an FP64 tensor-core GEMM) or "mixed" (tcgen05 fp16
        increments with FP64-accurate anchors; every result still passes an FP64-accurate KKT check).  Default: the
        environment variable NNMPC_PRECISION, else "mixed"."""
        if regulator._dev != target_selector._dev:
            raise ValueError("regulator and target selector live on different devices")
        self.regulator, self.target_selector = regulator, target_selector
        self.nx, self.nu = B.shape
        self.nd = Bd.shape[1]
        self.ny = target_selector.Ny
        self._dev = regulator._dev
        L = _lib.lib()
        ABd = _lib.host(np.hstack([A, B, Bd]))
        hnd = C.c_void_p()
        rc = L.nnmpc_sim_create(C.byref(hnd), regulator._handle, target_selector._handle, self.nx, self.nu, self.nd,
                                self.ny, _lib.hptr(ABd), self._dev)
        _lib.check(rc, "nnmpc_sim_create")
        self._handle = hnd
        self.set_precision(precision or os.environ.get("NNMPC_PRECISION", "mixed"))
        slots = os.environ.get("NNMPC_SLOTS") if slots is None else slots
        if slots is not None:
            self.set_slots(slots)
        if os.environ.get("NNMPC_CADENCE"):
            _lib.check(L.nnmpc_sim_set_cadence(self._handle, int(os.environ["NNMPC_CADENCE"])), "nnmpc_sim_set_cadence")
        if os.environ.get("NNMPC_EXACT_GEMM"):      # "dmma" = FP64 tensor cores, "int8" (default) = sliced INT8 tcgen05
            mode = {"dmma": 0, "int8": 1}[os.environ["NNMPC_EXACT_GEMM"]]
            _lib.check(L.nnmpc_sim_set_exact_gemm(self._handle, mode), "nnmpc_sim_set_exact_gemm")
        if os.environ.get("NNMPC_T2_EVERY"):        # second fp16 operator term every k-th pass (0 = fused into every pass)
            _lib.check(L.nnmpc_sim_set_second_term_cadence(self._handle, int(os.environ["NNMPC_T2_EVERY"])),
                       "nnmpc_sim_set_second_term_cadence")
        if os.environ.get("NNMPC_T2_FACTOR"):       # late-phase threshold of the one-term tensor-core tiles (0 = off)
            _lib.check(L.nnmpc_sim_set_one_term_threshold(self._handle, float(os.environ["NNMPC_T2_FACTOR"])),
                       "nnmpc_sim_set_one_term_threshold")
        tail_rows = os.environ.get("NNMPC_TAIL_ROWS") if tail_rows is None else tail_rows
        if tail_rows is not None:     # mixed mode: live rows at or below which a call finishes in FP64 (-1 = automatic)
            _lib.check(L.nnmpc_sim_set_tail_rows(self._handle, int(tail_rows)), "nnmpc_sim_set_tail_rows")

    def set_second_term_cadence(self, every):
        """Mixed precision: the second fp16 operator term is delivered every ``every``-th tensor-core pass (default 8);
        0 = both terms in every pass."""
        _lib.check(_lib.lib().nnmpc_sim_set_second_term_cadence(self._handle, int(every)), "nnmpc_sim_set_second_term_cadence")

    def set_slots(self, slots):
        """Most trajectories advanced concurrently; a run with more chunks queues the rest (continuous batching)."""
        _lib.check(_lib.lib().nnmpc_sim_set_slots(self._handle, int(slots)), "nnmpc_sim_set_slots")
        self.slots = int(slots)

    def set_precision(self, precision):
        if precision not in _lib.PRECISION:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISION)}")
        _lib.check(_lib.lib().nnmpc_sim_set_precision(self._handle, _lib.PRECISION[precision]),
                   "nnmpc_sim_set_precision")
        self.precision = precision

    def stats(self):
        """Cumulative solver work since construction: row-iterations, FP64 anchors, exact KKT checks, QPs."""
        out = (C.c_longlong * 4)()
        _lib.check(_lib.lib().nnmpc_sim_stats(self._handle, out), "nnmpc_sim_stats")
        act = (C.c_longlong * 2)()
        _lib.check(_lib.lib().nnmpc_sim_active_stats(self._handle, act), "nnmpc_sim_active_stats")
        til = (C.c_longlong * 3)()
        _lib.check(_lib.lib().nnmpc_sim_tile_stats(self._handle, til), "nnmpc_sim_tile_stats")
        return dict(row_iterations=out[0], anchors=out[1], exact_checks=out[2], qps=out[3],
                    qps_with_active_bounds=act[0], active_bounds=act[1], tiles_one_term=til[0], tiles_two_terms=til[1],
                    tiles_second_term_delivery=til[2])

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _lib.lib().nnmpc_sim_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    def _check_out(self, out, Bn, T, kind):
        shapes = dict(x=(Bn, T, self.nx), uprev=(Bn, T, self.nu), xs=(Bn, T, self.nx), us=(Bn, T, self.nu),
                      u=(Bn, T, self.nu), iters=(Bn, T), kkt=(Bn, T))
        for k, shp in shapes.items():
            a = out.get(k)
            if not isinstance(a, kind) or tuple(a.shape) != shp:
                raise ValueError(f"out[{k!r}] must be a {kind.__name__} of shape {shp}")
            want = "int32" if k == "iters" else "float64"
            if str(a.dtype).replace("torch.", "") != want:
                raise ValueError(f"out[{k!r}] must have dtype {want}")
            contiguous = a.flags["C_CONTIGUOUS"] if isinstance(a, np.ndarray) else a.is_contiguous()
            if not contiguous:
                raise ValueError(f"out[{k!r}] must be contiguous")
        return {k: out[k] for k in shapes}

    def run(self, x0, uprev0, setpoints, disturbances, *, tol=None, max_iter=None, resume=False, out=None,
            capture=False):
        """Advance B trajectories T steps.

        ``capture=True`` additionally returns ``useq`` (B,T,N*Nu) - the whole optimal input sequence of
        every regulator QP, target added back, i.e. what ``get_control_sequence`` returns upstream
        (linearMPC.py:689) - and ``cost`` (B,T), the optimal value in deviation variables.  Meant for
        parity tests / diagnostics (N*Nu doubles per sample).

        ``resume=True`` says these are the same B trajectories as in the previous call (a long
        trajectory advanced slab by slab): step 0 is then warm-started from the kept solver
        state.  ``out`` may hold preallocated result arrays (e.g. pinned host memory) under the
        keys x, uprev, xs, us, u, iters, kkt.

        setpoints (B,T,Ny), disturbances (B,T,Nd); x0 (B,Nx), uprev0 (B,Nu) (or column vectors,
        broadcast to all trajectories).  NumPy in -> dict of NumPy arrays (host entry point, copies
        inside the call); CUDA tensors in -> dict of CUDA tensors.  Keys as the reference's h5
        files: x, uprev, xs, us, u with shapes (B,T,.), plus iters, kkt (B,T) and x_final/uprev_final.
        """
        L = _lib.lib()
        reg = self.regulator
        tol = reg.tol if tol is None else tol
        max_iter = reg.max_iter if max_iter is None else max_iter
        Bn, T = setpoints.shape[0], setpoints.shape[1]
        nx, nu = self.nx, self.nu
        if tuple(setpoints.shape) != (Bn, T, self.ny) or tuple(disturbances.shape) != (Bn, T, self.nd):
            raise ValueError(f"setpoints / disturbances must have shapes (B,T,{self.ny}) / (B,T,{self.nd})")
        if capture and isinstance(setpoints, np.ndarray):      # the capture sinks live on the device entry point
            torch = _torch()
            f64 = dict(dtype=torch.float64, device=torch.device("cuda", self._dev))
            res = self.run(torch.as_tensor(np.asarray(x0, float), **f64), torch.as_tensor(np.asarray(uprev0, float), **f64),
                           torch.as_tensor(_lib.host(setpoints), **f64), torch.as_tensor(_lib.host(disturbances), **f64),
                           tol=tol, max_iter=max_iter, resume=resume, capture=True)
            return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in res.items()}
        if isinstance(setpoints, np.ndarray):
            sp, dist = _lib.host(setpoints), _lib.host(disturbances)
            xio = _lib.host(np.broadcast_to(np.asarray(x0, float).reshape(-1, nx), (Bn, nx))).copy()
            uio = _lib.host(np.broadcast_to(np.asarray(uprev0, float).reshape(-1, nu), (Bn, nu))).copy()
            res = dict(x=np.empty((Bn, T, nx)), uprev=np.empty((Bn, T, nu)), xs=np.empty((Bn, T, nx)),
                       us=np.empty((Bn, T, nu)), u=np.empty((Bn, T, nu)), iters=np.empty((Bn, T), dtype=np.int32),
                       kkt=np.empty((Bn, T))) if out is None else self._check_out(out, Bn, T, np.ndarray)
            out = dict(res)
            rc = L.nnmpc_sim_run_host(self._handle, Bn, T, _lib.hptr(xio), _lib.hptr(uio), _lib.hptr(sp),
                                      _lib.hptr(dist), *[_lib.hptr(out[k]) for k in ("x", "uprev", "xs", "us", "u",
                                                                                      "iters", "kkt")],
                                      float(tol), int(max_iter), int(bool(resume)))
            out["maxiter_hit"] = _lib.check(rc, "nnmpc_sim_run_host")
        else:
            torch = _torch()
            dev = setpoints.device
            sp, dist = setpoints.contiguous(), disturbances.contiguous()
            f64 = dict(dtype=torch.float64, device=dev)
            xio = torch.as_tensor(x0, **f64).reshape(-1, nx).expand(Bn, nx).contiguous().clone()
            uio = torch.as_tensor(uprev0, **f64).reshape(-1, nu).expand(Bn, nu).contiguous().clone()
            res = dict(x=torch.empty((Bn, T, nx), **f64), uprev=torch.empty((Bn, T, nu), **f64),
                       xs=torch.empty((Bn, T, nx), **f64), us=torch.empty((Bn, T, nu), **f64),
                       u=torch.empty((Bn, T, nu), **f64),
                       iters=torch.empty((Bn, T), dtype=torch.int32, device=dev),
                       kkt=torch.empty((Bn, T), **f64)) if out is None else self._check_out(out, Bn, T, torch.Tensor)
            out = dict(res)
            dv = self._dev
            if sp.dtype != torch.float64 or dist.dtype != torch.float64:
                raise ValueError("setpoints / disturbances must be float64 tensors")
            if capture:
                out["useq"] = torch.empty((Bn, T, reg.N * nu), **f64)
                out["cost"] = torch.empty((Bn, T), **f64)
                _lib.check(L.nnmpc_sim_set_capture(self._handle, _lib.dptr(out["useq"], device=dv),
                                                   _lib.dptr(out["cost"], device=dv)), "nnmpc_sim_set_capture")
            try:
                rc = L.nnmpc_sim_run(self._handle, Bn, T, _lib.dptr(xio, device=dv), _lib.dptr(uio, device=dv),
                                     _lib.dptr(sp, device=dv), _lib.dptr(dist, device=dv),
                                     *[_lib.dptr(out[k], device=dv) for k in ("x", "uprev", "xs", "us", "u")],
                                     _lib.dptr_i32(out["iters"], dv), _lib.dptr(out["kkt"], device=dv),
                                     float(tol), int(max_iter), int(bool(resume)), _lib.stream_ptr(dv))
            finally:
                if capture:
                    L.nnmpc_sim_set_capture(self._handle, None, None)
            out["maxiter_hit"] = _lib.check(rc, "nnmpc_sim_run")
        out["x_final"], out["uprev_final"] = xio, uio
        return out


def simulate_offline(task_number, process_number, data_filename, x0, uprev0, A, B, Bd, regulator, ulb, uub,
                     target_selector, setpoints, disturbances):
    """One trajectory chunk, reference signature (linearMPC.py:827-880); writes
    ``{task}-{process}-{data_filename}`` with keys x, uprev, xs, us, u, data_gen_time."""
    t0 = time.time()
    # The reference shifts THESE bounds by the target for the regulator (:685-686) while the target selector keeps
    # its own; both reference scripts pass the same pair.  The fused engine builds the regulator bounds from the
    # target selector's, so different pairs would silently diverge from the reference: refuse them.
    if not (np.array_equal(np.asarray(ulb), np.asarray(target_selector.ulb))
            and np.array_equal(np.asarray(uub), np.asarray(target_selector.uub))):
        raise NotImplementedError("simulate_offline: ulb/uub must equal the target selector's input bounds")
    regulator.ulb, regulator.uub = ulb, uub
    eng = ClosedLoopEngine(regulator, target_selector, A, B, Bd)
    res = eng.run(x0, uprev0, np.asarray(setpoints)[None], np.asarray(disturbances)[None])
    data = {k: res[k][0] for k in ("x", "uprev", "xs", "us", "u")}
    data["data_gen_time"] = time.time() - t0
    return _save_training_data(data, f"{task_number}-{process_number}-{data_filename}")


class OfflineSimulator:
    """Offline data generator (linearMPC.py:720-825).

    The reference builds one regulator/target selector per OS process and forks
    ``num_process_per_task`` processes per task; here one regulator/target selector pair serves
    every trajectory and all chunks of a task (or of all tasks, ``generate_batch``) advance
    together as one GPU batch.
    """

    def __init__(self, *, A, B, C, H, Rs, Qs, Bd, Cd, usp, uprev, Q, R, S, ulb, uub, N, xprior, setpoints,
                 disturbances, num_data_gen_task, num_process_per_task, device=None, **solver_kwargs):
        self.A, self.B, self.C, self.H, self.Rs, self.Qs, self.Bd, self.Cd = A, B, C, H, Rs, Qs, Bd, Cd
        self.usp, self.Q, self.R, self.S, self.ulb, self.uub, self.N = usp, Q, R, S, ulb, uub, N
        self.num_data_gen_task, self.num_process_per_task = num_data_gen_task, num_process_per_task
        self.Nx, self.Nu, self.Ny, self.Nd = A.shape[0], B.shape[1], C.shape[0], Bd.shape[1]
        self.x0, self.uprev0 = xprior, uprev
        self.target_selector = LinearMPCController.setup_target_selector(
            A=A, B=B, C=C, H=H, Bd=Bd, Cd=Cd, usp=usp, Qs=Qs, Rs=Rs, ulb=ulb, uub=uub, device=device)
        self.regulator = LinearMPCController.setup_regulator(A=A, B=B, Q=Q, R=R, S=S, N=N, ulb=ulb, uub=uub,
                                                             device=device, **solver_kwargs)
        # reference attribute names: one entry per process (all aliases of the shared pair)
        self.regulators = [self.regulator] * num_process_per_task
        self.target_selectors = [self.target_selector] * num_process_per_task
        self.engine = ClosedLoopEngine(self.regulator, self.target_selector, A, B, Bd)
        self.setpoints, self.disturbances = self._split_scenarios(setpoints=setpoints, disturbances=disturbances)

    def _split_scenarios(self, *, setpoints, disturbances):
        """Equal contiguous chunks, remainder dropped; lists indexed [task][process]
        (linearMPC.py:786-801)."""
        nproc = self.num_data_gen_task * self.num_process_per_task
        Lc = int(setpoints.shape[0] / nproc)
        self.Nsim_each_process = Lc
        sp = [setpoints[i * Lc:(i + 1) * Lc, :] for i in range(nproc)]
        ds = [disturbances[i * Lc:(i + 1) * Lc, :] for i in range(nproc)]
        k = self.num_process_per_task
        return ([sp[t * k:(t + 1) * k] for t in range(self.num_data_gen_task)],
                [ds[t * k:(t + 1) * k] for t in range(self.num_data_gen_task)])

    def generate_batch(self, tasks=None, distributed=None):
        """All chunks of the given tasks (default: all) as one batch; returns the engine's dict
        with arrays shaped (num_chunks, L, .), chunk order = (task, process) order.

        Under an initialised ``torch.distributed`` group with more than one rank (one process per
        GPU; ``distributed=None`` auto-detects) the chunks are sharded in contiguous blocks over the
        ranks - no collective on the solve path - and the dataset arrays x, uprev, xs, us, u are
        all-gathered over NCCL so every rank returns the full dataset (CUDA tensors) in the
        reference's concatenation order (controller_evaluation.py:281-292)."""
        from . import distributed as _d
        tasks = range(self.num_data_gen_task) if tasks is None else tasks
        sp = np.stack([c for t in tasks for c in self.setpoints[t]])
        ds = np.stack([c for t in tasks for c in self.disturbances[t]])
        if distributed is None:
            distributed = _d.is_distributed()
        if not distributed:
            return self.engine.run(self.x0, self.uprev0, sp, ds)
        torch = _torch()
        dev = torch.device("cuda", self.engine._dev)

        def run_local(sp_l, ds_l):
            f64 = dict(dtype=torch.float64, device=dev)
            return self.engine.run(self.x0, self.uprev0, torch.as_tensor(np.ascontiguousarray(sp_l), **f64),
                                   torch.as_tensor(np.ascontiguousarray(ds_l), **f64))
        return _d.generate_sharded(run_local, sp, ds, device=dev)

    def generate_data(self, *, task_number, data_filename, stdout_filename):
        """Reference entry point (linearMPC.py:803-825): writes one file per process of the task."""
        t0 = time.time()
        res = self.generate_batch([task_number])
        dt = time.time() - t0
        with open(stdout_filename, "w") as log:
            for proc in range(len(self.setpoints[task_number])):
                print(f"Process:{proc}\nSimulation Steps:{res['x'].shape[1]}\nComputation time:{dt}", file=log)
        files = []
        for proc in range(len(self.setpoints[task_number])):
            data = {k: res[k][proc] for k in ("x", "uprev", "xs", "us", "u")}
            data["data_gen_time"] = dt
            files.append(_save_training_data(data, f"{task_number}-{proc}-{data_filename}"))
        return files
