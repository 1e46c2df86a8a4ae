"""GPU: the target selector with pinned outputs (H non-empty) or an integrating plant (I - A singular) - the reduced
mode of k_ts_general - against the oracle's formulation of the reference problem (lib/linearMPC.py:229-311) solved
through a null-space basis (ts_equality_cases.EqualityTargetOracle), alone, inside the closed-loop engine and inside
the online loop.

No reference artefact pins the H rows of tA / tb (the reference code is not in this tree and no fixture covers
H != 0), so besides the oracle every target is checked against the formulation itself: the equality residual and a
solver-independent KKT check."""
import os
import pickle
import sys

import numpy as np
import pytest

from oracle import linear_mpc as om

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ts_equality_cases as tc        # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda(built_lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def cdu_full_problem():
    from industrial_nnmpc_2021_b200.plants import get_cdu_problem
    return get_cdu_problem(with_scenarios=False)


@pytest.fixture
def problems(cstrs_problem, cdu_small_problem, cdu_full_problem):
    return dict(cstrs=cstrs_problem, cdu_small=cdu_small_problem, cdu_full=cdu_full_problem)


def _pair(kw):
    from industrial_nnmpc_2021_b200.linearMPC import TargetSelector
    return TargetSelector(**kw), tc.EqualityTargetOracle(**kw)


def _check_kkt(ots, y, d, xs, us):
    """Stationarity of the (xs, us) QP with least-squares multipliers of the equalities and of the bounds the point
    sits on, their signs, and complementarity."""
    q, h, b = ots.changing(y[:, None], d[:, None])
    w = np.concatenate([xs, us])
    g = ots.P @ w + q[:, 0]
    slack = h[:, 0] - ots.G @ w
    act = np.flatnonzero(slack <= 1e-8 * (1.0 + np.abs(h[:, 0])))
    J = np.vstack([ots.tA, ots.G[act]]).T
    mult = np.linalg.lstsq(J, -g, rcond=None)[0]
    scale = max(np.abs(ots.P).max() * np.abs(w).max(), np.abs(q).max(), 1e-300)
    assert np.max(np.abs(g + J @ mult)) <= 1e-7 * scale
    lam = mult[ots.tA.shape[0]:]
    assert np.all(lam >= -1e-6 * max(1.0, np.abs(mult).max()))
    assert np.max(np.abs(lam * slack[act]), initial=0.0) <= 1e-8 * max(1.0, np.abs(mult).max())


@pytest.mark.parametrize("name", tc.CASES)
def test_targets_match_oracle(torch_cuda, problems, name):
    kw, YSP, D = tc.case(name, problems["cstrs"], problems["cdu_small"], problems["cdu_full"])
    ts, ots = _pair(kw)
    assert ts.reduced
    keep, ref = [], []
    for i in range(YSP.shape[0]):
        try:
            ref.append(ots.solve(YSP[i][:, None], D[i][:, None]))
            keep.append(i)
        except ValueError:
            pass                                       # infeasible output cut: covered by the mixed batch below
    assert len(keep) >= 4
    xs, us, it = ts.solve_batch(YSP[keep], D[keep], return_iters=True)
    assert it.min() >= 0
    for k, (oxs, ous) in enumerate(ref):
        y, d = YSP[keep[k]], D[keep[k]]
        assert np.all(us[k] >= kw["ulb"][:, 0]) and np.all(us[k] <= kw["uub"][:, 0])
        w = np.concatenate([xs[k], us[k]])
        b = ots.tb @ np.concatenate([y, d])
        assert np.max(np.abs(ots.tA @ w - b)) <= 1e-9 * max(1.0, np.abs(b).max(), np.abs(w).max())
        q = ots.changing(y[:, None], d[:, None])[0][:, 0]
        ow = np.vstack([oxs, ous])[:, 0]
        c, oc = 0.5 * w @ ots.P @ w + q @ w, 0.5 * ow @ ots.P @ ow + q @ ow
        assert abs(c - oc) <= 1e-7 * max(1.0, abs(oc)), (k, c, oc)
        assert np.max(np.abs(us[k] - ous[:, 0])) <= 1e-6 * max(1.0, np.abs(ous).max()), k
        assert np.max(np.abs(xs[k] - oxs[:, 0])) <= 1e-5 * max(1.0, np.abs(oxs).max()), k
        _check_kkt(ots, y, d, xs[k], us[k])
    # the CUDA-tensor entry point returns the same bits
    torch = torch_cuda
    f64 = dict(dtype=torch.float64, device="cuda")
    xd, ud, itd = ts.solve_batch(torch.as_tensor(YSP[keep], **f64), torch.as_tensor(D[keep], **f64), return_iters=True)
    assert np.array_equal(xd.cpu().numpy(), xs) and np.array_equal(ud.cpu().numpy(), us)
    assert np.array_equal(itd.cpu().numpy(), it)
    oxs1, ous1 = ts.solve(YSP[keep[0]][:, None], D[keep[0]][:, None])
    assert oxs1.shape == (ts.Nx, 1) and ous1.shape == (ts.Nu, 1) and len(ts.us) == 1


@pytest.mark.parametrize("name", ["cstrs_z", "cdu_small_h2", "cdu_hsel", "integrating_h"])
def test_unreachable_and_nonfinite_samples_are_flagged_alone(torch_cuda, problems, name):
    """A pinned output moved far out of reach makes the target infeasible; NaN / Inf in ysp or d make it undefined.
    Exactly those samples carry negative iteration counts, and every other sample is bitwise what a batch without
    them gives."""
    from industrial_nnmpc_2021_b200._lib import NnmpcError
    torch = torch_cuda
    kw, YSP, D = tc.case(name, problems["cstrs"], problems["cdu_small"], problems["cdu_full"])
    ts, ots = _pair(kw)
    hrow = int(np.flatnonzero(kw["H"][0])[0])
    bad = {1: "far", 4: "nan_y", 6: "far", 7: "inf_d", 11: "ninf_y"}
    Y, Dm = YSP.copy(), D.copy()
    for i, what in bad.items():
        if what == "far":
            Y[i, hrow] += 50.0 * (1.0 + np.abs(YSP[:, hrow]).max())
            with pytest.raises(ValueError):
                ots.solve(Y[i][:, None], Dm[i][:, None])
        elif what == "nan_y":
            Y[i, -1] = np.nan
        elif what == "ninf_y":
            Y[i, 0] = -np.inf
        else:
            Dm[i, -1] = np.inf
    with pytest.raises(NnmpcError):
        ts.solve_batch(Y[[1]], Dm[[1]])
    f64 = dict(dtype=torch.float64, device="cuda")
    xs, us, it = ts.solve_batch(torch.as_tensor(Y, **f64), torch.as_tensor(Dm, **f64), return_iters=True)
    it = it.cpu().numpy()
    assert sorted(np.flatnonzero(it < 0).tolist()) == sorted(bad)
    good = [i for i in range(Y.shape[0]) if i not in bad]
    xg, ug, itg = ts.solve_batch(torch.as_tensor(Y[good], **f64), torch.as_tensor(Dm[good], **f64), return_iters=True)
    assert np.array_equal(xs.cpu().numpy()[good], xg.cpu().numpy())
    assert np.array_equal(us.cpu().numpy()[good], ug.cpu().numpy())
    assert np.array_equal(it[good], itg.cpu().numpy())


def test_pickle_round_trip(torch_cuda, problems):
    kw, YSP, D = tc.case("cdu_small_h2", problems["cstrs"], problems["cdu_small"], problems["cdu_full"])
    ts, _ = _pair(kw)
    ts2 = pickle.loads(pickle.dumps(ts))
    assert ts2.reduced and ts2._handle is not ts._handle
    a, b = ts.solve_batch(YSP[:3], D[:3]), ts2.solve_batch(YSP[:3], D[:3])
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def _held(levels, T):
    """Consecutive pairs of rows of ``levels``, each row held for T // 2 steps: (len(levels) // 2 * T, n)."""
    out = [np.repeat(levels[[j, j + 1]], T // 2, axis=0) for j in range(0, len(levels) - 1, 2)]
    return np.concatenate(out)


def test_closed_loop_integrating_plant_with_h(torch_cuda):
    """simulate_offline (:827-880) on an integrating plant with two pinned outputs: the reduced target selector and
    the re-parameterised regulator inside the continuously batched engine, both precisions."""
    from industrial_nnmpc_2021_b200.linearMPC import OfflineSimulator
    ts_kw = tc.integrating_plant(with_h=True)
    A, B, C, Bd = ts_kw["A"], ts_kw["B"], ts_kw["C"], ts_kw["Bd"]
    nx, nu = B.shape
    T, chunks = 10, 3
    sts = tc.steady_states(ts_kw, 2 * chunks, seed=5, frac=0.4, dscale=0.2)
    Y0 = np.array([C @ xs + ts_kw["Cd"] @ d for xs, _, d in sts])
    sp, ds = _held(Y0, T), _held(np.array([d for _, _, d in sts]), T)
    kw = dict(ts_kw, uprev=np.zeros((nu, 1)), Q=0.05 * (C.T @ C) + 1e-3 * np.eye(nx), R=np.eye(nu), S=0.2 * np.eye(nu),
              N=12)
    xprior = np.zeros((nx, 1))
    sim = OfflineSimulator(**kw, xprior=xprior, setpoints=sp, disturbances=ds, num_data_gen_task=1,
                           num_process_per_task=chunks)
    assert sim.target_selector.reduced and sim.regulator.reparameterize
    oreg = om.setup_regulator(A, B, kw["Q"], kw["R"], kw["S"], 12, kw["ulb"], kw["uub"])
    ots = tc.EqualityTargetOracle(**ts_kw)
    for precision in ("f64", "mixed"):
        sim.engine.set_precision(precision)
        res = sim.generate_batch()
        assert float(res["kkt"].max()) <= 1e-8 and not res["maxiter_hit"]
        for c in range(chunks):
            od = om.simulate_offline(x0=xprior, uprev0=kw["uprev"], A=A, B=B, Bd=Bd, regulator=oreg, ulb=kw["ulb"],
                                     uub=kw["uub"], target_selector=ots, setpoints=sp[c * T:(c + 1) * T],
                                     disturbances=ds[c * T:(c + 1) * T])
            for k in ("x", "xs", "us", "u"):
                err = np.max(np.abs(res[k][c] - od[k])) / max(1.0, np.max(np.abs(od[k])))
                assert err <= 2e-6, (precision, c, k, err)
            ys = od["xs"] @ C.T + ds[c * T:(c + 1) * T] @ ts_kw["Cd"].T
            assert np.allclose((ys @ ts_kw["H"].T), sp[c * T:(c + 1) * T] @ ts_kw["H"].T, atol=1e-9)


def test_batched_online_mpc_cstrs_with_h(torch_cuda, cstrs_problem):
    """BatchedOnlineSimulation(kind="mpc") on the CSTRs with the z outputs pinned (nw = 0: the target is K s of the
    filter's disturbance estimate) against the one-scenario-at-a-time oracle loop."""
    from industrial_nnmpc_2021_b200.controller_evaluation import BatchedOnlineSimulation
    from industrial_nnmpc_2021_b200.linearMPC import LinearPlantSimulator
    p = cstrs_problem
    H = np.eye(p.Ny)[list(p.extra["z_indices"])]
    kw = dict(A=p.A, B=p.B, C=p.C, H=H, Qwx=1e-6 * np.eye(p.Nx), Qwd=1e-2 * np.eye(p.Nd), Rv=1e-4 * np.eye(p.Ny),
              xprior=np.zeros((p.Nx, 1)), dprior=np.zeros((p.Nd, 1)), Rs=p.Rs, Qs=p.Qs, Bd=p.Bd, Cd=p.Cd, usp=p.usp,
              uprev=np.zeros((p.Nu, 1)), Q=p.Q, R=p.R, S=p.S, ulb=p.ulb, uub=p.uub, N=30)
    S_, T = 4, 10
    sts = tc.steady_states(tc.ts_kwargs(p, H), 2 * S_, seed=9, frac=0.3, dscale=0.02)
    Y0 = np.array([p.C @ xs + p.Cd @ d for xs, _, d in sts])
    sp = _held(Y0, T).reshape(S_, T, p.Ny)
    ds = _held(np.array([d for _, _, d in sts]), T).reshape(S_, T, p.Nd)
    sim = BatchedOnlineSimulation(kind="mpc", **kw)
    assert sim.target_selector.reduced and sim.target_selector.nw == 0
    res = sim.run(sp, ds, seed=3)
    assert float(res["kkt"].max()) <= 1e-8 and not res["maxiter_hit"]
    for c in range(S_):
        octrl = om.OnlineControllerOracle(**kw)
        octrl.target_selector = tc.EqualityTargetOracle(**tc.ts_kwargs(p, H))     # the oracle loop's own cannot reduce H rows
        np.random.seed(3)
        plant = LinearPlantSimulator(A=p.A, B=p.B, C=p.C, Bp=p.Bd, Rv=kw["Rv"], sample_time=10.0, x0=np.zeros((p.Nx, 1)))
        uo = om.online_simulation(plant.step, plant.y[0], octrl, sp[c], ds[c], T)
        assert np.max(np.abs(res["u"][c] - uo)) <= 1e-6 * max(1.0, np.abs(uo).max()), c
        oxs = np.array([t[0][:, 0] for t in octrl.targets])
        ous = np.array([t[1][:, 0] for t in octrl.targets])
        assert np.max(np.abs(res["us"][c] - ous)) <= 1e-6 * max(1.0, np.abs(ous).max()), c
        assert np.max(np.abs(res["xs"][c] - oxs)) <= 1e-5 * max(1.0, np.abs(oxs).max()), c
