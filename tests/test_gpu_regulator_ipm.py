"""GPU tests of the interior-point regulator (csrc/ipm.cu): re-parameterised plants whose input-space box QP the
Douglas-Rachford path refuses (cond(P_u) >= 1e10, or P_u not positive definite in floating point) are solved in v by
interior point, against the oracle that follows the reference literally (general-G QP in v, lib/linearMPC.py:476-509)."""
import ctypes
import pickle

import numpy as np
import pytest
import scipy.linalg

pytestmark = pytest.mark.gpu

from oracle import linear_mpc as om

U_RTOL = 1e-6
COST_RTOL = 1e-6
MAX_ITERS = 50


@pytest.fixture(scope="module")
def torch_cuda(built_lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def unstable_plant(nx=6, nu=2, seed=5, rho=1.04):
    """Random plant with one unstable real mode (rho) and one marginally damped pair; controllable."""
    rng = np.random.default_rng(seed)
    lam = np.concatenate([[rho, 0.97], rng.uniform(0.3, 0.9, nx - 2)])
    V = rng.standard_normal((nx, nx)) + 2.0 * np.eye(nx)
    A = V @ np.diag(lam) @ np.linalg.inv(V)
    B = rng.standard_normal((nx, nu))
    return A, B


def rate_penalty_kwargs(nx, nu, seed, rho, N):
    """Regulator arguments as LinearMPCController.setup_regulator builds them, with a rate penalty S (M != 0)."""
    A, B = unstable_plant(nx=nx, nu=nu, seed=seed, rho=rho)
    C = np.random.default_rng(1).standard_normal((min(4, nx), nx))
    return dict(A=A, B=B, Q=0.05 * (C.T @ C) + 1e-3 * np.eye(nx), R=np.eye(nu), S=0.2 * np.eye(nu),
                ulb=-np.ones((nu, 1)), uub=np.ones((nu, 1)), N=N)


def make_plant(name, golden=None):
    """(regulator keyword arguments of DenseQPRegulator, or of setup_regulator when 'S' is present)."""
    if name.startswith("rho"):
        rho, N = {"rho1.3_N40": (1.3, 40), "rho1.5_N30": (1.5, 30), "rho1.5_N60": (1.5, 60), "rho2.0_N30": (2.0, 30)}[name]
        A, B = unstable_plant(rho=rho)
        nx, nu = B.shape
        return dict(A=A, B=B, Q=np.eye(nx), R=0.5 * np.eye(nu), M=np.zeros((nx, nu)), N=N, ulb=-np.ones((nu, 1)),
                    uub=np.ones((nu, 1)))
    if name == "rate_nu1":
        return rate_penalty_kwargs(4, 1, 3, 1.4, 40)
    if name == "rate_nu4":
        return rate_penalty_kwargs(6, 4, 9, 1.5, 30)
    assert name == "golden_unst_N200"
    return dict(A=golden["unst_A"], B=golden["unst_B"], Q=np.eye(2), R=np.eye(1), M=np.zeros((2, 1)), N=200,
                ulb=-np.ones((1, 1)), uub=np.ones((1, 1)))


def build(kw):
    from industrial_nnmpc_2021_b200.linearMPC import DenseQPRegulator, LinearMPCController
    if "S" in kw:
        reg = LinearMPCController.setup_regulator(**kw)
        oreg = om.setup_regulator(kw["A"], kw["B"], kw["Q"], kw["R"], kw["S"], kw["N"], kw["ulb"], kw["uub"])
    else:
        reg, oreg = DenseQPRegulator(**kw), om.DenseQPRegulatorOracle(**kw)
    return reg, oreg


def refused_by_box_path(reg):
    """The parent commit's refusal: non-finite P_u, a failed Cholesky, or cond(P_u) >= 1e10."""
    Pu = reg._Pu
    if not np.all(np.isfinite(Pu)):
        return True
    try:
        scipy.linalg.cho_factor(Pu, lower=True)
    except np.linalg.LinAlgError:
        return True
    ev = np.linalg.eigvalsh(0.5 * (Pu + Pu.T))
    return not (ev[0] > 0 and ev[-1] / ev[0] < 1e10)


def sample_x0(reg, count, seed, top=8.0):
    """x0 from deep inside the unconstrained region to most inputs saturated: random directions scaled so that the
    LQR roll-out S x0 peaks at 0.1 .. `top` times the bound."""
    rng = np.random.default_rng(seed)
    nxa = reg.Nx
    D = rng.standard_normal((count, nxa))
    peak = np.abs(D @ reg._S.T).max(axis=1)
    return D / peak[:, None] * np.logspace(-1.0, np.log10(top), count)[:, None]


# Where the inputs stay saturated, the state runs away like rho^k over the horizon.  The reference's variables
# u = K x + v then carry a cancellation of |K x| ~ rho^N |x0|: at rho = 1.5, N = 60 (rho^N = 4e10) u is only
# representable to ~1e-5 once most inputs saturate, for this solver and for the oracle alike, so that plant stops at
# 2.5 times the bound, and so does rho = 2.0, N = 30 (rho^N = 1e9); rho = 1.3, N = 40 (where the oracle's own solve
# breaks down beyond) stops at 4 times; the others run to 8.  The horizon of 200 with its 1.05 pole recovers from every
# such x0 within the horizon, so that plant saturates only a small share of its inputs.
TOP = {"rho1.5_N60": 2.5, "rho2.0_N30": 2.5, "rho1.3_N40": 4.0}
MOSTLY_SATURATED = {"rho1.5_N30", "rate_nu1", "rate_nu4"}


PLANTS = ["rho1.3_N40", "rho1.5_N30", "rho1.5_N60", "rho2.0_N30", "rate_nu1", "rate_nu4", "golden_unst_N200"]


@pytest.mark.parametrize("name", PLANTS)
def test_refused_plants_solve_by_interior_point(torch_cuda, golden_formulation, name):
    reg, oreg = build(make_plant(name, golden_formulation))
    assert reg.reparameterize and refused_by_box_path(reg)
    assert reg.solver == "ipm"
    with pytest.raises(AttributeError):
        reg.solver = "dr"
    X0 = sample_x0(reg, 64, seed=len(name), top=TOP.get(name, 8.0))
    U, info = reg.solve_batch(X0)
    assert not info["maxiter_hit"]
    assert float(np.max(info["kkt"])) <= reg.tol
    assert int(np.max(info["iters"])) <= MAX_ITERS, info["iters"]
    V = reg.to_v(U, X0)
    nact, sat = 0, []
    for i in range(X0.shape[0]):
        x0 = X0[i][:, None]
        uo = oreg.solve(x0)[:, 0]
        assert np.max(np.abs(U[i] - uo)) <= U_RTOL * max(1.0, np.abs(uo).max()), (i, np.max(np.abs(U[i] - uo)))
        # v = to_v(u) goes through T^-1, whose entries grow like rho^k (1.5^60 ~ 4e10): rounding in u reaches the
        # v-space objective at ~1e-8 absolute, so objectives below 1 are compared absolutely
        q = (oreg.tq @ x0)[:, 0]
        cost_v = float(0.5 * V[i] @ (oreg.P @ V[i]) + q @ V[i])
        v_or = reg.to_v(uo, X0[i])[0]
        cost_o = float(0.5 * v_or @ (oreg.P @ v_or) + q @ v_or)
        assert abs(cost_v - cost_o) <= COST_RTOL * max(abs(cost_o), 1.0), (i, cost_v, cost_o)
        # the kernel's cost output is the same reference objective
        assert abs(info["cost"][i] - cost_o) <= COST_RTOL * max(abs(cost_o), 1.0), (i, info["cost"][i], cost_o)
        assert np.all(oreg.G @ V[i][:, None] <= oreg.get_h(x0) + 1e-9)
        nact += int(np.any(np.abs(np.abs(uo) - 1.0) < 1e-7))
        sat.append(np.mean(np.abs(np.abs(uo) - 1.0) < 1e-7))
    assert nact >= X0.shape[0] // 4, nact
    if name in MOSTLY_SATURATED:
        assert max(sat) > 0.5, max(sat)        # most inputs saturated
    print(f"\n{name}: saturated share of the inputs up to {max(sat):.2f}")
    print(f"\n{name}: mean IPM iterations {np.mean(info['iters']):.2f}, max {np.max(info['iters'])}")


def test_known_answer_lqr_rollout(torch_cuda):
    """With S x0 inside the box the optimum is v = 0 (tq_v vanishes): u is the LQR roll-out."""
    reg, _ = build(make_plant("rho1.5_N60"))
    assert reg.solver == "ipm"
    X0 = sample_x0(reg, 16, seed=3)[:8]        # peaks of S x0 at 0.1 .. 0.7 of the bound
    assert np.all(np.abs(X0 @ reg._S.T) < 1.0)
    U, info = reg.solve_batch(X0)
    Uref = X0 @ reg._S.T
    assert np.max(np.abs(U - Uref)) <= 1e-12 * max(1.0, np.abs(Uref).max()), np.max(np.abs(U - Uref))
    assert not info["maxiter_hit"] and float(np.max(info["kkt"])) <= reg.tol


def test_batch_independence_and_host_device_entry_points(torch_cuda):
    torch = torch_cuda
    reg, _ = build(make_plant("rho2.0_N30"))
    X0 = sample_x0(reg, 3000, seed=11)
    Xd = torch.as_tensor(X0, device="cuda")
    Ub, ib = reg.solve_batch(Xd)
    Uh, ih = reg.solve_batch(X0)
    assert torch.equal(Ub.cpu(), torch.as_tensor(Uh))
    for k in ("kkt", "cost", "iters"):
        assert np.array_equal(ib[k].cpu().numpy(), ih[k]), k
    for i in (0, 1234, 2999):
        Ui, ii = reg.solve_batch(Xd[i:i + 1].clone())
        assert torch.equal(Ui[0], Ub[i]) and torch.equal(ii["kkt"][0], ib["kkt"][i])
    # the batched-engine form (precision has no effect) and the lock-step form agree bitwise
    for precision in ("mixed", "f64"):
        Ue, _ = reg.solve_batch(Xd, precision=precision)
        assert torch.equal(Ue, Ub), precision
    # warm_state is accepted and ignored
    ws = torch.zeros_like(Ub)
    Uw, _ = reg.solve_batch(Xd, warm_state=ws)
    Uw2, _ = reg.solve_batch(Xd, warm_state=ws)
    assert torch.equal(Uw, Ub) and torch.equal(Uw2, Ub)


@pytest.mark.parametrize("bad", ["nan_x0", "inf_x0", "lb_eq_ub", "lb_gt_ub", "nan_bound"])
def test_bad_samples_are_isolated(torch_cuda, bad):
    reg, _ = build(make_plant("rho1.5_N30"))
    nu = reg.Nu
    X0 = sample_x0(reg, 9, seed=5)
    LB, UB = -np.ones((9, nu)), np.ones((9, nu))
    U0, i0 = reg.solve_batch(X0, LB.copy(), UB.copy())
    assert not i0["maxiter_hit"]
    X1, LB1, UB1 = X0.copy(), LB.copy(), UB.copy()
    bad_rows = (0, 4, 8)
    for r in bad_rows:
        if bad == "nan_x0":
            X1[r, 1] = np.nan
        elif bad == "inf_x0":
            X1[r, 0] = -np.inf
        elif bad == "lb_eq_ub":
            LB1[r, 0] = UB1[r, 0] = 0.5
        elif bad == "lb_gt_ub":
            LB1[r, 1], UB1[r, 1] = 0.3, -0.3
        else:
            LB1[r, 0] = np.nan
    U1, i1 = reg.solve_batch(X1, LB1, UB1)
    assert i1["maxiter_hit"]
    for r in range(9):
        if r in bad_rows:
            assert np.all(np.isnan(U1[r])) and i1["iters"][r] == reg.max_iter and np.isnan(i1["kkt"][r])
        else:
            assert np.array_equal(U1[r], U0[r]) and i1["iters"][r] == i0["iters"][r] and i1["kkt"][r] == i0["kkt"][r]


def test_infinite_bounds_are_absent(torch_cuda):
    reg, oreg = build(make_plant("rho1.5_N30"))
    nu = reg.Nu
    X0 = sample_x0(reg, 9, seed=6)
    LB, UB = -np.ones((9, nu)), np.ones((9, nu))
    U0, _ = reg.solve_batch(X0, LB, UB)
    LB1, UB1 = LB.copy(), UB.copy()
    LB1[3, :] = -np.inf                 # one-sided box
    UB1[5, :], LB1[5, :] = np.inf, -np.inf   # unconstrained: the LQR roll-out
    U1, i1 = reg.solve_batch(X0, LB1, UB1)
    assert not i1["maxiter_hit"] and float(np.max(i1["kkt"])) <= reg.tol
    for r in range(9):
        if r not in (3, 5):
            assert np.array_equal(U1[r], U0[r])
    Uref = X0[5] @ reg._S.T
    assert np.max(np.abs(U1[5] - Uref)) <= 1e-12 * max(1.0, np.abs(Uref).max())
    # one-sided sample against the oracle with the lower bounds dropped
    assert np.all(U1[3] <= 1.0 + 1e-9)
    o1 = om.DenseQPRegulatorOracle(**dict(make_plant("rho1.5_N30"), ulb=-1e6 * np.ones((nu, 1))))
    uo = o1.solve(X0[3][:, None])[:, 0]
    assert np.max(np.abs(U1[3] - uo)) <= U_RTOL * max(1.0, np.abs(uo).max())


def _closed_loop_setup():
    kw = rate_penalty_kwargs(8, 4, 9, 1.6, 24)
    A, B = kw["A"], kw["B"]
    nx, nu = B.shape
    rng = np.random.default_rng(1)
    C = rng.standard_normal((4, nx))
    Bd = B[:, :2].copy()
    full = dict(A=A, B=B, C=C, H=np.zeros((0, 4)), Rs=1e-3 * np.eye(nu), Qs=np.eye(4), Bd=Bd, Cd=np.zeros((4, 2)),
                usp=np.zeros((nu, 1)), uprev=np.zeros((nu, 1)), Q=kw["Q"], R=kw["R"], S=kw["S"], ulb=kw["ulb"],
                uub=kw["uub"], N=kw["N"])
    return full


def test_closed_loop_with_strongly_unstable_plant(torch_cuda):
    """OfflineSimulator.generate_batch (simulate_offline, :827-880) on a plant the box path refuses: lock-step engine
    (target selector -> interior-point QPs -> plant step) against the oracle chunk by chunk."""
    from industrial_nnmpc_2021_b200.linearMPC import OfflineSimulator
    from industrial_nnmpc_2021_b200.controller_evaluation import sample_prbs_like
    torch = torch_cuda
    kw = _closed_loop_setup()
    A, B, C, Bd = kw["A"], kw["B"], kw["C"], kw["Bd"]
    nx, nu = B.shape
    T, chunks = 10, 3
    sp = sample_prbs_like(num_change=8, num_steps=T * chunks, lb=-1.0 * np.ones((4, 1)), ub=1.0 * np.ones((4, 1)),
                          mean_change=4, sigma_change=1, seed=3)
    ds = sample_prbs_like(num_change=8, num_steps=T * chunks, lb=-0.3 * np.ones((2, 1)), ub=0.3 * np.ones((2, 1)),
                          mean_change=4, sigma_change=1, seed=4)
    xprior = np.zeros((nx, 1))
    sim = OfflineSimulator(**kw, xprior=xprior, setpoints=sp, disturbances=ds, num_data_gen_task=1,
                           num_process_per_task=chunks)
    assert sim.regulator.reparameterize and refused_by_box_path(sim.regulator) and sim.regulator.solver == "ipm"
    oreg = om.setup_regulator(A, B, kw["Q"], kw["R"], kw["S"], kw["N"], kw["ulb"], kw["uub"])
    ots = om.TargetSelectorOracle(A=A, B=B, C=C, H=kw["H"], Bd=Bd, Cd=kw["Cd"], usp=kw["usp"], Rs=kw["Rs"],
                                  Qs=kw["Qs"], ulb=kw["ulb"], uub=kw["uub"])
    results = {}
    for precision in ("f64", "mixed"):
        sim.engine.set_precision(precision)
        results[precision] = res = sim.generate_batch()
        assert float(res["kkt"].max()) <= sim.regulator.tol and not res["maxiter_hit"]
        assert int(res["iters"].max()) <= MAX_ITERS
    for k in ("x", "uprev", "xs", "us", "u", "iters", "kkt"):
        assert np.array_equal(results["f64"][k], results["mixed"][k]), k
    res = results["f64"]
    assert np.sum(np.abs(res["u"]) >= 1.0 - 1e-7) >= 3, "saturated inputs wanted"
    for c in range(chunks):
        od = om.simulate_offline(x0=xprior, uprev0=kw["uprev"], A=A, B=B, Bd=Bd, regulator=oreg, ulb=kw["ulb"],
                                 uub=kw["uub"], target_selector=ots, setpoints=sp[c * T:(c + 1) * T],
                                 disturbances=ds[c * T:(c + 1) * T])
        for k in ("x", "xs", "us", "u"):
            err = np.max(np.abs(res[k][c] - od[k])) / max(1.0, np.max(np.abs(od[k])))
            assert err <= 2e-6, (c, k, err)
    st = sim.engine.stats()
    assert st["qps"] >= 2 * chunks * T and st["row_iterations"] > 0
    # capture: the whole optimal sequence of every QP, target added back, is the oracle's useq
    eng = sim.engine
    f64 = dict(dtype=torch.float64, device="cuda")
    cap = eng.run(torch.as_tensor(xprior, **f64), torch.as_tensor(kw["uprev"], **f64),
                  torch.as_tensor(np.stack(sim.setpoints[0]), **f64), torch.as_tensor(np.stack(sim.disturbances[0]), **f64),
                  capture=True)
    useq = cap["useq"].cpu().numpy()
    for c in range(chunks):
        assert np.array_equal(useq[c][:, :nu], res["u"][c])
        for t in (0, 4, 9):
            us = res["us"][c, t][:, None]
            oreg.ulb, oreg.uub = kw["ulb"] - us, kw["uub"] - us
            x0 = np.concatenate([res["x"][c, t] - res["xs"][c, t], res["uprev"][c, t] - res["us"][c, t]])[:, None]
            ou = oreg.solve(x0)[:, 0] + np.tile(us[:, 0], kw["N"])
            assert np.max(np.abs(useq[c, t] - ou)) <= 1e-6 * max(1.0, np.abs(ou).max()), (c, t)
    # resume: two slabs of 5 steps equal one run of 10
    sp0, ds0 = np.stack(sim.setpoints[0]), np.stack(sim.disturbances[0])
    first = eng.run(xprior, kw["uprev"], sp0[:, :5], ds0[:, :5])
    second = eng.run(first["x_final"], first["uprev_final"], sp0[:, 5:], ds0[:, 5:], resume=True)
    for k in ("x", "u", "xs", "us"):
        assert np.array_equal(np.concatenate([first[k], second[k]], axis=1), res[k]), k


def test_online_loop_with_strongly_unstable_plant(torch_cuda):
    from industrial_nnmpc_2021_b200.controller_evaluation import BatchedOnlineSimulation, sample_prbs_like
    from industrial_nnmpc_2021_b200.linearMPC import LinearPlantSimulator
    kw = _closed_loop_setup()
    nx, nu = kw["B"].shape
    ny = kw["C"].shape[0]
    kw = dict(kw, Qwx=1e-6 * np.eye(nx), Qwd=1e-2 * np.eye(2), Rv=1e-4 * np.eye(ny), xprior=np.zeros((nx, 1)),
              dprior=np.zeros((2, 1)))
    T = 10
    sp = np.stack([sample_prbs_like(num_change=4, num_steps=T, lb=-1.0 * np.ones((ny, 1)), ub=1.0 * np.ones((ny, 1)),
                                    mean_change=3, sigma_change=1, seed=s) for s in (5, 6)])
    ds = np.stack([sample_prbs_like(num_change=4, num_steps=T, lb=-0.3 * np.ones((2, 1)), ub=0.3 * np.ones((2, 1)),
                                    mean_change=3, sigma_change=1, seed=s) for s in (7, 8)])
    sim = BatchedOnlineSimulation(kind="mpc", **kw)
    assert sim.regulator.solver == "ipm"
    res = sim.run(sp, ds, seed=3)
    assert float(res["kkt"].max()) <= sim.regulator.tol and not res["maxiter_hit"]
    for c in range(2):
        octrl = om.OnlineControllerOracle(**kw)
        np.random.seed(3)
        plant = LinearPlantSimulator(A=kw["A"], B=kw["B"], C=kw["C"], Bp=kw["Bd"], Rv=kw["Rv"], sample_time=1.0,
                                     x0=np.zeros((nx, 1)))
        uo = om.online_simulation(plant.step, plant.y[0], octrl, sp[c], ds[c], T)
        assert np.max(np.abs(res["u"][c] - uo)) <= 2e-6 * max(1.0, np.abs(uo).max()), c
        xo = np.asarray(plant.x)[:, :, 0]
        assert np.max(np.abs(res["x"][c] - xo)) <= 2e-6 * max(1.0, np.abs(xo).max()), c


def test_refusals_and_pickle(torch_cuda):
    from industrial_nnmpc_2021_b200 import _lib
    from industrial_nnmpc_2021_b200.linearMPC import DenseQPRegulator
    reg, _ = build(make_plant("rho1.3_N40"))
    L = _lib.lib()
    rho = np.ones(reg.N * reg.Nu)
    rc = L.nnmpc_qp_set_penalty(reg._handle, _lib.hptr(rho))
    assert rc == -1 and b"interior point" in L.nnmpc_last_error()
    # C ABI size limits
    h = ctypes.c_void_p()
    for nxa, nu in ((66, 2), (8, 33)):
        ops = [np.zeros((nxa, nxa)), np.zeros((nxa, nu)), np.zeros((nxa, nxa)), np.eye(nu), np.zeros((nxa, nu)),
               np.zeros((nxa, nxa)), np.zeros((nu, nxa))]
        rc = L.nnmpc_qp_create_ipm(ctypes.byref(h), nxa, nu, 10, *[_lib.hptr(a) for a in ops], 0)
        assert rc == -4 and b"nxa <= 64 and nu <= 32" in L.nnmpc_last_error()
    # Python: a refused plant above the limit (nxa = 65 -> 66 after padding)
    A, B = unstable_plant(nx=65, nu=2, seed=2, rho=2.0)
    with pytest.raises(NotImplementedError, match="Nxa = 64"):
        DenseQPRegulator(A=A, B=B, Q=np.eye(65), R=0.5 * np.eye(2), M=np.zeros((65, 2)), N=40, ulb=-np.ones((2, 1)),
                         uub=np.ones((2, 1)))
    # pickle round trip re-runs the set-up and takes the same path; solves are bitwise equal
    reg2 = pickle.loads(pickle.dumps(reg))
    assert reg2.solver == "ipm"
    X0 = sample_x0(reg, 32, seed=2)
    U1, i1 = reg.solve_batch(X0)
    U2, i2 = reg2.solve_batch(X0)
    assert np.array_equal(U1, U2) and np.array_equal(i1["kkt"], i2["kkt"])
    u = reg2.solve(X0[5][:, None])
    assert np.array_equal(u[:, 0], U1[5])
