"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle.

Tolerances are the north-star ones: first move u0 and optimal cost within 1e-6 relative, KKT
residual <= 1e-8 (the solver stops at 1e-9), NN outputs within 1e-5.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import linear_mpc as om
from oracle import qp as oq
from oracle import nn as onn

U0_RTOL = 1e-6
COST_RTOL = 1e-6
KKT_TOL = 1e-8
NN_TOL = 1e-5


@pytest.fixture(scope="module")
def torch_cuda(built_lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _rel(a, b, floor=1e-3):
    """max |a-b| relative to max(|b|_inf, floor) per row."""
    a, b = np.atleast_2d(a), np.atleast_2d(b)
    return np.max(np.abs(a - b), axis=1) / np.maximum(np.max(np.abs(b), axis=1), floor)


# ------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K", [(1, 8, 4), (7, 13, 18), (64, 64, 64), (130, 540, 18), (257, 540, 540),
                                    (300, 129, 290), (1000, 252, 290)])
def test_gemm_tn_matches_numpy(torch_cuda, M, N, K):
    torch = torch_cuda
    from industrial_nnmpc_2021_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(M * 1000 + N)
    lda = (K + 1) & ~1
    A = np.zeros((M, lda)); A[:, :K] = rng.standard_normal((M, K))
    Bt = np.zeros((N, lda)); Bt[:, :K] = rng.standard_normal((N, K))
    At, Btt = torch.tensor(A, device="cuda"), torch.tensor(Bt, device="cuda")
    Cd = torch.full((M, N), np.nan, dtype=torch.float64, device="cuda")
    rc = L.nnmpc_gemm_tn(M, N, K, _lib.dptr(At), lda, _lib.dptr(Btt), lda, _lib.dptr(Cd), N, None, None)
    _lib.check(rc, "gemm")
    torch.cuda.synchronize()
    ref = A[:, :K] @ Bt[:, :K].T
    assert np.allclose(Cd.cpu().numpy(), ref, rtol=1e-13, atol=1e-12 * np.sqrt(K))


def test_gemm_row_gather(torch_cuda):
    torch = torch_cuda
    from industrial_nnmpc_2021_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(5)
    Mtot, M, N, K = 500, 200, 96, 128
    A, Bt = rng.standard_normal((Mtot, K)), rng.standard_normal((N, K))
    rows = rng.permutation(Mtot)[:M].astype(np.int32)
    At, Btt = torch.tensor(A, device="cuda"), torch.tensor(Bt, device="cuda")
    rt = torch.tensor(rows, device="cuda")
    Cd = torch.zeros((Mtot, N), dtype=torch.float64, device="cuda")
    rc = L.nnmpc_gemm_tn(M, N, K, _lib.dptr(At), K, _lib.dptr(Btt), K, _lib.dptr(Cd), N, _lib.vp(rt.data_ptr()), None)
    _lib.check(rc, "gemm")
    out = Cd.cpu().numpy()
    ref = np.zeros((Mtot, N)); ref[rows] = A[rows] @ Bt.T
    assert np.allclose(out, ref, rtol=1e-13, atol=1e-12)


# ------------------------------------------------------------------------------------ regulator QP
def _closed_loop_samples(p, T, starts):
    """(x0, us) pairs visited by the ORACLE's closed loop, so the QPs are realistic."""
    reg = om.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    ts = om.TargetSelectorOracle(A=p.A, B=p.B, C=p.C, H=p.H, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs,
                                 ulb=p.ulb, uub=p.uub)
    datas = [om.simulate_offline(x0=p.xprior, uprev0=p.uprev, A=p.A, B=p.B, Bd=p.Bd, regulator=reg, ulb=p.ulb,
                                 uub=p.uub, target_selector=ts, setpoints=p.setpoints[s:s + T],
                                 disturbances=p.disturbances[s:s + T]) for s in starts]
    return reg, ts, datas


@pytest.fixture(scope="module")
def cstr_case(cstrs_problem):
    reg, ts, datas = _closed_loop_samples(cstrs_problem, 40, (0, 30000))
    return reg, ts, datas


def test_regulator_batch_matches_oracle_cstr(torch_cuda, cstrs_problem, cstr_case):
    torch = torch_cuda
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    p = cstrs_problem
    oreg, _, datas = cstr_case
    d = {k: np.vstack([x[k] for x in datas]) for k in datas[0]}
    X0 = np.hstack([d["x"] - d["xs"], d["uprev"] - d["us"]])
    LB, UB = p.ulb.T - d["us"], p.uub.T - d["us"]
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    assert np.allclose(reg.P, oreg.P, atol=1e-11 * np.abs(oreg.P).max())
    # device entry point
    U, info = reg.solve_batch(torch.tensor(X0, device="cuda"), torch.tensor(LB, device="cuda"),
                              torch.tensor(UB, device="cuda"))
    U = U.cpu().numpy()
    box = oq.BoxQP(oreg.P)
    nact = 0
    for i in range(X0.shape[0]):
        q = oreg.tq @ X0[i]
        lb, ub = np.tile(LB[i], p.N), np.tile(UB[i], p.N)
        ue, ei = box.solve(q, lb, ub)
        nact += ei["n_active"] > 0
        assert oq.box_kkt_residual(oreg.P, q, U[i], lb, ub) <= KKT_TOL
        assert _rel(U[i][:p.Nu], ue[:p.Nu])[0] <= U0_RTOL
        assert abs(info["cost"][i].item() - ei["cost"]) <= COST_RTOL * max(abs(ei["cost"]), 1e-6)
    assert nact > 10, "test should exercise active constraints"
    assert float(info["kkt"].max()) <= KKT_TOL and not info["maxiter_hit"]
    # host entry point returns the same numbers
    U2, info2 = reg.solve_batch(X0, LB, UB)
    assert np.array_equal(U2, U)
    assert np.array_equal(info2["iters"], info["iters"].cpu().numpy())


def test_regulator_dropin_solve_and_lqr_identity(torch_cuda, cstrs_problem):
    """DenseQPRegulator.solve(x0) signature; unconstrained solves equal the LQR law (Pf = DARE)."""
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    p = cstrs_problem
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    rng = np.random.default_rng(3)
    x0 = 1e-4 * rng.standard_normal((reg.Nx, 1))
    useq = reg.solve(x0)
    assert useq.shape == (p.N * p.Nu, 1) and len(reg.useq) == 1 and reg.x0[0] is not None
    assert np.allclose(useq[:p.Nu], reg.Krep @ x0, rtol=1e-8, atol=1e-14)
    assert int(reg.last_info["iters"][0]) == 1
    # get_control_sequence mutates bounds and adds us back (linearMPC.py:682-689)
    us = 0.1 * np.ones((p.Nu, 1)); xs = np.zeros((p.Nx, 1))
    seq = LinearMPCController.get_control_sequence(reg, 0.5 * np.ones((p.Nx, 1)), np.zeros((p.Nu, 1)), xs, us,
                                                   p.ulb, p.uub)
    assert np.allclose(reg.ulb, p.ulb - us) and seq.shape == (p.N * p.Nu, 1)
    assert np.all(seq <= np.tile(p.uub, (p.N, 1)) + 1e-12) and np.all(seq >= np.tile(p.ulb, (p.N, 1)) - 1e-12)


def test_regulator_edge_cases(torch_cuda, cstrs_problem):
    torch = torch_cuda
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    p = cstrs_problem
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, 20, p.ulb, p.uub)
    n = 20 * p.Nu
    # empty batch
    U, info = reg.solve_batch(torch.zeros((0, reg.Nx), dtype=torch.float64, device="cuda"))
    assert tuple(U.shape) == (0, n)
    # x0 = 0 -> u = 0, one iteration
    U, info = reg.solve_batch(np.zeros((3, reg.Nx)))
    assert np.all(U == 0) and np.all(info["iters"] == 1)
    # ragged batch sizes around the tile boundaries give identical per-sample answers
    rng = np.random.default_rng(0)
    X0 = rng.standard_normal((131, reg.Nx)) * 0.5
    Ufull, _ = reg.solve_batch(X0)
    for Bn in (1, 63, 65, 129):
        Ub, _ = reg.solve_batch(X0[:Bn])
        assert np.array_equal(Ub, Ufull[:Bn])
    # heavily saturated: huge x0 pins almost everything; still exact KKT
    X0 = 50.0 * rng.standard_normal((4, reg.Nx))
    U, info = reg.solve_batch(X0)
    assert float(np.max(info["kkt"])) <= KKT_TOL
    assert np.mean(np.abs(np.abs(U) - 1.0) < 1e-12) > 0.3
    # degenerate bounds lb == ub
    U, info = reg.solve_batch(X0[:2], np.full((2, p.Nu), 0.25), np.full((2, p.Nu), 0.25))
    assert np.all(U == 0.25)
    # max_iter reached -> warning flag, per-sample iters == max_iter
    U, info = reg.solve_batch(X0, max_iter=5)
    assert info["maxiter_hit"] and np.all(info["iters"] == 5)


def test_regulator_warm_start_reduces_iterations(torch_cuda, cstrs_problem, cstr_case):
    torch = torch_cuda
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    p = cstrs_problem
    _, _, datas = cstr_case
    d = datas[0]
    X0 = torch.tensor(np.hstack([d["x"] - d["xs"], d["uprev"] - d["us"]]), device="cuda")
    LB = torch.tensor(p.ulb.T - d["us"], device="cuda"); UB = torch.tensor(p.uub.T - d["us"], device="cuda")
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    state = torch.zeros((X0.shape[0], p.N * p.Nu), dtype=torch.float64, device="cuda")
    U1, i1 = reg.solve_batch(X0, LB, UB, warm_state=state)
    U2, i2 = reg.solve_batch(X0, LB, UB, warm_state=state)     # same problems again, warm
    assert float((U1 - U2).abs().max()) <= 1e-8
    assert int(i2["iters"].max()) <= 5 and int(i1["iters"].max()) > 5


# ------------------------------------------------------------------------------------ target selector
@pytest.mark.parametrize("which", ["cstrs", "cdu_small"])
def test_target_selector_matches_oracle(torch_cuda, which, cstrs_problem, cdu_small_problem):
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    p = cstrs_problem if which == "cstrs" else cdu_small_problem
    ts = LinearMPCController.setup_target_selector(p.A, p.B, p.C, p.H, p.Bd, p.Cd, p.usp, p.Qs, p.Rs, p.ulb, p.uub)
    ots = om.TargetSelectorOracle(A=p.A, B=p.B, C=p.C, H=p.H, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs,
                                  ulb=p.ulb, uub=p.uub)
    for k in ("P", "G", "h", "tA", "tb"):
        assert np.allclose(getattr(ts, k), getattr(ots, k))
    idx = np.arange(0, 60000, 1500)
    YSP, D = p.setpoints[idx], p.disturbances[idx]
    # scale some rows up so that input bounds become active
    YSP = np.vstack([YSP, 4.0 * YSP]); D = np.vstack([D, 4.0 * D])
    xs, us, it = ts.solve_batch(YSP, D, return_iters=True)
    nb = 0
    for i in range(YSP.shape[0]):
        (oxs, ous), info = ots.solve(YSP[i][:, None], D[i][:, None], return_info=True)
        nb += info["n_active"] > 0
        w, ow = np.concatenate([xs[i], us[i]]), np.vstack([oxs, ous])[:, 0]
        q, _, _ = ots.changing(YSP[i][:, None], D[i][:, None])
        c = 0.5 * w @ ots.P @ w + q[:, 0] @ w
        oc = 0.5 * ow @ ots.P @ ow + q[:, 0] @ ow
        assert c <= oc + 1e-9 * max(1.0, abs(oc))                # as good as the oracle's optimum
        assert np.all(us[i] >= p.ulb[:, 0] - 1e-14) and np.all(us[i] <= p.uub[:, 0] + 1e-14)
        assert np.max(np.abs(ots.tA @ w - (ots.tb @ np.concatenate([YSP[i], D[i]])))) <= 1e-9
        assert np.max(np.abs(us[i] - ous[:, 0])) <= 1e-6 and np.max(np.abs(xs[i] - oxs[:, 0])) <= 1e-5
    assert nb > 0 and it.max() < 10 * p.Nu + 20
    # drop-in single solve signature
    oxs1, ous1 = ts.solve(YSP[0][:, None], D[0][:, None])
    assert oxs1.shape == (p.Nx, 1) and ous1.shape == (p.Nu, 1) and len(ts.xs) == 1


# ------------------------------------------------------------------------------------ tcgen05 GEMM
@pytest.mark.parametrize("pair", [0, 1, 2])
@pytest.mark.parametrize("M,n", [(128, 128), (1, 64), (300, 540), (1000, 40), (257, 4480), (2688, 1000)])
def test_lp_split_gemm_matches_fp64(torch_cuda, M, n, pair):
    """The tcgen05 pass C = fp16(A) (T1 + T2)' / s (TMA-fed, TMEM-accumulated) against FP64 NumPy: the
    two-term fp16 operator split carries ~22 bits, the fp32 accumulation ~2^-24 sqrt(K) of sum |a||t|."""
    torch = torch_cuda
    from industrial_nnmpc_2021_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(M * 7 + n)
    A = rng.standard_normal((M, n)) * np.exp(rng.uniform(-6, 2, (M, 1)))
    Bt = rng.standard_normal((n, n)) * np.exp(rng.uniform(-8, 0, (n, n)))
    At, Btt = torch.tensor(A, device="cuda"), torch.tensor(Bt, device="cuda")
    Cd = torch.full((M, n), np.nan, dtype=torch.float64, device="cuda")
    rc = L.nnmpc_lp_gemm_test(M, n, n, _lib.dptr(At), _lib.dptr(Btt), float(np.abs(Bt).max()), _lib.dptr(Cd), pair, None)
    _lib.check(rc, "nnmpc_lp_gemm_test")
    torch.cuda.synchronize()
    A16 = A.astype(np.float16).astype(np.float64)
    ref = A16 @ Bt.T
    bound = 3e-6 * (np.abs(A16) @ np.abs(Bt).T) + 1e-10 * np.abs(A16).sum(axis=1, keepdims=True) * np.abs(Bt).max()
    err = np.abs(Cd.cpu().numpy() - ref)
    assert np.all(np.isfinite(err)) and np.all(err <= bound), float((err / bound).max())


@pytest.mark.parametrize("M,N,K", [(128, 64, 128), (1, 8, 4), (37, 100, 540), (300, 540, 540), (257, 4480, 4480),
                                   (2200, 1000, 1000)])
def test_oz_int8_gemm_is_fp64_accurate(torch_cuda, M, N, K):
    """C = A Bt' on the INT8 tensor cores (error-free base-128 slicing, exact INT32 accumulation) against FP64
    NumPy.  Worst-case bound per element, with 2^f, 2^e the row scales (2^(f+e) < 16 max|a_row| max|b_row|):
    truncation 8 K 2^-58 2^(f+e) plus the FP64 fold of the levels K 2^-55 2^(f+e) - i.e. K 2^-50 max|a| max|b|,
    the worst-case rounding level of an FP64 dot product of that length."""
    torch = torch_cuda
    from industrial_nnmpc_2021_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(M * 7 + N + K)
    A = rng.standard_normal((M, K)) * np.exp(rng.uniform(-6, 2, (M, 1)))
    Bt = rng.standard_normal((N, K)) * np.exp(rng.uniform(-8, 0, (N, K))) * np.exp(rng.uniform(-3, 3, (N, 1)))
    At, Btt = torch.tensor(A, device="cuda"), torch.tensor(Bt, device="cuda")
    Cd = torch.full((M, N), np.nan, dtype=torch.float64, device="cuda")
    _lib.check(L.nnmpc_oz_gemm_test(M, N, K, _lib.dptr(At), _lib.dptr(Btt), _lib.dptr(Cd), None), "nnmpc_oz_gemm_test")
    torch.cuda.synchronize()
    ref = A @ Bt.T
    scale = np.abs(A).max(axis=1, keepdims=True) * np.abs(Bt).max(axis=1)[None, :]
    bound = K * 2.0 ** -50 * scale + 4 * K * 2.0 ** -53 * (np.abs(A) @ np.abs(Bt).T)
    err = np.abs(Cd.cpu().numpy() - ref)
    assert np.all(np.isfinite(err)) and np.all(err <= bound), float((err / bound).max())


# ------------------------------------------------------------------------------------ closed loop
@pytest.fixture(params=["f64", "mixed", "mixed-notail", "mixed-fused", "mixed-oneterm"])
def precision(request, monkeypatch):
    """Arithmetic of the closed-loop iteration: FP64 DMMA, or tcgen05 fp16 increments + FP64 anchors - with the
    automatic switch to skinny FP64 GEMMs for the last few live rows ("mixed"), or tensor-core passes to the end:
    "mixed-notail"  the form large QPs run by default: one fp16 operator term per pass, the second delivered every 8th
                    pass from the pending sums (lp_iter.cuh, deferred second term); the delivery loops are global, so
                    a row's arithmetic path (not its certified optimum) depends on when it started relative to them;
    "mixed-fused"   both operator terms in every pass (the round-1 form, NNMPC_T2_EVERY=0): a row's arithmetic is
                    independent of its neighbours;
    "mixed-oneterm" both terms, except one-term tiles for late-phase rows at an aggressive threshold."""
    monkeypatch.setenv("NNMPC_PRECISION", request.param.split("-")[0])
    for k in ("NNMPC_TAIL_ROWS", "NNMPC_T2_FACTOR", "NNMPC_T2_EVERY"):
        monkeypatch.delenv(k, raising=False)
    if request.param in ("mixed-notail", "mixed-fused", "mixed-oneterm"):
        monkeypatch.setenv("NNMPC_TAIL_ROWS", "0")
    if request.param == "mixed-oneterm":
        monkeypatch.setenv("NNMPC_T2_FACTOR", "10000")
    if request.param == "mixed-notail":
        monkeypatch.setenv("NNMPC_T2_EVERY", "8")       # forced: the default defers only for n >= 1536
    if request.param == "mixed-fused":
        monkeypatch.setenv("NNMPC_T2_EVERY", "0")
    return request.param


@pytest.mark.parametrize("which", ["cstrs", "cdu_small"])
def test_closed_loop_matches_oracle(torch_cuda, which, cstrs_problem, cdu_small_problem, cstr_case, precision):
    """OfflineSimulator data == oracle simulate_offline, sample by sample (SURVEY 4.6)."""
    from industrial_nnmpc_2021_b200.linearMPC import OfflineSimulator
    if which == "cstrs":
        p, T, starts = cstrs_problem, 40, (0, 30000)
        datas = cstr_case[2]
    else:
        p, T, starts = cdu_small_problem, 60, (0, 4000, 9000)
        datas = _closed_loop_samples(p, T, starts)[2]
    sp = np.vstack([p.setpoints[s:s + T] for s in starts])
    ds = np.vstack([p.disturbances[s:s + T] for s in starts])
    sim = OfflineSimulator(**p.controller_kwargs(), xprior=p.xprior, setpoints=sp, disturbances=ds,
                           num_data_gen_task=1, num_process_per_task=len(starts))
    res = sim.generate_batch()
    assert res["x"].shape == (len(starts), T, p.Nx) and not res["maxiter_hit"]
    assert float(res["kkt"].max()) <= KKT_TOL
    for c, od in enumerate(datas):
        assert np.array_equal(res["x"][c][0], p.xprior[:, 0])                     # row 0 = initial state
        for k, tol in (("xs", 1e-6), ("us", 1e-6), ("u", 1e-6), ("uprev", 1e-6), ("x", 1e-6)):
            err = np.max(np.abs(res[k][c] - od[k])) / max(1.0, np.max(np.abs(od[k])))
            assert err <= tol, (which, c, k, err)
        assert np.max(_rel(res["u"][c] - res["us"][c], od["u"] - od["us"], floor=1e-2)) <= 10 * U0_RTOL
    assert res["iters"].min() >= 1


def test_generate_data_files_and_sharding_invariance(torch_cuda, cdu_small_problem, tmp_path, monkeypatch, precision):
    """generate_data writes {task}-{proc}-file per process with the reference's keys; results do not
    depend on how chunks are grouped into batches (SURVEY 4.7)."""
    from industrial_nnmpc_2021_b200.linearMPC import OfflineSimulator, load_training_data
    p = cdu_small_problem
    monkeypatch.chdir(tmp_path)
    sp, ds = p.setpoints[:4 * 25 + 3], p.disturbances[:4 * 25 + 3]      # remainder rows are dropped
    sim = OfflineSimulator(**p.controller_kwargs(), xprior=p.xprior, setpoints=sp, disturbances=ds,
                           num_data_gen_task=2, num_process_per_task=2)
    assert sim.Nsim_each_process == 25
    all4 = sim.generate_batch()
    files = sim.generate_data(task_number=1, data_filename="cdu_offline_data.h5py", stdout_filename="1-out.txt")
    assert len(files) == 2
    for proc in range(2):
        d = load_training_data(f"1-{proc}-cdu_offline_data.h5py")
        assert set(d) == {"x", "uprev", "xs", "us", "u", "data_gen_time"}
        assert d["x"].shape == (25, p.Nx) and d["u"].shape == (25, p.Nu)
        for k in ("x", "uprev", "xs", "us", "u"):
            if precision == "mixed-notail":     # global delivery loops of the second operator term: equal to the solver tolerance
                assert np.max(np.abs(d[k] - all4[k][2 + proc])) <= 1e-7 * max(1.0, np.max(np.abs(d[k]))), k
            else:
                assert np.array_equal(d[k], all4[k][2 + proc]), k     # bitwise: batching does not change results


def test_closed_loop_engine_across_tile_shapes(torch_cuda, cdu_small_problem, precision):
    """Many trajectories of different lengths-to-convergence in one continuously batched run: as
    trajectories finish, the row lists cross the two lower row-count windows of the FP64 GEMM tile
    shapes (<= 48, <= 512 rows; the <= 896 and larger windows start above these 450 trajectories and
    are reached by tests/test_gpu_exact_applies.py), and every trajectory must come out bitwise
    identical to the same trajectory run in a small batch, and equal to the oracle's closed loop
    within the north-star tolerance."""
    from industrial_nnmpc_2021_b200.linearMPC import OfflineSimulator
    p = cdu_small_problem
    Bn, T = 450, 5
    sp, ds = p.setpoints[:Bn * T], p.disturbances[:Bn * T]
    sim = OfflineSimulator(**p.controller_kwargs(), xprior=p.xprior, setpoints=sp, disturbances=ds,
                           num_data_gen_task=1, num_process_per_task=Bn)
    big = sim.generate_batch()
    assert not big["maxiter_hit"] and float(big["kkt"].max()) <= KKT_TOL and big["iters"].min() >= 1
    spc = np.stack(sim.setpoints[0]); dsc = np.stack(sim.disturbances[0])
    for sel in (slice(0, 40), slice(100, 230), slice(449, 450)):
        sub = sim.engine.run(p.xprior, p.uprev, spc[sel], dsc[sel])
        for k in ("x", "uprev", "xs", "us", "u", "iters"):
            if precision in ("mixed", "mixed-notail", "mixed-oneterm"):
                # the automatic FP64 tail / the one-term tiles make the arithmetic path (not the optimum) depend on
                # which other trajectories are live, so batches agree to the solver tolerance, not bitwise
                if k != "iters":
                    assert np.max(np.abs(sub[k] - big[k][sel])) <= 1e-7 * max(1.0, np.max(np.abs(big[k][sel]))), (sel, k)
            else:
                assert np.array_equal(sub[k], big[k][sel]), (sel, k)
    oreg = om.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    ots = om.TargetSelectorOracle(A=p.A, B=p.B, C=p.C, H=p.H, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs,
                                  ulb=p.ulb, uub=p.uub)
    for c in (0, 77, 301, 449):
        od = om.simulate_offline(x0=p.xprior, uprev0=p.uprev, A=p.A, B=p.B, Bd=p.Bd, regulator=oreg, ulb=p.ulb,
                                 uub=p.uub, target_selector=ots, setpoints=spc[c], disturbances=dsc[c])
        for k in ("x", "xs", "us", "u"):
            assert np.max(np.abs(big[k][c] - od[k])) / max(1.0, np.max(np.abs(od[k]))) <= 1e-6, (c, k)


def test_closed_loop_chunk_queue(torch_cuda, cdu_small_problem, precision):
    """More trajectory chunks than slots: finished slots take the next queued chunk (continuous batching).
    Every chunk must come out as when all chunks run side by side."""
    from industrial_nnmpc_2021_b200.linearMPC import OfflineSimulator
    p = cdu_small_problem
    Bn, T = 300, 6
    sim = OfflineSimulator(**p.controller_kwargs(), xprior=p.xprior, setpoints=p.setpoints[:Bn * T],
                           disturbances=p.disturbances[:Bn * T], num_data_gen_task=1, num_process_per_task=Bn)
    wide = sim.generate_batch()
    spc = np.stack(sim.setpoints[0]); dsc = np.stack(sim.disturbances[0])
    rng = np.random.default_rng(3)
    x0 = np.tile(p.xprior.T, (Bn, 1)) + 0.01 * rng.standard_normal((Bn, p.Nx))     # per-chunk initial states
    wide2 = sim.engine.run(x0, p.uprev, spc, dsc)
    for slots in (64, 7):
        sim.engine.set_slots(slots)
        for ref, x_init in ((wide, p.xprior), (wide2, x0)):
            q = sim.engine.run(x_init, p.uprev, spc, dsc)
            assert not q["maxiter_hit"] and float(q["kkt"].max()) <= KKT_TOL
            for k in ("x", "uprev", "xs", "us", "u", "x_final", "uprev_final"):
                if precision in ("mixed", "mixed-notail", "mixed-oneterm"):
                    assert np.max(np.abs(q[k] - ref[k])) <= 1e-7 * max(1.0, np.max(np.abs(ref[k]))), (slots, k)
                else:
                    assert np.array_equal(q[k], ref[k]), (slots, k)
    sim.engine.set_slots(8192)


def test_closed_loop_resume_in_slabs(torch_cuda, cdu_small_problem, precision):
    """A trajectory advanced slab by slab (resume=True keeps the solver state) reproduces the
    single-call run within tolerance and needs no more iterations on the slab boundaries."""
    from industrial_nnmpc_2021_b200.linearMPC import OfflineSimulator
    p = cdu_small_problem
    Bn, T = 6, 24
    sim = OfflineSimulator(**p.controller_kwargs(), xprior=p.xprior, setpoints=p.setpoints[:Bn * T],
                           disturbances=p.disturbances[:Bn * T], num_data_gen_task=1, num_process_per_task=Bn)
    whole = sim.generate_batch()
    spc = np.stack(sim.setpoints[0]); dsc = np.stack(sim.disturbances[0])
    x, up, parts = p.xprior, p.uprev, []
    for i in range(0, T, 8):
        r = sim.engine.run(x, up, spc[:, i:i + 8], dsc[:, i:i + 8], resume=i > 0)
        x, up = r["x_final"], r["uprev_final"]
        parts.append(r)
    for k in ("x", "uprev", "xs", "us", "u"):
        cat = np.concatenate([r[k] for r in parts], axis=1)
        assert np.max(np.abs(cat - whole[k])) <= 1e-7 * max(1.0, np.max(np.abs(whole[k]))), k
    it_cat = np.concatenate([r["iters"] for r in parts], axis=1)
    assert it_cat[:, 8].max() <= whole["iters"][:, 8].max() + 5


# ------------------------------------------------------------------------------------ structured NN
def _random_weights(rng, dims):
    ws = []
    for i in range(len(dims) - 1):
        lim = np.sqrt(6.0 / (dims[i] + dims[i + 1]))
        ws.append(rng.uniform(-lim, lim, (dims[i], dims[i + 1])))
        if i < len(dims) - 2:
            ws.append(0.1 * rng.standard_normal(dims[i + 1]))
    return ws


@pytest.mark.parametrize("nn_precision,nn_tol", [("tc", 1e-6), ("f64", 1e-10), ("fp16", 1e-4)])
@pytest.mark.parametrize("with_uprev,nx,nu,hidden,B", [(True, 12, 6, [224, 224, 224], 300),
                                                        (False, 12, 6, [32, 48], 129),
                                                        (False, 252, 32, [832, 832, 832], 70),
                                                        (True, 252, 32, [832, 1024, 896], 513),
                                                        (True, 7, 3, [33, 17], 50)])
def test_structured_network_matches_numpy(torch_cuda, with_uprev, nx, nu, hidden, B, nn_precision, nn_tol):
    """Arithmetic modes of the layers: "tc" (INT8 tcgen05 digit-plane products with exact accumulation, the default)
    and "f64" (FP64 DMMA) far inside the north-star 1e-5; "fp16" (split-fp16 tcgen05, fp32 accumulation) is the
    measured-and-rejected alternative, checked at its own 1e-4.  Steady-state invariance is exact in all."""
    torch = torch_cuda
    from industrial_nnmpc_2021_b200.LinearMPCLayers import RegulatorLayerWithUprev, RegulatorLayerWithoutUprev
    from industrial_nnmpc_2021_b200.controller_evaluation import NeuralNetworkController
    rng = np.random.default_rng(nx * 100 + nu)
    in_w = 2 * nx + (2 if with_uprev else 1) * nu
    ws = _random_weights(rng, [in_w] + hidden + [nu])
    x, xs = rng.standard_normal((B, nx)), rng.standard_normal((B, nx))
    up, us = rng.uniform(-1, 1, (B, nu)), rng.uniform(-1, 1, (B, nu))
    layer = (RegulatorLayerWithUprev if with_uprev else RegulatorLayerWithoutUprev)(layer_dims=hidden + [nu],
                                                                                    precision=nn_precision)
    layer.set_weights(ws)
    got = [w.shape for w in layer.get_weights()]
    assert got == [w.shape for w in ws]
    inputs = [x, up, xs, us] if with_uprev else [x, xs, us]
    out = layer(inputs)
    ref = onn.layer_call(ws, inputs, with_uprev)
    assert out.shape == (B, nu) and np.max(np.abs(out - ref)) <= nn_tol, np.max(np.abs(out - ref))
    # inputs an order of magnitude away from O(1) (unscaled states): the per-row scales follow them
    big = [a * 37.0 for a in inputs[:-1]] + [inputs[-1]]
    assert np.max(np.abs(layer(big) - onn.layer_call(ws, big, with_uprev))) <= nn_tol * 37.0
    # device tensors in -> device tensor out, same numbers
    tin = [torch.tensor(a, device="cuda") for a in inputs]
    assert np.array_equal(layer(tin).cpu().numpy(), out)
    # steady-state invariance (paper eq. 8): x = xs (and uprev = us) => output == us for ANY weights
    inv = [xs, us, xs, us] if with_uprev else [xs, xs, us]
    assert np.array_equal(layer(inv), us)
    # deployment form: scaling + clip, column by column vs controller_evaluation.py:863-892
    xscale = rng.uniform(0.5, 2.0, nx)
    ulb, uub = -0.3 * np.ones((nu, 1)), 0.4 * np.ones((nu, 1))
    ctl = NeuralNetworkController(regulator_weights=ws, xscale=xscale, nnwithuprev=with_uprev, ulb=ulb, uub=uub,
                                  precision=nn_precision)
    ub = ctl.control_input_batch(x, up, xs, us)
    for i in range(0, B, max(1, B // 7)):
        col = lambda a: a[i][:, None]
        r = onn.control_input(ws, col(x), col(up), col(xs), col(us), with_uprev, xscale[:, None], ulb, uub)
        assert np.max(np.abs(ub[i] - r[:, 0])) <= nn_tol
    assert np.all(ub <= 0.4) and np.all(ub >= -0.3)


def test_regulator_model_wrapper(torch_cuda):
    from industrial_nnmpc_2021_b200.LinearMPCLayers import RegulatorModel
    m = RegulatorModel(Nx=12, Nu=6, regulator_dims=[999, 64, 64, 6], nnwithuprev=False, seed=1, precision="f64")
    ws = m.get_weights()
    assert [w.shape for w in ws] == [(30, 64), (64,), (64, 64), (64,), (64, 6)]     # dims[0] ignored (:128)
    rng = np.random.default_rng(0)
    x, xs, us = rng.standard_normal((10, 12)), rng.standard_normal((10, 12)), rng.standard_normal((10, 6))
    assert np.max(np.abs(m([x, xs, us]) - onn.layer_call(ws, [x, xs, us], False))) <= 1e-10


# ------------------------------------------------------------------------------------ batched QPs through the engine
@pytest.mark.parametrize("qp_precision", ["mixed", "f64"])
def test_regulator_batch_through_engine_matches_oracle(torch_cuda, cstrs_problem, cstr_case, qp_precision):
    """solve_batch(precision=...): cold QPs through the continuously batched engine (nnmpc_sim_solve_qps), more QPs
    than slots, against the exact CPU optimum and the lock-step FP64 solver."""
    torch = torch_cuda
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    p = cstrs_problem
    oreg, _, datas = cstr_case
    d = {k: np.vstack([x[k] for x in datas]) for k in datas[0]}
    X0 = np.hstack([d["x"] - d["xs"], d["uprev"] - d["us"]])
    LB, UB = p.ulb.T - d["us"], p.uub.T - d["us"]
    rng = np.random.default_rng(1)
    X0 = np.vstack([X0, X0 * rng.uniform(0.2, 3.0, (X0.shape[0], 1))])          # 160 QPs
    LB, UB = np.vstack([LB, LB]), np.vstack([UB, UB])
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    t = lambda a: torch.tensor(a, device="cuda")
    U, info = reg.solve_batch(t(X0), t(LB), t(UB), precision=qp_precision, slots=48)
    Uref, iref = reg.solve_batch(t(X0), t(LB), t(UB))
    assert not info["maxiter_hit"] and float(info["kkt"].max()) <= KKT_TOL
    assert float((U - Uref).abs().max()) <= 1e-7
    U, cost = U.cpu().numpy(), info["cost"].cpu().numpy()
    box = oq.BoxQP(oreg.P)
    nact = 0
    for i in range(0, X0.shape[0], 3):
        q = oreg.tq @ X0[i]
        lb, ub = np.tile(LB[i], p.N), np.tile(UB[i], p.N)
        ue, ei = box.solve(q, lb, ub)
        nact += ei["n_active"] > 0
        assert oq.box_kkt_residual(oreg.P, q, U[i], lb, ub) <= KKT_TOL
        assert _rel(U[i][:p.Nu], ue[:p.Nu])[0] <= U0_RTOL
        assert abs(cost[i] - ei["cost"]) <= COST_RTOL * max(abs(ei["cost"]), 1e-6)
    assert nact > 10
    # NumPy in -> NumPy out through the same engine
    U2, info2 = reg.solve_batch(X0, LB, UB, precision=qp_precision, slots=48)
    assert np.max(np.abs(U2 - U)) <= 1e-7 and float(np.max(info2["kkt"])) <= KKT_TOL
