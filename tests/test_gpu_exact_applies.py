"""The exact operator applies of the closed-loop engine, called as the engine calls them (nnmpc_exact_apply_test):
the anchor x = Top w - c, the KKT check g = P z + q with its residual ||z - clip(z - g, lb, ub)||_inf folded into kres,
and the plain apply, on the FP64 DMMA pipe and on every kernel variant of the INT8 digit-plane pipe.  Each call goes
through a permuted row list whose length lives on the device, as in the engine, against a float64 NumPy reference.

Error bounds per element, with scale = max|a_row| max|op_row| and 2^(f+e) <= 16 scale the power-of-two row scales of the
INT8 slicing:  truncation (LMAX+1) K 2^(-7 (LMAX+1) - 2) 2^(f+e) (LMAX = 5 for the anchor, 7 for the check and the
plain apply) plus the FP64 fold of the levels K 2^-55 2^(f+e) (test_gpu_parity.test_oz_int8_gemm_is_fp64_accurate);
on either pipe plus 4 K 2^-53 sum |a||op| for the float64 reference and the DMMA accumulation, and 2^-52 |result| for
the final add.  The residual r = |z - clip(z - g)| is 1-Lipschitz in g, so kres may differ from the reference residual
by the largest g bound of its row plus the rounding of the two subtractions.

The INT8 variants agree within these bounds.  Bitwise (test_int8_variants_agree prints the counts; measured on one B200):
the 6-level anchors agree in all four variants; the 8-level applies agree between variants 0 and 1 (all levels folded
in one FP64 Horner scheme) and between 2 and 3 (low level window folded in integers), and the two pairs differ in the
last bits of a few per cent of the entries.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import linear_mpc as om
from oracle import qp as oq

TOL = 1e-9                      # the engine's certification tolerance (linearMPC.DEFAULT_TOL)
ANCHOR, CHECK, STORE = 0, 1, 2
PIPES = [pytest.param((0, -1), id="dmma")] + [pytest.param((1, v), id=f"int8-v{v}") for v in range(4)]
INT8 = [p for p in PIPES if p.values[0][0] == 1]
B = 1000                        # physical rows of the operands
# device row counts: every window of gemm_by_count (<= 48, <= 512, <= 896, above) and the 128-row INT8 tiles, each edge
# from both sides; 1000 = max_rows
COUNTS = (0, 1, 47, 48, 49, 127, 128, 129, 511, 512, 513, 895, 896, 897, 1000)
COUNTS_LARGE_N = (1, 49, 513, 897, 1000)
SENTINEL = -1.2345e300
EPS = 2.0 ** -53
INF_BITS = 0x7FF0000000000000
NNMPC_ERR_BADARG = -1


@pytest.fixture(scope="module")
def torch_cuda(built_lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _apply(torch, kind, pipe, Op, A, rows, count, C=None, lb=None, ub=None, X=None, kres=None, nu=1, max_rows=None):
    """One call of the hook on device tensors; returns (status, message)."""
    from industrial_nnmpc_2021_b200 import _lib
    L = _lib.lib()
    cnt = torch.tensor([count], dtype=torch.int32, device="cuda")
    rc = L.nnmpc_exact_apply_test(kind, pipe[0], pipe[1], A.shape[0], A.shape[1], nu, _lib.dptr(Op),
                                  None if rows is None else _lib.dptr_i32(rows), _lib.dptr_i32(cnt),
                                  A.shape[0] if max_rows is None else max_rows, _lib.dptr(A), _lib.dptr(C),
                                  _lib.dptr(lb), _lib.dptr(ub), _lib.dptr(X),
                                  None if kres is None else _lib.dptr(kres, torch.int64), None)
    return rc, L.nnmpc_last_error().decode(errors="replace")


def _call(torch, *args, **kw):
    rc, msg = _apply(torch, *args, **kw)
    assert rc == 0, msg


def _bound(pipe, kind, K, ref, absref, scale):
    b = 4 * K * EPS * absref + 2 * EPS * np.abs(ref)
    if pipe[0] == 1:
        lmax = 5 if kind == ANCHOR else 7
        b = b + 16 * ((lmax + 1) * K * 2.0 ** (-7 * (lmax + 1) - 2) + K * 2.0 ** -55) * scale
    return b


def _residual(z, g, lb, ub):
    """per row max |z - clip(z - g, lb[k], ub[k])|, k = column % nu (float64, as the kernels compute it)."""
    nu = lb.shape[1]
    k = np.arange(z.shape[1]) % nu
    return np.max(np.abs(z - np.minimum(np.maximum(z - g, lb[:, k]), ub[:, k])), axis=1)


def _spd(rng, n, spread):
    """Symmetric, diagonally dominant (hence SPD) n x n matrix with row scales 2^U(-spread, spread)."""
    S = rng.standard_normal((n, n)) * np.exp(rng.uniform(-4, 0, (n, n)))
    M = S + S.T
    M[np.diag_indices(n)] = np.abs(M).sum(axis=1) + 1.0
    d = 2.0 ** rng.uniform(-spread, spread, n)
    return d[:, None] * M * d[None, :]


def _regulator(p):
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    assert not reg.reparameterize
    Minv = np.linalg.inv(reg.P + np.diag(reg.rho_vec))
    Top = 0.5 * (Minv + Minv.T) * reg.rho_vec[None, :]
    return reg, Top


# ------------------------------------------------------------------------------------ operators
CASES = ["cstrs", "cdu_small", "syn130_nu2", "syn258_nu3", "syn540_nu4", "syn1000_nu4", "syn4480_nu32",
         "syn8960_nu32"]


@pytest.fixture(scope="module", params=CASES)
def case(request, torch_cuda, cstrs_problem, cdu_small_problem):
    """Operators (anchor: Top, check and plain apply: P), B operand rows with row scales over 2^-6 .. 2^2, per-row
    stage bounds, and the float64 references of both operators."""
    torch = torch_cuda
    name = request.param
    rng = np.random.default_rng(CASES.index(name))
    if name in ("cstrs", "cdu_small"):
        p = cstrs_problem if name == "cstrs" else cdu_small_problem
        reg, Top = _regulator(p)
        P, nu = reg.P, p.Nu
    else:
        n, nu = (int(s) for s in name[3:].split("_nu"))
        P = _spd(rng, n, 8.0)
        Top = P                 # |Top| <= 1 only matters to the engine; the bounds scale with the rows
    n = P.shape[0]
    A = rng.standard_normal((B, n)) * 2.0 ** rng.uniform(-6, 2, (B, 1))
    C = rng.standard_normal((B, n)) * 2.0 ** rng.uniform(-4, 4, (B, 1))
    lb = -rng.uniform(0.01, 1.0, (B, nu)) * 2.0 ** rng.uniform(-6, 2, (B, 1))
    ub = rng.uniform(0.01, 1.0, (B, nu)) * 2.0 ** rng.uniform(-6, 2, (B, 1))
    d = dict(name=name, n=n, nu=nu, A=A, C=C, lb=lb, ub=ub, perm=rng.permutation(B).astype(np.int32),
             prior_f=rng.choice([0.0, 0.5, 2.0], B))
    amax = np.abs(A).max(axis=1)[:, None]
    for key, Op in (("P", P), ("top", Top)):
        if key == "top" and Op is P:
            d["top"] = d["P"]
            continue
        d[key] = dict(host=Op, dev=torch.tensor(Op, device="cuda"), ref=A @ Op.T, absref=np.abs(A) @ np.abs(Op).T,
                      scale=amax * np.abs(Op).max(axis=1)[None, :])
    return d


@pytest.mark.parametrize("kind", [ANCHOR, CHECK, STORE], ids=["anchor", "check", "store"])
@pytest.mark.parametrize("pipe", PIPES)
def test_listed_rows_match_reference(torch_cuda, case, pipe, kind):
    """Every device row count, over a permuted row list: the listed rows within the bound of the pipe, every other row
    of X / G / kres bitwise as it was; kres = max(prior, residual) with priors below and above the residual."""
    torch = torch_cuda
    d, n, nu = case, case["n"], case["nu"]
    op = d["top"] if kind == ANCHOR else d["P"]
    sign = {ANCHOR: -1.0, CHECK: 1.0, STORE: 0.0}[kind]
    ref = op["ref"] + sign * d["C"]
    bound = _bound(pipe, kind, n, ref, op["absref"], op["scale"])
    tdev = lambda a: torch.tensor(a, device="cuda")
    A, Cd, lb, ub, rows = tdev(d["A"]), tdev(d["C"]), tdev(d["lb"]), tdev(d["ub"]), tdev(d["perm"])
    if kind == CHECK:
        rref = _residual(d["A"], ref, d["lb"], d["ub"])
        gb = bound.max(axis=1) + 4 * EPS * (np.abs(d["A"]) + np.abs(ref)).max(axis=1)
        prior = rref * d["prior_f"]
        prior[d["perm"][::7]] = SENTINEL * -1.0      # huge priors stay
    for count in (COUNTS_LARGE_N if n >= 4096 else COUNTS):
        X = torch.full((B, n), SENTINEL, dtype=torch.float64, device="cuda")
        kres = torch.tensor(prior, device="cuda").view(torch.int64) if kind == CHECK else None
        _call(torch, kind, pipe, op["dev"], A, rows, count, C=None if kind == STORE else Cd, lb=lb, ub=ub, X=X,
              kres=kres, nu=nu, max_rows=B)
        on, off = d["perm"][:count], d["perm"][count:]
        Xh = X.cpu().numpy()
        assert np.all(Xh[off] == SENTINEL), (count, "unlisted rows written")
        err = np.abs(Xh[on] - ref[on])
        assert np.all(err <= bound[on]), (count, float(np.max(err / bound[on])) if err.size else 0.0)
        if kind == CHECK:
            kh = kres.cpu().numpy().view(np.float64)
            assert np.array_equal(kh[off].view(np.uint64), prior[off].view(np.uint64)), (count, "unlisted kres")
            want = np.maximum(prior[on], rref[on])
            assert np.all(np.abs(kh[on] - want) <= gb[on]), (count, float(np.max(np.abs(kh[on] - want) / gb[on])))
            above = prior[on] > rref[on] + gb[on]
            assert np.array_equal(kh[on][above], prior[on][above]), (count, "a larger prior was overwritten")
            if count == B:      # without G the same residuals
                k2 = torch.tensor(prior, device="cuda").view(torch.int64)
                _call(torch, kind, pipe, op["dev"], A, rows, count, C=Cd, lb=lb, ub=ub, X=None, kres=k2, nu=nu)
                assert torch.equal(k2, kres)


# ------------------------------------------------------------------------------------ certification at tol
def _closed_loop_qps(p, T, starts):
    """Regulator QPs (x0, stage bounds) visited by the oracle's closed loop, so that bounds are active."""
    reg = om.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    ts = om.TargetSelectorOracle(A=p.A, B=p.B, C=p.C, H=p.H, Bd=p.Bd, Cd=p.Cd, usp=p.usp, Rs=p.Rs, Qs=p.Qs,
                                 ulb=p.ulb, uub=p.uub)
    ds = [om.simulate_offline(x0=p.xprior, uprev0=p.uprev, A=p.A, B=p.B, Bd=p.Bd, regulator=reg, ulb=p.ulb, uub=p.uub,
                              target_selector=ts, setpoints=p.setpoints[s:s + T], disturbances=p.disturbances[s:s + T])
          for s in starts]
    d = {k: np.vstack([x[k] for x in ds]) for k in ("x", "xs", "uprev", "us")}
    return np.hstack([d["x"] - d["xs"], d["uprev"] - d["us"]]), p.ulb.T - d["us"], p.uub.T - d["us"]


@pytest.fixture(scope="module", params=["cstrs", "cdu_small", "syn130_nu2"])
def optima(request, torch_cuda, cstrs_problem, cdu_small_problem):
    """Exact box-QP optima z (oracle.qp.BoxQP) with active bounds and distinct bounds per stage index, then two
    copies of every row moved off the optimum: one free coordinate (the last one), and one coordinate at a bound."""
    rng = np.random.default_rng(11)
    if request.param == "syn130_nu2":
        n, nu, S = 130, 2, 60
        P = _spd(rng, n, 2.0)
        LB, UB = -rng.uniform(0.2, 1.0, (S, nu)), rng.uniform(0.2, 1.0, (S, nu))
        Q = -(P @ rng.uniform(-2.0, 2.0, (n, S))).T
    else:
        p = cstrs_problem if request.param == "cstrs" else cdu_small_problem
        reg, _ = _regulator(p)
        X0, LB, UB = _closed_loop_qps(p, 40 if request.param == "cstrs" else 30, (0, 30000) if request.param == "cstrs"
                                      else (0, 4000))
        P, nu = reg.P, p.Nu
        Q = X0 @ reg.tq.T
    n = P.shape[0]
    span = (UB - LB).max(axis=1, keepdims=True)
    LB, UB = LB - 0.031 * span * np.arange(nu), UB + 0.023 * span * np.arange(nu)    # distinct per stage index
    assert all(len(np.unique(LB[i])) == nu and len(np.unique(UB[i])) == nu for i in range(len(LB)))
    box = oq.BoxQP(P)
    Z = np.array([box.solve(Q[i], np.tile(LB[i], n // nu), np.tile(UB[i], n // nu))[0] for i in range(len(Q))])
    assert np.all(_residual(Z, Z @ P.T + Q, LB, UB) <= 1e-11)
    k = np.arange(n) % nu
    act = (Z <= LB[:, k]) | (Z >= UB[:, k])
    assert act.any(axis=1).sum() >= 10, "the optima must have active bounds"
    Zf = Z.copy()
    for i in range(len(Z)):
        j = np.flatnonzero(~act[i])[-1]                        # last free coordinate
        step = 1e-7 / max(P[j, j], 1e-3)
        Zf[i, j] += step if UB[i, k[j]] - Z[i, j] > LB[i, k[j]] - Z[i, j] + 2 * step else -step
    ia = np.flatnonzero(act.any(axis=1))
    Za = Z[ia].copy()
    G = Z @ P.T + Q
    for r, i in enumerate(ia):
        j = np.flatnonzero(act[i])[np.argmax(np.abs(G[i, act[i]]))]   # strongest active bound
        Za[r, j] += 1e-7 if Z[i, j] <= LB[i, k[j]] else -1e-7           # moved inward by 1e-7
    Zall = np.vstack([Z, Zf, Za])
    Qall, LBall, UBall = np.vstack([Q, Q, Q[ia]]), np.vstack([LB, LB, LB[ia]]), np.vstack([UB, UB, UB[ia]])
    rref = _residual(Zall, Zall @ P.T + Qall, LBall, UBall)
    moved = np.arange(len(Zall)) >= len(Z)
    assert np.all(rref[moved] >= 10 * TOL)
    return dict(P=P, nu=nu, Z=Zall, Q=Qall, LB=LBall, UB=UBall, rref=rref, moved=moved)


@pytest.mark.parametrize("pipe", PIPES)
def test_check_certifies_optima_at_tol(torch_cuda, optima, pipe):
    """The property the engine relies on: at the exact optimum kres <= tol, and a point moved by one coordinate so
    that its residual is >= 10 tol fails.  A wrong stage index of the bounds, swapped bounds or a dropped column chunk
    certify the wrong rows."""
    torch = torch_cuda
    o = optima
    t = lambda a: torch.tensor(a, device="cuda")
    Bn, n = o["Z"].shape
    rows = t(np.random.default_rng(5).permutation(Bn).astype(np.int32))
    kres = torch.zeros(Bn, dtype=torch.int64, device="cuda")
    G = torch.full((Bn, n), SENTINEL, dtype=torch.float64, device="cuda")
    _call(torch, CHECK, pipe, t(o["P"]), t(o["Z"]), rows, Bn, C=t(o["Q"]), lb=t(o["LB"]), ub=t(o["UB"]), X=G,
          kres=kres, nu=o["nu"])
    kh = kres.cpu().numpy().view(np.float64)
    bad = np.flatnonzero(~o["moved"] & (kh > TOL))
    assert bad.size == 0, ("optimum not certified", bad[:8], kh[bad[:8]])
    missed = np.flatnonzero(o["moved"] & ~(kh > TOL))
    assert missed.size == 0, ("moved point certified", missed[:8], o["rref"][missed[:8]], kh[missed[:8]])
    gref = o["Z"] @ o["P"].T + o["Q"]
    bound = _bound(pipe, CHECK, n, gref, np.abs(o["Z"]) @ np.abs(o["P"]).T + np.abs(o["Q"]),
                   np.abs(o["Z"]).max(axis=1)[:, None] * np.abs(o["P"]).max(axis=1)[None, :])
    assert np.all(np.abs(G.cpu().numpy() - gref) <= bound)


# ------------------------------------------------------------------------------------ non-finite and zero rows
@pytest.mark.parametrize("pipe", PIPES)
def test_nonfinite_and_zero_rows(torch_cuda, pipe):
    """A NaN in z or an infinite q gives kres = +Inf for that row only, a NaN in w a NaN anchor row only, and an
    all-zero z (a cold start from x0 = 0) gives exactly g = q; the other rows of the same 128-row tiles stay exact.
    (The NaN row once sliced as if the NaN were 0: the row-maximum reduction of k_oz_slice dropped a NaN it held.)"""
    torch = torch_cuda
    rng = np.random.default_rng(7)
    n, nu, Bn = 258, 3, 300
    P = _spd(rng, n, 3.0)
    Z = rng.standard_normal((Bn, n)) * 2.0 ** rng.uniform(-4, 2, (Bn, 1))
    Q = rng.standard_normal((Bn, n))
    LB, UB = -rng.uniform(0.1, 1.0, (Bn, nu)), rng.uniform(0.1, 1.0, (Bn, nu))
    perm = rng.permutation(Bn).astype(np.int32)
    nan_z, inf_q, minf_q, zero = perm[3], perm[40], perm[41], perm[100]    # list positions inside the first tile
    Z[nan_z, 17] = np.nan
    Q[inf_q, n - 1] = np.inf
    Q[minf_q, 5] = -np.inf
    Z[zero] = 0.0
    t = lambda a: torch.tensor(a, device="cuda")
    Pd, rows = t(P), t(perm)
    kres = torch.zeros(Bn, dtype=torch.int64, device="cuda")
    G = torch.full((Bn, n), SENTINEL, dtype=torch.float64, device="cuda")
    _call(torch, CHECK, pipe, Pd, t(Z), rows, Bn, C=t(Q), lb=t(LB), ub=t(UB), X=G, kres=kres, nu=nu)
    kb, Gh = kres.cpu().numpy(), G.cpu().numpy()
    special = [nan_z, inf_q, minf_q]
    assert np.all(kb[special] == INF_BITS), kb[special]
    assert np.isposinf(Gh[inf_q, n - 1]) and np.isneginf(Gh[minf_q, 5]) and np.all(np.isnan(Gh[nan_z]))
    assert np.array_equal(Gh[zero], Q[zero])                               # g = P 0 + q exactly
    ok = np.setdiff1d(np.arange(Bn), special)
    Zs = np.where(np.isfinite(Z), Z, 0.0)
    gref = Zs @ P.T + Q
    bound = _bound(pipe, CHECK, n, gref, np.abs(Zs) @ np.abs(P).T + np.abs(Q),
                   np.abs(Zs).max(axis=1)[:, None] * np.abs(P).max(axis=1)[None, :])
    assert np.all(np.abs(Gh[ok] - gref[ok]) <= bound[ok])
    rref = _residual(Zs[ok], gref[ok], LB[ok], UB[ok])
    kh = kb.view(np.float64)
    assert np.all(np.abs(kh[ok] - rref) <= bound[ok].max(axis=1) + 4 * EPS * (np.abs(Zs[ok]) + np.abs(gref[ok])).max(axis=1))
    assert kh[zero] == _residual(Z[zero:zero + 1], Q[zero:zero + 1], LB[zero:zero + 1], UB[zero:zero + 1])[0] > 0
    # anchor: a NaN in w poisons its own row of x and no other
    W = rng.standard_normal((Bn, n))
    W[nan_z, 200] = np.nan
    X = torch.full((Bn, n), SENTINEL, dtype=torch.float64, device="cuda")
    _call(torch, ANCHOR, pipe, Pd, t(W), rows, Bn, C=t(Q), X=X)
    Xh = X.cpu().numpy()
    assert np.all(np.isnan(Xh[nan_z]))
    rest = np.setdiff1d(np.arange(Bn), [nan_z])
    Ws = np.where(np.isfinite(W), W, 0.0)
    xref = Ws @ P.T - Q
    xb = _bound(pipe, ANCHOR, n, xref, np.abs(Ws) @ np.abs(P).T + np.abs(Q),
                np.abs(Ws).max(axis=1)[:, None] * np.abs(P).max(axis=1)[None, :])
    ok = np.setdiff1d(rest, [inf_q, minf_q])
    assert np.all(np.abs(Xh[ok] - xref[ok]) <= xb[ok])


# ------------------------------------------------------------------------------------ variants against each other
def test_int8_variants_agree(torch_cuda, cstrs_problem):
    """All INT8 variants within the bound of each other (twice the bound against the reference); bitwise agreement is
    not required, the counts of differing entries are printed."""
    torch = torch_cuda
    reg, Top = _regulator(cstrs_problem)
    rng = np.random.default_rng(3)
    n = reg.P.shape[0]
    A = rng.standard_normal((B, n)) * 2.0 ** rng.uniform(-6, 2, (B, 1))
    C = rng.standard_normal((B, n))
    t = lambda a: torch.tensor(a, device="cuda")
    rows = t(rng.permutation(B).astype(np.int32))
    for kind, Op in ((ANCHOR, Top), (STORE, reg.P)):
        outs = []
        for v in range(4):
            X = torch.zeros((B, n), dtype=torch.float64, device="cuda")
            _call(torch, kind, (1, v), t(Op), t(A), rows, 700, C=t(C), X=X, max_rows=B)
            outs.append(X.cpu().numpy())
        ref = A @ Op.T - (C if kind == ANCHOR else 0.0)
        bound = _bound((1, 0), kind, n, ref, np.abs(A) @ np.abs(Op).T, np.abs(A).max(axis=1)[:, None] * np.abs(Op).max(axis=1)[None, :])
        for v in range(1, 4):
            assert np.all(np.abs(outs[v] - outs[0]) <= 2 * bound)
        diff = {f"{a}-{b}": int(np.sum(outs[a].view(np.uint64) != outs[b].view(np.uint64)))
                for a in range(4) for b in range(a + 1, 4)}
        print(f"kind {kind}: entries differing bitwise between variants {diff}")


# ------------------------------------------------------------------------------------ the length limit
@pytest.fixture(scope="module")
def longest(torch_cuda):
    """K = 32768, the longest contraction the INT8 pipe accepts, with the digits that make every level sum as large as
    the slicing allows: all entries of a row of one sign and of magnitude 126/127 2^e, whose base-128 digits are all 63.
    The exact result is K a b."""
    torch = torch_cuda
    K, Bn = 32768, 130
    c, a = 126.0 / 127.0, 126.0 / 127.0 * 0.125
    osc = 2.0 ** np.arange(-3, 5)[np.arange(K) % 8] * np.where(np.arange(K) % 3 == 0, -1.0, 1.0)    # per operator row
    asc = 2.0 ** np.arange(-2, 3)[np.arange(Bn) % 5] * np.where(np.arange(Bn) % 2 == 0, -1.0, 1.0)  # per sample row
    Op = torch.full((K, K), c, dtype=torch.float64, device="cuda").mul_(torch.tensor(osc, device="cuda")[:, None])
    A = torch.full((Bn, K), a, dtype=torch.float64, device="cuda") * torch.tensor(asc, device="cuda")[:, None]
    ref = (np.longdouble(K) * np.longdouble(a) * np.longdouble(c)) * asc[:, None].astype(np.longdouble) \
        * osc[None, :].astype(np.longdouble)
    yield Op, A, ref.astype(np.float64), np.abs(a * asc)[:, None] * np.abs(c * osc)[None, :]
    del Op, A
    torch.cuda.empty_cache()


@pytest.mark.parametrize("pipe", INT8)
def test_int8_length_limit(torch_cuda, longest, pipe):
    torch = torch_cuda
    Op, A, ref, scale = longest
    K, Bn = Op.shape[0], A.shape[0]
    rows = torch.tensor(np.random.default_rng(2).permutation(Bn).astype(np.int32), device="cuda")
    X = torch.full((Bn, K), SENTINEL, dtype=torch.float64, device="cuda")
    _call(torch, STORE, pipe, Op, A, rows, Bn, X=X)
    absref = np.abs(ref)
    err = np.abs(X.cpu().numpy() - ref)
    assert np.all(err <= _bound(pipe, STORE, K, ref, absref, scale)), float(err.max())


@pytest.mark.parametrize("pipe", INT8)
def test_int8_rejects_longer_contractions(torch_cuda, pipe):
    """One column more than 32768 is refused with a message, before the operator is read."""
    torch = torch_cuda
    for K in (32769, 32770):
        Op = torch.empty((K, K), dtype=torch.float64, device="cuda")
        A = torch.zeros((4, K), dtype=torch.float64, device="cuda")
        X = torch.zeros((4, K), dtype=torch.float64, device="cuda")
        rc, msg = _apply(torch, STORE, pipe, Op, A, None, 4, X=X)
        assert rc == NNMPC_ERR_BADARG and msg, (K, rc, msg)
        if K % 2 == 0:
            assert "32768" in msg, msg
        del Op
    torch.cuda.empty_cache()
