"""The mixed-precision iteration of the regulator QP at kernel level (nnmpc_lp_step_test): the tcgen05 pass with its
Douglas-Rachford epilogue (EpiDelta) in every tile variant, the deferred second-term delivery (EpiAddX), the fp16
operator split and the FP64 kernels around the anchors, each called as the closed-loop engine calls it and compared
with a float64 NumPy restatement of the formulas in the header of lp_iter.cuh.

The closed-loop tests cannot see a pass that is subtly wrong: every returned point is re-certified by an FP64 KKT check
and a failed check re-anchors the row, so a wrong epilogue costs iterations, not answers.  Here each output is checked
on its own.

Bounds.  The pass accumulates  acc = dq . (T1 + T2)^T  (dq, T1, T2 fp16) in fp32 on the tensor cores, K = 16 products
per MMA step, steps = terms * ceil(n / 16) (terms = 2 for a two-term tile, 1 for a one-term pass or a tile whose need2
flag is 0).  The fp16 products are exact in fp32 and in float64, so the float64 reference of the same products is exact
to 2^-53 n relative.  As a model of the accumulation (not a hardware specification) each step adds its 16 products to
the fp32 accumulator with an error of at most 2^-22 (one truncation of the sum and one of the operand alignment, each
below one fp32 ulp) relative to the sum of |products| so far, so
    |acc - ref| <= steps 2^-22 sum_k |dq_k| (|T1_jk| + |T2_jk|)          (|T2| only when the tile has two terms).
At n = 4480 this is 1.3e-4 of sum |dq||T|; profiles/r02c_fp16_accumulation_error.txt measured at most 2.2e-6, split
error included.  The state moves by acc / (s_T sc_in), both powers of two, so X_out - X_in must lie within that bound
over s_T sc_in of ref / (s_T sc_in), plus the rounding of the FP64 add.

Downstream of the GPU's own X_out everything is checked to one FP64 rounding per operation (FMA contraction allowed),
and bitwise where the operation order leaves no freedom: V_out = V + alpha (X_out - clip(V)) to two roundings;
dw = (2 clip(V_out) - V_out) - ((2 clip(V) - V) - E), from V_out, exactly; q = fp16(clamp(dw sc_out, +-60000)) within
one fp16 ulp under any rounding; E_out = fp32(dw - q / sc_out) bitwise; the conservation law
(w_out - E_out) - (w_in - E_in) = q / sc_out up to the fp32 rounding of E_out; dres = max(prior, fp32 max |d|)
bitwise, +Inf when that maximum is not finite; the pending sums bitwise.  The FP64 helper kernels are checked bitwise
where their arithmetic is a fixed sequence of correctly rounded operations, to one rounding where an FMA may be
formed, and their power-of-two scales exactly.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OPS = {"split": 0, "anchor_prep": 1, "dr_first": 2, "reanchor": 3, "emit": 4, "iterate": 5, "correct": 6}
ITER, CAND, EMIT = 1, 2, 6          # row states of the engine (sim.cu SlotState)
# (s_mode, kernel): every tile variant of the pass
PASSES = [pytest.param((0, 0), id="2term-128"), pytest.param((0, 1), id="2term-256"),
          pytest.param((0, 2), id="2term-pair"), pytest.param((1, 0), id="1term-128-add"),
          pytest.param((1, 1), id="1term-256-add"), pytest.param((2, 0), id="1term-128-new"),
          pytest.param((2, 1), id="1term-256-new")]
EPS = 2.0 ** -53
INF_BITS = 0x7FF0000000000000
SENT16 = 0x5A5A                      # fp16 sentinel of operand rows no kernel may write
SENT64 = -1.2345e300
NNMPC_ERR_BADARG = -1


@pytest.fixture(scope="module")
def torch_cuda(built_lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


# ------------------------------------------------------------------------------------ the hook
def _step(torch, op, n, nu, B, kernel=-1, s_mode=0, alpha=1.6, Top=None, top_max=0.0, rows=None, count=0,
          list_r=None, len_r=0, pos_w=None, pos_r=None, state=None, iter_state=ITER, emit_state=EMIT, need2=None,
          X=None, V=None, W=None, E=None, sc_in=None, sc_out=None, sS=None, dres=None, it=None, dtrig=None,
          rinv=None, Z=None, lb=None, ub=None, D_in=None, S_in=None, D_out=None, S_out=None, tile_stat=None,
          lb_dev=None, ub_dev=None):
    """One call on device copies of the given NumPy arrays.  Returns (status, message, outputs): the outputs are the
    arrays after the call, as NumPy (fp16 as uint16 bit patterns)."""
    from industrial_nnmpc_2021_b200 import _lib
    L = _lib.lib()
    dev = {}

    def put(name, a, dt):
        if a is None:
            return None
        a = np.ascontiguousarray(a)
        if dt is torch.int16:
            a = a.view(np.int16)
        elif dt is torch.int64:
            a = a.view(np.int64)
        t = torch.tensor(a, dtype=dt, device="cuda")
        dev[name] = t
        return _lib.dptr(t, dt)
    f64, f32, i32, i16, i64, u8 = torch.float64, torch.float32, torch.int32, torch.int16, torch.int64, torch.uint8
    args = [OPS[op], kernel, s_mode, alpha, n, nu, B, put("Top", Top, f64), float(top_max),
            put("rows", rows, i32), put("count", None if rows is None else np.array([count]), i32),
            put("list_r", list_r, i32), put("len_r", np.array([len_r]) if op in ("iterate", "correct") else None, i32),
            put("pos_w", pos_w, i32), put("pos_r", pos_r, i32), put("state", state, i32), iter_state, emit_state,
            put("need2", need2, u8), put("X", X, f64), put("V", V, f64), put("W", W, f64), put("E", E, f32),
            put("sc_in", sc_in, f64), put("sc_out", sc_out, f64), put("sS", sS, f64), put("dres", dres, i64),
            put("it", it, i32), put("dtrig", dtrig, f64), put("rinv", rinv, f64), put("Z", Z, f64),
            lb_dev if lb_dev is not None else put("lb", lb, f64), ub_dev if ub_dev is not None else put("ub", ub, f64),
            put("D_in", D_in, i16), put("S_in", S_in, i16), put("D_out", D_out, i16), put("S_out", S_out, i16),
            put("tile_stat", tile_stat, i64), None]
    rc = L.nnmpc_lp_step_test(*args)
    msg = L.nnmpc_last_error().decode(errors="replace")
    out = {}
    for k, t in dev.items():
        a = t.cpu().numpy()
        out[k] = a.view(np.uint16) if t.dtype is i16 else (a.view(np.uint64) if t.dtype is i64 else a)
    return rc, msg, out


def _call(torch, op, n, nu, B, **kw):
    rc, msg, out = _step(torch, op, n, nu, B, **kw)
    assert rc == 0, msg
    return out


# ------------------------------------------------------------------------------------ float64 restatements
def f16(a):
    """float64 -> fp16 bit patterns, correctly rounded (NumPy converts float64 -> float16 in one rounding)."""
    return np.asarray(a, dtype=np.float64).astype(np.float16).view(np.uint16)


def h2d(bits):
    return np.asarray(bits, dtype=np.uint16).view(np.float16).astype(np.float64)


def split_ref(T, top_max):
    _, e = np.frexp(top_max if top_max > 0 else 1.0)
    s = 2.0 ** (10 - int(e))
    sT = T * s
    T1 = f16(sT)
    return T1, f16(sT - h2d(T1)), s


def pow2_scale(est):
    """lp.cuh pow2_scale: the largest power of two s with s est in [8, 16], clamped to 2^+-60."""
    est = np.asarray(est, dtype=np.float64)
    out = np.empty_like(est)
    for i, x in np.ndenumerate(est):
        if not x > 0.0:
            out[i] = 2.0 ** 60
        elif not x <= 1.7e308:
            out[i] = 2.0 ** -60
        else:
            sh = 4 - int(np.frexp(x)[1])
            out[i] = 2.0 ** min(60, max(-60, sh))
    return out


def clip_sel(v, l, u):
    """compare/select clip of the epilogue: a NaN stays NaN"""
    r = np.where(v < l, l, v)
    return np.where(r > u, u, r)


def clipd(v, l, u):
    """fmin(fmax(v, l), u) of the FP64 kernels: a NaN becomes l"""
    return np.fmin(np.fmax(v, l), u)


def bits(a):
    """the bit patterns of an array (NaN payloads included), for 'unchanged' checks"""
    a = np.asarray(a)
    return a.view({8: np.uint64, 4: np.uint32, 2: np.uint16, 1: np.uint8}[a.dtype.itemsize])


def same(a, b):
    """bitwise equal, except that any NaN matches any NaN (payloads differ between the GPU and NumPy)"""
    a, b = np.asarray(a), np.asarray(b)
    u = np.uint64 if a.dtype == np.float64 else np.uint32
    return bool(np.all((a.view(u) == b.view(u)) | (np.isnan(a) & np.isnan(b))))


def ulp16(t):
    a = np.abs(t)
    e = np.floor(np.log2(np.maximum(a, 2.0 ** -24)))
    return 2.0 ** np.maximum(e - 10, -24)


def nanmax_rows(a):
    """row maximum that keeps a NaN"""
    return np.where(np.isnan(a).any(axis=1), np.nan, np.max(np.where(np.isnan(a), 0.0, a), axis=1))


def bounds_cols(lb, ub, n):
    k = np.arange(n) % lb.shape[1]
    return lb[:, k], ub[:, k]


# ------------------------------------------------------------------------------------ operators and state
def _regulator_top(p):
    from industrial_nnmpc_2021_b200.linearMPC import LinearMPCController
    reg = LinearMPCController.setup_regulator(p.A, p.B, p.Q, p.R, p.S, p.N, p.ulb, p.uub)
    Minv = np.linalg.inv(reg.P + np.diag(reg.rho_vec))
    return 0.5 * (Minv + Minv.T) * reg.rho_vec[None, :]


@pytest.fixture(scope="module")
def plant_tops(cstrs_problem):
    """Top = (P + D)^-1 D of the real CSTR (n = 540, nu = 6) and CDU (n = 4480, nu = 32) regulators, built as
    test_gpu_exact_applies._regulator builds them."""
    from industrial_nnmpc_2021_b200.plants import get_cdu_problem
    return {540: (_regulator_top(cstrs_problem), 6), 4480: (_regulator_top(get_cdu_problem(N=140, Nsim=1600)), 32)}


def _synthetic_top(rng, n):
    return rng.standard_normal((n, n)) * 2.0 ** rng.uniform(-8, 0, (1, n)) / np.sqrt(n)


def _state(rng, B, n, nu, inf_bounds=False):
    """Engine-like state: row scales over 2^-4 .. 2^2, v outside its box in about a third of the entries, power-of-two
    operand scales with a few rows whose sc_out saturates the increment, pending sums, priors of dres below and above."""
    rs = 2.0 ** rng.uniform(-4, 2, (B, 1))
    lb = -rng.uniform(0.1, 1.0, (B, nu)) * rs
    ub = rng.uniform(0.1, 1.0, (B, nu)) * rs
    if inf_bounds:
        lb[::3] = -np.inf
        ub[1::3] = np.inf
    sc_out = 2.0 ** rng.integers(2, 12, B).astype(np.float64)
    sc_out[::17] = 2.0 ** 24
    return dict(
        X=rng.standard_normal((B, n)) * rs, V=rng.standard_normal((B, n)) * rs * 1.3,
        E=(rng.standard_normal((B, n)) * 1e-4 * rs).astype(np.float32), lb=lb, ub=ub,
        sc_in=2.0 ** rng.integers(0, 10, B).astype(np.float64), sc_out=sc_out,
        sS=2.0 ** rng.integers(-3, 8, B).astype(np.float64),
        D_in=f16(rng.standard_normal((B, n)) * 8.0), S_in=f16(rng.standard_normal((B, n)) * 4.0),
        dres=rng.choice([0.0, 1e-300, 1e300], B).view(np.uint64))


# ------------------------------------------------------------------------------------ the pass and its reference
def _pass(torch, T, st, B, n, nu, s_mode, kernel, list_r, len_r, pos_w, state, need2=None, alpha=1.6, **kw):
    top_max = float(np.abs(T).max())
    return _call(torch, "iterate", n, nu, B, kernel=kernel, s_mode=s_mode, alpha=alpha, Top=T, top_max=top_max,
                 list_r=list_r, len_r=len_r, pos_w=pos_w, state=state, need2=need2, X=st["X"], V=st["V"], E=st["E"],
                 sc_in=st["sc_in"], sc_out=st["sc_out"], sS=st["sS"], dres=st["dres"], lb=st["lb"], ub=st["ub"],
                 D_in=st["D_in"], S_in=st["S_in"] if s_mode == 1 else None,
                 D_out=np.full((B, n), SENT16, np.uint16), S_out=np.full((B, n), SENT16, np.uint16) if s_mode else None,
                 tile_stat=np.zeros(2, np.uint64), **kw)


def _terms(s_mode, kernel, need2, pos):
    """operator terms of the tile that holds operand position pos"""
    if s_mode:
        return np.ones(len(pos), int)
    if need2 is None:
        return np.full(len(pos), 2)
    if kernel == 0:
        return np.where(need2[pos >> 7] != 0, 2, 1)
    return np.where((need2[(pos >> 8) * 2] | need2[(pos >> 8) * 2 + 1]) != 0, 2, 1)


def _tile_counts(s_mode, kernel, need2, M, n):
    """expected tile_stat = [one-term, two-term] tiles in 128 x 128 units"""
    tm, tn, unit = (128, 128, 1) if kernel == 0 else ((256, 128, 2) if kernel == 1 else (256, 256, 4))
    ntm, ntn = -(-M // tm), -(-n // tn)
    if s_mode:
        return [ntm * ntn * unit, 0]
    two = sum(1 for b in range(ntm) for _ in range(ntn) if _terms(0, kernel, need2, np.array([b * tm]))[0] == 2)
    return [(ntm * ntn - two) * unit, two * unit]


def _check_pass(T, st, out, B, n, nu, s_mode, kernel, list_r, len_r, pos_w, state, need2=None, alpha=1.6,
                tile_counts=True):
    """Everything the pass wrote or must not have written; returns the participating rows."""
    T1, T2, sT = split_ref(T, float(np.abs(T).max()))
    M = min(len_r, B)
    pos = np.arange(M)
    lr = np.arange(B) if list_r is None else np.asarray(list_r)
    pw_all = np.arange(B) if pos_w is None else np.asarray(pos_w)
    take = state[lr[pos]] == ITER
    pos = pos[take]
    r = lr[pos]
    pw = pw_all[r]
    lb, ub = bounds_cols(st["lb"][r], st["ub"][r], n)
    A = h2d(st["D_in"][pos])
    t1, t2 = h2d(T1), h2d(T2)
    terms = _terms(s_mode, kernel, need2, pos)[:, None]
    ref = A @ t1.T + np.where(terms == 2, A @ t2.T, 0.0)
    absref = np.abs(A) @ np.abs(t1).T + np.where(terms == 2, np.abs(A) @ np.abs(t2).T, 0.0)
    inv_in = (1.0 / sT) / st["sc_in"][r][:, None]
    bound = terms * -(-n // 16) * 2.0 ** -22 * absref * inv_in
    x0, x1 = st["X"][r], out["X"][r]
    err = np.abs((x1 - x0) - ref * inv_in)
    assert np.all(err <= bound + 2 * EPS * (np.abs(x0) + np.abs(x1))), float(np.max(err / np.maximum(bound, 1e-300)))
    # downstream of the GPU's own x
    v0, v1, e0 = st["V"][r], out["V"][r], st["E"][r].astype(np.float64)
    z0 = clip_sel(v0, lb, ub)
    d = x1 - z0
    vref = v0 + alpha * d
    assert np.all(np.abs(v1 - vref) <= 2 * EPS * (np.abs(vref) + np.abs(alpha * d))), "V"
    wl = (2.0 * z0 - v0) - e0
    z1 = clip_sel(v1, lb, ub)
    dw = (2.0 * z1 - v1) - wl
    so = st["sc_out"][r][:, None]
    q = h2d(out["D_out"][pw])
    t = np.clip(dw * so, -60000.0, 60000.0)
    assert np.all(np.abs(q - t) <= ulp16(t)), "q"
    e1 = out["E"][r]
    assert np.array_equal(e1, (dw - q * (1.0 / so)).astype(np.float32)), "E"
    w0, w1, e1d = 2.0 * z0 - v0, 2.0 * z1 - v1, e1.astype(np.float64)
    cons = ((w1 - e1d) - (w0 - e0)) - q / so
    assert np.all(np.abs(cons) <= 2.0 ** -24 * np.abs(e1d) + 4 * EPS * (np.abs(w0) + np.abs(w1) + np.abs(e0) + np.abs(e1d))), "conservation"
    m = np.abs(d).astype(np.float32).max(axis=1).astype(np.float64)
    m = np.where(m <= 3.0e38, m, np.inf)
    prior = st["dres"][r].view(np.float64)
    assert np.array_equal(out["dres"][r], np.maximum(prior, m).view(np.uint64)), "dres"
    # deferred second term
    if s_mode == 2:
        want = f16(h2d(out["D_out"][pw]) * 0.125 + 0.0)      # fmaf(q, 0.125, +0): exact, and -0 + 0 = +0
        assert np.array_equal(out["S_out"][pw], want), "S (new sum)"
        assert np.array_equal(out["sS"][r], 0.125 * st["sc_out"][r]), "sS"
    elif s_mode == 1:
        g = (st["sS"][r] * (1.0 / st["sc_out"][r])).astype(np.float32).astype(np.float64)[:, None]
        so_in = h2d(st["S_in"][pos])
        prod = q * g
        s64 = prod + so_in
        assert np.all((s64 - prod == so_in) & (s64 - so_in == prod)), "test data: the fp32 FMA is not exact in float64"
        want = f16(np.clip(s64.astype(np.float32), -65504.0, 65504.0).astype(np.float64))
        assert np.array_equal(out["S_out"][pw], want), "S (added)"
        assert np.array_equal(out["sS"], st["sS"]), "sS"
    # nothing else written
    rest = np.setdiff1d(np.arange(B), r)
    for k in ("X", "V"):
        assert np.array_equal(out[k][rest].view(np.uint64), st[k][rest].view(np.uint64)), k
    assert np.array_equal(out["E"][rest].view(np.uint32), st["E"][rest].view(np.uint32)), "E"
    assert np.array_equal(out["dres"][rest], st["dres"][rest]), "dres"
    if s_mode:
        assert np.array_equal(out["sS"][rest], st["sS"][rest]), "sS"
    unw = np.setdiff1d(np.arange(B), pw)
    assert np.all(out["D_out"][unw] == SENT16), "D_out rows written that no row owns"
    if s_mode:
        assert np.all(out["S_out"][unw] == SENT16), "S_out rows written that no row owns"
    if tile_counts:
        assert list(out["tile_stat"]) == _tile_counts(s_mode, kernel, need2, M, n), (list(out["tile_stat"]), M)
    return r


SHAPES = [(2, 1, 129), (62, 2, 130), (64, 2, 127), (66, 33, 257), (126, 3, 255), (128, 4, 256), (130, 3, 128),
          (254, 2, 1), (256, 4, 300), (258, 6, 129), (540, 6, 257), (4480, 32, 257), (1000, 4, 2688)]


@pytest.mark.parametrize("mode", PASSES)
def test_pass_shapes(torch_cuda, plant_tops, mode):
    """Every tile variant at the 64-, 128- and 256-column edges, B at the 128- and 256-row tile edges, the real CSTR and
    CDU operators (the CDU's 35 column tiles end in a partial L2 column group in every variant), more tiles than SMs,
    nu = 1, an odd nu whose column pairs cross a stage, and nu = 33 > n / 2; permuted list, re-compacting pos_w, rows
    in the list that do not iterate."""
    torch = torch_cuda
    s_mode, kernel = mode
    for i, (n, nu, B) in enumerate(SHAPES):
        rng = np.random.default_rng(100 + i)
        T = plant_tops[n][0] if n in plant_tops else _synthetic_top(rng, n)
        st = _state(rng, B, n, nu)
        list_r = rng.permutation(B).astype(np.int32)
        pos_w = rng.permutation(B).astype(np.int32)
        state = np.where(rng.random(B) < 0.1, CAND, ITER).astype(np.int32)
        out = _pass(torch, T, st, B, n, nu, s_mode, kernel, list_r, B, pos_w, state)
        _check_pass(T, st, out, B, n, nu, s_mode, kernel, list_r, B, pos_w, state)


def test_pass_8960(torch_cuda):
    """One pass at n = 8960 (70 column tiles, 2 x 160 MB of fp16 operator) in the default variant."""
    torch = torch_cuda
    rng = np.random.default_rng(8960)
    n, nu, B = 8960, 32, 130
    T = _synthetic_top(rng, n)
    st = _state(rng, B, n, nu)
    list_r = rng.permutation(B).astype(np.int32)
    state = np.full(B, ITER, np.int32)
    out = _pass(torch, T, st, B, n, nu, 0, 0, list_r, B, None, state)
    _check_pass(T, st, out, B, n, nu, 0, 0, list_r, B, None, state)


@pytest.mark.parametrize("mode", PASSES)
def test_pass_bounds_paths(torch_cuda, mode):
    """The scalar bounds path (lb / ub one double off a 16-byte boundary with even nu) and infinite bounds as data."""
    torch = torch_cuda
    s_mode, kernel = mode
    rng = np.random.default_rng(7)
    n, nu, B = 130, 2, 200
    T = _synthetic_top(rng, n)
    st = _state(rng, B, n, nu, inf_bounds=True)
    state = np.full(B, ITER, np.int32)
    list_r = rng.permutation(B).astype(np.int32)
    lbuf = torch.tensor(np.concatenate([[0.0], st["lb"].ravel()]), device="cuda")
    ubuf = torch.tensor(np.concatenate([[0.0], st["ub"].ravel()]), device="cuda")
    from industrial_nnmpc_2021_b200 import _lib
    out = _pass(torch, T, st, B, n, nu, s_mode, kernel, list_r, B, None, state,
                lb_dev=_lib.dptr(lbuf[1:]), ub_dev=_lib.dptr(ubuf[1:]))
    _check_pass(T, st, out, B, n, nu, s_mode, kernel, list_r, B, None, state)
    out2 = _pass(torch, T, st, B, n, nu, s_mode, kernel, list_r, B, None, state)     # the vector path: same bits
    for k in ("X", "V", "E", "dres", "D_out"):
        assert np.array_equal(out[k], out2[k]), k


@pytest.mark.parametrize("mode", PASSES)
def test_pass_lists_and_layout(torch_cuda, mode):
    """len_r on both sides of every 128- and 256-row edge and 0, a permuted list with rows that do not iterate, and a
    pos_w that re-compacts: the rows that take part are exact, every other row and operand position keeps its bits."""
    torch = torch_cuda
    s_mode, kernel = mode
    rng = np.random.default_rng(3)
    n, nu, B = 130, 3, 300
    T = _synthetic_top(rng, n)
    st = _state(rng, B, n, nu)
    list_r = rng.permutation(B).astype(np.int32)
    state = np.where(rng.random(B) < 0.15, CAND, ITER).astype(np.int32)
    state[list_r[126:131]] = CAND
    pos_w = rng.permutation(B).astype(np.int32)
    for len_r in (0, 1, 127, 128, 129, 255, 256, 257, 300):
        out = _pass(torch, T, st, B, n, nu, s_mode, kernel, list_r, len_r, pos_w, state)
        _check_pass(T, st, out, B, n, nu, s_mode, kernel, list_r, len_r, pos_w, state)


def _one_sign_top(rng, n):
    """T = (h + 0.375 ulp(h)) 2^-10 with fp16 h in [512, 1024): s_T = 2^10, T1 = h and T2 = 0.375 ulp(h) > 0 exactly,
    so with non-negative increments the second term adds at least 1.8e-4 of the first - far above the bound."""
    h = h2d(f16(rng.uniform(512.0, 1023.0, (n, n))))
    return (h + 0.375 * 0.5) * 2.0 ** -10


@pytest.mark.parametrize("mode", PASSES)
def test_one_term_or_two(torch_cuda, mode):
    """Each tile runs with exactly the operator terms its need2 flags ask for (a 256-row or pair tile with two when
    either 128-row half is flagged; one-term passes always with one): within the bound of the right reference and
    outside it of the other, and tile_stat counts exactly."""
    torch = torch_cuda
    s_mode, kernel = mode
    rng = np.random.default_rng(12)
    n, nu, B = 256, 4, 600
    T = _one_sign_top(rng, n)
    T1, T2, sT = split_ref(T, float(np.abs(T).max()))
    assert sT == 2.0 ** 10 and np.all(h2d(T2) > 0)
    st = _state(rng, B, n, nu)
    st["D_in"] = f16(np.abs(rng.standard_normal((B, n))) * 8.0)
    st["X"][:] = 0.0
    state = np.full(B, ITER, np.int32)
    A = h2d(st["D_in"])
    ref1, ref2 = A @ h2d(T1).T, A @ (h2d(T1) + h2d(T2)).T
    ntile = (B + 255) // 256 * 2 + 2
    patterns = {"all0": np.zeros(ntile, np.uint8), "all1": np.ones(ntile, np.uint8),
                "alternating": (np.arange(ntile) % 2 == 0).astype(np.uint8),
                "second": (np.arange(ntile) == 1).astype(np.uint8), "last": (np.arange(ntile) == (B - 1) // 128).astype(np.uint8)}
    for name, need2 in patterns.items():
        out = _pass(torch, T, st, B, n, nu, s_mode, kernel, None, B, None, state, need2=need2)
        _check_pass(T, st, out, B, n, nu, s_mode, kernel, None, B, None, state, need2=need2)
        acc = out["X"] * sT * st["sc_in"][:, None]
        terms = _terms(s_mode, kernel, need2, np.arange(B))[:, None]
        steps = terms * (n // 16)
        bnd = steps * 2.0 ** -22 * np.where(terms == 2, ref2, ref1)
        right, wrong = np.where(terms == 2, ref2, ref1), np.where(terms == 2, ref1, ref2)
        assert np.all(np.abs(acc - right) <= bnd), name
        assert np.all(np.abs(acc - wrong) > bnd), (name, "the other number of operator terms fits too")


# ------------------------------------------------------------------------------------ deferred second term
@pytest.mark.parametrize("kernel", [0, 1], ids=["128", "256"])
def test_correct_adds_the_second_term(torch_cuda, kernel):
    """x += T2 S / (s_T sS) over the rows a pass would take, within the bound and never with T1; every other row keeps
    its bits; tile_stat[0] counts the one-term tiles."""
    torch = torch_cuda
    rng = np.random.default_rng(21)
    n, nu, B = 258, 3, 300
    T = _synthetic_top(rng, n)
    T1, T2, sT = split_ref(T, float(np.abs(T).max()))
    st = _state(rng, B, n, nu)
    list_r = rng.permutation(B).astype(np.int32)
    state = np.where(rng.random(B) < 0.2, CAND, ITER).astype(np.int32)
    for len_r in (0, 129, 257, 300):
        out = _call(torch, "correct", n, nu, B, kernel=kernel, Top=T, top_max=float(np.abs(T).max()), list_r=list_r,
                    len_r=len_r, state=state, X=st["X"], S_in=st["S_in"], sS=st["sS"], tile_stat=np.zeros(2, np.uint64))
        pos = np.arange(len_r)
        pos = pos[state[list_r[pos]] == ITER]
        r = list_r[pos]
        Sv = h2d(st["S_in"][pos])
        inv = (1.0 / sT) / st["sS"][r][:, None]
        ref, ref1 = Sv @ h2d(T2).T * inv, Sv @ h2d(T1).T * inv
        bound = -(-n // 16) * 2.0 ** -22 * (np.abs(Sv) @ np.abs(h2d(T2)).T) * inv
        dx = out["X"][r] - st["X"][r]
        slack = 2 * EPS * (np.abs(out["X"][r]) + np.abs(st["X"][r]))
        assert np.all(np.abs(dx - ref) <= bound + slack)
        assert np.all(np.abs(dx - ref1) > bound + slack)
        rest = np.setdiff1d(np.arange(B), r)
        assert np.array_equal(out["X"][rest].view(np.uint64), st["X"][rest].view(np.uint64))
        ntm = -(-len_r // (128 * (kernel + 1)))
        assert list(out["tile_stat"]) == [ntm * -(-n // 128) * (kernel + 1), 0]


# ------------------------------------------------------------------------------------ operator split
def test_operator_split_bitwise(torch_cuda):
    """s = 2^(10 - e) for frexp(top_max) = (m, e), T1 = fp16(s T), T2 = fp16(s T - T1) bitwise, with top_max a power of
    two and just below one, T2 in the fp16 subnormal range and rounding to 0, and zero padding beyond n."""
    torch = torch_cuda
    rng = np.random.default_rng(5)
    n = 130
    ldh = 192
    base = rng.uniform(-1.0, 1.0, (n, n)) * 0.5
    for top in (1.0, np.nextafter(1.0, 0.0), 0.75, 2.0 ** -20):
        T = base * top
        T[0, 0] = top
        _, e = np.frexp(top)
        s = 2.0 ** (10 - int(e))
        h = h2d(f16(rng.uniform(16.0, 512.0, 40)))
        T[1, :40] = (h + 2.0 ** -20) / s             # T2 = 2^-20: fp16 subnormal
        T[2, :40] = (h + 2.0 ** -26) / s             # T2 = 2^-26 rounds to 0 (below half the smallest subnormal)
        T[3, :40] = (h + 3 * 2.0 ** -25) / s         # 1.5 x the smallest subnormal: rounds to even
        out = _call(torch, "split", n, 1, 1, Top=T, top_max=top, sc_out=np.zeros(1),
                    D_out=np.full((n, ldh), SENT16, np.uint16), S_out=np.full((n, ldh), SENT16, np.uint16))
        T1, T2, sref = split_ref(T, top)
        assert out["sc_out"][0] == sref == s, (out["sc_out"][0], s)
        assert np.array_equal(out["D_out"][:, :n], T1) and np.array_equal(out["S_out"][:, :n], T2)
        assert np.all(out["D_out"][:, n:] == 0) and np.all(out["S_out"][:, n:] == 0), "padding"
        t2 = h2d(T2)
        assert np.all(t2[1, :40] == 2.0 ** -20) and np.all(t2[2, :40] == 0.0) and np.all(t2[3, :40] == 2.0 ** -23)


# ------------------------------------------------------------------------------------ FP64 helper kernels
def _helper_state(rng, B, n, nu):
    st = _state(rng, B, n, nu)
    st["W"] = rng.standard_normal((B, n)) * 0.5
    st["state"] = np.where(rng.random(B) < 0.4, EMIT, ITER).astype(np.int32)
    st["it"] = rng.integers(0, 50, B).astype(np.int32)
    st["dtrig"] = np.abs(rng.standard_normal(B)) * 1e-6
    return st


def test_anchor_prep_and_reanchor(torch_cuda):
    """anchor_prep: W = 2 clip(V) - V and E = 0 bitwise for listed rows; reanchor: listed rows in emit_state get X = Z
    bitwise and W = Z + W rinv to one rounding; every other row keeps its bits."""
    torch = torch_cuda
    rng = np.random.default_rng(31)
    n, nu, B = 258, 3, 300
    st = _helper_state(rng, B, n, nu)
    rows = rng.permutation(B).astype(np.int32)
    for count in (0, 1, 200, 300):
        out = _call(torch, "anchor_prep", n, nu, B, rows=rows, count=count, V=st["V"], W=st["W"], E=st["E"],
                    lb=st["lb"], ub=st["ub"])
        on, off = rows[:count], rows[count:]
        lb, ub = bounds_cols(st["lb"][on], st["ub"][on], n)
        assert np.array_equal(out["W"][on], 2.0 * clipd(st["V"][on], lb, ub) - st["V"][on])
        assert np.all(out["E"][on].view(np.uint32) == 0)
        assert np.array_equal(out["W"][off], st["W"][off]) and np.array_equal(out["E"][off], st["E"][off])
        Z = rng.standard_normal((B, n))
        rinv = rng.uniform(0.1, 10.0, n)
        out = _call(torch, "reanchor", n, nu, B, rows=rows, count=count, state=st["state"], Z=Z, W=st["W"],
                    rinv=rinv, X=st["X"])
        on = rows[:count][st["state"][rows[:count]] == EMIT]
        off = np.setdiff1d(np.arange(B), on)
        assert np.array_equal(out["X"][on], Z[on])
        # the kernel may round once (FMA: u |W|), the reference rounds the product and the sum (u |W rinv| + u |ref|)
        ref = Z[on] + st["W"][on] * rinv
        assert np.all(np.abs(out["W"][on] - ref) <= 2 * EPS * (np.abs(ref) + np.abs(st["W"][on] * rinv)))
        assert np.array_equal(out["X"][off], st["X"][off]) and np.array_equal(out["W"][off], st["W"][off])


def _first_increment_check(st, out, rows_on, n, nu, dw, wmax, est, s_mode, pos_r, need2_in, iter_state=ITER):
    """what dr_first and emit share: scales, increment, residual, pending sum, state, need2"""
    sq = pow2_scale(wmax)
    assert np.array_equal(out["sc_in"][rows_on], sq), "sc_in"
    assert np.array_equal(out["sc_out"][rows_on], pow2_scale(est)), "sc_out"
    t = np.fmin(np.fmax(dw * sq[:, None], -60000.0), 60000.0)
    q = f16(t)
    pos = pos_r[rows_on]
    w = pos >= 0
    assert np.array_equal(out["D_out"][pos[w]], q[w]), "D"
    e = (dw - h2d(q) * (1.0 / sq)[:, None]).astype(np.float32)
    assert same(out["E"][rows_on], e), "E"
    assert np.all(out["state"][rows_on] == iter_state)
    if s_mode:
        sref = f16((h2d(q).astype(np.float32) * np.float32(0.125)).astype(np.float64))
        assert np.array_equal(out["S_out"][pos[w]], sref[w]), "S start"
        assert np.array_equal(out["sS"][rows_on], 0.125 * sq), "sS"
    flags = need2_in.copy()
    flags[pos[w] >> 7] = 1
    assert np.array_equal(out["need2"], flags), "need2"
    written = set(pos[w].tolist())
    unw = np.array([p for p in range(len(st["X"])) if p not in written], dtype=int)
    assert np.all(out["D_out"][unw] == SENT16), "operand rows written that no row owns"
    if s_mode:
        assert np.all(out["S_out"][unw] == SENT16)
    else:
        assert "S_out" not in out or np.all(out["S_out"] == SENT16)


def _edge_rows(st, rows, n):
    """rows whose max |dw| is 0, subnormal, huge, NaN and +Inf (W is the operand the step subtracts)"""
    r0, r1, r2, r3, r4 = rows[:5]
    lb, ub = bounds_cols(st["lb"], st["ub"], n)
    for r in (r0, r1, r2, r3, r4):
        st["V"][r] = 0.5 * (lb[r] + ub[r])             # inside the box: clip(v) = v
        st["X"][r] = st["V"][r]                         # d = 0
        st["W"][r] = st["V"][r]                         # dw = (2 v - v) - v = 0
    st["W"][r1, 7] -= 3e-310
    st["W"][r2, n - 1] -= 1e300
    st["W"][r3, 5] = np.nan
    st["W"][r4, 0] = -np.inf
    return [r0, r1, r2, r3, r4]


@pytest.mark.parametrize("s_mode", [0, 2], ids=["plain", "pending-sum"])
def test_dr_first(torch_cuda, s_mode):
    """One FP64 step from the exact x, first increment at pos_r (none for a negative position), exact power-of-two
    scales including estimates of 0, subnormal, huge, NaN and +Inf (clamped to 2^+-60), it + 1, need2 at pos >> 7,
    and the pending-sum start with s_mode != 0."""
    torch = torch_cuda
    rng = np.random.default_rng(41)
    n, nu, B, alpha = 258, 3, 300, 1.6
    st = _helper_state(rng, B, n, nu)
    rows = rng.permutation(B).astype(np.int32)
    edge = _edge_rows(st, rows, n)
    pos_r = rng.permutation(B).astype(np.int32)
    pos_r[rows[5:9]] = -1
    need2 = np.zeros((B + 127) // 128 + 2, np.uint8)
    for count in (0, 1, 129, 300):
        out = _call(torch, "dr_first", n, nu, B, s_mode=s_mode, alpha=alpha, rows=rows, count=count, pos_r=pos_r,
                    state=st["state"], iter_state=ITER, need2=need2, X=st["X"], V=st["V"], W=st["W"], E=st["E"],
                    sc_in=st["sc_in"], sc_out=st["sc_out"], sS=st["sS"], it=st["it"], lb=st["lb"], ub=st["ub"],
                    D_out=np.full((B, n), SENT16, np.uint16), S_out=np.full((B, n), SENT16, np.uint16))
        on = rows[:count]
        lb, ub = bounds_cols(st["lb"][on], st["ub"][on], n)
        x, v = st["X"][on], st["V"][on]
        z0 = clipd(v, lb, ub)
        d = x - z0
        vref = v + alpha * d
        v1 = out["V"][on]
        ok = np.isfinite(vref)
        assert np.all(np.abs(v1 - vref)[ok] <= 2 * EPS * (np.abs(vref) + np.abs(alpha * d))[ok]), "V"
        dw = (2.0 * clipd(v1, lb, ub) - v1) - st["W"][on]
        assert same(out["W"][on], dw), "W"
        wmax, dmax = nanmax_rows(np.abs(dw)), nanmax_rows(np.abs(d))
        _first_increment_check(st, out, on, n, nu, dw, wmax, 3.0 * alpha * dmax, s_mode, pos_r, need2)
        assert np.array_equal(out["it"][on], st["it"][on] + 1)
        if count == B:
            sc = out["sc_in"][edge]
            assert list(sc) == [2.0 ** 60, 2.0 ** 60, 2.0 ** -60, 2.0 ** 60, 2.0 ** -60], sc
        off = rows[count:]
        for k in ("X", "V", "W", "E", "sc_in", "sc_out", "it", "state"):
            assert np.array_equal(bits(out[k][off]), bits(st[k][off])), k
        assert np.array_equal(out["sS"][off] if s_mode else out["sS"], st["sS"][off] if s_mode else st["sS"])


@pytest.mark.parametrize("s_mode", [0, 2], ids=["plain", "pending-sum"])
def test_emit(torch_cuda, s_mode):
    """Listed rows in emit_state: dw = (2 clip(v) - v) - w_lp into W, first increment at pos_r (none for a negative
    position), sc_out = pow2_scale(3 alpha (dtrig + max |dw|)) exactly; rows in other states and unlisted rows keep
    their bits."""
    torch = torch_cuda
    rng = np.random.default_rng(43)
    n, nu, B, alpha = 130, 2, 300, 1.6
    st = _helper_state(rng, B, n, nu)
    rows = rng.permutation(B).astype(np.int32)
    edge = _edge_rows(st, rows, n)
    st["state"][edge] = EMIT
    st["dtrig"][edge] = 0.0
    pos_r = rng.permutation(B).astype(np.int32)
    pos_r[rows[5:12]] = -1
    need2 = np.zeros((B + 127) // 128 + 2, np.uint8)
    for count in (0, 1, 129, 300):
        out = _call(torch, "emit", n, nu, B, s_mode=s_mode, alpha=alpha, rows=rows, count=count, pos_r=pos_r,
                    state=st["state"], emit_state=EMIT, iter_state=ITER, need2=need2, V=st["V"], W=st["W"], E=st["E"],
                    sc_in=st["sc_in"], sc_out=st["sc_out"], sS=st["sS"], dtrig=st["dtrig"], lb=st["lb"], ub=st["ub"],
                    D_out=np.full((B, n), SENT16, np.uint16), S_out=np.full((B, n), SENT16, np.uint16))
        on = rows[:count][st["state"][rows[:count]] == EMIT]
        lb, ub = bounds_cols(st["lb"][on], st["ub"][on], n)
        v = st["V"][on]
        dw = (2.0 * clipd(v, lb, ub) - v) - st["W"][on]
        assert same(out["W"][on], dw), "W"
        wmax = nanmax_rows(np.abs(dw))
        _first_increment_check(st, out, on, n, nu, dw, wmax, 3.0 * alpha * (st["dtrig"][on] + wmax), s_mode, pos_r,
                               need2)
        if count == B:
            sc = out["sc_in"][edge]
            assert list(sc) == [2.0 ** 60, 2.0 ** 60, 2.0 ** -60, 2.0 ** 60, 2.0 ** -60], sc
        off = np.setdiff1d(np.arange(B), on)
        for k in ("V", "W", "E", "sc_in", "sc_out", "state"):
            assert np.array_equal(bits(out[k][off]), bits(st[k][off])), k


# ------------------------------------------------------------------------------------ non-finite rows
@pytest.mark.parametrize("mode", PASSES)
def test_nonfinite_rows_do_not_look_converged(torch_cuda, mode):
    """A NaN, +Inf or -Inf in one column of V, X or E of one row (column 0, an odd column, the last column, the first
    and the last column tile; rows on both sides of a 128-row tile edge) gives that row dres = +Inf exactly; every
    other row is bitwise what a clean run gives.  (The epilogue's maxima used to drop a NaN, and a non-finite V or E
    left d finite.)"""
    torch = torch_cuda
    s_mode, kernel = mode
    rng = np.random.default_rng(51)
    n, nu, B = 386, 3, 300
    T = _synthetic_top(rng, n)
    st = _state(rng, B, n, nu)
    state = np.full(B, ITER, np.int32)
    list_r = rng.permutation(B).astype(np.int32)
    clean = _pass(torch, T, st, B, n, nu, s_mode, kernel, list_r, B, None, state)
    # columns: 0, odd, inside the first / last 128- and 256-column tiles, the last; operand positions on both sides of
    # the 128-, 256- and last row-tile edges
    cols = [0, 1, 77, 127, 129, 255, 258, n - 2, n - 1]
    positions = [0, 1, 126, 127, 128, 129, 254, 255, 256, 257, 298, 299, 30, 60, 90, 140, 170, 200, 230, 270, 290,
                 10, 20, 40, 50, 70, 80]
    pois = {k: st[k].copy() for k in ("X", "V", "E")}
    bad = []
    i = 0
    for field in ("V", "X", "E"):
        for val in (np.nan, np.inf, -np.inf):
            for _ in range(3):
                r = list_r[positions[i]]
                pois[field][r, cols[i % len(cols)]] = val
                bad.append(r)
                i += 1
    sp = dict(st, **pois)
    out = _pass(torch, T, sp, B, n, nu, s_mode, kernel, list_r, B, None, state)
    got = out["dres"][bad]
    assert np.all(got == INF_BITS), [(int(r), hex(int(g))) for r, g in zip(bad, got) if g != INF_BITS]
    ok = np.setdiff1d(np.arange(B), bad)
    for k in ("X", "V", "dres", "sS"):
        assert np.array_equal(out[k][ok].view(np.uint64), clean[k][ok].view(np.uint64)), k
    assert np.array_equal(out["E"][ok].view(np.uint32), clean["E"][ok].view(np.uint32))
    pw_ok = ok                      # pos_w = identity
    assert np.array_equal(out["D_out"][pw_ok], clean["D_out"][pw_ok])
    if s_mode:
        assert np.array_equal(out["S_out"][pw_ok], clean["S_out"][pw_ok])


# ------------------------------------------------------------------------------------ refusals
def test_refuses_bad_shapes_before_any_launch(torch_cuda):
    torch = torch_cuda
    z = np.zeros((4, 4))
    for n, nu, s_mode, kernel in ((3, 1, 0, 0), (0, 1, 0, 0), (-2, 1, 0, 0), (4, 0, 0, 0), (4, 1, 1, 2), (4, 1, 2, 2),
                                  (4, 1, 3, 0), (4, 1, 0, 3)):
        rc, msg, _ = _step(torch, "iterate", n, nu, 4, kernel=kernel, s_mode=s_mode, Top=z, top_max=1.0, len_r=4,
                           state=np.ones(4, np.int32), X=z, V=z, E=z.astype(np.float32), sc_in=np.ones(4),
                           sc_out=np.ones(4), sS=np.ones(4), dres=np.zeros(4, np.uint64), lb=z, ub=z,
                           D_in=np.zeros((4, 4), np.uint16), S_in=np.zeros((4, 4), np.uint16),
                           D_out=np.zeros((4, 4), np.uint16), S_out=np.zeros((4, 4), np.uint16))
        assert rc == NNMPC_ERR_BADARG and msg, (n, nu, s_mode, kernel, rc, msg)
