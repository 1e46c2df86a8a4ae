"""The structured regulator network u = us + f(x, [uprev], xs, us) - f(xs, [us], xs, us) in all three arithmetic
modes ("tc": INT8 tcgen05 digit planes, "f64": FP64 DMMA, "fp16": split-fp16 tcgen05) against the float64 NumPy
restatement of oracle/nn.py, at the edges where the kernels go wrong: no hidden layer and 15 of them, widths at the
64-column and 128-row tile edges, the K = 32768 contraction limit, the batch chunking of each mode, extreme
magnitudes, zero rows, dead units, non-finite inputs, and one handle reused across batch sizes and modes."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import nn as onn

MODES = ("tc", "f64", "fp16")
MODE_CODE = {"f64": 0, "tc": 1, "fp16": 2}
U = 2.0 ** -53


@pytest.fixture(scope="module")
def torch_cuda(built_lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _layer(ws, with_uprev, mode):
    from industrial_nnmpc_2021_b200.LinearMPCLayers import RegulatorLayerWithUprev, RegulatorLayerWithoutUprev
    kernels = ws[0::2]
    layer = (RegulatorLayerWithUprev if with_uprev else RegulatorLayerWithoutUprev)(
        layer_dims=[k.shape[1] for k in kernels], precision=mode)
    layer.set_weights(ws)
    return layer


def _set_mode(layer, mode):
    from industrial_nnmpc_2021_b200 import _lib
    _lib.check(_lib.lib().nnmpc_mlp_set_precision(layer._handle, MODE_CODE[mode]), "nnmpc_mlp_set_precision")


def _weights(rng, dims, bias_scale=3.0):
    """Glorot kernels and large biases (+-bias_scale, beyond the O(1) pre-activations).  In every hidden layer of
    width >= 2 unit 0 is dead (zero kernel column, zero bias); in every layer of width >= 3 unit 1 takes incoming
    weights spanning 1e-8..1.  In the first hidden layer input 0 (x[:, 0]) feeds every live unit with a positive
    weight, so a sample with x[0] = +1e4 switches every unit of that layer on and x[0] = -1e4 every unit off."""
    ws = []
    nl = len(dims) - 1
    for i in range(nl):
        K, N = dims[i], dims[i + 1]
        lim = np.sqrt(6.0 / (K + N))
        W = rng.uniform(-lim, lim, (K, N))
        if N >= 3:
            W[:, 1] = rng.choice([-1.0, 1.0], K) * np.logspace(0, -8, K)
        b = bias_scale * rng.uniform(0.2, 1.0, N) * rng.choice([-1.0, 1.0], N)
        if i == 0 and nl > 1:
            W[0, :] = np.abs(W[0, :]) + lim
        if i < nl - 1 and N >= 2:
            W[:, 0] = 0.0
            b[0] = 0.0
        ws.append(W)
        if i < nl - 1:
            ws.append(b)
    return ws


def _inputs(rng, B, nx, nu, with_uprev):
    """Random samples with a per-sample magnitude over 3 decades, and by sample index mod 7: all-zero samples,
    samples that mix 1e6 and 1e-6 entries, and samples with x[0] = +1e4 / -1e4."""
    mag = np.exp(rng.uniform(-3, 3, (B, 1)))
    x, xs = rng.standard_normal((B, nx)) * mag, rng.standard_normal((B, nx)) * mag
    up, us = rng.uniform(-1, 1, (B, nu)) * mag, rng.uniform(-1, 1, (B, nu)) * mag
    k = np.arange(B) % 7
    for a in (x, xs, up, us):
        a[k == 0] = 0.0
        mix = np.where(np.arange(a.shape[1]) % 2 == 0, 1e6, 1e-6)
        a[k == 1] = rng.standard_normal((int(np.sum(k == 1)), a.shape[1])) * mix
    x[k == 2, 0], x[k == 3, 0] = 1e4, -1e4
    return [x, up, xs, us] if with_uprev else [x, xs, us]


def _operands(inputs, with_uprev, xscale):
    """The two network inputs of every sample, as the kernels and controller_evaluation.py:863-866 form them."""
    if with_uprev:
        x, up, xs, us = inputs
    else:
        (x, xs, us), up = inputs, None
    if xscale is not None:
        x, xs = x / xscale, xs / xscale
    a1 = np.concatenate([x, up, xs, us] if with_uprev else [x, xs, us], axis=1)
    a2 = np.concatenate([xs, us, xs, us] if with_uprev else [xs, xs, us], axis=1)
    return a1, a2, us, ([x, up, xs, us] if with_uprev else [x, xs, us])


def _reference(ws, inputs, with_uprev, xscale=None, ulb=None, uub=None):
    """oracle/nn.py in float64, with the deployment form's scaling and clip (controller_evaluation.py:863-892)."""
    scaled = _operands(inputs, with_uprev, xscale)[3]
    u = onn.layer_call(ws, scaled, with_uprev)
    if ulb is not None:
        u = np.where(u > uub, uub, u)
        u = np.where(u < ulb, ulb, u)
    return u


def _pow2_scale(m):
    """2^(ex + 1) for m = mant 2^ex, mant in [0.5, 1), and 2 for m = 0: the digit-plane scale the slicing kernels
    give a row (operator row) whose largest magnitude is m; non-decreasing in m."""
    return np.ldexp(1.0, np.frexp(m)[1] + 1)


def _gamma(k):
    return k * U / (1.0 - k * U)


def _pass_bound(ws, a, mode):
    """f(a) in float64 and a worst-case bound of |f_kernel(a) - f_reference(a)| per element.

    Layer by layer, with h, d the reference activation and the bound of the kernel's deviation from it (d = 0 for the
    input, which both form with the same IEEE divisions), |h|+d bounds what the kernel holds, S = (|h|+d) |W|, and
      - both float64 GEMMs (the reference's, and the DMMA chain of "f64") round within gamma_(K+1) S each;
      - "tc": a row of max m is cut into 4 base-128 digits of 2^f = 2^(ex+1) <= 4 m, |digit| <= 64, leaving a
        residual <= 2^f 2^-29 per entry; a weight column likewise with 2^e.  Levels 0..3 keep the digit pairs i+j <= 3,
        INT32 sums are exact and the fold is exact, so the error is the three dropped levels 4..6
        (K 2^12 2^(f+e) (3 128^-6 + 2 128^-7 + 128^-8)) plus the two residual products (2 K 2^(f+e) 2^-30), at most
        (5 + 2^-5) K 2^-30 2^(f+e) (< 1.3 K 2^-24 max|a| max|w|); 2^f, 2^e from the bound of the row maximum;
      - "fp16": a value t of a row scaled by s (s bound < 2^14, 1/s <= 2^-13 bound; weights: 1/s_w <= 2^-9 max|W|)
        is split into fp16 hi + lo with |t - hi - lo| <= 2^-22 |t| + 2^-25 and |lo| <= 2^-11 |t| + 2^-24; the products
        hi hi + hi lo + lo hi then miss at most 2^-20 |t_a t_w| + 2^-24 (|t_a| + |t_w|) + 2^-47 per term; the fp32
        accumulator takes 3 kp / 16 MMA steps of K = 16 (kp = K rounded up to 64; hi and lo of the activation, the
        weights read twice), each adding at most 2^-22 of the magnitudes summed so far (fp32 rounding with a
        truncating alignment).  The row bound of layer 0 is the exact row maximum, of layer l+1 the fp32 maximum of
        the row layer l read (<= (1 + 2^-21) max) times max_j sum_i |W_ij| (1 + 2^-22) plus max |b|;
      - the bias add rounds in the kernel and the reference (2u of |y| + err);
      - "tc" stores hidden activations as fp32: 2^-24 of |h| + err, plus 2^-149 for the subnormal range.
    The deviation propagates through |W| (ReLU is 1-Lipschitz)."""
    nl = (len(ws) + 1) // 2
    h, d = a, np.zeros_like(a)
    rowb = np.abs(a).max(axis=1)                 # fp16: the bound the row scale of the operand is taken from
    for l in range(nl):
        W = ws[2 * l]
        b = ws[2 * l + 1] if l < nl - 1 else None
        K = W.shape[0]
        Wa = np.abs(W)
        ha = np.abs(h) + d
        S = ha @ Wa
        y = h @ W + (0.0 if b is None else b)
        e = d @ Wa + 2 * _gamma(K + 1) * S
        if mode == "tc":
            e = e + (5 + 2.0 ** -5) * K * 2.0 ** -30 * np.outer(_pow2_scale(ha.max(axis=1)), _pow2_scale(Wa.max(axis=0)))
        elif mode == "fp16":
            steps = 3 * ((K + 63) // 64 * 64) // 16
            wmax = Wa.max()
            inv_s = np.where(rowb > 0, np.maximum(2.0 ** -13 * rowb, 2.0 ** -100), 0.0)
            small = (2.0 ** -33 * wmax * ha.sum(axis=1)[:, None] + 2.0 ** -24 * np.outer(inv_s, Wa.sum(axis=0))
                     + K * 2.0 ** -56 * wmax * inv_s[:, None])
            e = e + (2.0 ** -20 + steps * 2.0 ** -22 * 1.002) * S + (1 + steps * 2.0 ** -22) * small
            rowb = (ha.max(axis=1) * (1 + 2.0 ** -21) * Wa.sum(axis=0).max() * (1 + 2.0 ** -22)
                    + (np.abs(b).max() if b is not None else 0.0)) * (1 + 2.0 ** -50)
        e = e * (1 + 2 * U) + 2 * U * np.abs(y)
        if b is None:
            return y, e
        h = onn.relu(y)
        if mode == "tc":
            e = e + 2.0 ** -24 * (h + e) + 2.0 ** -149
        d = e


def _bound(ws, inputs, with_uprev, mode, xscale=None):
    """Bound of |u_kernel - u_reference| per element (the clip is 1-Lipschitz, so it holds with and without it): the
    two network passes, then us + (f1 - f2) in the kernel and (us + f1) - f2 in the reference, 2 roundings each."""
    a1, a2, us, _ = _operands(inputs, with_uprev, xscale)
    f1, e1 = _pass_bound(ws, a1, mode)
    f2, e2 = _pass_bound(ws, a2, mode)
    return (e1 + e2) * (1 + 4 * U) + 4 * U * (np.abs(us) + np.abs(f1) + np.abs(f2))


def _check_within(out, ref, bound, what):
    err = np.abs(out - ref)
    ok = np.isfinite(out) & (err <= bound)
    worst = float(np.max(np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))))
    assert np.all(ok), (what, worst, np.argwhere(~ok)[:5].tolist())
    return worst


def _clip_bounds(rng, nu):
    return -rng.uniform(0.5, 2.0, nu), rng.uniform(0.5, 2.0, nu)


# --------------------------------------------------------------------------------------------- (a) shape sweep
SHAPES = [  # with_uprev, nx, nu, hidden widths, B (the kernels see M = 2B rows)
    (False, 1, 1, [], 1),                          # no hidden layer, input width 3, M = 2
    (True, 3, 1, [], 63),                          # no hidden layer, nx = 3 with uprev, M = 126
    (False, 3, 2, [1], 64),                        # width-1 hidden layer, M = 128
    (True, 3, 3, [63], 65),                        # M = 130
    (False, 5, 33, [64, 65], 337),                 # 6 tiles of 128 rows, the last one partial
    (True, 4, 32, [127, 128, 129], 200),
    (True, 12, 2, [2049], 65),
    (False, 3, 3, [65, 64, 63, 129, 128, 127, 33, 2, 65, 64, 48, 31, 129, 17, 5], 97),   # 16 layers
]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("with_uprev,nx,nu,hidden,B", SHAPES)
def test_forward_within_derived_bound(torch_cuda, with_uprev, nx, nu, hidden, B, mode):
    """Every output element within the worst-case bound of _pass_bound / _bound, with and without the state scaling
    and the per-column clip.  The weights hold dead units, a unit whose weights span 1e-8..1 and large biases; the
    samples hold zero rows, rows mixing 1e6 and 1e-6, and rows that switch the whole first hidden layer on or off."""
    rng = np.random.default_rng(1000 * nx + 10 * nu + len(hidden))
    in_w = 2 * nx + (2 if with_uprev else 1) * nu
    ws = _weights(rng, [in_w] + hidden + [nu])
    inputs = _inputs(rng, B, nx, nu, with_uprev)
    if hidden and hidden[0] >= 2 and B >= 4:       # the data does what the docstring says
        pre = _operands(inputs, with_uprev, None)[0] @ ws[0] + ws[1]
        live = pre[:, 1:]
        assert np.any(np.all(live > 0, axis=1)) and np.any(np.all(live <= 0, axis=1))
    layer = _layer(ws, with_uprev, mode)
    xscale = rng.uniform(0.5, 2.0, nx)
    ulb, uub = _clip_bounds(rng, nu)
    worst = 0.0
    for sc, lb, ub in ((None, None, None), (xscale, ulb, uub)):
        out = layer.forward(*(inputs if with_uprev else [inputs[0], None, inputs[1], inputs[2]]),
                            xscale=sc, ulb=lb, uub=ub)
        ref = _reference(ws, inputs, with_uprev, sc, lb, ub)
        bound = _bound(ws, inputs, with_uprev, mode, sc)
        worst = max(worst, _check_within(out, ref, bound, (mode, sc is not None)))
        if lb is not None:
            assert np.all(out >= lb) and np.all(out <= ub)
    print(f"{mode} L={len(hidden) + 1} widths={hidden} nu={nu} B={B}: worst error / bound = {worst:.3g}")


# --------------------------------------------------------------------------------------------- (b) homogeneity
@pytest.mark.parametrize("mode,ks", [("f64", (1, -1, 60, -60, 200, -200)), ("tc", (1, -1, 20, -20, 60, -60)),
                                     ("fp16", (1, -1, 20, -20, 60, -60))])
@pytest.mark.parametrize("with_uprev,nx,nu,hidden,B", [(True, 3, 2, [65, 64], 130), (False, 5, 33, [129], 64),
                                                        (True, 4, 3, [], 65)])
def test_power_of_two_homogeneity_is_bitwise(torch_cuda, with_uprev, nx, nu, hidden, B, mode, ks):
    """A ReLU network with biases b satisfies f_(2^k b)(2^k a) = 2^k f_b(a), and every row scale of the three modes is
    a power of two taken from an exact maximum, so a handle with biases x 2^k fed x, uprev, xs, us x 2^k (no clip)
    returns exactly 2^k x the first handle's output.  This holds while nothing leaves the normal range: the fp32
    hidden store of "tc" (and the fp32 row maxima of "fp16") keep |h| 2^k inside [2^-126, 2^128), checked below on
    the reference activations; |k| <= 60 there, |k| <= 200 for "f64"."""
    rng = np.random.default_rng(7 * nx + nu)
    in_w = 2 * nx + (2 if with_uprev else 1) * nu
    ws = _weights(rng, [in_w] + hidden + [nu])
    mag = np.exp(rng.uniform(-2, 2, (B, 1)))
    x, xs = rng.standard_normal((B, nx)) * mag, rng.standard_normal((B, nx)) * mag
    up, us = rng.uniform(-1, 1, (B, nu)) * mag, rng.uniform(-1, 1, (B, nu)) * mag
    for a in (x, up, xs, us):
        a[0] = 0.0
    xscale = rng.uniform(0.5, 2.0, nx)
    if mode != "f64" and hidden:
        for a in _operands([x, up, xs, us] if with_uprev else [x, xs, us], with_uprev, xscale)[:2]:
            for i in range(len(hidden)):
                a = onn.relu(a @ ws[2 * i] + ws[2 * i + 1])
                nz = np.abs(a[a != 0])
                assert nz.min() * 2.0 ** -60 >= 2.0 ** -126 and nz.max() * 2.0 ** 60 < 2.0 ** 127
    base = _layer(ws, with_uprev, mode)
    out0 = base.forward(x, up if with_uprev else None, xs, us, xscale=xscale)
    assert np.all(np.isfinite(out0))
    for k in ks:
        wk = [w if i % 2 == 0 else np.ldexp(w, k) for i, w in enumerate(ws)]
        lk = _layer(wk, with_uprev, mode)
        s = lambda a: np.ldexp(a, k)
        outk = lk.forward(s(x), s(up) if with_uprev else None, s(xs), s(us), xscale=xscale)
        assert np.array_equal(outk, np.ldexp(out0, k)), (mode, k, float(np.max(np.abs(np.ldexp(outk, -k) - out0))))


# --------------------------------------------------------------------------------------------- (c) non-finite
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("with_uprev,nx,nu,hidden", [(True, 3, 3, [65, 64]), (False, 2, 2, [])])
def test_nonfinite_samples(torch_cuda, with_uprev, nx, nu, hidden, mode):
    """NaN, +Inf and -Inf in one entry of x, uprev, xs or us of samples 63 and 64 (rows 126/127 and 128/129: the last
    rows of one 128-row tile and the first of the next) and of the last sample, with and without the clip.  Every
    other sample is bitwise what a run without the bad entries gives.  A NaN sample is NaN in every component, as
    in the reference (its ReLU and clip are np.where forms that keep a NaN).  With an infinity the output is
    non-finite wherever the reference is; "f64" is finite exactly where the reference is, while "tc" and "fp16" may
    return NaN where the reference is finite (for example where the clip catches an infinity): a row holding an
    infinity has no finite scale."""
    rng = np.random.default_rng(31 + nx)
    B = 200
    in_w = 2 * nx + (2 if with_uprev else 1) * nu
    ws = _weights(rng, [in_w] + hidden + [nu])
    clean = _inputs(rng, B, nx, nu, with_uprev)
    layer = _layer(ws, with_uprev, mode)
    xscale = rng.uniform(0.5, 2.0, nx)
    ulb, uub = _clip_bounds(rng, nu)
    bad = np.array([63, 64, B - 1])
    good = np.setdiff1d(np.arange(B), bad)
    names = ["x", "uprev", "xs", "us"] if with_uprev else ["x", "xs", "us"]
    call = lambda ins, sc, lb, ub: layer.forward(*(ins if with_uprev else [ins[0], None, ins[1], ins[2]]),
                                                 xscale=sc, ulb=lb, uub=ub)
    for sc, lb, ub in ((None, None, None), (xscale, ulb, uub)):
        out_clean = call(clean, sc, lb, ub)
        for blk in range(len(names)):
            for val in (np.nan, np.inf, -np.inf):
                ins = [a.copy() for a in clean]
                cols = rng.integers(0, ins[blk].shape[1], bad.size)
                ins[blk][bad, cols] = val
                out = call(ins, sc, lb, ub)
                ref = _reference(ws, ins, with_uprev, sc, lb, ub)
                what = (mode, names[blk], val, sc is not None)
                assert np.array_equal(out[good], out_clean[good]), what
                if np.isnan(val):
                    assert np.all(np.isnan(ref[bad])) and np.all(np.isnan(out[bad])), what
                else:
                    assert np.all(~np.isfinite(out[bad][~np.isfinite(ref[bad])])), what
                    if mode == "f64":
                        assert np.array_equal(np.isfinite(out[bad]), np.isfinite(ref[bad])), what


# --------------------------------------------------------------------------------------------- (d) chunks, K limit
CHUNK = {"tc": 1 << 18, "f64": 1 << 20, "fp16": 131072}


@pytest.mark.parametrize("mode", MODES)
def test_batch_chunk_boundaries(torch_cuda, mode):
    """A batch just above the mode's internal chunk (input and hidden widths <= 128, so the chunk is the cap: 2^18
    samples for "tc", 2^20 for "f64", 131072 for "fp16"): the samples on both sides of the boundary, the first and
    the last are within the bound, and bitwise equal to a separate call that holds just those samples."""
    torch = torch_cuda
    with_uprev, nx, nu, hidden = True, 4, 3, [32, 17]
    c = CHUNK[mode]
    B = c + 3
    rng = np.random.default_rng(5)
    ws = _weights(rng, [2 * nx + 2 * nu] + hidden + [nu])
    layer = _layer(ws, with_uprev, mode)
    g = torch.Generator(device="cuda").manual_seed(11)
    dev = lambda n: torch.randn((B, n), generator=g, device="cuda", dtype=torch.float64)
    x, up, xs, us = dev(nx), dev(nu), dev(nx), dev(nu)
    out = layer.forward(x, up, xs, us).cpu().numpy()
    idx = np.array([0, c - 2, c - 1, c, c + 1, B - 1])
    ti = torch.tensor(idx, device="cuda")
    sub = [a.index_select(0, ti).contiguous() for a in (x, up, xs, us)]
    small = layer.forward(*sub).cpu().numpy()
    assert np.array_equal(out[idx], small), mode
    host = [a.cpu().numpy() for a in sub]
    _check_within(out[idx], _reference(ws, host, with_uprev), _bound(ws, host, with_uprev, mode), mode)


@pytest.mark.parametrize("mode", MODES)
def test_contraction_length_limit(torch_cuda, mode):
    """Input width 32768, the longest contraction the INT8 digit planes take (int32 accumulators), is accepted and
    within the bound in every mode; width 32769 is refused when the handle is created, naming the limit."""
    from industrial_nnmpc_2021_b200 import _lib
    rng = np.random.default_rng(3)
    nx, nu, B = 16383, 2, 5
    ws = _weights(rng, [2 * nx + nu, 8, nu])
    ins = _inputs(rng, B, nx, nu, False)
    out = _layer(ws, False, mode)(ins)
    _check_within(out, _reference(ws, ins, False), _bound(ws, ins, False, mode), mode)
    ws = _weights(rng, [2 * 16384 + 1, 8, 1])
    with pytest.raises(_lib.NnmpcError, match=r"status -1\).*32768"):
        _layer(ws, False, mode)


# --------------------------------------------------------------------------------------------- (e) one handle
def test_one_handle_across_batches_and_modes(torch_cuda):
    """One handle, B = 3000 -> 5 -> 70000 -> 64, switching f64 -> tc -> fp16 -> tc between the calls: every result is
    bitwise what a fresh handle in that mode returns, and within the bound.  Catches digit planes, padding rows and
    per-row scale buffers that the modes share and that a smaller or earlier call left behind."""
    rng = np.random.default_rng(17)
    with_uprev, nx, nu, hidden = True, 4, 3, [65, 64]
    ws = _weights(rng, [2 * nx + 2 * nu] + hidden + [nu])
    shared = _layer(ws, with_uprev, "f64")
    for B, mode in ((3000, "f64"), (5, "tc"), (70000, "fp16"), (64, "tc")):
        ins = _inputs(rng, B, nx, nu, with_uprev)
        _set_mode(shared, mode)
        out = shared(ins)
        assert np.array_equal(out, _layer(ws, with_uprev, mode)(ins)), (B, mode)
        _check_within(out, _reference(ws, ins, with_uprev), _bound(ws, ins, with_uprev, mode), (B, mode))
