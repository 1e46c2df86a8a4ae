"""Training step of the structured network on the GPU (cdu_train.py:24-62, cstrs_train.py:24-61: Keras
compile(optimizer='adam', loss='mean_squared_error') + fit) against a hand-written NumPy backpropagation + Adam."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import nn as onn


@pytest.fixture(scope="module")
def torch_cuda(built_lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _problem(rng, with_uprev, nx, nu, hidden, B):
    in_w = 2 * nx + (2 if with_uprev else 1) * nu
    dims = [in_w] + hidden + [nu]
    ws = []
    for i in range(len(dims) - 1):
        lim = np.sqrt(6.0 / (dims[i] + dims[i + 1]))
        ws.append(rng.uniform(-lim, lim, (dims[i], dims[i + 1])))
        if i < len(dims) - 2:
            ws.append(0.05 * rng.standard_normal(dims[i + 1]))
    x, xs = rng.standard_normal((B, nx)), rng.standard_normal((B, nx))
    up, us = rng.uniform(-1, 1, (B, nu)), rng.uniform(-1, 1, (B, nu))
    u = np.clip(us + 0.3 * rng.standard_normal((B, nu)), -1, 1)
    return ws, ([x, up, xs, us] if with_uprev else [x, xs, us]), u


@pytest.mark.parametrize("with_uprev,nx,nu,hidden,B", [(True, 12, 6, [40, 32, 24], 257), (False, 12, 6, [33, 17], 64),
                                                        (False, 252, 32, [128, 96, 64], 300),
                                                        (False, 1, 1, [], 33),           # no hidden layer, nu = 1
                                                        (False, 4, 3, [17], 45)])        # odd input width 11
def test_training_steps_match_numpy_backprop_and_adam(torch_cuda, with_uprev, nx, nu, hidden, B):
    from industrial_nnmpc_2021_b200.LinearMPCLayers import RegulatorLayerWithUprev, RegulatorLayerWithoutUprev
    rng = np.random.default_rng(nx + nu + B)
    ws, inputs, u = _problem(rng, with_uprev, nx, nu, hidden, B)
    layer = (RegulatorLayerWithUprev if with_uprev else RegulatorLayerWithoutUprev)(layer_dims=hidden + [nu], precision="f64")
    layer.set_weights(ws)
    w, m, v = [a.copy() for a in ws], [np.zeros_like(a) for a in ws], [np.zeros_like(a) for a in ws]
    for t in range(1, 5):
        loss_o, grads = onn.mse_loss_and_grads(w, inputs, u, with_uprev)
        w, m, v = onn.adam_step(w, grads, m, v, t)
        loss_g = layer.train_on_batch(inputs, u)
        assert abs(loss_g - loss_o) <= 1e-12 * max(1.0, loss_o), (t, loss_g, loss_o)
        got = layer.get_weights()
        for k, (a, b) in enumerate(zip(got, w)):
            assert a.shape == b.shape and np.max(np.abs(a - b)) <= 1e-11, (t, k, np.max(np.abs(a - b)))
    # the trained weights drive the inference paths (operators are rebuilt after training steps)
    out = layer(inputs)
    assert np.max(np.abs(out - onn.layer_call(w, inputs, with_uprev))) <= 1e-10
    assert abs(layer.evaluate(inputs, u) - onn.mse_loss_and_grads(w, inputs, u, with_uprev)[0]) <= 1e-12


def test_fit_reduces_validation_loss_and_restores_best_weights(torch_cuda):
    """RegulatorModel.compile / fit as cdu_train.py uses them (validation_split, best-val-loss weights), on a
    target that IS a structured network, so the loss must fall steadily (measured: 0.192 -> 0.0186 in 30 epochs of 15 Adam steps at the Keras default rate)."""
    from industrial_nnmpc_2021_b200.LinearMPCLayers import RegulatorModel
    rng = np.random.default_rng(0)
    nx, nu, B = 6, 3, 4096
    teacher = RegulatorModel(Nx=nx, Nu=nu, regulator_dims=[0, 24, 24, nu], nnwithuprev=False, seed=5, precision="f64")
    x, xs, us = rng.standard_normal((B, nx)), 0.3 * rng.standard_normal((B, nx)), rng.uniform(-1, 1, (B, nu))
    u = teacher([x, xs, us])
    model = RegulatorModel(Nx=nx, Nu=nu, regulator_dims=[0, 24, 24, nu], nnwithuprev=False, seed=9)
    model.compile(optimizer="adam", loss="mean_squared_error")
    l0 = model.evaluate([x, xs, us], [u])
    hist = model.fit(x=[x, xs, us], y=[u], epochs=30, batch_size=256, validation_split=0.05)
    assert len(hist["loss"]) == 30 and len(hist["val_loss"]) == 30
    assert hist["loss"][-1] < 0.2 * l0 and min(hist["val_loss"]) < 0.2 * l0
    assert hist["loss"][-1] < hist["loss"][9] < hist["loss"][0]
    nval = int(B * 0.05)
    # the restored weights are those of the best validation epoch, and the default (INT8 tensor-core) forward uses them
    best = model.evaluate([a[B - nval:] for a in (x, xs, us)], [u[B - nval:]])
    assert abs(best - min(hist["val_loss"])) <= 1e-12 * max(1.0, best)
    pred = model.predict([x[:64], xs[:64], us[:64]])
    from oracle import nn as onn2
    assert np.max(np.abs(pred - onn2.layer_call(model.get_weights(), [x[:64], xs[:64], us[:64]], False))) <= 1e-6
