"""CPU checks of the fp64 activation reference (tests/activation_reference.py) that the GPU tests of
vbnn_mlp_set_activation compare against: without operand rounding it is torch fp64 autograd through torch.tanh,
torch.sigmoid and F.elu, and at ReLU it is custom_loss_reference bit for bit."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import activation_reference as A
from custom_loss_reference import classnll_grad, custom_minibatch
from oracle import vbnn_oracle as O
from test_custom_loss_cpu import make_pair, noise_for, state

TORCH_ACT = {"relu": torch.relu, "tanh": torch.tanh, "sigmoid": torch.sigmoid, "elu": F.elu}


@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("kind", ["tanh", "sigmoid", "elu"])
def test_matches_fp64_autograd(kind, reparam):
    """One sample through a 11-9-8-5 net: the outputs, the input gradient and every layer's gradWeight (and, in local
    mode, gradSum = H^T X^2, the derivative with respect to s2 written as autograd's d/ds2) agree with fp64 autograd
    through the torch module to <= 1e-12."""
    N = 7
    lrt = reparam == "local"
    ref, _, opt = make_pair(reparam, True, 1)
    rng = np.random.RandomState(1)
    x = torch.from_numpy(rng.randn(N, opt["input_size"]))
    noise = noise_for(ref, 1, N, lrt, rng)[0]
    G = torch.from_numpy(rng.randn(N, len(opt["classes"])))
    ref.resetGradients()
    ref.sample(None if lrt else noise)
    acts, Y = A.forward(ref, x, kind, noise if lrt else None)
    dX = A.backward(ref, acts, G, kind)

    xa = x.clone().requires_grad_(True)
    h, leaves = xa, []
    layers = ref.vb + [ref.out]
    for k, lyr in enumerate(layers):
        if lrt:
            mu = lyr.means.clone().requires_grad_(True)
            s2 = torch.exp(lyr.lvars).requires_grad_(True)
            y = h @ mu.t() + lyr.bias + torch.sqrt((h * h) @ s2.t()) * noise[k]
            leaves.append((mu, s2))
        else:
            w = lyr.weight.clone().requires_grad_(True)
            y = h @ w.t() + lyr.bias
            leaves.append((w, None))
        h = TORCH_ACT[kind](y) if k < len(layers) - 1 else y
    assert float((h.detach() - Y).abs().max()) <= 1e-12
    grads = torch.autograd.grad((h * G).sum(), [xa] + [t for pair in leaves for t in pair if t is not None])
    assert float((grads[0] - dX).abs().max()) <= 1e-12 * max(1.0, float(dX.abs().max()))
    it = iter(grads[1:])
    for lyr, (w, s2) in zip(layers, leaves):
        gw = next(it)
        assert float((gw - lyr.gradWeight).abs().max()) <= 1e-12 * max(1.0, float(gw.abs().max()))
        if s2 is not None:
            gs = next(it)
            # d/ds2 of sqrt(X^2 s2^T) zeta is H^T X^2 with H = G zeta / (2 sqrt V): the reference's gradSum
            assert float((gs - lyr.gradSum).abs().max()) <= 1e-12 * max(1.0, float(gs.abs().max()))


@pytest.mark.parametrize("operand_round", [None, O.round_bf16], ids=["fp64", "bf16_round"])
@pytest.mark.parametrize("vb_output", [False, True])
@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_relu_is_custom_loss_reference(reparam, vb_output, operand_round):
    """Two minibatches under the ClassNLL gradient: at ReLU the activation reference leaves outputs, dX, gradients,
    parameters and Adam state bit-identical to custom_loss_reference.custom_minibatch."""
    S, N = 3, 6
    lrt = reparam == "local"
    a, b, opt = make_pair(reparam, vb_output, S, operand_round)
    rng = np.random.RandomState(0)
    for _ in range(2):
        X = torch.from_numpy(rng.randn(N, opt["input_size"]))
        T = torch.from_numpy(rng.randint(1, len(opt["classes"]) + 1, N).astype(np.float64))
        noise = noise_for(a, S, N, lrt, rng)
        Ya, Ga, dXa = custom_minibatch(a, X, classnll_grad(T), noise, lrt, opt)
        Yb, Gb, dXb = A.minibatch(b, X, classnll_grad(T), noise, lrt, "relu", opt)
        assert torch.equal(Ya, Yb) and torch.equal(Ga, Gb) and torch.equal(dXa, dXb)
        for x, y in zip(state(a), state(b)):
            assert torch.equal(x, y)


@pytest.mark.parametrize("kind", A.KINDS)
def test_rounding_points(kind):
    """With operand rounding the stored activation is q(f(y)) and f' is formed from it: the hidden layer's gradient
    is q(g_in * f'(q(a)))."""
    ref, _, opt = make_pair("weight", False, 1, O.round_bf16)
    rng = np.random.RandomState(3)
    N = 5
    x = ref.q(torch.from_numpy(rng.randn(N, opt["input_size"])))
    noise = noise_for(ref, 1, N, False, rng)[0]
    ref.sample(noise)
    acts, _ = A.forward(ref, x, kind)
    for a in acts[1:]:
        assert torch.equal(a, O.round_bf16(a))
    ref.resetGradients()
    G = torch.from_numpy(rng.randn(N, len(opt["classes"])))
    A.backward(ref, acts, G, kind)
    # the last hidden layer's gradient operand, restated: q(q(G) W_out * f'(a)) with a the stored (rounded) output
    want = O.round_bf16((O.round_bf16(G) @ O.round_bf16(ref.out.weight)) * A.act_grad(kind, acts[-1]))
    assert torch.equal(ref.vb[-1].gradWeight, want.t() @ acts[-2])


def test_saturation_and_derivatives():
    """The derivatives from the output at the saturated and the exact-zero ends: tanh(+-100) = +-1 and sigmoid(100) = 1
    with f' exactly 0, ELU(-100) = -1 with f' exactly 0; f'(0) is 1, 1/4 and 1."""
    y = torch.tensor([-100.0, 0.0, 100.0], dtype=torch.float64)
    a = A.act("tanh", y)
    assert torch.equal(a, torch.tensor([-1.0, 0.0, 1.0], dtype=torch.float64))
    assert torch.equal(A.act_grad("tanh", a), torch.tensor([0.0, 1.0, 0.0], dtype=torch.float64))
    s = A.act("sigmoid", y)
    assert s[2] == 1.0 and A.act_grad("sigmoid", s)[2] == 0.0 and A.act_grad("sigmoid", s)[1] == 0.25
    e = A.act("elu", y)
    assert e[0] == -1.0 and A.act_grad("elu", e)[0] == 0.0 and A.act_grad("elu", e)[1] == 1.0
    z = torch.linspace(-6, 6, 97, dtype=torch.float64)
    for kind in ("tanh", "sigmoid", "elu"):
        za = z.clone().requires_grad_(True)
        (d,) = torch.autograd.grad(TORCH_ACT[kind](za).sum(), za)
        assert float((A.act_grad(kind, A.act(kind, z)) - d).abs().max()) <= 1e-15


def test_predict_forward_map_uses_the_means():
    """predict_forward's MAP pass (vbnn_mlp_test / predict with 0 samples) is the forward with W = mu."""
    ref, _, opt = make_pair("weight", False, 1)
    twin = copy.deepcopy(ref)
    rng = np.random.RandomState(4)
    x = torch.from_numpy(rng.randn(4, opt["input_size"]))
    got = A.predict_forward(ref, x, "tanh", None, False, map_mode=True)[0]
    for lyr in twin.vb_all:
        lyr.weight.copy_(lyr.means)
    _, want = A.forward(twin, x, "tanh")
    assert torch.equal(got, want)
