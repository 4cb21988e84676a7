"""CPU checks of the fp64 split-minibatch reference that the GPU tests of vbnn_mlp_forward_train /
vbnn_mlp_backward_update compare against: fed the ClassNLL gradient it IS the oracle's fused minibatch."""
import copy

import numpy as np
import pytest
import torch

from custom_loss_reference import autograd_grad, classnll_grad, custom_minibatch
from oracle import vbnn_oracle as O


def make_pair(reparam, vb_output, S, operand_round=None, sizes=(11, 9, 8, 5)):
    opt = O.default_opt(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])],
                        S=S, B=30.0, mu_init=1, var_init=0.01, reparam=reparam, vb_output=vb_output,
                        strict_reference=False, log=False)
    a = O.MLPOracle(opt, torch.float64, seed=3, operand_round=operand_round)
    return a, copy.deepcopy(a), opt


def noise_for(ref, S, N, lrt, rng):
    if lrt:
        return [[torch.from_numpy(rng.randn(N, l.O)) for l in ref.vb_all] for _ in range(S)]
    return [[torch.from_numpy(rng.randn(l.O, l.I)) for l in ref.vb_all] for _ in range(S)]


def state(ref):
    out = []
    for l in ref.vb + [ref.out]:
        out += [l.weight, l.bias, l.gradWeight, l.gradBias]
        if isinstance(l, O.VBLinearOracle):
            out += [l.means, l.lvars, l.gradSum, l.meanState["m"], l.meanState["v"], l.varState["m"], l.varState["v"]]
    return out


@pytest.mark.parametrize("operand_round", [None, O.round_bf16], ids=["fp64", "bf16_round"])
@pytest.mark.parametrize("vb_output", [False, True])
@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_classnll_gradient_reproduces_the_oracle_minibatch(reparam, vb_output, operand_round):
    """Two minibatches: the reference fed the ClassNLL gradient leaves the parameters, gradients and Adam state of
    O.train_minibatch to <= 1e-12, and its dX is the oracle's sum over samples of the first layer's gradInput."""
    S, N = 3, 6
    lrt = reparam == "local"
    a, b, opt = make_pair(reparam, vb_output, S, operand_round)
    rng = np.random.RandomState(0)
    first = a.vb[0]
    for it in range(2):
        X = torch.from_numpy(rng.randn(N, opt["input_size"]))
        T = torch.from_numpy(rng.randint(1, len(opt["classes"]) + 1, N).astype(np.float64))
        noise = noise_for(a, S, N, lrt, rng)
        # the oracle's minibatch, summing the first layer's gradInput over the samples as it goes
        a.resetGradients()
        dx_want = 0
        for s in range(S):
            a.sample(None if lrt else noise[s])
            a.run(X, T, noise[s] if lrt else None)
            dx_want = dx_want + first.gradInput
        logits_last = a.out.output.clone()
        a.update(opt)
        Y, G, dX = custom_minibatch(b, X, classnll_grad(T), noise, lrt, opt)
        assert torch.allclose(Y[-1], logits_last, rtol=0, atol=1e-12)
        assert float((dX - dx_want).abs().max()) <= 1e-12 * max(1.0, float(dx_want.abs().max()))
        for x, y in zip(state(a), state(b)):
            assert float((x - y).abs().max()) <= 1e-12 * max(1.0, float(x.abs().max())), it


def test_autograd_gradient_of_the_summed_nll_is_the_classnll_gradient():
    """loss = sum_s nll_loss(log_softmax(Y_s)) through autograd equals the per-sample ClassNLL gradient: the
    convention the split path documents for reproducing vbnn_mlp_step."""
    g = torch.Generator().manual_seed(1)
    Y = torch.randn(3, 7, 5, generator=g, dtype=torch.float64)
    T = torch.randint(1, 6, (7,), generator=g).double()
    want = classnll_grad(T)(Y)
    got = autograd_grad(lambda y: sum(torch.nn.functional.nll_loss(torch.log_softmax(y[s], -1), T.long() - 1)
                                      for s in range(y.shape[0])))(Y)
    assert torch.allclose(got, want, rtol=0, atol=1e-15)


def test_mse_gradient_reaches_the_parameters():
    """A regression loss: the reference's output-layer gradWeight is sum_s G_s^T A_s with G = dMSE/dY."""
    S, N = 2, 5
    _, ref, opt = make_pair("weight", False, S)
    rng = np.random.RandomState(2)
    X = torch.from_numpy(rng.randn(N, opt["input_size"]))
    R = torch.from_numpy(rng.randn(N, len(opt["classes"])))
    noise = noise_for(ref, S, N, False, rng)
    Y, G, _ = custom_minibatch(ref, X, autograd_grad(lambda y: ((y - R) ** 2).mean(dim=(1, 2)).sum()), noise, False,
                               opt, update=False)
    assert torch.allclose(G, 2 * (Y - R) / (N * len(opt["classes"])), rtol=0, atol=1e-15)
    assert float(ref.out.gradWeight.abs().max()) > 0
