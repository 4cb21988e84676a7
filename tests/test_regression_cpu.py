"""CPU checks of the regression criteria (vbnn_mlp_set_criterion) in fp64: the references of
tests/regression_reference.py against torch's own losses, autograd and the closed forms, including NaN-masked targets,
log-variances of +-100 and y == m; the fp32 statements of k_loss_reg stay finite wherever the exact value is
representable and give dm == 0 exactly where y == m; the fp64 minibatch of tests/custom_loss_reference.py runs under
them; and MLP.set_criterion rejects an unknown name before it reaches the library."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from custom_loss_reference import autograd_grad, custom_minibatch
from oracle import vbnn_oracle as O
from regression_reference import closed_form_grad, emulate_fp32, loss_sum, scalars

F32_MAX = float(np.finfo(np.float32).max)


def extreme_case(crit, S=2, N=5, K=3, seed=0):
    """Y [S x N x C], y [N x K] with a NaN row, a NaN column entry, y == m entries and s in {-100, 100}."""
    rng = np.random.RandomState(seed)
    C = 2 * K if crit == "gaussian_nll" else K
    Y = rng.randn(S, N, C)
    y = rng.randn(N, K)
    y[1, :] = np.nan                                   # a padding row
    y[3, 2] = np.nan                                   # one missing element
    y[0, 0] = Y[0, 0, 0] = Y[1, 0, 0]                  # y == m in both samples
    if crit == "gaussian_nll":
        Y[:, 2, K + 0] = -100.0                        # e^{-s} = 2.7e43 overflows fp32 ...
        y[2, 0] = Y[0, 2, 0] + 1e-20                   # ... but the terms with (y - m) = 1e-20 are representable
        Y[1, 2, 0] = Y[0, 2, 0]
        Y[:, 4, K + 1] = 100.0                         # e^{-s} = 3.7e-44: subnormal in fp32
        Y[:, 0, K + 0] = -100.0                        # y == m under s = -100: dm must be 0, not 0 * inf
        y[0, 0] = Y[0, 0, 0]
    return Y, y


def test_losses_match_torch():
    rng = np.random.RandomState(1)
    Y = torch.from_numpy(rng.randn(3, 7, 4))
    y = torch.from_numpy(rng.randn(7, 4))
    want = sum(F.mse_loss(Y[s], y) for s in range(3))
    assert abs(float(loss_sum("mse", y)(Y)) - float(want)) <= 1e-14 * abs(float(want))
    Yg = torch.from_numpy(rng.randn(3, 7, 4))
    yg = torch.from_numpy(rng.randn(7, 2))
    m, s = Yg[..., :2], Yg[..., 2:]
    want = (0.5 * (s + (yg - m) ** 2 * torch.exp(-s))).mean(dim=(1, 2)).sum()
    assert abs(float(loss_sum("gaussian_nll", yg)(Yg)) - float(want)) <= 1e-14 * abs(float(want))
    # gaussian_nll is torch's gaussian_nll_loss with var = e^s, less its constant
    g = sum(F.gaussian_nll_loss(m[i], yg, torch.exp(s[i]), full=False) for i in range(3))
    assert abs(float(g) - float(want)) <= 1e-12 * abs(float(want))


@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
def test_autograd_equals_closed_form_with_masking_and_extremes(crit):
    Y, y = extreme_case(crit)
    Yt, yt = torch.from_numpy(Y), torch.from_numpy(y)
    G = autograd_grad(loss_sum(crit, yt, n_global=4 * Y.shape[1]))(Yt).numpy()
    Gc = closed_form_grad(crit, Y, y, 4 * Y.shape[1])
    assert np.isfinite(G).all() and np.isfinite(Gc).all()
    np.testing.assert_allclose(G, Gc, rtol=1e-12, atol=0)
    K = y.shape[1]
    assert (G[:, 1, :] == 0).all()                                     # NaN row: no gradient
    assert G[0, 3, 2] == 0 and (crit == "mse" or G[0, 3, K + 2] == 0)   # NaN element
    assert G[0, 0, 0] == 0 and G[1, 0, 0] == 0                          # y == m
    # the NaN elements add nothing to either scalar; the means still divide by N K
    e, a = scalars(crit, Y, y)
    mask = ~np.isnan(y)
    se = np.where(mask, np.nan_to_num(y) - Y[..., :K], 0) ** 2
    assert abs(a - se.sum(axis=(1, 2)).mean() / y.size) <= 1e-14 * a
    if crit == "mse":
        assert e == a


@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
def test_kernel_statements_finite_and_exact(crit):
    """k_loss_reg's fp32 statements: every gradient element whose exact value is representable is finite and within
    1e-6 of it (relative, or of 1 / (N K) where 1 - q^2 cancels), the loss sum is finite (its exact value is), and dm
    is exactly 0 where y == m (s = -100 included)."""
    Y, y = extreme_case(crit)
    ng = Y.shape[1]
    G32, loss = emulate_fp32(crit, Y.astype(np.float32), y.astype(np.float32), ng)
    Gx = closed_form_grad(crit, Y.astype(np.float32).astype(np.float64), y.astype(np.float32).astype(np.float64), ng)
    rep = np.abs(Gx) < F32_MAX
    assert rep.all()
    assert np.isfinite(G32).all()
    # relative 1e-6, or 1e-6 of the scale 1 / (N K) where ds = (1 - q^2) / (2 N K) cancels
    np.testing.assert_allclose(G32, Gx, rtol=1e-6, atol=1e-6 / (ng * y.shape[1]))
    assert G32[0, 0, 0] == 0 and G32[1, 0, 0] == 0
    want, _ = scalars(crit, Y.astype(np.float32), y.astype(np.float32))
    got = loss / (ng * y.shape[1]) / Y.shape[0]
    assert np.isfinite(got) and abs(got - want) <= 1e-6 * abs(want)
    if crit == "gaussian_nll":
        # the naive (y - m)^2 e^{-s} of the s = -100 element overflows fp32; q^2 does not
        d = np.float32(y[2, 0]) - np.float32(Y[0, 2, 0])
        with np.errstate(over="ignore"):
            assert not np.isfinite(np.float32(d * d) * np.exp(np.float32(100.0)))


@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
@pytest.mark.parametrize("lrt", [False, True])
def test_fp64_minibatch_runs_under_the_criteria(crit, lrt):
    """custom_minibatch with the criterion's autograd gradient equals the one with the closed form (fp64, 1e-12) and
    moves the parameters."""
    sizes, N, S = [9, 7, 4], 6, 2
    over = dict(input_size=sizes[0], hidden=[sizes[1]], classes=[str(i) for i in range(sizes[-1])], S=S, B=30.0,
                batchSize=N, mu_init=1, var_init=0.01, reparam="local" if lrt else "weight", strict_reference=False,
                log=False)
    oopt = O.default_opt(**over)
    rng = np.random.RandomState(3)
    x = torch.from_numpy(rng.randn(N, sizes[0]))
    K = sizes[-1] // 2 if crit == "gaussian_nll" else sizes[-1]
    y = rng.randn(N, K)
    y[2, :] = np.nan
    outs = []
    for grad_fn in (autograd_grad(loss_sum(crit, torch.from_numpy(y))),
                    lambda Yv: torch.from_numpy(closed_form_grad(crit, Yv.numpy(), y, N))):
        ref = O.MLPOracle(oopt, torch.float64, seed=3)
        g = torch.Generator().manual_seed(5)
        if lrt:
            noise = [[torch.randn(N, o, generator=g, dtype=torch.float64) for o in sizes[1:]] for _ in range(S)]
        else:
            noise = [[torch.randn(o, i, generator=g, dtype=torch.float64) for i, o in zip(sizes[:-2], sizes[1:-1])]
                     for _ in range(S)]
        m0 = ref.vb[0].means.clone()
        _, G, dX = custom_minibatch(ref, x, grad_fn, noise, lrt, oopt)
        assert torch.isfinite(G).all() and (G[:, 2, :] == 0).all()
        assert not torch.equal(ref.vb[0].means, m0)
        outs.append((ref.vb[0].means.clone(), ref.out.weight.clone() if hasattr(ref.out, "weight") else None, dX))
    for a, b in zip(*outs):
        if a is not None:
            torch.testing.assert_close(a, b, rtol=1e-12, atol=1e-15)


def test_set_criterion_rejects_unknown_names():
    import vbnn_b200
    from vbnn_b200 import _lib as L
    net = vbnn_b200.MLP()
    with pytest.raises(vbnn_b200.VbnnError) as e:
        net.set_criterion("huber")
    assert e.value.code == L.E_INVALID
    assert L.CRITERIA == {"class_nll": 0, "mse": 1, "gaussian_nll": 2}
