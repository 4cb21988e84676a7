"""CPU checks of the fp64 reference that the GPU tests of vbnn_mlp_predict_outputs compare against: closed forms of
every statistic, the MAP stack, and proof that the cancellation case of the GPU tests defeats a naive fp32 variance."""
import math

import numpy as np
import torch

from oracle import vbnn_oracle as O
from predict_outputs_reference import gaussian_log_density, moments, raw_stack
from predict_reference import logp_stack


def stack(T, N, C, seed, loc=0.0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return loc + scale * torch.randn(T, N, C, generator=g, dtype=torch.float64)


def cancellation_stack(T=16, N=64, K=3):
    """outputs near 1e4 with a spread near 1e-2 over the samples: the regime of test_cancellation in the GPU tests"""
    return stack(T, N, K, 11, loc=1.0e4, scale=1.0e-2)


def test_one_sample_has_zero_epistemic_variance():
    for model, C in (("raw", 5), ("gaussian", 6)):
        r = moments(stack(1, 7, C, 0), model)
        assert float(r["epistemic"].abs().max()) == 0.0
        assert torch.equal(r["mean"], stack(1, 7, C, 0)[0, :, :C // 2 if model == "gaussian" else C])


def test_one_gaussian_sample_nll_is_the_normal_log_density():
    f = stack(1, 9, 6, 1)
    y = stack(1, 9, 3, 2)[0]
    m, s = f[0, :, :3], f[0, :, 3:]
    want = -float(torch.distributions.Normal(m, torch.exp(s / 2)).log_prob(y).sum(-1).mean())
    got = moments(f, "gaussian", y)["nll"]
    assert abs(got - want) <= 1e-12 * abs(want)
    assert torch.allclose(moments(f, "gaussian")["aleatoric"], torch.exp(s), rtol=1e-15, atol=0)


def test_mixture_log_likelihood_is_the_log_of_the_mean_density():
    T, N, K = 5, 8, 2
    f = stack(T, N, 2 * K, 3, scale=0.5)
    y = stack(1, N, K, 4)[0]
    dens = torch.zeros(N, dtype=torch.float64)
    for t in range(T):
        dens += torch.exp(torch.distributions.Normal(f[t, :, :K], torch.exp(f[t, :, K:] / 2)).log_prob(y).sum(-1)) / T
    want = -float(torch.log(dens).mean())
    got = moments(f, "gaussian", y)["nll"]
    assert abs(got - want) <= 1e-12 * abs(want)
    # the joint per-row mixture, not a product of per-column mixtures
    per_col = 0.0
    for k in range(K):
        d = torch.exp(torch.distributions.Normal(f[:, :, k], torch.exp(f[:, :, K + k] / 2)).log_prob(y[:, k])).mean(0)
        per_col += float(-torch.log(d).mean())
    assert abs(per_col - want) > 1e-3


def test_rmse_mean_and_epistemic_definitions():
    f = stack(6, 10, 4, 5)
    y = stack(1, 10, 4, 6)[0]
    r = moments(f, "raw", y)
    mean = f.mean(0)
    assert torch.allclose(r["mean"], mean, rtol=1e-15, atol=1e-15)
    assert torch.allclose(r["epistemic"], f.var(0, unbiased=False), rtol=1e-12, atol=0)
    assert abs(r["rmse"] - math.sqrt(float(((y - mean) ** 2).sum()) / 40)) <= 1e-14
    assert r["aleatoric"] is None and r["nll"] is None


def test_degenerate_log_variances_stay_finite():
    # y == m exactly, s = -100 and +100: e^{-s} or e^{s} overflows fp32, the log density does not
    N, K = 4, 2
    m = stack(1, N, K, 7)[0]
    for sv in (-100.0, 100.0):
        f = torch.cat([m, torch.full((N, K), sv, dtype=torch.float64)], -1).unsqueeze(0)
        r = moments(f, "gaussian", m)
        want = 0.5 * (math.log(2 * math.pi) + sv) * K
        assert math.isfinite(r["nll"]) and abs(r["nll"] - want) <= 1e-12 * abs(want)
        ll = gaussian_log_density(m.float(), m.float(), torch.full((N, K), sv))
        assert bool(torch.isfinite(ll).all())                              # also in fp32


def test_naive_fp32_variance_fails_on_the_cancellation_case():
    f = cancellation_stack()
    want = moments(f)["epistemic"]
    x = f.float()
    T = x.shape[0]
    s1 = torch.zeros_like(x[0]); s2 = torch.zeros_like(x[0])
    for t in range(T):                                                      # sequential fp32 sums, as a kernel would
        s1 = s1 + x[t]; s2 = s2 + x[t] * x[t]
    naive = (s2 / T - (s1 / T) ** 2).double()
    assert float(((naive - want).abs() / want).max()) > 0.1
    # sums of deviations from the first sample, in fp32, meet the 1e-4 bar of the GPU tests
    f0 = x[0]
    a = torch.zeros_like(f0); b = torch.zeros_like(f0)
    for t in range(1, T):
        d = x[t] - f0
        a = a + d; b = b + d * d
    shifted = ((b - a * (a / T)) / T).double()
    exact = moments(x.double())["epistemic"]                                # of the fp32 samples themselves
    assert float(((shifted - exact).abs() / exact).max()) <= 1e-4


def test_raw_stack_is_the_pre_logsoftmax_of_logp_stack():
    over = dict(input_size=12, hidden=[10, 8], classes=[str(i) for i in range(5)], S=1, B=10.0, mu_init=1,
                var_init=0.01, testSamples=3, log=False)
    rng = np.random.RandomState(4)
    X = torch.from_numpy(rng.randn(9, 12))
    eps = [[torch.from_numpy(rng.randn(10, 12)), torch.from_numpy(rng.randn(8, 10))] for _ in range(3)]
    a = raw_stack(O.MLPOracle(O.default_opt(**over), torch.float64, seed=3), X, eps_lists=eps)
    b = logp_stack(O.MLPOracle(O.default_opt(**over), torch.float64, seed=3), X, eps_lists=eps)
    assert a.shape == (3, 9, 5)
    assert torch.allclose(O.log_softmax(a.reshape(-1, 5)).reshape(3, 9, 5), b, rtol=0, atol=1e-12)
    # MAP under n_samples = 0
    a = raw_stack(O.MLPOracle(O.default_opt(**over), torch.float64, seed=3), X, n_samples=0)
    b = logp_stack(O.MLPOracle(O.default_opt(**over), torch.float64, seed=3), X, n_samples=0)
    assert a.shape == (1, 9, 5)
    assert torch.allclose(O.log_softmax(a[0]), b[0], rtol=0, atol=1e-12)
