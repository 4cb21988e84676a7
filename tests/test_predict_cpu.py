"""CPU checks of the fp64 predictive reference that the GPU tests of vbnn_mlp_predict compare against."""
import math

import numpy as np
import torch

from oracle import vbnn_oracle as O
from predict_reference import logp_stack, nll_accuracy, oracle_predict, predictive


def random_stack(T, N, C, seed, scale=3.0):
    g = torch.Generator().manual_seed(seed)
    return O.log_softmax(scale * torch.randn(T * N, C, generator=g, dtype=torch.float64)).reshape(T, N, C)


def test_one_sample_is_that_sample():
    lp = random_stack(1, 7, 5, 0)
    p = predictive(lp)
    assert torch.allclose(p["logp"], lp[0], rtol=0, atol=1e-12)
    assert float(p["mutual_info"].abs().max()) <= 1e-12
    assert torch.allclose(p["entropy"], p["expected_entropy"], rtol=0, atol=1e-12)


def test_identical_samples_carry_no_epistemic_uncertainty():
    lp = random_stack(1, 6, 9, 1).expand(4, -1, -1)
    p = predictive(lp)
    assert float(p["mutual_info"].max()) <= 1e-12
    assert torch.allclose(p["logp"], lp[0], rtol=0, atol=1e-12)


def test_sample_order_does_not_matter():
    lp = random_stack(6, 5, 7, 2)
    a = predictive(lp)
    b = predictive(lp[torch.tensor([3, 0, 5, 1, 4, 2])])
    for k in ("logp", "entropy", "expected_entropy", "mutual_info"):
        assert torch.allclose(a[k], b[k], rtol=0, atol=1e-12), k
    assert torch.equal(a["label"], b["label"])


def test_mutual_information_is_nonnegative():
    for seed in range(5):
        p = predictive(random_stack(8, 16, 10, 10 + seed))
        assert float((p["entropy"] - p["expected_entropy"]).min()) >= -1e-12        # Jensen: H[mean] >= mean H
        assert float(p["mutual_info"].max()) > 0.0


def test_large_logit_gaps_stay_finite():
    # class 2 has logp near -300 in every sample: summing probabilities would underflow to log(0) = -inf
    x = torch.tensor([[[0.0, -10.0, -300.0]], [[0.0, -5.0, -310.0]], [[0.0, -20.0, -250.0]]], dtype=torch.float64)
    lp = O.log_softmax(x.reshape(3, 3)).reshape(3, 1, 3)
    p = predictive(lp)
    assert bool(torch.isfinite(p["logp"]).all())
    v = [float(lp[t, 0, 2]) for t in range(3)]
    m = max(v)
    hand = m + math.log(sum(math.exp(a - m) for a in v)) - math.log(3)
    assert abs(float(p["logp"][0, 2]) - hand) <= 1e-9 * abs(hand)
    nll, acc = nll_accuracy(p, torch.tensor([3.0]))
    assert math.isfinite(nll) and abs(nll + hand) <= 1e-9 * abs(hand) and acc == 0.0


def test_one_sample_predict_matches_test_nll():
    over = dict(input_size=12, hidden=[10, 8], classes=[str(i) for i in range(5)], S=1, B=10.0, mu_init=1,
                var_init=0.01, testSamples=1, log=False)
    rng = np.random.RandomState(4)
    X = torch.from_numpy(rng.randn(9, 12))
    T = torch.from_numpy(rng.randint(1, 6, 9).astype(np.float64))
    eps = [[torch.from_numpy(rng.randn(10, 12)), torch.from_numpy(rng.randn(8, 10))]]
    ref = O.MLPOracle(O.default_opt(**over), torch.float64, seed=3)
    err, acc = ref.test(X, T, eps_lists=eps)
    ref = O.MLPOracle(O.default_opt(**over), torch.float64, seed=3)
    p = oracle_predict(ref, X, T, eps_lists=eps)
    assert abs(p["nll"] - err) <= 1e-12 * abs(err)
    assert abs(p["accuracy"] - acc) <= 1e-9


def test_map_stack_is_the_quicktest_pass():
    over = dict(input_size=12, hidden=[10], classes=[str(i) for i in range(4)], S=1, B=10.0, mu_init=1,
                var_init=0.01, quicktest=True, log=False)
    rng = np.random.RandomState(5)
    X = torch.from_numpy(rng.randn(6, 12))
    T = torch.from_numpy(rng.randint(1, 5, 6).astype(np.float64))
    ref = O.MLPOracle(O.default_opt(**over), torch.float64, seed=3)
    err, _ = ref.test(X, T)
    ref = O.MLPOracle(O.default_opt(**over), torch.float64, seed=3)
    st = logp_stack(ref, X)
    assert st.shape == (1, 6, 4)
    assert abs(nll_accuracy(predictive(st), T)[0] - err) <= 1e-12 * abs(err)
