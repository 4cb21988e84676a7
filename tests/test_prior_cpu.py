"""The fp64 prior reference (tests/prior_reference.py) against the oracle and against its own calc_lc."""
import math

import numpy as np
import pytest
import torch

from oracle import vbnn_oracle as O
from prior_reference import kl_terms, set_prior


def make_layer(seed=0, I=7, O_=5, B=30.0, strict=True):
    opt = O.default_opt(input_size=I, hidden=[O_], B=B, S=3, mu_init=1, var_init=0.01, strict_reference=strict)
    rng = np.random.RandomState(seed)
    lyr = O.VBLinearOracle(I, O_, opt, torch.float64, np.random.RandomState(3))
    lyr.means.copy_(torch.from_numpy(rng.randn(O_, I) * 0.3))
    lyr.lvars.copy_(torch.from_numpy(rng.uniform(math.log(1e-4), math.log(1e-1), (O_, I))))
    lyr.compute_prior()
    return lyr, opt, rng


def feed_grads(lyr, rng):
    lyr.gradWeight.copy_(torch.from_numpy(rng.randn(lyr.O, lyr.I)))
    lyr.gradSum.copy_(torch.from_numpy(rng.randn(lyr.O, lyr.I)))
    lyr.gradBias.copy_(torch.from_numpy(rng.randn(lyr.O)))


@pytest.mark.parametrize("strict", [True, False])
def test_empirical_reference_equals_the_oracle(strict):
    a, opt, rng_a = make_layer(strict=strict)
    b, _, rng_b = make_layer(strict=strict)
    set_prior(b, "empirical")
    for _ in range(3):
        feed_grads(a, rng_a); feed_grads(b, rng_b)
        a.update(opt); b.update(opt)
        assert torch.equal(a.means, b.means) and torch.equal(a.lvars, b.lvars)
        assert a.var_hat == b.var_hat and a.mu_hat == b.mu_hat == 0.0
    assert torch.equal(a.calc_lc(opt), b.calc_lc(opt))


def fd_grads(lyr, opt, h=1e-5):
    """central differences of sum calc_lc w.r.t. each mean and each log-variance (no re-estimate of the prior)."""
    def total():
        lyr.compute_prior()
        return float(lyr.calc_lc(opt).sum())
    out = []
    for t in (lyr.means, lyr.lvars):
        g = torch.zeros_like(t)
        for idx in np.ndindex(*t.shape):
            x0 = float(t[idx])
            t[idx] = x0 + h; fp = total()
            t[idx] = x0 - h; fm = total()
            t[idx] = x0
            g[idx] = (fp - fm) / (2 * h)
        out.append(g)
    lyr.compute_prior()
    return out


@pytest.mark.parametrize("kind", ["fixed", "per_weight"])
def test_kl_gradients_are_the_derivative_of_calc_lc(kind):
    lyr, opt, rng = make_layer(seed=1, B=7.0)
    if kind == "fixed":
        set_prior(lyr, "fixed", mean=0.15, var=0.04)
    else:
        set_prior(lyr, "per_weight", prior_means=rng.randn(lyr.O, lyr.I) * 0.2,
                  prior_lvars=rng.uniform(math.log(1e-3), math.log(1e-1), (lyr.O, lyr.I)))
    fd_mu, fd_lv = fd_grads(lyr, opt)
    mlcg, vlcg = kl_terms(lyr, opt)
    assert float((mlcg - fd_mu).norm() / mlcg.norm()) <= 1e-7
    assert float((vlcg - fd_lv).norm() / vlcg.norm()) <= 1e-7
    # the oracle's own compute_mugrads / compute_vargrads give the same KL terms under the reference's prior
    _, lcg = lyr.compute_mugrads(opt)
    _, vlc = lyr.compute_vargrads(opt)
    assert torch.allclose(lcg, mlcg, rtol=1e-14, atol=0) and torch.allclose(vlc, vlcg, rtol=1e-14, atol=0)


def test_fixed_at_the_empirical_values_is_the_empirical_prior():
    a, opt, _ = make_layer(seed=2)
    b, _, _ = make_layer(seed=2)
    set_prior(b, "fixed", mean=0.0, var=a.var_hat)
    assert torch.equal(kl_terms(a, opt)[0], kl_terms(b, opt)[0])
    assert torch.allclose(a.calc_lc(opt), b.calc_lc(opt), rtol=1e-13, atol=1e-16)


@pytest.mark.parametrize("strict", [True, False])
def test_snapshot_has_zero_kl_and_zero_kl_gradients(strict):
    lyr, opt, rng = make_layer(seed=3, strict=strict)
    set_prior(lyr, "per_weight")
    mlcg, vlcg = kl_terms(lyr, opt)
    assert float(mlcg.abs().max()) == 0.0 and float(vlcg.abs().max()) == 0.0
    assert float(lyr.calc_lc(opt).abs().max()) <= 1e-15
    # and an update under it moves the parameters by the data terms only
    feed_grads(lyr, rng)
    gw, gs = lyr.gradWeight.clone(), lyr.gradSum.clone()
    leg, lcg = lyr.compute_mugrads(opt)
    assert float(lcg.abs().max()) == 0.0 and torch.equal(leg, gw / opt["S"])
    _, vlc = lyr.compute_vargrads(opt)
    assert float(vlc.abs().max()) == 0.0


def test_refusals():
    lyr, _, _ = make_layer()
    for bad in (dict(var=None), dict(var=0.0), dict(var=-1.0), dict(var=float("inf")), dict(mean=float("nan"), var=1.0)):
        with pytest.raises(ValueError):
            set_prior(lyr, "fixed", **bad)
    with pytest.raises(ValueError):
        set_prior(lyr, "mixture")
