"""fp64 reference of the prior kinds of vbnn_layer_set_prior, built on the CPU oracle's VBLinearOracle.

The reference's KL algebra (VBLinear.lua:91, 96-97, 100-101) is written in terms of mu_hat and var_hat; the oracle's
compute_mugrads / compute_vargrads already read them from the layer, so only where they come from changes:
compute_prior() sets them from the prior instead of re-estimating var_hat, and calc_lc() accepts a per-weight var_hat.

set_prior(layer, kind, ...) turns an oracle layer into a PriorVBLinearOracle in place:
  "empirical"   the oracle's own compute_prior / calc_lc (mu_hat = 0, var_hat = mean(sigma^2 + mu^2));
  "fixed"       mu_hat = mean, var_hat = var (scalars);
  "per_weight"  mu_hat = prior_means, var_hat = exp(prior_lvars) ([O x I]); by default a copy of the layer's current
                means / lvars, as the device's snapshot."""
import math

import torch

from oracle.vbnn_oracle import VBLinearOracle


class PriorVBLinearOracle(VBLinearOracle):
    prior_kind = "empirical"

    def compute_prior(self):
        if self.prior_kind == "empirical":
            return super().compute_prior()
        self.vars = torch.exp(self.lvars)                                   # :78
        self.stdv = torch.sqrt(self.vars)                                   # :79
        if self.prior_kind == "fixed":
            self.mu_hat, self.var_hat = float(self.prior_mean), float(self.prior_var)
        else:
            self.mu_hat, self.var_hat = self.prior_means.clone(), torch.exp(self.prior_lvars)
        self.mu_sqe = (self.means - self.mu_hat).pow(2)                     # :82
        return self.mu_hat, self.var_hat

    def calc_lc(self, opt):
        if self.prior_kind == "empirical":
            return super().calc_lc(opt)
        vh = torch.as_tensor(self.var_hat, dtype=self.dtype)
        first = -torch.log(torch.sqrt(self.vars)) + 0.5 * torch.log(vh)                 # :100
        second = (self.mu_sqe + (self.vars - vh)) / (2 * vh)                            # :101
        return (first + second) * (1.0 / opt["B"])                                       # :102


def set_prior(layer, kind, mean=0.0, var=None, prior_means=None, prior_lvars=None):
    """Give oracle layer `layer` (a VBLinearOracle) the prior `kind`; refreshes its compute_prior caches."""
    if kind not in ("empirical", "fixed", "per_weight"):
        raise ValueError(kind)
    layer.__class__ = PriorVBLinearOracle
    layer.prior_kind = kind
    if kind == "fixed":
        if not (var is not None and math.isfinite(var) and var > 0 and math.isfinite(mean)):
            raise ValueError("fixed prior needs a finite mean and a finite var > 0")
        layer.prior_mean, layer.prior_var = float(mean), float(var)
    if kind == "per_weight":
        layer.prior_means = (layer.means if prior_means is None else torch.as_tensor(prior_means)).to(layer.dtype).clone()
        layer.prior_lvars = (layer.lvars if prior_lvars is None else torch.as_tensor(prior_lvars)).to(layer.dtype).clone()
    layer.compute_prior()
    return layer


def kl_terms(layer, opt):
    """(mlcg, vlcg): the KL gradients w.r.t. means and lvars (divided by B) under the layer's prior, without touching
    its gradient accumulators."""
    layer.compute_prior()
    mlcg = (layer.means - layer.mu_hat) / (opt["B"] * layer.var_hat)                     # :91
    vlcg = (-layer.vars.pow(-1) + 1.0 / layer.var_hat) / (2 * opt["B"]) * layer.vars    # :96-97
    return mlcg, vlcg
