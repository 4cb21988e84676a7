"""fp64 reference of vbnn_mlp_predict_outputs, built on the CPU oracle's forward pass (oracle/vbnn_oracle.py).

raw_stack() draws the [T x N x C] pre-LogSoftMax outputs of an MLPOracle as predict_reference.logp_stack draws its
samples (same noise injection, MAP under n_samples = 0); moments() computes every statistic of the call from such a
stack: mean, epistemic and aleatoric variance, the Gaussian mixture's NLL and the RMSE."""
import math

import torch

from custom_loss_reference import forward


def raw_stack(ref, inputs, eps_lists=None, zeta_lists=None, n_samples=None):
    """[T x N x C] raw outputs of T forward passes of MLPOracle `ref` (n_samples = 0: one MAP pass; default: 0 under
    quicktest, else testSamples)."""
    if n_samples is None:
        n_samples = 0 if ref.opt.get("quicktest") else ref.opt["testSamples"]
    x = torch.as_tensor(inputs)
    x = ref.q(x.reshape(x.shape[0], -1).to(ref.dtype))                  # nn.Reshape, as MLPOracle.run
    if n_samples == 0:
        for lyr in ref.vb_all:
            lyr.clamp_to_map()
            lyr._map = True
        y = forward(ref, x)[1].clone()
        for lyr in ref.vb_all:
            lyr._map = False
        return y.unsqueeze(0)
    out = []
    for t in range(n_samples):
        ref.sample(None if eps_lists is None else eps_lists[t])
        out.append(forward(ref, x, None if zeta_lists is None else zeta_lists[t])[1].clone())
    return torch.stack(out)


def gaussian_log_density(y, m, s):
    """sum over the last axis of log N(y; m, e^s), in the log domain: -1/2 (log 2 pi + s + (y - m)^2 e^{-s})."""
    d = y - m
    q = torch.where(d == 0, torch.zeros_like(d), d * torch.exp(-0.5 * s))
    return (-0.5 * (math.log(2 * math.pi) + s + q * q)).sum(-1)


def moments(stack, model="raw", targets=None):
    """stack [T x N x C] (fp64) -> dict of mean / epistemic [N x K], aleatoric [N x K] (gaussian, else None), and with
    targets [N x K]: nll (gaussian, else None) and rmse, as floats."""
    f = torch.as_tensor(stack).to(torch.float64)
    T, N, C = f.shape
    gaussian = model == "gaussian"
    K = C // 2 if gaussian else C
    m = f[..., :K]
    mean = m.mean(0)
    out = dict(mean=mean, epistemic=((m - mean) ** 2).mean(0), aleatoric=None, nll=None, rmse=None)
    if gaussian:
        s = f[..., K:]
        out["aleatoric"] = torch.exp(s).mean(0)
    if targets is not None:
        y = torch.as_tensor(targets).to(torch.float64).reshape(N, K)
        out["rmse"] = float(torch.sqrt(((y - mean) ** 2).mean()))
        if gaussian:
            ll = gaussian_log_density(y.unsqueeze(0), m, s)                # [T x N]: the joint density of a row
            out["nll"] = float(-(torch.logsumexp(ll, 0) - math.log(T)).mean())
    return out
