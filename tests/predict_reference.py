"""fp64 reference of vbnn_mlp_predict, built on the CPU oracle's forward pass (oracle/vbnn_oracle.py).

predictive() averages the per-sample probabilities of a [T x N x C] stack of log-probabilities; oracle_predict()
draws that stack from an MLPOracle exactly as MLPOracle.test() draws its samples (same noise injection, same
MAP pass under quicktest)."""
import math

import torch


def predictive(logp_stack):
    """[T x N x C] per-sample logp -> dict of fp64 tensors: logp (log p-bar, via logsumexp), entropy H[p-bar],
    expected_entropy mean_t H[p_t], mutual_info max(H - E, 0), label (1-based argmax of p-bar)."""
    lp = torch.as_tensor(logp_stack).to(torch.float64)
    T = lp.shape[0]
    lpb = torch.logsumexp(lp, dim=0) - math.log(T)
    H = -(torch.exp(lpb) * lpb).sum(-1)
    E = -(torch.exp(lp) * lp).sum(-1).mean(0)
    return dict(logp=lpb, entropy=H, expected_entropy=E, mutual_info=torch.clamp(H - E, min=0.0),
                label=lpb.argmax(-1) + 1)


def nll_accuracy(pred, targets):
    """mean -log p-bar(target) and % argmax p-bar == target (targets 1-based)."""
    t = torch.as_tensor(targets).long()
    n = t.shape[0]
    nll = float(-pred["logp"][torch.arange(n), t - 1].mean())
    acc = float((pred["label"] == t).double().mean() * 100.0)
    return nll, acc


def logp_stack(ref, inputs, eps_lists=None, zeta_lists=None, n_samples=None):
    """[T x N x C] LogSoftMax outputs of T forward passes of MLPOracle `ref`, sampled as ref.test() samples them
    (n_samples = 0: one MAP pass; default: 0 under quicktest, else testSamples)."""
    if n_samples is None:
        n_samples = 0 if ref.opt.get("quicktest") else ref.opt["testSamples"]
    x = torch.as_tensor(inputs)
    dummy = torch.ones(x.shape[0], dtype=torch.float64)       # run() scores its outputs; predict ignores that
    if n_samples == 0:
        for lyr in ref.vb_all:
            lyr.clamp_to_map()
            lyr._map = True
        ref.run(x, dummy, backward=False)
        for lyr in ref.vb_all:
            lyr._map = False
        return ref.outputs.unsqueeze(0).clone()
    out = []
    for t in range(n_samples):
        ref.sample(None if eps_lists is None else eps_lists[t])
        ref.run(x, dummy, None if zeta_lists is None else zeta_lists[t], backward=False)
        out.append(ref.outputs.clone())
    return torch.stack(out)


def oracle_predict(ref, inputs, targets=None, eps_lists=None, zeta_lists=None, n_samples=None):
    """predictive() of logp_stack(); with targets also "nll" and "accuracy" (else None)."""
    pred = predictive(logp_stack(ref, inputs, eps_lists, zeta_lists, n_samples))
    pred["nll"], pred["accuracy"] = nll_accuracy(pred, targets) if targets is not None else (None, None)
    return pred
