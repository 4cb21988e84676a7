"""fp64 references of the regression criteria of vbnn_mlp_set_criterion (VBNN_CRIT_MSE, VBNN_CRIT_GAUSSIAN_NLL).

loss_sum(crit, y, n_global) is the differentiable loss of the stacked outputs Y [S x N x C]: the SUM over samples of
the per-sample mean criterion, which custom_loss_reference.autograd_grad turns into the fused step's dL/dY.  A NaN
target element adds nothing; the mean still divides by n_global * K.  closed_form_grad is the same gradient written
out; emulate_fp32 restates the kernel's fp32 statements (q = (y - m) e^{-s/2}) for the finiteness checks."""
import numpy as np
import torch


def target_cols(crit, C):
    return C // 2 if crit == "gaussian_nll" else C


def terms(crit, Y, y):
    """Per-element loss terms [.., N x K] and squared errors of the means; 0 where y is NaN."""
    K = target_cols(crit, Y.shape[-1])
    m = Y[..., :K]
    mask = ~torch.isnan(y)
    yf = torch.where(mask, y, m.detach())                # d = 0 at a missing target: finite terms and gradients
    d = yf - m
    if crit == "mse":
        t = d ** 2
    else:
        s = Y[..., K:]
        t = 0.5 * (s + d ** 2 * torch.exp(-s))
    zero = torch.zeros((), dtype=Y.dtype)
    return torch.where(mask, t, zero), torch.where(mask, d.detach() ** 2, zero)


def loss_sum(crit, y, n_global=None):
    """L(Y) = sum_s l_s, l_s = 1 / (n_global K) sum_{n,k} term: torch.mse_loss / the Gaussian NLL of the issue's
    (0.5 * (s + (y - m)**2 * exp(-s))).mean() per sample on one GPU."""
    def fn(Y):
        t, _ = terms(crit, Y, y.to(Y.dtype))
        K = t.shape[-1]
        ng = Y.shape[1] if n_global is None else n_global
        return t.sum() / (ng * K)
    return fn


def scalars(crit, Y, y):
    """The fused step's {error, accuracy} pair: mean over samples of l_s and of the MSE of the means (this rank)."""
    Y = torch.as_tensor(Y, dtype=torch.float64)
    t, se = terms(crit, Y, torch.as_tensor(y, dtype=torch.float64))
    nk = t.shape[-2] * t.shape[-1]
    return float(t.sum(dim=(-1, -2)).mean() / nk), float(se.sum(dim=(-1, -2)).mean() / nk)


def closed_form_grad(crit, Y, y, n_global):
    """dl_s/dY_s in fp64 numpy, Y [.., N x C], y [N x K]."""
    Y = np.asarray(Y, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    K = target_cols(crit, Y.shape[-1])
    D = n_global * K
    miss = np.isnan(y)
    d = np.where(miss, 0.0, y - Y[..., :K])
    G = np.zeros_like(Y)
    if crit == "mse":
        G[...] = -2.0 * d / D
    else:
        s = Y[..., K:]
        with np.errstate(over="ignore", invalid="ignore"):
            es = np.exp(-s)
            G[..., :K] = np.where(d == 0, 0.0, -d * es / D)
            G[..., K:] = np.where(miss, 0.0, 0.5 * (1.0 - d * d * es) / D)
    return G


def emulate_fp32(crit, Y, y, n_global):
    """The kernel's statements in fp32 (fmaf as one rounding of the exact fp64 result): (G, sum of loss terms)."""
    f = np.float32
    Y = np.asarray(Y, dtype=f)
    y = np.asarray(y, dtype=f)
    K = target_cols(crit, Y.shape[-1])
    scale = f(1.0 / (n_global * K))
    half, two = f(0.5) * scale, f(2.0) * scale
    fma = lambda a, b, c: f(np.float64(a) * np.float64(b) + np.float64(c))
    G = np.zeros_like(Y)
    loss = np.float64(0.0)
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        for idx in np.ndindex(*Y.shape[:-1]):
            for k in range(K):
                t, m = y[idx[-1], k], Y[idx + (k,)]
                miss = np.isnan(t)
                d = f(0.0) if miss else f(t - m)
                if crit == "mse":
                    G[idx + (k,)] = -two * d
                    loss += np.float64(f(d * d))
                    continue
                s = Y[idx + (K + k,)]
                eh = f(np.exp(f(-0.5) * s))
                q = f(0.0) if d == 0 else f(d * eh)
                G[idx + (k,)] = f(0.0) if d == 0 else -f(f(q * scale) * eh)
                G[idx + (K + k,)] = f(0.0) if miss else fma(-q, f(q * half), half)
                if not miss:
                    loss += np.float64(fma(f(0.5) * q, q, f(0.5) * s))
    return G, loss
