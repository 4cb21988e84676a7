"""fp64 restatement of one fused KL + Adam update (k_update, csrc/elementwise.cu) with per-element error bounds.

Input: the layer's state read back just before the update (means, log-variances, the four Adam moments, the step
counter t, the bias, gradWeight / gradSum / gradBias as the device left them), its options and its prior.  Every
value is restated in fp64 from those fp32 numbers with the device's fp32 constants and statement order, and paired
with a bound on |device - reference| built from how the device computes it (the edge_reference.py style):
  * every fp32 operation rounds once, |fl(x) - x| <= 2^-24 |x|; the bound allows a rounding after every operation,
    so it holds with or without FMA contraction.  An exact result that fp32 represents (1 - f32(beta1), 0.5 / S, mu -
    mu where equal) is not rounded.
  * __expf: edge_reference.expf_err at the argument's interval (the device is built without --use_fast_math, so
    sqrtf and divisions are IEEE and __expf is the only approximate function).
  * an error on an operand propagates exactly through the operation (absolute errors through cancellations such as
    b1 m + (1 - b1) g and var / var_hat - 1).
  * var_hat (EMPIRICAL) is the fp64 mean of __expf(lvar) + mu^2 over the pre-update state.  Its bound follows the
    partial sums it came from: each thread sums `terms` values in fp32 before the fp64 reduction -- 4 ceil(quads /
    (grid TPB)) when the previous update wrote them, 256 (chunks of 64 quads) when k_prior_partials did (creation,
    vbnn_layer_set, vbnn_layer_set_t, vbnn_layer_compute_prior).
All tensors are fp64 torch tensors holding fp32 values, on any device."""
import math

import numpy as np
import torch

from edge_reference import ETA, FLT_MIN, INF, U32, expf_err, mul_err

KMAX_PARTIALS = 1184       # kMaxPartials (csrc/kernels.h): 148 SMs x 8 blocks
NUM_SMS = 148
TPB = 256                  # k_update's block size; 128 for the co-resident variant
PRIOR_CHUNK_TERMS = 256    # k_prior_partials: fp32 chunks of 64 quads


def f32(x):
    """The fp32 value of a Python / numpy scalar, as a float."""
    return float(np.float32(x))


def update_grid(O, I, bps=4):
    """update_grid(O, I) of csrc/elementwise.cu under the upd_bps knob at the layer's creation."""
    quads = O * ((I + 3) // 4)
    blocks = max(1, (quads + 255) // 256)
    return min(blocks, NUM_SMS * bps, KMAX_PARTIALS)


def update_terms(O, I, grid, tpb=TPB):
    """fp32 terms each thread of a k_update launch sums into its partial of the next var_hat."""
    quads = O * ((I + 3) // 4)
    return 4 * -(-quads // (grid * tpb))


class V:
    """A value (fp64 tensor) and a bound on the device's distance from it."""

    def __init__(self, v, e=None):
        self.v = v
        self.e = torch.zeros_like(v) if e is None else e

    def __neg__(self):
        return V(-self.v, self.e)

    def __add__(self, o):
        o = _v(o, self.v)
        return _rnd(self.v + o.v, self.e + o.e)

    def __sub__(self, o):
        o = _v(o, self.v)
        return _rnd(self.v - o.v, self.e + o.e)

    def __mul__(self, o):
        o = _v(o, self.v)
        return _rnd(self.v * o.v, mul_err(self.v, self.e, o.v, o.e))

    def __truediv__(self, o):
        o = _v(o, self.v)
        v = self.v / o.v
        room = o.v.abs() - o.e
        e = torch.where(room > 0, (self.e + v.abs() * o.e) / room.clamp(min=1e-300), torch.full_like(v, INF))
        return _rnd(v, torch.where((self.e == 0) & (o.e == 0), torch.zeros_like(e), e))

    def pair(self):
        return self.v, self.e


def _v(x, like):
    if isinstance(x, V):
        return x
    return V(torch.full_like(like, float(x)))


def _rnd(v, e):
    """One fp32 rounding of a result whose operands carry a total error e.  Exact where the operands are exact and
    fp32 holds the result."""
    exact = (e == 0) & (v == v.float().double())
    out = e + U32 * (v.abs() + e) + ETA
    return V(v, torch.where(exact, torch.zeros_like(e), torch.nan_to_num(out, nan=INF)))


def sqrtf(a):
    v = a.v.clamp(min=0).sqrt()
    lo = (a.v - a.e).clamp(min=0).sqrt()
    e = torch.where(a.v > 0, a.e / (v + lo), a.e.sqrt())
    return _rnd(v, torch.where(a.e == 0, torch.zeros_like(e), e))


def expf(x):
    """__expf(x') for |x' - x.v| <= x.e: exp's own spread over the interval plus the intrinsic's error at its top."""
    v = torch.exp(x.v)
    top = torch.exp(x.v + x.e)
    e = v * torch.expm1(x.e) + top * (2.0 + torch.floor(1.173 * (x.v.abs() + x.e))) * 2.0 ** -23
    e = torch.where(top < FLT_MIN, top, e)       # flushed to 0 or subnormal: anything in [0, top]
    return V(v, torch.nan_to_num(e, nan=INF))


def var_hat(mu, lv, terms):
    """The EMPIRICAL prior's var_hat as the device forms it from partial sums of `terms` fp32 values per thread:
    (value, bound), 0-d tensors."""
    W = mu.numel()
    s = torch.exp(lv) + mu * mu
    tot = s.sum()
    # per element: __expf's error and the add / square roundings; per thread: a recursive fp32 sum of `terms` values
    e_terms = expf_err(lv).sum() + 2 * U32 * tot
    e = (e_terms + terms * U32 * (tot + e_terms)) / W + 1e-12 * tot / W      # + the fp64 reduction
    v = tot / W
    return v, e + U32 * (v + e) + ETA                                       # (float)(r / W)


class Prior:
    """kind "empirical" (terms: see var_hat), "fixed" (mu0, var0) or "per_weight" (pm, pl as read back)."""

    def __init__(self, kind, terms=None, mu0=0.0, var0=None, pm=None, pl=None):
        self.kind, self.terms, self.mu0, self.var0, self.pm, self.pl = kind, terms, mu0, var0, pm, pl


def _kl_terms(mu, lv, prior, inv_2B):
    """kl_mu / kl_lvar of FIXED and PER_WEIGHT: (d, klm, klv) as V."""
    if prior.kind == "fixed":
        pm = torch.full_like(mu, f32(prior.mu0))
        l0v = math.log(f32(prior.var0))
        l0 = V(torch.full_like(mu, l0v), torch.full_like(mu, 2 * U32 * abs(l0v)))   # host logf: within 1 ulp
    else:
        pm, l0 = prior.pm, V(prior.pl)
    d = V(mu) - V(pm)
    eh = expf(l0 * -0.5)
    klm = d * (2.0 * inv_2B) * eh * eh
    zero = (d.v == 0) & (d.e == 0)
    klm = V(torch.where(zero, torch.zeros_like(klm.v), klm.v), torch.where(zero, torch.zeros_like(klm.e), klm.e))
    klv = (expf(V(lv) - l0) - 1.0) * inv_2B
    return d, klm, klv


def update(st, opt, prior):
    """One k_update from the pre-update state st (dict of mu, lv, m_mu, v_mu, m_var, v_var, gW, gS, bias, gB, t) under
    opt (dict of B, S, lr_mu, lr_var, lr_bias, beta1, beta2, eps, lrt).  Returns dict name -> (value, bound): the new
    mu, lv, m_mu, v_mu, m_var, v_var, bias, s2 (__expf of the new lv), the caches stdv / mu_sqe, the four gradient
    terms mleg / mlcg / vleg / vlcg, dmu / dlv, and var_hat as used (EMPIRICAL; 0-d)."""
    mu, lv = st["mu"], st["lv"]
    B, S = f32(opt["B"]), int(opt["S"])
    inv_S = f32(np.float32(1) / np.float32(S))
    inv_2B = f32(np.float32(1) / (np.float32(2) * np.float32(B)))
    b1, b2 = f32(opt["beta1"]), f32(opt["beta2"])
    omb1, omb2 = f32(np.float32(1) - np.float32(b1)), f32(np.float32(1) - np.float32(b2))
    eps = f32(opt["eps"])
    t = int(st["t"]) + 1                                                    # state.t = state.t + 1
    bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
    step_mu = f32(f32(opt["lr_mu"]) * math.sqrt(bc2) / bc1)
    step_var = f32(f32(opt["lr_var"]) * math.sqrt(bc2) / bc1)

    var = expf(V(lv))
    sd = sqrtf(var)
    out = {}
    mleg = V(st["gW"]) * inv_S
    if opt["lrt"]:
        vleg = V(st["gS"]) * inv_S * var
    else:
        vleg = V(st["gS"]) * (0.5 * inv_S) * sd
    if prior.kind == "empirical":
        vh, evh = var_hat(mu, lv, prior.terms)
        vhV = V(vh.expand_as(mu).clone(), evh.expand_as(mu).clone())
        inv_BV = _v(1.0, mu) / (vhV * B)
        inv_vh = _v(1.0, mu) / vhV
        musq = V(mu) * V(mu)
        mlcg = V(mu) * inv_BV
        vlcg = (var * inv_vh - 1.0) * inv_2B
        out["var_hat"] = (vh, evh)
    else:
        d, mlcg, vlcg = _kl_terms(mu, lv, prior, inv_2B)
        musq = d * d
    gmu = mleg + mlcg
    gvar = vleg + vlcg
    m_mu = V(st["m_mu"]) * b1 + gmu * omb1
    v_mu = V(st["v_mu"]) * b2 + gmu * omb2 * gmu
    # the steps: the kernel's pow() in fp64 may differ from this one in the last bit, which can move the fp32 step by an ulp
    step = lambda c: V(torch.full_like(mu, -c), torch.full_like(mu, 2 * U32 * c))
    dmu = (m_mu * step(step_mu)) / (sqrtf(v_mu) + eps)
    m_var = V(st["m_var"]) * b1 + gvar * omb1
    v_var = V(st["v_var"]) * b2 + gvar * omb2 * gvar
    dlv = (m_var * step(step_var)) / (sqrtf(v_var) + eps)
    mu_new = V(mu) + dmu
    lv_new = V(lv) + dlv
    bias = V(st["bias"]) - V(st["gB"]) * f32(opt["lr_bias"])
    for k, x in dict(mu=mu_new, lv=lv_new, m_mu=m_mu, v_mu=v_mu, m_var=m_var, v_var=v_var, bias=bias,
                     s2=expf(lv_new), stdv=sd, mu_sqe=musq, mleg=mleg, mlcg=mlcg, vleg=vleg, vlcg=vlcg,
                     dmu=dmu, dlv=dlv).items():
        out[k] = x.pair()
    return out


def sgd(w, g, lr):
    """k_sgd: w - lr g (the output layer's weight and every bias)."""
    return (V(w) - V(g) * f32(lr)).pair()


def grads(st, opt, prior, vh=None):
    """k_grads (vbnn_layer_grads): mleg, mlcg, vleg, vlcg from the state, in its own forms (divisions by S, B var_hat,
    2 S and 2 B).  vh: (value, bound) of the var_hat it reads (EMPIRICAL)."""
    mu, lv = st["mu"], st["lv"]
    B, S = f32(opt["B"]), float(int(opt["S"]))
    var = expf(V(lv))
    sd = sqrtf(var)
    mleg = V(st["gW"]) / S
    vleg = V(st["gS"]) / S * var if opt["lrt"] else V(st["gS"]) / (2.0 * S) * sd
    inv_B = f32(np.float32(1) / np.float32(B))
    inv_2B = f32(np.float32(1) / (np.float32(2) * np.float32(B)))
    if prior.kind == "empirical":
        vhV = V(vh[0].expand_as(mu).clone(), vh[1].expand_as(mu).clone())
        mlcg = V(mu) / (vhV * B)
        vlcg = (var * (_v(1.0, mu) / vhV) - 1.0) / (2.0 * B)
    else:
        _, mlcg, vlcg = _kl_terms(mu, lv, prior, inv_2B)
        # k_grads passes 1 / B itself: the same fp32 value as 2 * inv_2B (B and 2B scale by an exact power of 2)
        assert inv_B == 2.0 * inv_2B
    return dict(mleg=mleg.pair(), mlcg=mlcg.pair(), vleg=vleg.pair(), vlcg=vlcg.pair())


# ---------------------------------------------------------------- the 14 diagnostics (vbnn_stats)
STAT_FIELDS = ("vlc_grad", "vle_grad", "mlc_grad", "mle_grad", "min_variance", "max_variance", "mean_variance",
               "var_hat", "mean_means", "std_means", "min_means", "max_means", "mu_normratio", "var_normratio")


def _norm(p):
    v, e = p
    return float(v.norm()), float(e.norm()) + 1e-12 * float(v.norm())


def _ratio(a, b):
    (av, ae), (bv, be) = a, b
    if bv <= be:
        return av / bv if bv > 0 else INF, INF
    r = av / bv
    return r, (ae + r * be) / (bv - be)


def stats(out, prior_kind, var_hat0=None):
    """The 14 diagnostics of the update whose reference is `out`, each (value, bound); the device sums in fp64 and
    stores fp32.  var_hat0: the scalar the layer reports for FIXED (var0); PER_WEIGHT reports NaN."""
    nl, nm = _norm(out["lv"]), _norm(out["mu"])
    mu, emu = out["mu"]
    s2, es2 = out["s2"]
    n = mu.numel()
    mean = float(mu.mean())
    if n > 1:
        std = float(mu.std())
        estd = float(emu.norm()) / math.sqrt(n - 1) + math.sqrt(float((mu * mu).sum()) * 2.0 ** -50 / (n - 1))
    else:
        std, estd = 0.0, 0.0                                               # (s5 - n mean^2) = 0 exactly: fmax(0, NaN)
    if prior_kind == "empirical":
        vh = (float(out["var_hat"][0]), float(out["var_hat"][1]))
    elif prior_kind == "fixed":
        vh = (f32(var_hat0), 0.0)
    else:
        vh = (float("nan"), 0.0)
    raw = dict(
        vlc_grad=_ratio(_norm(out["vlcg"]), nl), vle_grad=_ratio(_norm(out["vleg"]), nl),
        mlc_grad=_ratio(_norm(out["mlcg"]), nm), mle_grad=_ratio(_norm(out["mleg"]), nm),
        min_variance=(float(s2.min()), float(es2.max())), max_variance=(float(s2.max()), float(es2.max())),
        mean_variance=(float(s2.mean()), float(es2.mean()) + 1e-12 * float(s2.abs().mean())),
        var_hat=vh, mean_means=(mean, float(emu.mean()) + 1e-12 * float(mu.abs().mean())),
        std_means=(std, estd), min_means=(float(mu.min()), float(emu.max())),
        max_means=(float(mu.max()), float(emu.max())),
        mu_normratio=_ratio(_norm(out["dmu"]), nm), var_normratio=_ratio(_norm(out["dlv"]), nl))
    res = {}
    for k in STAT_FIELDS:
        v, e = raw[k]
        res[k] = (v, e if k == "var_hat" else e + U32 * (abs(v) + e) + 2.0 ** -149)
    return res
