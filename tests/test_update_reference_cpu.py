"""CPU checks of tests/update_reference.py, the per-element fp64 reference of the fused KL + Adam update (k_update):
  * it agrees with the oracle's VBLinear.update (optim.adam in fp64 with the exact constants) up to the fp32
    constants the device uses (beta1, 1 - beta1, 1/S, 1/(2B), the bias-correction step);
  * an fp32 emulation of k_update in its statement order, with and without FMA contraction, lands inside the
    bounds on every element, with var_hat from per-thread fp32 partial sums as the device forms them;
  * the bounds are tight enough to flag each of a set of plausible slips in the kernel (wrong ping-pong half of
    var_hat, S - 1, t instead of t + 1 in the bias correction, the other reparameterisation's vleg, EMPIRICAL KL
    terms under FIXED, one tail quad left un-updated) on at least a stated share of elements: the GPU tests
    (tests/test_gpu_update.py) can fail."""
import math

import numpy as np
import pytest
import torch

import update_reference as R
from edge_reference import violations
from oracle import vbnn_oracle as O

F = np.float32


# ---------------------------------------------------------------- an fp32 emulation of k_update
def _mad(fma, a, b, c):
    """a * b + c with one rounding (FMA) or two."""
    if fma:
        return (a.astype(np.float64) * b + c).astype(F)
    return (a * b).astype(F) + c


def partial_sums(mu, lv, nthreads):
    """The device's var_hat numerator: each of nthreads threads walks the row quads grid-stride and sums
    __expf(lv) + mu^2 in fp32, then the partials are summed in fp64.  Returns float32 var_hat."""
    O_, I = mu.shape
    Q = (I + 3) // 4
    pad = np.zeros((O_, 4 * Q), F)
    pad[:, :I] = np.exp(lv.astype(F)) + mu.astype(F) * mu.astype(F)
    quads = pad.reshape(O_ * Q, 4)
    K = -(-quads.shape[0] // nthreads)
    q = np.zeros((K * nthreads, 4), F)
    q[:quads.shape[0]] = quads
    q = q.reshape(K, nthreads, 4)
    acc = np.zeros(nthreads, F)
    for k in range(K):
        for j in range(4):
            acc = acc + q[k, :, j]
    return F(acc.astype(np.float64).sum() / mu.size)


def emulate(st, opt, prior, nthreads, fma=False, vh=None, S=None, t_used=None, lrt=None, empirical_kl=False,
            skip_quad=None):
    """k_update in fp32 numpy, statement by statement.  The keyword arguments after fma are slips to inject:
    vh (a var_hat to use instead), S (for the 1/S), t_used (the bias-correction exponent instead of t + 1), lrt (the
    reparameterisation vleg follows), empirical_kl (EMPIRICAL terms whatever the prior), skip_quad ((o, c): that
    quad's outputs are not stored)."""
    mu, lv = st["mu"].numpy().astype(F), st["lv"].numpy().astype(F)
    gw, gs = st["gW"].numpy().astype(F), st["gS"].numpy().astype(F)
    B, Sv = F(opt["B"]), int(opt["S"] if S is None else S)
    inv_S = F(1) / F(Sv)
    inv_2B = F(1) / (F(2) * B)
    b1, b2 = F(opt["beta1"]), F(opt["beta2"])
    omb1, omb2 = F(1) - b1, F(1) - b2
    eps = F(opt["eps"])
    t = int(st["t"]) + 1 if t_used is None else t_used
    bc1, bc2 = 1.0 - float(b1) ** t, 1.0 - float(b2) ** t
    step_mu = F(float(F(opt["lr_mu"])) * math.sqrt(bc2) / bc1)
    step_var = F(float(F(opt["lr_var"])) * math.sqrt(bc2) / bc1)
    lrt = opt["lrt"] if lrt is None else lrt
    var = np.exp(lv)
    sd = np.sqrt(var)
    mleg = gw * inv_S
    vleg = (gs * inv_S) * var if lrt else (gs * (F(0.5) * inv_S)) * sd
    if prior.kind == "empirical" or empirical_kl:
        v = partial_sums(mu, lv, nthreads) if vh is None else F(vh)
        inv_BV = F(1) / (B * v)
        inv_vh = F(1) / v
        musq = mu * mu
        mlcg = mu * inv_BV
        vlcg = _mad(fma, var, inv_vh, F(-1)) * inv_2B
        gmu = _mad(fma, mu, inv_BV, mleg)
    else:
        pm = np.full_like(mu, F(prior.mu0)) if prior.kind == "fixed" else prior.pm.numpy().astype(F)
        l0 = np.full_like(mu, F(math.log(F(prior.var0)))) if prior.kind == "fixed" else prior.pl.numpy().astype(F)
        d = mu - pm
        musq = d * d
        e = np.exp(F(-0.5) * l0)
        mlcg = np.where(d == 0, F(0), ((d * (F(2) * inv_2B)) * e) * e).astype(F)
        vlcg = (np.exp(lv - l0) - F(1)) * inv_2B
        gmu = _mad(fma, gw, inv_S, mlcg)
    gvar = vleg + vlcg
    mm = _mad(fma, F(b1), st["m_mu"].numpy().astype(F), omb1 * gmu)
    vm = _mad(fma, F(b2), st["v_mu"].numpy().astype(F), (omb2 * gmu) * gmu)
    dmu = (-step_mu * mm) / (np.sqrt(vm) + eps)
    mv = _mad(fma, F(b1), st["m_var"].numpy().astype(F), omb1 * gvar)
    vv = _mad(fma, F(b2), st["v_var"].numpy().astype(F), (omb2 * gvar) * gvar)
    dlv = (-step_var * mv) / (np.sqrt(vv) + eps)
    out = dict(mu=mu + dmu, lv=lv + dlv, m_mu=mm, v_mu=vm, m_var=mv, v_var=vv, stdv=sd, mu_sqe=musq, mleg=mleg,
               mlcg=mlcg, vleg=vleg, vlcg=vlcg, dmu=dmu, dlv=dlv)
    out["s2"] = np.exp(out["lv"])
    if skip_quad is not None:
        o, c = skip_quad
        cols = slice(4 * c, min(4 * c + 4, mu.shape[1]))
        for k, old in dict(mu=mu, lv=lv, m_mu=st["m_mu"], v_mu=st["v_mu"], m_var=st["m_var"], v_var=st["v_var"]).items():
            out[k][o, cols] = np.asarray(old, F)[o, cols]
    out["bias"] = (st["bias"].numpy().astype(F) - F(opt["lr_bias"]) * st["gB"].numpy().astype(F))
    return out


# ---------------------------------------------------------------- states
OPT = dict(B=10.0, S=3, lr_mu=1e-4, lr_var=0.05, lr_bias=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, lrt=False)


def _grads(rng, O_, I):
    """Gradients mixed in sign and over three decades of scale."""
    scale = lambda: 10.0 ** rng.uniform(-2, 1, (O_, I))
    return (torch.from_numpy(F(rng.randn(O_, I) * scale()).astype(np.float64)),
            torch.from_numpy(F(rng.randn(O_, I) * 10 * scale()).astype(np.float64)))


def advanced_state(O_, I, opt, prior, nthreads, steps=3, seed=0):
    """A state after `steps` emulated updates from zero moments (t = steps): returns (state, the state one update
    earlier).  Fresh gradients for the next update."""
    rng = np.random.RandomState(seed)
    d = lambda a: torch.from_numpy(np.asarray(a, F).astype(np.float64))
    st = dict(mu=d(rng.randn(O_, I) * 0.2), lv=d(rng.uniform(math.log(1e-3), math.log(1e-1), (O_, I))),
              m_mu=d(np.zeros((O_, I))), v_mu=d(np.zeros((O_, I))), m_var=d(np.zeros((O_, I))),
              v_var=d(np.zeros((O_, I))), bias=d(rng.randn(O_) * 0.1), t=0)
    prev = None
    for _ in range(steps + 1):
        st["gW"], st["gS"] = _grads(rng, O_, I)
        st["gB"] = d(rng.randn(O_))
        if st["t"] == steps:
            return st, prev
        prev = dict(st)
        e = emulate(st, opt, prior, nthreads)
        st = dict(st, **{k: d(e[k]) for k in ("mu", "lv", "m_mu", "v_mu", "m_var", "v_var", "bias")}, t=st["t"] + 1)
    raise AssertionError


def flagged(got, pair):
    """Share of elements outside the bound."""
    ref, bound = pair
    got = torch.as_tensor(np.asarray(got, np.float64))
    return float(((got - ref).abs() > bound).double().mean())


KEYS = ("mu", "lv", "m_mu", "v_mu", "m_var", "v_var", "bias", "s2", "stdv", "mu_sqe", "mleg", "mlcg", "vleg", "vlcg")
PRIORS = ["empirical", "fixed", "per_weight"]


def make_prior(kind, st, nthreads, O_, I, rng=None):
    if kind == "empirical":
        return R.Prior("empirical", terms=R.update_terms(O_, I, 1, nthreads))
    if kind == "fixed":
        return R.Prior("fixed", mu0=0.05, var0=0.02)
    rng = rng or np.random.RandomState(5)
    f = lambda a: torch.from_numpy(np.asarray(a, F).astype(np.float64))
    pm = f(st["mu"].numpy() + rng.randn(O_, I) * 0.05)
    pl = f(st["lv"].numpy() + rng.randn(O_, I) * 0.5)
    pm[0, 0] = st["mu"][0, 0]                     # mu == mu_hat: kl_mu is exactly 0
    return R.Prior("per_weight", pm=pm, pl=pl)


# ---------------------------------------------------------------- the reference vs the oracle
def test_reference_matches_oracle_update():
    """EMPIRICAL, both reparameterisations: the reference equals optim.adam of the oracle in fp64 to within the
    bound plus 2e-5 of each element, the fp32-constant difference: 1 - f32(0.999) = 0.001 (1 - 1.3e-5) is the
    largest (1 - f32(0.9) = 0.1 (1 + 2.4e-7); 1/S and the bias-corrected step are rounded to fp32)."""
    O_, I, nth = 6, 11, 8
    for lrt in (False, True):
        opt = dict(OPT, lrt=lrt)
        prior = R.Prior("empirical", terms=R.update_terms(O_, I, 1, nth))
        st, _ = advanced_state(O_, I, opt, prior, nth)
        ref = R.update(st, opt, prior)
        oo = dict(var_init=1e-3, mu_init=0, B=opt["B"], S=opt["S"], state=dict(learningRate=opt["lr_bias"]),
                  meanState=dict(learningRate=opt["lr_mu"]), varState=dict(learningRate=opt["lr_var"]),
                  reparam="local" if lrt else "weight")
        ol = O.VBLinearOracle(I, O_, oo)
        ol.means.copy_(st["mu"]); ol.lvars.copy_(st["lv"]); ol.bias.copy_(st["bias"])
        ol.gradWeight.copy_(st["gW"]); ol.gradSum.copy_(st["gS"]); ol.gradBias.copy_(st["gB"])
        ol.meanState.update(t=st["t"], m=st["m_mu"].clone(), v=st["v_mu"].clone())
        ol.varState.update(t=st["t"], m=st["m_var"].clone(), v=st["v_var"].clone())
        ol.update(oo)
        got = dict(mu=ol.means, lv=ol.lvars, m_mu=ol.meanState["m"], v_mu=ol.meanState["v"], m_var=ol.varState["m"],
                   v_var=ol.varState["v"], bias=ol.bias)
        for k, v in got.items():
            r, b = ref[k]
            tol = b + 2e-5 * r.abs()
            assert ((v - r).abs() <= tol).all(), (lrt, k, float((v - r).abs().max()), float(tol.max()))
        assert abs(float(ref["var_hat"][0]) - ol.var_hat) <= float(ref["var_hat"][1]), lrt


# ---------------------------------------------------------------- the emulation lands inside the bounds
CASES = [(prior, lrt, fma) for prior in PRIORS for lrt in (False, True) for fma in (False, True)]


@pytest.mark.parametrize("prior_kind,lrt,fma", CASES)
def test_emulation_inside_bounds(prior_kind, lrt, fma):
    O_, I, nth = 9, 14, 8                          # I % 4 = 2: tail quads; 4 quads per thread
    opt = dict(OPT, lrt=lrt)
    base = R.Prior("empirical", terms=R.update_terms(O_, I, 1, nth))
    st, _ = advanced_state(O_, I, opt, base, nth, seed=1)
    prior = make_prior(prior_kind, st, nth, O_, I)
    ref = R.update(st, opt, prior)
    got = emulate(st, opt, prior, nth, fma=fma)
    for k in KEYS:
        v = violations(got[k], *ref[k])
        assert v == [], (k, v)
        assert torch.isfinite(ref[k][1]).all(), k
    # ulp-level: the new means and log-variances within a few ulps of themselves
    for k in ("mu", "lv"):
        r, b = ref[k]
        assert float((b / r.abs().clamp(min=1e-30)).max()) < 8 * R.U32, (k, float((b / r.abs()).max()))
    if prior_kind == "empirical":
        vh, evh = ref["var_hat"]
        assert abs(float(partial_sums(st["mu"].numpy(), st["lv"].numpy(), nth)) - float(vh)) <= float(evh)


def test_stats_inside_bounds():
    """The 14 diagnostics restated from the emulated update, as the layer forms them from fp64 sums."""
    O_, I, nth = 9, 14, 8
    prior = R.Prior("empirical", terms=R.update_terms(O_, I, 1, nth))
    st, _ = advanced_state(O_, I, OPT, prior, nth, seed=2)
    ref = R.update(st, OPT, prior)
    e = emulate(st, OPT, prior, nth)
    mu, lv, s2 = e["mu"].astype(np.float64), e["lv"].astype(np.float64), e["s2"].astype(np.float64)
    mu0, lv0 = st["mu"].numpy(), st["lv"].numpy()
    nl, nm, n = np.linalg.norm(lv), np.linalg.norm(mu), mu.size
    nrm = lambda k: np.linalg.norm(e[k].astype(np.float64))
    mean = mu.sum() / n
    got = dict(vlc_grad=nrm("vlcg") / nl, vle_grad=nrm("vleg") / nl, mlc_grad=nrm("mlcg") / nm,
               mle_grad=nrm("mleg") / nm, min_variance=s2.min(), max_variance=s2.max(), mean_variance=s2.sum() / n,
               var_hat=partial_sums(mu0, lv0, nth), mean_means=mean,
               std_means=math.sqrt(max(0.0, ((mu * mu).sum() - n * mean * mean) / (n - 1))),
               min_means=mu.min(), max_means=mu.max(),
               mu_normratio=nrm("dmu") / nm, var_normratio=nrm("dlv") / nl)
    for k, (r, b) in R.stats(ref, "empirical").items():
        g = float(F(got[k]))
        assert abs(g - r) <= b, (k, g, r, b)


# ---------------------------------------------------------------- sensitivity: the slips the GPU tests must catch
# (name, prior, slip, the output checked, the share of its elements that must be flagged: measured 0.98-1.0 for the
# first five on this state, and both elements of the skipped tail quad (I % 4 = 2) for the last)
def _slips(st, prev, opt, nth, O_, I):
    Q = (I + 3) // 4
    return [
        ("var_hat of the other ping-pong half", "empirical", dict(vh=partial_sums(prev["mu"].numpy(), prev["lv"].numpy(), nth)), "m_mu", 0.95),
        ("S - 1 instead of S", "empirical", dict(S=opt["S"] - 1), "m_mu", 0.99),
        ("t instead of t + 1 in the bias correction", "empirical", dict(t_used=st["t"]), "mu", 0.99),
        ("the other reparameterisation's vleg", "empirical", dict(lrt=not opt["lrt"]), "m_var", 0.99),
        ("EMPIRICAL KL terms where FIXED was asked", "fixed", dict(empirical_kl=True), "m_mu", 0.99),
        ("one tail quad left un-updated", "empirical", dict(skip_quad=(O_ - 1, Q - 1)), "mu", 2.0 / (O_ * I)),
    ]


@pytest.mark.parametrize("lrt", [False, True])
def test_bounds_flag_each_slip(lrt):
    O_, I, nth = 9, 14, 8
    opt = dict(OPT, lrt=lrt)
    base = R.Prior("empirical", terms=R.update_terms(O_, I, 1, nth))
    st, prev = advanced_state(O_, I, opt, base, nth, steps=4, seed=3)
    assert st["t"] >= 3 and float(st["v_mu"].abs().min()) > 0
    for name, kind, kw, key, share in _slips(st, prev, opt, nth, O_, I):
        prior = make_prior(kind, st, nth, O_, I)
        ref = R.update(st, opt, prior)
        assert violations(emulate(st, opt, prior, nth)[key], *ref[key]) == [], name
        got = emulate(st, opt, prior, nth, **kw)[key]
        f = flagged(got, ref[key])
        assert f >= share, (name, key, f, share)
