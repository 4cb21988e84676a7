"""vbnn_layer_set_prior on the device (pytest -m gpu): the empirical default is untouched bit for bit, FIXED and
PER_WEIGHT priors match the fp64 reference (tests/prior_reference.py) fed the device-drawn noise, every update path
and the layer-level ABI obey the prior, graphs re-capture once per prior change, and checkpoints carry the prior.
Tolerances are those of test_gpu_mlp.py: fp32 <= 2e-4 after Adam, bf16 against the bf16-rounding oracle <= 5e-3."""
import ctypes as C
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import vbnn_oracle as O
from prior_reference import kl_terms, set_prior

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES, N, S = [40, 48, 36, 6], 24, 2
MU0, VAR0 = 0.05, 0.02


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def cpu(t):
    return t.detach().float().cpu().numpy()


def f32(x):
    return float(np.float32(x))


def build(ctx, precision="fp32", reparam="weight", vb_output=False, strict=True, seed=0, sizes=SIZES, n=N, s=S,
          B=30.0, operand_round=None):
    """device net + fp64 oracle with identical random parameters (as test_gpu_mlp.build_pair)."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    over = dict(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])], S=s, B=B,
                batchSize=n, testBatchSize=n, mu_init=1, var_init=0.01, reparam=reparam, strict_reference=strict,
                vb_output=vb_output, log=False)
    net = vbnn_b200.MLP(vbnn_b200.default_opt(precision=precision, **over), ctx, max_batch=n)
    oopt = O.default_opt(**over)
    ref = O.MLPOracle(oopt, torch.float64, seed=3, operand_round=operand_round)
    rng = np.random.RandomState(seed)
    for gl, ol in zip(net.model, ref.vb + [ref.out]):
        if isinstance(ol, O.VBLinearOracle):
            mu = rng.randn(ol.O, ol.I).astype(np.float32) * math.sqrt(2.0 / ol.I)
            lv = rng.uniform(math.log(1e-4), math.log(1e-2), (ol.O, ol.I)).astype(np.float32)
            ol.means.copy_(torch.from_numpy(mu.astype(np.float64)))
            ol.lvars.copy_(torch.from_numpy(lv.astype(np.float64)))
            ol.compute_prior()
            gl.set(L.BUF_MEANS, mu); gl.set(L.BUF_LVARS, lv)
            gl.compute_prior()
        else:
            w = (rng.randn(*ol.weight.shape) * math.sqrt(2.0 / ol.weight.shape[1])).astype(np.float32)
            ol.weight.copy_(torch.from_numpy(w.astype(np.float64))); ol.bias.zero_()
            gl.set(L.BUF_WEIGHT, w)
    return net, ref, oopt


def random_prior(net, seed):
    """PER_WEIGHT on every VB layer, arrays replaced by random (mu0, l0); returns {model index: (mu0, l0)} float32."""
    from vbnn_b200 import _lib as L
    rng = np.random.RandomState(seed)
    net.set_prior("per_weight")
    arrays = {}
    for k in net.vb_indices:
        m = net.model[k]
        pm = (rng.randn(m.outputSize, m.inputSize) * 0.1).astype(np.float32)
        pl = rng.uniform(math.log(1e-3), math.log(1e-1), (m.outputSize, m.inputSize)).astype(np.float32)
        m.set(L.BUF_PRIOR_MEANS, pm); m.set(L.BUF_PRIOR_LVARS, pl)
        arrays[k] = (pm, pl)
    return arrays


def data(rng, n=N, sizes=SIZES):
    X = rng.randn(n, sizes[0]); T = rng.randint(1, sizes[-1] + 1, n).astype(np.float64)
    return X, T, torch.from_numpy(X).float().cuda(), torch.from_numpy(T).float().cuda()


def batches(seed, k, n=N, sizes=SIZES):
    rng = np.random.RandomState(seed)
    return [data(rng, n, sizes)[2:] for _ in range(k)]


def assert_same_state(a, b, what=""):
    sa, sb = a.state_dict(), b.state_dict()
    assert sorted(sa) == sorted(sb), what
    for k in sa:
        if isinstance(sa[k], torch.Tensor):
            assert torch.equal(sa[k], sb[k]), (what, k)
        else:
            assert sa[k] == sb[k], (what, k)


def assert_same_results(ra, rb):
    """(error, accuracy) per minibatch: the loss sums are accumulated with float atomics, so the last bit of the error
    may differ between two runs of the same state (test_gpu_mlp.py's resume test compares them the same way)"""
    assert np.allclose(np.array(ra), np.array(rb), rtol=1e-6, atol=1e-7), (ra, rb)


def nll_sum(T):
    t = T.long() - 1
    return lambda Y: sum(F.nll_loss(F.log_softmax(Y[s], -1), t) for s in range(Y.shape[0]))


def split_step(net, X, T, G):
    """forward_train + torch ClassNLL + backward_update with the gradient in the caller's buffer G, so that the
    backward half's graph keeps its key"""
    Y = net.forward_train(X)
    leaf = Y.detach().requires_grad_(True)
    with torch.enable_grad():
        (g,) = torch.autograd.grad(nll_sum(T)(leaf), leaf)
    G.copy_(g)
    net.backward_update(G)


# ---------------------------------------------------------------- 1. the default is untouched
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_a_round_trip_back_to_the_empirical_prior_changes_nothing(ctx, precision, reparam):
    """A net that goes FIXED -> PER_WEIGHT -> EMPIRICAL after two minibatches (the switch back recomputes var_hat and
    re-captures the step graph once) and its untouched twin: parameters, Adam state and caches stay bitwise equal over
    the next three, and so do the results up to the last bit of the atomically summed error."""
    a = build(ctx, precision, reparam)[0]
    b = build(ctx, precision, reparam)[0]
    step0 = ctx.get_step()
    runs = []
    for net, switch in ((a, False), (b, True)):
        ctx.set_step(step0)
        res = []
        for it, (X, T) in enumerate(batches(1, 5)):
            if switch and it == 2:
                c0 = net.graph_captures()
                net.set_prior("fixed", MU0, VAR0)
                net.set_prior("per_weight")
                net.set_prior("empirical")
                assert net.model[0].prior == ("empirical", None, None)
            res.append(net.train_step(X, T))
            if switch and it == 2:
                assert net.graph_captures() == c0 + 1
        runs.append(res)
    assert_same_results(runs[0], runs[1])
    assert_same_state(a, b)


# ---------------------------------------------------------------- 2. parity with the reference
def apply_prior(net, ref, kind, seed=7):
    if kind == "fixed":
        net.set_prior("fixed", MU0, VAR0)
        for ol in ref.vb_all:
            set_prior(ol, "fixed", f32(MU0), f32(VAR0))
    else:
        arrays = random_prior(net, seed)
        for ol, k in zip(ref.vb_all, net.vb_indices):
            pm, pl = arrays[k]
            set_prior(ol, "per_weight", prior_means=pm.astype(np.float64), prior_lvars=pl.astype(np.float64))


def run_parity(ctx, kind, precision, reparam, vb_output, strict, steps=3):
    bf = precision == "bf16"
    net, ref, oopt = build(ctx, precision, reparam, vb_output, strict, operand_round=O.round_bf16 if bf else None)
    apply_prior(net, ref, kind)
    tol = 5e-3 if bf else 2e-4
    rng = np.random.RandomState(5)
    nvb = len(ref.vb_all)
    gidx = lambda k: k if k < len(ref.vb) else len(net.model) - 1
    for it in range(steps):
        Xn, Tn, X, T = data(rng)
        step = ctx.get_step()
        noise = [[torch.from_numpy(cpu(net.model[gidx(k)].draw_noise(step, s, rows=N)).astype(np.float64))
                  for k in range(nvb)] for s in range(S)]
        err, _ = net.train_step(X, T)
        kw = dict(zeta=noise) if reparam == "local" else dict(eps=noise)
        rerr, _ = O.train_minibatch(ref, torch.from_numpy(Xn), torch.from_numpy(Tn), oopt, **kw)
        assert abs(err - rerr) < (2e-3 if bf else 1e-4) * abs(rerr), (it, err, rerr)
        for k, ol in enumerate(ref.vb_all):
            gl = net.model[gidx(k)]
            assert rel(cpu(gl.means), ol.means.numpy()) < tol, (it, k, "means")
            assert rel(cpu(gl.lvars), ol.lvars.numpy()) < tol, (it, k, "lvars")
        if not vb_output:
            assert rel(cpu(net.model[-1].weight), ref.out.weight.numpy()) < tol
    return net, ref


@pytest.mark.parametrize("strict", [True, False])
@pytest.mark.parametrize("reparam,vb_output", [("weight", False), ("local", False), ("weight", True), ("local", True)])
@pytest.mark.parametrize("kind", ["fixed", "per_weight"])
def test_fp32_parity_with_the_reference(ctx, kind, reparam, vb_output, strict):
    run_parity(ctx, kind, "fp32", reparam, vb_output, strict)


@pytest.mark.parametrize("reparam,vb_output", [("weight", False), ("local", True)])
@pytest.mark.parametrize("kind", ["fixed", "per_weight"])
def test_bf16_parity_with_the_rounding_reference(ctx, kind, reparam, vb_output):
    run_parity(ctx, kind, "bf16", reparam, vb_output, True)


def test_the_prior_changes_the_trajectory(ctx):
    """The same minibatches under the empirical and a per-weight prior end in different parameters (B = 30, so the
    KL terms weigh): far above fp32 noise, though Adam moves each mean by at most about lr_mu = 1e-4 per step."""
    a = build(ctx)[0]
    b = build(ctx)[0]
    random_prior(b, 3)
    step0 = ctx.get_step()
    for net in (a, b):
        ctx.set_step(step0)
        for X, T in batches(2, 2):
            net.train_step(X, T)
    assert rel(cpu(a.model[0].means), cpu(b.model[0].means)) > 1e-4


# ---------------------------------------------------------------- 3-4. the layer-level ABI
def layer_pair(ctx, strict, I=37, O_=29, B=30.0, seed=11):
    import vbnn_b200
    from vbnn_b200 import _lib as L
    opt = vbnn_b200.default_opt(input_size=I, hidden=[O_], B=B, S=3, mu_init=1, var_init=0.01,
                                strict_reference=strict, log=False)
    lyr = vbnn_b200.VBLinear(I, O_, opt, ctx)
    oopt = O.default_opt(input_size=I, hidden=[O_], B=B, S=3, mu_init=1, var_init=0.01, strict_reference=strict)
    ol = O.VBLinearOracle(I, O_, oopt, torch.float64, np.random.RandomState(3))
    rng = np.random.RandomState(seed)
    mu = (rng.randn(O_, I) * 0.2).astype(np.float32)
    lv = rng.uniform(math.log(1e-4), math.log(1e-1), (O_, I)).astype(np.float32)
    lyr.set(L.BUF_MEANS, mu); lyr.set(L.BUF_LVARS, lv); lyr.compute_prior()
    ol.means.copy_(torch.from_numpy(mu.astype(np.float64))); ol.lvars.copy_(torch.from_numpy(lv.astype(np.float64)))
    ol.compute_prior()
    return lyr, ol, opt, oopt, rng


@pytest.mark.parametrize("strict", [True, False])
@pytest.mark.parametrize("kind", ["fixed", "per_weight"])
def test_layer_abi_follows_the_prior(ctx, kind, strict):
    """vbnn_layer_compute_prior's scalars, vbnn_layer_grads' KL terms, vbnn_layer_calc_lc, the vbnn_stats.var_hat rule
    and the Q6 mu_sqe cache under the prior, against the reference."""
    from vbnn_b200 import _lib as L
    lyr, ol, opt, oopt, rng = layer_pair(ctx, strict)
    if kind == "fixed":
        lyr.set_prior("fixed", MU0, VAR0)
        set_prior(ol, "fixed", f32(MU0), f32(VAR0))
        assert lyr.prior == ("fixed", f32(MU0), f32(VAR0))
    else:
        lyr.set_prior("per_weight")
        pm = (rng.randn(lyr.outputSize, lyr.inputSize) * 0.1).astype(np.float32)
        pl = rng.uniform(math.log(1e-3), math.log(1e-1), pm.shape).astype(np.float32)
        lyr.set(L.BUF_PRIOR_MEANS, pm); lyr.set(L.BUF_PRIOR_LVARS, pl)
        assert np.array_equal(cpu(lyr.prior_means), pm) and np.array_equal(lyr.get(L.BUF_PRIOR_LVARS).numpy(), pl)
        set_prior(ol, "per_weight", prior_means=pm.astype(np.float64), prior_lvars=pl.astype(np.float64))
        assert lyr.prior == ("per_weight", None, None)
    mu_hat, var_hat = lyr.compute_prior()
    if kind == "fixed":
        assert (mu_hat, var_hat) == (f32(MU0), f32(VAR0))
    else:
        assert math.isnan(mu_hat) and math.isnan(var_hat)
    mlcg_ref, vlcg_ref = kl_terms(ol, oopt)
    _, mlcg = lyr.compute_mugrads()
    _, vlcg = lyr.compute_vargrads()
    assert rel(cpu(mlcg), mlcg_ref.numpy()) < 1e-5
    assert rel(cpu(vlcg), vlcg_ref.numpy()) < 1e-5
    assert rel(cpu(lyr.calc_lc()), ol.calc_lc(oopt).numpy()) < 1e-5
    assert abs(lyr.calc_lc_sum() - float(ol.calc_lc(oopt).sum())) < 1e-5 * float(ol.calc_lc(oopt).abs().sum())
    # one update with the diagnostics: var_hat follows compute_prior's rule, the mu_sqe cache holds (mu - mu_hat)^2
    # of the parameters before the update, in the device's fp32 arithmetic
    mu_old = lyr.get(L.BUF_MEANS).numpy()
    lyr.set(L.BUF_GRAD_WEIGHT, (rng.randn(lyr.outputSize, lyr.inputSize) * 0.01).astype(np.float32))
    lyr.set(L.BUF_GRAD_SUM, (rng.randn(lyr.outputSize, lyr.inputSize) * 0.01).astype(np.float32))
    st = lyr.update(dict(opt, log=True))
    if kind == "fixed":
        assert st["var hat"] == f32(VAR0)
    else:
        assert math.isnan(st["var hat"])
    if strict:
        hat = np.float32(MU0) if kind == "fixed" else pm
        assert np.array_equal(lyr.get(L.BUF_MU_SQE).numpy(), (mu_old - hat) * (mu_old - hat))
    # back to the reference's prior: the empirical var_hat of the current parameters
    lyr.set_prior("empirical")
    assert lyr.prior == ("empirical", None, None)
    mu, lv = lyr.get(L.BUF_MEANS).double(), lyr.get(L.BUF_LVARS).double()
    _, vh = lyr.compute_prior()
    assert abs(vh - float((torch.exp(lv) + mu * mu).mean())) < 1e-5 * vh


@pytest.mark.parametrize("strict", [False, True])
def test_snapshot_is_exact(ctx, strict):
    """Right after set_prior(PER_WEIGHT) the KL terms of vbnn_layer_grads are exactly 0 and calc_lc vanishes: exactly
    from the log-variances, and within 1e-6 * O * I / B from strict_reference's sigma cache."""
    lyr, ol, opt, oopt, _ = layer_pair(ctx, strict)
    lyr.set_prior("per_weight")
    _, mlcg = lyr.compute_mugrads()
    _, vlcg = lyr.compute_vargrads()
    assert float(mlcg.abs().max()) == 0.0 and float(vlcg.abs().max()) == 0.0
    lyr.compute_prior()                               # strict_reference: calc_lc reads the caches it refreshes
    lc = lyr.calc_lc_sum()
    bound = 1e-6 * lyr.W / opt["B"]
    if strict:
        assert abs(lc) <= bound, (lc, bound)
    else:
        assert lc == 0.0 and float(lyr.calc_lc().abs().max()) == 0.0


def test_extreme_log_variances_stay_finite(ctx):
    """A snapshot of a layer whose log-variances are -90 and -100 (below ln FLT_MIN, as test_gpu_edge_values.py): the KL
    terms of vbnn_layer_grads are exactly 0 and calc_lc is exactly 0; with the sigma cache of strict_reference calc_lc
    is finite.  A FIXED prior with a subnormal var0 gives exactly 0 where mu == mu0 and no NaN anywhere (where the
    exact gradient exceeds fp32 it is inf)."""
    from vbnn_b200 import _lib as L
    for strict in (False, True):
        lyr, _, opt, _, _ = layer_pair(ctx, strict)
        lv = lyr.get(L.BUF_LVARS).numpy().copy()
        lv.flat[0::3] = -90.0
        lv.flat[1::3] = -100.0
        lyr.set(L.BUF_LVARS, lv)
        lyr.set_prior("per_weight")
        lyr.compute_prior()
        _, mlcg = lyr.compute_mugrads()
        _, vlcg = lyr.compute_vargrads()
        assert float(mlcg.abs().max()) == 0.0 and float(vlcg.abs().max()) == 0.0, strict
        lc = cpu(lyr.calc_lc())
        assert np.isfinite(lc).all(), strict
        if not strict:
            assert float(np.abs(lc).max()) == 0.0
        # FIXED with a subnormal variance
        mu = lyr.get(L.BUF_MEANS).numpy().copy()
        mu.flat[0::2] = np.float32(MU0)
        lyr.set(L.BUF_MEANS, mu)
        lyr.set(L.BUF_LVARS, np.full(mu.shape, -90.0, np.float32))
        lyr.set_prior("fixed", MU0, 1e-40)
        lyr.compute_prior()
        _, mlcg = lyr.compute_mugrads()
        _, vlcg = lyr.compute_vargrads()
        m, v = cpu(mlcg), cpu(vlcg)
        assert (m.flat[0::2] == 0).all() and not np.isnan(m).any() and np.isfinite(v).all(), strict
        assert not np.isnan(cpu(lyr.calc_lc())).any(), strict


@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_fused_step_after_a_snapshot_at_extreme_log_variances(ctx, reparam):
    """One fused minibatch after snapshotting a net whose first layer holds log-variances of -90 and -100: the result,
    parameters and Adam state stay finite, and the snapshot's KL terms moved nothing beyond the data terms."""
    from vbnn_b200 import _lib as L
    net = build(ctx, reparam=reparam)[0]
    m = net.model[0]
    lv = m.get(L.BUF_LVARS).numpy().copy()
    lv.flat[0::3] = -90.0
    lv.flat[1::3] = -100.0
    m.set(L.BUF_LVARS, lv)
    net.set_prior("per_weight")
    X, T = batches(18, 1)[0]
    err, acc = net.train_step(X, T)
    assert math.isfinite(err) and math.isfinite(acc)
    for k, v in net.state_dict().items():
        if isinstance(v, torch.Tensor):
            assert torch.isfinite(v).all(), k


# ---------------------------------------------------------------- 5. FIXED == PER_WEIGHT filled with its scalars
def test_fixed_equals_per_weight_filled_with_the_same_prior(ctx):
    from vbnn_b200 import _lib as L
    a = build(ctx)[0]
    b = build(ctx)[0]
    a.set_prior("fixed", MU0, VAR0)
    b.set_prior("per_weight")
    for k in b.vb_indices:
        m = b.model[k]
        m.set(L.BUF_PRIOR_MEANS, np.full((m.outputSize, m.inputSize), MU0, np.float32))
        m.set(L.BUF_PRIOR_LVARS, np.full((m.outputSize, m.inputSize), math.log(f32(VAR0)), np.float32))
    step0 = ctx.get_step()
    for net in (a, b):
        ctx.set_step(step0)
        for X, T in batches(4, 3):
            net.train_step(X, T)
    for k in a.vb_indices:
        assert rel(cpu(b.model[k].means), cpu(a.model[k].means)) <= 1e-5, k
        assert rel(cpu(b.model[k].lvars), cpu(a.model[k].lvars)) <= 1e-5, k


# ---------------------------------------------------------------- 6. every update path
@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_every_update_path_obeys_the_prior(ctx, reparam):
    """One minibatch under the same PER_WEIGHT prior through vbnn_mlp_step, _step_grad_input and submit_host leaves
    bitwise-equal state; forward_train + torch ClassNLL + backward_update agrees within 1e-6 (torch's LogSoftMax
    against k_loss's, as in test_gpu_custom_loss.py)."""
    nets = [build(ctx, reparam=reparam)[0] for _ in range(4)]
    for net in nets:
        random_prior(net, 21)
    rng = np.random.RandomState(8)
    Xn, Tn, X, T = data(rng)
    step0 = ctx.get_step()
    ctx.set_step(step0); nets[0].train_step(X, T)
    ctx.set_step(step0); nets[1].train_step(X, T, grad_input=torch.empty(N, SIZES[0], device="cuda"))
    ctx.set_step(step0); nets[2].submit_host(torch.from_numpy(Xn).float(), torch.from_numpy(Tn).float())
    nets[2].collect()
    ctx.set_step(step0); nets[3].train_step_loss(X, nll_sum(T))
    torch.cuda.synchronize()
    assert_same_state(nets[0], nets[1], "step_grad_input")
    assert_same_state(nets[0], nets[2], "submit_host")
    s0, s3 = nets[0].state_dict(), nets[3].state_dict()
    for k in s0:
        if isinstance(s0[k], torch.Tensor):
            assert rel(s3[k], s0[k]) <= 1e-6, k


# ---------------------------------------------------------------- 7. graphs
def test_graphs_recapture_once_per_prior_change(ctx):
    net = build(ctx)[0]
    random_prior(net, 5)
    X, T = batches(6, 1)[0]
    G = torch.empty(S, N, SIZES[-1], device="cuda")
    for _ in range(2):
        net.train_step(X, T)
        split_step(net, X, T, G)
    c0 = net.graph_captures()
    for _ in range(2):                                # replays: no capture
        net.train_step(X, T)
        split_step(net, X, T, G)
    assert net.graph_captures() == c0
    net.set_prior("fixed", MU0, VAR0)
    net.train_step(X, T)
    assert net.graph_captures() == c0 + 1
    split_step(net, X, T, G)
    assert net.graph_captures() == c0 + 3             # the forward and the backward half
    for _ in range(2):
        net.train_step(X, T)
        split_step(net, X, T, G)
    assert net.graph_captures() == c0 + 3
    random_prior(net, 6)                              # set_prior + array edits
    net.train_step(X, T)
    assert net.graph_captures() == c0 + 4
    from vbnn_b200 import _lib as L
    m = net.model[0]
    m.set(L.BUF_PRIOR_MEANS, np.zeros((m.outputSize, m.inputSize), np.float32))
    m.prior_lvars.fill_(-3.0)
    net.train_step(X, T)
    assert net.graph_captures() == c0 + 4


def test_graph_replay_equals_no_graph(ctx):
    from vbnn_b200 import _lib as L
    a = build(ctx)[0]
    L.knob("no_graph", 1)
    try:
        b = build(ctx)[0]
    finally:
        L.knob("no_graph")
    step0 = ctx.get_step()
    for net in (a, b):
        ctx.set_step(step0)
        random_prior(net, 9)
        for it, (X, T) in enumerate(batches(10, 5)):
            if it == 3:
                net.set_prior("fixed", MU0, VAR0)
            net.train_step(X, T)
    assert b.graph_captures() == 0 and a.graph_captures() > 0
    assert_same_state(a, b)


def test_array_edit_between_steps_equals_a_fresh_net(ctx):
    """An edit through vbnn_layer_set between two replays of a captured step takes effect at the next update, as in a
    fresh net loaded with the same state and arrays."""
    from vbnn_b200 import _lib as L
    a = build(ctx)[0]
    random_prior(a, 12)
    data_ = batches(13, 4)
    for X, T in data_[:3]:
        a.train_step(X, T)                            # eager, capture, replay
    rng = np.random.RandomState(14)
    edits = {}
    for k in a.vb_indices:
        m = a.model[k]
        edits[k] = ((rng.randn(m.outputSize, m.inputSize) * 0.1).astype(np.float32),
                    rng.uniform(-6.0, -2.0, (m.outputSize, m.inputSize)).astype(np.float32))
        m.set(L.BUF_PRIOR_MEANS, edits[k][0]); m.set(L.BUF_PRIOR_LVARS, edits[k][1])
    sd = a.state_dict()
    b = build(ctx, seed=99)[0]
    b.load_state_dict(sd)
    for k in b.vb_indices:
        assert np.array_equal(b.model[k].get(L.BUF_PRIOR_MEANS).numpy(), edits[k][0])
    step0 = ctx.get_step()
    X, T = data_[3]
    a.train_step(X, T)                                # replay
    ctx.set_step(step0)
    b.train_step(X, T)                                # eager
    assert_same_state(a, b)


# ---------------------------------------------------------------- 8. refusals
def test_refusals(ctx):
    import vbnn_b200
    from vbnn_b200 import _lib as L
    net = build(ctx)[0]
    lib = L.lib()
    out = net.model[-1]
    with pytest.raises(L.VbnnError) as e:
        out.set_prior("fixed", 0.0, 1.0)                          # plain nn.Linear output layer
    assert e.value.code == L.E_INVALID
    h = net.model[0].handle
    for kind, mu0, var0 in ((3, 0.0, 1.0), (-1, 0.0, 1.0), (1, float("nan"), 1.0), (1, float("inf"), 1.0),
                            (1, 0.0, 0.0), (1, 0.0, -1.0), (1, 0.0, float("inf")), (1, 0.0, float("nan"))):
        assert lib.vbnn_layer_set_prior(h, kind, C.c_float(mu0), C.c_float(var0)) == L.E_INVALID, (kind, mu0, var0)
    assert net.model[0].prior == ("empirical", None, None)       # refused calls change nothing
    with pytest.raises(L.VbnnError) as e:
        net.model[0].set_prior("fixed", 0.0)                      # no var
    assert e.value.code == L.E_INVALID
    with pytest.raises(L.VbnnError):
        net.model[0].set_prior("mixture")
    # the PRIOR buffers exist under PER_WEIGHT only
    for kind in ("empirical", "fixed"):
        net.set_prior(kind, MU0, VAR0)
        for which in (L.BUF_PRIOR_MEANS, L.BUF_PRIOR_LVARS):
            p, n = C.c_void_p(), C.c_size_t()
            assert lib.vbnn_layer_device_ptr(h, which, C.byref(p), C.byref(n)) == L.E_STATE
            buf = np.zeros(net.model[0].W, np.float32)
            assert lib.vbnn_layer_get(h, which, C.c_void_p(buf.ctypes.data)) == L.E_STATE
            assert lib.vbnn_layer_set(h, which, C.c_void_p(buf.ctypes.data)) == L.E_STATE
    # an open split step
    X, T = batches(15, 1)[0]
    net.forward_train(X)
    assert lib.vbnn_layer_set_prior(h, L.PRIOR_PER_WEIGHT, C.c_float(0), C.c_float(0)) == L.E_STATE
    net.resetGradients()
    net.set_prior("per_weight")
    # the arrays stay allocated across kind changes: a pointer handed out earlier stays valid
    p0, n = C.c_void_p(), C.c_size_t()
    assert lib.vbnn_layer_device_ptr(h, L.BUF_PRIOR_MEANS, C.byref(p0), C.byref(n)) == L.VBNN_OK
    net.set_prior("fixed", MU0, VAR0)
    net.set_prior("per_weight")
    p1 = C.c_void_p()
    assert lib.vbnn_layer_device_ptr(h, L.BUF_PRIOR_MEANS, C.byref(p1), C.byref(n)) == L.VBNN_OK
    assert p0.value == p1.value
    assert torch.equal(net.model[0].prior_means.cpu(), net.model[0].get(L.BUF_MEANS))
    # opt keys: 'fixed' is applied by buildModel, anything but 'empirical' / 'fixed' is refused
    over = dict(input_size=8, hidden=[16], classes=list("abc"), batchSize=4, log=False)
    fixed = vbnn_b200.MLP(vbnn_b200.default_opt(prior="fixed", prior_mean=0.5, prior_var=2.0, vb_output=True, **over),
                          ctx, max_batch=4)
    assert [fixed.model[k].prior for k in fixed.vb_indices] == [("fixed", 0.5, 2.0)] * 2
    with pytest.raises(L.VbnnError):
        vbnn_b200.MLP(vbnn_b200.default_opt(prior="per_weight", **over), ctx, max_batch=4)


# ---------------------------------------------------------------- 9. checkpoint
def test_checkpoint_carries_the_prior(ctx, tmp_path):
    from vbnn_b200 import checkpoint
    a = build(ctx, vb_output=True)[0]
    a.set_prior("fixed", MU0, VAR0)
    a.model[0].set_prior("per_weight")
    for X, T in batches(16, 2):
        a.train_step(X, T)
    sd = a.state_dict()
    assert sd["0.prior"] == 2 and sd["1.prior"] == 1 and "0.prior_means" in sd and "1.prior_means" not in sd
    checkpoint.save_net(a, str(tmp_path))
    b = build(ctx, vb_output=True, seed=50)[0]
    b.load_state_dict(sd)
    c = build(ctx, vb_output=True, seed=51)[0]
    checkpoint.load_net(c, str(tmp_path))
    assert [m.prior for m in (c.model[0], c.model[1], c.model[2])] == \
        [("per_weight", None, None), ("fixed", f32(MU0), f32(VAR0)), ("fixed", f32(MU0), f32(VAR0))]
    step0 = ctx.get_step()
    runs = []
    for net in (a, b, c):
        ctx.set_step(step0)
        runs.append([net.train_step(X, T) for X, T in batches(17, 3)])
    assert_same_results(runs[0], runs[1])
    assert_same_results(runs[0], runs[2])
    assert_same_state(a, b, "state_dict")
    assert_same_state(a, c, "save_net")
    # a checkpoint without prior keys (older files) loads as the empirical prior
    old = {k: v for k, v in sd.items() if ".prior" not in k}
    c.load_state_dict(old)
    assert all(c.model[k].prior == ("empirical", None, None) for k in c.vb_indices)


# ---------------------------------------------------------------- 10. peer and NCCL modes
@pytest.mark.parametrize("mode,transport", [("peer", "1"), ("peer", "3"), ("nccl", "0")])
def test_data_parallel_prior(mode, transport):
    """Two GPUs under torchrun (skipped on one): sync the replicas, snapshot a PER_WEIGHT prior on every rank and train
    on; data-parallel equals one GPU (tools/dp_prior_check.py), and peer mode refuses a snapshot over stale rows."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, VBNN_DP=mode, VBNN_PEER_TRANSPORT=transport)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dp_prior_check.py")],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dp_prior_check OK" in r.stdout
