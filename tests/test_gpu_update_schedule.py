"""Live hyper-parameters on the device (pytest -m gpu): vbnn_layer_set_opts / vbnn_mlp_set_opts (VBLinear.set_opt,
MLP.set_opt) change B, the learning rates and the Adam constants between minibatches without re-capturing a step graph.
A set before the first step equals creating the net with the new values, a set between replays equals a fresh net
loaded with the same state, every update path follows the values, the updates match the fp64 references under a
per-step schedule, refused calls change nothing, and checkpoints carry the values.  Tolerances as test_gpu_mlp.py."""
import ctypes as C
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

import update_reference as R
from oracle import vbnn_oracle as O
from test_gpu_edge_values import knobs
from test_gpu_prior import (N, S, SIZES, assert_same_results, assert_same_state, batches, build, cpu, data, nll_sum,
                            rel, split_step)
from test_gpu_update import (buf, check, check_update, make_prior, prior_of, read_state, run_stats_update,
                             set_random_grads, set_random_state)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# B, lr_bias, lr_mu, lr_var, beta1, beta2, eps: every live value changes at every step
SCHEDULE = [
    (30.0, 1e-3, 1e-4, 0.05, 0.9, 0.999, 1e-8),
    (12.0, 3e-3, 4e-4, 0.02, 0.8, 0.99, 1e-6),
    (80.0, 5e-4, 2e-4, 0.08, 0.95, 0.995, 1e-7),
    (5.0, 2e-3, 1e-3, 0.01, 0.6, 0.9, 1e-5),
    (200.0, 1e-4, 5e-5, 0.03, 0.85, 0.98, 1e-8),
    (40.0, 0.0, 3e-4, 0.0, 0.0, 0.5, 1e-4),
]


def L_():
    from vbnn_b200 import _lib as L
    return L


def opt_with(opt, row):
    """opt with the live values of a schedule row, in the config dict's own keys (buildModel's mapping)"""
    B, lr_bias, lr_mu, lr_var, b1, b2, eps = row
    return dict(opt, B=B, state=dict(opt["state"], learningRate=lr_bias), varState=dict(opt["varState"], learningRate=lr_var),
                meanState=dict(opt["meanState"], learningRate=lr_mu, beta1=b1, beta2=b2, epsilon=eps))


def ref_opt(row, S_, lrt):
    B, lr_bias, lr_mu, lr_var, b1, b2, eps = row
    return dict(B=B, S=S_, lr_bias=lr_bias, lr_mu=lr_mu, lr_var=lr_var, beta1=b1, beta2=b2, eps=eps, lrt=lrt)


def set_tables(ref, oopt, row):
    """The Torch7 idiom on the oracle: opt.B and every layer's optimiser tables rewritten"""
    B, lr_bias, lr_mu, lr_var, b1, b2, eps = row
    oopt["B"] = B
    oopt["state"] = dict(oopt["state"], learningRate=lr_bias)
    for ol in ref.vb_all:
        ol.biasState["learningRate"] = lr_bias
        ol.meanState.update(learningRate=lr_mu, beta1=b1, beta2=b2, epsilon=eps)
        ol.varState.update(learningRate=lr_var, beta1=b1, beta2=b2, epsilon=eps)
    ref.state["learningRate"] = lr_bias             # the plain nn.Linear output layer (mlp.lua:120-123)


def build_with(ctx, row, precision="fp32", reparam="weight", vb_output=False, strict=True, seed=0, operand_round=None):
    """test_gpu_prior.build, the net and the oracle created with a schedule row's live values"""
    import vbnn_b200
    from test_gpu_prior import build as build0
    net, ref, oopt = build0(ctx, precision, reparam, vb_output, strict, seed, B=row[0], operand_round=operand_round)
    y = opt_with(net.opt, row)
    created = vbnn_b200.MLP(y, ctx, max_batch=N)
    # the same random parameters, under the options it was created with
    created.load_state_dict({k: v for k, v in net.state_dict().items() if not k.endswith(".opts")})
    return created, ref, oopt


def live(net):
    return [m.opts for m in net.model]


# ---------------------------------------------------------------- 1. a set before the first step equals create
@pytest.mark.parametrize("vb_output,strict", [(False, True), (True, False)])
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_set_at_step_0_equals_create(ctx, precision, reparam, vb_output, strict):
    """Net A created with X and set to Y, net B created with Y: four fused steps (eager, capture, replay, replay) leave
    bitwise-equal state, Adam moments, caches and live values."""
    a = build(ctx, precision, reparam, vb_output, strict, B=30.0)[0]
    b = build_with(ctx, SCHEDULE[1], precision, reparam, vb_output, strict)[0]
    y = opt_with(a.opt, SCHEDULE[1])
    c0 = a.graph_captures()
    a.set_opt(y)
    assert live(a) == live(b)
    step0 = ctx.get_step()
    runs = []
    for net in (a, b):
        ctx.set_step(step0)
        runs.append([net.train_step(X, T) for X, T in batches(2, 4)])
    assert a.graph_captures() == c0 + 1
    assert_same_results(runs[0], runs[1])
    assert_same_state(a, b)


def test_set_changes_the_trajectory(ctx):
    a = build(ctx)[0]
    b = build(ctx)[0]
    b.set_opt(opt_with(b.opt, SCHEDULE[3]))
    step0 = ctx.get_step()
    for net in (a, b):
        ctx.set_step(step0)
        for X, T in batches(3, 2):
            net.train_step(X, T)
    for k in a.vb_indices:
        assert not torch.equal(a.model[k].get(L_().BUF_MEANS), b.model[k].get(L_().BUF_MEANS))
        assert not torch.equal(a.model[k].get(L_().BUF_LVARS), b.model[k].get(L_().BUF_LVARS))


# ---------------------------------------------------------------- 2. a switch between replays equals a fresh net
PATHS = ["step", "grad_input", "split", "submit_host", "run_update", "layer_update"]


def one_step(net, ctx, path, Xn, Tn, X, T, G, gi):
    if path == "step":
        net.train_step(X, T)
    elif path == "grad_input":
        net.train_step(X, T, grad_input=gi)
    elif path == "split":
        split_step(net, X, T, G)
    elif path == "submit_host":
        net.submit_host(torch.from_numpy(Xn).float(), torch.from_numpy(Tn).float())
        net.collect()
    elif path == "run_update":
        net.resetGradients()
        for s in range(S):
            net.sample(s)
            net.run(X, T)
        net.update()
    elif path == "layer_update":                       # the reference's loop, each layer's update on its own
        L = L_()
        net.resetGradients()
        for s in range(S):
            net.sample(s)
            net.run(X, T)
        for m in net.model:
            L.check(L.lib().vbnn_layer_update(m.handle, None))
        ctx.set_step(ctx.get_step() + 1)


@pytest.mark.parametrize("path", PATHS)
def test_switch_between_replays_equals_a_fresh_net(ctx, path):
    """Net A runs three steps (eager, capture, replay), is set to Y and runs one more; net B is created with Y, loaded
    with A's state from before the switch and runs that step: bitwise-equal state."""
    a = build(ctx)[0]
    rng = np.random.RandomState(20)
    steps = [data(rng) for _ in range(4)]
    G = torch.empty(S, N, SIZES[-1], device="cuda")
    gi = torch.empty(N, SIZES[0], device="cuda")
    for Xn, Tn, X, T in steps[:3]:
        one_step(a, ctx, path, Xn, Tn, X, T, G, gi)
    torch.cuda.synchronize()
    sd = a.state_dict()
    y = opt_with(a.opt, SCHEDULE[2])
    c0 = a.graph_captures()
    a.set_opt(y)
    b = build_with(ctx, SCHEDULE[2], seed=99)[0]
    b.load_state_dict({k: v for k, v in sd.items() if not k.endswith(".opts")})
    assert live(a) == live(b)
    step0 = ctx.get_step()
    one_step(a, ctx, path, *steps[3], G, gi)
    assert a.graph_captures() == c0
    ctx.set_step(step0)
    one_step(b, ctx, path, *steps[3], G, gi)           # eager: b's first step
    torch.cuda.synchronize()
    assert_same_state(a, b, path)


@pytest.mark.parametrize("strict", [True, False])
def test_calc_lc_and_grads_follow_b(ctx, strict):
    """vbnn_layer_grads / calc_lc and vbnn_mlp_calc_lc after a change of B equal a fresh net created with that B."""
    a = build(ctx, strict=strict, B=30.0)[0]
    for X, T in batches(21, 3):
        a.train_step(X, T)
    a.set_opt(opt_with(a.opt, SCHEDULE[4]))
    b = build(ctx, strict=strict, B=SCHEDULE[4][0], seed=98)[0]
    b.load_state_dict(a.state_dict())
    for net in (a, b):                                 # var_hat and the strict caches of the current parameters
        for k in net.vb_indices:
            net.model[k].compute_prior()
    torch.cuda.synchronize()
    assert a.calc_lc() == b.calc_lc()
    for k in a.vb_indices:
        la, lb = a.model[k], b.model[k]
        assert torch.equal(la.calc_lc(), lb.calc_lc())
        for fa, fb in ((la.compute_mugrads, lb.compute_mugrads), (la.compute_vargrads, lb.compute_vargrads)):
            ga, gb = fa(), fb()
            assert torch.equal(ga[1], gb[1])
    # and 1/B scales calc_lc as the reference does
    c = build(ctx, strict=strict, B=30.0, seed=97)[0]
    c.load_state_dict(a.state_dict())
    c.set_opt(opt_with(c.opt, SCHEDULE[0]))
    for k in c.vb_indices:
        c.model[k].compute_prior()
    torch.cuda.synchronize()
    assert abs(c.calc_lc() * 30.0 / SCHEDULE[4][0] - a.calc_lc()) <= 1e-5 * abs(a.calc_lc())


# ---------------------------------------------------------------- 3. element by element against fp64
LAYER_CASES = [
    # O, I, prior, reparam, precision, strict, S, coresident
    (5, 13, "empirical", "local", "fp32", False, 3, False),         # scalar quads
    (9, 16, "fixed", "weight", "bf16", True, 1, False),             # VEC
    (7, 12, "per_weight", "local", "bf16", True, 3, False),
    (1000, 4096, "empirical", "local", "bf16", False, 3, False),
    (9, 16, "empirical", "weight", "fp32", True, 1, True),          # 128-thread co-resident variant
    (7, 12, "fixed", "local", "bf16", False, 3, True),
    (1000, 4096, "per_weight", "weight", "fp32", True, 1, True),
]


@pytest.mark.parametrize("case", LAYER_CASES, ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}-{c[3]}-{c[4]}-core{int(c[7])}")
def test_layer_update_under_a_schedule(ctx, case):
    """vbnn_layer_update with a set before each call, STATS and not alternating (the co-resident cases run the 128-thread
    variant on their non-STATS calls), against tests/update_reference.py fed that call's values; vbnn_layer_grads too."""
    import vbnn_b200
    L = L_()
    O_, I, kind, reparam, precision, strict, S_, core = case
    rng = np.random.RandomState(O_ + I)
    opt = vbnn_b200.default_opt(B=20.0, S=S_, reparam=reparam, precision=precision, strict_reference=strict,
                                var_init=0.01, mu_init=1, log=False)
    layer = vbnn_b200.VBLinear(I, O_, opt, ctx)
    grid = R.update_grid(O_, I)
    set_random_state(layer, rng, t=4)
    make_prior(layer, kind, rng)
    terms = R.PRIOR_CHUNK_TERMS
    with knobs(**({"upd_coresident": 1} if core else {})):
        for i, row in enumerate(SCHEDULE[:4]):
            stats = i % 2 == 1
            layer.set_opt(opt_with(opt, row))
            uopt = ref_opt(row, S_, reparam == "local")
            set_random_grads(layer, rng)
            if i == 0:
                layer.compute_prior()
                st = read_state(layer)
                outs = {k: layer._new() for k in ("mleg", "mlcg", "vleg", "vlcg")}
                L.check(L.lib().vbnn_layer_grads(layer.handle, *[C.c_void_p(outs[k].data_ptr()) for k in outs]))
                vh = R.var_hat(st["mu"], st["lv"], R.PRIOR_CHUNK_TERMS)
                ref_g = R.grads(st, uopt, prior_of(layer, kind, None), vh)
                for k in outs:
                    check(f"{case} grads {k}", outs[k], ref_g[k])
                layer.set(L.BUF_GRAD_WEIGHT, st["gW"].cpu().numpy())
                layer.set(L.BUF_GRAD_SUM, st["gS"].cpu().numpy())
            st = read_state(layer)
            ref = R.update(st, uopt, prior_of(layer, kind, terms))
            run_stats_update(layer, stats)
            check_update(f"{case} call {i}", layer, st, ref, strict)
            terms = R.update_terms(O_, I, grid, 128 if core and I % 4 == 0 and not stats else R.TPB)


@pytest.mark.parametrize("mode", ["step", "grad_input", "backward_update"])
@pytest.mark.parametrize("precision,reparam", [("fp32", "weight"), ("bf16", "local")])
def test_fused_step_under_a_schedule(ctx, precision, reparam, mode):
    """The fused net (eager, capture, replays) with vbnn_mlp_set_opts before every step: every VB layer's update and the
    output layer's SGD element by element against the reference fed that step's values."""
    import vbnn_b200
    L = L_()
    sizes, n = (40, 64, 30, 10), 96
    rng = np.random.RandomState(1)
    over = dict(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])], S=2,
                B=50.0, batchSize=n, testBatchSize=n, mu_init=1, var_init=0.01, reparam=reparam, log=False)
    net = vbnn_b200.MLP(vbnn_b200.default_opt(precision=precision, **over), ctx, max_batch=n)
    for k, m in enumerate(net.model):
        if m.kind == L.KIND_VB:
            set_random_state(m, rng, t=3 + k, mu_scale=math.sqrt(2.0 / m.inputSize))
        else:
            m.set(L.BUF_WEIGHT, rng.randn(m.outputSize, m.inputSize) * math.sqrt(2.0 / m.inputSize))
            m.set(L.BUF_BIAS, rng.randn(m.outputSize) * 0.1)
    terms = {k: R.PRIOR_CHUNK_TERMS for k in net.vb_indices}
    X = torch.from_numpy(rng.randn(n, sizes[0]).astype(np.float32)).cuda()
    T = torch.from_numpy(rng.randint(1, sizes[-1] + 1, n).astype(np.float32)).cuda()
    gi = torch.empty(n, sizes[0], device="cuda") if mode == "grad_input" else None
    G = torch.empty(2, n, sizes[-1], device="cuda")
    c0 = None
    for s, row in enumerate(SCHEDULE):
        net.set_opt(opt_with(net.opt, row))
        before = [read_state(m) if m.kind == L.KIND_VB else dict(w=buf(m, L.BUF_WEIGHT), b=buf(m, L.BUF_BIAS))
                  for m in net.model]
        if mode == "backward_update":
            y = net.forward_train(X)
            G.copy_(torch.from_numpy(rng.randn(*y.shape).astype(np.float32) * 1e-2))
            net.backward_update(G)
        else:
            net.train_step(X, T, sync=False, grad_input=gi)
        torch.cuda.synchronize()
        if s == 1:
            c0 = net.graph_captures()
        for k, m in enumerate(net.model):
            st = before[k]
            name = f"{precision} {reparam} {mode} step {s} layer {k}"
            if m.kind == L.KIND_VB:
                st.update(gW=buf(m, L.BUF_GRAD_WEIGHT), gS=buf(m, L.BUF_GRAD_SUM), gB=buf(m, L.BUF_GRAD_BIAS))
                ref = R.update(st, ref_opt(row, 2, reparam == "local"), prior_of(m, "empirical", terms[k]))
                check_update(name, m, st, ref, True)
                terms[k] = R.update_terms(m.outputSize, m.inputSize, R.update_grid(m.outputSize, m.inputSize))
            else:
                check(f"{name} weight", m._view(L.BUF_WEIGHT), R.sgd(st["w"], buf(m, L.BUF_GRAD_WEIGHT), row[1]))
                check(f"{name} bias", m._view(L.BUF_BIAS), R.sgd(st["b"], buf(m, L.BUF_GRAD_BIAS), row[1]))
    assert net.graph_captures() == c0


# ---------------------------------------------------------------- 4. the trajectory against the oracle
@pytest.mark.parametrize("precision,reparam,vb_output", [("fp32", "weight", False), ("fp32", "local", True),
                                                         ("bf16", "weight", False), ("bf16", "local", True)])
def test_trajectory_against_the_oracle(ctx, precision, reparam, vb_output):
    bf = precision == "bf16"
    net, ref, oopt = build(ctx, precision, reparam, vb_output, operand_round=O.round_bf16 if bf else None)
    tol = 5e-3 if bf else 2e-4
    rng = np.random.RandomState(5)
    nvb = len(ref.vb_all)
    gidx = lambda k: k if k < len(ref.vb) else len(net.model) - 1
    for it, row in enumerate(SCHEDULE):
        net.set_opt(opt_with(net.opt, row))
        set_tables(ref, oopt, row)
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


# ---------------------------------------------------------------- 5. no re-capture; replay equals no graph
def test_no_step_graph_recaptures(ctx):
    net = build(ctx)[0]
    X, T = batches(6, 1)[0]
    G = torch.empty(S, N, SIZES[-1], device="cuda")
    gi = torch.empty(N, SIZES[0], device="cuda")
    gi2 = torch.empty(N, SIZES[0], device="cuda")

    def all_five():
        net.train_step(X, T)
        net.train_step(X, T, grad_input=gi)
        split_step(net, X, T, G)
        y = net.forward_train(X)
        net.backward_update(G, grad_input=gi2)
    for _ in range(2):
        all_five()
    c0 = net.graph_captures()
    assert c0 == 5
    for row in SCHEDULE:
        net.set_opt(opt_with(net.opt, row))
        net.model[0].set_opt(opt_with(net.opt, SCHEDULE[0]))
        all_five()
        assert net.graph_captures() == c0


def test_graph_replay_equals_no_graph_under_a_schedule(ctx):
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
        for (X, T), row in zip(batches(10, 6), SCHEDULE):
            net.set_opt(opt_with(net.opt, row))
            net.train_step(X, T)
    assert b.graph_captures() == 0 and a.graph_captures() > 0
    assert_same_state(a, b)


# ---------------------------------------------------------------- 6. ordering in the host pipeline
def test_set_between_submits_is_stream_ordered(ctx):
    """submit_host(t), set, submit_host(t+1) without a collect in between equals the eager sequence with the set
    between the two steps."""
    from vbnn_b200 import _lib as L
    a = build(ctx)[0]
    L.knob("no_graph", 1)
    try:
        b = build(ctx)[0]
    finally:
        L.knob("no_graph")
    rng = np.random.RandomState(30)
    steps = [data(rng) for _ in range(6)]
    h = lambda Xn, Tn: (torch.from_numpy(Xn).float(), torch.from_numpy(Tn).float())
    step0 = ctx.get_step()
    for i in range(0, 6, 2):
        a.submit_host(*h(*steps[i][:2]))
        a.set_opt(opt_with(a.opt, SCHEDULE[i + 1]))
        a.submit_host(*h(*steps[i + 1][:2]))
        a.collect(); a.collect()
    ctx.set_step(step0)
    for i in range(6):
        b.train_step(*steps[i][2:])
        if i % 2 == 0:
            b.set_opt(opt_with(b.opt, SCHEDULE[i + 1]))
    torch.cuda.synchronize()
    assert_same_state(a, b)


# ---------------------------------------------------------------- 7. per-layer sets
def test_a_set_on_one_layer_leaves_the_others_alone(ctx):
    a = build(ctx, vb_output=True)[0]
    b = build(ctx, vb_output=True)[0]
    b.model[1].set_opt(opt_with(b.opt, SCHEDULE[3]))
    assert b.model[1].opts != b.model[0].opts == a.model[0].opts
    step0 = ctx.get_step()
    for net in (a, b):                                 # one step: every layer's gradient comes before any update
        ctx.set_step(step0)
        net.train_step(*batches(11, 1)[0])
    sa, sb = a.state_dict(), b.state_dict()
    for key in sa:
        if key.split(".")[0] in ("0", "2"):
            assert (torch.equal(sa[key], sb[key]) if isinstance(sa[key], torch.Tensor) else sa[key] == sb[key]), key
    assert not torch.equal(sa["1.means"], sb["1.means"])


# ---------------------------------------------------------------- 8. refusals
def test_refusals_change_nothing(ctx):
    L = L_()
    lib = L.lib()
    a = build(ctx, vb_output=True)[0]
    b = build(ctx, vb_output=True)[0]
    X, T = batches(12, 1)[0]
    h = a.model[0].handle
    base = a.model[0]._get_opts()
    bad = [("B", float("nan")), ("B", float("inf")), ("B", -float("inf")), ("B", 0.0), ("B", -1.0),
           ("lr_mu", -1e-4), ("lr_var", float("nan")), ("lr_bias", float("inf")), ("adam_beta1", 1.0),
           ("adam_beta2", 1.0), ("adam_beta1", -0.1), ("adam_beta2", float("nan")), ("adam_eps", 0.0),
           ("adam_eps", float("inf")), ("adam_eps", -1e-8),
           ("var_init", 0.5), ("msr_init", 1), ("mu_init", 2.0), ("S", 3), ("reparam", 1), ("precision", 1),
           ("strict_reference", 0)]
    for f, v in bad:
        o = L.VbnnOpts.from_buffer_copy(base)
        setattr(o, f, v)
        assert lib.vbnn_layer_set_opts(h, C.byref(o)) == L.E_INVALID, (f, v)
        assert f in lib.vbnn_last_error().decode(), (f, lib.vbnn_last_error())
        assert lib.vbnn_mlp_set_opts(a.handle, C.byref(o)) == L.E_INVALID, (f, v)
    assert lib.vbnn_layer_set_opts(h, None) == L.E_INVALID
    assert lib.vbnn_layer_set_opts(None, C.byref(base)) == L.E_INVALID
    assert lib.vbnn_mlp_set_opts(a.handle, None) == L.E_INVALID
    assert lib.vbnn_layer_get_opts(h, None) == L.E_INVALID
    # every refusal above left the values and the next step as they were
    assert [m.opts for m in a.model] == [m.opts for m in b.model]
    step0 = ctx.get_step()
    for net in (a, b):
        ctx.set_step(step0)
        net.train_step(X, T)
    assert_same_state(a, b)


@pytest.mark.parametrize("key,value", [("S", 1), ("reparam", "local"), ("precision", "bf16"), ("strict_reference", False),
                                       ("var_init", 0.5), ("msr_init", True), ("mu_init", 0)])
def test_set_opt_refuses_a_changed_build_key(ctx, key, value):
    """MLP.set_opt / VBLinear.set_opt with a dict whose build keys differ from the net's: VbnnError(E_INVALID) naming
    the field, and the net's opt, the layers' values and the next split step (whose buffers are sized by opt["S"]) are
    as if the call had not happened."""
    from vbnn_b200 import _lib as L
    a = build(ctx)[0]
    b = build(ctx)[0]
    opt0 = a.opt
    bad = dict(opt_with(a.opt, SCHEDULE[3]), **{key: value})
    field = {"reparam": "reparam", "precision": "precision"}.get(key, key)
    for call in (a.set_opt, a.model[0].set_opt):
        with pytest.raises(L.VbnnError) as e:
            call(bad)
        assert e.value.code == L.E_INVALID and field in str(e.value), str(e.value)
    assert a.opt is opt0 and a.model[0].opt is opt0
    assert live(a) == live(b)
    X, T = batches(18, 1)[0]
    G = torch.empty(S, N, SIZES[-1], device="cuda")
    step0 = ctx.get_step()
    for net in (a, b):
        ctx.set_step(step0)
        split_step(net, X, T, G)
    torch.cuda.synchronize()
    assert_same_state(a, b)


def test_set_opt_replaces_only_the_live_keys_of_opt(ctx):
    """After set_opt the net's opt (what save_net records) has the new B and optimiser tables and every other key as
    built; after load_state_dict it has the values the checkpoint carried."""
    a = build(ctx)[0]
    built = dict(a.opt)
    new = dict(opt_with(a.opt, SCHEDULE[2]), hidden=[1], testSamples=1, quicktest=True)
    a.set_opt(new)
    for k in built:
        if k in ("B", "state", "meanState", "varState"):
            assert a.opt[k] == new[k], k
        else:
            assert a.opt[k] == built[k], k
    assert all(m.opt is a.opt for m in a.model)
    b = build(ctx, seed=3)[0]
    b.load_state_dict(a.state_dict())
    f = lambda v: float(np.float32(v))
    row = SCHEDULE[2]
    assert b.opt["B"] == f(row[0]) and b.opt["state"]["learningRate"] == f(row[1])
    assert b.opt["meanState"]["learningRate"] == f(row[2]) and b.opt["varState"]["learningRate"] == f(row[3])
    assert (b.opt["meanState"]["beta1"], b.opt["meanState"]["beta2"], b.opt["meanState"]["epsilon"]) == \
        (f(row[4]), f(row[5]), f(row[6]))
    assert b.opt["S"] == built["S"] and b.opt["hidden"] == built["hidden"]


def test_refused_during_stream_capture(ctx):
    """A set while the context's stream is being captured: VBNN_E_STATE from both calls, and nothing changes."""
    L = L_()
    lib = L.lib()
    net = build(ctx)[0]
    X, T = batches(13, 1)[0]
    net.train_step(X, T)
    torch.cuda.synchronize()
    before = live(net)
    o = net.model[0]._get_opts()
    o.B = 3.0
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(ctx.stream):
        g.capture_begin(capture_error_mode="thread_local")
        try:
            rc_layer = lib.vbnn_layer_set_opts(net.model[0].handle, C.byref(o))
            rc_net = lib.vbnn_mlp_set_opts(net.handle, C.byref(o))
        finally:
            g.capture_end()
    assert rc_layer == L.E_STATE and rc_net == L.E_STATE
    assert live(net) == before


# ---------------------------------------------------------------- 9. checkpoints
def test_checkpoint_carries_the_values(ctx, tmp_path):
    from vbnn_b200 import checkpoint
    a = build(ctx, vb_output=True)[0]
    a.set_opt(opt_with(a.opt, SCHEDULE[1]))
    a.model[1].set_opt(opt_with(a.opt, SCHEDULE[2]))
    for X, T in batches(16, 2):
        a.train_step(X, T)
    sd = a.state_dict()
    assert torch.equal(sd["1.opts"], torch.tensor(SCHEDULE[2], dtype=torch.float32))
    assert torch.equal(sd["0.opts"], torch.tensor(SCHEDULE[1], dtype=torch.float32))
    checkpoint.save_net(a, str(tmp_path))
    b = build(ctx, vb_output=True, seed=50)[0]
    b.load_state_dict(sd)
    c = build(ctx, vb_output=True, seed=51)[0]
    opt = checkpoint.load_net(c, str(tmp_path))
    assert opt["B"] == SCHEDULE[1][0]                  # save_net records the net's opt after set_opt
    assert live(a) == live(b) == live(c)
    step0 = ctx.get_step()
    runs = []
    for net in (a, b, c):
        ctx.set_step(step0)
        runs.append([net.train_step(X, T) for X, T in batches(17, 3)])
    assert_same_results(runs[0], runs[1])
    assert_same_results(runs[0], runs[2])
    assert_same_state(a, b, "state_dict")
    assert_same_state(a, c, "save_net")
    # a checkpoint without the key (older files) keeps the net's values
    d = build(ctx, vb_output=True, seed=52)[0]
    d.set_opt(opt_with(d.opt, SCHEDULE[4]))
    mine = live(d)
    d.load_state_dict({k: v for k, v in sd.items() if not k.endswith(".opts")})
    assert live(d) == mine


# ---------------------------------------------------------------- 10. peer and NCCL modes
@pytest.mark.parametrize("mode,transport", [("peer", "1"), ("peer", "3"), ("nccl", "0")])
def test_data_parallel_schedule(mode, transport):
    """Two GPUs under torchrun (skipped on one): a per-minibatch schedule set on every rank; data-parallel equals one
    GPU stepping the full minibatch under the same schedule (tools/dp_hparams_check.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, VBNN_DP=mode, VBNN_PEER_TRANSPORT=transport)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dp_hparams_check.py")],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dp_hparams_check OK" in r.stdout
