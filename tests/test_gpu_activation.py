"""GPU tests of the hidden-layer activation of the fused net (pytest -m gpu): vbnn_mlp_set_activation with tanh, sigmoid
and ELU.  The fused step matches the fp64 reference of tests/activation_reference.py on the device-drawn noise in both
engines, also where the LRT GEMMs run several work units per CTA; every net-level entry point follows the kind; ReLU is
untouched by a round trip through another kind; saturated layers stay finite and pass exactly 0; the setter refuses
what it must; checkpoints carry the kind; and data-parallel training matches one GPU."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import activation_reference as A
import work_units as W
from custom_loss_reference import classnll_grad
from oracle import vbnn_oracle as O
from test_gpu_custom_loss import nll_sum, split_step, state_tensors
from test_gpu_input_grad import build_pair, cpu, data, device_noise, rel, snapshot

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMOOTH = ("tanh", "sigmoid", "elu")


def nll_scalars(Y, Tn):
    """The fused step's {error, accuracy %} from reference outputs Y [S x N x C] and 1-based labels."""
    T = torch.as_tensor(Tn, dtype=torch.float64)
    err = acc = 0.0
    for s in range(Y.shape[0]):
        logp = O.log_softmax(Y[s])
        err += float(O.class_nll_forward(logp, T))
        acc += float(O.get_accuracy(logp, T))
    return err / Y.shape[0], acc / Y.shape[0]


def check_state(net, ref, it, tol_par, tol_adam, tol_bias):
    from vbnn_b200 import _lib as L
    for gl, ol in zip(net.model, ref.vb + [ref.out]):
        if isinstance(ol, O.VBLinearOracle):
            pairs = [(L.BUF_MEANS, ol.means, tol_par), (L.BUF_LVARS, ol.lvars, tol_par), (L.BUF_BIAS, ol.bias, tol_bias),
                     (L.BUF_ADAM_M_MU, ol.meanState["m"], tol_adam), (L.BUF_ADAM_V_MU, ol.meanState["v"], tol_adam),
                     (L.BUF_ADAM_M_VAR, ol.varState["m"], tol_adam), (L.BUF_ADAM_V_VAR, ol.varState["v"], tol_adam)]
        else:
            pairs = [(L.BUF_WEIGHT, ol.weight, tol_par), (L.BUF_BIAS, ol.bias, tol_bias)]
        for b, want, t in pairs:
            e = rel(gl.get(b), want)
            assert e <= t, (it, b, e)


# ---------------------------------------------------------------- 1. the fused step against the reference
@pytest.mark.parametrize("vb_output", [False, True])
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", SMOOTH)
def test_fused_step_vs_reference(ctx, kind, precision, reparam, S, vb_output):
    """Ragged 37-29-23-10 net, N = 45, ClassNLL, two minibatches (the second replays the captured graph) against the fp64
    reference (bf16: with its operand rounding) on the device-drawn noise: parameters, Adam state and both scalars at the
    tolerances of test_fused_regression_vs_reference; the accuracy may differ by one row per sample in bf16."""
    sizes, N = [37, 29, 23, 10], 45
    bf = precision == "bf16"
    lrt = reparam == "local"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, precision, reparam, seed=7, strict=False, vb_output=vb_output,
                                      operand_round=O.round_bf16 if bf else None)
    net.set_activation(kind)
    tol = (5e-3 if lrt else 1e-2) if bf else 1e-5
    tol_par = 5e-3 if bf else 2e-4
    tol_adam = 2e-2 if bf else 1e-4
    rng = np.random.RandomState(5)
    for it in range(2):
        Xn, Tn, X, Tt = data(rng, N, sizes[0], sizes[-1])
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        err, acc = net.train_step(X, Tt)
        Yr, _, _ = A.minibatch(ref, torch.from_numpy(Xn), classnll_grad(torch.from_numpy(Tn)), noise, lrt, kind, oopt)
        we, wa = nll_scalars(Yr, Tn)
        assert abs(err - we) <= tol * abs(we) + 1e-7, (it, err, we)
        assert abs(acc - wa) <= (100.0 / N + 1e-4 if bf else 1e-4), (it, acc, wa)
        check_state(net, ref, it, tol_par, tol_adam, max(tol_par, tol, 1e-4))


@pytest.mark.parametrize("lrt_split", [0, 3])
@pytest.mark.parametrize("kind", SMOOTH)
def test_lrt_gemms_run_several_units_per_cta(ctx, kind, lrt_split):
    """bf16 LRT 256-1024-1024-10, N = 4096, S = 2 on 128 x 128 tiles: the hidden layers' fwd-lrt and dx-lrt GEMMs
    (dual with lrt_split 0, split with 3) run >= 3 work units per resident CTA (tests/work_units.py), so each CTA
    carries its epilogue state across tiles.  One minibatch against the bf16-rounding reference: the error scalar, dX,
    parameters and Adam state."""
    import vbnn_b200
    sizes, N, S = [256, 1024, 1024, 10], 4096, 2
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert W.per_slot(N, sizes[2], 128, 1, sms, S) >= 3        # fwd-lrt of the second hidden layer
    assert W.per_slot(N, sizes[1], 128, 1, sms, S) >= 3        # dx-lrt into the first hidden layer
    names = ("tc_bn", "tc_cg", "lrt_split")
    old = [vbnn_b200.knob(n) for n in names]
    vbnn_b200.knob("tc_bn", 128); vbnn_b200.knob("tc_cg", 1); vbnn_b200.knob("lrt_split", lrt_split)
    try:
        net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, "bf16", "local", seed=2, strict=False,
                                          operand_round=O.round_bf16)
        net.set_activation(kind)
        Xn, Tn, X, Tt = data(np.random.RandomState(3), N, sizes[0], sizes[-1])
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        dx = torch.empty(N, sizes[0], device="cuda")
        err, _ = net.train_step(X, Tt, grad_input=dx)
        Yr, _, dXr = A.minibatch(ref, torch.from_numpy(Xn), classnll_grad(torch.from_numpy(Tn)), noise, True, kind, oopt)
    finally:
        for n, v in zip(names, old):
            vbnn_b200.knob(n, v)
    we, _ = nll_scalars(Yr, Tn)
    assert abs(err - we) <= 5e-3 * abs(we), (err, we)
    assert rel(cpu(dx), dXr.numpy()) <= 5e-3
    check_state(net, ref, 0, 5e-3, 2e-2, 5e-3)


# ---------------------------------------------------------------- 2. every net-level path follows the kind
CONFIGS = [("fp32", "weight", 3), ("bf16", "local", 2), ("bf16", "weight", 2)]


@pytest.mark.parametrize("precision,reparam,S", CONFIGS)
@pytest.mark.parametrize("kind", SMOOTH)
def test_step_grad_input_vs_reference(ctx, kind, precision, reparam, S):
    """step_grad_input over two minibatches (eager, then captured): dX and the error scalar against the reference."""
    sizes, N = [37, 29, 23, 10], 45
    bf = precision == "bf16"
    lrt = reparam == "local"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, precision, reparam, seed=7, strict=False,
                                      operand_round=O.round_bf16 if bf else None)
    net.set_activation(kind)
    tol = (5e-3 if lrt else 1e-2) if bf else 1e-5
    rng = np.random.RandomState(6)
    dx = torch.empty(N, sizes[0], device="cuda")
    for it in range(2):
        Xn, Tn, X, Tt = data(rng, N, sizes[0], sizes[-1])
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        dx.fill_(float("nan"))
        err, _ = net.train_step(X, Tt, grad_input=dx)
        Yr, _, dXr = A.minibatch(ref, torch.from_numpy(Xn), classnll_grad(torch.from_numpy(Tn)), noise, lrt, kind, oopt)
        assert np.isfinite(cpu(dx)).all()
        assert rel(cpu(dx), dXr.numpy()) <= tol, it
        we, _ = nll_scalars(Yr, Tn)
        assert abs(err - we) <= tol * abs(we) + 1e-7


@pytest.mark.parametrize("precision,reparam,S", CONFIGS)
@pytest.mark.parametrize("kind", SMOOTH)
def test_split_step_equals_fused(ctx, kind, precision, reparam, S):
    """forward_train + torch log_softmax / nll_loss + backward_update against train_step from identical state, three
    minibatches: state within the tolerances of test_split_equals_fused_step (fp32 1e-6, bf16 1e-3)."""
    sizes, N = [200, 136, 96, 10], 160
    a, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=3, strict=False)
    b, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=4, strict=False)
    a.set_activation(kind); b.set_activation(kind)
    tol = 1e-6 if precision == "fp32" else 1e-3
    rng = np.random.RandomState(9)
    for it in range(3):
        _, _, X, Tt = data(rng, N, sizes[0], sizes[-1])
        sd = a.state_dict()
        b.load_state_dict(sd)
        a.train_step(X, Tt)
        outs = [a.outputs(s, N) for s in range(S)]
        ctx.set_step(sd["step"])
        Y, _, _ = split_step(b, X, nll_sum(Tt))
        for s in range(S):
            assert rel(cpu(F.log_softmax(Y[s], -1)), cpu(outs[s])) <= max(tol, 1e-6), (it, s)
        sa, sb = state_tensors(a), state_tensors(b)
        for k in sa:
            assert rel(sa[k], sb[k]) <= tol, (it, k)


@pytest.mark.parametrize("precision,reparam,S", CONFIGS)
@pytest.mark.parametrize("kind", SMOOTH)
def test_evaluation_paths_vs_reference(ctx, kind, precision, reparam, S):
    """test (MC and MAP), predict and predict_outputs against the reference forward on the noise the evaluation draws
    (sample indices 2^20 + t at the current step), and run against the reference forward / backward of its sample."""
    from vbnn_b200 import _lib as L
    sizes, N, T = [37, 29, 23, 10], 45, 5
    bf = precision == "bf16"
    lrt = reparam == "local"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, precision, reparam, seed=7, strict=False,
                                      operand_round=O.round_bf16 if bf else None)
    net.set_activation(kind)
    tol = (5e-3 if lrt else 1e-2) if bf else 1e-5
    Xn, Tn, X, Tt = data(np.random.RandomState(11), N, sizes[0], sizes[-1])
    xr = torch.from_numpy(Xn)
    step = ctx.get_step()
    gidx = lambda k: k if k < len(ref.vb) else len(net.model) - 1
    noise = [[torch.from_numpy(cpu(net.model[gidx(k)].draw_noise(step, (1 << 20) + t, rows=N)).astype(np.float64))
              for k in range(len(ref.vb_all))] for t in range(T)]
    Yr = A.predict_forward(ref, xr, kind, noise, lrt)                                  # [T x N x C]
    Ymap = A.predict_forward(ref, xr, kind, None, lrt, map_mode=True)
    po = net.predict_outputs(X, n_samples=T, return_samples=True)
    assert rel(cpu(po.samples), Yr.numpy()) <= tol
    assert rel(cpu(po.mean), Yr.mean(0).numpy()) <= tol
    pm = net.predict_outputs(X, n_samples=0, return_samples=True)
    assert rel(cpu(pm.samples[0]), Ymap[0].numpy()) <= tol
    pr = net.predict(X, n_samples=T)
    want = torch.logsumexp(torch.log_softmax(Yr, -1), 0) - np.log(T)
    assert rel(cpu(pr.logp), want.numpy()) <= tol
    for ns, Y in ((T, Yr), (0, Ymap)):
        net.opt["testSamples"] = ns
        net.opt["quicktest"] = ns == 0
        err, _ = net.test(X, Tt)
        we, _ = nll_scalars(Y, Tn)
        assert abs(err - we) <= tol * abs(we) + 1e-7, (ns, err, we)
    net.opt["quicktest"] = False
    # run: one sample's forward + backward, gradients accumulated
    net.resetGradients()
    net.sample(0)
    sidx = 0 if not lrt else net._s
    rn = [torch.from_numpy(cpu(net.model[gidx(k)].draw_noise(step, sidx, rows=N)).astype(np.float64))
          for k in range(len(ref.vb_all))]
    err, _ = net.run(X, Tt)
    ref.resetGradients()
    ref.sample(None if lrt else rn)
    x = ref.q(xr)
    acts, Y1 = A.forward(ref, x, kind, rn if lrt else None)
    A.backward(ref, acts, classnll_grad(torch.from_numpy(Tn))(Y1[None])[0], kind)
    we, _ = nll_scalars(Y1[None], Tn)
    assert abs(err - we) <= tol * abs(we) + 1e-7
    for gl, ol in zip(net.model, ref.vb + [ref.out]):
        assert rel(gl.get(L.BUF_GRAD_WEIGHT), ol.gradWeight) <= tol


@pytest.mark.parametrize("kind", SMOOTH)
def test_host_pipeline_equals_step_host(ctx, kind):
    """From one state and step: submit_host + collect against step_host leaves bit-identical exact state (the error
    scalar, a sum of fp32 atomics, within 1e-6).  submit_host_u8 against step_host of the same pixels normalised on the
    host: within 1e-6 (the u8 staging kernel normalises and squares its own operand).  Two minibatches in flight against
    two step_host calls: within 1e-6 (the second starts from biases finished by fp32 atomics)."""
    sizes, N, S = [64, 48, 32, 10], 50, 2
    a, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    b, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    a.set_activation(kind); b.set_activation(kind)
    rng = np.random.RandomState(4)
    X = [torch.from_numpy(rng.randn(N, sizes[0])).float() for _ in range(2)]
    T = [torch.from_numpy(rng.randint(1, 11, N).astype(np.float32)) for _ in range(3)]
    U = torch.from_numpy(rng.randint(0, 256, (N, sizes[0]))).to(torch.uint8)
    mean, std = 33.0, 78.0
    Xu = (U.float() - mean) * np.float32(1.0 / std)
    ctx.set_step(30)
    for it, (x, u8) in enumerate(((X[0], False), (X[1], False), (Xu, True), (Xu, True))):
        sd = a.state_dict()
        b.load_state_dict(sd)
        ea_, ma = a.train_step_host(x, T[it % 3])
        ctx.set_step(sd["step"])
        if u8:
            b.submit_host_u8(U, T[it % 3], mean, std)
        else:
            b.submit_host(x, T[it % 3])
        eb_, mb = b.collect()
        assert abs(ea_ - eb_) <= 1e-6 * abs(ea_) and (u8 or ma == mb), it
        for p, q in zip(snapshot(a)[0], snapshot(b)[0]):
            assert rel(p, q) <= 1e-6 if u8 else torch.equal(p, q), it
    sd = a.state_dict()
    b.load_state_dict(sd)
    want = [a.train_step_host(X[0], T[0]), a.train_step_host(X[1], T[1])]
    ctx.set_step(sd["step"])
    b.submit_host(X[0], T[0]); b.submit_host(X[1], T[1])
    got = [b.collect(), b.collect()]
    for (e1, m1), (e2, m2) in zip(want, got):
        assert abs(e1 - e2) <= 1e-6 * abs(e1) and abs(m1 - m2) <= 100.0 / N
    for p, q in zip(snapshot(a)[0], snapshot(b)[0]):
        assert rel(p, q) <= 1e-6


def test_gaussian_nll_tanh_net_trains_and_evaluates(ctx):
    """The 1-D heteroscedastic problem of test_heteroscedastic_regression_learns_fused (noise growing with |x|, the same
    rates) on a tanh net built with opt["activation"]: the median loss of minibatches 200-250 is below that of the
    first 20, and predict_outputs(gaussian) then gives finite means, epistemic and positive aleatoric variances, a
    finite mixture NLL and a lower RMSE than before training."""
    import vbnn_b200
    N, S = 256, 2
    opt = vbnn_b200.default_opt(input_size=1, hidden=[64, 64], outputs=2, criterion="gaussian_nll", S=S, B=2000.0,
                                batchSize=N, testSamples=8, mu_init=1, msr_init=True, vb_output=False, reparam="local",
                                strict_reference=False, log=False, seed=5, meanState=dict(learningRate=1e-3),
                                state=dict(learningRate=1e-4), activation="tanh")
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    assert net.activation == "tanh"
    net.init_params(seed=4, he_means=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    xe = torch.rand(N, 1, device="cuda", generator=g) * 4 - 2
    ye = torch.sin(2 * xe) + (0.05 + 0.3 * xe.abs()) * torch.randn(N, 1, device="cuda", generator=g)
    r0 = net.predict_outputs(xe, model="gaussian", targets=ye).rmse
    losses = []
    for _ in range(250):
        x = torch.rand(N, 1, device="cuda", generator=g) * 4 - 2
        y = torch.sin(2 * x) + (0.05 + 0.3 * x.abs()) * torch.randn(N, 1, device="cuda", generator=g)
        losses.append(net.train_step(x, y)[0])
    assert np.isfinite(losses).all()
    first, late = float(np.median(losses[:20])), float(np.median(losses[200:]))
    print(f"tanh heteroscedastic NLL: median of the first 20 {first:.4f}, of 200-250 {late:.4f}")
    assert late < first, (first, late)
    p = net.predict_outputs(xe, model="gaussian", targets=ye)
    for t in (p.mean, p.epistemic, p.aleatoric):
        assert torch.isfinite(t).all()
    assert float(p.aleatoric.min()) > 0 and np.isfinite(p.nll)
    assert p.rmse < r0, (p.rmse, r0)


# ---------------------------------------------------------------- 3. ReLU untouched, graphs, launches
def test_relu_round_trip_is_bit_identical(ctx):
    """Net A set to tanh, stepped, and set back to ReLU; net B never set.  Loaded with one state at one step, three
    minibatches leave bit-identical exact state, scalars and outputs (the biases, finished by fp32 atomics, within
    1e-6).  Each change re-captures the step graph once at its next use; a same-value set re-captures nothing."""
    sizes, N, S = [64, 48, 32, 10], 40, 2
    a, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    b, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    rng = np.random.RandomState(8)
    Xc = torch.from_numpy(rng.randn(N, sizes[0])).float().cuda()
    Tc = torch.from_numpy(rng.randint(1, 11, N).astype(np.float64)).float().cuda()
    for net in (a, b):
        net.train_step(Xc, Tc); net.train_step(Xc, Tc); net.train_step(Xc, Tc)      # eager, capture, replay
    c0 = a.graph_captures()
    a.set_activation("tanh")
    assert a.graph_captures() == c0
    a.train_step(Xc, Tc)
    assert a.graph_captures() == c0 + 1
    a.set_activation("tanh")
    a.train_step(Xc, Tc)
    assert a.graph_captures() == c0 + 1
    a.set_activation("relu")
    sd = b.state_dict()
    a.load_state_dict(sd); b.load_state_dict(sd)
    cb = b.graph_captures()
    res = []
    for net in (a, b):
        ctx.set_step(77)
        r = [net.train_step(Xc, Tc) for _ in range(3)]
        res.append((r, snapshot(net), [net.outputs(s, N) for s in range(S)]))
    assert a.graph_captures() == c0 + 2 and b.graph_captures() == cb + 1      # (a load drops the graphs)
    (ra, (ea, fa), oa), (rb, (eb, fb), ob) = res
    for x, w in zip(ea, eb):
        assert torch.equal(x, w)
    for x, w in zip(fa, fb):
        assert rel(x, w) <= 1e-6
    for p, q in zip(ra, rb):
        assert abs(p[0] - q[0]) <= 1e-6 * abs(q[0]) and p[1] == q[1]
    for x, w in zip(oa, ob):
        assert rel(x, w) <= 1e-6


@pytest.mark.parametrize("precision,reparam", [("bf16", "local"), ("bf16", "weight"), ("fp32", "local")])
def test_launch_count_is_the_same_for_every_kind(ctx, precision, reparam):
    """One step per kind on one net: the launch count per step is the same for all four kinds."""
    from vbnn_b200 import _lib as L
    sizes, N, S = [64, 48, 32, 10], 40, 2
    net, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=3, strict=False)
    _, _, X, Tt = data(np.random.RandomState(1), N, sizes[0], sizes[-1])
    counts = {}
    for kind in A.KINDS:
        net.set_activation(kind)
        v = C.c_int()
        L.check(L.lib().vbnn_mlp_get_activation(net.handle, C.byref(v)))
        assert v.value == L.ACTIVATIONS[kind]
        n0 = net.launch_count()
        net.train_step(X, Tt)
        counts[kind] = net.launch_count() - n0
    assert len(set(counts.values())) == 1, counts


# ---------------------------------------------------------------- 4. edges
@pytest.mark.parametrize("precision,reparam", [("fp32", "weight"), ("fp32", "local"), ("bf16", "weight"),
                                               ("bf16", "local")])
@pytest.mark.parametrize("kind", SMOOTH)
def test_saturation(ctx, kind, precision, reparam):
    """First-layer biases of +-100 (alternating units): outputs, dX and every parameter stay finite.  Then all of them at
    the saturating end (+100 tanh, -100 ELU): the first layer passes exactly 0 gradient (its gradWeight and dX are 0)."""
    from vbnn_b200 import _lib as L
    sizes, N, S = [40, 32, 24, 10], 30, 2
    net, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=5, strict=False)
    net.set_activation(kind)
    _, _, X, Tt = data(np.random.RandomState(2), N, sizes[0], sizes[-1])
    dx = torch.empty(N, sizes[0], device="cuda")
    b = np.where(np.arange(sizes[1]) % 2 == 0, 100.0, -100.0)
    net.model[0].set(L.BUF_BIAS, b)
    err, _ = net.train_step(X, Tt, grad_input=dx)
    assert np.isfinite(err) and np.isfinite(cpu(dx)).all()
    assert all(np.isfinite(cpu(net.outputs(s, N))).all() for s in range(S))
    for v in state_tensors(net).values():
        assert torch.isfinite(v).all()
    if kind == "sigmoid":
        return
    net.model[0].set(L.BUF_BIAS, np.full(sizes[1], 100.0 if kind == "tanh" else -100.0))
    net.train_step(X, Tt, grad_input=dx)
    assert (cpu(dx) == 0).all()
    assert (cpu(net.model[0].get(L.BUF_GRAD_WEIGHT)) == 0).all()
    assert (cpu(net.model[0].get(L.BUF_GRAD_BIAS)) == 0).all()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_zero_row_under_tanh_keeps_r_zero(ctx, precision):
    """LRT, tanh, zero biases: an all-zero input row stays all-zero through the hidden layers (tanh(0) = 0), so every
    layer has V = 0 and R = 0 there; the row's outputs are exactly the (zero) output biases and every gradient is
    finite."""
    from vbnn_b200 import _lib as L
    sizes, N, S = [40, 32, 24, 10], 30, 2
    net, _, _, _ = build_pair(ctx, sizes, N, S, precision, "local", seed=5, strict=False, vb_output=True)
    net.set_activation("tanh")
    for m in net.model:
        m.set(L.BUF_BIAS, np.zeros(m.get(L.BUF_BIAS).shape[0]))
    _, _, X, Tt = data(np.random.RandomState(2), N, sizes[0], sizes[-1])
    X[7] = 0
    Y = net.forward_train(X).clone()
    net.backward_update(torch.randn_like(Y))
    assert (cpu(Y[:, 7]) == 0).all()
    for v in state_tensors(net).values():
        assert torch.isfinite(v).all()


# ---------------------------------------------------------------- 5. refusals
def test_refusals(ctx):
    from vbnn_b200 import _lib as L
    import vbnn_b200
    lib = L.lib()
    net, _, _, _ = build_pair(ctx, [13, 7, 3], 4, 2, "fp32", "weight")
    h = net.handle
    assert lib.vbnn_mlp_set_activation(None, 1) == L.E_INVALID
    assert lib.vbnn_mlp_get_activation(None, C.byref(C.c_int())) == L.E_INVALID
    assert lib.vbnn_mlp_get_activation(h, None) == L.E_INVALID
    for bad in (-1, 4, 99):
        assert lib.vbnn_mlp_set_activation(h, bad) == L.E_INVALID
    with pytest.raises(vbnn_b200.VbnnError):
        net.set_activation("gelu")
    X = torch.randn(4, 13, device="cuda")
    net.forward_train(X)                                                              # an open split step
    assert lib.vbnn_mlp_set_activation(h, L.ACT_TANH) == L.E_STATE
    net.resetGradients()
    net.submit_host(torch.randn(4, 13), torch.ones(4))                                # uncollected minibatch
    assert lib.vbnn_mlp_set_activation(h, L.ACT_TANH) == L.E_STATE
    net.collect()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(ctx.stream):
        g.capture_begin(capture_error_mode="thread_local")
        try:
            rc = lib.vbnn_mlp_set_activation(h, L.ACT_TANH)
        finally:
            g.capture_end()
    assert rc == L.E_STATE
    v = C.c_int()
    L.check(lib.vbnn_mlp_get_activation(h, C.byref(v)))
    assert v.value == L.ACT_RELU
    # a net without hidden layers accepts the call, and nothing it computes changes
    one, _, _, _ = build_pair(ctx, [13, 3], 4, 1, "fp32", "weight")
    _, _, Xo, To = data(np.random.RandomState(0), 4, 13, 3)
    one.train_step(Xo, To); one.train_step(Xo, To)
    c0 = one.graph_captures()
    one.set_activation("elu")
    one.train_step(Xo, To)
    assert one.graph_captures() == c0


# ---------------------------------------------------------------- 6. checkpoints
def test_checkpoint_carries_the_activation(ctx):
    """state_dict records the kind and load_state_dict restores it, so a tanh checkpoint loaded into a net built with
    ReLU predicts with tanh; a checkpoint without the key loads as ReLU."""
    sizes, N = [20, 16, 10], 12
    a, _, _, _ = build_pair(ctx, sizes, N, 1, "fp32", "weight", seed=1)
    b, _, _, _ = build_pair(ctx, sizes, N, 1, "fp32", "weight", seed=2)
    a.set_activation("tanh")
    sd = a.state_dict()
    assert sd["activation"] == "tanh"
    b.load_state_dict(sd)
    assert b.activation == "tanh"
    _, _, X, _ = data(np.random.RandomState(0), N, sizes[0], sizes[-1])
    pa, pb = a.predict_outputs(X, n_samples=0), b.predict_outputs(X, n_samples=0)
    assert torch.equal(pa.mean, pb.mean)
    old = {k: v for k, v in sd.items() if k != "activation"}
    b.load_state_dict(old)
    assert b.activation == "relu"
    assert not torch.equal(b.predict_outputs(X, n_samples=0).mean, pa.mean)


# ---------------------------------------------------------------- 7. two GPUs
@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_data_parallel_matches_one_gpu(mode):
    """Two GPUs under torchrun (skipped on one): tools/dp_activation_check.py."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, VBNN_DP=mode)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dp_activation_check.py")],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "ACTIVATION DP CHECK OK" in r.stdout
