"""GPU tests of the split minibatch (pytest -m gpu): vbnn_mlp_forward_train / vbnn_mlp_backward_update and
MLP.forward_train / backward_update / train_step_loss.  Fed the ClassNLL gradient it is the fused step; under other
losses (MSE regression, label-smoothed cross-entropy) it matches the fp64 reference of tests/custom_loss_reference.py
on the device-drawn noise; it holds with the CTA-pair tiles forced, is deterministic, keys its graphs on its buffers,
refuses what the open-step rules refuse, and trains end to end (a conv extractor under a VB head, a heteroscedastic
regression, BASELINE C3 at full size)."""
import copy
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from custom_loss_reference import autograd_grad, custom_minibatch
from oracle import vbnn_oracle as O
from test_gpu_input_grad import build_pair, cpu, data, device_noise, rel, snapshot

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def nll_sum(t1):
    """sum_s of the batch-mean ClassNLL(LogSoftMax(Y_s)): the loss of vbnn_mlp_step.  t1: 1-based targets."""
    return lambda Y: sum(F.nll_loss(F.log_softmax(Y[s], -1), t1.long() - 1) for s in range(Y.shape[0]))


def mse_sum(R):
    return lambda Y: ((Y - R) ** 2).mean(dim=(1, 2)).sum()


def smooth_ce_sum(t1, eps=0.1):
    return lambda Y: sum(F.cross_entropy(Y[s], t1.long() - 1, label_smoothing=eps) for s in range(Y.shape[0]))


def split_step(net, X, loss_fn, dx=None):
    """forward_train, torch loss + autograd on the device, backward_update; returns (logits copy, grad, loss)."""
    Y = net.forward_train(X)
    leaf = Y.detach().clone().requires_grad_(True)
    loss = loss_fn(leaf)
    (g,) = torch.autograd.grad(loss, leaf)
    net.backward_update(g.contiguous(), dx)
    return leaf.detach(), g, loss.detach()


def state_tensors(net):
    from vbnn_b200 import _lib as L
    out = {}
    for k, m in enumerate(net.model):
        out[f"{k}.t"] = torch.tensor([float(m.t)])
        out[f"{k}.bias"] = m.get(L.BUF_BIAS)
        out[f"{k}.gb"] = m.get(L.BUF_GRAD_BIAS)
        out[f"{k}.gW"] = m.get(L.BUF_GRAD_WEIGHT)
        if m.kind == L.KIND_LINEAR:
            out[f"{k}.weight"] = m.get(L.BUF_WEIGHT)
        else:
            for n, b in (("means", L.BUF_MEANS), ("lvars", L.BUF_LVARS), ("gS", L.BUF_GRAD_SUM),
                         ("m_mu", L.BUF_ADAM_M_MU), ("v_mu", L.BUF_ADAM_V_MU), ("m_var", L.BUF_ADAM_M_VAR),
                         ("v_var", L.BUF_ADAM_V_VAR)):
                out[f"{k}.{n}"] = m.get(b)
    return out


# ---------------------------------------------------------------- 1. equals the fused step
@pytest.mark.parametrize("precision,reparam,S,vb_output", [("fp32", "weight", 3, False), ("fp32", "local", 2, True),
                                                           ("bf16", "weight", 3, False), ("bf16", "local", 1, True),
                                                           ("bf16", "local", 2, False)])
def test_split_equals_fused_step(ctx, precision, reparam, S, vb_output):
    """From identical state, K = 3 minibatches of forward_train + torch log_softmax / nll_loss + backward_update match
    train_step: parameters, gradients, Adam state and step counters within 1e-6 (fp32: torch's LogSoftMax against
    k_loss's fast exp / log is the only difference) or 1e-3 (bf16: that difference can flip a bf16 rounding of G).
    The logits equal the fused run's outputs after log_softmax, and the launch count of the two halves is the step's
    minus {k_loss, finalize, [mul_act of an LRT output layer]} plus one k_grad_logits."""
    sizes, N = [200, 136, 96, 10], 160
    a, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=3, strict=False, vb_output=vb_output)
    b, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=4, strict=False, vb_output=vb_output)
    tol = 1e-6 if precision == "fp32" else 1e-3
    delta = 1 + (1 if reparam == "local" and vb_output else 0)     # k_loss + finalize + [mul_act] - k_grad_logits
    rng = np.random.RandomState(9)
    for it in range(3):
        _, _, X, Tt = data(rng, N, sizes[0], sizes[-1])
        sd = a.state_dict()
        b.load_state_dict(sd)
        step = sd["step"]
        n0 = a.launch_count()
        a.train_step(X, Tt)
        na = a.launch_count() - n0
        outs = [a.outputs(s, N) for s in range(S)]
        ctx.set_step(step)
        n0 = b.launch_count()
        Y, _, _ = split_step(b, X, nll_sum(Tt))
        nb = b.launch_count() - n0
        assert ctx.get_step() == step + 1
        assert na - nb == delta, (it, na, nb)
        for s in range(S):
            e = rel(cpu(F.log_softmax(Y[s], -1)), cpu(outs[s]))
            assert e <= 1e-6, (it, s, e)
        sa, sb = state_tensors(a), state_tensors(b)
        for k in sa:
            e = rel(sa[k], sb[k])
            assert e <= tol, (it, k, e)


# ---------------------------------------------------------------- 2. non-NLL losses against the reference
@pytest.mark.parametrize("loss", ["mse", "smooth_ce"])
@pytest.mark.parametrize("vb_output", [False, True])
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_custom_loss_vs_reference(ctx, precision, reparam, S, vb_output, loss):
    """Ragged 37-29-23-7 net, N = 45, two minibatches (the second replays captured graphs), dX requested on the second,
    against the fp64 reference fed the device-drawn noise.  Logits and dX at the tolerances of
    test_grad_input_vs_oracle (fp32 1e-5; bf16 against the bf16-rounding reference 5e-3 LRT / 1e-2 weight mode);
    parameters at those of test_fused_step_vs_oracle (fp32 2e-4, bf16 5e-3: Adam's first steps are sign-like, so an
    element whose gradient nearly cancels may step either way); the Adam moments at twice the gradient tolerance
    (fp32 1e-4, bf16 2e-2: v squares the gradient)."""
    from vbnn_b200 import _lib as L
    sizes, N = [37, 29, 23, 7], 45
    bf = precision == "bf16"
    lrt = reparam == "local"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, precision, reparam, seed=7, strict=False, vb_output=vb_output,
                                      operand_round=O.round_bf16 if bf else None)
    tol = (5e-3 if lrt else 1e-2) if bf else 1e-5
    tol_par = 5e-3 if bf else 2e-4
    tol_adam = 2e-2 if bf else 1e-4
    rng = np.random.RandomState(5)
    dx = torch.empty(N, sizes[0], device="cuda")
    for it in range(2):
        Xn, Tn, X, Tt = data(rng, N, sizes[0], sizes[-1])
        Rn = rng.randn(N, sizes[-1])
        if loss == "mse":
            fn_dev, fn_ref = mse_sum(torch.from_numpy(Rn).float().cuda()), mse_sum(torch.from_numpy(Rn))
        else:
            fn_dev, fn_ref = smooth_ce_sum(Tt), smooth_ce_sum(torch.from_numpy(Tn))
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        dx.fill_(float("nan"))
        Y, _, _ = split_step(net, X, fn_dev, dx if it == 1 else None)
        Yr, _, dXr = custom_minibatch(ref, torch.from_numpy(Xn), autograd_grad(fn_ref), noise, lrt, oopt)
        assert rel(cpu(Y), Yr.numpy()) <= tol, (it, "logits")
        if it == 1:
            assert np.isfinite(cpu(dx)).all()
            assert rel(cpu(dx), dXr.numpy()) <= tol, (it, "dX")
        for gl, ol in zip(net.model, ref.vb + [ref.out]):
            if isinstance(ol, O.VBLinearOracle):
                pairs = [(L.BUF_MEANS, ol.means, tol_par), (L.BUF_LVARS, ol.lvars, tol_par),
                         (L.BUF_BIAS, ol.bias, max(tol_par, 1e-4)),
                         (L.BUF_ADAM_M_MU, ol.meanState["m"], tol_adam), (L.BUF_ADAM_V_MU, ol.meanState["v"], tol_adam),
                         (L.BUF_ADAM_M_VAR, ol.varState["m"], tol_adam), (L.BUF_ADAM_V_VAR, ol.varState["v"], tol_adam)]
            else:
                pairs = [(L.BUF_WEIGHT, ol.weight, tol_par), (L.BUF_BIAS, ol.bias, max(tol_par, 1e-4))]
            for b, want, t in pairs:
                e = rel(gl.get(b), want)
                assert e <= t, (it, b, e)


# ---------------------------------------------------------------- 3. pair tiles
def test_split_pair_tiles(ctx):
    """CTA-pair 256 x 256 tiles forced at 600-552-530-10 with 540 rows (bf16, LRT, S = 2, label-smoothed CE): logits,
    dX and the updated parameters against the default tiling from the same state <= 1e-3, and three forced reruns
    from that state give bitwise-identical logits, dX and bit-reproducible state."""
    import vbnn_b200
    names = ("tc_bn", "tc_cg")
    sizes, N, S = [600, 552, 530, 10], 540, 2
    net, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=2, strict=False)
    sd = net.state_dict()
    _, _, X, Tt = data(np.random.RandomState(1), N, sizes[0], sizes[-1])
    dx = torch.empty(N, sizes[0], device="cuda")
    res = {}
    for forced in (False, True, True, True):
        old = [vbnn_b200.knob(n) for n in names]
        if forced:
            vbnn_b200.knob("tc_bn", 256); vbnn_b200.knob("tc_cg", 2)
        try:
            net.load_state_dict(sd)
            Y, _, _ = split_step(net, X, smooth_ce_sum(Tt), dx)
            exact, _ = snapshot(net)
            res.setdefault(forced, []).append((Y.clone(), dx.clone(), exact))
        finally:
            for n, v in zip(names, old):
                vbnn_b200.knob(n, v)
    (Yd, dxd, ed), = res[False]
    for Yf, dxf, ef in res[True]:
        assert rel(cpu(Yf), cpu(Yd)) <= 1e-3
        assert rel(cpu(dxf), cpu(dxd)) <= 1e-3
        for x, y in zip(ef, ed):
            assert rel(x, y) <= 1e-3
    Y0, dx0, e0 = res[True][0]
    for Yf, dxf, ef in res[True][1:]:
        assert torch.equal(Yf, Y0) and torch.equal(dxf, dx0)
        for x, y in zip(ef, e0):
            assert torch.equal(x, y)


# ---------------------------------------------------------------- 4. determinism and graph keying
def test_graphs_keyed_on_buffers(ctx):
    """Graph keying, observed through vbnn_mlp_graph_captures on a net replaying graphs, with a second net created
    with graphs off (every call eager) as the reference.  Each half runs eagerly on its first call, is captured on the
    second and replayed after; a new logits or gradient buffer re-captures only its own half; the backward with and
    without dX are separate graphs, so alternating them never re-captures; and interleaving with step /
    step_grad_input never re-captures their graphs.  The buffer a call does not name is filled with NaN before it,
    so a graph that read a stale address would show: every logits tensor, dX, result and the final state agree with
    the eager net (<= 1e-5: fp32-atomic gradBias) and the unnamed logits buffer stays untouched."""
    import ctypes as C
    import vbnn_b200
    from vbnn_b200 import _lib as L
    sizes, N, S = [200, 136, 96, 10], 160, 2
    a, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    old = vbnn_b200.knob("no_graph", 1)
    try:
        b, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    finally:
        vbnn_b200.knob("no_graph", old)
    P = lambda t: C.c_void_p(t.data_ptr())
    nan = float("nan")
    # (call, logits buffer, gradient buffer, with dX) -> captures it must add on the graph net
    seq = [("split", 0, 0, False, 0), ("split", 0, 0, False, 2), ("split", 0, 0, False, 0),
           ("split", 0, 1, False, 1),             # new gradient buffer: the backward re-captures
           ("split", 1, 1, False, 1),             # new logits buffer: the forward re-captures
           ("split", 1, 1, True, 0), ("split", 1, 1, True, 1),   # the dX backward: eager, then captured
           ("split", 1, 1, False, 0),             # back to no dX: its graph is still there
           ("step", 0, 0, False, 0), ("step", 0, 0, False, 1), ("split", 1, 1, True, 0), ("step", 0, 0, False, 0),
           ("stepdx", 0, 0, True, 0), ("stepdx", 0, 0, True, 1), ("split", 1, 1, False, 0),
           ("step", 0, 0, False, 0), ("stepdx", 0, 0, True, 0), ("split", 1, 1, True, 0)]
    rng = np.random.RandomState(4)
    batches = [data(rng, N, sizes[0], sizes[-1])[2:] for _ in range(len(seq))]
    traces = []
    for net in (a, b):
        ctx.set_step(50)
        logits = [torch.empty(S, N, sizes[-1], device="cuda") for _ in range(2)]
        grads = [torch.empty(S, N, sizes[-1], device="cuda") for _ in range(2)]
        dx = torch.empty(N, sizes[0], device="cuda")
        trace = []
        for (X, Tt), (call, li, gi, with_dx, new_captures) in zip(batches, seq):
            c0 = net.graph_captures()
            dx.fill_(nan)
            if call != "split":
                trace.append(net.train_step(X, Tt, grad_input=dx if with_dx else None))
            else:
                logits[li].fill_(nan); logits[1 - li].fill_(nan)
                L.check(L.lib().vbnn_mlp_forward_train(net.handle, P(X), N, P(logits[li])))
                Y = logits[li].clone()
                assert bool(torch.isnan(logits[1 - li]).all())         # the other buffer is left as it was
                leaf = Y.requires_grad_(True)
                (g,) = torch.autograd.grad(smooth_ce_sum(Tt)(leaf), leaf)
                grads[gi].copy_(g); grads[1 - gi].fill_(nan)
                L.check(L.lib().vbnn_mlp_backward_update(net.handle, P(grads[gi]), P(dx) if with_dx else None))
                trace.append(Y.detach())
            if with_dx:
                trace.append(dx.clone())
            got = net.graph_captures() - c0
            assert got == (new_captures if net is a else 0), (call, li, gi, with_dx, got)
        torch.cuda.synchronize()
        traces.append(trace)
    for va, vb in zip(*traces):
        if isinstance(va, torch.Tensor):
            assert bool(torch.isfinite(va).all())
            assert rel(cpu(va), cpu(vb)) <= 1e-5
        else:
            assert abs(va[0] - vb[0]) <= 1e-5 * abs(vb[0])
    (ea, qa), (eb, qb) = snapshot(a), snapshot(b)
    for x, y in zip(ea + qa, eb + qb):
        assert rel(x, y) <= 1e-5


def test_split_is_deterministic(ctx):
    """Three split minibatches from one state (eager, capture, replay): bit-identical logits, dX and state."""
    sizes, N, S = [600, 552, 530, 10], 540, 2
    net, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "weight", seed=2, strict=False)
    sd = net.state_dict()
    _, _, X, Tt = data(np.random.RandomState(1), N, sizes[0], sizes[-1])
    dx = torch.empty(N, sizes[0], device="cuda")
    outs = []
    for rep in range(3):
        net.load_state_dict(sd)
        Y, _, _ = split_step(net, X, smooth_ce_sum(Tt), dx)
        outs.append((Y.clone(), dx.clone(), snapshot(net)[0]))
    for Y, d, e in outs[1:]:
        assert torch.equal(Y, outs[0][0]) and torch.equal(d, outs[0][1])
        for x, y in zip(e, outs[0][2]):
            assert torch.equal(x, y)


# ---------------------------------------------------------------- 5. state and argument errors
def test_state_and_argument_errors(ctx):
    import ctypes as C
    import vbnn_b200
    from vbnn_b200 import _lib as L
    sizes, N, S = [13, 7, 3], 4, 2
    net, _, _, _ = build_pair(ctx, sizes, N, S, "fp32", "weight")
    lib = L.lib()
    h = net.handle
    P = lambda t: C.c_void_p(t.data_ptr())
    X = torch.randn(N, 13, device="cuda"); T = torch.ones(N, device="cuda")
    Y = torch.empty(S, N, 3, device="cuda"); G = torch.zeros(S, N, 3, device="cuda")
    res = torch.zeros(2, device="cuda"); dx = torch.empty(N, 13, device="cuda")
    # arguments
    assert lib.vbnn_mlp_forward_train(h, None, N, P(Y)) == L.E_INVALID
    assert lib.vbnn_mlp_forward_train(h, P(X), N, None) == L.E_INVALID
    assert lib.vbnn_mlp_forward_train(h, P(X), 0, P(Y)) == L.E_INVALID
    X5 = torch.randn(N + 1, 13, device="cuda"); Y5 = torch.empty(S, N + 1, 3, device="cuda")
    assert lib.vbnn_mlp_forward_train(h, P(X5), N + 1, P(Y5)) == L.E_INVALID
    Yb = torch.empty(S * N * 3 + 1, device="cuda")
    assert lib.vbnn_mlp_forward_train(h, P(X), N, C.c_void_p(Yb.data_ptr() + 4)) == L.E_INVALID   # misaligned
    assert lib.vbnn_mlp_backward_update(h, P(G), None) == L.E_STATE                              # no open step
    # the open step refuses everything that enqueues work, except backward_update and reset_gradients
    net.train_step(X, T)                                                   # outputs() works after a step
    net.outputs(0, N)
    step = ctx.get_step()
    assert lib.vbnn_mlp_forward_train(h, P(X), N, P(Y)) == L.VBNN_OK
    assert lib.vbnn_mlp_backward_update(h, None, None) == L.E_INVALID
    f = C.c_float()
    refused = [
        lib.vbnn_mlp_forward_train(h, P(X), N, P(Y)),
        lib.vbnn_mlp_step(h, P(X), P(T), N, P(res)),
        lib.vbnn_mlp_step_grad_input(h, P(X), P(T), N, P(res), P(dx)),
        lib.vbnn_mlp_test(h, P(X), P(T), N, 1, C.byref(f), C.byref(f)),
        lib.vbnn_mlp_predict(h, P(X), N, 1, None, None, None, None, None),
        lib.vbnn_mlp_run(h, P(X), P(T), N, 0, None, None),
        lib.vbnn_mlp_sample(h, 0),
        lib.vbnn_mlp_update(h),
        lib.vbnn_mlp_calc_lc(h, C.byref(f)),
        lib.vbnn_mlp_init_params(h, C.c_uint64(1), 0),
        lib.vbnn_mlp_get_outputs(h, 0, P(torch.empty(N, 3))),
        lib.vbnn_mlp_sync_replicas(h),
    ]
    assert all(r == L.E_STATE for r in refused), refused
    with pytest.raises(vbnn_b200.VbnnError) as e:
        net.submit_host(torch.randn(N, 13), torch.ones(N))
    assert e.value.code == L.E_STATE
    # Python argument checks of backward_update (the step stays open through them)
    net._open_n = N
    for bad in (torch.zeros(S, N, 4, device="cuda"), torch.zeros(S, N, 3, device="cuda", dtype=torch.float64),
                torch.zeros(S, N, 3), torch.zeros(3, N, S, device="cuda").transpose(0, 2)):
        with pytest.raises(vbnn_b200.VbnnError) as e:
            net.backward_update(bad)
        assert e.value.code == L.E_INVALID
    with pytest.raises(vbnn_b200.VbnnError) as e:
        net.backward_update(G, grad_input=torch.zeros(N, 12, device="cuda"))
    assert e.value.code == L.E_INVALID
    # reset_gradients abandons the step: no update, the counter stays, and train_step works afterwards
    means = net.model[0].get(L.BUF_MEANS)
    net.resetGradients()
    assert ctx.get_step() == step
    assert torch.equal(net.model[0].get(L.BUF_MEANS), means)
    assert lib.vbnn_mlp_backward_update(h, P(G), None) == L.E_STATE
    net.train_step(X, T)
    assert ctx.get_step() == step + 1
    # get_outputs after forward_train refuses until the next step / test / predict
    net.forward_train(X)
    net.backward_update(G)
    assert ctx.get_step() == step + 2
    assert lib.vbnn_mlp_get_outputs(h, 0, P(torch.empty(N, 3))) == L.E_STATE
    net.test(X, T)
    net.outputs(0, N)
    # forward_train waits for the host pipeline to be collected
    net.submit_host(torch.randn(N, 13), torch.ones(N))
    assert lib.vbnn_mlp_forward_train(h, P(X), N, P(Y)) == L.E_STATE
    net.collect()
    net.forward_train(X)
    net.backward_update(G)
    # train_step_loss abandons the step when the loss raises
    step = ctx.get_step()
    with pytest.raises(ZeroDivisionError):
        net.train_step_loss(X, lambda y: 1 / 0)
    assert ctx.get_step() == step
    loss = net.train_step_loss(X, nll_sum(T))
    assert loss.is_cuda and ctx.get_step() == step + 1


# ---------------------------------------------------------------- 6. end to end
def test_convnet_head_smoothed_ce(ctx):
    """BASELINE C4's shape: a torch conv extractor under MLP(256-100-10, vb_output = 1), fp32, weight mode, S = 2,
    trained under label-smoothed CE through train_step_loss(grad_input=g): g and the conv parameter gradients after
    feats.backward(g) equal autograd through the same extractor with the head in fp64 on the same sampled weights
    (<= 1e-5 / 1e-4 relative)."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    torch.manual_seed(0)
    N, Cn, S = 64, 10, 2
    conv = torch.nn.Sequential(torch.nn.Conv2d(3, 16, 5), torch.nn.ReLU(), torch.nn.MaxPool2d(2),
                               torch.nn.Conv2d(16, 16, 5), torch.nn.ReLU(), torch.nn.MaxPool2d(2),
                               torch.nn.Flatten(), torch.nn.Linear(16 * 5 * 5, 256), torch.nn.ReLU()).cuda()
    conv_ref = copy.deepcopy(conv)
    opt = vbnn_b200.default_opt(input_size=256, hidden=[100], classes=[str(i) for i in range(Cn)], S=S, B=50.0,
                                batchSize=N, mu_init=1, var_init=0.01, vb_output=True, strict_reference=False,
                                log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    x = torch.randn(N, 3, 32, 32, device="cuda")
    t = torch.randint(0, Cn, (N,), device="cuda")
    step = ctx.get_step()
    W = [[(m.get(L.BUF_MEANS).double() + torch.exp(0.5 * m.get(L.BUF_LVARS).double()) *
           m.draw_noise(step, s).double().cpu()).cuda() for m in net.model] for s in range(S)]
    b = [m.get(L.BUF_BIAS).double().cuda() for m in net.model]
    feats = conv(x)
    g = torch.empty(N, 256, device="cuda")
    net.train_step_loss(feats.detach(), smooth_ce_sum(t.float() + 1), grad_input=g)
    feats.backward(g)
    f64 = feats.detach().double().requires_grad_(True)
    loss = sum(F.cross_entropy(torch.relu(f64 @ W[s][0].t() + b[0]) @ W[s][1].t() + b[1], t, label_smoothing=0.1)
               for s in range(S))
    loss.backward()
    assert rel(cpu(g), f64.grad.cpu().numpy()) < 1e-5
    conv_ref(x).backward(f64.grad.float())
    for p, q in zip(conv.parameters(), conv_ref.parameters()):
        assert rel(cpu(p.grad), cpu(q.grad)) < 1e-4


def test_heteroscedastic_regression_learns(ctx):
    """C = 2 outputs read as (mean, log-variance) under the Gaussian NLL 0.5 (log var + (y - mean)^2 / var) on a
    seeded 1-D regression whose noise grows with |x|: the mean loss of the last 20 minibatches is well below that of
    the first 20."""
    import vbnn_b200
    N, S = 256, 2
    opt = vbnn_b200.default_opt(input_size=1, hidden=[64, 64], classes=["mean", "logvar"], S=S, B=2000.0,
                                batchSize=N, mu_init=1, msr_init=True, vb_output=False, reparam="local",
                                strict_reference=False, log=False, seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    g = torch.Generator(device="cuda").manual_seed(0)

    def loss_fn(y_true):
        def fn(Y):
            mean, logvar = Y[..., 0], Y[..., 1]
            return (0.5 * (logvar + (y_true - mean) ** 2 * torch.exp(-logvar))).mean(dim=1).sum()
        return fn
    losses = []
    for it in range(300):
        x = torch.rand(N, 1, device="cuda", generator=g) * 4 - 2
        y = torch.sin(2 * x[:, 0]) + (0.05 + 0.3 * x[:, 0].abs()) * torch.randn(N, device="cuda", generator=g)
        losses.append(net.train_step_loss(x, loss_fn(y)))
    losses = torch.stack(losses).cpu() / S
    first, last = float(losses[:20].mean()), float(losses[-20:].mean())
    print(f"heteroscedastic NLL: first 20 {first:.4f}, last 20 {last:.4f}")
    assert np.isfinite(last) and last < first - 0.3, (first, last)


def test_c3_full_size_split_vs_fused(ctx):
    """BASELINE C3 at its exact size (4096-4096x4-1000, N = 8192, bf16, LRT, S = 1): one split minibatch under torch
    ClassNLL against one fused step from the same state: logits after log_softmax, parameters and Adam state within
    the bf16 tolerance 1e-3 (measured values printed)."""
    import vbnn_b200
    sizes, N = [4096, 4096, 4096, 4096, 4096, 1000], 8192
    gen = torch.Generator().manual_seed(3)
    X = torch.randn(N, sizes[0], generator=gen).cuda()
    T = torch.randint(1, sizes[-1] + 1, (N,), generator=gen).float().cuda()
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=1, B=100.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.001,
                                reparam="local", precision="bf16", strict_reference=False, log=False, seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    sd = net.state_dict()
    ctx.set_step(21)
    net.train_step(X, T)
    lp = net.outputs(0, N)
    fused = state_tensors(net)
    net.load_state_dict(sd)
    ctx.set_step(21)
    Y, _, _ = split_step(net, X, nll_sum(T))
    e_lp = rel(cpu(F.log_softmax(Y[0], -1)), cpu(lp))
    split = state_tensors(net)
    e = max(rel(fused[k], split[k]) for k in fused)
    print(f"C3 split vs fused: logp rel {e_lp:.2e}, state max rel {e:.2e}")
    assert e_lp <= 1e-6 and e <= 1e-3, (e_lp, e)


@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_data_parallel_split(mode):
    """Two GPUs under torchrun (skipped on one): each rank's split step under a global-mean MSE matches one GPU
    stepping the whole minibatch (tools/dp_custom_loss_check.py)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, VBNN_DP=mode)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dp_custom_loss_check.py")],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "CUSTOM LOSS DP CHECK OK" in r.stdout
