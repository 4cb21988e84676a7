"""GPU tests of the regression criteria of the fused minibatch (pytest -m gpu): vbnn_mlp_set_criterion with
VBNN_CRIT_MSE and VBNN_CRIT_GAUSSIAN_NLL.  The fused step matches the fp64 reference of tests/custom_loss_reference.py
fed the criterion's gradient, matches the split path under the same torch loss with fewer kernels, returns the same
input gradient, handles NaN targets, extreme log-variances and exact zeros, runs through the host pipeline, test, run
and get_outputs, switches criterion without disturbing classification, refuses what it must, is deterministic, learns a
heteroscedastic problem, and holds at BASELINE C3's size with a 500-output Gaussian head."""
import ctypes as C
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from custom_loss_reference import autograd_grad, custom_minibatch
from oracle import vbnn_oracle as O
from regression_reference import closed_form_grad, loss_sum, scalars
from test_gpu_custom_loss import state_tensors
from test_gpu_input_grad import build_pair, cpu, device_noise, rel, snapshot

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reg_data(rng, N, I, K, nan_rows=(), nan_elems=()):
    Xn, yn = rng.randn(N, I), rng.randn(N, K)
    for r in nan_rows:
        yn[r, :] = np.nan
    for r, k in nan_elems:
        yn[r, k] = np.nan
    return Xn, yn, torch.from_numpy(Xn).float().cuda(), torch.from_numpy(yn).float().cuda()


def kcols(crit, C_):
    return C_ // 2 if crit == "gaussian_nll" else C_


# ---------------------------------------------------------------- 1. against the fp64 reference
@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
@pytest.mark.parametrize("vb_output", [False, True])
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_fused_regression_vs_reference(ctx, precision, reparam, S, vb_output, crit):
    """Ragged 37-29-23-8 net, N = 45, a NaN target row and element, two minibatches (the second replays the captured
    graph) against custom_minibatch fed the criterion's fp64 autograd gradient on the device-drawn noise: parameters,
    Adam state and both result scalars at the tolerances of test_custom_loss_vs_reference (the biases at the logits'
    tolerance)."""
    from vbnn_b200 import _lib as L
    sizes, N = [37, 29, 23, 8], 45
    bf = precision == "bf16"
    lrt = reparam == "local"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, precision, reparam, seed=7, strict=False, vb_output=vb_output,
                                      operand_round=O.round_bf16 if bf else None)
    net.set_criterion(crit)
    tol = (5e-3 if lrt else 1e-2) if bf else 1e-5
    tol_par = 5e-3 if bf else 2e-4
    # Adam's v squares the gradient: twice the gradient tolerance, and under GAUSSIAN_NLL in bf16 weight mode 3e-2, where
    # the log-variance gradients 1/2 (1 - q^2) / (N K) cancel and a bf16 flip of G is a larger share of them
    tol_adam = (3e-2 if crit == "gaussian_nll" and not lrt else 2e-2) if bf else 1e-4
    # a bias moves by lr x the column sums of G, which carry G's (the logits') error; the Gaussian log-variance
    # columns sum 1/2 (1 - q^2) terms that nearly cancel, so their relative error is that of G, not of a parameter
    tol_bias = max(tol, 1e-4)
    rng = np.random.RandomState(5)
    K = kcols(crit, sizes[-1])
    for it in range(2):
        Xn, yn, X, y = reg_data(rng, N, sizes[0], K, nan_rows=(3,), nan_elems=((10, 1),))
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        err, mse = net.train_step(X, y)
        Yr, _, _ = custom_minibatch(ref, torch.from_numpy(Xn), autograd_grad(loss_sum(crit, torch.from_numpy(yn))),
                                    noise, lrt, oopt)
        we, wm = scalars(crit, Yr, yn)
        assert abs(err - we) <= tol * abs(we) + 1e-7 and abs(mse - wm) <= tol * abs(wm) + 1e-7, (it, err, we, mse, wm)
        if crit == "mse":
            assert err == mse
        for gl, ol in zip(net.model, ref.vb + [ref.out]):
            if isinstance(ol, O.VBLinearOracle):
                pairs = [(L.BUF_MEANS, ol.means, tol_par), (L.BUF_LVARS, ol.lvars, tol_par),
                         (L.BUF_BIAS, ol.bias, max(tol_par, tol_bias)),
                         (L.BUF_ADAM_M_MU, ol.meanState["m"], tol_adam), (L.BUF_ADAM_V_MU, ol.meanState["v"], tol_adam),
                         (L.BUF_ADAM_M_VAR, ol.varState["m"], tol_adam), (L.BUF_ADAM_V_VAR, ol.varState["v"], tol_adam)]
            else:
                pairs = [(L.BUF_WEIGHT, ol.weight, tol_par), (L.BUF_BIAS, ol.bias, max(tol_par, tol_bias))]
            for b, want, t in pairs:
                e = rel(gl.get(b), want)
                assert e <= t, (it, b, e)


# ---------------------------------------------------------------- 2 + 3. against the split path, with dX
def torch_loss(crit, y):
    """the torch equivalent a user of the split path writes: sum over samples of the per-sample mean criterion"""
    K = y.shape[1]
    if crit == "mse":
        return lambda Y: ((Y - y) ** 2).mean(dim=(1, 2)).sum()
    return lambda Y: (0.5 * (Y[..., K:] + (y - Y[..., :K]) ** 2 * torch.exp(-Y[..., K:]))).mean(dim=(1, 2)).sum()


@pytest.mark.parametrize("precision,reparam,S,vb_output", [("fp32", "weight", 3, False), ("fp32", "local", 2, True),
                                                           ("bf16", "weight", 3, False), ("bf16", "local", 1, True),
                                                           ("bf16", "local", 2, False)])
@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
def test_fused_equals_split(ctx, crit, precision, reparam, S, vb_output):
    """From identical state, three minibatches of train_step against train_step_loss under the torch loss: state within
    1e-6 (fp32) / 1e-3 (bf16, where a different fp32 rounding of G can flip a bf16 one), the error scalar against the
    torch loss / S.  The third minibatch passes grad_input to both: dX agrees likewise.  Launches per step: the library
    enqueues one more for the fused step (k_loss_reg + finalize against k_grad_logits; an LRT output layer's H is
    fused in both), and the split step's torch loss and autograd add more than one kernel of their own."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    sizes, N = [200, 136, 96, 10], 160
    a, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=3, strict=False, vb_output=vb_output)
    b, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=4, strict=False, vb_output=vb_output)
    a.set_criterion(crit)
    tol = 1e-6 if precision == "fp32" else 1e-3
    rng = np.random.RandomState(9)
    K = kcols(crit, sizes[-1])
    dxa, dxb = torch.empty(N, sizes[0], device="cuda"), torch.empty(N, sizes[0], device="cuda")
    leaf = torch.randn(S, N, sizes[-1], device="cuda").requires_grad_(True)
    y0 = torch.randn(N, K, device="cuda")
    torch.autograd.grad(torch_loss(crit, y0)(leaf), leaf)                      # warm up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        (g,) = torch.autograd.grad(torch_loss(crit, y0)(leaf), leaf)
        g.contiguous()
        torch.cuda.synchronize()
    torch_kernels = sum(1 for e in prof.events() if e.device_type == DeviceType.CUDA)
    assert torch_kernels > 1, torch_kernels
    for it in range(3):
        _, _, X, y = reg_data(rng, N, sizes[0], K)
        sd = a.state_dict()
        b.load_state_dict(sd)
        step = sd["step"]
        gi = it == 2
        n0 = a.launch_count()
        err, _ = a.train_step(X, y, grad_input=dxa if gi else None)
        na = a.launch_count() - n0
        ctx.set_step(step)
        n0 = b.launch_count()
        loss = b.train_step_loss(X, torch_loss(crit, y), grad_input=dxb if gi else None)
        nb = b.launch_count() - n0
        assert ctx.get_step() == step + 1
        assert na == nb + 1 and na < nb + torch_kernels, (it, na, nb, torch_kernels)
        assert abs(err - float(loss) / S) <= max(tol, 1e-5) * abs(err), (it, err, float(loss) / S)
        sa, sb = state_tensors(a), state_tensors(b)
        for k in sa:
            e = rel(sa[k], sb[k])
            assert e <= tol, (it, k, e)
        if gi:
            assert np.isfinite(cpu(dxa)).all()
            assert rel(cpu(dxa), cpu(dxb)) <= tol


# ---------------------------------------------------------------- 4. masking, extremes, exact zeros
@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
def test_masking_extremes_and_zeros(ctx, crit):
    """A one-layer fp32 net C -> C with W = I, b = 0, S = 1: its outputs are its inputs and dX is G.  NaN target rows
    and elements give G = 0 there; log-variances of -100 (e^{-s} overflows fp32) and +100 (subnormal), y == m (dm exactly
    0, also at s = -100); every element of G within 1e-5 of the fp64 closed form, and both scalars within 1e-5."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    N, K = 40, 6
    Cn = 2 * K if crit == "gaussian_nll" else K
    opt = vbnn_b200.default_opt(input_size=Cn, hidden=[], classes=[str(i) for i in range(Cn)], S=1, B=30.0,
                                batchSize=N, strict_reference=False, log=False, criterion=crit, outputs=Cn)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.model[0].set(L.BUF_WEIGHT, np.eye(Cn))
    net.model[0].set(L.BUF_BIAS, np.zeros(Cn))
    rng = np.random.RandomState(2)
    Y = rng.randn(N, Cn).astype(np.float32)
    y = rng.randn(N, K).astype(np.float32)
    y[[1, 17], :] = np.nan
    y[5, 2] = y[20, 0] = np.nan
    y[0, :3] = Y[0, :3]                                # y == m
    if crit == "gaussian_nll":
        Y[7, :K] = 0.0
        Y[7, K:] = -100.0
        y[7, :] = np.float32(1e-20) * np.arange(1, K + 1)   # (y - m) e^{-s} = 2.7e23 k: fp32 overflows, q^2 does not
        y[7, 1] = 0.0                                  # y == m under s = -100
        Y[8, K:] = 100.0
        Y[0, K:K + 3] = -100.0
    dx = torch.empty(N, Cn, device="cuda")
    err, mse = net.train_step(torch.from_numpy(Y).cuda(), torch.from_numpy(y).cuda(), grad_input=dx)
    G = cpu(dx)
    Gx = closed_form_grad(crit, Y.astype(np.float64), y.astype(np.float64), N)
    assert np.isfinite(G).all()
    assert (G[[1, 17]] == 0).all() and G[5, 2] == 0 and G[20, 0] == 0
    assert (G[0, :3] == 0).all()
    if crit == "gaussian_nll":
        assert G[7, 1] == 0 and G[5, K + 2] == 0
        assert np.abs(G[7, [0, 2, 3, 4, 5]]).min() > 1e10        # e^{100} / (N K) scale, representable
    np.testing.assert_allclose(G, Gx, rtol=1e-5, atol=1e-5 / (N * K))
    we, wm = scalars(crit, Y[None].astype(np.float64), y.astype(np.float64))
    assert abs(err - we) <= 1e-5 * abs(we) and abs(mse - wm) <= 1e-5 * abs(wm), (err, we, mse, wm)


# ---------------------------------------------------------------- 5. host pipeline
@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
def test_host_pipeline_matches_device_step(ctx, crit):
    """submit_host, submit_host (two in flight), submit_host_u8 and their collects on one net; train_step on device
    copies of the same data (u8 normalised by the same fp32 expression) on a twin from the same state and step: state
    within 1e-6 (the u8 staging kernel squares its own operand for the LRT copy), scalars within 1e-5."""
    sizes, N, S = [64, 48, 32, 6], 50, 2
    a, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    b, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    a.set_criterion(crit); b.set_criterion(crit)
    K = kcols(crit, sizes[-1])
    rng = np.random.RandomState(4)
    X = [torch.from_numpy(rng.randn(N, sizes[0])).float() for _ in range(2)]
    U = torch.from_numpy(rng.randint(0, 256, (N, sizes[0]))).to(torch.uint8)
    mean, std = 33.0, 78.0
    Xu = (U.float() - mean) * np.float32(1.0 / std)
    y = [torch.from_numpy(rng.randn(N, K)).float() for _ in range(3)]
    y[1][4, :] = float("nan")
    ctx.set_step(30)
    want = [a.train_step(X[0].cuda(), y[0].cuda()), a.train_step(X[1].cuda(), y[1].cuda()),
            a.train_step(Xu.cuda(), y[2].cuda())]
    ctx.set_step(30)
    b.submit_host(X[0], y[0]); b.submit_host(X[1], y[1])
    got = [b.collect()]
    b.submit_host_u8(U, y[2], mean, std)
    got += [b.collect(), b.collect()]
    for (e1, m1), (e2, m2) in zip(want, got):
        assert abs(e1 - e2) <= 1e-5 * abs(e1) and abs(m1 - m2) <= 1e-5 * abs(m1)
    (ea, _), (eb, _) = snapshot(a), snapshot(b)
    for p, q in zip(ea, eb):
        assert rel(p, q) <= 1e-6
    e, m = b.train_step_host(X[0], y[0])
    assert math.isfinite(e) and math.isfinite(m)


# ---------------------------------------------------------------- 6. test, run, get_outputs
@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
def test_test_run_and_outputs(ctx, crit):
    """get_outputs after a regression step returns the raw outputs, equal to forward_train's at the same state and
    step; test() over T passes returns the mean over the passes of (loss, MSE of the means) of the outputs that
    predict_outputs samples at the same step (and of the MAP pass under quicktest); run() returns those of its
    single pass."""
    sizes, N, S, T = [30, 24, 8], 20, 2, 5
    a, _, _, _ = build_pair(ctx, sizes, N, S, "fp32", "local", seed=3, strict=False, vb_output=True)
    b, _, _, _ = build_pair(ctx, sizes, N, S, "fp32", "local", seed=3, strict=False, vb_output=True)
    a.set_criterion(crit)
    K = kcols(crit, sizes[-1])
    rng = np.random.RandomState(6)
    _, yn, X, y = reg_data(rng, N, sizes[0], K, nan_elems=((2, 1),))
    ctx.set_step(40)
    a.train_step(X, y)
    outs = [a.outputs(s, N) for s in range(S)]
    ctx.set_step(40)
    Yb = b.forward_train(X).clone()
    b.resetGradients()
    for s in range(S):
        assert torch.equal(outs[s], Yb[s].cpu())
    # test(): T sampled passes, then the MAP pass
    a.opt["testSamples"] = T
    step = ctx.get_step()
    pr = a.predict_outputs(X, n_samples=T, model="raw", return_samples=True)
    assert ctx.get_step() == step
    err, mse = a.test(X, y)
    per = [scalars(crit, cpu(pr.samples[t])[None].astype(np.float64), yn) for t in range(T)]
    we, wm = float(np.mean([p[0] for p in per])), float(np.mean([p[1] for p in per]))
    assert abs(err - we) <= 1e-5 * abs(we) and abs(mse - wm) <= 1e-5 * abs(wm), (err, we, mse, wm)
    a.opt["quicktest"] = True
    pm = a.predict_outputs(X, n_samples=0, model="raw", return_samples=True)
    err, mse = a.test(X, y)
    we, wm = scalars(crit, cpu(pm.samples[0])[None].astype(np.float64), yn)
    assert abs(err - we) <= 1e-5 * abs(we) and abs(mse - wm) <= 1e-5 * abs(wm)
    if crit == "mse":
        assert err == mse
    # run(): one sampled pass with a backward; its scalars are those of the outputs it leaves
    a.resetGradients()
    a.sample()
    err, mse = a.run(X, y)
    we, wm = scalars(crit, a.outputs(0, N).double().numpy()[None], yn)
    assert abs(err - we) <= 1e-5 * abs(we) and abs(mse - wm) <= 1e-5 * abs(wm)


# ---------------------------------------------------------------- 7. switching
def test_switching_keeps_classification_bit_identical(ctx):
    """Net A: ClassNLL steps, MSE steps, ClassNLL again; net B never switches.  Loaded with one state at one step, a
    ClassNLL step of A equals B's bit for bit (exact state and the error / accuracy scalars), and each switch makes
    the step graph re-capture exactly once.  A set to the current criterion changes nothing."""
    from vbnn_b200 import _lib as L
    sizes, N, S = [64, 48, 32, 10], 40, 2
    a, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    b, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False, vb_output=True)
    rng = np.random.RandomState(8)
    Xc = torch.from_numpy(rng.randn(N, sizes[0])).float().cuda()
    Tc = torch.from_numpy(rng.randint(1, 11, N).astype(np.float64)).float().cuda()
    yr = torch.from_numpy(rng.randn(N, sizes[-1])).float().cuda()
    for net in (a, b):
        net.train_step(Xc, Tc); net.train_step(Xc, Tc); net.train_step(Xc, Tc)     # eager, capture, replay
    c0 = a.graph_captures()
    a.set_criterion("mse")
    assert a.graph_captures() == c0
    a.train_step(Xc, yr)
    assert a.graph_captures() == c0 + 1
    a.train_step(Xc, yr)
    assert a.graph_captures() == c0 + 1
    a.set_criterion("mse")
    a.train_step(Xc, yr)
    assert a.graph_captures() == c0 + 1
    a.set_criterion("class_nll")
    v = C.c_int()
    L.check(L.lib().vbnn_mlp_get_criterion(a.handle, C.byref(v)))
    assert v.value == L.CRIT_CLASS_NLL
    sd = b.state_dict()
    a.load_state_dict(sd)
    b.load_state_dict(sd)                                   # (a load resets the priors, which drops the graphs)
    cb = b.graph_captures()
    res = []
    for net in (a, b):
        ctx.set_step(77)
        res.append([net.train_step(Xc, Tc) for _ in range(2)] + [snapshot(net)[0]])
    assert a.graph_captures() == c0 + 2 and b.graph_captures() == cb + 1
    (ra1, ra2, ea), (rb1, rb2, eb) = res
    for x, w in zip(ea, eb):
        assert torch.equal(x, w)
    for p, q in ((ra1, rb1), (ra2, rb2)):
        assert abs(p[0] - q[0]) <= 1e-6 * abs(q[0]) and p[1] == q[1]


# ---------------------------------------------------------------- 8. refusals
def test_refusals(ctx):
    from vbnn_b200 import _lib as L
    lib = L.lib()
    net, _, _, _ = build_pair(ctx, [13, 7, 3], 4, 2, "fp32", "weight")
    h = net.handle
    assert lib.vbnn_mlp_set_criterion(None, 1) == L.E_INVALID
    assert lib.vbnn_mlp_get_criterion(None, C.byref(C.c_int())) == L.E_INVALID
    assert lib.vbnn_mlp_get_criterion(h, None) == L.E_INVALID
    for bad in (-1, 3, 99):
        assert lib.vbnn_mlp_set_criterion(h, bad) == L.E_INVALID
    assert lib.vbnn_mlp_set_criterion(h, L.CRIT_GAUSSIAN_NLL) == L.E_INVALID          # C = 3 is odd
    X = torch.randn(4, 13, device="cuda")
    net.forward_train(X)                                                              # an open split step
    assert lib.vbnn_mlp_set_criterion(h, L.CRIT_MSE) == L.E_STATE
    net.resetGradients()
    net.submit_host(torch.randn(4, 13), torch.ones(4))                                # uncollected minibatch
    assert lib.vbnn_mlp_set_criterion(h, L.CRIT_MSE) == L.E_STATE
    net.collect()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(ctx.stream):
        g.capture_begin(capture_error_mode="thread_local")
        try:
            rc = lib.vbnn_mlp_set_criterion(h, L.CRIT_MSE)
        finally:
            g.capture_end()
    assert rc == L.E_STATE
    v = C.c_int()
    L.check(lib.vbnn_mlp_get_criterion(h, C.byref(v)))
    assert v.value == L.CRIT_CLASS_NLL
    net.set_criterion("mse")
    import vbnn_b200
    with pytest.raises(vbnn_b200.VbnnError):
        net.train_step(X, torch.ones(4, device="cuda"))                                # [N] targets under MSE


# ---------------------------------------------------------------- 9. determinism
@pytest.mark.parametrize("crit", ["mse", "gaussian_nll"])
def test_deterministic(ctx, crit):
    """Two nets built from one seed, three steps each (eager, capture, replay) at the same steps on the same data:
    bit-identical exact state."""
    sizes, N, S = [96, 80, 64, 12], 70, 3
    nets = [build_pair(ctx, sizes, N, S, "bf16", "local", seed=5, strict=False, vb_output=True)[0] for _ in range(2)]
    rng = np.random.RandomState(2)
    data = [reg_data(rng, N, sizes[0], kcols(crit, sizes[-1]), nan_rows=(1,))[2:] for _ in range(3)]
    for net in nets:
        net.set_criterion(crit)
        ctx.set_step(90)
        for X, y in data:
            net.train_step(X, y)
    for p, q in zip(snapshot(nets[0])[0], snapshot(nets[1])[0]):
        assert torch.equal(p, q)


# ---------------------------------------------------------------- 10. learns
def test_heteroscedastic_regression_learns_fused(ctx):
    """The problem of test_heteroscedastic_regression_learns (1-D, noise growing with |x|) trained through the fused
    step under opt.criterion = "gaussian_nll" with opt.outputs = 2, beside a twin from the same state trained through
    the split step under the torch loss at the same steps on the same data: the two loss curves agree within 1e-3 over
    the first 250 minibatches, and the median loss of minibatches 200-250 is well below that of the first 20."""
    import vbnn_b200
    N, S = 256, 2
    # rates for which the curve falls at every Philox step offset tried (0, 1000, 77777): the means' Adam at 1e-3, the
    # output layer's SGD at 1e-4 (its gradient carries e^{-s}, and SGD does not bound the step as Adam does)
    opt = vbnn_b200.default_opt(input_size=1, hidden=[64, 64], outputs=2, criterion="gaussian_nll", S=S, B=2000.0,
                                batchSize=N, mu_init=1, msr_init=True, vb_output=False, reparam="local",
                                strict_reference=False, log=False, seed=5, meanState=dict(learningRate=1e-3),
                                state=dict(learningRate=1e-4))
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    assert net.sizes == [1, 64, 64, 2] and net.criterion == "gaussian_nll"
    net.init_params(seed=4, he_means=True)
    split = vbnn_b200.MLP(dict(opt, criterion="class_nll", classes=["mean", "logvar"]), ctx, max_batch=N)
    split.load_state_dict(net.state_dict())
    g = torch.Generator(device="cuda").manual_seed(0)
    fused, lsplit = [], []

    def loss_fn(y):
        return lambda Y: (0.5 * (Y[..., 1:] + (y - Y[..., :1]) ** 2 * torch.exp(-Y[..., 1:]))).mean(dim=(1, 2)).sum()
    for it in range(250):
        x = torch.rand(N, 1, device="cuda", generator=g) * 4 - 2
        y = torch.sin(2 * x) + (0.05 + 0.3 * x.abs()) * torch.randn(N, 1, device="cuda", generator=g)
        step = ctx.get_step()
        fused.append(net.train_step(x, y)[0])
        ctx.set_step(step)
        lsplit.append(float(split.train_step_loss(x, loss_fn(y))) / S)
    first, late = float(np.median(fused[:20])), float(np.median(fused[200:]))
    print(f"heteroscedastic NLL (fused): median of the first 20 {first:.4f}, of 200-250 {late:.4f}")
    assert rel(fused, lsplit) <= 1e-3, rel(fused, lsplit)
    assert np.isfinite(late) and late < first - 0.3, (first, late)


# ---------------------------------------------------------------- 11. C3 with a Gaussian head
def test_c3_gaussian_head_fused_vs_split(ctx):
    """BASELINE C3's topology (4096-4096x4-1000, N = 8192, bf16, LRT, S = 1) with the 1000 outputs read as a 500-output
    Gaussian head: one fused step against one split step under the torch loss from the same state, parameters and Adam
    state within the bf16 tolerance 1e-3 (measured values printed)."""
    import vbnn_b200
    sizes, N = [4096, 4096, 4096, 4096, 4096, 1000], 8192
    gen = torch.Generator().manual_seed(3)
    X = torch.randn(N, sizes[0], generator=gen).cuda()
    y = torch.randn(N, 500, generator=gen).cuda()
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], outputs=1000, criterion="gaussian_nll",
                                S=1, B=100.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.001,
                                reparam="local", precision="bf16", strict_reference=False, log=False, seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    sd = net.state_dict()
    ctx.set_step(21)
    err, _ = net.train_step(X, y)
    fused = state_tensors(net)
    net.load_state_dict(sd)
    ctx.set_step(21)
    loss = net.train_step_loss(X, torch_loss("gaussian_nll", y))
    split = state_tensors(net)
    e = max(rel(fused[k], split[k]) for k in fused)
    print(f"C3 Gaussian head fused vs split: state max rel {e:.2e}, loss {err:.6f} vs {float(loss):.6f}")
    assert e <= 1e-3 and abs(err - float(loss)) <= 1e-4 * abs(float(loss)), (e, err, float(loss))


@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_data_parallel_regression(mode):
    """Two GPUs under torchrun (skipped on one): tools/dp_regression_check.py."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, VBNN_DP=mode)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dp_regression_check.py")],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "REGRESSION DP CHECK OK" in r.stdout
