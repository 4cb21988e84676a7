"""GPU tests of vbnn_mlp_predict_outputs / MLP.predict_outputs (pytest -m gpu): the sampled raw outputs against the
fp64 oracle fed the device-drawn noise, every statistic against the fp64 moments of those samples, agreement with
vbnn_mlp_predict, the samples buffer, chunking, cancellation, degenerate log-variances, determinism, side effects,
argument checks, profiling and a full-size run."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import vbnn_oracle as O
from predict_outputs_reference import moments, raw_stack
from predict_reference import predictive
from test_gpu_predict import build_pair, cpu, data, device_noise, rel

pytestmark = pytest.mark.gpu

SIZES = [40, 48, 36]                     # hidden widths before the output layer


def targets(N, K, seed):
    return torch.from_numpy(np.random.RandomState(seed).randn(N, K)).float().cuda()


def check_moments(p, samples, model, y, tol_epi=1e-4):
    """every statistic of p against the fp64 moments() of the samples the call returned"""
    want = moments(samples.double().cpu(), model, None if y is None else y.double().cpu())
    assert rel(cpu(p.mean), want["mean"].numpy()) <= 1e-5
    e = rel(cpu(p.epistemic), want["epistemic"].numpy())
    assert e <= tol_epi or float(want["epistemic"].abs().max()) == 0.0, e
    if model == "gaussian":
        assert rel(cpu(p.aleatoric), want["aleatoric"].numpy()) <= 1e-5
    else:
        assert p.aleatoric is None
    if y is not None:
        assert abs(p.rmse - want["rmse"]) <= 1e-5 * abs(want["rmse"])
        if model == "gaussian":
            assert abs(p.nll - want["nll"]) <= 1e-5 * abs(want["nll"]), (p.nll, want["nll"])
        else:
            assert p.nll is None


# ---------------------------------------------------------------- 1. against the oracle
@pytest.mark.parametrize("model,C", [("raw", 6), ("raw", 1), ("gaussian", 6), ("gaussian", 2)])
@pytest.mark.parametrize("reparam,vb_output", [("weight", False), ("local", False), ("local", True)])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_predict_outputs_vs_oracle(ctx, precision, reparam, vb_output, model, C):
    """T = 5 samples in chunks of S = 2 (the last one ragged) and the MAP pass: the samples against the fp64 oracle fed
    the device-drawn noise (bf16: the reference restating the bf16 operand rounding), every statistic against the
    fp64 moments of the returned samples."""
    sizes, N, S, T = SIZES + [C], 24, 2, 5
    K = C // 2 if model == "gaussian" else C
    bf = precision == "bf16"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, 30.0, precision, reparam, vb_output=vb_output,
                                      operand_round=O.round_bf16 if bf else None)
    tol = 5e-3 if bf else 1e-5
    Xn, _, X, _ = data(N, sizes[0], sizes[-1], 7)
    y = targets(N, K, 8)
    step = ctx.get_step()
    noise = device_noise(net, ref, step, T, N)
    p = net.predict_outputs(X, n_samples=T, model=model, targets=y, return_samples=True)
    assert ctx.get_step() == step
    assert p.samples.shape == (T, N, C)
    kw = dict(zeta_lists=noise) if reparam == "local" else dict(eps_lists=noise)
    want = raw_stack(ref, torch.from_numpy(Xn), n_samples=T, **kw)
    e = rel(cpu(p.samples), want.numpy())
    assert e <= tol, e
    check_moments(p, p.samples, model, y)
    # MAP
    p = net.predict_outputs(X, n_samples=0, model=model, targets=y, return_samples=True)
    assert p.samples.shape == (1, N, C)
    want = raw_stack(ref, torch.from_numpy(Xn), n_samples=0)
    e = rel(cpu(p.samples), want.numpy())
    assert e <= tol, e
    check_moments(p, p.samples, model, y)
    assert float(p.epistemic.abs().max()) == 0.0


# ---------------------------------------------------------------- 2. the samples of predict
def test_same_samples_as_predict(ctx):
    """A classification net at one step: predict's log p-bar is the fp64 average of log_softmax of the samples that
    predict_outputs returns."""
    sizes, N, T = SIZES + [6], 24, 5
    net, _, _, _ = build_pair(ctx, sizes, N, 2, 30.0, "fp32", "local", seed=2)
    _, _, X, _ = data(N, sizes[0], sizes[-1], 3)
    p = net.predict_outputs(X, n_samples=T, return_samples=True)
    pred = net.predict(X, n_samples=T)
    want = predictive(torch.log_softmax(p.samples.double().cpu(), -1))
    assert rel(cpu(pred.logp), want["logp"].numpy()) <= 1e-5


# ---------------------------------------------------------------- 3. the samples buffer changes nothing else
@pytest.mark.parametrize("model", ["raw", "gaussian"])
def test_samples_buffer_changes_nothing_else(ctx, model):
    from vbnn_b200 import _lib as L
    sizes, N, S, T = SIZES + [6], 24, 2, 5
    net, _, _, _ = build_pair(ctx, sizes, N, S, 30.0, "bf16", "local", seed=4)
    _, Tn, X, Tt = data(N, sizes[0], sizes[-1], 5)
    K = 3 if model == "gaussian" else 6
    y = targets(N, K, 6)
    a = net.predict_outputs(X, n_samples=T, model=model, targets=y, return_samples=True)
    with pytest.raises(L.VbnnError) as ei:
        net.outputs(0, n=N)
    assert ei.value.code == L.E_STATE
    b = net.predict_outputs(X, n_samples=T, model=model, targets=y)
    for k in ("mean", "epistemic", "aleatoric"):
        if getattr(a, k) is not None:
            assert torch.equal(getattr(a, k), getattr(b, k)), k
    assert a.nll == b.nll and a.rmse == b.rmse
    # get_outputs after a call without samples: LogSoftMax of the last chunk's samples (t = 4 is its only one)
    out = net.outputs(0, n=N)
    assert float((out - torch.log_softmax(a.samples[T - 1].cpu(), -1)).abs().max()) <= 1e-5
    # a train step after either call leaves the parameters of a twin that never called it
    params = []
    for variant in ("none", "samples", "plain"):
        ctx.set_step(30)
        twin, _, _, _ = build_pair(ctx, sizes, N, S, 30.0, "bf16", "local", seed=4)
        for it in range(2):
            if variant != "none":
                twin.predict_outputs(X, n_samples=3, model=model, targets=y, return_samples=variant == "samples")
            twin.train_step(X, Tt)
        params.append([m.get(bb).numpy().copy() for m in twin.model[:-1] for bb in (L.BUF_MEANS, L.BUF_LVARS)]
                      + [twin.model[-1].get(L.BUF_WEIGHT).numpy().copy()])
    for x, z in zip(params[0], params[1]):
        assert np.array_equal(x, z)
    for x, z in zip(params[0], params[2]):
        assert np.array_equal(x, z)


# ---------------------------------------------------------------- 4. chunking
@pytest.mark.parametrize("model", ["raw", "gaussian"])
def test_predict_outputs_does_not_depend_on_chunking(ctx, model):
    sizes, N, T = SIZES + [6], 24, 4
    _, _, X, _ = data(N, sizes[0], sizes[-1], 9)
    y = targets(N, 3 if model == "gaussian" else 6, 10)
    ps = []
    for S in (1, 4):
        net, _, _, _ = build_pair(ctx, sizes, N, S, 30.0, "fp32", "local", seed=5)
        ps.append(net.predict_outputs(X, n_samples=T, model=model, targets=y))
    a, b = ps
    for k in ("mean", "epistemic", "aleatoric"):
        if getattr(a, k) is not None:
            assert rel(cpu(getattr(a, k)), cpu(getattr(b, k))) <= 1e-6, k
    assert abs(a.rmse - b.rmse) <= 1e-6 * abs(b.rmse)
    if model == "gaussian":
        assert abs(a.nll - b.nll) <= 1e-6 * abs(b.nll)


# ---------------------------------------------------------------- 5. cancellation
def test_cancellation(ctx):
    """Plain output layer's bias at 1e4: outputs near 1e4 whose spread over samples is far smaller.  The epistemic
    variance is positive and within 1e-4 of the fp64 variance of the returned samples."""
    from vbnn_b200 import _lib as L
    sizes, N, T = SIZES + [3], 24, 16
    net, _, _, _ = build_pair(ctx, sizes, N, 4, 30.0, "fp32", "local", seed=6)
    net.model[-1].set(L.BUF_BIAS, np.full(3, 1.0e4))
    _, _, X, _ = data(N, sizes[0], sizes[-1], 11)
    p = net.predict_outputs(X, n_samples=T, return_samples=True)
    f = p.samples.double().cpu()
    want = f.var(0, unbiased=False)
    spread = float(want.sqrt().mean())
    print(f"cancellation: |mean| ~ {float(f.abs().mean()):.1f}, spread ~ {spread:.3g}")
    assert float(f.abs().min()) > 1e3 * spread
    assert float(p.epistemic.min()) > 0.0
    e = float(((p.epistemic.double().cpu() - want).abs() / want).max())
    assert e <= 1e-4, e


# ---------------------------------------------------------------- 6. degenerate Gaussian
@pytest.mark.parametrize("sv", [-100.0, 100.0])
def test_degenerate_gaussian(ctx, sv):
    """Log-variance rows of the plain output layer zeroed, their bias at s = -100 / +100; targets are the MAP means
    of a previous call (y - m = 0 exactly): the MAP nll is 1/2 (log 2 pi + s) K, nothing is NaN."""
    from vbnn_b200 import _lib as L
    sizes, N, K = SIZES + [4], 24, 2
    net, ref, _, _ = build_pair(ctx, sizes, N, 2, 30.0, "fp32", "weight", seed=7)
    w = ref.out.weight.clone()
    w[K:] = 0.0
    net.model[-1].set(L.BUF_WEIGHT, w.numpy())
    net.model[-1].set(L.BUF_BIAS, np.array([0.0, 0.0, sv, sv]))
    _, _, X, _ = data(N, sizes[0], sizes[-1], 12)
    y = net.predict_outputs(X, n_samples=0, model="gaussian").mean.clone()
    p = net.predict_outputs(X, n_samples=0, model="gaussian", targets=y, return_samples=True)
    assert bool((p.samples[0, :, K:] == sv).all())
    want = 0.5 * (math.log(2 * math.pi) + sv) * K
    assert math.isfinite(p.nll) and abs(p.nll - want) <= 1e-5 * abs(want), (p.nll, want)
    assert p.rmse == 0.0
    for k in ("mean", "epistemic", "aleatoric"):
        assert not bool(torch.isnan(getattr(p, k)).any()), k
    assert float(p.aleatoric.min()) >= 0.0
    if sv < 0:
        assert bool(torch.isfinite(p.aleatoric).all())
    # sampled passes over the same head: y - m != 0 now, and at s = -100 (y - m)^2 e^{100} may exceed fp32, which
    # makes nll +inf, never NaN
    q = net.predict_outputs(X, n_samples=3, model="gaussian", targets=y)
    assert not math.isnan(q.nll) and not bool(torch.isnan(q.epistemic).any())
    if sv > 0:
        assert math.isfinite(q.nll)


# ---------------------------------------------------------------- 7. degenerate cases
@pytest.mark.parametrize("model", ["raw", "gaussian"])
def test_one_sample_and_map_have_zero_epistemic(ctx, model):
    sizes, N = SIZES + [6], 24
    K = 3 if model == "gaussian" else 6
    net, _, _, _ = build_pair(ctx, sizes, N, 2, 30.0, "bf16", "local", seed=8)
    _, _, X, _ = data(N, sizes[0], sizes[-1], 13)
    p = net.predict_outputs(X, n_samples=1, model=model, return_samples=True)
    assert float(p.epistemic.abs().max()) == 0.0
    assert torch.equal(p.mean, p.samples[0, :, :K])
    p = net.predict_outputs(X, n_samples=0, model=model, return_samples=True)
    assert float(p.epistemic.abs().max()) == 0.0
    assert torch.equal(p.mean, p.samples[0, :, :K])


# ---------------------------------------------------------------- 8. determinism, no side effects
def test_predict_outputs_is_deterministic_and_has_no_side_effects(ctx):
    from vbnn_b200 import _lib as L
    sizes, N = SIZES + [6], 24
    _, _, X, Tt = data(N, sizes[0], sizes[-1], 10)
    net, _, _, _ = build_pair(ctx, sizes, N, 2, 30.0, "fp32", "weight", seed=6)
    net.train_step(X, Tt)                                   # non-zero gradients and Adam moments
    bufs = [L.BUF_MEANS, L.BUF_LVARS, L.BUF_BIAS, L.BUF_GRAD_WEIGHT, L.BUF_GRAD_SUM, L.BUF_GRAD_BIAS,
            L.BUF_ADAM_M_MU, L.BUF_ADAM_V_MU, L.BUF_ADAM_M_VAR, L.BUF_ADAM_V_VAR]

    def snapshot():
        out = [ctx.get_step()] + [m.t for m in net.model]
        for m in net.model:
            for b in (bufs if m.kind == L.KIND_VB else [L.BUF_WEIGHT, L.BUF_BIAS, L.BUF_GRAD_WEIGHT, L.BUF_GRAD_BIAS]):
                out.append(m.get(b).numpy().copy())
        return out

    y = targets(N, 3, 14)
    before = snapshot()
    p1 = net.predict_outputs(X, n_samples=5, model="gaussian", targets=y, return_samples=True)
    p2 = net.predict_outputs(X, n_samples=5, model="gaussian", targets=y, return_samples=True)
    after = snapshot()
    for a, b in zip(before, after):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    for k in ("mean", "epistemic", "aleatoric", "samples"):
        assert torch.equal(getattr(p1, k), getattr(p2, k)), k
    assert p1.nll == p2.nll and p1.rmse == p2.rmse


# ---------------------------------------------------------------- 9. argument errors
def test_predict_outputs_argument_errors(ctx):
    from vbnn_b200 import _lib as L
    N = 8
    net, _, _, _ = build_pair(ctx, SIZES + [5], N, 2, 30.0, "fp32", "weight", seed=1)
    X = torch.zeros(N + 1, SIZES[0], device="cuda")
    y = torch.zeros(N + 1, 5, device="cuda")
    buf = torch.zeros(2 * (N + 1) * 5 + 4, device="cuda")
    mean = torch.zeros(N, 5, device="cuda")
    f = C.c_float()
    lib = L.lib()
    xp, yp, mp = C.c_void_p(X.data_ptr()), C.c_void_p(y.data_ptr()), C.c_void_p(mean.data_ptr())
    call = lambda *a: lib.vbnn_mlp_predict_outputs(*a)
    RAW, GAU = L.OUTPUT_RAW, L.OUTPUT_GAUSSIAN
    assert call(net.handle, xp, N + 1, 2, RAW, None, None, mp, None, None, None, None) == L.E_INVALID   # N > max_batch
    assert call(net.handle, xp, 0, 2, RAW, None, None, mp, None, None, None, None) == L.E_INVALID
    assert call(net.handle, xp, N, -1, RAW, None, None, mp, None, None, None, None) == L.E_INVALID      # n_samples < 0
    assert call(net.handle, None, N, 2, RAW, None, None, mp, None, None, None, None) == L.E_INVALID     # null X
    assert call(None, xp, N, 2, RAW, None, None, mp, None, None, None, None) == L.E_INVALID
    assert call(net.handle, xp, N, 2, 2, None, None, mp, None, None, None, None) == L.E_INVALID         # unknown model
    assert call(net.handle, xp, N, 2, GAU, None, None, mp, None, None, None, None) == L.E_INVALID       # odd C
    assert call(net.handle, xp, N, 2, RAW, None, None, mp, None, mp, None, None) == L.E_INVALID         # aleatoric, RAW
    assert call(net.handle, xp, N, 2, RAW, yp, None, mp, None, None, C.byref(f), None) == L.E_INVALID   # nll, RAW
    assert call(net.handle, xp, N, 2, RAW, None, None, mp, None, None, None, C.byref(f)) == L.E_INVALID  # rmse, no y
    unaligned = C.c_void_p(buf.data_ptr() + 4)
    assert call(net.handle, xp, N, 2, RAW, None, unaligned, mp, None, None, None, None) == L.E_INVALID
    assert call(net.handle, xp, N, 2, RAW, yp, None, mp, None, None, None, C.byref(f)) == L.VBNN_OK
    with pytest.raises(L.VbnnError):
        net.predict_outputs(X[:N], n_samples=2, model="gaussian")
    with pytest.raises(L.VbnnError):
        net.predict_outputs(X[:N], n_samples=2, model="laplace")
    # even C, GAUSSIAN: nll without targets; an open split step
    net2, _, _, _ = build_pair(ctx, SIZES + [4], N, 2, 30.0, "fp32", "weight", seed=2)
    assert call(net2.handle, xp, N, 2, GAU, None, None, mp, None, None, C.byref(f), None) == L.E_INVALID
    net2.forward_train(X[:N])
    assert call(net2.handle, xp, N, 2, GAU, None, None, mp, None, None, None, None) == L.E_STATE
    net2.resetGradients()
    assert call(net2.handle, xp, N, 2, GAU, yp, None, mp, None, None, C.byref(f), C.byref(f)) == L.VBNN_OK


# ---------------------------------------------------------------- 10. profiling
@pytest.mark.parametrize("model", ["raw", "gaussian"])
def test_predict_outputs_profile_class(ctx, model):
    """Class 8 counts one launch per chunk (T = 5, S = 2: three) with 28 B per (row, mean column, sample) and 12 B
    per (row, log-variance column, sample)."""
    sizes, N, S, T = SIZES + [6], 24, 2, 5
    net, _, _, _ = build_pair(ctx, sizes, N, S, 30.0, "bf16", "local", seed=9)
    _, _, X, _ = data(N, sizes[0], sizes[-1], 15)
    y = targets(N, 3 if model == "gaussian" else 6, 16)
    net.predict_outputs(X, n_samples=1, model=model)                   # allocates the state outside the window
    ctx.profile(True)
    try:
        net.predict_outputs(X, n_samples=T, model=model, targets=y)
        prof = ctx.profile_read()
    finally:
        ctx.profile(False)
    ms, launches, nbytes = prof["predict"]
    want = T * N * (40.0 * 3 if model == "gaussian" else 28.0 * 6)
    assert launches == 3 and nbytes == want and ms > 0, (launches, nbytes, want)


# ---------------------------------------------------------------- 11. full size
def test_predict_outputs_full_size_bf16_lrt(ctx):
    """[1024, 1024, 1024, 2] GAUSSIAN, bf16, local reparameterisation, N = 2048, S = 1."""
    import vbnn_b200
    sizes, N = [1024, 1024, 1024, 2], 2048
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=["mean", "logvar"], S=1, B=100.0,
                                batchSize=N, reparam="local", precision="bf16", var_init=0.01, mu_init=1, log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    _, _, X, _ = data(N, sizes[0], sizes[-1], 17)
    y = targets(N, 1, 18)
    epi = []
    for T in (1, 2, 3):
        p = net.predict_outputs(X, n_samples=T, model="gaussian", targets=y)
        for k in ("mean", "epistemic", "aleatoric"):
            assert bool(torch.isfinite(getattr(p, k)).all()), (T, k)
        assert math.isfinite(p.nll) and math.isfinite(p.rmse)
        epi.append(float(p.epistemic.mean()))
    assert epi[0] == 0.0 and epi[1] > 0.0 and epi[2] > 0.0, epi
    again = net.predict_outputs(X, n_samples=3, model="gaussian", targets=y)
    for k in ("mean", "epistemic", "aleatoric"):
        assert torch.equal(getattr(p, k), getattr(again, k)), k
    assert p.nll == again.nll and p.rmse == again.rmse
