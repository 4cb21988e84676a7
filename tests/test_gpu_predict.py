"""GPU tests of vbnn_mlp_predict / MLP.predict (pytest -m gpu): the Bayesian model average against the fp64
reference fed the device-drawn noise, against its own per-sample outputs, against vbnn_mlp_test, across chunkings,
and for determinism, side effects, numerical range and argument checks."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import vbnn_oracle as O
from predict_reference import oracle_predict, predictive

pytestmark = pytest.mark.gpu

TEST_BASE = 1 << 20                      # noise index of test / predict sample 0 (mlp.cu)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def cpu(t):
    return t.detach().float().cpu().numpy()


def build_pair(ctx, sizes, N, S, B, precision, reparam, seed=0, strict=True, vb_output=False, lr_mu=None,
               operand_round=None, dtype=torch.float64):
    """A device net and a CPU oracle holding the same parameters (copy of tests/test_gpu_mlp.py's helper)."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    over = dict(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])],
                S=S, B=B, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.01, reparam=reparam,
                strict_reference=strict, vb_output=vb_output, log=False)
    if lr_mu:
        over["meanState"] = dict(learningRate=lr_mu)
    gopt = vbnn_b200.default_opt(precision=precision, **over)
    net = vbnn_b200.MLP(gopt, ctx, max_batch=N)
    oopt = O.default_opt(**over)
    ref = O.MLPOracle(oopt, dtype, seed=3, operand_round=operand_round)
    rng = np.random.RandomState(seed)
    layers = ref.vb + [ref.out]
    for k, (gl, ol) in enumerate(zip(net.model, layers)):
        if isinstance(ol, O.VBLinearOracle):
            mu = rng.randn(ol.O, ol.I) * math.sqrt(2.0 / ol.I)
            lv = rng.uniform(math.log(1e-4), math.log(1e-2), (ol.O, ol.I))
            ol.means.copy_(torch.from_numpy(mu)); ol.lvars.copy_(torch.from_numpy(lv))
            ol.compute_prior()
            gl.set(L.BUF_MEANS, mu); gl.set(L.BUF_LVARS, lv)
            gl.compute_prior()
        else:
            w = rng.randn(ol.weight.shape[0], ol.weight.shape[1]) * math.sqrt(2.0 / ol.weight.shape[1])
            ol.weight.copy_(torch.from_numpy(w)); ol.bias.zero_()
            gl.set(L.BUF_WEIGHT, w)
    return net, ref, gopt, oopt


def device_noise(net, ref, step, T, N):
    """The noise of test / predict sample t at `step`, per VB layer of the oracle: eps (weight) or zeta (local)."""
    nvb = len(ref.vb_all)
    gidx = lambda k: k if k < len(ref.vb) else len(net.model) - 1
    return [[torch.from_numpy(cpu(net.model[gidx(k)].draw_noise(step, TEST_BASE + t, rows=N)).astype(np.float64))
             for k in range(nvb)] for t in range(T)]


def data(N, I, C, seed):
    rng = np.random.RandomState(seed)
    Xn = rng.randn(N, I)
    Tn = rng.randint(1, C + 1, N).astype(np.float64)
    return Xn, Tn, torch.from_numpy(Xn).float().cuda(), torch.from_numpy(Tn).float().cuda()


def check_against(pred, want, Tn, tol_lp, tol_u, tol_nll):
    assert rel(cpu(pred.logp), want["logp"].numpy()) <= tol_lp
    for k in ("entropy", "expected_entropy", "mutual_info"):
        d = float(np.abs(cpu(getattr(pred, k)) - want[k].numpy()).max())
        assert d <= tol_u, (k, d)
    assert abs(pred.nll - want["nll"]) <= tol_nll * abs(want["nll"])
    # labels: identical wherever the reference's top two classes are not within rounding of each other
    top2 = torch.topk(want["logp"], 2, dim=-1).values
    clear = (top2[:, 0] - top2[:, 1] > 1e-4).numpy()
    lab = pred.label.cpu().numpy()
    assert (lab[clear] == want["label"].numpy()[clear]).all()
    assert abs(pred.accuracy - want["accuracy"]) <= 1e-3 + 100.0 * (~clear).sum() / len(Tn)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("reparam,vb_output", [("weight", False), ("local", False), ("local", True)])
def test_predict_vs_oracle(ctx, precision, reparam, vb_output):
    """T = 5 samples in chunks of S = 2 (2, 2, 1: the last one ragged) and the MAP pass, against the fp64
    reference fed the device-drawn noise (bf16: the reference restating the bf16 operand rounding)."""
    sizes, N, S, T = [40, 48, 36, 6], 24, 2, 5
    bf = precision == "bf16"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, 30.0, precision, reparam, vb_output=vb_output,
                                      operand_round=O.round_bf16 if bf else None)
    tol = (5e-3, 5e-3, 5e-3) if bf else (1e-5, 1e-5, 1e-4)
    Xn, Tn, X, Tt = data(N, sizes[0], sizes[-1], 7)
    step = ctx.get_step()
    noise = device_noise(net, ref, step, T, N)
    pred = net.predict(X, n_samples=T, targets=Tt)
    assert ctx.get_step() == step
    kw = dict(zeta_lists=noise) if reparam == "local" else dict(eps_lists=noise)
    want = oracle_predict(ref, torch.from_numpy(Xn), torch.from_numpy(Tn), n_samples=T, **kw)
    check_against(pred, want, Tn, *tol)
    # MAP (quicktest): n_samples defaults to 0
    net.opt["quicktest"] = True; oopt["quicktest"] = True
    pred = net.predict(X, targets=Tt)
    want = oracle_predict(ref, torch.from_numpy(Xn), torch.from_numpy(Tn))
    check_against(pred, want, Tn, *tol)
    assert float(pred.mutual_info.abs().max()) == 0.0


def test_predict_matches_its_own_sample_outputs(ctx):
    """C = 1000, one chunk of S = T = 4: the fp64 average of the four LogSoftMax outputs get_outputs(s) returns
    afterwards equals what the kernel produced; profile class 8 counts the launch and its bytes."""
    sizes, N, S = [256, 512, 1000], 512, 4
    net, _, _, _ = build_pair(ctx, sizes, N, S, 30.0, "bf16", "local", seed=2)
    _, _, X, Tt = data(N, sizes[0], sizes[-1], 3)
    ctx.profile(True)
    try:
        pred = net.predict(X, n_samples=S, targets=Tt)
        prof = ctx.profile_read()
    finally:
        ctx.profile(False)
    ms, launches, nbytes = prof["predict"]
    assert launches == 1 and nbytes == 20.0 * S * N * sizes[-1] and ms > 0
    stack = torch.stack([net.outputs(s, n=N).double() for s in range(S)])
    want = predictive(stack)
    assert rel(cpu(pred.logp), want["logp"].numpy()) <= 1e-5
    for k in ("entropy", "expected_entropy", "mutual_info"):
        assert float(np.abs(cpu(getattr(pred, k)) - want[k].numpy()).max()) <= 1e-5, k
    assert bool(torch.isfinite(pred.logp).all())


def test_predict_agrees_with_test(ctx):
    """One sample: predict's NLL / accuracy are test()'s error / accuracy and the mutual information is 0.
    MAP: log p-bar is the LogSoftMax of the MAP pass."""
    sizes, N = [40, 48, 36, 6], 20
    net, _, _, _ = build_pair(ctx, sizes, N, 2, 30.0, "fp32", "weight", seed=3)
    _, _, X, Tt = data(N, sizes[0], sizes[-1], 8)
    net.opt["testSamples"] = 1
    e, a = net.test(X, Tt)
    pred = net.predict(X, targets=Tt)
    assert abs(pred.nll - e) <= 1e-6 * abs(e) and abs(pred.accuracy - a) <= 1e-3
    assert float(pred.mutual_info.max()) <= 1e-6
    net.opt["quicktest"] = True
    pred = net.predict(X)
    assert pred.nll is None and pred.accuracy is None
    assert float(np.abs(cpu(pred.logp) - cpu(net.outputs(0, n=N))).max()) <= 1e-6


@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_predict_does_not_depend_on_chunking(ctx, reparam):
    """Nets with S = 1 and S = 4, same parameters, same step: four samples in four chunks or in one."""
    sizes, N, T = [40, 48, 36, 6], 24, 4
    _, _, X, Tt = data(N, sizes[0], sizes[-1], 9)
    preds = []
    for S in (1, 4):
        net, _, _, _ = build_pair(ctx, sizes, N, S, 30.0, "fp32", reparam, seed=5)
        preds.append(net.predict(X, n_samples=T, targets=Tt))
    a, b = preds
    assert rel(cpu(a.logp), cpu(b.logp)) <= 1e-6
    for k in ("entropy", "expected_entropy", "mutual_info"):
        assert rel(cpu(getattr(a, k)), cpu(getattr(b, k))) <= 1e-6, k
    assert abs(a.nll - b.nll) <= 1e-6 * abs(b.nll) and torch.equal(a.label, b.label)


def test_predict_is_deterministic_and_has_no_side_effects(ctx):
    from vbnn_b200 import _lib as L
    sizes, N = [40, 48, 36, 6], 24
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

    before = snapshot()
    p1 = net.predict(X, n_samples=5, targets=Tt)
    p2 = net.predict(X, n_samples=5, targets=Tt)
    after = snapshot()
    for x, y in zip(before, after):
        assert np.array_equal(np.asarray(x), np.asarray(y))
    for k in ("logp", "entropy", "expected_entropy", "mutual_info", "label"):
        assert torch.equal(getattr(p1, k), getattr(p2, k)), k
    assert p1.nll == p2.nll and p1.accuracy == p2.accuracy
    # twin nets train three minibatches from the same step; a predict between them changes nothing
    params = []
    for with_predict in (False, True):
        ctx.set_step(40)
        twin, _, _, _ = build_pair(ctx, sizes, N, 2, 30.0, "fp32", "weight", seed=11)
        for it in range(3):
            twin.train_step(X, Tt)
            if with_predict and it < 2:
                twin.predict(X, n_samples=3, targets=Tt)
        params.append([m.get(b).numpy().copy() for m in twin.model[:-1] for b in (L.BUF_MEANS, L.BUF_LVARS)]
                      + [twin.model[-1].get(L.BUF_WEIGHT).numpy().copy()])
    for x, y in zip(*params):
        assert np.array_equal(x, y)


def test_predict_is_finite_with_huge_logit_gaps(ctx):
    """Output weights scaled so that logits of one row lie hundreds apart: per-sample logp far below -87 (where
    exp underflows in fp32) still gives a finite log p-bar, equal to the fp64 reference."""
    from vbnn_b200 import _lib as L
    sizes, N, T = [40, 48, 36, 6], 24, 3
    net, ref, _, oopt = build_pair(ctx, sizes, N, 3, 30.0, "fp32", "weight", seed=12)
    w = ref.out.weight * 400.0
    ref.out.weight.copy_(w)
    net.model[-1].set(L.BUF_WEIGHT, w.numpy())
    Xn, Tn, X, Tt = data(N, sizes[0], sizes[-1], 13)
    noise = device_noise(net, ref, ctx.get_step(), T, N)
    pred = net.predict(X, n_samples=T, targets=Tt)
    want = oracle_predict(ref, torch.from_numpy(Xn), torch.from_numpy(Tn), eps_lists=noise, n_samples=T)
    assert float(want["logp"].min()) < -200.0
    for k in ("logp", "entropy", "expected_entropy", "mutual_info"):
        assert bool(torch.isfinite(getattr(pred, k)).all()), k
    assert math.isfinite(pred.nll) and pred.nll > 1.0
    assert rel(cpu(pred.logp), want["logp"].numpy()) <= 1e-5
    for k in ("entropy", "expected_entropy", "mutual_info"):
        assert float(np.abs(cpu(getattr(pred, k)) - want[k].numpy()).max()) <= 1e-3, k
    assert abs(pred.nll - want["nll"]) <= 1e-4 * abs(want["nll"])


def test_predict_argument_errors(ctx):
    from vbnn_b200 import _lib as L
    sizes, N = [40, 48, 36, 6], 8
    net, _, _, _ = build_pair(ctx, sizes, N, 2, 30.0, "fp32", "weight", seed=1)
    X = torch.zeros(N + 1, sizes[0], device="cuda")
    Tt = torch.ones(N + 1, device="cuda")
    f = C.c_float()
    lib = L.lib()
    xp, tp = C.c_void_p(X.data_ptr()), C.c_void_p(Tt.data_ptr())
    assert lib.vbnn_mlp_predict(net.handle, xp, N + 1, 2, None, None, None, None, None) == L.E_INVALID   # N > max_batch
    assert lib.vbnn_mlp_predict(net.handle, xp, 0, 2, None, None, None, None, None) == L.E_INVALID
    assert lib.vbnn_mlp_predict(net.handle, xp, N, -1, None, None, None, None, None) == L.E_INVALID     # n_samples < 0
    assert lib.vbnn_mlp_predict(net.handle, None, N, 2, None, None, None, None, None) == L.E_INVALID    # null X
    assert lib.vbnn_mlp_predict(None, xp, N, 2, None, None, None, None, None) == L.E_INVALID
    assert lib.vbnn_mlp_predict(net.handle, xp, N, 2, None, None, None, C.byref(f), None) == L.E_INVALID  # nll, no targets
    assert lib.vbnn_mlp_predict(net.handle, xp, N, 2, tp, None, None, C.byref(f), None) == L.VBNN_OK
    with pytest.raises(L.VbnnError):
        net.predict(X)


def test_predict_full_size_bf16_lrt(ctx):
    """[1024, 1024, 1024, 1000], bf16, local reparameterisation, N = 2048, S = 1 (T > S: one chunk per sample)."""
    import vbnn_b200
    sizes, N = [1024, 1024, 1024, 1000], 2048
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=1, B=100.0, batchSize=N, reparam="local", precision="bf16", var_init=0.01,
                                mu_init=1, log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    _, _, X, Tt = data(N, sizes[0], sizes[-1], 14)
    mi = []
    for T in (1, 2, 3):
        p = net.predict(X, n_samples=T, targets=Tt)
        for k in ("logp", "entropy", "expected_entropy", "mutual_info"):
            assert bool(torch.isfinite(getattr(p, k)).all()), (T, k)
        assert math.isfinite(p.nll) and 0.0 <= p.accuracy <= 100.0
        assert int(p.label.min()) >= 1 and int(p.label.max()) <= sizes[-1]
        mi.append(float(p.mutual_info.mean()))
    assert mi[0] <= 1e-6 and mi[1] > mi[0] and mi[2] > mi[0], mi
    again = net.predict(X, n_samples=3, targets=Tt)
    for k in ("logp", "entropy", "expected_entropy", "mutual_info", "label"):
        assert torch.equal(getattr(p, k), getattr(again, k)), k
    assert p.nll == again.nll
