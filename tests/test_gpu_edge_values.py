"""GPU tests at degenerate values (pytest -m gpu), element by element against tests/edge_reference.py: all-zero and
tiny input rows on both sides of every 128- and 256-row tile edge, log-variances below ln(FLT_MIN), logit gaps up to
1e4 with tied, and out-of-range targets, and the layer-level ABI at ragged tile edges with scratch regrowth.  Every
comparison is |device - fp64| <= a bound derived from how the device computes the value (edge_reference.py), not a
whole-tensor norm, so one wrong element, row or 32-column chunk fails."""
import math

import numpy as np
import pytest
import torch

import edge_reference as E
from oracle import vbnn_oracle as O
from test_gpu_input_grad import cpu, device_noise, rel

pytestmark = pytest.mark.gpu

EDGE_ROWS = (0, 127, 128, 255, 256, 299)          # both sides of every 128- and 256-row tile edge of N = 300


def f32(a):
    """fp64 array holding fp32 values: what both the device and the oracle are given."""
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def check(name, got, pair, finite_share=0.95):
    ref, bound = pair
    got = np.asarray(got, dtype=np.float64)
    ref = ref.detach().double()
    bound = bound.detach().double()
    assert got.shape == tuple(ref.shape), (name, got.shape, tuple(ref.shape))
    assert np.isfinite(got).all(), (name, "non-finite", np.argwhere(~np.isfinite(got))[:8].tolist())
    v = E.violations(got, ref, bound)
    assert v == [], (name, v)
    share = float(torch.isfinite(bound).double().mean())
    assert share >= finite_share, (name, "bound is +inf on too many elements", share)


class knobs:
    """Set library knobs for a with-block and restore them."""

    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        import vbnn_b200
        self.old = {k: vbnn_b200.knob(k) for k in self.kv}
        for k, v in self.kv.items():
            vbnn_b200.knob(k, v)

    def __exit__(self, *a):
        import vbnn_b200
        for k, v in self.old.items():
            vbnn_b200.knob(k, v)


def pair_knobs(pair, lrt_split=None):
    kv = dict(tc_bn=256, tc_cg=2) if pair else {}
    if lrt_split is not None:
        kv["lrt_split"] = lrt_split
    return knobs(**kv)


def build(ctx, sizes, N, S, precision, reparam, strict=True, vb_output=False, hidden_bias="neg", seed=7,
          lvar_range=(math.log(1e-4), math.log(1e-2))):
    """A device net and a bf16-rounding (or plain) fp64 oracle holding the same fp32 parameters.  hidden_bias: "neg"
    draws biases <= 0 with half of them exactly 0, "pos" draws them in (0.05, 0.25).  The output layer gets a small
    random bias, so that a zero row's logits are a known non-zero vector."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    over = dict(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])],
                S=S, B=30.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.01, reparam=reparam,
                strict_reference=strict, vb_output=vb_output, log=False)
    net = vbnn_b200.MLP(vbnn_b200.default_opt(precision=precision, **over), ctx, max_batch=N)
    oopt = O.default_opt(**over)
    ref = O.MLPOracle(oopt, torch.float64, seed=3, operand_round=O.round_bf16 if precision == "bf16" else None)
    rng = np.random.RandomState(seed)
    layers = ref.vb + [ref.out]
    for k, (gl, ol) in enumerate(zip(net.model, layers)):
        last = k == len(layers) - 1
        if last:
            b = f32(rng.randn(ol.bias.shape[0]) * 0.1)
        elif hidden_bias == "neg":
            b = f32(-rng.uniform(0.0, 0.2, ol.bias.shape[0]) * (rng.rand(ol.bias.shape[0]) < 0.5))
        else:
            b = f32(rng.uniform(0.05, 0.25, ol.bias.shape[0]))
        if isinstance(ol, O.VBLinearOracle):
            mu = f32(rng.randn(ol.O, ol.I) * math.sqrt(2.0 / ol.I))
            lv = f32(rng.uniform(lvar_range[0], lvar_range[1], (ol.O, ol.I)))
            ol.means.copy_(torch.from_numpy(mu)); ol.lvars.copy_(torch.from_numpy(lv))
            gl.set(L.BUF_MEANS, mu); gl.set(L.BUF_LVARS, lv)
        else:
            w = f32(rng.randn(ol.weight.shape[0], ol.weight.shape[1]) * math.sqrt(2.0 / ol.weight.shape[1]))
            ol.weight.copy_(torch.from_numpy(w))
            gl.set(L.BUF_WEIGHT, w)
        ol.bias.copy_(torch.from_numpy(b))
        gl.set(L.BUF_BIAS, b)
        if isinstance(ol, O.VBLinearOracle):
            ol.compute_prior()
            gl.compute_prior()
    return net, ref, oopt


def edge_inputs(rng, N, I, kind):
    """N x I normal rows with EDGE_ROWS replaced: all zero ("zero"), or zero but one feature = 1e-20 ("tiny20": V is
    subnormal in fp32) or 1e-15 ("tiny15": V small but normal)."""
    X = f32(rng.randn(N, I))
    for j, r in enumerate(EDGE_ROWS):
        if r >= N:
            continue
        X[r] = 0.0
        if kind != "zero":
            X[r, (7 * j) % I] = f32(1e-20 if kind == "tiny20" else 1e-15) * (1 if j % 2 == 0 else -1)
    return X


def grads_of(net, k):
    from vbnn_b200 import _lib as L
    m = net.model[k]
    out = {f"gW{k}": cpu(m.get(L.BUF_GRAD_WEIGHT)), f"gB{k}": cpu(m.get(L.BUF_GRAD_BIAS))}
    if m.kind == L.KIND_VB:
        out[f"gS{k}"] = cpu(m.get(L.BUF_GRAD_SUM))
    return out


# ---------------------------------------------------------------- (a), (b): zero and tiny rows through the fused net
ROW_CASES = [
    # precision, reparam, S, lrt_split, pair, rows, hidden_bias, vb_output
    ("fp32", "weight", 2, None, False, "zero", "neg", False),
    ("fp32", "local", 1, None, False, "zero", "neg", True),
    ("fp32", "local", 2, None, False, "zero", "pos", False),
    ("fp32", "local", 2, None, False, "tiny20", "neg", False),
    ("fp32", "local", 1, None, False, "tiny15", "neg", True),
    ("fp32", "weight", 1, None, False, "tiny20", "pos", False),
    ("bf16", "weight", 2, None, False, "zero", "neg", False),
    ("bf16", "weight", 1, None, True, "zero", "pos", False),
    ("bf16", "local", 1, 0, False, "zero", "neg", True),
    ("bf16", "local", 2, 1, False, "zero", "pos", False),
    ("bf16", "local", 2, 2, True, "zero", "neg", False),
    ("bf16", "local", 1, 3, True, "zero", "neg", False),
    ("bf16", "local", 2, 0, True, "tiny20", "neg", False),
    ("bf16", "local", 1, 3, False, "tiny20", "neg", True),
    ("bf16", "local", 2, 1, True, "tiny15", "neg", False),
    ("bf16", "weight", 2, None, False, "tiny20", "neg", False),
]


@pytest.mark.parametrize("precision,reparam,S,lrt_split,pair,rows,hidden_bias,vb_output", ROW_CASES)
def test_edge_rows(ctx, precision, reparam, S, lrt_split, pair, rows, hidden_bias, vb_output):
    """N = 300, 150-136-10 net.  forward_train / backward_update with a chosen dL/dY: logits, dX and every layer's
    gradWeight, gradSum and gradBias within the derived bound element by element and finite.  On a zero row with
    hidden biases <= 0: the hidden pre-activation is b <= 0, so the ReLU mask is 0 (as torch: x > 0), the row's logits
    are the output bias exactly and its dX is exactly 0.  Then the parameters after the update against the oracle
    (existing tolerances), and a fused train_step on the same rows stays finite."""
    from vbnn_b200 import _lib as L
    sizes, N = [150, 136, 10], 300
    bf = precision == "bf16"
    lrt = reparam == "local"
    with pair_knobs(pair, lrt_split):
        net, ref, oopt = build(ctx, sizes, N, S, precision, reparam, strict=False, vb_output=vb_output,
                               hidden_bias=hidden_bias)
        rng = np.random.RandomState(11)
        X = edge_inputs(rng, N, sizes[0], rows)
        G = f32(rng.randn(S, N, sizes[-1]) / N)
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        Xd = torch.from_numpy(X).float().cuda()
        dx = torch.full((N, sizes[0]), float("nan"), device="cuda")
        Y = net.forward_train(Xd).clone()
        net.backward_update(torch.from_numpy(G).float().cuda().contiguous(), dx)
        got = {"logits": cpu(Y), "dX": cpu(dx)}
        for k in range(len(net.model)):
            got.update(grads_of(net, k))
        want = E.mlp_minibatch(ref, torch.from_numpy(X), torch.from_numpy(G), noise, lrt, bf, False, oopt)
        if bf:                                         # the output layer's bias gradient may sum G or its bf16 copy
            last = len(net.model) - 1
            v, e = want[f"gB{last}"]
            want[f"gB{last}"] = (v, e + E.UBF * torch.from_numpy(np.abs(G)).sum(dim=(0, 1)))
        for key in want:
            check(key, got[key], want[key])
        edge = [r for r in EDGE_ROWS if r < N]
        if rows == "zero" and hidden_bias == "neg":
            if not bf:                                 # 0 + b, and in LRT + sqrt(0) * zeta: no rounding at all
                bout = ref.out.bias.numpy()
                assert (got["logits"][:, edge] == bout).all(), "a zero row's logits are not the output bias"
            assert (got["dX"][edge] == 0).all(), "a zero pre-activation must mask the gradient (ReLU: x > 0)"
        ref.update(oopt)
        tol_par = 5e-3 if bf else 2e-4
        for gl, ol in zip(net.model, ref.vb + [ref.out]):
            pairs = ([(L.BUF_MEANS, ol.means), (L.BUF_LVARS, ol.lvars)] if isinstance(ol, O.VBLinearOracle)
                     else [(L.BUF_WEIGHT, ol.weight)]) + [(L.BUF_BIAS, ol.bias)]
            for b, w in pairs:
                g = cpu(gl.get(b))
                assert np.isfinite(g).all(), b
                assert rel(g, w) <= max(tol_par, 1e-4), (b, rel(g, w))
        T = torch.from_numpy(rng.randint(1, sizes[-1] + 1, N).astype(np.float32)).cuda()
        err, acc = net.train_step(Xd, T, grad_input=dx)
        assert math.isfinite(err) and math.isfinite(acc)
        assert torch.isfinite(dx).all()
        for k in range(len(net.model)):
            for key, v in grads_of(net, k).items():
                assert np.isfinite(v).all(), key
        for key, v in net.state_dict().items():
            if isinstance(v, torch.Tensor):
                assert torch.isfinite(v).all(), key


# ---------------------------------------------------------------- (c): log-variances below ln(FLT_MIN)
@pytest.mark.parametrize("strict", [True, False])
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_underflowing_lvars(ctx, precision, reparam, strict):
    """A few log-variances at -90 and -100 (exp underflows fp32: __expf gives 0) in every VB layer.  After one and two
    fused steps every parameter and Adam moment is finite and matches the fp64 oracle at the tolerances of
    test_custom_loss_vs_reference; so do the clamped elements themselves.  compute_vargrads and the 14 layer stats
    stay finite.  (The reference's (1/var_hat - 1/var) * var is inf * 0 = NaN there; the finite limit is -1/(2B).)"""
    from vbnn_b200 import _lib as L
    sizes, N, S = [40, 24, 6], 64, 2
    bf = precision == "bf16"
    lrt = reparam == "local"
    net, ref, oopt = build(ctx, sizes, N, S, precision, reparam, strict=strict, vb_output=True)
    rng = np.random.RandomState(3)
    low = {}
    for k, (gl, ol) in enumerate(zip(net.model, ref.vb_all)):
        lv = ol.lvars.clone()
        idx = [(i % ol.O, (5 * i) % ol.I) for i in range(6)]
        for j, (o, i) in enumerate(idx):
            lv[o, i] = -90.0 if j % 2 == 0 else -100.0
        low[k] = idx
        ol.lvars.copy_(lv); ol.compute_prior()
        gl.set(L.BUF_LVARS, lv.numpy()); gl.compute_prior()
    tol_par = 5e-3 if bf else 2e-4
    tol_adam = 2e-2 if bf else 1e-4
    for it in range(2):
        Xn = f32(rng.randn(N, sizes[0]))
        Tn = rng.randint(1, sizes[-1] + 1, N).astype(np.float64)
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        err, acc = net.train_step(torch.from_numpy(Xn).float().cuda(), torch.from_numpy(Tn).float().cuda())
        assert math.isfinite(err) and math.isfinite(acc), it
        kw = dict(zeta=noise) if lrt else dict(eps=noise)
        O.train_minibatch(ref, torch.from_numpy(Xn), torch.from_numpy(Tn), oopt, **kw)
        for k, (gl, ol) in enumerate(zip(net.model, ref.vb_all)):
            for b, want, t in [(L.BUF_MEANS, ol.means, tol_par), (L.BUF_LVARS, ol.lvars, tol_par),
                               (L.BUF_BIAS, ol.bias, max(tol_par, 1e-4)),
                               (L.BUF_ADAM_M_MU, ol.meanState["m"], tol_adam),
                               (L.BUF_ADAM_V_MU, ol.meanState["v"], tol_adam),
                               (L.BUF_ADAM_M_VAR, ol.varState["m"], tol_adam),
                               (L.BUF_ADAM_V_VAR, ol.varState["v"], tol_adam)]:
                g = cpu(gl.get(b))
                assert np.isfinite(g).all(), (it, k, b)
                assert rel(g, want) <= t, (it, k, b, rel(g, want))
            lvd, lvr = cpu(gl.get(L.BUF_LVARS)), ol.lvars.numpy()
            mvd, mvr = cpu(gl.get(L.BUF_ADAM_M_VAR)), ol.varState["m"].numpy()
            for o, i in low[k]:
                # Adam's first steps are sign-like: the clamped elements move by ~lr_var per step on both sides
                assert abs(lvd[o, i] - lvr[o, i]) <= 1e-4 * abs(lvr[o, i]), (it, k, o, i, lvd[o, i], lvr[o, i])
                assert abs(mvd[o, i] - mvr[o, i]) <= 1e-3 * abs(mvr[o, i]) + 1e-9, (it, k, o, i, mvd[o, i], mvr[o, i])
    for k, gl in enumerate(net.model):
        vleg, vlcg = gl.compute_vargrads()
        assert torch.isfinite(vleg).all() and torch.isfinite(vlcg).all(), k
        for o, i in low[k]:
            assert abs(float(vlcg[o, i]) + 1.0 / (2.0 * oopt["B"])) <= 1e-6 / oopt["B"], (k, float(vlcg[o, i]))
        stats = gl.update(dict(net.opt, log=True))
        assert all(math.isfinite(v) for v in stats.values()), (k, stats)


# ---------------------------------------------------------------- (d): the loss at its edges (k_loss, k_predict)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_loss_edges(ctx, precision):
    """Output weights scaled so that logit gaps run from ~100 to ~1e4; zero rows with zero biases everywhere (the
    mlp.lua initialisation) give exactly tied logits; targets 0 and C+1 on some rows.  The fused step's error,
    accuracy and output-layer gradBias (sum over rows of dL/dY) are compared with fp64 computed from the same logits
    (forward_train at the same step, then abandoned): out-of-range targets add 0, have no -1 in the gradient and never
    count; ties go to the lowest index in k_loss, in k_predict and in the reference."""
    from vbnn_b200 import _lib as L
    sizes, N, S = [32, 24, 5], 256, 1
    C = sizes[-1]
    net, ref, oopt = build(ctx, sizes, N, S, precision, "weight", strict=False)
    for gl, ol in zip(net.model, ref.vb + [ref.out]):
        zb = np.zeros(ol.bias.shape[0])
        gl.set(L.BUF_BIAS, zb); ol.bias.zero_()
    w = cpu(net.model[-1].get(L.BUF_WEIGHT)).astype(np.float64)
    scales = f32(np.geomspace(300.0, 1e4, C))[:, None]
    net.model[-1].set(L.BUF_WEIGHT, f32(w * scales))
    rng = np.random.RandomState(8)
    Xn = f32(rng.randn(N, sizes[0]))
    tied = [0, 1, 127, 128, 200]
    Xn[tied] = 0.0
    Tn = rng.randint(1, C + 1, N).astype(np.float64)
    Tn[[0, 127]] = 1                                       # tied rows: class 1 is the lowest index: correct
    Tn[[1, 128]] = 2                                       # tied rows: not correct
    Tn[[5, 9, 200]] = 0
    Tn[[6, 10, 201]] = C + 1
    X, T = torch.from_numpy(Xn).float().cuda(), torch.from_numpy(Tn).float().cuda()
    step = ctx.get_step()
    Y = net.forward_train(X).clone()
    net.resetGradients()                                  # abandon: no update, no step bump
    assert ctx.get_step() == step
    Yd = torch.from_numpy(cpu(Y[0]).astype(np.float64))
    assert (Yd[tied] == 0).all()
    gaps = (Yd.max(1).values - Yd.min(1).values)
    assert float(gaps.max()) > 1e3 and float(gaps.median()) > 100, (float(gaps.max()), float(gaps.median()))
    # k_predict, before the step's update moves the biases off 0 (a zero row is then no longer tied): ties go to the
    # lowest index, out-of-range targets never count and add 0 to the nll.  predict leaves the step counter alone.
    pr = net.predict(X, n_samples=1, targets=T)
    assert ctx.get_step() == step
    lab = pr.label.cpu().numpy()
    lpb = cpu(pr.logp).astype(np.float64)
    assert (lpb[tied] == lpb[tied][:, :1]).all()          # exactly tied: log p-bar is the same for every class
    assert (lab[tied] == 1).all(), lab[tied]
    valid = (Tn >= 1) & (Tn <= C)
    assert pr.accuracy == pytest.approx(float((lab[valid] == Tn[valid]).sum()) / N * 100.0, abs=1e-4)
    want_nll = -sum(lpb[r, int(Tn[r]) - 1] for r in range(N) if valid[r]) / N
    assert pr.nll == pytest.approx(want_nll, rel=1e-5, abs=1e-6)
    err, acc = net.train_step(X, T)
    rerr, racc, g, logp = E.classnll_device(Yd, torch.from_numpy(Tn))
    # k_loss: lse = mx + __logf(sum __expf(x - mx)); lp = x - lse rounds to u |x| (6e-4 at 1e4: the fp32 loss of
    # precision at large logits, not an error of the kernel)
    # |d lp| <= rounding of x - mx, lse and x - lse (each u |.| <= 2u max|x|), __logf's 2^-21.41 absolute error, and the
    # sum of __expf terms ((2 + 1.173 |x - mx|) ulps, weighted by p: < 3 ulps each) over C terms
    row_err = 8 * E.U32 * Yd.abs().max(1).values + 2.0 ** -20 + 16 * C * E.U32
    e_err = float(row_err.sum()) / N + E.C_ACC * N * E.U32 * abs(rerr)
    assert abs(err - rerr) <= e_err, (err, rerr, e_err)
    assert acc == pytest.approx(racc, abs=1e-4), (acc, racc)
    p = torch.exp(logp)
    e_p = p * row_err[:, None] + E.expf_err(logp)            # __expf(lp): flushed to 0 below FLT_MIN
    e_g = e_p / N
    if precision == "bf16":
        e_g = e_g + E.UBF * g.abs()                         # the gradient operand is bf16; gradBias may sum it
    gb_bound = e_g.sum(0) + E.C_ACC * N * E.U32 * g.abs().sum(0)
    check("gradBias(out)", cpu(net.model[-1].get(L.BUF_GRAD_BIAS)), (g.sum(0), gb_bound))
    # outputs(): the LogSoftMax k_loss wrote, element by element
    lp_bound = row_err[:, None].expand(N, C)
    check("logp", cpu(net.outputs(0, N)), (logp, lp_bound))


# ---------------------------------------------------------------- (e): the layer-level ABI at tile edges
@pytest.mark.parametrize("injected", [False, True])
@pytest.mark.parametrize("precision,pair", [("fp32", False), ("bf16", False), ("bf16", True)])
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("I,Ol", [(300, 257), (8, 129)])
def test_layer_abi_tile_edges(ctx, I, Ol, reparam, precision, pair, injected):
    """One VBLinear(I, O) called with N = 16, then 300, then 129 (scratch regrowth, then a smaller N in the grown
    buffers): updateOutput, updateGradInput and accGradParameters element by element.  Noise is the device's Philox
    (read back with draw_noise: the staged epilogue path) or injected.  Rows 127 and 128 of the larger calls are an
    all-zero row and a row with one feature at 1e-20."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    bf = precision == "bf16"
    lrt = reparam == "local"
    opt = vbnn_b200.default_opt(B=40.0, S=1, mu_init=1, var_init=0.01, precision=precision, reparam=reparam,
                                strict_reference=False, log=False)
    oopt = O.default_opt(B=40.0, S=1, mu_init=1, var_init=0.01, reparam=reparam, strict_reference=False)
    rng = np.random.RandomState(I + Ol)
    mu = f32(rng.randn(Ol, I) * math.sqrt(2.0 / I))
    lv = f32(rng.uniform(math.log(1e-4), math.log(1e-2), (Ol, I)))
    b = f32(rng.randn(Ol) * 0.1)
    with pair_knobs(pair):
        lyr = vbnn_b200.VBLinear(I, Ol, opt, ctx)
        lyr.set(L.BUF_MEANS, mu); lyr.set(L.BUF_LVARS, lv); lyr.set(L.BUF_BIAS, b)
        lyr.compute_prior()
        for call, N in enumerate((16, 300, 129)):
            ol = O.VBLinearOracle(I, Ol, oopt, torch.float64, np.random.RandomState(1),
                                  operand_round=O.round_bf16 if bf else None)
            ol.means.copy_(torch.from_numpy(mu)); ol.lvars.copy_(torch.from_numpy(lv)); ol.bias.copy_(torch.from_numpy(b))
            ol.compute_prior()
            X = f32(rng.randn(N, I))
            if N > 128:
                X[127] = 0.0
                X[128] = 0.0; X[128, call % I] = f32(1e-20)
            G = f32(rng.randn(N, Ol) / N)
            step = ctx.get_step()
            lyr.resetAcc()
            ps = E.LayerPass(ol, bf, strict=False)
            Xd, Gd = torch.from_numpy(X).float().cuda(), torch.from_numpy(G).float().cuda()
            if lrt:
                zeta = f32(rng.randn(N, Ol)) if injected else f32(cpu(lyr.draw_noise(step, call, rows=N)))
                lyr.sample(sample_idx=call)
                Y = lyr.updateOutput(Xd, torch.from_numpy(zeta).float().cuda() if injected else None)
                Yr, eY = ps.forward(ol.q(torch.from_numpy(X)), torch.zeros(N, I, dtype=torch.float64),
                                    torch.from_numpy(zeta))
                eps = None
            else:
                eps = f32(rng.randn(Ol, I)) if injected else f32(cpu(lyr.draw_noise(step, call)))
                if injected:
                    lyr.sample(eps=torch.from_numpy(eps).float().cuda(), sample_idx=call)
                else:
                    lyr.sample(sample_idx=call)
                Y = lyr.updateOutput(Xd)
                ol.sample(torch.from_numpy(eps))
                ps.eW = ps.sample_bound(torch.from_numpy(eps))
                Yr, eY = ps.forward(ol.q(torch.from_numpy(X)), torch.zeros(N, I, dtype=torch.float64))
            check(f"Y[N={N}]", cpu(Y), (Yr, eY))
            dX = lyr.updateGradInput(Xd, Gd)
            lyr.accGradParameters(Xd, Gd, 1.0)
            gi, egi = ps.backward(ol.q(torch.from_numpy(G)), torch.zeros(N, Ol, dtype=torch.float64),
                                  None if eps is None else torch.from_numpy(eps))
            check(f"dX[N={N}]", cpu(dX), (gi, egi))
            ew, es, eb = ps.grad_bounds()
            if bf:
                eb = eb + E.UBF * torch.from_numpy(np.abs(G)).sum(0)
            check(f"gradWeight[N={N}]", cpu(lyr.gradWeight), (ol.gradWeight, ew))
            check(f"gradSum[N={N}]", cpu(lyr.gradSum), (ol.gradSum, es))
            check(f"gradBias[N={N}]", cpu(lyr.gradBias), (ol.gradBias, eb))
