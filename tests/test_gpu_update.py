"""The fused KL + Adam update (k_update) element by element against fp64 (pytest -m gpu).

Every update is checked from the state read back just before it (tests/update_reference.py), so errors cannot
compound and the bounds stay at a few ulps in fp32 and bf16 mode alike.  Every case starts from a non-trivial state:
random Adam moments, t > 1, gradients mixed in sign and over three decades of scale.

Which test checks each k_update<VEC, STATS, TPB, PK> element by element (VEC: I % 4 == 0; each layer-ABI case runs
its three updates with, without and with diagnostics, so STATS and non-STATS hand var_hat to each other):
  VEC      STATS  256  EMPIRICAL / FIXED / PER_WEIGHT   test_layer_update (9x16, 1000x4096 / 4096x4096 / 7x12)
  VEC      -      256  EMPIRICAL / FIXED / PER_WEIGHT   test_layer_update (the same cases), test_fused_step
  scalar   STATS  256  EMPIRICAL / FIXED / PER_WEIGHT   test_layer_update (1x1, 5x13, 148x4090 / 3x5, 6x14 / 4x15, 148x4097)
  scalar   -      256  EMPIRICAL / FIXED / PER_WEIGHT   test_layer_update (the same cases), test_fused_step (I % 4 != 0 layer)
  VEC      -      128  EMPIRICAL / FIXED / PER_WEIGHT   test_layer_update_coresident (knob upd_coresident)"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import update_reference as R
from test_gpu_edge_values import knobs

pytestmark = pytest.mark.gpu

STATE_BUFS = dict(mu=0, lv=1, m_mu=7, v_mu=8, m_var=9, v_var=10)     # vbnn_b200._lib BUF_* ids


def lib():
    from vbnn_b200 import _lib as L
    return L


def buf(layer, which):
    return layer._view(which).double().clone()


def read_state(layer):
    L = lib()
    st = {k: buf(layer, b) for k, b in STATE_BUFS.items()}
    st.update(gW=buf(layer, L.BUF_GRAD_WEIGHT), gS=buf(layer, L.BUF_GRAD_SUM), bias=buf(layer, L.BUF_BIAS),
              gB=buf(layer, L.BUF_GRAD_BIAS), t=layer.t)
    return st


def check(name, got, pair):
    ref, bound = pair
    got = got.double().to(ref.device)
    bad = ~torch.isfinite(got) | ((got - ref).abs() > bound)
    if bool(bad.any()):
        idx = bad.nonzero()[:6].tolist()
        detail = [(i, float(got[tuple(i)]), float(ref[tuple(i)]), float(bound[tuple(i)])) for i in idx]
        raise AssertionError((name, int(bad.sum()), "of", bad.numel(), detail))
    assert bool(torch.isfinite(bound).all()), (name, "infinite bound")


def layer_opt(layer):
    o = layer.opt
    return dict(B=o["B"], S=o["S"], lr_mu=o["meanState"]["learningRate"], lr_var=o["varState"]["learningRate"],
                lr_bias=o["state"]["learningRate"], beta1=0.9, beta2=0.999, eps=1e-8,
                lrt=o.get("reparam", "weight") == "local")


def f32t(a, dev):
    return torch.from_numpy(np.asarray(a, np.float32)).to(dev)


def set_random_state(layer, rng, t, mu_scale=0.2):
    """Parameters, Adam moments and t of a VB layer: a state several steps into training."""
    L = lib()
    O_, I = layer.outputSize, layer.inputSize
    layer.set(L.BUF_MEANS, rng.randn(O_, I) * mu_scale)
    layer.set(L.BUF_LVARS, rng.uniform(math.log(1e-3), math.log(1e-1), (O_, I)))
    layer.set(L.BUF_ADAM_M_MU, rng.randn(O_, I) * 0.05)
    layer.set(L.BUF_ADAM_V_MU, rng.rand(O_, I) * 1e-2 + 1e-6)
    layer.set(L.BUF_ADAM_M_VAR, rng.randn(O_, I) * 0.05)
    layer.set(L.BUF_ADAM_V_VAR, rng.rand(O_, I) * 1e-2 + 1e-6)
    layer.set(L.BUF_BIAS, rng.randn(O_) * 0.1)
    L.check(L.lib().vbnn_layer_set_t(layer.handle, int(t)))


def set_random_grads(layer, rng):
    L = lib()
    O_, I = layer.outputSize, layer.inputSize
    sc = lambda: 10.0 ** rng.uniform(-2, 1, (O_, I))
    layer.set(L.BUF_GRAD_WEIGHT, rng.randn(O_, I) * sc())
    layer.set(L.BUF_GRAD_SUM, rng.randn(O_, I) * 10 * sc())
    layer.set(L.BUF_GRAD_BIAS, rng.randn(O_))


def make_prior(layer, kind, rng):
    """Set the layer's prior; PER_WEIGHT: the snapshot, then edited arrays (a few means left equal: kl_mu == 0)."""
    L = lib()
    if kind == "fixed":
        layer.set_prior("fixed", 0.05, 0.02)
    elif kind == "per_weight":
        layer.set_prior("per_weight")
        O_, I = layer.outputSize, layer.inputSize
        mu = layer.get(L.BUF_MEANS).numpy()
        pm = mu + rng.randn(O_, I) * 0.05 * (rng.rand(O_, I) < 0.9)
        layer.set(L.BUF_PRIOR_MEANS, pm)
        layer.set(L.BUF_PRIOR_LVARS, layer.get(L.BUF_LVARS).numpy() + rng.randn(O_, I) * 0.5)


def prior_of(layer, kind, terms):
    L = lib()
    if kind == "empirical":
        return R.Prior("empirical", terms=terms)
    if kind == "fixed":
        return R.Prior("fixed", mu0=0.05, var0=0.02)
    return R.Prior("per_weight", pm=buf(layer, L.BUF_PRIOR_MEANS), pl=buf(layer, L.BUF_PRIOR_LVARS))


def check_update(name, layer, st, ref, strict):
    L = lib()
    for k, b in STATE_BUFS.items():
        check(f"{name} {k}", layer._view(b), ref[k])
    check(f"{name} bias", layer._view(L.BUF_BIAS), ref["bias"])
    if strict:
        check(f"{name} stdv", layer._view(L.BUF_STDV), ref["stdv"])
        check(f"{name} mu_sqe", layer._view(L.BUF_MU_SQE), ref["mu_sqe"])


def run_stats_update(layer, stats):
    L = lib()
    if not stats:
        L.check(L.lib().vbnn_layer_update(layer.handle, None))
        return None
    s = L.VbnnStats()
    L.check(L.lib().vbnn_layer_update(layer.handle, C.byref(s)))
    return {f: getattr(s, f) for f, _ in L.VbnnStats._fields_}


def check_stats(name, got, ref):
    for k, (v, e) in ref.items():
        if math.isnan(v):
            assert math.isnan(got[k]), (name, k, got[k])
        else:
            assert abs(got[k] - v) <= e, (name, k, got[k], v, e)


def layer_case(ctx, O_, I, prior_kind, reparam, precision, strict, S, seed, create_bps=None, run_bps=None,
               coresident=False, calls=(True, False, True), check_grads=True):
    """Three vbnn_layer_update calls on one layer, each checked element by element from the state before it."""
    import vbnn_b200
    L = lib()
    rng = np.random.RandomState(seed)
    opt = vbnn_b200.default_opt(B=20.0, S=S, reparam=reparam, precision=precision, strict_reference=strict,
                                var_init=0.01, mu_init=1, log=False)
    with knobs(**({"upd_bps": create_bps} if create_bps else {})):
        layer = vbnn_b200.VBLinear(I, O_, opt, ctx)
        grid = R.update_grid(O_, I, create_bps or 4)
    set_random_state(layer, rng, t=5 + seed % 3)
    make_prior(layer, prior_kind, rng)
    uopt = layer_opt(layer)
    terms = R.PRIOR_CHUNK_TERMS                   # the partials vbnn_layer_set_t / set left behind
    kv = {}
    if run_bps:
        kv["upd_bps"] = run_bps
    if coresident:
        kv["upd_coresident"] = 1
    with knobs(**kv):
        for i, stats in enumerate(calls):
            name = f"{O_}x{I} {prior_kind} {reparam} {precision} strict={strict} S={S} call {i}"
            set_random_grads(layer, rng)
            if check_grads and i == 0:
                # vbnn_layer_grads after compute_prior (var_hat from k_prior_partials' chunks); it rescales the
                # gradients in place, so they are set again for the update
                layer.compute_prior()
                st = read_state(layer)
                outs = {k: layer._new() for k in ("mleg", "mlcg", "vleg", "vlcg")}
                L.check(L.lib().vbnn_layer_grads(layer.handle, *[C.c_void_p(outs[k].data_ptr()) for k in
                                                                 ("mleg", "mlcg", "vleg", "vlcg")]))
                vh = R.var_hat(st["mu"], st["lv"], R.PRIOR_CHUNK_TERMS)
                ref_g = R.grads(st, uopt, prior_of(layer, prior_kind, None), vh)
                for k in outs:
                    check(f"{name} grads {k}", outs[k], ref_g[k])
                layer.set(L.BUF_GRAD_WEIGHT, st["gW"].cpu().numpy())
                layer.set(L.BUF_GRAD_SUM, st["gS"].cpu().numpy())
            st = read_state(layer)
            prior = prior_of(layer, prior_kind, terms)
            ref = R.update(st, uopt, prior)
            got_stats = run_stats_update(layer, stats)
            check_update(name, layer, st, ref, strict)
            if stats:
                check_stats(name, got_stats, R.stats(ref, prior_kind, 0.02))
            assert layer.t == st["t"] + 1
            tpb = 128 if coresident and I % 4 == 0 and not stats else R.TPB
            terms = R.update_terms(O_, I, grid, tpb)
    return layer, opt


# ---------------------------------------------------------------- (a) the layer ABI
LAYER_CASES = [
    # O, I, prior, reparam, precision, strict, S
    (1, 1, "empirical", "weight", "fp32", True, 1),
    (3, 5, "fixed", "local", "bf16", False, 3),
    (7, 12, "per_weight", "weight", "bf16", True, 3),
    (5, 13, "empirical", "local", "fp32", False, 3),
    (6, 14, "fixed", "weight", "fp32", True, 1),
    (4, 15, "per_weight", "local", "fp32", True, 1),
    (9, 16, "empirical", "local", "bf16", True, 1),
    (1000, 4096, "empirical", "local", "bf16", False, 3),       # ~7 quads per thread
    (4096, 4096, "fixed", "local", "bf16", True, 1),            # C3's hidden layer, ~28 quads per thread
    (148, 4097, "per_weight", "weight", "fp32", False, 3),      # 151700 quads: just above 592 x 256
    (148, 4090, "empirical", "weight", "fp32", True, 3),        # 151404: just below
]


@pytest.mark.parametrize("case", LAYER_CASES, ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}-{c[3]}-{c[4]}-s{int(c[5])}-S{c[6]}")
def test_layer_update(ctx, case):
    layer_case(ctx, *case, seed=sum(case[:2]))


@pytest.mark.parametrize("case", [c for c in LAYER_CASES if c[1] % 4 == 0],
                         ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}")
def test_layer_update_coresident(ctx, case):
    """(e) the 128-thread co-resident variant (kl_first for FIXED / PER_WEIGHT) on one GPU: the non-diagnostic calls
    run it, the diagnostic ones the 256-thread STATS variant, and they hand var_hat to each other."""
    layer_case(ctx, *case, seed=3 + case[0], coresident=True, calls=(False, True, False, False), check_grads=False)


# ---------------------------------------------------------------- (b) the GEMM operand copies
@pytest.mark.parametrize("precision,I", [("bf16", 13), ("bf16", 64), ("fp32", 13), ("fp32", 64)])
def test_operand_copies_match_set(ctx, precision, I):
    """After updates, the layer's GEMM operands (bf16 mu / sigma^2 at pitch ld_bf16 from k_update's vector and tail
    stores, or the fp32 sigma^2 copy) equal those vbnn_layer_set makes from the same fp32 state on a twin: the forward
    outputs on the same X and zeta are ==.  The output Linear layer's k_sgd bf16 copy likewise."""
    import vbnn_b200
    L = lib()
    O_, N = 37, 70
    layer, opt = layer_case(ctx, O_, I, "empirical", "local", precision, False, 3, seed=I, check_grads=False)
    twin = vbnn_b200.VBLinear(I, O_, opt, ctx)
    for b in (L.BUF_MEANS, L.BUF_LVARS, L.BUF_BIAS):
        twin.set(b, layer.get(b).numpy())
    rng = np.random.RandomState(1)
    X = f32t(rng.randn(N, I), "cuda")
    Z = f32t(rng.randn(N, O_), "cuda")
    y1, y2 = layer.updateOutput(X, Z).clone(), twin.updateOutput(X, Z).clone()
    assert torch.equal(y1, y2), float((y1 - y2).abs().max())
    # nn.Linear output layer: optim.sgd and its bf16 operand
    lin = vbnn_b200.Linear(I, O_, opt, ctx)
    lin.set(L.BUF_WEIGHT, rng.randn(O_, I))
    lin.set(L.BUF_GRAD_WEIGHT, rng.randn(O_, I))
    lin.set(L.BUF_BIAS, rng.randn(O_))
    lin.set(L.BUF_GRAD_BIAS, rng.randn(O_))
    w, gw = buf(lin, L.BUF_WEIGHT), buf(lin, L.BUF_GRAD_WEIGHT)
    b, gb = buf(lin, L.BUF_BIAS), buf(lin, L.BUF_GRAD_BIAS)
    L.check(L.lib().vbnn_layer_update(lin.handle, None))
    check("linear weight", lin._view(L.BUF_WEIGHT), R.sgd(w, gw, opt["state"]["learningRate"]))
    check("linear bias", lin._view(L.BUF_BIAS), R.sgd(b, gb, opt["state"]["learningRate"]))
    ltwin = vbnn_b200.Linear(I, O_, opt, ctx)
    ltwin.set(L.BUF_WEIGHT, lin.get(L.BUF_WEIGHT).numpy())
    ltwin.set(L.BUF_BIAS, lin.get(L.BUF_BIAS).numpy())
    y1, y2 = lin.updateOutput(X).clone(), ltwin.updateOutput(X).clone()
    assert torch.equal(y1, y2), float((y1 - y2).abs().max())


# ---------------------------------------------------------------- (c) in situ in the fused net
def fused_case(ctx, sizes, N, precision, reparam, prior_kind, vb_output, strict, mode="step", steps=5, seed=0,
               run_bps=None, create_bps=None, no_graph=0):
    """`steps` minibatches of the fused net (eager, capture, replays); before each the state and t of every layer are
    read, after it the gradients, and every VB layer's update and the output layer's SGD are checked."""
    import vbnn_b200
    L = lib()
    rng = np.random.RandomState(seed)
    over = dict(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])], S=2,
                B=50.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.01, reparam=reparam,
                strict_reference=strict, vb_output=vb_output, log=False)
    with knobs(**({"upd_bps": create_bps} if create_bps else {})):
        net = vbnn_b200.MLP(vbnn_b200.default_opt(precision=precision, **over), ctx, max_batch=N)
    bps = create_bps or 4
    for k, m in enumerate(net.model):
        if m.kind == L.KIND_VB:
            set_random_state(m, rng, t=3 + k, mu_scale=math.sqrt(2.0 / m.inputSize))
        else:
            m.set(L.BUF_WEIGHT, rng.randn(m.outputSize, m.inputSize) * math.sqrt(2.0 / m.inputSize))
            m.set(L.BUF_BIAS, rng.randn(m.outputSize) * 0.1)
    if prior_kind != "empirical":
        for k in net.vb_indices:
            make_prior(net.model[k], prior_kind, rng)
    terms = {k: R.PRIOR_CHUNK_TERMS for k in net.vb_indices}
    X = f32t(rng.randn(N, sizes[0]), "cuda")
    T = f32t(rng.randint(1, sizes[-1] + 1, N), "cuda")
    gi = torch.empty(N, sizes[0], dtype=torch.float32, device="cuda") if mode == "grad_input" else None
    kv = dict(no_graph=no_graph)
    if run_bps:
        kv["upd_bps"] = run_bps
    with knobs(**kv):
        for s in range(steps):
            before = [read_state(m) if m.kind == L.KIND_VB else
                      dict(w=buf(m, L.BUF_WEIGHT), b=buf(m, L.BUF_BIAS)) for m in net.model]
            if mode == "backward_update":
                y = net.forward_train(X)
                net.backward_update(f32t(rng.randn(*y.shape) * 10.0 ** rng.uniform(-3, -1, y.shape), "cuda"))
            else:
                net.train_step(X, T, sync=False, grad_input=gi)
            torch.cuda.synchronize()
            for k, m in enumerate(net.model):
                name = f"{sizes} {precision} {reparam} {prior_kind} {mode} step {s} layer {k}"
                st = before[k]
                if m.kind == L.KIND_VB:
                    st.update(gW=buf(m, L.BUF_GRAD_WEIGHT), gS=buf(m, L.BUF_GRAD_SUM), gB=buf(m, L.BUF_GRAD_BIAS))
                    ref = R.update(st, layer_opt(m), prior_of(m, prior_kind, terms[k]))
                    check_update(name, m, st, ref, strict)
                    assert m.t == st["t"] + 1, name
                    terms[k] = R.update_terms(m.outputSize, m.inputSize, R.update_grid(m.outputSize, m.inputSize, bps))
                else:
                    lr = m.opt["state"]["learningRate"]
                    check(f"{name} weight", m._view(L.BUF_WEIGHT), R.sgd(st["w"], buf(m, L.BUF_GRAD_WEIGHT), lr))
                    check(f"{name} bias", m._view(L.BUF_BIAS), R.sgd(st["b"], buf(m, L.BUF_GRAD_BIAS), lr))
    return net


FUSED_CASES = [
    # sizes, N, precision, reparam, prior, vb_output, strict, mode
    ((40, 64, 30, 10), 96, "fp32", "weight", "empirical", False, True, "step"),
    ((40, 64, 30, 10), 96, "fp32", "local", "fixed", True, False, "step"),
    ((37, 64, 48, 10), 96, "bf16", "local", "per_weight", False, True, "step"),     # I % 4 != 0 first layer
    ((48, 64, 32, 10), 96, "bf16", "weight", "empirical", True, False, "backward_update"),
    ((48, 66, 32, 12), 96, "bf16", "local", "empirical", False, True, "grad_input"),  # I % 4 = 2 second layer
]


@pytest.mark.parametrize("case", FUSED_CASES, ids=lambda c: f"{c[2]}-{c[3]}-{c[4]}-vbout{int(c[5])}-{c[7]}")
def test_fused_step(ctx, case):
    fused_case(ctx, *case)


def test_fused_step_c3(ctx):
    """The C3 network bench.py times (4096-4096x4-1000, N = 8192, bf16, local): the grid-stride regime, every thread
    ~28 quads."""
    fused_case(ctx, (4096, 4096, 4096, 4096, 4096, 1000), 8192, "bf16", "local", "empirical", False, False, steps=3)


# ---------------------------------------------------------------- (d) upd_bps changed around a layer's creation
BPS = [(4, 2), (4, 8), (2, None), (8, None), (2, 8)]      # (at creation, while updating: None = the default 4)


@pytest.mark.parametrize("create_bps,run_bps", BPS)
def test_upd_bps_layer(ctx, create_bps, run_bps):
    """var_hat of each update (its diagnostic, and every element through mlcg / vlcg) from the partials the previous
    update wrote: their count is fixed at creation, so the grid that writes them must be too."""
    layer_case(ctx, 4096, 4096, "empirical", "local", "bf16", False, 3, seed=11, create_bps=create_bps,
               run_bps=run_bps or 4, check_grads=False)


@pytest.mark.parametrize("no_graph", [1, 0])
@pytest.mark.parametrize("create_bps,run_bps", [(4, 2), (4, 8), (8, 2)])
def test_upd_bps_fused(ctx, create_bps, run_bps, no_graph):
    fused_case(ctx, (64, 1024, 1024, 10), 128, "fp32", "local", "empirical", False, False, steps=3, seed=2,
               create_bps=create_bps, run_bps=run_bps, no_graph=no_graph)
