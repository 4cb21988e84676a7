"""GPU tests of the tcgen05 GEMMs where each persistent CTA (or CTA pair) runs several work units (pytest -m gpu).

From its second unit on, a CTA carries its pipeline state from tile to tile: the smem ring's stage and phase, the
TMEM accumulator ring, the CLC response ring and the band position of decode_tile.  A stale accumulator, a phase off
by one or a unit decoded into the wrong (m, n, z) shows only there, so every case here asserts at least 3 units per
resident slot (tests/work_units.py) for the GEMMs it targets.

Operands are small integers (ternary inputs, dL/dY and sparse means, integer biases) and the log-variances flush
sigma to 0.  Every partial sum is then an integer below 2^24, exact in fp32 in any order, tile shape, schedule or
K-split, so logits, dX and every gradWeight and gradBias must equal plain fp64 bit for bit (== on the whole tensor;
tests/edge_reference.py, exactness rule).  The fp64 reference runs on the device; it asserts the 2^24 condition on
every contraction.  Each knob of csrc/knobs.h that changes a GEMM's tiles, schedule or form runs at a shape where
that GEMM is multi-wave.  A net captures its step graphs on the second call, so each knob setting builds a fresh
net and calls it once (eagerly)."""
import math

import numpy as np
import pytest
import torch

import edge_reference as E
from oracle import vbnn_oracle as O
from test_gpu_edge_values import check, knobs
from work_units import per_slot

pytestmark = pytest.mark.gpu

SIGMA0 = -300.0                      # lvars: __expf flushes sigma and sigma^2 to 0
SIGMA10 = float(np.float32(-10.0 * math.log(2.0)))   # lvars: sigma^2 = 2^-10 exactly after the bf16 store
PAIR = dict(tc_bn=256, tc_cg=2)
SINGLE = dict(tc_bn=128, tc_cg=1)
DUAL_PAIR = dict(tc_bn=128, tc_cg=2)  # the 256 x 128 pair form of the dual (LRT) GEMMs


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def multiwave(what, M, N, tiles, batch=1, z_once=False):
    """Assert >= 3 units per resident slot on every tile shape in `tiles` ((bn, cg) pairs)."""
    for bn, cg in tiles:
        u = per_slot(M, N, bn, cg, sms(), batch, z_once)
        assert u >= 3.0, (what, M, N, (bn, cg), u)


def tern(shape, density, gen):
    """Ternary {-1, 0, 1} with P(non-zero) = density, fp64 on the device."""
    r = torch.rand(shape, generator=gen, device="cuda", dtype=torch.float64)
    s = torch.randint(0, 2, shape, generator=gen, device="cuda").double() * 2 - 1
    return torch.where(r < density, s, torch.zeros_like(s))


def same(name, got, want):
    """got (device, fp32) == want (fp64) on every element; reports the first mismatches."""
    got = got.detach().double()
    assert got.shape == want.shape, (name, tuple(got.shape), tuple(want.shape))
    bad = ~(got == want)
    if bool(bad.any()):
        idx = bad.nonzero()[:6].tolist()
        raise AssertionError((name, int(bad.sum()), [(i, float(got[tuple(i)]), float(want[tuple(i)])) for i in idx]))


def within(name, got, want, bound):
    got = got.detach().double()
    bad = ~torch.isfinite(got) | ((got - want).abs() > bound)
    if bool(bad.any()):
        idx = bad.nonzero()[:6].tolist()
        raise AssertionError((name, int(bad.sum()), [(i, float(got[tuple(i)]), float(want[tuple(i)]),
                                                      float(bound[tuple(i)])) for i in idx]))


# ---------------------------------------------------------------- (a) the raw GEMM
RAW = [
    # name, M, N, K, batch, a_kmajor, b_kmajor, B shared by the batch
    ("fwd ragged", 2000, 1960, 200, 4, 1, 1, False),
    ("dx ragged, shared B", 2000, 1960, 200, 4, 1, 0, True),
    ("dW ragged", 2000, 1960, 200, 4, 0, 0, False),
    ("C3 fwd", 8192, 4096, 4096, 1, 1, 1, False),
    ("C3 dx", 8192, 4096, 4096, 1, 1, 0, False),
    ("C3 dW", 4096, 4096, 8192, 1, 0, 0, False),
    ("C3 out fwd", 8192, 1000, 4096, 1, 1, 1, False),
]
RAW_KNOBS = [{}, SINGLE, PAIR, dict(tc_clc=0), dict(tc_clc=0, **SINGLE), dict(tc_gm=1), dict(tc_gm=3),
             dict(tc_staged=0), dict(tc_l2hint=1)]


@pytest.mark.parametrize("name,M,N,K,batch,ak,bk,shared", RAW, ids=[r[0] for r in RAW])
def test_raw_gemm_multiwave_exact(ctx, name, M, N, K, batch, ak, bk, shared):
    """vbnn_gemm_bf16 on ternary operands in the step's three operand-major combinations, into a NaN canvas with guard
    rows and pitch columns: the whole output == fp64 and every canary left NaN, under each tile shape and schedule
    knob.  The C3 output layer's GEMM (N = 1000) has 1.7 units per pair slot; every other case >= 3 on both tiles."""
    import ctypes as C
    from vbnn_b200 import _lib as L
    multiwave(name, M, N, [(128, 1)] if N == 1000 else [(128, 1), (256, 2)], batch)
    g = torch.Generator(device="cuda").manual_seed(M + N + K + batch + 2 * ak + bk)
    A = tern((batch, M, K), 0.5, g)
    B = tern((1 if shared else batch, N, K), 0.5, g)
    want = torch.matmul(A, B.transpose(1, 2))
    assert float(torch.matmul(A.abs(), B.abs().transpose(1, 2)).max()) < E.EXACT
    r8 = lambda v: (v + 7) // 8 * 8
    # device layouts: K-major [rows x K] or MN-major [K x rows], each row padded to a multiple of 8 elements
    def lay(T, kmajor, rows):
        ld = r8(K) if kmajor else r8(rows)
        D = torch.zeros(T.shape[0], *((rows, ld) if kmajor else (K, ld)), dtype=torch.bfloat16, device="cuda")
        if kmajor:
            D[:, :, :K] = T.bfloat16()
        else:
            D[:, :, :rows] = T.transpose(1, 2).bfloat16()
        return D, ld, D.shape[1] * ld
    Ad, lda, sA = lay(A, ak, M)
    Bd, ldb, sB = lay(B, bk, N)
    if shared:
        sB = 0
    ldd, guard = N + 12, 64
    for kv in RAW_KNOBS:
        with knobs(**kv):
            buf = torch.full((batch, M + 2 * guard, ldd), float("nan"), device="cuda")
            D = buf[:, guard:guard + M, :]
            L.check(L.lib().vbnn_gemm_bf16(ctx.handle, C.c_void_p(Ad.data_ptr()), lda, ak, C.c_void_p(Bd.data_ptr()),
                                           ldb, bk, C.c_void_p(D[0].data_ptr()), ldd, M, N, K, batch, sA, sB,
                                           (M + 2 * guard) * ldd))
            ctx.synchronize()
            assert bool(buf[:, :guard].isnan().all() and buf[:, guard + M:].isnan().all()), (name, kv, "guard rows")
            assert bool(D[:, :, N:].isnan().all()), (name, kv, "pitch columns")
            same(f"{name} {kv}", D[:, :, :N], want)
        del buf, D


# ---------------------------------------------------------------- the fused net
def make_params(sizes, dens_mu, gen):
    """Ternary means / weights of density dens_mu and integer biases in [-2, 2], per layer (fp64, device)."""
    out = []
    for I, O_ in zip(sizes[:-1], sizes[1:]):
        W = tern((O_, I), dens_mu, gen)
        b = torch.randint(-2, 3, (O_,), generator=gen, device="cuda").double()
        out.append((W, b))
    return out


def build_net(ctx, sizes, N, S, reparam, vb_output, params, lvar=SIGMA0):
    import vbnn_b200
    from vbnn_b200 import _lib as L
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=list(sizes[1:-1]),
                                classes=[str(i) for i in range(sizes[-1])], S=S, B=30.0, batchSize=N,
                                testBatchSize=N, mu_init=1, var_init=0.01, reparam=reparam, precision="bf16",
                                strict_reference=False, vb_output=vb_output, log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    for gl, (W, b) in zip(net.model, params):
        if gl.kind == L.KIND_VB:
            gl.set(L.BUF_MEANS, W.cpu()); gl.set(L.BUF_LVARS, torch.full(W.shape, lvar))
            gl.set(L.BUF_GRAD_SUM, torch.full(W.shape, float("nan")))
            gl.compute_prior()
        else:
            gl.set(L.BUF_WEIGHT, W.cpu())
        gl.set(L.BUF_BIAS, b.cpu())
        # the step overwrites gradWeight / gradSum with its first sample: a tile it skips stays NaN
        gl.set(L.BUF_GRAD_WEIGHT, torch.full(W.shape, float("nan")))
    return net


def run_net(ctx, sizes, N, S, reparam, vb_output, params, X, G, step, want, label, eps=None):
    """One forward_train / backward_update(G, dX) on a fresh net: logits, dX and every layer's gW / gB == want, gS
    == 0 (local) or within its bound (weight).  Returns the device results."""
    from vbnn_b200 import _lib as L
    net = build_net(ctx, sizes, N, S, reparam, vb_output, params)
    try:
        ctx.set_step(step)
        for s in range(S if eps is not None else 0):      # the reference's gradSum used this net's epsilon
            for k, gl in enumerate(net.model):
                if gl.kind == L.KIND_VB:
                    assert torch.equal(gl.draw_noise(step, s).double(), eps[s][k]), (label, s, k)
        Y = net.forward_train(X.float().contiguous()).clone()
        dx = torch.full((N, sizes[0]), float("nan"), device="cuda")
        net.backward_update(G.float().contiguous(), dx)
        torch.cuda.synchronize()
        got = {"logits": Y, "dX": dx}
        for k, gl in enumerate(net.model):
            got[f"gW{k}"] = gl.gradWeight.clone()
            got[f"gB{k}"] = gl.gradBias.clone()
            if gl.kind == L.KIND_VB:
                got[f"gS{k}"] = gl.gradSum.clone()
    finally:
        del net
    for key, (v, e) in ((k, p) for k, p in want.items() if k != "worst"):
        if key.startswith("gS") and reparam == "weight":
            within(f"{label} {key}", got[key], v, e)
        else:
            same(f"{label} {key}", got[key], v)
    return got


def eps_of(ctx, sizes, N, S, reparam, vb_output, params, step):
    """The weight-mode epsilon of every VB layer and sample at `step` (fp64, device)."""
    from vbnn_b200 import _lib as L
    if reparam == "local":
        return None
    net = build_net(ctx, sizes, N, S, reparam, vb_output, params)
    try:
        return [[gl.draw_noise(step, s).double() if gl.kind == L.KIND_VB else None for gl in net.model]
                for s in range(S)]
    finally:
        del net


def exact_case(ctx, sizes, N, S, reparam, vb_output, variants, seed, dens=(0.5, 1 / 16, 0.5), step=40):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    params = make_params(sizes, dens[1], gen)
    X = tern((N, sizes[0]), dens[0], gen)
    G = tern((S, N, sizes[-1]), dens[2], gen)
    vb = [True] * (len(sizes) - 2) + [vb_output]
    eps = eps_of(ctx, sizes, N, S, reparam, vb_output, params, step)
    want = E.exact_minibatch(X, params, G, reparam == "local", vb, eps)
    for kv in variants:
        with knobs(**kv):
            run_net(ctx, sizes, N, S, reparam, vb_output, params, X, G, step, want, f"{sizes} {reparam} {kv}", eps)
    return want


def crossed(tiles, extra=()):
    """Every tile shape under both schedules, then the extra knob sets."""
    return [dict(t, tc_clc=c) for t in tiles for c in (1, 0)] + list(extra)


# (c) the smallest multi-wave shapes of each step form
@pytest.mark.parametrize("reparam,vb_output,C", [("weight", False, 64), ("weight", True, 10),
                                                ("local", False, 10), ("local", True, 64)])
def test_fused_hidden_forward_and_dx_multiwave(ctx, reparam, vb_output, C):
    """[128, 2048, C], N = 4096, S = 2: the hidden layer's forward and the dx into it run 1024 single-CTA units and
    256 pair units (6.9 / 3.5 per slot).  Under local reparameterisation every lrt_split value (split or dual
    forward and backward-data) and the dual 256 x 128 pair form; C = 64 takes the staged logits store, C = 10 the
    direct one."""
    sizes, N, S = [128, 2048, C], 4096, 2
    multiwave("hidden fwd", N, 2048, [(128, 1), (256, 2)], batch=S)
    multiwave("dx into hidden", N, 2048, [(128, 1), (256, 2)], batch=S)
    lrt = reparam == "local"
    tiles = [{}, SINGLE, PAIR] + ([DUAL_PAIR] if lrt else [])
    extra = [dict(tc_gm=1), dict(tc_gm=3), dict(tc_staged=0)]
    if lrt:
        extra += [dict(lrt_split=v) for v in (0, 2, 3)] + [dict(lrt_split=v, **PAIR) for v in (0, 3)]
        extra += [dict(lrt_split=0, **DUAL_PAIR), dict(lrt_split=0, tc_clc=0, **DUAL_PAIR)]
    exact_case(ctx, sizes, N, S, reparam, vb_output, crossed(tiles, extra), seed=1 + 2 * lrt + vb_output)


@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_fused_multi_sample_dw_multiwave(ctx, reparam):
    """[3840, 3840, 16], N = 256, S = 2: layer 0's dW accumulates both samples in one tile: 900 single-CTA units
    (6.1 per slot), 450 on 256 x 128 pairs, 225 on 256 x 256 pairs (3.04).  Weight mode: the TMEM-accumulating
    forms (tc_tacc 1, 2), the 128 x 64 register form (tc_dw64) and the plain ZACC tiles, each with epsilon kept
    in fp16 or regenerated (dw_eps16).  Local: the dual and the split (dw_split) dW."""
    sizes, N, S = [3840, 3840, 16], 256, 2
    multiwave("layer-0 dW", 3840, 3840, [(128, 1), (256, 2), (128, 2)], z_once=True)
    if reparam == "weight":
        forms = [dict(tc_tacc=1), dict(tc_tacc=2), dict(tc_tacc=0, tc_dw64=1), dict(tc_tacc=0, tc_dw64=0)]
        variants = [dict(f, dw_eps16=e, tc_clc=c) for f in forms for e in (1, 0) for c in (1, 0)]
        variants += [dict(tc_tacc=0, tc_dw64=0, tc_gm=3), dict(tc_tacc=2, tc_gm=1)]
    else:
        variants = crossed([{}, SINGLE, PAIR, DUAL_PAIR], [dict(dw_split=1), dict(dw_split=1, tc_clc=0),
                                                         dict(dw_split=1, **PAIR), dict(dw_split=0, **DUAL_PAIR),
                                                         dict(dw_split=0, tc_gm=3)])
    exact_case(ctx, sizes, N, S, reparam, False, variants, seed=21, dens=(0.5, 1 / 16, 0.5))


@pytest.mark.parametrize("reparam", ["weight", "local"])
def test_fused_sample_summing_dx_multiwave(ctx, reparam):
    """[4096, 64, 16], N = 4096, S = 2: the first layer's dX sums the samples in one K-concatenated GEMM (zsum):
    1024 single-CTA units, 256 pair units.  Local: the split form (lrt_split bit 1) and the dual one."""
    sizes, N, S = [4096, 64, 16], 4096, 2
    multiwave("zsum dX", N, 4096, [(128, 1), (256, 2)], z_once=True)
    tiles = [{}, SINGLE, PAIR] + ([DUAL_PAIR] if reparam == "local" else [])
    extra = [dict(tc_gm=3), dict(tc_staged=0)]
    if reparam == "local":
        extra += [dict(lrt_split=v, tc_clc=c) for v in (0, 1, 3) for c in (1, 0)] + [dict(lrt_split=0, **DUAL_PAIR)]
    exact_case(ctx, sizes, N, S, reparam, False, crossed(tiles, extra), seed=31)


@pytest.mark.parametrize("sizes,N,S", [([16, 9472, 100], 256, 10), ([16, 9600, 768], 256, 2)],
                         ids=["partials", "kconcat"])
def test_fused_output_layer_dw_forms_multiwave(ctx, sizes, N, S):
    """The plain output layer's S > 1 dW forms.  100 x 9472 at S = 10: 74 tiles (2 x 74 <= 148), each (tile, sample)
    its own unit of a batched store into per-sample partials that k_sum_partials adds: 740 units, 5 per slot.
    768 x 9600 at S = 2: 450 tiles (2 x 450 > 148), one GEMM over K = S * N: 450 units, 3.04 per slot on the forced
    128 x 128 tiles; the cost model picks 256 x 256 pairs there by default (114 units, 1.5 per pair slot), so only the
    forced variants are multi-wave for that GEMM."""
    O_, I = sizes[-1], sizes[-2]
    partials = 2 * math.ceil(O_ / 128) * math.ceil(I / 128) <= 148
    multiwave("output dW", O_, I, [(128, 1)], batch=S if partials else 1)
    exact_case(ctx, sizes, N, S, "weight", False, crossed([{}, SINGLE], [dict(tc_gm=3), dict(tc_staged=0)]),
               seed=41, dens=(0.5, 1 / 4, 0.5))


# ---------------------------------------------------------------- (b) the layer ABI at C3 layer sizes
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("O_", [4096, 1000])
def test_layer_abi_c3_sizes_exact(ctx, O_, reparam):
    """VBLinear(4096, O), N = 8192, bf16: updateOutput, updateGradInput and accGradParameters == fp64 on the whole
    tensors (gradSum == 0 under local reparameterisation, within its bound in weight mode), on the default tiles,
    forced 128 x 128, 256 x 256 pairs and (local) the 256 x 128 dual pair form, each under both schedules."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    I, N = 4096, 8192
    multiwave("layer fwd", N, O_, [(128, 1)])
    multiwave("layer dx", N, I, [(128, 1), (256, 2)])
    if O_ == 4096:
        multiwave("layer dW", O_, I, [(128, 1), (256, 2)])
    gen = torch.Generator(device="cuda").manual_seed(O_ + (reparam == "local"))
    W = tern((O_, I), 1 / 16, gen)
    b = torch.randint(-2, 3, (O_,), generator=gen, device="cuda").double()
    X = tern((N, I), 0.5, gen)
    G = tern((N, O_), 0.125, gen)
    Y0, dX0, gW0, gB0 = X @ W.t() + b, G @ W, G.t() @ X, G.sum(0)
    for mag in (X.abs() @ W.abs().t(), G.abs() @ W.abs(), G.abs().t() @ X.abs()):
        assert float(mag.max()) < E.EXACT
    opt = vbnn_b200.default_opt(B=40.0, S=1, mu_init=1, var_init=0.01, precision="bf16", reparam=reparam,
                                strict_reference=False, log=False)
    Xd, Gd = X.float().contiguous(), G.float().contiguous()
    # the dual 256 x 128 pair form exists only for the LRT (dual) GEMMs: in weight mode it would repeat the default
    for kv in crossed([{}, SINGLE, PAIR] + ([DUAL_PAIR] if reparam == "local" else [])):
        with knobs(**kv):
            lyr = vbnn_b200.VBLinear(I, O_, opt, ctx)
            try:
                lyr.set(L.BUF_MEANS, W.cpu()); lyr.set(L.BUF_LVARS, torch.full((O_, I), SIGMA0))
                lyr.set(L.BUF_BIAS, b.cpu())
                lyr.compute_prior()
                lyr.resetAcc()
                step = ctx.get_step()
                eps = None if reparam == "local" else lyr.draw_noise(step, 0).double()
                lyr.sample(sample_idx=0)
                label = f"VBLinear({I}, {O_}) {reparam} {kv}"
                same(f"{label} Y", lyr.updateOutput(Xd), Y0)
                same(f"{label} dX", lyr.updateGradInput(Xd, Gd), dX0)
                lyr.accGradParameters(Xd, Gd, 1.0)
                torch.cuda.synchronize()
                same(f"{label} gradWeight", lyr.gradWeight, gW0)
                same(f"{label} gradBias", lyr.gradBias, gB0)
                if reparam == "local":
                    same(f"{label} gradSum", lyr.gradSum, torch.zeros_like(gW0))
                else:
                    dS = gW0 * eps
                    within(f"{label} gradSum", lyr.gradSum, dS,
                           gW0.abs() * (eps.abs() * E.U16 + E.ETA16) + E.U32 * dS.abs())
            finally:
                del lyr
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- (d) the C3 step bench.py times
def test_c3_step_exact(ctx):
    """BASELINE C3 at its exact size (4096-4096x4-1000, N = 8192, S = 1, local reparameterisation, bf16) with exact
    operands: logits, dX and every layer's gradWeight and gradBias == fp64, gradSum == 0, under the default knobs
    (split forward, dual dx and dW on 256 x 256 pairs: 3.5 to 6.9 units per pair slot), forced 128 x 128 tiles and
    the static schedule.  The inputs' density 1/2, the means' 1/64 and dL/dY's 1/8 keep every sum below 2^24
    (largest, a hidden dW: about 6e6)."""
    sizes, N, S = [4096, 4096, 4096, 4096, 4096, 1000], 8192, 1
    multiwave("C3 hidden fwd / dx", N, 4096, [(128, 1), (256, 2)])
    multiwave("C3 hidden dW", 4096, 4096, [(128, 1), (256, 2)], z_once=True)
    gen = torch.Generator(device="cuda").manual_seed(3)
    params = make_params(sizes, 1 / 64, gen)
    X = tern((N, sizes[0]), 0.5, gen)
    G = tern((S, N, sizes[-1]), 0.125, gen)
    want = E.exact_minibatch(X, params, G, True, [True] * 4 + [False])
    acts = (want["logits"][0] != 0).double().mean()
    assert float(acts) > 0.1, "the chain died out: the test would compare zeros"
    for kv in ({}, SINGLE, dict(tc_clc=0)):
        with knobs(**kv):
            run_net(ctx, sizes, N, S, "local", False, params, X, G, 21, want, f"C3 {kv}")
        torch.cuda.empty_cache()


# ---------------------------------------------------------------- sigma^2 = 2^-10: the variance accumulators
# With sigma = 0 the second accumulator of every dual or split LRT GEMM (V = X^2 s2^T, H s2, gradSum = H^T X^2)
# multiplies zeros.  Here s2 = 2^-10 exactly on both sides, so those accumulators carry real values and the
# epilogue's rsqrt / zeta / R branch runs; V is still exact, and everything is checked element by element against
# tests/edge_reference.py's bounds (the mean-side contractions on integer operands keep bound 0 there).
def oracle_of(sizes, N, S, vb_output, params, lvar):
    """The bf16-rounding fp64 oracle net of build_net's parameters, local reparameterisation."""
    over = dict(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])], S=S,
                B=30.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.01, reparam="local",
                strict_reference=False, vb_output=vb_output, log=False)
    oopt = O.default_opt(**over)
    ref = O.MLPOracle(oopt, torch.float64, seed=3, operand_round=O.round_bf16)
    for ol, (W, b) in zip(ref.vb + [ref.out], params):
        if isinstance(ol, O.VBLinearOracle):
            ol.means.copy_(W.cpu()); ol.lvars.fill_(lvar); ol.compute_prior()
        else:
            ol.weight.copy_(W.cpu())
        ol.bias.copy_(b.cpu())
    return ref, oopt


def step_once(ctx, sizes, N, S, vb_output, params, X, G, step, lvar):
    """forward_train / backward_update(G, dX) of a fresh LRT net at `step`; returns every output (device)."""
    from vbnn_b200 import _lib as L
    net = build_net(ctx, sizes, N, S, "local", vb_output, params, lvar)
    try:
        ctx.set_step(step)
        got = {"logits": net.forward_train(X.float().contiguous()).clone()}
        got["dX"] = torch.full((N, sizes[0]), float("nan"), device="cuda")
        net.backward_update(G.float().contiguous(), got["dX"])
        torch.cuda.synchronize()
        for k, gl in enumerate(net.model):
            got[f"gW{k}"] = gl.gradWeight.clone()
            got[f"gB{k}"] = gl.gradBias.clone()
            if gl.kind == L.KIND_VB:
                got[f"gS{k}"] = gl.gradSum.clone()
        noise = [[gl.draw_noise(step, s, rows=N).double().cpu() for gl in net.model if gl.kind == L.KIND_VB]
                 for s in range(S)]
    finally:
        del net
    return got, noise


SIGMA_CASES = [
    # name, sizes, N, vb_output, GEMMs that must be multi-wave (M, N, z_once), variants
    ("hidden fwd and dx", [128, 2048, 64], 4096, True, [(4096, 2048, False)],
     crossed([{}, SINGLE, PAIR, DUAL_PAIR], [dict(lrt_split=v) for v in (0, 2, 3)]
             + [dict(lrt_split=0, **DUAL_PAIR), dict(lrt_split=3, **PAIR), dict(lrt_split=0, tc_clc=0, **PAIR)])),
    ("hidden fwd and dx, C = 10", [128, 2048, 10], 4096, False, [(4096, 2048, False)],
     [{}, PAIR, dict(lrt_split=0, **PAIR), dict(lrt_split=2, tc_clc=0, **PAIR), dict(lrt_split=0, **DUAL_PAIR)]),
    ("multi-sample dW", [3840, 3840, 16], 256, False, [(3840, 3840, True)],
     crossed([{}, SINGLE, PAIR, DUAL_PAIR], [dict(dw_split=1), dict(dw_split=1, tc_clc=0), dict(dw_split=1, **PAIR),
                                            dict(dw_split=1, tc_clc=0, **PAIR)])),
    ("sample-summing dX", [4096, 64, 16], 4096, False, [(4096, 4096, True)],
     [dict(lrt_split=v, tc_clc=c, **t) for v in (0, 1, 3) for c in (1, 0) for t in ({}, PAIR)]
     + [dict(lrt_split=0, **DUAL_PAIR), dict(lrt_split=0, tc_clc=0, **DUAL_PAIR)]),
]


@pytest.mark.parametrize("name,sizes,N,vb_output,gemms,variants", SIGMA_CASES, ids=[c[0] for c in SIGMA_CASES])
def test_fused_lrt_variance_multiwave(ctx, name, sizes, N, vb_output, gemms, variants):
    """The LRT cases of the fused forms at sigma^2 = 2^-10, S = 2: every tensor (gradSum included) within its
    edge_reference bound element by element under each dual / split form, tile shape and schedule; then three
    reruns on the default knobs (CLC) bit-identical.  The hidden layers' gradBias is a column sum finished with fp32
    atomics (order-dependent on non-integer dL/dY), so it is held to its bound there; the output layer's, a sum of
    integers, must be bit-identical too."""
    S, step = 2, 50
    for M_, N_, z_once in gemms:
        multiwave(name, M_, N_, [(128, 1), (256, 2)], batch=S, z_once=z_once)
    gen = torch.Generator(device="cuda").manual_seed(sum(sizes) + N)
    params = make_params(sizes, 1 / 16, gen)
    X = tern((N, sizes[0]), 0.5, gen)
    G = tern((S, N, sizes[-1]), 0.5, gen)
    runs = []
    with knobs():
        for _ in range(3):
            runs.append(step_once(ctx, sizes, N, S, vb_output, params, X, G, step, SIGMA10))
    noise = runs[0][1]
    ref, oopt = oracle_of(sizes, N, S, vb_output, params, SIGMA10)
    want = E.mlp_minibatch(ref, X.cpu(), G.cpu(), noise, True, True, False, oopt)
    last = len(sizes) - 2
    for got, nz in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(sum(nz, []), sum(noise, [])))
        for key, v in got.items():
            if key.startswith("gB") and key != f"gB{last}":
                continue
            assert torch.equal(v, runs[0][0][key]), (name, "rerun differs", key)
    for kv in [None] + variants:
        if kv is None:
            got = runs[0][0]
        else:
            with knobs(**kv):
                got, nz = step_once(ctx, sizes, N, S, vb_output, params, X, G, step, SIGMA10)
            assert all(torch.equal(a, b) for a, b in zip(sum(nz, []), sum(noise, [])))
        for key, pair in want.items():
            check(f"{name} {kv} {key}", got[key].double().cpu().numpy(), pair)


@pytest.mark.parametrize("O_", [4096, 1000])
def test_layer_abi_c3_sizes_variance(ctx, O_):
    """VBLinear(4096, O) at sigma^2 = 2^-10, N = 8192, local reparameterisation, bf16, on the default tiles, forced
    128 x 128, 256 x 256 pairs and the dual 256 x 128 pair form under both schedules.  gradWeight (ternary G and X)
    stays == fp64 on the whole tensor; Y and dX on both edge rows of every 256-row tile and one interior row, and
    gradSum on the same sample of output rows over all columns and all N rows, within edge_reference's bounds.
    zeta is this layer's Philox stream (draw_noise); one layer runs every knob setting (the layer ABI launches
    eagerly), so every setting sees the same noise."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    I, N, step = 4096, 8192, 60
    multiwave("layer dx", N, I, [(128, 1), (256, 2)])
    multiwave("layer fwd", N, O_, [(128, 1)])
    gen = torch.Generator(device="cuda").manual_seed(O_ + 7)
    W = tern((O_, I), 1 / 16, gen)
    b = torch.randint(-2, 3, (O_,), generator=gen, device="cuda").double()
    X = tern((N, I), 0.5, gen)
    G = tern((N, O_), 0.125, gen)
    gW0 = G.t() @ X
    assert float((G.abs().t() @ X.abs()).max()) < E.EXACT
    tile_rows = lambda n: sorted({r for t in range(0, n, 256) for r in (t, min(t + 128, n - 1), min(t + 255, n - 1))})
    rows, outs = tile_rows(N), tile_rows(O_)
    opt = vbnn_b200.default_opt(B=40.0, S=1, mu_init=1, var_init=0.01, precision="bf16", reparam="local",
                                strict_reference=False, log=False)
    oopt = O.default_opt(B=40.0, S=1, mu_init=1, var_init=0.01, reparam="local", strict_reference=False)
    lyr = vbnn_b200.VBLinear(I, O_, opt, ctx)
    try:
        lyr.set(L.BUF_MEANS, W.cpu()); lyr.set(L.BUF_LVARS, torch.full((O_, I), SIGMA10)); lyr.set(L.BUF_BIAS, b.cpu())
        lyr.compute_prior()
        zeta = lyr.draw_noise(step, 0, rows=N).double().cpu()

        def oracle(Wo, bo):
            ol = O.VBLinearOracle(I, Wo.shape[0], oopt, torch.float64, np.random.RandomState(1),
                                  operand_round=O.round_bf16)
            ol.means.copy_(Wo); ol.lvars.fill_(SIGMA10); ol.bias.copy_(bo); ol.compute_prior()
            return E.LayerPass(ol, True, strict=False)
        Xc, Gc = X.cpu(), G.cpu()
        pr = oracle(W.cpu(), b.cpu())                           # sampled rows, every output
        Yr = pr.forward(Xc[rows], torch.zeros(len(rows), I, dtype=torch.float64), zeta[rows])
        dXr = pr.backward(Gc[rows], torch.zeros(len(rows), O_, dtype=torch.float64))
        po = oracle(W.cpu()[outs], b.cpu()[outs])               # sampled outputs, every row
        po.forward(Xc, torch.zeros_like(Xc), zeta[:, outs])
        po.backward(Gc[:, outs], torch.zeros(N, len(outs), dtype=torch.float64))
        gSo = (po.l.gradSum.clone(), po.grad_bounds()[1])
        del Xc, po
        Xd, Gd = X.float().contiguous(), G.float().contiguous()
        for kv in crossed([{}, SINGLE, PAIR, DUAL_PAIR]):
            with knobs(**kv):
                label = f"VBLinear({I}, {O_}) sigma^2 = 2^-10 {kv}"
                lyr.resetAcc()
                ctx.set_step(step)
                lyr.sample(sample_idx=0)
                check(f"{label} Y", lyr.updateOutput(Xd)[rows].double().cpu().numpy(), Yr)
                check(f"{label} dX", lyr.updateGradInput(Xd, Gd)[rows].double().cpu().numpy(), dXr)
                lyr.accGradParameters(Xd, Gd, 1.0)
                torch.cuda.synchronize()
                same(f"{label} gradWeight", lyr.gradWeight, gW0)
                same(f"{label} gradBias", lyr.gradBias, G.sum(0))
                check(f"{label} gradSum", lyr.gradSum[outs].double().cpu().numpy(), gSo)
    finally:
        del lyr
    torch.cuda.empty_cache()
