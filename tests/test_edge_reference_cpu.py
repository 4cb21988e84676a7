"""CPU checks of tests/edge_reference.py: the conventions it adds to the oracle (R := 0 where V == 0, the ClassNLL
target rule, lowest-index argmax), and that its per-element bound catches a single corrupted element while accepting
an fp32 sum taken in another order."""
import copy
import math

import numpy as np
import torch

import edge_reference as E
from custom_loss_reference import custom_minibatch
from oracle import vbnn_oracle as O


def lrt_layer(I=24, Ol=10, seed=0, bf=False):
    opt = O.default_opt(reparam="local", B=20.0, S=1, mu_init=1, var_init=0.01)
    lyr = O.VBLinearOracle(I, Ol, opt, torch.float64, np.random.RandomState(seed),
                           operand_round=O.round_bf16 if bf else None)
    rng = np.random.RandomState(seed + 1)
    lyr.means.copy_(torch.from_numpy(rng.randn(Ol, I) * 0.3))
    lyr.lvars.copy_(torch.from_numpy(rng.uniform(math.log(1e-4), math.log(1e-2), (Ol, I))))
    lyr.bias.copy_(torch.from_numpy(rng.randn(Ol) * 0.1))
    lyr.compute_prior()
    return lyr


def test_zero_row_convention():
    """An all-zero input row under local reparameterisation: the oracle's R is +-inf there and its gradInput NaN;
    the reference keeps R = 0, so the row's output is the bias, its gradInput is G mu, and it adds nothing to gradSum."""
    rng = np.random.RandomState(2)
    N, I, Ol = 6, 24, 10
    x = torch.from_numpy(rng.randn(N, I)); x[2] = 0.0
    zeta = torch.from_numpy(rng.randn(N, Ol))
    G = torch.from_numpy(rng.randn(N, Ol))
    raw = lrt_layer()
    raw.updateOutput(x, zeta)
    assert not torch.isfinite(raw._R[2]).any()
    assert not torch.isfinite(raw.updateGradInput(x, G)[2]).all()

    lyr = lrt_layer()
    ps = E.LayerPass(lyr, bf=False)
    Y, eY = ps.forward(x, torch.zeros_like(x), zeta)
    assert torch.equal(Y[2], lyr.bias) and float(eY[2].max()) == 0.0      # exact: no rounding on a zero row
    assert torch.equal(lyr._R[2], torch.zeros(Ol, dtype=torch.float64))
    gi, egi = ps.backward(G, torch.zeros_like(G))
    assert torch.isfinite(gi).all() and torch.isfinite(egi).all()
    assert torch.allclose(gi[2], G[2] @ lyr.means, rtol=0, atol=1e-15)
    gs_with = lyr.gradSum.clone()
    lyr2 = lrt_layer()
    ps2 = E.LayerPass(lyr2, bf=False)
    keep = [0, 1, 3, 4, 5]
    ps2.forward(x[keep], torch.zeros(5, I, dtype=torch.float64), zeta[keep])
    ps2.backward(G[keep], torch.zeros(5, Ol, dtype=torch.float64))
    assert torch.allclose(gs_with, lyr2.gradSum, rtol=1e-14, atol=0)     # the zero row adds nothing
    # the other rows are the oracle's
    assert torch.allclose(Y[keep], raw.output[keep], rtol=1e-14, atol=0)


def test_subnormal_variance_is_finite():
    """x = 1e-20 at one feature: V ~ 1e-43 (subnormal in fp32) has the finite R = zeta / (2 sqrt V) ~ 1e20 zeta, and
    gradInput's variance term 2 x (H s2) = sign(x) G zeta sqrt(s2) is O(1); the bounds stay finite and below it."""
    rng = np.random.RandomState(3)
    N, I, Ol = 4, 24, 10
    x = torch.from_numpy(rng.randn(N, I)); x[1] = 0.0; x[1, 5] = 1e-20
    zeta = torch.from_numpy(rng.randn(N, Ol))
    G = torch.from_numpy(rng.randn(N, Ol))
    lyr = lrt_layer()
    ps = E.LayerPass(lyr, bf=False)
    Y, eY = ps.forward(x, torch.zeros_like(x), zeta)
    assert float(ps.V[1].max()) < E.FLT_MIN and float(ps.V[1].min()) > 0
    assert torch.isfinite(lyr._R).all() and torch.isfinite(ps.eR).all()
    assert float((ps.eR[1] / lyr._R[1].abs()).max()) < 0.05            # the subnormal V costs a few bits, no more
    gi, egi = ps.backward(G, torch.zeros_like(G))
    s2 = torch.exp(lyr.lvars[:, 5])
    want = G[1] @ lyr.means[:, 5] + (G[1] * zeta[1] * s2.sqrt()).sum()
    assert abs(float(gi[1, 5]) - float(want)) <= 1e-12 * abs(float(want))
    assert float(egi[1, 5]) < 0.05 * abs(float(want))


def test_target_rule_and_ties():
    """Targets 0 and C+1 add 0 to the loss, give softmax / N with no -1 and never count; tied rows predict the
    lowest index."""
    C, N = 5, 6
    Y = torch.tensor([[1.0, 3.0, 3.0, 0.0, 3.0],
                      [0.0] * 5,
                      [2.0, 1.0, 0.0, 0.0, 0.0],
                      [0.0, 1e4, 0.0, 0.0, -1e4],
                      [0.0, 1.0, 2.0, 3.0, 4.0],
                      [0.0, 0.0, 0.0, 0.0, 0.0]], dtype=torch.float64)
    t = torch.tensor([2.0, 1.0, 0.0, 2.0, 6.0, 2.0])
    err, acc, g, logp = E.classnll_device(Y, t)
    assert first_argmax_list(Y) == [1, 0, 0, 1, 4, 0]
    assert acc == 3 / N * 100.0                                        # rows 0, 1, 3; never rows 2 and 4
    p = torch.exp(logp)
    for r in (2, 4):
        assert torch.allclose(g[r], p[r] / N, rtol=0, atol=0)
    want = -(logp[0, 1] + logp[1, 0] + logp[3, 1] + logp[5, 1]) / N
    assert abs(err - float(want)) < 1e-15
    assert abs(float(g[3].sum())) < 1e-15 and float(g[3, 4]) == 0.0     # exp(-2e4) underflows to 0


def first_argmax_list(Y):
    return [int(i) for i in E.first_argmax(Y)]


def _fp32_sum(A, B, order):
    """A @ B^T summed in fp32 in a chosen order over k."""
    a, b = A.float(), B.float()
    if order == "matmul":
        return (a @ b.t()).double()
    if order == "reverse":
        acc = torch.zeros(A.shape[0], B.shape[0])
        for k in range(A.shape[1] - 1, -1, -1):
            acc = acc + a[:, k:k + 1] * b[:, k:k + 1].t()
        return acc.double()
    if order == "blocks":                                              # 64-wide k-blocks, partial sums added last
        parts = [a[:, k:k + 64] @ b[:, k:k + 64].t() for k in range(0, A.shape[1], 64)]
        acc = torch.zeros_like(parts[0])
        for p in parts[::-1]:
            acc = acc + p
        return acc.double()
    raise ValueError(order)


def test_bound_accepts_fp32_orders_and_flags_corruption():
    """An fp32 sum of bf16-rounded operands in three different orders lies within the bound everywhere; dropping one
    k-block of 64 products from one element, or shifting one output row by one, is flagged."""
    rng = np.random.RandomState(4)
    M, N, K = 48, 40, 256
    A = O.round_bf16(torch.from_numpy(rng.randn(M, K)))
    B = O.round_bf16(torch.from_numpy(rng.randn(N, K)))
    ref = A @ B.t()
    bound = E.contraction_bound(A, B) + E.U32 * ref.abs()
    for order in ("matmul", "reverse", "blocks"):
        got = _fp32_sum(A, B, order)
        assert E.violations(got.numpy(), ref, bound) == [], order
    # one k-block missing from one element: the first element of row 7 whose block 64..127 is at least 1 in size
    # (a block of 64 N(0,1) products is ~8; one near 0 is invisible to any sound bound)
    part = A[7, 64:128] @ B[:, 64:128].t()
    j = int((part.abs() >= 1.0).nonzero()[0])
    got = _fp32_sum(A, B, "matmul").clone()
    got[7, j] -= float(part[j])
    v = E.violations(got.numpy(), ref, bound)
    assert [x[0] for x in v] == [(7, j)]
    got = _fp32_sum(A, B, "matmul").clone()
    got[20] = got[21].clone()                                           # a row written one row off
    v = E.violations(got.numpy(), ref, bound)
    assert len(v) >= 1 and all(x[0][0] == 20 for x in v if x[0] != "...")
    # a single ulp-scale slip does not need the bound to be loose: the bound is a small fraction of the values
    assert float((bound / ref.abs().clamp(min=1.0)).median()) < 1e-3


def test_bias_gradient_bound():
    """The bias gradient's bound is the contraction of G with ones: C_ACC * N * 2^-24 * sum |G| (+ subnormal floor)."""
    rng = np.random.RandomState(5)
    G = torch.from_numpy(rng.randn(300, 7))
    b = E.contraction_bound(G.t(), torch.ones(1, 300, dtype=torch.float64))[:, 0]
    want = E.C_ACC * 300 * E.U32 * G.abs().sum(0) + 300 * E.ETA
    assert torch.allclose(b, want, rtol=1e-14, atol=0)
    got = G.float().sum(0).double()
    assert E.violations(got.numpy(), G.sum(0), b) == []


def test_minibatch_matches_split_reference():
    """Without degenerate rows the edge reference's minibatch values equal tests/custom_loss_reference.py's (the same
    oracle methods), and every bound is finite."""
    sizes, N, S = [20, 16, 5], 12, 2
    for reparam in ("weight", "local"):
        for vb_output in (False, True):
            opt = O.default_opt(input_size=sizes[0], hidden=[sizes[1]], classes=list("abcde"), S=S, B=10.0,
                                mu_init=1, var_init=0.01, reparam=reparam, vb_output=vb_output)
            ref = O.MLPOracle(opt, torch.float64, seed=3)
            rng = np.random.RandomState(6)
            for l in ref.vb_all:
                l.means.copy_(torch.from_numpy(rng.randn(l.O, l.I) * 0.3)); l.compute_prior()
            ref2 = copy.deepcopy(ref)
            x = torch.from_numpy(rng.randn(N, sizes[0]))
            G = torch.from_numpy(rng.randn(S, N, 5) / N)
            lrt = reparam == "local"
            noise = [[torch.from_numpy(rng.randn(*((N, l.O) if lrt else (l.O, l.I)))) for l in ref.vb_all]
                     for _ in range(S)]
            out = E.mlp_minibatch(ref, x, G, noise, lrt, bf=False, strict=True, opt=opt)
            Y, _, dX = custom_minibatch(ref2, x, lambda Y_: G, noise, lrt, opt, update=False)
            assert torch.allclose(out["logits"][0], Y, rtol=1e-13, atol=1e-15)
            assert torch.allclose(out["dX"][0], dX, rtol=1e-12, atol=1e-15)
            for k, l in enumerate(ref2.vb + [ref2.out]):
                assert torch.allclose(out[f"gW{k}"][0], l.gradWeight, rtol=1e-12, atol=1e-15)
            for key, (v, e) in out.items():
                assert torch.isfinite(v).all() and torch.isfinite(e).all(), key


# ---------------------------------------------------------------- the exactness rule
def _ternary(rng, shape, density=0.5):
    return torch.from_numpy(rng.choice([-1.0, 1.0], size=shape) * (rng.rand(*shape) < density))


def test_exact_operands_any_order():
    """Ternary operands at K = 8192: an fp32 sum in each of three orders equals fp64 exactly and the exactness rule
    gives the bound 0; one off-grid operand element restores the old bound on its row; under the zero bound a dropped
    64-wide k-block or a row written one row off is flagged."""
    rng = np.random.RandomState(9)
    M, N, K = 12, 10, 8192
    A, B = _ternary(rng, (M, K)), _ternary(rng, (N, K))
    ref = A @ B.t()
    bound = E.contraction_bound(A, B)
    assert float(bound.abs().max()) == 0.0
    for order in ("matmul", "reverse", "blocks"):
        got = _fp32_sum(A, B, order)
        assert torch.equal(got, ref), order
        assert E.violations(got.numpy(), ref, bound) == [], order
    A2 = A.clone()
    A2[3, 100] = 0.5 + 2.0 ** -9                                    # a bf16 value off the integer grid
    b2 = E.contraction_bound(A2, B)
    assert float(b2[3].min()) > 0 and float(b2[[i for i in range(M) if i != 3]].abs().max()) == 0.0
    old = E.C_ACC * ((A2[3].abs() > 0).double() @ (B.abs() > 0).double().t()) * E.U32 * (A2[3].abs() @ B.abs().t())
    assert torch.allclose(b2[3], old + ((A2[3].abs() > 0).double() @ (B.abs() > 0).double().t()) * E.ETA, rtol=1e-15)
    e = torch.zeros_like(A); e[5, 7] = 1e-3                          # an operand error does the same
    assert float(E.contraction_bound(A, B, e, None)[5].min()) > 0
    part = A[7, 64:128] @ B[:, 64:128].t()
    j = int(part.abs().argmax())
    assert float(part[j]) != 0
    got = _fp32_sum(A, B, "blocks").clone()
    got[7, j] -= float(part[j])
    assert [x[0] for x in E.violations(got.numpy(), ref, bound)] == [(7, j)]
    got = _fp32_sum(A, B, "matmul").clone()
    got[4] = got[5].clone()
    v = E.violations(got.numpy(), ref, bound)
    assert len(v) >= 1 and all(x[0][0] == 4 for x in v if x[0] != "...")
    # past 2^24 the rule does not apply: a sum of 2^25 ones
    big = torch.ones(1, 2 ** 25, dtype=torch.float64)
    assert float(E.contraction_bound(big, big)) > 0


def _exact_oracle(sizes, N, S, reparam, vb_output, seed):
    """An oracle net with integer means / weights and biases and sigma flushed to 0, and its minibatch inputs."""
    opt = O.default_opt(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])],
                        S=S, B=10.0, mu_init=1, var_init=0.01, reparam=reparam, vb_output=vb_output,
                        strict_reference=False)
    ref = O.MLPOracle(opt, torch.float64, seed=3, operand_round=O.round_bf16)
    rng = np.random.RandomState(seed)
    params = []
    for l in ref.vb + [ref.out]:
        W = _ternary(rng, (l.weight.shape[0], l.weight.shape[1]), 0.3)
        b = torch.from_numpy(rng.randint(-2, 3, l.bias.shape[0]).astype(np.float64))
        if isinstance(l, O.VBLinearOracle):
            l.means.copy_(W); l.lvars.fill_(-300.0); l.compute_prior()
        else:
            l.weight.copy_(W)
        l.bias.copy_(b)
        params.append((W, b))
    x = _ternary(rng, (N, sizes[0]))
    G = _ternary(rng, (S, N, sizes[-1]), 0.25)
    lrt = reparam == "local"
    noise = [[torch.from_numpy(rng.randn(*((N, l.O) if lrt else (l.O, l.I)))) for l in ref.vb_all] for _ in range(S)]
    return ref, opt, params, x, G, noise


def test_exact_minibatch_is_the_edge_reference():
    """On exact operands with sigma flushed to 0, tests/edge_reference.py's minibatch gives bound 0 on logits, dX,
    gW, gB (and gS under local reparameterisation), and exact_minibatch -- the plain fp64 chain the multi-wave GPU
    tests use at full size -- reproduces its values bit for bit; weight-mode gradSum agrees with it in value and
    bound."""
    sizes, N, S = [40, 24, 20, 6], 64, 2
    for reparam in ("weight", "local"):
        for vb_output in (False, True):
            ref, opt, params, x, G, noise = _exact_oracle(sizes, N, S, reparam, vb_output, seed=12)
            lrt = reparam == "local"
            want = E.mlp_minibatch(ref, x, G, noise, lrt, bf=True, strict=False, opt=opt)
            vb = [True] * (len(sizes) - 2) + [vb_output]
            eps = None if lrt else [[noise[s][k] if vb[k] else None for k in range(len(vb))] for s in range(S)]
            got = E.exact_minibatch(x, params, G, lrt, vb, eps)
            assert max(got["worst"].values()) < E.EXACT
            for key, (v, e) in want.items():
                gv, ge = got[key]
                assert torch.equal(gv, v), (reparam, vb_output, key)
                if key.startswith("gS") and not lrt:
                    assert float(e.max()) > 0
                    assert torch.allclose(ge, e, rtol=1e-12, atol=0), (reparam, vb_output, key)
                else:
                    assert float(e.abs().max()) == 0.0, (reparam, vb_output, key, float(e.max()))
                    assert float(ge.abs().max()) == 0.0


def test_exact_minibatch_refuses_past_2_24():
    """exact_minibatch asserts the 2^24 condition instead of trusting an estimate."""
    X = torch.ones(4, 8, dtype=torch.float64)
    W = torch.full((3, 8), 2.0 ** 22, dtype=torch.float64)
    G = torch.ones(1, 4, 3, dtype=torch.float64)
    with np.testing.assert_raises(AssertionError):
        E.exact_minibatch(X, [(W, torch.zeros(3, dtype=torch.float64))], G, True, [False])


def test_exactness_across_samples_counts_terms():
    """The cross-sample rule tests the magnitudes of the terms the device may sum in one fp32 accumulator, not of the
    per-sample results: terms 2^23 .. 2^16 in sample 1 (sum 16711680) and +65536, +1, -65536 in sample 2 (sum 1) have
    results summing below 2^24, yet one fp32 accumulator over all terms loses the 1."""
    lyr = O.LinearOracle(1, 1, torch.float64)
    lyr.weight.fill_(1.0); lyr.bias.zero_()
    ps = E.LayerPass(lyr, bf=False)
    lyr.gradWeight.zero_(); lyr.gradBias.zero_()
    for xs in ([2.0 ** k for k in range(23, 15, -1)], [65536.0, 1.0, -65536.0]):
        x = torch.tensor(xs, dtype=torch.float64)[:, None]
        g = torch.ones_like(x)
        ps.forward(x, torch.zeros_like(x))
        ps.backward(g, torch.zeros_like(g))
    ew, _, eb = ps.grad_bounds()
    want = float(lyr.gradWeight[0, 0])
    assert want == 16711681.0
    fused = np.float32(0)
    for v in [2.0 ** k for k in range(23, 15, -1)] + [65536.0, 1.0, -65536.0]:
        fused = np.float32(fused + np.float32(v))
    assert float(fused) != want and abs(float(fused) - want) <= float(ew[0, 0])
    assert float(eb[0]) == 0.0                                       # 11 ones: exact
