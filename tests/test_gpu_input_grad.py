"""GPU tests of vbnn_mlp_step_grad_input / MLP.train_step(grad_input=...) (pytest -m gpu): the input gradient of the
fused minibatch, dX = sum_s d l_s / dX, against the fp64 oracle fed the device-drawn noise (the oracle's first layer
computes its gradInput on every run), with the CTA-pair tiles forced, through a torch conv extractor (BASELINE C4),
at C3's full size, and for the guarantees around it: the step itself is unchanged bit for bit, the launch-count
delta is the one first-layer GEMM, dX is deterministic, the graphs are keyed on (N, dX), arguments are checked, and
each data-parallel rank receives its rows of the single-GPU dX."""
import copy
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import vbnn_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def cpu(t):
    return t.detach().float().cpu().numpy()


def build_pair(ctx, sizes, N, S, precision, reparam, seed=0, strict=True, vb_output=False, operand_round=None):
    """A device net and a CPU fp64 oracle holding the same parameters."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    over = dict(input_size=sizes[0], hidden=list(sizes[1:-1]), classes=[str(i) for i in range(sizes[-1])],
                S=S, B=30.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.01, reparam=reparam,
                strict_reference=strict, vb_output=vb_output, log=False)
    gopt = vbnn_b200.default_opt(precision=precision, **over)
    net = vbnn_b200.MLP(gopt, ctx, max_batch=N)
    oopt = O.default_opt(**over)
    ref = O.MLPOracle(oopt, torch.float64, seed=3, operand_round=operand_round)
    rng = np.random.RandomState(seed)
    for gl, ol in zip(net.model, ref.vb + [ref.out]):
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


def device_noise(net, ref, step, S, N):
    """eps (weight mode) or zeta (local) of training sample s at `step`, per VB layer of the oracle."""
    gidx = lambda k: k if k < len(ref.vb) else len(net.model) - 1
    return [[torch.from_numpy(cpu(net.model[gidx(k)].draw_noise(step, s, rows=N)).astype(np.float64))
             for k in range(len(ref.vb_all))] for s in range(S)]


def oracle_grad_input(ref, oopt, X, T, noise, lrt):
    """One reference minibatch (main.lua:28-40); returns sum_s of the first layer's gradInput (mlp.lua:79)."""
    first = ref.vb[0] if ref.vb else ref.out
    ref.resetGradients()
    dX = 0
    for s in range(oopt["S"]):
        ref.sample(None if lrt else noise[s])
        ref.run(X, T, noise[s] if lrt else None)
        dX = dX + first.gradInput
    ref.update(oopt)
    return dX


def data(rng, N, I, C):
    Xn = rng.randn(N, I)
    Tn = rng.randint(1, C + 1, N).astype(np.float64)
    return Xn, Tn, torch.from_numpy(Xn).float().cuda(), torch.from_numpy(Tn).float().cuda()


def run_vs_oracle(ctx, sizes, N, S, precision, reparam, vb_output, iters=2, strict=True):
    bf = precision == "bf16"
    lrt = reparam == "local"
    net, ref, gopt, oopt = build_pair(ctx, sizes, N, S, precision, reparam, seed=7, strict=strict, vb_output=vb_output,
                                      operand_round=O.round_bf16 if bf else None)
    tol = (5e-3 if lrt else 1e-2) if bf else 1e-5
    rng = np.random.RandomState(5)
    g = torch.empty(N, sizes[0], device="cuda")
    out = []
    for it in range(iters):                 # the second minibatch replays a captured graph
        Xn, Tn, X, Tt = data(rng, N, sizes[0], sizes[-1])
        noise = device_noise(net, ref, ctx.get_step(), S, N)
        g.fill_(float("nan"))                # every element must be written
        net.train_step(X, Tt, grad_input=g)
        want = oracle_grad_input(ref, oopt, torch.from_numpy(Xn), torch.from_numpy(Tn), noise, lrt).numpy()
        got = cpu(g)
        assert np.isfinite(got).all(), it
        e = rel(got, want)
        assert e <= tol, (it, e, tol)
        out.append(got.copy())
    return net, out


@pytest.mark.parametrize("vb_output", [False, True])
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("reparam", ["weight", "local"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_grad_input_vs_oracle(ctx, precision, reparam, S, vb_output):
    """Ragged 37-29-23-7 net, N = 45: fp32 <= 1e-5; bf16 against the bf16-rounding oracle <= 5e-3 (LRT) / 1e-2
    (weight mode: the sampled weight is one more bf16 operand)."""
    run_vs_oracle(ctx, [37, 29, 23, 7], 45, S, precision, reparam, vb_output)


@pytest.mark.parametrize("precision,reparam,vb_output", [("fp32", "weight", False), ("bf16", "weight", True),
                                                         ("bf16", "local", True)])
def test_grad_input_without_hidden_layer(ctx, precision, reparam, vb_output):
    """One layer (37-7): the input gradient is the output layer's gradInput (plain nn.Linear or a VBLinear)."""
    run_vs_oracle(ctx, [37, 7], 45, 2, precision, reparam, vb_output)


@pytest.mark.parametrize("reparam,S,lrt_split", [("local", 1, 1),      # dual dx-lrt, one sample
                                                 ("local", 2, 3),      # split dx-lrt, two samples summed
                                                 ("weight", 3, 1)])    # EPI_DX over three sampled weights
def test_grad_input_pair_tiles(ctx, reparam, S, lrt_split):
    """CTA-pair 256 x 256 tiles forced at a size with >= 2 pair tiles per dimension and ragged edges (first-layer
    dX: 540 x 600, K = S x 552): against the bf16-rounding oracle, and against this library's default tiling on the
    same inputs and noise (same rounding points, only the fp32 summation order differs: <= 1e-3)."""
    import vbnn_b200
    names = ("tc_bn", "tc_cg", "lrt_split")
    sizes, N = [600, 552, 530, 10], 540
    res = {}
    for forced in (False, True):
        old = [vbnn_b200.knob(n) for n in names]
        vbnn_b200.knob("lrt_split", lrt_split)
        if forced:
            vbnn_b200.knob("tc_bn", 256); vbnn_b200.knob("tc_cg", 2)
        try:
            ctx.set_step(40)
            net, outs = run_vs_oracle(ctx, sizes, N, S, "bf16", reparam, False, strict=False)
            res[forced] = outs
            del net
        finally:
            for n, v in zip(names, old):
                vbnn_b200.knob(n, v)
    for a, b in zip(res[True], res[False]):
        assert rel(a, b) < 1e-3
        for c0 in range(0, a.shape[1], 64):
            assert rel(a[:, c0:c0 + 64], b[:, c0:c0 + 64]) < 3e-3, c0
        for r0 in range(0, a.shape[0], 64):
            assert rel(a[r0:r0 + 64], b[r0:r0 + 64]) < 3e-3, r0


def snapshot(net):
    """(exact, rounded): the state a minibatch leaves that is bit-reproducible -- means, log-variances, Adam moments,
    sampled weights, gradWeight / gradSum, step counters -- and the part finished by fp32 atomics (the gradBias
    column sums, hence the biases, and the loss / accuracy sums of the result), which is order-dependent by design."""
    from vbnn_b200 import _lib as L
    exact, rounded = [], []
    for m in net.model:
        exact += [m.get(L.BUF_GRAD_WEIGHT), torch.tensor([m.t])]
        if m.kind == L.KIND_LINEAR or net.opt.get("reparam") == "weight":     # (LRT keeps no sampled weight)
            exact.append(m.get(L.BUF_WEIGHT))
        rounded += [m.get(L.BUF_BIAS), m.get(L.BUF_GRAD_BIAS)]
        if m.kind == L.KIND_VB:
            exact += [m.get(b) for b in (L.BUF_MEANS, L.BUF_LVARS, L.BUF_GRAD_SUM, L.BUF_ADAM_M_MU, L.BUF_ADAM_V_MU,
                                         L.BUF_ADAM_M_VAR, L.BUF_ADAM_V_VAR)]
    return exact, rounded


@pytest.mark.parametrize("precision,reparam,S,lrt_split,dx_launches", [("bf16", "local", 1, 1, 1),
                                                                       ("bf16", "local", 2, 3, 2),
                                                                       ("bf16", "weight", 3, 1, 1),
                                                                       ("fp32", "local", 2, 1, 1),
                                                                       ("fp32", "weight", 3, 1, 1)])
def test_step_is_unchanged_bit_for_bit(ctx, precision, reparam, S, lrt_split, dx_launches):
    """From one state_dict and step counter, step and step_grad_input leave bit-identical parameters, Adam state,
    gradients and step counters, over three minibatches (eager, capture, replay); what fp32 atomics finish (gradBias,
    bias, the result scalars) agrees to 1e-6.  The launch-count delta is exactly the first-layer dX GEMM (2 with
    the split dx-lrt form)."""
    import vbnn_b200
    old = vbnn_b200.knob("lrt_split", lrt_split)
    try:
        sizes, N = [200, 136, 96, 10], 160
        a, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=3, strict=False)
        b, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=4, strict=False)
        rng = np.random.RandomState(9)
        g = torch.empty(N, sizes[0], device="cuda")
        for it in range(3):
            _, _, X, Tt = data(rng, N, sizes[0], sizes[-1])
            sd = a.state_dict()
            b.load_state_dict(sd)                 # same state, so the atomics' rounding cannot carry over
            step = sd["step"]
            n0 = a.launch_count()
            ra = a.train_step(X, Tt)
            na = a.launch_count() - n0
            ctx.set_step(step)
            n0 = b.launch_count()
            rb = b.train_step(X, Tt, grad_input=g)
            nb = b.launch_count() - n0
            assert ctx.get_step() == step + 1
            assert abs(ra[0] - rb[0]) <= 1e-6 * abs(ra[0]) and abs(ra[1] - rb[1]) <= 1e-4, (it, ra, rb)
            assert nb - na == dx_launches, (it, na, nb)
            (ea, qa), (eb, qb) = snapshot(a), snapshot(b)
            for x, y in zip(ea, eb):
                assert torch.equal(x, y), it
            for x, y in zip(qa, qb):
                assert rel(x, y) <= 1e-6, it
            assert bool(torch.isfinite(g).all())
    finally:
        vbnn_b200.knob("lrt_split", old)


@pytest.mark.parametrize("precision,reparam,S", [("bf16", "local", 2), ("bf16", "weight", 3), ("fp32", "local", 2)])
def test_grad_input_is_deterministic(ctx, precision, reparam, S):
    """Two calls from the same state (the first eager, the later ones a captured graph) give a bit-identical dX."""
    sizes, N = [600, 552, 530, 10], 540
    net, _, _, _ = build_pair(ctx, sizes, N, S, precision, reparam, seed=2, strict=False)
    sd = net.state_dict()
    _, _, X, Tt = data(np.random.RandomState(1), N, sizes[0], sizes[-1])
    g = torch.empty(N, sizes[0], device="cuda")
    outs = []
    for rep in range(3):
        net.load_state_dict(sd)
        net.train_step(X, Tt, grad_input=g)
        outs.append(g.clone())
    for o in outs[1:]:
        assert torch.equal(outs[0], o)


def test_graphs_keyed_on_buffer(ctx):
    """One net replaying graphs against a second one created with graphs off (every call eager), through
    step / grad(g1) / grad(g1) / grad(g2) / step / grad(g1) / grad(g2) / step: every dX, result and the final
    parameters agree (<= 1e-5: the biases carry the rounding of the fp32-atomic gradBias from one minibatch to the
    next); a call into a new buffer leaves the old one untouched, bit for bit."""
    import vbnn_b200
    sizes, N, S = [200, 136, 96, 10], 160, 2
    a, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False)
    old = vbnn_b200.knob("no_graph", 1)
    try:
        b, _, _, _ = build_pair(ctx, sizes, N, S, "bf16", "local", seed=3, strict=False)
    finally:
        vbnn_b200.knob("no_graph", old)
    rng = np.random.RandomState(4)
    batches = [data(rng, N, sizes[0], sizes[-1])[2:] for _ in range(8)]
    seq = [None, 0, 0, 1, None, 0, 1, None]
    traces = []
    for net in (a, b):
        bufs = [torch.empty(N, sizes[0], device="cuda") for _ in range(2)]
        ctx.set_step(50)
        trace = []
        for (X, Tt), k in zip(batches, seq):
            if k is None:
                trace.append(net.train_step(X, Tt))
                continue
            other = bufs[1 - k].clone()
            trace.append(net.train_step(X, Tt, grad_input=bufs[k]))
            trace.append(bufs[k].clone())
            assert torch.equal(other, bufs[1 - k])             # the other buffer is left as it was
        traces.append(trace)
    for va, vb in zip(*traces):
        if isinstance(va, torch.Tensor):
            assert rel(cpu(va), cpu(vb)) <= 1e-5
        else:
            assert abs(va[0] - vb[0]) <= 1e-5 * abs(vb[0])
    (ea, qa), (eb, qb) = snapshot(a), snapshot(b)
    for x, y in zip(ea + qa, eb + qb):
        assert rel(x, y) <= 1e-5


def test_argument_errors(ctx):
    import ctypes as C
    import vbnn_b200
    from vbnn_b200 import _lib as L
    sizes, N = [13, 7, 2], 4
    net, _, _, _ = build_pair(ctx, sizes, N, 1, "fp32", "weight")
    X = torch.zeros(N, 13, device="cuda"); T = torch.ones(N, device="cuda")
    res = torch.zeros(2, device="cuda")
    lib = L.lib()
    assert lib.vbnn_mlp_step_grad_input(net.handle, C.c_void_p(X.data_ptr()), C.c_void_p(T.data_ptr()), N,
                                        C.c_void_p(res.data_ptr()), None) == L.E_INVALID
    g5 = torch.zeros(5, 13, device="cuda")
    X5 = torch.zeros(5, 13, device="cuda")
    assert lib.vbnn_mlp_step_grad_input(net.handle, C.c_void_p(X5.data_ptr()), C.c_void_p(T.data_ptr()), 5,
                                        C.c_void_p(res.data_ptr()), C.c_void_p(g5.data_ptr())) == L.E_INVALID
    for bad in (torch.zeros(N, 12, device="cuda"), torch.zeros(N + 1, 13, device="cuda"),
                torch.zeros(N, 13, device="cuda", dtype=torch.float64), torch.zeros(N, 13),
                torch.zeros(13, N, device="cuda").t()):
        with pytest.raises(vbnn_b200.VbnnError) as e:
            net.train_step(X, T, grad_input=bad)
        assert e.value.code == L.E_INVALID
    step = ctx.get_step()
    net.train_step(X, T, grad_input=torch.zeros(N, 13, device="cuda"))     # and a valid call still works
    assert ctx.get_step() == step + 1


@pytest.mark.parametrize("S", [1, 2])
def test_convnet_head_end_to_end(ctx, S):
    """BASELINE C4 (convnet.lua:14-33): a torch conv extractor under MLP(256-100-10, vb_output = 1), fp32, weight
    mode.  train_step(feats.detach(), t, grad_input=g) then feats.backward(g) gives the conv parameters the
    gradients of autograd through the same extractor with the head in fp64 on the same sampled weights, summed over
    the S samples as the reference's model:backward does (main.lua:32-37): g itself <= 1e-5, the conv parameter
    gradients <= 1e-4 relative."""
    import vbnn_b200
    from vbnn_b200 import _lib as L
    torch.manual_seed(0)
    N, Cn = 64, 10
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
    # the head's parameters before the update, and the sampled weights W_s = mu + exp(lvars / 2) eps_s
    W = [[(m.get(L.BUF_MEANS).double() + torch.exp(0.5 * m.get(L.BUF_LVARS).double()) *
           m.draw_noise(step, s).double().cpu()).cuda() for m in net.model] for s in range(S)]
    b = [m.get(L.BUF_BIAS).double().cuda() for m in net.model]
    feats = conv(x)
    g = torch.empty(N, 256, device="cuda")
    net.train_step(feats.detach(), t.float() + 1, grad_input=g)
    feats.backward(g)
    assert torch.allclose(net.model[0].get(L.BUF_WEIGHT).double().cuda(), W[0][0], rtol=1e-5, atol=1e-6)  # same W_0
    f64 = feats.detach().double().requires_grad_(True)
    loss = sum(torch.nn.functional.cross_entropy(torch.relu(f64 @ W[s][0].t() + b[0]) @ W[s][1].t() + b[1], t)
               for s in range(S))
    loss.backward()
    assert rel(cpu(g), f64.grad.cpu().numpy()) < 1e-5
    conv_ref(x).backward(f64.grad.float())
    for p, q in zip(conv.parameters(), conv_ref.parameters()):
        assert rel(cpu(p.grad), cpu(q.grad)) < 1e-4


def test_c3_full_size(ctx):
    """BASELINE C3 at its exact size (4096-4096x4-1000, N = 8192, local reparameterisation, S = 1): dX is finite,
    and the bf16 tcgen05 path against this library's fp32 CUDA-core path with identical Philox noise stays within
    0.12 relative (the bound of the first-layer parameter gradients in tests/test_gpu_mlp.py; the same G_0 feeds
    both; measured value printed)."""
    import vbnn_b200
    sizes, N = [4096, 4096, 4096, 4096, 4096, 1000], 8192
    gen = torch.Generator().manual_seed(3)
    X = torch.randn(N, sizes[0], generator=gen).cuda()
    T = torch.randint(1, sizes[-1] + 1, (N,), generator=gen).float().cuda()
    out = {}
    for precision in ("fp32", "bf16"):
        opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                    S=1, B=100.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.001,
                                    reparam="local", precision=precision, strict_reference=False, log=False, seed=5)
        net = vbnn_b200.MLP(opt, ctx, max_batch=N)
        net.init_params(seed=4, he_means=True)
        ctx.set_step(21)
        g = torch.empty(N, sizes[0], device="cuda")
        net.train_step(X, T, grad_input=g)
        assert bool(torch.isfinite(g).all()) and float(g.norm()) > 0
        out[precision] = g.double().cpu()
        del net
        torch.cuda.empty_cache()
    e = float((out["bf16"] - out["fp32"]).norm() / out["fp32"].norm())
    print(f"C3 first-layer dX, bf16 vs fp32: rel {e:.3e}")
    assert e < 0.12, e


@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_data_parallel_rows(mode):
    """Two GPUs under torchrun (skipped on one): each rank's dX equals its rows of a single-GPU step over the whole
    batch (whose 1 / N_global scale is the data-parallel 1 / (N_local x nranks)) within 1e-4 in fp32."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ, VBNN_DP=mode)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "dp_grad_input_check.py")],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "GRAD INPUT DP CHECK OK" in r.stdout
