"""Time vbnn_mlp_step_grad_input against vbnn_mlp_step, in one process, alternating the two on one net.

Workloads (bf16 GEMMs):
  C3     4096-4096x4-1000, N = 8192, local reparameterisation, S = 1: the first-layer dX is a dual dx-lrt GEMM of
         the same shape as the hidden layers' ones;
  C2     784-1200-1200-10, N = 1024, weight mode, S = 10: the first-layer dX sums ten samples (K = 10 x 1200) in one
         TMEM accumulator per 128 x 128 tile.  For the choice of that form, the same products as per-sample work
         units (the batched plain-store GEMM the per-sample-partials alternative would run before a fixed-order sum)
         are timed through vbnn_gemm_bf16;
  C4     a torch conv extractor (3x32x32 -> 256) under MLP(256-100-10, vb_output = 1), N = 512, S in {1, 10}: the
         whole minibatch -- extractor forward and backward plus head -- through the fused path (train_step with
         grad_input, then feats.backward) against the layer-level chain (per sample: sample, updateOutput,
         updateGradInput, accGradParameters per layer; then update), as in tests/test_gpu_mlp.py.
Per workload: median CUDA-event ms of each entry point and their ratio; from one profiled call of each, the
first-layer dX GEMM (the difference of the dx / dx-lrt profile classes between the two calls) with its time and
TFLOP/s next to the mean of the other dx / dx-lrt launches of the same step.  Prints one JSON object; the GPU name
and power limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/input_grad_bench.py [--reps 10] [--warmup 3] [--only C3 C2 C4]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def median(v):
    return sorted(v)[len(v) // 2]


def timed(fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def alternate(a, b, reps, warmup):
    for _ in range(warmup):
        a(); b()
    ta, tb = [], []
    for _ in range(reps):                       # alternating: drifts in clock / power hit both alike
        ta.append(timed(a))
        tb.append(timed(b))
    ma, mb = median(ta), median(tb)
    return dict(step_ms=round(ma, 4), grad_input_ms=round(mb, 4), ratio=round(mb / ma, 4),
                step_ms_all=[round(v, 4) for v in ta], grad_input_ms_all=[round(v, 4) for v in tb])


def profiled(ctx, fn):
    ctx.profile(True)
    try:
        fn()
        return ctx.profile_read()
    finally:
        ctx.profile(False)


def first_layer_dx(ctx, step, grad):
    """The first-layer dX GEMM(s): what the dx / dx-lrt classes of a grad-input call hold beyond a plain call."""
    p0, p1 = profiled(ctx, step), profiled(ctx, grad)
    out = {}
    for k in ("dx", "dx_lrt", "store"):
        a, b = p0.get(k, (0.0, 0, 0.0)), p1.get(k, (0.0, 0, 0.0))
        d_ms, d_n, d_fl = b[0] - a[0], b[1] - a[1], b[2] - a[2]
        if d_n:
            out[k] = dict(launches=d_n, ms=round(d_ms, 4), tflops=round(d_fl / d_ms / 1e9, 1), flop=d_fl)
        if a[1] and k != "store":
            out[k + "_other_launches"] = dict(launches=a[1], mean_ms=round(a[0] / a[1], 4),
                                              tflops=round(a[2] / a[0] / 1e9, 1))
    return out


def mlp_workload(ctx, name, sizes, N, S, reparam, a):
    import torch
    import vbnn_b200
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=S, B=100.0, batchSize=N, reparam=reparam, precision="bf16", strict_reference=False,
                                log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn(N, sizes[0], device="cuda", generator=g)
    T = torch.randint(1, sizes[-1] + 1, (N,), device="cuda", generator=g).float()
    dX = torch.empty(N, sizes[0], device="cuda")
    step = lambda: net.train_step(X, T, sync=False)
    grad = lambda: net.train_step(X, T, sync=False, grad_input=dX)
    row = dict(workload=name, sizes=sizes, N=N, S=S, reparam=reparam, **alternate(step, grad, a.reps, a.warmup))
    row["first_layer_dx"] = first_layer_dx(ctx, step, grad)
    del net
    torch.cuda.empty_cache()
    return row


def per_sample_units(ctx, N, I, O, Z, reps):
    """The C2 first-layer dX products as Z separate work units (batched plain-store GEMM into per-sample partials)."""
    import torch
    from vbnn_b200 import _lib as L
    A = torch.randn(Z, N, O, device="cuda").to(torch.bfloat16)
    B = torch.randn(Z, O, I, device="cuda").to(torch.bfloat16)
    D = torch.empty(Z, N, I, device="cuda")
    run = lambda: L.check(L.lib().vbnn_gemm_bf16(ctx.handle, C.c_void_p(A.data_ptr()), O, 1, C.c_void_p(B.data_ptr()),
                                                 I, 0, C.c_void_p(D.data_ptr()), I, N, I, O, Z, N * O, O * I, N * I))
    for _ in range(3):
        run()
    prof = profiled(ctx, lambda: [run() for _ in range(reps)])
    ms, n, fl = prof["store"]
    return dict(form="per-sample work units, plain store (before any partial sum)", launches=n,
                mean_ms=round(ms / n, 4), tflops=round(fl / ms / 1e9, 1),
                partials_bytes_written=Z * N * I * 4)


def c4_workload(ctx, S, a):
    import torch
    import vbnn_b200
    N, Cn = 512, 10
    torch.manual_seed(0)
    conv = torch.nn.Sequential(torch.nn.Conv2d(3, 16, 5), torch.nn.ReLU(), torch.nn.MaxPool2d(2),
                               torch.nn.Conv2d(16, 16, 5), torch.nn.ReLU(), torch.nn.MaxPool2d(2),
                               torch.nn.Flatten(), torch.nn.Linear(16 * 5 * 5, 256), torch.nn.ReLU()).cuda()
    x = torch.randn(N, 3, 32, 32, device="cuda")
    t = torch.randint(0, Cn, (N,), device="cuda")
    t1 = t.float() + 1
    opt = vbnn_b200.default_opt(input_size=256, hidden=[100], classes=[str(i) for i in range(Cn)], S=S, B=50.0,
                                batchSize=N, mu_init=1, var_init=0.01, vb_output=True, strict_reference=False,
                                precision="bf16", log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    g = torch.empty(N, 256, device="cuda")

    def fused():
        conv.zero_grad(set_to_none=False)
        feats = conv(x)
        net.train_step(feats.detach(), t1, sync=False, grad_input=g)
        feats.backward(g)

    lopt = vbnn_b200.default_opt(S=S, B=50.0, batchSize=N, mu_init=1, var_init=0.01, strict_reference=False,
                                 precision="bf16", log=False)
    h1 = vbnn_b200.VBLinear(256, 100, lopt, ctx)
    h2 = vbnn_b200.VBLinear(100, Cn, lopt, ctx)

    def layered():                              # test_convnet_head_behind_the_same_abi, S samples
        conv.zero_grad(set_to_none=False)
        feats = conv(x)
        f = feats.detach().contiguous()
        gf = torch.zeros_like(f)
        for h in (h1, h2):
            h.resetAcc()
        for s in range(S):
            for h in (h1, h2):
                h.sample(sample_idx=s)
            a1 = h1.updateOutput(f)
            r1 = torch.clamp(a1, min=0)
            logits = h2.updateOutput(r1).clone().requires_grad_(True)
            torch.nn.functional.cross_entropy(logits, t).backward()
            g2 = logits.grad.contiguous()
            gr1 = h2.updateGradInput(r1, g2); h2.accGradParameters(r1, g2)
            g1 = (gr1 * (a1 > 0)).contiguous()
            gf += h1.updateGradInput(f, g1); h1.accGradParameters(f, g1)
        feats.backward(gf)
        h1.update(lopt); h2.update(lopt)

    r = alternate(layered, fused, a.reps, a.warmup)
    return dict(workload="C4", head=[256, 100, 10], N=N, S=S, extractor="torch conv 3x32x32 -> 256 (fp32, cuDNN)",
                layer_level_ms=r["step_ms"], fused_ms=r["grad_input_ms"], fused_over_layer_level=r["ratio"],
                layer_level_ms_all=r["step_ms_all"], fused_ms_all=r["grad_input_ms_all"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10, help="timed calls of each entry point per workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", nargs="+", default=["C3", "C2", "C4"])
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("input_grad_bench: no CUDA device (there is no CPU fallback)")
    import vbnn_b200
    ctx = vbnn_b200.default_context(0, seed=5)
    rows = []
    if "C3" in a.only:
        rows.append(mlp_workload(ctx, "C3", [4096, 4096, 4096, 4096, 4096, 1000], 8192, 1, "local", a))
    if "C2" in a.only:
        row = mlp_workload(ctx, "C2 shape", [784, 1200, 1200, 10], 1024, 10, "weight", a)
        row["first_layer_dx_alternative"] = per_sample_units(ctx, 1024, 784, 1200, 10, a.reps)
        rows.append(row)
    if "C4" in a.only:
        for S in (1, 10):
            rows.append(c4_workload(ctx, S, a))
    out = dict(bench="vbnn_mlp_step_grad_input vs vbnn_mlp_step", precision="bf16 GEMMs", reps=a.reps,
               warmup=a.warmup, timing="median of CUDA-event times per call", **gpu_info(), results=rows)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
