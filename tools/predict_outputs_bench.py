"""Time vbnn_mlp_predict_outputs, in one process, against what a user would otherwise run.

(a) C3 (4096-4096x4-1000, local reparameterisation, bf16 GEMMs), N = 8192, S = 1, T in {1, 8, 32}:
    predict_outputs (RAW, no samples buffer) against predict, alternating the two.  Both run the same sampled
    forward passes; they differ only in the kernel that folds each pass (class 8): k_predict_moments against k_predict.
(b) A regression shape, 1024-4096-4096-2 GAUSSIAN (same settings, T in {8, 32}): predict_outputs against the
    layer-level chain a user writes today: VBLinear.forward per layer (each LRT layer draws its own noise), torch
    ReLU, T times, then torch mean / var / logsumexp for the moments and the mixture NLL.

Calls are timed with CUDA events after warm-up; every timed call ends in a stream synchronise (the fused calls return
host scalars, the chain converts its NLL to a float).  A separate profiled call per T gives the class-8 time and bytes.
Prints one JSON object; the GPU name and power limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/predict_outputs_bench.py [--N 8192] [--reps 5] [--warmup 2]"""
import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from predict_bench import gpu_info  # noqa: E402

C3 = [4096, 4096, 4096, 4096, 4096, 1000]
REG = [1024, 4096, 4096, 2]


def make_net(vbnn_b200, ctx, sizes, N):
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=1, B=100.0, batchSize=N, reparam="local", precision="bf16", log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    return net


def median(v):
    return sorted(v)[len(v) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=5, help="timed calls of each entry point per T")
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("predict_outputs_bench: no CUDA device (there is no CPU fallback)")
    import vbnn_b200
    ctx = vbnn_b200.default_context(0, seed=5)
    g = torch.Generator(device="cuda").manual_seed(0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        ev0.record()
        fn()
        ev1.record()
        ev1.synchronize()
        return ev0.elapsed_time(ev1)

    def profiled(fn):
        ctx.profile(True)
        try:
            fn()
            return ctx.profile_read()
        finally:
            ctx.profile(False)

    # ---- (a) C3: predict_outputs (RAW) against predict
    net = make_net(vbnn_b200, ctx, C3, a.N)
    X = torch.randn(a.N, C3[0], device="cuda", generator=g)
    Tt = torch.randint(1, C3[-1] + 1, (a.N,), device="cuda", generator=g).float()
    net.train_step(X, Tt)                                     # a trained step: non-trivial posterior state
    Y = torch.randn(a.N, C3[-1], device="cuda", generator=g)
    rows_a = []
    for T in (1, 8, 32):
        run_pred = lambda: net.predict(X, n_samples=T, targets=Tt)
        run_out = lambda: net.predict_outputs(X, n_samples=T, targets=Y)
        for _ in range(a.warmup):
            run_pred(); run_out()
        p_ms, o_ms = [], []
        for _ in range(a.reps):                               # alternating: drifts in clock / power hit both alike
            p_ms.append(timed(run_pred))
            o_ms.append(timed(run_out))
        kp = profiled(run_pred)["predict"]
        ko = profiled(run_out)["predict"]
        pm, om = median(p_ms), median(o_ms)
        rows_a.append(dict(
            T=T, predict_ms=round(pm, 3), predict_outputs_ms=round(om, 3), outputs_over_predict=round(om / pm, 4),
            predict_ms_all=[round(v, 3) for v in p_ms], predict_outputs_ms_all=[round(v, 3) for v in o_ms],
            k_predict=dict(launches=kp[1], ms=round(kp[0], 4), share_of_call=round(kp[0] / pm, 4),
                           gb_per_s=round(kp[2] / kp[0] / 1e6, 1)),
            k_predict_moments=dict(launches=ko[1], ms=round(ko[0], 4), share_of_call=round(ko[0] / om, 4),
                                   gb_per_s=round(ko[2] / ko[0] / 1e6, 1), bytes=ko[2])))
    del net

    # ---- (b) regression shape: predict_outputs (GAUSSIAN) against the layer-level chain
    net = make_net(vbnn_b200, ctx, REG, a.N)
    X = torch.randn(a.N, REG[0], device="cuda", generator=g)
    y = torch.randn(a.N, 1, device="cuda", generator=g)

    def chain(T):
        outs = []
        for t in range(T):
            h = X
            for k, lyr in enumerate(net.model):
                h = lyr.forward(h)                            # LRT: each VB layer draws its own zeta
                if k < len(net.model) - 1:
                    h = torch.relu(h)
            outs.append(h)
        f = torch.stack(outs)                                 # [T x N x 2]
        m, s = f[..., :1], f[..., 1:]
        mean = m.mean(0)
        epi = m.var(0, unbiased=False)
        ale = s.exp().mean(0)
        ll = (-0.5 * (math.log(2 * math.pi) + s + (y - m) ** 2 * torch.exp(-s))).sum(-1)
        nll = -(torch.logsumexp(ll, 0) - math.log(T)).mean()
        return mean, epi, ale, float(nll)

    rows_b = []
    for T in (8, 32):
        run_out = lambda: net.predict_outputs(X, n_samples=T, model="gaussian", targets=y)
        run_chain = lambda: chain(T)
        for _ in range(a.warmup):
            run_out(); run_chain()
        o_ms, c_ms = [], []
        for _ in range(a.reps):
            o_ms.append(timed(run_out))
            c_ms.append(timed(run_chain))
        ko = profiled(run_out)["predict"]
        om, cm = median(o_ms), median(c_ms)
        rows_b.append(dict(T=T, predict_outputs_ms=round(om, 3), layer_chain_ms=round(cm, 3),
                           chain_over_fused=round(cm / om, 3),
                           predict_outputs_ms_all=[round(v, 3) for v in o_ms],
                           layer_chain_ms_all=[round(v, 3) for v in c_ms],
                           k_predict_moments=dict(launches=ko[1], ms=round(ko[0], 4), share_of_call=round(ko[0] / om, 4))))
    out = dict(c3=dict(workload="C3 4096-4096x4-1000, local reparameterisation, bf16 GEMMs, RAW", N=a.N, S=1,
                       results=rows_a),
               regression=dict(workload="1024-4096-4096-2 GAUSSIAN, local reparameterisation, bf16 GEMMs", N=a.N, S=1,
                               results=rows_b),
               reps=a.reps, warmup=a.warmup, timing="median of CUDA-event times per call", **gpu_info())
    print(json.dumps(out))


if __name__ == "__main__":
    main()
