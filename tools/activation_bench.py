"""Time the fused minibatch (vbnn_mlp_step) under each hidden-layer activation of vbnn_mlp_set_activation on one net,
switching the kind between groups of calls, in one process.

Workloads (bf16 GEMMs, ClassNLL):
  C3     4096-4096x4-1000, N = 8192, local reparameterisation, S = 1 (fwd-lrt / dx-lrt epilogues);
  C2     784-1200-1200-10, N = 1024, weight mode, S = 10 (fwd / dx epilogues).
Per workload and kind: the median CUDA-event ms of `reps` calls, taken in alternating rounds (round r times one call of
every kind in turn, so drifts in clock and power hit all kinds alike; the switch between kinds re-captures the step
graph, so each kind's graph is captured in warm-up and every timed call replays it after one untimed call), and from one
profiled call per kind the time of the GEMM classes fwd, fwd_lrt, dx and dx_lrt.  Prints one JSON object; the GPU name
and power limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/activation_bench.py [--reps 7] [--warmup 2] [--only C3 C2]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from custom_loss_bench import gpu_info, median, timed  # noqa: E402

WORKLOADS = {
    "C3": dict(sizes=[4096, 4096, 4096, 4096, 4096, 1000], N=8192, reparam="local", S=1),
    "C2": dict(sizes=[784, 1200, 1200, 10], N=1024, reparam="weight", S=10),
}
KINDS = ("relu", "tanh", "sigmoid", "elu")
CLASSES = ("fwd", "fwd_lrt", "dx", "dx_lrt")


def run(ctx, name, w, reps, warmup):
    import torch
    import vbnn_b200
    sizes, N, S = w["sizes"], w["N"], w["S"]
    C = sizes[-1]
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(C)], S=S,
                                B=100.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.001, reparam=w["reparam"],
                                precision="bf16", strict_reference=False, log=False, seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    gen = torch.Generator().manual_seed(3)
    X = torch.randn(N, sizes[0], generator=gen).cuda()
    T = torch.randint(1, C + 1, (N,), generator=gen).float().cuda()
    step = lambda: net.train_step(X, T, sync=False)
    launches = {}
    for kind in KINDS:
        net.set_activation(kind)
        for _ in range(max(warmup, 2)):          # eager, then capture
            step()
        n0 = net.launch_count()
        step()
        launches[kind] = net.launch_count() - n0
    times = {k: [] for k in KINDS}
    for _ in range(reps):
        for kind in KINDS:
            net.set_activation(kind)
            step()                               # re-captures the graph of this kind (untimed)
            times[kind].append(timed(step))
    gemm_ms = {}
    for kind in KINDS:
        net.set_activation(kind)
        torch.cuda.synchronize()
        ctx.profile(True)
        step()
        torch.cuda.synchronize()
        prof = ctx.profile_read()
        ctx.profile(False)
        gemm_ms[kind] = {c: round(prof[c][0], 4) for c in CLASSES if c in prof}
    torch.cuda.synchronize()
    del net
    torch.cuda.empty_cache()
    med = {k: median(v) for k, v in times.items()}
    return dict(workload=name, S=S, N=N, sizes=sizes, reparam=w["reparam"],
                step_ms={k: round(v, 4) for k, v in med.items()},
                spread_ms={k: [round(min(v), 4), round(max(v), 4)] for k, v in times.items()},
                over_relu={k: round(med[k] / med["relu"], 4) for k in KINDS}, gemm_ms=gemm_ms, launches=launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("activation_bench: no GPU", file=sys.stderr)
        sys.exit(2)
    import vbnn_b200
    ctx = vbnn_b200.default_context(0, seed=5)
    out = dict(gpu_info(), reps=a.reps, results=[])
    for name in a.only:
        out["results"].append(run(ctx, name, WORKLOADS[name], a.reps, a.warmup))
        print(json.dumps(out["results"][-1]), file=sys.stderr)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
