"""Time the fused regression minibatch (vbnn_mlp_set_criterion(VBNN_CRIT_GAUSSIAN_NLL) + vbnn_mlp_step) against the
split minibatch under the equivalent torch loss (vbnn_mlp_forward_train + torch + vbnn_mlp_backward_update) and against
the fused classification step of the same topology, in one process, alternating the three.

Workloads (bf16 GEMMs), each with a heteroscedastic Gaussian head (C = 2K outputs: K means, K log-variances):
  C3     4096-4096x4-1000, N = 8192, local reparameterisation, S = 1: a 500-output Gaussian head;
  C2     784-1200-1200-2, N = 1024, weight mode, S = 10: one Gaussian output (UCI-style regression);
  C4     the 256-100-2 VB head of BASELINE C4 (vb_output = 1, weight mode, N = 512) at S = 1 and S = 10.
The classification arm uses the same sizes under ClassNLL (C classes).  Per workload: the median CUDA-event ms over
alternating calls of each arm, the ratios, and from one profiled call of each fused arm the time of its "loss" phase
(k_loss_reg, or k_loss [+ the H = G .* R pass of an LRT output layer]).  Prints one JSON object; the GPU name and power
limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/regression_bench.py [--reps 7] [--warmup 3] [--only C3 C2 C4]"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from custom_loss_bench import gpu_info, median, timed  # noqa: E402

WORKLOADS = {
    "C3": dict(sizes=[4096, 4096, 4096, 4096, 4096, 1000], N=8192, reparam="local", S=[1], vb_output=False),
    "C2": dict(sizes=[784, 1200, 1200, 2], N=1024, reparam="weight", S=[10], vb_output=False),
    "C4": dict(sizes=[256, 100, 2], N=512, reparam="weight", S=[1, 10], vb_output=True),
}


def run(ctx, name, w, S, reps, warmup):
    import torch
    import vbnn_b200
    sizes, N = w["sizes"], w["N"]
    C = sizes[-1]
    K = C // 2

    def build(criterion):
        opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(C)],
                                    criterion=criterion, S=S, B=100.0, batchSize=N, testBatchSize=N, mu_init=1,
                                    var_init=0.001, reparam=w["reparam"], precision="bf16", strict_reference=False,
                                    log=False, seed=5, vb_output=w["vb_output"])
        net = vbnn_b200.MLP(opt, ctx, max_batch=N)
        net.init_params(seed=4, he_means=True)
        return net
    reg, cls = build("gaussian_nll"), build("class_nll")
    gen = torch.Generator().manual_seed(3)
    X = torch.randn(N, sizes[0], generator=gen).cuda()
    y = torch.randn(N, K, generator=gen).cuda()
    T = torch.randint(1, C + 1, (N,), generator=gen).float().cuda()

    def loss_fn(Y):
        m, s = Y[..., :K], Y[..., K:]
        return (0.5 * (s + (y - m) ** 2 * torch.exp(-s))).mean(dim=(1, 2)).sum()

    arms = {"fused": lambda: reg.train_step(X, y, sync=False), "split": lambda: reg.train_step_loss(X, loss_fn),
            "class": lambda: cls.train_step(X, T, sync=False)}
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    times = {k: [] for k in arms}
    for _ in range(reps):                       # alternating: drifts in clock / power hit all arms alike
        for k, fn in arms.items():
            times[k].append(timed(fn))
    med = {k: median(v) for k, v in times.items()}
    loss_ms = {}
    for arm in ("fused", "class"):
        ctx.profile(True)
        arms[arm]()
        torch.cuda.synchronize()
        loss_ms[arm] = ctx.phase_read()["loss"][0]
        ctx.profile(False)
    launches = {}
    for arm in ("fused", "class"):
        net = reg if arm == "fused" else cls
        n0 = net.launch_count()
        arms[arm]()
        launches[arm] = net.launch_count() - n0
    torch.cuda.synchronize()
    del reg, cls
    torch.cuda.empty_cache()
    return dict(workload=name, S=S, N=N, sizes=sizes, fused_ms=round(med["fused"], 4), split_ms=round(med["split"], 4),
                class_ms=round(med["class"], 4), split_over_fused=round(med["split"] / med["fused"], 4),
                fused_over_class=round(med["fused"] / med["class"], 4), k_loss_reg_ms=round(loss_ms["fused"], 4),
                class_loss_phase_ms=round(loss_ms["class"], 4), launches_fused=launches["fused"],
                launches_class=launches["class"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("regression_bench: no GPU", file=sys.stderr)
        sys.exit(2)
    import vbnn_b200
    ctx = vbnn_b200.default_context(0, seed=5)
    out = dict(gpu_info(), reps=a.reps, results=[])
    for name in a.only:
        for S in WORKLOADS[name]["S"]:
            out["results"].append(run(ctx, name, WORKLOADS[name], S, a.reps, a.warmup))
            print(json.dumps(out["results"][-1]), file=sys.stderr)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
