"""Time the split minibatch (vbnn_mlp_forward_train + a torch ClassNLL + vbnn_mlp_backward_update) against the fused
vbnn_mlp_step, in one process, alternating the two on one net.

Workloads (bf16 GEMMs):
  C3     4096-4096x4-1000, N = 8192, local reparameterisation, S = 1;
  C2     784-1200-1200-10, N = 1024, weight mode, S = 10;
  C4     the 256-100-10 VB head of BASELINE C4 (vb_output = 1, weight mode, N = 512) at S = 1 and S = 10, on fixed
         features: a conv extractor below it would run the same work in both arms.
The split arm's loss is sum_s nll_loss(log_softmax(Y_s)) through torch autograd, i.e. what the fused step computes.
Per workload: the median CUDA-event ms over alternating calls of each arm and their ratio; from one profiled call of
each, the time of the "loss" phase -- k_grad_logits alone in the split arm, k_loss (+ the H = G .* R pass of an LRT
output layer) in the fused one -- and k_grad_logits' algorithmic bytes (fp32 gradient read, G written over its padded
width, R read and H written for an LRT output layer) over its time.  Prints one JSON object; the GPU name and power
limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/custom_loss_bench.py [--reps 7] [--warmup 3] [--only C3 C2 C4]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "C3": dict(sizes=[4096, 4096, 4096, 4096, 4096, 1000], N=8192, reparam="local", S=[1], vb_output=False),
    "C2": dict(sizes=[784, 1200, 1200, 10], N=1024, reparam="weight", S=[10], vb_output=False),
    "C4": dict(sizes=[256, 100, 10], N=512, reparam="weight", S=[1, 10], vb_output=True),
}


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


def run(ctx, name, w, S, reps, warmup):
    import torch
    import torch.nn.functional as F
    import vbnn_b200
    sizes, N = w["sizes"], w["N"]
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=S, B=100.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.001,
                                reparam=w["reparam"], precision="bf16", strict_reference=False, log=False, seed=5,
                                vb_output=w["vb_output"])
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    gen = torch.Generator().manual_seed(3)
    X = torch.randn(N, sizes[0], generator=gen).cuda()
    T = torch.randint(1, sizes[-1] + 1, (N,), generator=gen).float().cuda()
    t0 = T.long() - 1

    def loss_fn(Y):
        return sum(F.nll_loss(F.log_softmax(Y[s], -1), t0) for s in range(Y.shape[0]))

    fused = lambda: net.train_step(X, T, sync=False)
    split = lambda: net.train_step_loss(X, loss_fn)
    for _ in range(warmup):
        fused(); split()
    ta, tb = [], []
    for _ in range(reps):                       # alternating: drifts in clock / power hit both alike
        ta.append(timed(fused))
        tb.append(timed(split))
    ma, mb = median(ta), median(tb)
    phases = {}
    for arm, fn in (("fused", fused), ("split", split)):
        ctx.profile(True)
        fn()
        torch.cuda.synchronize()
        phases[arm] = ctx.phase_read()
        ctx.profile(False)
    C, ld = sizes[-1], (sizes[-1] + 7) // 8 * 8
    lrt_out = w["reparam"] == "local" and w["vb_output"]
    rows = S * N
    nbytes = rows * (4 * C + 2 * ld) + (rows * 2 * C * 2 if lrt_out else 0)
    gl_ms = phases["split"]["loss"][0]
    del net
    torch.cuda.empty_cache()
    return dict(workload=name, S=S, N=N, sizes=sizes, fused_ms=round(ma, 4), split_ms=round(mb, 4),
                ratio=round(mb / ma, 4), fused_loss_phase_ms=round(phases["fused"]["loss"][0], 4),
                k_grad_logits_ms=round(gl_ms, 4), k_grad_logits_bytes=nbytes,
                k_grad_logits_GBps=round(nbytes / (gl_ms * 1e-3) / 1e9, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("custom_loss_bench: no GPU", file=sys.stderr)
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
