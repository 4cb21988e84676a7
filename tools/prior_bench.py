"""Time the fused minibatch under the three prior kinds of vbnn_layer_set_prior, in one process, alternating the kinds
on one net (set_prior between calls; each kind keeps its own warmed-up step graph only until the next switch, so
every timed call is preceded by one untimed call of the same kind that re-captures the graph).

Workloads (bf16 GEMMs):
  C3     4096-4096x4-1000, N = 8192, local reparameterisation, S = 1;
  C2     784-1200-1200-10, N = 1024, weight mode, S = 10.
Per workload and kind: the median CUDA-event ms of the whole step over the alternating calls, and the median (and
range) over as many profiled steps, in a loop of their own, of the fused KL + Adam update's time (profile class 7,
summed over the VB layers) with its algorithmic bytes (56 B per weight, 64 under PER_WEIGHT) over that median.
Prints one JSON object; the GPU name and power limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/prior_bench.py [--reps 7] [--warmup 3] [--only C3 C2]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "C3": dict(sizes=[4096, 4096, 4096, 4096, 4096, 1000], N=8192, reparam="local", S=1),
    "C2": dict(sizes=[784, 1200, 1200, 10], N=1024, reparam="weight", S=10),
}
KINDS = ("empirical", "fixed", "per_weight")


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


def run(ctx, name, w, reps, warmup):
    import torch
    import vbnn_b200
    sizes, N = w["sizes"], w["N"]
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=w["S"], B=100.0, batchSize=N, testBatchSize=N, mu_init=1, var_init=0.001,
                                reparam=w["reparam"], precision="bf16", strict_reference=False, log=False, seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    gen = torch.Generator().manual_seed(3)
    X = torch.randn(N, sizes[0], generator=gen).cuda()
    T = torch.randint(1, sizes[-1] + 1, (N,), generator=gen).float().cuda()
    step = lambda: net.train_step(X, T, sync=False)

    def switch(kind):
        net.set_prior(kind, 0.0, 0.01)                 # per_weight: a snapshot of the current posterior
        step()                                         # untimed: re-captures the step graph
        step()

    for _ in range(warmup):
        for kind in KINDS:
            switch(kind)
    times = {k: [] for k in KINDS}
    for _ in range(reps):                              # alternating: drifts in clock / power hit every kind alike
        for kind in KINDS:
            switch(kind)
            times[kind].append(timed(step))
    out = dict(workload=name, S=w["S"], N=N, sizes=sizes)
    upd = {k: [] for k in KINDS}
    for _ in range(reps):                              # profiled steps in a loop of their own, kinds alternated
        for kind in KINDS:
            switch(kind)
            torch.cuda.synchronize()
            ctx.profile(True)
            step()
            torch.cuda.synchronize()
            ms, launches, nbytes = ctx.profile_read()["update"]
            ctx.profile(False)
            upd[kind].append((ms, launches, nbytes))
    for kind in KINDS:
        ms = median([u[0] for u in upd[kind]])
        _, launches, nbytes = upd[kind][0]
        out[kind] = dict(step_ms=round(median(times[kind]), 4), update_ms=round(ms, 4),
                         update_ms_range=[round(min(u[0] for u in upd[kind]), 4), round(max(u[0] for u in upd[kind]), 4)],
                         update_launches=launches, update_bytes=int(nbytes),
                         update_TBps=round(nbytes / (ms * 1e-3) / 1e12, 3) if ms else None)
    out["per_weight_over_empirical_update"] = round(out["per_weight"]["update_ms"] / out["empirical"]["update_ms"], 4)
    del net
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", nargs="*", default=list(WORKLOADS))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("prior_bench: no GPU", file=sys.stderr)
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
