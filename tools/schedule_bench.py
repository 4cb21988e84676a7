"""Time the fused minibatch with and without a hyper-parameter set (MLP.set_opt -> vbnn_mlp_set_opts) before every step,
in one process, alternating the two arms on one net.  The "set" arm walks a learning-rate decay with a KL warm-up (B
changes at every step), so every set writes new values; neither arm re-captures a step graph.

Workloads: bench.py's C1 (launch-bound: one more launch per step shows most there), C2 and C3, each at bench.py's
sizes, batch, S, reparameterisation and precision.  Per workload and arm: the median over the alternating windows of
the CUDA-event ms per step of a window of `--steps` steps (host work of the set included, as a training loop pays it),
the launches per step, and the step graph captures during the timed windows.  Prints one JSON object; the GPU name and
power limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/schedule_bench.py [--reps 7] [--warmup 3] [--only c1 c2 c3]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STEPS = {"c1": 200, "c2": 50, "c3": 20}          # per timed window: >= ~50 ms of work on a B200


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def median(v):
    return sorted(v)[len(v) // 2]


def run(ctx, name, w, steps, reps, warmup):
    import torch
    import vbnn_b200
    sizes, N = w["sizes"], w["N"]
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=w["S"], B=w["B"], batchSize=N, testBatchSize=N, mu_init=1, var_init=0.001,
                                reparam=w["reparam"], precision=w["precision"], strict_reference=False, log=False,
                                seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    gen = torch.Generator().manual_seed(3)
    data = [(torch.randn(N, sizes[0], generator=gen).cuda(),
             torch.randint(1, sizes[-1] + 1, (N,), generator=gen).float().cuda()) for _ in range(2)]
    count = [0]

    def scheduled():
        """a decaying rate and a KL weight warming up towards w["B"]: new values at every call"""
        i = count[0] = count[0] + 1
        decay = 1.0 / (1.0 + 1e-3 * (i % 1000))
        o = dict(opt, B=w["B"] * (1.0 + 10.0 / (1 + i % 1000)))
        o["meanState"] = dict(opt["meanState"], learningRate=opt["meanState"]["learningRate"] * decay)
        o["varState"] = dict(opt["varState"], learningRate=opt["varState"]["learningRate"] * decay)
        o["state"] = dict(opt["state"], learningRate=opt["state"]["learningRate"] * decay)
        return o

    def window(with_set):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0, c0 = net.launch_count(), net.graph_captures()
        e0.record()
        for s in range(steps):
            if with_set:
                net.set_opt(scheduled())
            X, T = data[s & 1]
            net.train_step(X, T, sync=False)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / steps, (net.launch_count() - l0) / steps, net.graph_captures() - c0

    for _ in range(warmup):
        window(False)
        window(True)
    res = {False: [], True: []}
    for _ in range(reps):                             # alternating: drifts in clock / power hit both arms alike
        for arm in (False, True):
            res[arm].append(window(arm))
    out = dict(workload=name, N=N, S=w["S"], sizes=sizes, steps_per_window=steps)
    for arm, key in ((False, "no_set"), (True, "set_every_step")):
        ms = [r[0] for r in res[arm]]
        out[key] = dict(ms_per_step=round(median(ms), 5), ms_range=[round(min(ms), 5), round(max(ms), 5)],
                        launches_per_step=res[arm][0][1], captures_in_timed_windows=sum(r[2] for r in res[arm]))
    out["set_over_no_set"] = round(out["set_every_step"]["ms_per_step"] / out["no_set"]["ms_per_step"], 4)
    del net
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", nargs="*", default=["c1", "c2", "c3"])
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print("schedule_bench: no GPU", file=sys.stderr)
        sys.exit(2)
    import vbnn_b200
    from bench import WORKLOADS
    ctx = vbnn_b200.default_context(0, seed=5)
    out = dict(gpu_info(), reps=a.reps, results=[])
    for name in a.only:
        out["results"].append(run(ctx, name, WORKLOADS[name], STEPS[name], a.reps, a.warmup))
        print(json.dumps(out["results"][-1]), file=sys.stderr)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
