"""Time vbnn_mlp_predict against vbnn_mlp_test at T samples, in one process, alternating the two.

Default workload: C3 (4096-4096x4-1000, local reparameterisation, bf16 GEMMs), N = 8192 rows, S = 1, T in {1, 8, 32}.
Both calls run the same sampled forward passes; test() scores each pass into two scalars, predict() folds every
pass into the per-(row, class) log-sum-exp state of the Bayesian average.  Calls are timed with CUDA events after
warm-up (both return host scalars, so both end in a stream synchronise).  A separate profiled call per T gives the
forward GEMM rate (profile classes 1 and 2) and the time and bytes of the averaging kernel (class 8).  Prints one
JSON object; the GPU name and power limit are read in the same run.  Without a GPU it exits non-zero.

    python tools/predict_bench.py [--T 1 8 32] [--N 8192] [--reps 5] [--warmup 2]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

C3 = dict(sizes=[4096, 4096, 4096, 4096, 4096, 1000], S=1, reparam="local", precision="bf16", B=100.0)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, nargs="+", default=[1, 8, 32])
    ap.add_argument("--N", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=5, help="timed calls of each entry point per T")
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("predict_bench: no CUDA device (there is no CPU fallback)")
    import vbnn_b200
    w = C3
    s = w["sizes"]
    ctx = vbnn_b200.default_context(0, seed=5)
    opt = vbnn_b200.default_opt(input_size=s[0], hidden=s[1:-1], classes=[str(i) for i in range(s[-1])], S=w["S"],
                                B=w["B"], batchSize=a.N, reparam=w["reparam"], precision=w["precision"], log=False)
    net = vbnn_b200.MLP(opt, ctx, max_batch=a.N)
    net.init_params(seed=4, he_means=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn(a.N, s[0], device="cuda", generator=g)
    Tt = torch.randint(1, s[-1] + 1, (a.N,), device="cuda", generator=g).float()
    net.train_step(X, Tt)                                     # a trained step: non-trivial posterior state
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        ev0.record()
        fn()
        ev1.record()
        ev1.synchronize()
        return ev0.elapsed_time(ev1)

    rows = []
    for T in a.T:
        net.opt["testSamples"], net.opt["quicktest"] = T, False
        run_test = lambda: net.test(X, Tt)
        run_pred = lambda: net.predict(X, n_samples=T, targets=Tt)
        for _ in range(a.warmup):
            run_test(); run_pred()
        t_ms, p_ms = [], []
        for _ in range(a.reps):                               # alternating: drifts in clock / power hit both alike
            t_ms.append(timed(run_test))
            p_ms.append(timed(run_pred))
        ctx.profile(True)
        try:
            pred = run_pred()
            prof = ctx.profile_read()
        finally:
            ctx.profile(False)
        fwd_ms = sum(prof[k][0] for k in ("fwd", "fwd_lrt") if k in prof)
        fwd_fl = sum(prof[k][2] for k in ("fwd", "fwd_lrt") if k in prof)
        k_ms, k_n, k_bytes = prof["predict"]
        tm, pm = sorted(t_ms)[len(t_ms) // 2], sorted(p_ms)[len(p_ms) // 2]
        rows.append(dict(
            T=T, test_ms=round(tm, 3), predict_ms=round(pm, 3), predict_over_test=round(pm / tm, 4),
            test_ms_all=[round(v, 3) for v in t_ms], predict_ms_all=[round(v, 3) for v in p_ms],
            test_rows_per_s=round(a.N / tm * 1e3), predict_rows_per_s=round(a.N / pm * 1e3),
            forward_tflops=round(fwd_fl / fwd_ms / 1e9, 1) if fwd_ms else None,
            predict_kernel=dict(launches=k_n, ms=round(k_ms, 4), share_of_predict_call=round(k_ms / pm, 4),
                                gb_per_s=round(k_bytes / k_ms / 1e6, 1), bytes=k_bytes),
            nll=pred.nll, accuracy=pred.accuracy, mean_mutual_info=float(pred.mutual_info.mean())))
    out = dict(workload="C3 4096-4096x4-1000, local reparameterisation, bf16 GEMMs", N=a.N, S=w["S"],
               reps=a.reps, warmup=a.warmup, timing="median of CUDA-event times per call", **gpu_info(), results=rows)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
