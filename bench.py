#!/usr/bin/env python
"""bench.py -- VB-MLP train samples/sec on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--workload c3|c2|c1] [--scaling weak|strong]
                  [--batch ROWS_PER_GPU] [--impl reference] [--dump-outputs DIR]

One "step" = one minibatch of main.lua:28-40: S x (sample, forward, loss, backward), the gradient exchange
when N > 1, and the fused KL + Adam update.  Default workload: BASELINE configs[2], the wide VB-MLP
4096-4096x4-1000, batch 8192 per GPU, local reparameterisation, bf16 GEMMs with fp32 accumulate -- the config
the metric's "tensor-pipe % of peak" is quoted on.

Prints ONE JSON line (rank 0):
  value / ms_per_step   device-resident throughput over exactly K timed minibatches (CUDA events, max over ranks;
                        the library's auxiliary streams are joined before the closing event);
  e2e, e2e_u8           the same metric through the public host-buffer API (pinned fp32 -- the reference's format
                        -- or the dataset's native uint8 bytes), H2D of every minibatch + D2H of its loss inside;
  roofline              the dominant kernel instantiation (largest share of the step), from CUDA events around
                        every tensor-core GEMM launch during an instrumented repeat of the same K minibatches;
                        roofline_all_gemms = all tensor-core GEMM launches together; roofline_hbm = k_update;
  cpu_baseline          the oracle ("port" of the reference's Torch7 CPU path, which cannot run here), 8 threads
                        (config.lua:5); a full timed minibatch for C1 / C2, a bounded row sample for C3 (flagged);
  extra_workloads       (N = 1) BASELINE configs[0] and [1] -- C1, C2 -- measured the same way in the same run;
  strong_scaling        (N > 1) the same network with the GLOBAL batch fixed at 8192 rows (BASELINE configs[2]
                        read as strong scaling; at N = 8 that is 1024 rows per GPU, the hard regime);
  dp_parity             (N > 1) a short data-parallel-vs-single-GPU parity check run before timing; the run fails
                        if it is not ok.
Every timed loop runs exactly K minibatches (extra_workloads: 500 unless --steps is given; their warm-up stays 20).
--dump-outputs DIR (one GPU; DIR must hold no .npy files yet) writes what the last timed minibatch left the caller as DIR/<name>.npy, float32: see
dump_outputs().  Inputs, initial parameters and noise are seeded, so two builds run with the same arguments can be
compared array for array.  Compare with a tolerance: fp32 atomics (bias gradients, the loss sum) make two runs of the
same build differ in the last bits, and bf16 operands carry that forward -- two C3 runs of 10 + 50 minibatches on one
B200 (1000 W power limit) differed by <= 7e-4 relative (Frobenius norm) per array, 2.3e-3 on the worst log-probability.
The oracle is only ever the checker / CPU baseline, never the product."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CPU_THREADS = 8          # opt.threads (config.lua:5, main.lua:142)

WORKLOADS = {
    # name: sizes, per-GPU batch, S, reparam, precision, B (trainSize/N)
    "c1": dict(sizes=[784, 100, 10], N=100, S=1, reparam="weight", precision="fp32", B=600.0,
               l2="no flush: the whole working set (78 k weights x 36 B + activations < 4 MB) is L2-resident in real "
                  "training too; two alternating input minibatches",
               desc="mlp.lua VBLinear MLP 784-100-10, batch 100, 1 weight sample (BASELINE configs[0])"),
    "c2": dict(sizes=[784, 1200, 1200, 10], N=1024, S=10, reparam="weight", precision="bf16", B=58.59,
               l2="working set (2.38 M weights x 36 B state + 10 sampled bf16 weight sets + 10 x activations ~ 200 MB) "
                  "> 126 MB L2; two alternating input minibatches",
               desc="VBLinear MLP 784-1200-1200-10, batch 1024, 10 MC weight samples (BASELINE configs[1])"),
    "c3": dict(sizes=[4096, 4096, 4096, 4096, 4096, 1000], N=8192, S=1, reparam="local", precision="bf16",
               B=100.0,
               l2="working set (parameters + optimizer state + activations ~ 3.3 GB) >> 126 MB L2; two alternating "
                  "input minibatches",
               desc="wide VB-MLP 4096-4096x4-1000, local reparameterization, batch 8192/GPU, bf16 GEMMs fp32 "
                    "accumulate (BASELINE configs[2])"),
}


def flops_per_sample(w):
    """SURVEY.md 8(d): weight sampling c=4 (first layer) / 6; LRT c=8 / 12; plain nn.Linear output c=6."""
    s = w["sizes"]
    lrt = w["reparam"] == "local"
    total = 0
    for j in range(len(s) - 1):
        last = j == len(s) - 2
        if last:
            c = 6
        elif lrt:
            c = 8 if j == 0 else 12
        else:
            c = 4 if j == 0 else 6
        total += c * s[j] * s[j + 1]
    return w["S"] * total


def config_dict(w, world, n_per_gpu, scaling):
    """The workload description; identical in the GPU arm and the --impl reference arm."""
    return dict(workload=w["desc"], sizes=w["sizes"], global_batch=n_per_gpu * world, per_gpu_batch=n_per_gpu,
                S=w["S"], reparam=w["reparam"], parallelism=f"dp{world}", scaling=scaling,
                output_layer="nn.Linear (mlp.lua:29)", l2=w["l2"], flops_per_sample=flops_per_sample(w))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=float(d["bf16_tflops_sustained"]), tflops_burst=float(d["bf16_tflops"]),
                    hbm=float(d["hbm_gbs"]), source="measured (MEASURED_PEAKS.json, sustained)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=10)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                self.proc.wait()

    def summary(self, t0, t1):
        sm, mx, reasons, pw = [], 0.0, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                c, m = float(f[0]), float(f[1])
            except ValueError:
                continue
            mx = max(mx, m)
            if t0 - 0.05 <= t <= t1 + 0.05:
                sm.append(c)
                try:
                    pw.append(float(f[2]))
                except ValueError:
                    pass
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        if not sm:
            sm = [float(l.split(",")[0]) for _, l in self.rows[-3:] if l and l.split(",")[0].strip().replace(".", "").isdigit()] or [0.0]
        return dict(sm_mhz=statistics.median(sm), sm_min_mhz=min(sm), sm_max_mhz=mx, reasons=sorted(reasons),
                    samples=len(sm), power_w_max=max(pw) if pw else None)


def bind_to_gpu_numa_node(index):
    """Host side of the end-to-end path: run this rank's host thread (and so first-touch its pinned staging
    buffers) on the NUMA node the GPU hangs off.  Best effort; returns the node or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, z = part.partition("-")
            cpus.update(range(int(a), int(z or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:                                            # noqa: BLE001
        pass
    return None


def build_net(w, ctx, N):
    import vbnn_b200
    s = w["sizes"]
    opt = vbnn_b200.default_opt(input_size=s[0], hidden=s[1:-1], classes=[str(i) for i in range(s[-1])],
                                S=w["S"], B=w["B"], batchSize=N, testBatchSize=N, mu_init=1, msr_init=False,
                                var_init=0.001,
                                reparam=w["reparam"], precision=w["precision"], strict_reference=False, log=False,
                                seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    return net, opt


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's Torch7 CPU path, CPU_THREADS threads
# ------------------------------------------------------------------------------------------------
def cpu_baseline(w, n_global=None, threads=CPU_THREADS):
    """One minibatch of main.lua:19-51 through the oracle (fp32, the reference's exact op sequence: redundant
    GEMM Q2, first-layer dX, host Gaussian fill).  C1 / C2: the FULL minibatch is timed.  C3 (6e12 flop per
    minibatch, ~10 s on 8 cores): a bounded row sample through the full-size net plus ONE full-size update is
    timed and scaled to the full batch -- `estimated` says so and `seconds_timed` is what was really spent."""
    import numpy as np
    import torch
    from oracle import vbnn_oracle as O
    torch.set_num_threads(threads)
    s = w["sizes"]
    N = n_global or w["N"]
    opt = O.default_opt(input_size=s[0], hidden=s[1:-1], classes=[str(i) for i in range(s[-1])], S=w["S"],
                        B=w["B"], batchSize=N, mu_init=1, msr_init=False, var_init=0.001, reparam=w["reparam"],
                        strict_reference=False)
    net = O.MLPOracle(opt, torch.float32, seed=3)
    budget = 2.0e11                                                     # flop of forward / backward per timed step
    rows = N if flops_per_sample(w) * N <= budget else max(16, int(budget / flops_per_sample(w)))
    rows = min(rows, N)
    rng = np.random.RandomState(0)
    X = torch.from_numpy(rng.randn(rows, s[0]).astype(np.float32))
    T = torch.from_numpy(rng.randint(1, s[-1] + 1, rows).astype(np.float32))
    t0 = time.perf_counter()
    net.resetGradients()
    for _ in range(opt["S"]):
        net.sample()                                   # host randomkit-style Gaussian fill, as the reference
        net.run(X, T)
    t_fb = time.perf_counter() - t0
    t0 = time.perf_counter()
    net.update(opt)
    t_up = time.perf_counter() - t0
    estimated = rows < N
    full = t_fb * (N / rows) + t_up
    if estimated:
        sample = (f"{rows} of {N} rows x S={w['S']} through the full-size net ({t_fb:.2f} s) + one full update "
                  f"({t_up:.2f} s), fp32 torch-CPU oracle, scaled to the full minibatch")
    else:
        sample = f"one full minibatch ({N} rows x S={w['S']} + update) timed: {full:.3f} s, fp32 torch-CPU oracle"
    return dict(value=N / full, unit="samples/s", cores=threads, kind="port", sample=sample, estimated=estimated,
                rows_timed=rows, seconds_timed=t_fb + t_up, host_cpus=os.cpu_count())


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    n_per_gpu = args.batch or (w["N"] // world if args.scaling == "strong" else w["N"])
    n_global = n_per_gpu * world
    vals, spent = [], []
    for i in range(args.warmup + args.steps):
        r = cpu_baseline(w, n_global)
        if i >= args.warmup:
            vals.append(r)
            spent.append(r["seconds_timed"])
    v = statistics.mean(x["value"] for x in vals)
    r = dict(vals[-1])
    r["value"] = v
    line = dict(metric="VB-MLP train samples/sec", value=v, unit="samples/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup,
                # wall time really spent per timed step (for C3: the bounded sample, NOT a full minibatch)
                ms_per_step=1e3 * statistics.mean(spent),
                estimated=r["estimated"], ms_per_full_step_estimated=1e3 * n_global / v,
                higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f32", data="synthetic",
                impl="reference", config=config_dict(w, world, n_per_gpu, args.scaling),
                cpu_baseline=r, e2e=dict(value=v, unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Env:
    """Per-process plumbing: rank, torch.distributed, the libvbnn context."""

    def __init__(self, args):
        import torch
        import vbnn_b200
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", rank=self.rank, world_size=self.world,
                                    device_id=torch.device(f"cuda:{self.local_rank}"))
            self.dist = dist
        self.numa = bind_to_gpu_numa_node(self.local_rank)
        self.ctx = vbnn_b200.Context(self.local_rank, seed=5)
        if self.world > 1:
            self.ctx.init_comm(self.rank, self.world, self._bcast)
        self.dp_mode = "single" if self.world == 1 else os.environ.get("VBNN_DP", "peer")
        self.dev = f"cuda:{self.local_rank}"

    def _bcast(self, buf):
        torch = self.torch
        t = torch.zeros(128, dtype=torch.uint8, device=self.dev if hasattr(self, "dev") else f"cuda:{self.local_rank}")
        if self.rank == 0:
            t.copy_(torch.tensor(list(buf), dtype=torch.uint8))
        self.dist.broadcast(t, 0)
        return bytes(t.cpu().tolist())

    def gather_bytes(self, blob):
        torch = self.torch
        t = torch.tensor(list(blob), dtype=torch.uint8, device=self.dev)
        out = [torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [bytes(o.cpu().tolist()) for o in out]

    def barrier(self):
        """Every rank first drains ALL of its own streams (the peer-mode side stream included), then meets the
        others: after the barrier nobody's device still writes into a peer's buffers."""
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.dist is None:
            return ms
        t = self.torch.tensor([ms], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0])

    def make_net(self, w, N):
        """Build the net on this rank and, for N > 1, switch on the data-parallel exchange (peer mode unless
        VBNN_DP=nccl or CUDA IPC is unavailable on any rank)."""
        torch = self.torch
        net, opt = build_net(w, self.ctx, N)
        if self.world > 1 and self.dp_mode == "peer":
            ok = 1
            try:
                net.enable_peer(self.gather_bytes)
            except Exception as e:                                   # noqa: BLE001
                ok = 0
                print(f"[bench rank {self.rank}] peer mode unavailable ({e}); falling back to NCCL allreduce",
                      file=sys.stderr)
            flag = torch.tensor([ok], device=self.dev)
            self.dist.all_reduce(flag, op=self.dist.ReduceOp.MIN)
            if int(flag[0]) == 0:
                if net.peer_active:
                    raise SystemExit("peer mode is active on this rank but not on all ranks")
                self.dp_mode = "nccl (peer mode unavailable)"
        return net, opt

    def drop_net(self, net):
        """Peers hold IPC mappings of this rank's buffers: nobody frees before everybody is done."""
        self.ctx.synchronize()
        self.barrier()
        del net
        import gc
        gc.collect()
        self.barrier()


def gemm_algorithmic_bytes(cls, w, N):
    """Operands read once + epilogue inputs read once + outputs written once, per launch of a hidden layer
    (the shape that dominates): what `traffic` (measured DRAM bytes per launch) is compared with."""
    H = w["sizes"][1]
    e = 2                                                               # bf16
    if cls == "fwd_lrt":      # split: mean GEMM (A, B -> aux fp32) and variance GEMM (A2, B2, aux -> act, act2, R): mean of both
        return ((N * H * e + H * H * e + N * H * 4) + (N * H * e + H * H * e + N * H * 4 + 3 * N * H * e)) // 2
    if cls == "dx_lrt":       # G, H, mu, s2 -> G_prev, H_prev (reads xprev, rprev)
        return 2 * N * H * e + 2 * H * H * e + 4 * N * H * e
    if cls == "dw_lrt":       # G, H, X, X2 -> gW, gS fp32
        return 4 * N * H * e + 2 * H * H * 4
    if cls == "fwd":
        return N * H * e + H * H * e + N * H * e
    if cls == "dx":
        return N * H * e + H * H * e + 2 * N * H * e
    if cls == "dw":
        return 2 * N * H * e + 2 * H * H * 4
    return None


DUMP_MAX_ELEMS = 1 << 18                 # per array; keeps a C3 dump near 10 MB


def dump_outputs(net, out_dir):
    """What a caller of train_step holds after the last minibatch: its [error, accuracy], the LogSoftMax outputs of
    its forward pass ([S x N x classes]) and every layer's updated parameters, as out_dir/<name>.npy in float32.  An
    array of more than DUMP_MAX_ELEMS elements is flattened and replaced by the elements at a fixed set of indices
    (seed 0, sorted): the same sample in every run."""
    import numpy as np
    import torch
    from vbnn_b200 import _lib as VL
    arrays = {"result": net._res, "logp": torch.stack([net.outputs(s) for s in range(net.opt["S"])])}
    for k, m in enumerate(net.model):
        if m.kind == VL.KIND_VB:
            arrays.update({f"layer{k}_means": m.means, f"layer{k}_lvars": m.lvars, f"layer{k}_bias": m.bias})
        else:
            arrays.update({f"layer{k}_weight": m.weight, f"layer{k}_bias": m.bias})
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if t.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def measure(env, args, w, N, steps, warmup, sampler=None, e2e=True, dump_dir=None):
    """Time `steps` minibatches of workload w at N rows per GPU.  Returns the measurement dict.  With dump_dir, the
    outputs of the last timed minibatch are written there (dump_outputs) before anything else runs on the net."""
    torch = env.torch
    world, rank, ctx = env.world, env.rank, env.ctx
    net, opt = env.make_net(w, N)
    g = torch.Generator(device="cpu").manual_seed(3 + rank)
    nbuf = 2
    Xd = [torch.randn(N, w["sizes"][0], generator=g).cuda() for _ in range(nbuf)]
    Td = [torch.randint(1, w["sizes"][-1] + 1, (N,), generator=g).float().cuda() for _ in range(nbuf)]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed_region():
        """EXACTLY K minibatches between barrier + synchronize on both sides; device time, max over ranks.  The
        closing event waits for the library's auxiliary streams (peer-mode side stream: the last minibatch's
        layer-0 shard update + operand push), so the tail is inside the timed region."""
        env.barrier()
        t0 = sampler.mark() if sampler else 0
        ev0.record()
        for i in range(steps):
            net.train_step(Xd[i % nbuf], Td[i % nbuf], sync=False)
        net.join_streams()
        ev1.record()
        env.barrier()
        t1 = sampler.mark() if sampler else 0
        return env.max_over_ranks(ev0.elapsed_time(ev1)), t0, t1

    # ---------------- device-resident throughput (value): the path a user gets -------------------
    for i in range(warmup):
        net.train_step(Xd[i % nbuf], Td[i % nbuf], sync=False)
    l0 = net.launch_count()
    ms, t_mark0, t_mark1 = timed_region()
    launches = net.launch_count() - l0
    if dump_dir:
        dump_outputs(net, dump_dir)
    out = dict(value=steps * N * world / (ms / 1e3), ms_per_step=ms / steps, gpu_launches=launches,
               marks=(t_mark0, t_mark1), per_gpu_batch=N, global_batch=N * world)
    # ---------------- the same K minibatches again with CUDA events around every GEMM / update launch
    # and phase marks inside the minibatch (roofline, phases).  Instrumenting turns graph replay off and
    # adds two event records per launch, so it is a separate pass: `value` carries no instrumentation.
    if w["precision"] == "bf16":
        ctx.profile(True)
        for i in range(3):
            net.train_step(Xd[i % nbuf], Td[i % nbuf], sync=False)
        ctx.profile(False); ctx.profile(True)                       # drop the warm-up records
        ms_prof, _, _ = timed_region()
        out["prof"] = ctx.profile_read()
        out["phases"] = ctx.phase_read()
        out["ms_prof"] = ms_prof
        ctx.profile(False)
    out["last_error"] = float(net._res.cpu()[0])

    # ---------------- end to end through the host-buffer API ------------------------------
    if e2e:
        def e2e_run(submit, bufs):
            for i in range(3):
                submit(*bufs[i % nbuf]); net.collect()
            env.barrier()
            ev0.record()
            submit(*bufs[0])
            for i in range(1, steps):
                submit(*bufs[i % nbuf])                        # copy of minibatch i overlaps compute of i-1
                net.collect()
            net.collect()
            net.join_streams()
            ev1.record()
            env.barrier()
            return env.max_over_ranks(ev0.elapsed_time(ev1))
        Xh = [x.cpu().pin_memory() for x in Xd]
        Th = [t.cpu().pin_memory() for t in Td]
        ms_e = e2e_run(net.submit_host, list(zip(Xh, Th)))
        out["e2e"] = dict(value=steps * N * world / (ms_e / 1e3), unit="samples/s",
                          h2d_bytes_per_step=N * w["sizes"][0] * 4 + N * 4, d2h_bytes_per_step=8,
                          api="vbnn_mlp_submit_host/vbnn_mlp_collect (pinned fp32 host minibatch -- the reference's "
                              "FloatTensor format, main.lua:23-24 -- double-buffered)")
        # the dataset's native bytes (MNIST pixels are uint8 before utils.lua:29-35 normalises them): 4x fewer
        # host bytes, (x - mean) / std fused into the operand staging kernel
        P8 = [torch.randint(0, 256, (N, w["sizes"][0]), generator=g, dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
        sub8 = lambda p, t: net.submit_host_u8(p, t, 127.5, 73.9)
        ms_8 = e2e_run(sub8, list(zip(P8, Th)))
        out["e2e_u8"] = dict(value=steps * N * world / (ms_8 / 1e3), unit="samples/s",
                             h2d_bytes_per_step=N * w["sizes"][0] + N * 4, d2h_bytes_per_step=8,
                             api="vbnn_mlp_submit_host_u8/vbnn_mlp_collect (pinned uint8 pixels, normalisation "
                                 "(utils.lua:29-35) fused on the device, double-buffered)")
    env.drop_net(net)
    return out


def roofline_objects(m, w, N, steps, peaks, is_c3=False):
    """roofline (dominant instantiation), roofline_all_gemms, roofline_hbm from one measurement."""
    prof = dict(m.get("prof") or {})
    upd = prof.pop("update", None)
    res = {}
    tpath = os.path.join(ROOT, "profiles", "r02_c3_traffic.json")
    traffic = json.load(open(tpath)) if os.path.exists(tpath) else {}
    if prof:
        ms_prof = m["ms_prof"]
        per_class = {}
        for k, v in prof.items():
            d = dict(tflops=v[2] / (v[0] / 1e3) / 1e12, ms_per_step=v[0] / steps, launches=v[1],
                     avg_launch_ms=v[0] / max(v[1], 1), share_of_step=v[0] / ms_prof)
            tr = traffic.get("per_class", {}).get(k) if is_c3 else None
            if tr:
                d["traffic_bytes_per_launch"] = tr.get("dram_bytes_per_launch")
                d["algorithmic_bytes_per_launch"] = tr.get("algorithmic_bytes_per_launch") or gemm_algorithmic_bytes(k, w, N)
            per_class[k] = d
        tot_ms = sum(v[0] for v in prof.values())
        tot_fl = sum(v[2] for v in prof.values())
        tot_n = sum(v[1] for v in prof.values())
        timed = ("CUDA events on the launching stream around every launch during an instrumented repeat of the K timed "
                 "minibatches (graph replay off); `value` is the un-instrumented pass")
        top = max(per_class, key=lambda k: per_class[k]["share_of_step"])
        t = per_class[top]
        res["roofline"] = dict(bound="tensor", kernel=f"gemm_tc_kernel, epilogue class {top} (tcgen05 bf16; the class with the "
                               "largest share of the step)", achieved=t["tflops"], peak=peaks["tflops"], unit="TFLOP/s",
                               frac=t["tflops"] / peaks["tflops"], peak_source=peaks["source"], peak_burst=peaks["tflops_burst"],
                               traffic=t.get("traffic_bytes_per_launch"), algorithmic_bytes=t.get("algorithmic_bytes_per_launch"),
                               traffic_source=traffic.get("source"), launches=t["launches"], avg_launch_ms=t["avg_launch_ms"],
                               share_of_step=t["share_of_step"], timed=timed)
        achieved = tot_fl / (tot_ms / 1e3) / 1e12
        res["roofline_all_gemms"] = dict(bound="tensor", kernel="gemm_tc_kernel (tcgen05 bf16, all epilogue classes)",
                                         achieved=achieved, peak=peaks["tflops"], unit="TFLOP/s", frac=achieved / peaks["tflops"],
                                         launches=tot_n, avg_launch_ms=tot_ms / max(tot_n, 1), share_of_step=tot_ms / ms_prof,
                                         instrumented_ms_per_step=ms_prof / steps, per_class=per_class)
    if upd:
        gbs = upd[2] / (upd[0] / 1e3) / 1e9
        res["roofline_hbm"] = dict(bound="hbm", kernel="k_update (fused KL + 2x Adam, 56 B/weight algorithmic)", achieved=gbs,
                                   peak=peaks["hbm"], unit="GB/s", frac=gbs / peaks["hbm"], launches=upd[1],
                                   avg_launch_ms=upd[0] / max(upd[1], 1), share_of_step=upd[0] / m["ms_prof"],
                                   peak_source=peaks["source"])
    if m.get("phases"):
        res["phases_ms_per_step"] = {k: v[0] / steps for k, v in m["phases"].items()}
    return res


def dp_parity_check(env):
    """Data-parallel vs single-GPU parity on the exact paths the scaling runs time: the C3 network (4096 wide: 256 x 256
    CTA-pair tiles, co-resident shard updates, operand all-gather), 1024 rows per rank, 3 minibatches, once per gradient
    transport -- dW tiles stored into every owner's slot from the epilogue ("fused", what the weak-scaling run uses),
    staged locally + moved by the copy engines ("copy_engine"), staged locally + moved and signalled by one co-resident
    copy kernel per layer ("copy_kernel", what the strong-scaling run uses).  After
    sync_replicas every rank must hold -- parameters AND Adam state -- what ONE GPU stepping the whole global minibatch
    holds (identical Philox noise: zeta is indexed by the global row).  Differences are fp32 summation order only."""
    torch, dist = env.torch, env.dist
    import vbnn_b200
    from vbnn_b200 import _lib as VL
    w = dict(WORKLOADS["c3"])
    n_loc, steps = 1024, 3
    Ng = n_loc * env.world
    g = torch.Generator().manual_seed(11)
    X = torch.randn(Ng, w["sizes"][0], generator=g)
    T = torch.randint(1, w["sizes"][-1] + 1, (Ng,), generator=g).float()
    adam_ids = (VL.BUF_ADAM_M_MU, VL.BUF_ADAM_V_MU, VL.BUF_ADAM_M_VAR, VL.BUF_ADAM_V_VAR)
    relf = lambda a, b: float((a.double() - b.double()).norm() / max(float(b.double().norm()), 1e-30))
    sg_par = sg_adam = None
    if env.rank == 0:                                                   # the single-GPU reference, once
        ctx1 = vbnn_b200.Context(env.local_rank, seed=5)                # no communicator: nranks = 1
        one, _ = build_net(w, ctx1, Ng)
        ctx1.set_step(7)
        Xg, Tg = X.cuda(), T.cuda()
        for _ in range(steps):
            one.train_step(Xg, Tg)
        sg_par = [m.means.clone() for m in one.model[:-1]] + [m.lvars.clone() for m in one.model[:-1]] + [one.model[-1].weight.clone()]
        sg_adam = [m.get(b) for m in one.model[:-1] for b in adam_ids]
        ctx1.synchronize()
        del one, Xg, Tg
        torch.cuda.set_stream(env.ctx.stream)
    res = dict(config=f"C3 network, {n_loc} rows/rank x {env.world} ranks, {steps} minibatches, exchange: {env.dp_mode}",
               tol_params=1e-4, tol_adam=1e-3, ok=True)
    transports = ([("fused", 1, 0), ("copy_engine", 2, 0), ("copy_kernel", 3, 0), ("copy_kernel_bf16_wire", 3, 1)]
                  if env.dp_mode == "peer" else [(env.dp_mode, 0, 0)])
    for name, knob, wire in transports:
        old = vbnn_b200.knob("peer_transport", knob)
        old_wire = vbnn_b200.knob("peer_wire_bf16", wire)
        # bf16 gradient tiles add one rounding point per rank (2^-9 relative on each partial sum): stated separately
        tol_p, tol_a = (1e-4, 1e-3) if not wire else (1e-3, 2e-2)
        net, _ = env.make_net(w, n_loc)
        env.ctx.set_step(7)
        env.barrier()
        lo = env.rank * n_loc
        Xl, Tl = X[lo:lo + n_loc].cuda(), T[lo:lo + n_loc].cuda()
        for _ in range(steps):
            net.train_step(Xl, Tl)
        env.barrier()                                                   # all streams of all ranks drained
        net.sync_replicas()
        env.barrier()
        same = True
        for m in net.model[:-1]:                                        # every rank holds identical parameters
            t = m.means.clone(); ref = t.clone(); dist.broadcast(ref, 0)
            same &= bool(torch.equal(ref, t))
        flag = torch.tensor([1 if same else 0], device=env.dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        r = dict(replicas_identical=bool(int(flag[0])))
        if env.rank == 0:
            dp_par = [m.means for m in net.model[:-1]] + [m.lvars for m in net.model[:-1]] + [net.model[-1].weight]
            dp_adam = [m.get(b) for m in net.model[:-1] for b in adam_ids]
            e_par = max(relf(a, b) for a, b in zip(dp_par, sg_par))
            e_adam = max(relf(a, b) for a, b in zip(dp_adam, sg_adam))
            t_ok = all(m.t == steps for m in net.model)
            r.update(max_rel_params=e_par, max_rel_adam=e_adam, step_counters_ok=t_ok, tol_params=tol_p, tol_adam=tol_a,
                     ok=bool(r["replicas_identical"] and e_par < tol_p and e_adam < tol_a and t_ok))
        ok = torch.tensor([1 if r.get("ok", True) else 0], device=env.dev)
        dist.broadcast(ok, 0)
        r["ok"] = bool(int(ok[0]))
        res[name] = r
        res["ok"] = res["ok"] and r["ok"]
        env.drop_net(net)
        vbnn_b200.knob("peer_transport", old)
        vbnn_b200.knob("peer_wire_bf16", old_wire)
    if env.rank == 0:
        res["max_rel"] = max(max(r.get("max_rel_params", 0.0), r.get("max_rel_adam", 0.0)) for k, r in res.items()
                             if isinstance(r, dict) and not k.endswith("bf16_wire"))      # fp32-wire transports
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=None, help="rows per GPU (overrides the workload / scaling default)")
    ap.add_argument("--impl", default="vbnn", choices=["vbnn", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip extra_workloads / strong_scaling / dp_parity")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed minibatch as DIR/<name>.npy (one GPU only)")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    if args.dump_outputs and (args.impl == "reference" or args.gpus != 1 or os.environ.get("WORLD_SIZE", "1") != "1"):
        ap.error("--dump-outputs needs --impl vbnn on one GPU")
    # arrays left by an earlier run (another workload has other layers) would pass for this run's
    if args.dump_outputs and os.path.isdir(args.dump_outputs) and any(
            f.endswith(".npy") for f in os.listdir(args.dump_outputs)):
        ap.error(f"--dump-outputs: {args.dump_outputs} already holds .npy files; give an empty or new directory")
    # extra_workloads time their own (short) minibatches: 500 unless the command line says otherwise
    extra_steps = 500 if args.steps is None else args.steps
    if args.steps is None:
        args.steps = 3 if args.impl == "reference" else (200 if args.workload == "c3" else 500)
    if args.warmup is None:
        args.warmup = 1 if args.impl == "reference" else (10 if args.workload == "c3" else 20)
    if args.impl == "reference":
        return run_reference(args, w)
    args.warmup = max(args.warmup, 3)

    env = Env(args)
    world, rank = env.world, env.rank
    N = args.batch or (w["N"] // world if args.scaling == "strong" else w["N"])
    peaks = load_peaks()

    # ---------------- N > 1: parity of the exchange first; a wrong exchange is not worth timing -------------
    dp_parity = None
    if world > 1 and not args.no_extra and args.workload == "c3":
        dp_parity = dp_parity_check(env)
        if not dp_parity["ok"]:
            if rank == 0:
                print(json.dumps(dict(error="dp_parity failed", dp_parity=dp_parity)), flush=True)
            env.dist.destroy_process_group()
            sys.exit(1)

    sampler = ClockSampler(env.local_rank) if rank == 0 else None
    try:
        m = measure(env, args, w, N, args.steps, args.warmup, sampler, e2e=not args.no_e2e, dump_dir=args.dump_outputs)
    finally:                                        # the nvidia-smi poller would outlive a failed run
        if sampler:
            sampler.stop()

    # ---------------- strong scaling (N > 1): global batch fixed at the workload's 8192 rows ----------------
    strong = None
    if world > 1 and not args.no_extra and args.scaling == "weak" and args.workload == "c3" and not args.batch:
        Ns = w["N"] // world
        ms_ = measure(env, args, w, Ns, args.steps, args.warmup, None, e2e=False)
        strong = dict(global_batch=Ns * world, per_gpu_batch=Ns, value=ms_["value"], unit="samples/s",
                      ms_per_step=ms_["ms_per_step"], gpu_launches=ms_["gpu_launches"],
                      note="efficiency = value / (N x the 1-GPU value of the same global batch); computed by the reader")
        ro = roofline_objects(ms_, w, Ns, args.steps, peaks)
        if "roofline_all_gemms" in ro:
            strong["gemm_tflops"] = ro["roofline_all_gemms"]["achieved"]
            strong["per_class"] = {k: dict(tflops=v["tflops"], ms_per_step=v["ms_per_step"]) for k, v in
                                   ro["roofline_all_gemms"]["per_class"].items()}
        if "phases_ms_per_step" in ro:
            strong["phases_ms_per_step"] = ro["phases_ms_per_step"]
            # what the exchange exposes on the main stream: the next forward waiting for the owners' refreshed operands
            strong["exposed_exchange_ms"] = ro["phases_ms_per_step"].get("wait_params")
        if env.dp_mode == "peer":
            # the same with bf16 gradient tiles on the wire (opt-in: one more rounding point, see dp_parity)
            import vbnn_b200
            oldw = vbnn_b200.knob("peer_wire_bf16", 1)
            mw = measure(env, args, w, Ns, args.steps, args.warmup, None, e2e=False)
            vbnn_b200.knob("peer_wire_bf16", oldw)
            strong["bf16_wire"] = dict(value=mw["value"], ms_per_step=mw["ms_per_step"],
                                       phases_ms_per_step={k: v[0] / args.steps for k, v in (mw.get("phases") or {}).items()})

    # ---------------- N = 1: the other single-GPU BASELINE configs in the same record -----------------------
    extra = None
    if world == 1 and not args.no_extra and args.workload == "c3" and not args.batch:
        extra = {}
        for name in ("c1", "c2"):
            wx = WORKLOADS[name]
            mx = measure(env, args, wx, wx["N"], extra_steps, 20, None, e2e=not args.no_e2e)
            d = dict(config=config_dict(wx, 1, wx["N"], "weak"), value=mx["value"], unit="samples/s",
                     ms_per_step=mx["ms_per_step"], steps=extra_steps, warmup=20, gpu_launches=mx["gpu_launches"],
                     dtype="bf16" if wx["precision"] == "bf16" else "f32",
                     step_tflops=flops_per_sample(wx) * wx["N"] / (mx["ms_per_step"] / 1e3) / 1e12)
            for k in ("e2e", "e2e_u8"):
                if k in mx:
                    d[k] = mx[k]
            d.update(roofline_objects(mx, wx, wx["N"], extra_steps, peaks))
            if not args.no_cpu_baseline:
                cpu_baseline(wx)                                        # warm-up (MKL thread pool, page faults)
                d["cpu_baseline"] = cpu_baseline(wx)
            extra[name] = d

    if rank != 0:
        if env.dist is not None:
            env.dist.destroy_process_group()
        return
    clocks = sampler.summary(*m["marks"])
    fps = flops_per_sample(w)
    step_tf = fps * N / (m["ms_per_step"] / 1e3) / 1e12
    line = dict(metric="VB-MLP train samples/sec", value=m["value"], unit="samples/s", n_gpus=world, steps=args.steps,
                warmup=args.warmup, ms_per_step=m["ms_per_step"], higher_is_better=True, scaling=args.scaling,
                vs_baseline=None, dtype="bf16" if w["precision"] == "bf16" else "f32", data="synthetic",
                config=config_dict(w, world, N, args.scaling), dp_exchange=env.dp_mode, host_numa_node=env.numa,
                step_tflops=step_tf, step_frac_of_peak=step_tf / peaks["tflops"],
                gpu_launches=m["gpu_launches"], clocks=clocks, last_error=m["last_error"])
    for k in ("e2e", "e2e_u8"):
        if k in m:
            line[k] = m[k]
    line.update(roofline_objects(m, w, N, args.steps, peaks, is_c3=args.workload == "c3" and N == w["N"]))
    if dp_parity is not None:
        line["dp_parity"] = dp_parity
    if strong is not None:
        line["strong_scaling"] = strong
    if extra is not None:
        line["extra_workloads"] = extra
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(w, N * world)
    elif not args.no_cpu_baseline:
        line["cpu_baseline"] = None
    print(json.dumps(line), flush=True)
    if env.dist is not None:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
