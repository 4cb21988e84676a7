"""Data-parallel training under a per-minibatch hyper-parameter schedule on real GPUs (run under torchrun, world size
G; VBNN_DP=peer or nccl; in peer mode VBNN_PEER_TRANSPORT selects the gradient transport: 1 = NVLink stores from the dW
epilogue, 3 = the co-resident copy kernel).  Every rank steps rows [r*N/G, (r+1)*N/G) of one global minibatch.

Before every minibatch each rank sets the same B, learning rates and Adam constants with vbnn_mlp_set_opts
(MLP.set_opt), without draining the previous minibatch: in peer mode its shard updates may still run on the side
stream, which the set waits for.  One GPU stepping the whole minibatches under the same schedule is the reference:
parameters within 1e-4 and Adam state within 1e-3 (bench.py's dp_parity), no step graph re-captured by a set, and
the live values equal on every rank.

  VBNN_DP=peer VBNN_PEER_TRANSPORT=3 python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 \\
      --master-port 29514 tools/dp_hparams_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vbnn_b200


# B, lr_bias, lr_mu, lr_var, beta1, beta2, eps per minibatch: a KL warm-up (B falling towards its full-weight value)
# under decaying rates, with the Adam constants moved as well
SCHEDULE = [
    (2000.0, 1e-3, 1e-3, 0.05, 0.9, 0.999, 1e-8),
    (500.0, 8e-4, 8e-4, 0.04, 0.85, 0.99, 1e-7),
    (200.0, 6e-4, 6e-4, 0.03, 0.9, 0.995, 1e-8),
    (80.0, 4e-4, 4e-4, 0.02, 0.8, 0.99, 1e-6),
    (40.0, 2e-4, 2e-4, 0.01, 0.9, 0.999, 1e-8),
    (20.0, 1e-4, 1e-4, 0.005, 0.95, 0.999, 1e-8),
]


def scheduled(opt, it):
    """opt with row `it` of SCHEDULE in the config dict's keys; "_row" keeps the float32 values"""
    B, lr_bias, lr_mu, lr_var, b1, b2, eps = SCHEDULE[it]
    o = dict(opt, B=B, state=dict(opt["state"], learningRate=lr_bias), varState=dict(opt["varState"], learningRate=lr_var),
             meanState=dict(opt["meanState"], learningRate=lr_mu, beta1=b1, beta2=b2, epsilon=eps))
    o["_row"] = [float(torch.tensor(v, dtype=torch.float32)) for v in SCHEDULE[it]]
    return o


def build(ctx, sizes, N, S, reparam):
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=S, B=20.0, batchSize=N, mu_init=1, msr_init=True, reparam=reparam, vb_output=True,
                                precision="fp32", strict_reference=False, log=False, seed=5)
    net = vbnn_b200.MLP(opt, ctx, max_batch=N)
    net.init_params(seed=4, he_means=True)
    return net


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    lr = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(lr)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{lr}"))
    ctx = vbnn_b200.Context(lr, seed=5)

    def bcast(buf):
        t = torch.zeros(128, dtype=torch.uint8, device=f"cuda:{lr}")
        if rank == 0:
            t.copy_(torch.tensor(list(buf), dtype=torch.uint8))
        dist.broadcast(t, 0)
        return bytes(t.cpu().tolist())
    ctx.init_comm(rank, world, bcast)

    def gather_bytes(blob):
        t = torch.tensor(list(blob), dtype=torch.uint8, device=f"cuda:{lr}")
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [bytes(o.cpu().tolist()) for o in out]
    use_peer = os.environ.get("VBNN_DP", "peer") == "peer"
    from vbnn_b200 import _lib as L
    names = [("means", L.BUF_MEANS), ("lvars", L.BUF_LVARS), ("bias", L.BUF_BIAS), ("m_mu", L.BUF_ADAM_M_MU),
             ("v_mu", L.BUF_ADAM_V_MU), ("m_var", L.BUF_ADAM_M_VAR), ("v_var", L.BUF_ADAM_V_VAR)]

    def params(net):
        return {f"{k}.{n}": net.model[k].get(b) for k in net.vb_indices for n, b in names}

    def drain_and_sync(net):
        net.join_streams()
        torch.cuda.synchronize(); dist.barrier()
        net.sync_replicas()
        dist.barrier()

    ok = True
    steps = len(SCHEDULE)
    for reparam, sizes, N, S in [("weight", [64, 96, 80, 10], 64, 2), ("local", [64, 96, 80, 10], 64, 2)]:
        g = torch.Generator().manual_seed(11)
        X = [torch.randn(N, sizes[0], generator=g) for _ in range(steps)]
        T = [torch.randint(1, sizes[-1] + 1, (N,), generator=g).float() for _ in range(steps)]
        n_loc = N // world
        rows = slice(rank * n_loc, (rank + 1) * n_loc)
        net = build(ctx, sizes, n_loc, S, reparam)
        if use_peer:
            net.enable_peer(gather_bytes)
        ctx.set_step(7)
        dist.barrier()
        captures = []
        for it in range(steps):
            net.set_opt(scheduled(net.opt, it))
            net.train_step(X[it][rows].cuda(), T[it][rows].cuda(), sync=False)
            captures.append(net.graph_captures())
        if captures[-1] != captures[1]:
            ok = False
            print(f"rank {rank}: step graph captures {captures}: a set re-captured")
        drain_and_sync(net)
        dp_par = params(net)
        live = torch.tensor([[m.opts[f] for f in L.LIVE_OPTS] for m in net.model], device=f"cuda:{lr}")
        want = torch.tensor([list(scheduled(net.opt, steps - 1)["_row"])] * len(net.model), device=f"cuda:{lr}")
        if not torch.equal(live, want.float()):
            ok = False
            print(f"rank {rank}: live values {live.tolist()} are not the last row of the schedule")
        if rank == 0:
            ctx1 = vbnn_b200.Context(lr, seed=5)         # single-GPU reference: no communicator, nranks = 1
            one = build(ctx1, sizes, N, S, reparam)
            ctx1.set_step(7)
            for it in range(steps):
                one.set_opt(scheduled(one.opt, it))
                one.train_step(X[it].cuda(), T[it].cuda(), sync=False)
            torch.cuda.synchronize()
            sg_par = params(one)
            worst = {"params": 0.0, "adam": 0.0}
            for k in sg_par:
                e = float((dp_par[k].double() - sg_par[k].double()).norm() / max(float(sg_par[k].double().norm()), 1e-30))
                n = k.split(".", 1)[1]
                kind = "adam" if n[:2] in ("m_", "v_") else "params"
                worst[kind] = max(worst[kind], e)
            ok &= worst["params"] < 1e-4 and worst["adam"] < 1e-3
            print(f"{reparam} ({'peer' if net.peer_active else 'nccl'}): after {steps} scheduled minibatches, max rel "
                  f"parameters {worst['params']:.2e}, Adam {worst['adam']:.2e}")
            torch.cuda.set_stream(ctx.stream)
        ref = live.clone()
        dist.broadcast(ref, 0)
        if not torch.equal(live, ref):
            ok = False
            print(f"rank {rank}: live values differ from rank 0's")
        torch.cuda.synchronize(); dist.barrier()      # nobody still writes into a peer's buffers
        del net
        dist.barrier()
    flag = torch.tensor([1 if ok else 0], device=f"cuda:{lr}")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("dp_hparams_check", "OK" if int(flag[0]) == 1 else "FAILED")
    dist.destroy_process_group()
    sys.exit(0 if int(flag[0]) == 1 else 1)


if __name__ == "__main__":
    main()
