"""Data-parallel input gradient on real GPUs (run under torchrun, world size G; VBNN_DP=peer or nccl):
every rank steps rows [r*N/G, (r+1)*N/G) of one global minibatch through vbnn_mlp_step_grad_input, and its dX must
equal those rows of the dX of ONE rank stepping the whole minibatch (the data-parallel gradient scale 1 / (N/G * G)
is the single-GPU 1 / N; identical Philox eps on every rank, LRT zeta indexed by the global row).

  VBNN_DP=nccl python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \\
      tools/dp_grad_input_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vbnn_b200


def build(ctx, sizes, N, S, reparam):
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=S, B=50.0, batchSize=N, mu_init=1, msr_init=True, reparam=reparam,
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
    ok = True
    for reparam, sizes, N, S in [("weight", [64, 96, 80, 10], 64, 2), ("local", [64, 96, 80, 10], 64, 2)]:
        g = torch.Generator().manual_seed(11)
        X = torch.randn(N, sizes[0], generator=g)
        T = torch.randint(1, sizes[-1] + 1, (N,), generator=g).float()
        n_loc = N // world
        net = build(ctx, sizes, n_loc, S, reparam)
        if use_peer:
            net.enable_peer(gather_bytes)
        ctx.set_step(7)
        dist.barrier()
        dxs = []
        for it in range(2):                     # the second minibatch reads parameters updated by the exchange
            dx = torch.empty(n_loc, sizes[0], device=f"cuda:{lr}")
            net.train_step(X[rank * n_loc:(rank + 1) * n_loc].cuda(), T[rank * n_loc:(rank + 1) * n_loc].cuda(),
                           grad_input=dx)
            dxs.append(dx)
        net.join_streams()
        torch.cuda.synchronize(); dist.barrier()
        full = [[torch.empty_like(d) for _ in range(world)] for d in dxs]
        for f, d in zip(full, dxs):
            dist.all_gather(f, d)
        if rank == 0:
            ctx1 = vbnn_b200.Context(lr, seed=5)         # single-GPU reference: no communicator, nranks = 1
            one = build(ctx1, sizes, N, S, reparam)
            ctx1.set_step(7)
            for it in range(2):
                d1 = torch.empty(N, sizes[0], device=f"cuda:{lr}")
                one.train_step(X.cuda(), T.cuda(), grad_input=d1)
                got = torch.cat(full[it])
                e = float((got - d1).norm() / d1.norm())
                ok &= e < 1e-4
                print(f"{reparam} ({'peer' if net.peer_active else 'nccl'}) minibatch {it}: rel err DP vs single = {e:.2e}")
            torch.cuda.set_stream(ctx.stream)
        torch.cuda.synchronize(); dist.barrier()      # nobody still writes into a peer's buffers
        del net
        dist.barrier()
    flag = torch.tensor([1 if ok else 0], device=f"cuda:{lr}")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("GRAD INPUT DP CHECK", "OK" if int(flag[0]) == 1 else "FAILED")
    dist.destroy_process_group()
    sys.exit(0 if int(flag[0]) == 1 else 1)


if __name__ == "__main__":
    main()
