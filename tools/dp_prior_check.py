"""Data-parallel training under a per-weight prior on real GPUs (run under torchrun, world size G; VBNN_DP=peer or
nccl; in peer mode VBNN_PEER_TRANSPORT selects the gradient transport: 1 = NVLink stores from the dW epilogue, 3 = the
co-resident copy kernel).  Every rank steps rows [r*N/G, (r+1)*N/G) of one global minibatch.

After two minibatches under the empirical prior the ranks run the vbnn_mlp_sync_replicas protocol and snapshot a
PER_WEIGHT prior on every layer (the continual-learning step), then train three more minibatches.  Before the
protocol, peer mode must refuse the snapshot (rows owned by other ranks are stale).  One GPU stepping the whole
minibatches the same way is the reference: parameters within 1e-4 and Adam state within 1e-3 (bench.py's dp_parity),
and the prior arrays equal on every rank.

  VBNN_DP=peer VBNN_PEER_TRANSPORT=3 python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 \\
      --master-port 29513 tools/dp_prior_check.py
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
             ("v_mu", L.BUF_ADAM_V_MU), ("m_var", L.BUF_ADAM_M_VAR), ("v_var", L.BUF_ADAM_V_VAR),
             ("prior_means", L.BUF_PRIOR_MEANS), ("prior_lvars", L.BUF_PRIOR_LVARS)]

    def params(net):
        return {f"{k}.{n}": net.model[k].get(b) for k in net.vb_indices for n, b in names}

    def drain_and_sync(net):
        net.join_streams()
        torch.cuda.synchronize(); dist.barrier()
        net.sync_replicas()
        dist.barrier()

    ok = True
    for reparam, sizes, N, S in [("weight", [64, 96, 80, 10], 64, 2), ("local", [64, 96, 80, 10], 64, 2)]:
        g = torch.Generator().manual_seed(11)
        X = [torch.randn(N, sizes[0], generator=g) for _ in range(5)]
        T = [torch.randint(1, sizes[-1] + 1, (N,), generator=g).float() for _ in range(5)]
        n_loc = N // world
        rows = slice(rank * n_loc, (rank + 1) * n_loc)
        net = build(ctx, sizes, n_loc, S, reparam)
        if use_peer:
            net.enable_peer(gather_bytes)
        ctx.set_step(7)
        dist.barrier()
        for it in range(2):
            net.train_step(X[it][rows].cuda(), T[it][rows].cuda(), sync=False)
        if use_peer:
            net.join_streams()
            torch.cuda.synchronize()
            rc = L.lib().vbnn_layer_set_prior(net.model[0].handle, L.PRIOR_PER_WEIGHT, 0.0, 0.0)
            if rc != L.E_STATE:
                ok = False
                print(f"rank {rank}: PER_WEIGHT snapshot over stale rows returned {rc}, expected VBNN_E_STATE")
        drain_and_sync(net)
        net.set_prior("per_weight")
        for it in range(2, 5):
            net.train_step(X[it][rows].cuda(), T[it][rows].cuda(), sync=False)
        drain_and_sync(net)
        dp_par = params(net)
        if rank == 0:
            ctx1 = vbnn_b200.Context(lr, seed=5)         # single-GPU reference: no communicator, nranks = 1
            one = build(ctx1, sizes, N, S, reparam)
            ctx1.set_step(7)
            for it in range(5):
                if it == 2:
                    one.set_prior("per_weight")
                one.train_step(X[it].cuda(), T[it].cuda(), sync=False)
            torch.cuda.synchronize()
            sg_par = params(one)
            worst = {"params": 0.0, "adam": 0.0, "prior": 0.0}
            for k in sg_par:
                e = float((dp_par[k].double() - sg_par[k].double()).norm() / max(float(sg_par[k].double().norm()), 1e-30))
                n = k.split(".", 1)[1]
                kind = "adam" if n[:2] in ("m_", "v_") else "prior" if n.startswith("prior") else "params"
                worst[kind] = max(worst[kind], e)
            ok &= worst["params"] < 1e-4 and worst["adam"] < 1e-3 and worst["prior"] < 1e-4
            print(f"{reparam} ({'peer' if net.peer_active else 'nccl'}): after 5 minibatches, max rel parameters "
                  f"{worst['params']:.2e}, Adam {worst['adam']:.2e}, prior {worst['prior']:.2e}")
            torch.cuda.set_stream(ctx.stream)
        # every rank snapshotted the same posterior
        for k in sorted(dp_par):
            if ".prior" in k:
                t = dp_par[k].cuda()
                ref = t.clone()
                dist.broadcast(ref, 0)
                if not torch.equal(t, ref):
                    ok = False
                    print(f"rank {rank}: {k} differs from rank 0's")
        torch.cuda.synchronize(); dist.barrier()      # nobody still writes into a peer's buffers
        del net
        dist.barrier()
    flag = torch.tensor([1 if ok else 0], device=f"cuda:{lr}")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("dp_prior_check", "OK" if int(flag[0]) == 1 else "FAILED")
    dist.destroy_process_group()
    sys.exit(0 if int(flag[0]) == 1 else 1)


if __name__ == "__main__":
    main()
