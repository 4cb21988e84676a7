"""Data-parallel fused regression minibatch on real GPUs (run under torchrun, world size G; VBNN_DP=peer or nccl):
every rank steps rows [r*N/G, (r+1)*N/G) of one global minibatch through vbnn_mlp_step under VBNN_CRIT_MSE and
VBNN_CRIT_GAUSSIAN_NLL, whose means divide by the GLOBAL batch (N/G * G rows).  After three minibatches (a padding row of
NaN targets in the second) the parameters and Adam state must equal those of ONE GPU stepping the whole minibatch,
within the tolerances of bench.py's dp_parity (1e-4 / 1e-3), and each rank's error scalar must equal the single GPU's
loss over that rank's rows (the scalars are rank-local means).

  VBNN_DP=nccl python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \\
      tools/dp_regression_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vbnn_b200


def build(ctx, sizes, N, S, reparam, crit):
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], outputs=sizes[-1], criterion=crit, S=S,
                                B=50.0, batchSize=N, mu_init=1, msr_init=True, reparam=reparam, vb_output=True,
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
        return {f"{k}.{n}": m.get(b) for k, m in enumerate(net.model) for n, b in names}

    ok = True
    for crit in ("mse", "gaussian_nll"):
        for reparam in ("weight", "local"):
            sizes, N, S = [64, 96, 80, 10], 64, 2
            K = sizes[-1] // 2 if crit == "gaussian_nll" else sizes[-1]
            g = torch.Generator().manual_seed(11)
            X = [torch.randn(N, sizes[0], generator=g) for _ in range(3)]
            Y = [torch.randn(N, K, generator=g) for _ in range(3)]
            Y[1][5, :] = float("nan")
            n_loc = N // world
            rows = slice(rank * n_loc, (rank + 1) * n_loc)
            net = build(ctx, sizes, n_loc, S, reparam, crit)
            if use_peer:
                net.enable_peer(gather_bytes)
            ctx.set_step(7)
            dist.barrier()
            errs = [net.train_step(X[it][rows].cuda(), Y[it][rows].cuda())[0] for it in range(3)]
            net.join_streams()
            torch.cuda.synchronize(); dist.barrier()
            net.sync_replicas()
            dist.barrier()
            dp_par = params(net)
            e_all = [None] * world
            dist.all_gather_object(e_all, errs)
            if rank == 0:
                ctx1 = vbnn_b200.Context(lr, seed=5)         # single-GPU reference: no communicator, nranks = 1
                one = build(ctx1, sizes, N, S, reparam, crit)
                ctx1.set_step(7)
                worst_err = 0.0
                for it in range(3):
                    one.train_step(X[it].cuda(), Y[it].cuda())
                    # this minibatch's outputs on the single GPU; each rank's scalar is its rows' share
                    outs = torch.stack([one.outputs(s, N) for s in range(S)]).double()
                    for q in range(world):
                        r = slice(q * n_loc, (q + 1) * n_loc)
                        yq = Y[it][r].double()
                        mask = ~torch.isnan(yq)
                        m = outs[:, r, :K]
                        d = torch.where(mask, yq, m) - m
                        t = d ** 2 if crit == "mse" else 0.5 * (outs[:, r, K:] + d ** 2 * torch.exp(-outs[:, r, K:]))
                        want = float(torch.where(mask, t, torch.zeros_like(t)).sum(dim=(1, 2)).mean() / (n_loc * K))
                        worst_err = max(worst_err, abs(e_all[q][it] - want) / abs(want))
                sg_par = params(one)
                worst = {"params": 0.0, "adam": 0.0}
                for k in sg_par:
                    e = float((dp_par[k].double() - sg_par[k].double()).norm() /
                              max(float(sg_par[k].double().norm()), 1e-30))
                    kind = "adam" if k.split(".")[1][:2] in ("m_", "v_") else "params"
                    worst[kind] = max(worst[kind], e)
                ok &= worst["params"] < 1e-4 and worst["adam"] < 1e-3 and worst_err < 1e-4
                print(f"{crit} {reparam} ({'peer' if net.peer_active else 'nccl'}): after 3 minibatches max rel "
                      f"parameters {worst['params']:.2e}, Adam {worst['adam']:.2e}, rank error scalars {worst_err:.2e}")
                torch.cuda.set_stream(ctx.stream)
            torch.cuda.synchronize(); dist.barrier()      # nobody still writes into a peer's buffers
            del net
            dist.barrier()
    flag = torch.tensor([1 if ok else 0], device=f"cuda:{lr}")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("REGRESSION DP CHECK", "OK" if int(flag[0]) == 1 else "FAILED")
    dist.destroy_process_group()
    sys.exit(0 if int(flag[0]) == 1 else 1)


if __name__ == "__main__":
    main()
