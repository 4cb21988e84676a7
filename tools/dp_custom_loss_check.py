"""Data-parallel split minibatch on real GPUs (run under torchrun, world size G; VBNN_DP=peer or nccl): every rank
steps rows [r*N/G, (r+1)*N/G) of one global minibatch through vbnn_mlp_forward_train + a torch MSE whose mean runs
over the GLOBAL batch (it divides by N/G * G) + vbnn_mlp_backward_update.  Its logits and dX must equal those rows of
ONE rank stepping the whole minibatch the same way.  Between the second and the third minibatch every rank opens a
step and closes it without a loss twice: once through vbnn_mlp_reset_gradients, which peer mode must refuse (the step
is then closed with a zero gradient) and NCCL mode accepts (the step is abandoned), and once through
MLP.train_step_loss with a loss_fn that raises, which closes it the same way.  The single GPU mirrors both (a zero
gradient for peer mode, an abandoned step for NCCL), so afterwards the ranks' step counters, the third minibatch and
the parameters and Adam state must still equal the single GPU's, the last within the tolerances of bench.py's
dp_parity (1e-4 / 1e-3).

  VBNN_DP=nccl python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \\
      tools/dp_custom_loss_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vbnn_b200


def build(ctx, sizes, N, S, reparam, vb_output=False):
    opt = vbnn_b200.default_opt(input_size=sizes[0], hidden=sizes[1:-1], classes=[str(i) for i in range(sizes[-1])],
                                S=S, B=50.0, batchSize=N, mu_init=1, msr_init=True, reparam=reparam, vb_output=vb_output,
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

    def split(net, X, R, n_global, dx):
        Y = net.forward_train(X)
        leaf = Y.detach().clone().requires_grad_(True)
        loss = ((leaf - R) ** 2).sum() / (n_global * R.shape[1])     # per sample: the mean over the global batch
        (g,) = torch.autograd.grad(loss, leaf)
        net.backward_update(g.contiguous(), dx)
        return leaf.detach()

    def close_without_loss(net, X, peer):
        """Open a step twice and close it without a loss: reset_gradients (refused in peer mode, where a zero
        gradient closes it instead), then train_step_loss with a loss_fn that raises."""
        step = ctx.get_step()
        Y = net.forward_train(X)
        rc = L.lib().vbnn_mlp_reset_gradients(net.handle)
        good = rc == (L.E_STATE if peer else L.VBNN_OK)
        if peer:
            net.backward_update(torch.zeros_like(Y))
        else:
            net._open_n = None
        def failing_loss(y):
            raise ValueError("loss")
        try:
            net.train_step_loss(X, failing_loss)
            good = False
        except ValueError:
            pass
        good &= getattr(net, "_open_n", None) is None
        good &= ctx.get_step() == step + (2 if peer else 0)
        return bool(good)

    ok = True
    for reparam, sizes, N, S in [("weight", [64, 96, 80, 10], 64, 2), ("local", [64, 96, 80, 10], 64, 2)]:
        g = torch.Generator().manual_seed(11)
        X = [torch.randn(N, sizes[0], generator=g) for _ in range(4)]
        R = [torch.randn(N, sizes[-1], generator=g) for _ in range(4)]
        n_loc = N // world
        rows = slice(rank * n_loc, (rank + 1) * n_loc)
        net = build(ctx, sizes, n_loc, S, reparam, vb_output=True)
        if use_peer:
            net.enable_peer(gather_bytes)
        ctx.set_step(7)
        dist.barrier()
        outs = []
        for it in (0, 1, None, 3):              # the second minibatch reads parameters updated by the exchange
            if it is None:
                closed = close_without_loss(net, X[2][rows].cuda(), use_peer)
                ok &= closed
                if not closed:
                    print(f"rank {rank}: a step opened by forward_train was not closed as expected")
                continue
            dx = torch.empty(n_loc, sizes[0], device=f"cuda:{lr}")
            Y = split(net, X[it][rows].cuda(), R[it][rows].cuda(), N, dx)
            outs.append((Y.contiguous(), dx))
        steps = [torch.zeros(1, dtype=torch.int64, device=f"cuda:{lr}") for _ in range(world)]
        dist.all_gather(steps, torch.tensor([ctx.get_step()], device=f"cuda:{lr}"))
        steps = [int(t) for t in steps]
        net.join_streams()
        torch.cuda.synchronize(); dist.barrier()
        net.sync_replicas()                     # peer mode: every row's fp32 state, not just this rank's shard
        dist.barrier()
        dp_par = params(net)
        full = [[[torch.empty_like(t) for _ in range(world)] for t in o] for o in outs]
        for f, o in zip(full, outs):
            for ff, t in zip(f, o):
                dist.all_gather(ff, t)
        if rank == 0:
            ctx1 = vbnn_b200.Context(lr, seed=5)         # single-GPU reference: no communicator, nranks = 1
            one = build(ctx1, sizes, N, S, reparam, vb_output=True)
            ctx1.set_step(7)
            for k, it in enumerate((0, 1, 3)):
                if it == 3:                          # the two steps closed without a loss, as the ranks closed them
                    for _ in range(2):
                        one.forward_train(X[2].cuda())
                        if use_peer:
                            one.backward_update(torch.zeros(S, N, sizes[-1], device=f"cuda:{lr}"))
                        else:
                            one.resetGradients()
                d1 = torch.empty(N, sizes[0], device=f"cuda:{lr}")
                Y1 = split(one, X[it].cuda(), R[it].cuda(), N, d1)
                Yg = torch.cat(full[k][0], dim=1)
                dg = torch.cat(full[k][1])
                e_y = float((Yg - Y1).norm() / Y1.norm())
                e_dx = float((dg - d1).norm() / d1.norm())
                ok &= e_y < 1e-4 and e_dx < 1e-4
                print(f"{reparam} ({'peer' if net.peer_active else 'nccl'}) minibatch {it}: logits {e_y:.2e}, "
                      f"dX {e_dx:.2e}")
            step_ok = all(t == ctx1.get_step() for t in steps)
            ok &= step_ok
            print(f"{reparam}: step counters of the ranks {steps}, single GPU {ctx1.get_step()}")
            sg_par = params(one)
            worst = {"params": 0.0, "adam": 0.0}
            for k in sg_par:
                e = float((dp_par[k].double() - sg_par[k].double()).norm() / max(float(sg_par[k].double().norm()), 1e-30))
                kind = "adam" if k.split(".")[1][:2] in ("m_", "v_") else "params"
                worst[kind] = max(worst[kind], e)
            ok &= worst["params"] < 1e-4 and worst["adam"] < 1e-3
            print(f"{reparam}: after 3 minibatches, max rel parameters {worst['params']:.2e}, Adam {worst['adam']:.2e}")
            torch.cuda.set_stream(ctx.stream)
        torch.cuda.synchronize(); dist.barrier()      # nobody still writes into a peer's buffers
        del net
        dist.barrier()
    flag = torch.tensor([1 if ok else 0], device=f"cuda:{lr}")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("CUSTOM LOSS DP CHECK", "OK" if int(flag[0]) == 1 else "FAILED")
    dist.destroy_process_group()
    sys.exit(0 if int(flag[0]) == 1 else 1)


if __name__ == "__main__":
    main()
