"""fp64 reference of the split minibatch (vbnn_mlp_forward_train + vbnn_mlp_backward_update), built from the CPU
oracle's layer methods (oracle/vbnn_oracle.py) with the operand_round points of MLPOracle.run.

custom_minibatch() runs one minibatch of main.lua:28-40 in which the criterion is replaced by a caller's function of
the stacked logits: it forwards the S samples, asks grad_fn for dL/dY [S x N x C], backpropagates each sample's slice
of it (mlp.lua:79 model:backward, the ReLU masks and the LRT terms as MLPOracle.run has them) and updates."""
import torch

from oracle import vbnn_oracle as O


def forward(ref, x, zeta=None):
    """MLPOracle.run's forward of one sample: (activations, pre-LogSoftMax logits).  x is already operand-rounded."""
    q = ref.q
    acts = [x]
    for k, lyr in enumerate(ref.vb):
        z = None if zeta is None else zeta[k]
        y = lyr.updateOutput(acts[-1], z) if lyr.lrt else lyr.updateOutput(acts[-1])
        acts.append(q(torch.clamp(y, min=0)))                         # nn.ReLU
    if isinstance(ref.out, O.VBLinearOracle) and ref.out.lrt:
        logits = ref.out.updateOutput(acts[-1], None if zeta is None else zeta[len(ref.vb)])
    else:
        logits = ref.out.updateOutput(acts[-1])
    return acts, logits


def backward(ref, acts, grad):
    """MLPOracle.run's backward of one sample from dL/dlogits; returns the first layer's gradInput."""
    q = ref.q
    g = q(grad)
    g_in = ref.out.updateGradInput(acts[-1], g)
    ref.out.accGradParameters(acts[-1], g, 1.0)
    for k in range(len(ref.vb) - 1, -1, -1):
        g = q(g_in * (acts[k + 1] > 0).to(ref.dtype))                 # ReLU backward
        g_in = ref.vb[k].updateGradInput(acts[k], g)
        ref.vb[k].accGradParameters(acts[k], g, 1.0)
    return g_in


def classnll_grad(targets):
    """grad_fn of the fused step: per sample, the gradient of the batch-mean ClassNLL(LogSoftMax(Y_s)) (mlp.lua:78-79)."""
    def fn(Y):
        out = []
        for s in range(Y.shape[0]):
            logp = O.log_softmax(Y[s])
            out.append(O.log_softmax_backward(logp, O.class_nll_backward(logp, targets)))
        return torch.stack(out)
    return fn


def autograd_grad(loss_fn):
    """grad_fn from a differentiable loss of the stacked logits (fp64 autograd)."""
    def fn(Y):
        leaf = Y.detach().clone().requires_grad_(True)
        with torch.enable_grad():
            (g,) = torch.autograd.grad(loss_fn(leaf), leaf)
        return g
    return fn


def custom_minibatch(ref, inputs, grad_fn, noise, lrt, opt=None, update=True):
    """One minibatch under a caller's loss.  noise[s] is sample s's list of per-VB-layer epsilons (weight mode) or
    zetas (local reparameterisation), as for O.train_minibatch.  Returns (Y [S x N x C], dL/dY, dX = sum_s of the first
    layer's gradInput); ref's gradients, parameters and optimiser state are left as after the update."""
    opt = opt or ref.opt
    S = opt["S"]
    x = ref.q(inputs.reshape(inputs.shape[0], -1).to(ref.dtype))     # nn.Reshape
    ref.resetGradients()                                             # main.lua:28
    ys = []
    for s in range(S):
        ref.sample(None if lrt else noise[s])
        ys.append(forward(ref, x, noise[s] if lrt else None)[1].clone())
    Y = torch.stack(ys)
    G = grad_fn(Y)
    dX = 0
    for s in range(S):                                               # the forward again: the layers keep one sample
        ref.sample(None if lrt else noise[s])
        acts, _ = forward(ref, x, noise[s] if lrt else None)
        dX = dX + backward(ref, acts, G[s])
    if update:
        ref.update(opt)                                              # main.lua:40
    return Y, G, dX
