"""fp64 reference of the hidden-layer activations of vbnn_mlp_set_activation, built like custom_loss_reference's
forward / backward with a kind parameter and the same operand_round points: q after the activation, and f' formed from
the rounded output q(a), as Torch7's updateGradInput of nn.Tanh / nn.Sigmoid / nn.ELU forms it from self.output.

minibatch() is custom_loss_reference.custom_minibatch with the kind: one minibatch of main.lua:28-40 under a caller's
gradient of the stacked outputs."""
import torch

from oracle import vbnn_oracle as O

KINDS = ("relu", "tanh", "sigmoid", "elu")


def act(kind, y):
    """a = f(y) (nn.ELU with alpha 1)"""
    if kind == "relu":
        return torch.clamp(y, min=0)
    if kind == "tanh":
        return torch.tanh(y)
    if kind == "sigmoid":
        return torch.sigmoid(y)
    return torch.where(y > 0, y, torch.expm1(y))


def act_grad(kind, a):
    """f'(y) from the output a = f(y)"""
    if kind == "relu":
        return (a > 0).to(a.dtype)
    if kind == "tanh":
        return 1 - a * a
    if kind == "sigmoid":
        return a * (1 - a)
    return torch.where(a > 0, torch.ones_like(a), a + 1)


def forward(ref, x, kind, zeta=None):
    """One sample's forward: (activations, outputs of the linear output layer).  x is already operand-rounded."""
    q = ref.q
    acts = [x]
    for k, lyr in enumerate(ref.vb):
        z = None if zeta is None else zeta[k]
        y = lyr.updateOutput(acts[-1], z) if lyr.lrt else lyr.updateOutput(acts[-1])
        acts.append(q(act(kind, y)))
    if isinstance(ref.out, O.VBLinearOracle) and ref.out.lrt:
        logits = ref.out.updateOutput(acts[-1], None if zeta is None else zeta[len(ref.vb)])
    else:
        logits = ref.out.updateOutput(acts[-1])
    return acts, logits


def backward(ref, acts, grad, kind):
    """One sample's backward from dL/dY; returns the first layer's gradInput (no f' term: nothing is below the input)."""
    q = ref.q
    g = q(grad)
    g_in = ref.out.updateGradInput(acts[-1], g)
    ref.out.accGradParameters(acts[-1], g, 1.0)
    for k in range(len(ref.vb) - 1, -1, -1):
        g = q(g_in * act_grad(kind, acts[k + 1]))
        g_in = ref.vb[k].updateGradInput(acts[k], g)
        ref.vb[k].accGradParameters(acts[k], g, 1.0)
    return g_in


def minibatch(ref, inputs, grad_fn, noise, lrt, kind, opt=None, update=True):
    """custom_loss_reference.custom_minibatch under activation `kind`: returns (Y [S x N x C], dL/dY, dX)."""
    opt = opt or ref.opt
    S = opt["S"]
    x = ref.q(inputs.reshape(inputs.shape[0], -1).to(ref.dtype))
    ref.resetGradients()
    ys = []
    for s in range(S):
        ref.sample(None if lrt else noise[s])
        ys.append(forward(ref, x, kind, noise[s] if lrt else None)[1].clone())
    Y = torch.stack(ys)
    G = grad_fn(Y)
    dX = 0
    for s in range(S):
        ref.sample(None if lrt else noise[s])
        acts, _ = forward(ref, x, kind, noise[s] if lrt else None)
        dX = dX + backward(ref, acts, G[s], kind)
    if update:
        ref.update(opt)
    return Y, G, dX


def predict_forward(ref, x, kind, noise, lrt, map_mode=False):
    """Outputs [T x N x C] of evaluation passes: one MAP pass (map_mode, the means as weights) or one pass per entry of
    noise (eps lists in weight mode, zeta lists in local mode)."""
    x = ref.q(x.reshape(x.shape[0], -1).to(ref.dtype))
    if map_mode:
        for lyr in ref.vb_all:
            lyr.clamp_to_map()
            lyr._map = True
        try:
            return forward(ref, x, kind)[1].clone()[None]
        finally:
            for lyr in ref.vb_all:
                lyr._map = False
    out = []
    for nz in noise:
        ref.sample(None if lrt else nz)
        out.append(forward(ref, x, kind, nz if lrt else None)[1].clone())
    return torch.stack(out)
