"""nn.VBLinear over libvbnn.so: the same names, argument meaning and error behaviour as the
reference's Torch7 module (VBLinear.lua:7-166), so mlp.lua-style callers use it as a drop-in.
This is the host-side mirror SURVEY.md section 8(b) asks for in place of the LuaJIT shim
(lua/VBLinear.lua holds that shim; no Lua runtime exists in this image)."""
from __future__ import annotations

import ctypes as C

from . import _lib as L
from .config import opts_struct, with_live
from .context import Context, DevView, as_dev_f32, default_context


class VBLinear:
    """nn.VBLinear(inputSize, outputSize, opt)  -- VBLinear.lua:9-47."""

    kind = L.KIND_VB

    def __init__(self, inputSize, outputSize, opt, ctx: Context = None, _borrowed=None):
        self.opt = opt
        self.ctx = ctx or default_context(seed=opt.get("seed", 3))
        self.inputSize, self.outputSize = int(inputSize), int(outputSize)
        self.W = self.inputSize * self.outputSize                      # VBLinear.lua:21
        self._owned = _borrowed is None
        if _borrowed is not None:
            self.handle = _borrowed
        else:
            self.handle = C.c_void_p()
            o = opts_struct(opt)
            L.check(L.lib().vbnn_layer_create(self.ctx.handle, self.inputSize, self.outputSize, self.kind,
                                              C.byref(o), C.byref(self.handle)))
        self.var_init = 2.0 / self.inputSize if opt.get("msr_init") else opt["var_init"]
        self.mu_hat, self.var_hat = 0.0, None
        self.output = None
        self.gradInput = None
        self._sample_idx = 0
        self.stats = None

    def __del__(self):
        try:
            if self._owned and self.handle:
                L.lib().vbnn_layer_destroy(self.handle)
        except Exception:
            pass

    # ---- live views of the module's tensors (reference fields) ----
    def _view(self, which, shape=None):
        import torch
        p, n = C.c_void_p(), C.c_size_t()
        L.check(L.lib().vbnn_layer_device_ptr(self.handle, which, C.byref(p), C.byref(n)))
        if not p.value:
            raise L.VbnnError(L.E_STATE, f"buffer {which} is not materialised in this mode")
        if shape is None:
            shape = (self.outputSize, self.inputSize) if n.value == self.W else (n.value,)
        return torch.as_tensor(DevView(p.value, shape), device=f"cuda:{self.ctx.device}")

    means = property(lambda s: s._view(L.BUF_MEANS))
    lvars = property(lambda s: s._view(L.BUF_LVARS))
    bias = property(lambda s: s._view(L.BUF_BIAS))
    gradWeight = property(lambda s: s._view(L.BUF_GRAD_WEIGHT))
    gradSum = property(lambda s: s._view(L.BUF_GRAD_SUM))
    gradBias = property(lambda s: s._view(L.BUF_GRAD_BIAS))
    stdv = property(lambda s: s._view(L.BUF_STDV))
    mu_sqe = property(lambda s: s._view(L.BUF_MU_SQE))
    prior_means = property(lambda s: s._view(L.BUF_PRIOR_MEANS))      # "per_weight" prior only
    prior_lvars = property(lambda s: s._view(L.BUF_PRIOR_LVARS))

    @property
    def weight(self):
        import torch
        out = torch.empty(self.outputSize, self.inputSize, dtype=torch.float32)
        L.check(L.lib().vbnn_layer_get(self.handle, L.BUF_WEIGHT, C.c_void_p(out.data_ptr())))
        return out

    @property
    def e(self):
        return self._view(L.BUF_EPS)

    def get(self, which):
        import torch
        n = self.outputSize if which in (L.BUF_BIAS, L.BUF_GRAD_BIAS) else self.W
        out = torch.empty(n, dtype=torch.float32)
        L.check(L.lib().vbnn_layer_get(self.handle, which, C.c_void_p(out.data_ptr())))
        return out if n == self.outputSize else out.view(self.outputSize, self.inputSize)

    def set(self, which, value):
        import torch
        v = torch.as_tensor(value, dtype=torch.float32).contiguous().cpu()
        n = self.outputSize if which in (L.BUF_BIAS, L.BUF_GRAD_BIAS) else self.W
        if v.numel() != n:
            raise L.VbnnError(L.E_INVALID, f"set({which}): expected {n} elements, got {v.numel()}")
        L.check(L.lib().vbnn_layer_set(self.handle, which, C.c_void_p(v.data_ptr())))

    @property
    def t(self):
        v = C.c_int()
        L.check(L.lib().vbnn_layer_get_t(self.handle, C.byref(v)))
        return v.value

    # ---- VBLinear.lua:49-64 ----
    def sample(self, opt=None, eps=None, sample_idx=None):
        if sample_idx is not None:
            self._sample_idx = int(sample_idx)
        ptr = None
        if eps is not None:
            eps = as_dev_f32(eps, self.ctx.device)
            if eps.numel() != self.W:
                raise L.VbnnError(L.E_INVALID, "sample: eps must be [outputSize x inputSize]")
            self._eps_keep = eps
            ptr = C.c_void_p(eps.data_ptr())
        L.check(L.lib().vbnn_layer_sample(self.handle, self._sample_idx, ptr))
        self._sample_idx += 1

    def clamp_to_map(self):                                             # VBLinear.lua:105-107
        L.check(L.lib().vbnn_layer_clamp_to_map(self.handle))

    # ---- inherited nn.Linear protocol ----
    def _check_input(self, input):
        x = as_dev_f32(input, self.ctx.device)
        if x.dim() == 1:
            x = x.view(1, -1)
        if x.dim() != 2 or x.shape[1] != self.inputSize:
            raise L.VbnnError(L.E_INVALID, f"input must be [N x {self.inputSize}], got {tuple(x.shape)}")
        return x

    def updateOutput(self, input, zeta=None):
        import torch
        x = self._check_input(input)
        n = x.shape[0]
        self.output = torch.empty(n, self.outputSize, dtype=torch.float32, device=x.device)
        zp = None
        if zeta is not None:
            zeta = as_dev_f32(zeta, self.ctx.device)
            self._zeta_keep = zeta
            zp = C.c_void_p(zeta.data_ptr())
        L.check(L.lib().vbnn_layer_forward(self.handle, C.c_void_p(x.data_ptr()), n,
                                           C.c_void_p(self.output.data_ptr()), zp))
        self._x_keep = x
        return self.output

    def updateGradInput(self, input, gradOutput):
        import torch
        x = self._check_input(input)
        g = as_dev_f32(gradOutput, self.ctx.device)
        n = x.shape[0]
        if tuple(g.shape) != (n, self.outputSize):
            raise L.VbnnError(L.E_INVALID, f"gradOutput must be [{n} x {self.outputSize}]")
        self.gradInput = torch.empty(n, self.inputSize, dtype=torch.float32, device=x.device)
        L.check(L.lib().vbnn_layer_backward_data(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(g.data_ptr()),
                                                 n, C.c_void_p(self.gradInput.data_ptr())))
        return self.gradInput

    def accGradParameters(self, input, gradOutput, scale=1.0):           # VBLinear.lua:112-118
        x = self._check_input(input)
        g = as_dev_f32(gradOutput, self.ctx.device)
        n = x.shape[0]
        if tuple(g.shape) != (n, self.outputSize):
            raise L.VbnnError(L.E_INVALID, f"gradOutput must be [{n} x {self.outputSize}]")
        L.check(L.lib().vbnn_layer_acc_grad(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(g.data_ptr()),
                                            n, C.c_float(scale)))

    def forward(self, input, zeta=None):
        return self.updateOutput(input, zeta)

    def backward(self, input, gradOutput, scale=1.0):
        gi = self.updateGradInput(input, gradOutput)
        self.accGradParameters(input, gradOutput, scale)
        return gi

    def parameters(self):
        return [self.weight, self.bias], [self.gradWeight, self.gradBias]

    def resetAcc(self, opt=None):                                       # VBLinear.lua:120-122
        L.check(L.lib().vbnn_layer_reset_acc(self.handle))
        self._sample_idx = 0

    # ---- the prior of the KL terms (vbnn_layer_set_prior) ----
    def set_prior(self, kind, mean=0.0, var=None):
        """kind "empirical" (the reference's N(0, mean(sigma^2 + mu^2)), the default), "fixed" (N(mean, var),
        var > 0) or "per_weight": the prior becomes a copy of the current posterior, N(means, exp(lvars)), kept in
        prior_means / prior_lvars, which may be edited afterwards.  mean / var are read for "fixed" only."""
        if kind not in L.PRIOR_KINDS:
            raise L.VbnnError(L.E_INVALID, f"set_prior: kind must be one of {sorted(L.PRIOR_KINDS)}, got {kind!r}")
        if kind == "fixed" and var is None:
            raise L.VbnnError(L.E_INVALID, "set_prior('fixed') needs var")
        L.check(L.lib().vbnn_layer_set_prior(self.handle, L.PRIOR_KINDS[kind], C.c_float(mean),
                                             C.c_float(var if var is not None else 0.0)))

    @property
    def prior(self):
        """(kind, mean, var): the fixed prior's scalars, None for "empirical" and "per_weight"."""
        k, m, v = C.c_int(), C.c_float(), C.c_float()
        L.check(L.lib().vbnn_layer_get_prior(self.handle, C.byref(k), C.byref(m), C.byref(v)))
        name = {c: n for n, c in L.PRIOR_KINDS.items()}[k.value]
        return (name, m.value, v.value) if k.value == L.PRIOR_FIXED else (name, None, None)

    # ---- hyper-parameters read at every update (vbnn_layer_set_opts) ----
    def _get_opts(self):
        o = L.VbnnOpts()
        L.check(L.lib().vbnn_layer_get_opts(self.handle, C.byref(o)))
        return o

    def set_opt(self, opt):
        """This layer's B, learning rates and Adam constants from a config dict, mapped as buildModel maps it: opt["B"],
        state.learningRate (biases / nn.Linear), meanState.learningRate / beta1 / beta2 / epsilon (0.9, 0.999, 1e-8
        where absent), varState.learningRate.  The Torch7 idiom of writing layer.meanState.learningRate or opt.B between
        minibatches, made explicit: every later update, captured step graphs included, uses the new values.  The keys
        that describe the layer as created (S, reparam, precision, strict_reference, var_init, msr_init, mu_init) must
        be unchanged: otherwise VbnnError(E_INVALID) and nothing changes.  self.opt takes the live keys of opt only.  On
        a layer of an MLP it gives this layer its own values."""
        L.check(L.lib().vbnn_layer_set_opts(self.handle, C.byref(opts_struct(opt))))
        self.opt = with_live(self.opt, opt)

    @property
    def opts(self):
        """The live values {B, lr_bias, lr_mu, lr_var, adam_beta1, adam_beta2, adam_eps} the next update uses."""
        o = self._get_opts()
        return {f: getattr(o, f) for f in L.LIVE_OPTS}

    # ---- VBLinear.lua:77-103 ----
    def compute_prior(self):
        mu_hat, var_hat = C.c_float(), C.c_float()
        L.check(L.lib().vbnn_layer_compute_prior(self.handle, C.byref(mu_hat), C.byref(var_hat)))
        self.mu_hat, self.var_hat = mu_hat.value, var_hat.value
        return self.mu_hat, self.var_hat

    def _new(self):
        import torch
        return torch.empty(self.outputSize, self.inputSize, dtype=torch.float32, device=f"cuda:{self.ctx.device}")

    def compute_mugrads(self, opt=None):
        leg, lcg = self._new(), self._new()
        L.check(L.lib().vbnn_layer_grads(self.handle, C.c_void_p(leg.data_ptr()), C.c_void_p(lcg.data_ptr()), None, None))
        return leg, lcg

    def compute_vargrads(self, opt=None):
        leg, lcg = self._new(), self._new()
        L.check(L.lib().vbnn_layer_grads(self.handle, None, None, C.c_void_p(leg.data_ptr()), C.c_void_p(lcg.data_ptr())))
        return leg, lcg

    def calc_lc(self, opt=None):
        lc = self._new()
        L.check(L.lib().vbnn_layer_calc_lc(self.handle, C.c_void_p(lc.data_ptr()), None))
        return lc

    def calc_lc_sum(self):
        s = C.c_float()
        L.check(L.lib().vbnn_layer_calc_lc(self.handle, None, C.byref(s)))
        return s.value

    # ---- VBLinear.lua:124-166 ----
    def update(self, opt=None):
        opt = opt or self.opt
        if opt.get("log"):
            st = L.VbnnStats()
            L.check(L.lib().vbnn_layer_update(self.handle, C.byref(st)))
            self.stats = {name: getattr(st, f) for name, (f, _) in zip(L.STAT_NAMES, L.VbnnStats._fields_)}
            self.var_hat = st.var_hat
            from . import logger
            if logger.Log is not None:                                  # VBLinear.lua:150-163
                for name in L.STAT_NAMES:
                    logger.Log.add(name, self.stats[name])
            return self.stats
        L.check(L.lib().vbnn_layer_update(self.handle, None))
        return None

    def snr_prune_count(self, thresh=0.005):                            # mainviz.lua:20-24
        c = C.c_longlong()
        L.check(L.lib().vbnn_layer_snr_count(self.handle, C.c_float(thresh), None, C.byref(c)))
        return c.value

    def snr_prune_mask(self, thresh=0.005):
        """(mask [O x I] uint8 on the device, count): mainviz.lua:20-22 `torch.lt(|mu| / sigma, thresh)`."""
        import torch
        mask = torch.empty(self.outputSize, self.inputSize, dtype=torch.uint8, device=f"cuda:{self.ctx.device}")
        c = C.c_longlong()
        L.check(L.lib().vbnn_layer_snr_count(self.handle, C.c_float(thresh), C.c_void_p(mask.data_ptr()), C.byref(c)))
        return mask, c.value

    def draw_noise(self, step, sample_idx, rows=0, row0=0):
        """The epsilon [O x I] (or zeta [rows x O] under local reparameterisation) the fused
        kernels generate for (step, sample_idx)."""
        import torch
        lrt = self.opt.get("reparam", "weight") == "local" and self.kind == L.KIND_VB
        shape = (rows, self.outputSize) if lrt else (self.outputSize, self.inputSize)
        out = torch.empty(*shape, dtype=torch.float32, device=f"cuda:{self.ctx.device}")
        L.check(L.lib().vbnn_layer_draw_noise(self.handle, C.c_uint32(step), sample_idx, rows, row0,
                                              C.c_void_p(out.data_ptr())))
        return out


class Linear(VBLinear):
    """Plain nn.Linear behind the same ABI (mlp.lua:29 output layer; quirk Q8)."""
    kind = L.KIND_LINEAR

    @property
    def weight(self):
        return self._view(L.BUF_WEIGHT)
