"""The mlp.lua net object (reference mlp.lua:5-143) over libvbnn.so: buildModel, resetGradients,
sample, run, test, calc_lc, update -- same names and order as the reference so that a
main.lua-style loop drives it unchanged -- plus the fused per-minibatch entry points
(train_step / train_step_host) that keep minibatches, weights and noise on the GPU."""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Optional

from . import _lib as L
from .config import opts_struct, with_live
from .context import Context, as_dev_f32, default_context
from .vblinear import Linear, VBLinear


class Prediction(NamedTuple):
    """MLP.predict's result: device tensors over the N input rows, and the two scalars when targets were given."""
    logp: "torch.Tensor"                  # [N x C] log p-bar(c | x)
    entropy: "torch.Tensor"               # [N] H[p-bar]: total uncertainty
    expected_entropy: "torch.Tensor"      # [N] mean_t H[p_t]: aleatoric
    mutual_info: "torch.Tensor"           # [N] H[p-bar] - mean_t H[p_t] (clamped at 0): epistemic, "BALD"
    label: "torch.Tensor"                 # [N] int64, 1-based argmax of p-bar
    nll: Optional[float]                  # mean -log p-bar(target)
    accuracy: Optional[float]             # % argmax p-bar == target


class OutputPrediction(NamedTuple):
    """MLP.predict_outputs's result over the N input rows (K = C raw, C / 2 gaussian); None where not asked for."""
    mean: "torch.Tensor"                  # [N x K] mean_t m_t
    epistemic: "torch.Tensor"             # [N x K] mean_t (m_t - mean)^2: variance over the weight posterior
    aleatoric: Optional["torch.Tensor"]   # [N x K] mean_t exp(s_t) (gaussian): the head's noise variance
    samples: Optional["torch.Tensor"]     # [T x N x C] every sampled raw output (return_samples)
    nll: Optional[float]                  # mean -log p-bar(y | x) of the per-row Gaussian mixture (gaussian, targets)
    rmse: Optional[float]                 # sqrt(mean (y - mean)^2) (targets)


class MLP:
    def __init__(self, opt=None, ctx: Context = None, max_batch=None):
        self.handle = None
        if opt is not None:
            self.buildModel(opt, ctx, max_batch)

    # ---- mlp.lua:7-60 ----
    def buildModel(self, opt, ctx: Context = None, max_batch=None):
        self.opt = opt
        self.ctx = ctx or default_context(seed=opt.get("seed", 3))
        sizes = [int(opt["input_size"])] + [int(h) for h in opt["hidden"]] + [len(opt["classes"])]
        self.sizes = sizes
        self.max_batch = int(max_batch or max(opt["batchSize"], opt.get("testBatchSize", 1)))
        arr = (C.c_int * len(sizes))(*sizes)
        o = opts_struct(opt)
        self.handle = C.c_void_p()
        L.check(L.lib().vbnn_mlp_create(self.ctx.handle, arr, len(sizes), 1 if opt.get("vb_output") else 0,
                                        self.max_batch, C.byref(o), C.byref(self.handle)))
        self.model = []
        self.vb_indices = []                                            # mlp.lua:9,15,23
        n = L.lib().vbnn_mlp_num_layers(self.handle)
        for k in range(n):
            h = C.c_void_p()
            L.check(L.lib().vbnn_mlp_layer(self.handle, k, C.byref(h)))
            vb = k < n - 1 or opt.get("vb_output")
            cls = VBLinear if vb else Linear
            self.model.append(cls(sizes[k], sizes[k + 1], opt, self.ctx, _borrowed=h))
            if vb:
                self.vb_indices.append(k)
        self._s = 0
        prior = opt.get("prior", "empirical")
        if prior not in ("empirical", "fixed"):
            raise L.VbnnError(L.E_INVALID, f"opt.prior must be 'empirical' or 'fixed', got {prior!r}")
        if prior == "fixed":
            self.set_prior("fixed", opt.get("prior_mean", 0.0), opt.get("prior_var"))
        return self

    def set_prior(self, kind, mean=0.0, var=None):
        """VBLinear.set_prior on every VB layer (the hidden layers and a vb_output layer); "per_weight" makes each
        layer's current posterior its prior.  Each step graph of the net re-captures once at its next use."""
        for k in self.vb_indices:
            self.model[k].set_prior(kind, mean, var)

    def set_opt(self, opt):
        """VBLinear.set_opt on every layer in one call (vbnn_mlp_set_opts), for a learning-rate schedule or KL annealing:
        decay opt's learning rates or change opt["B"], then set_opt(opt) before the next step.  No step graph is
        re-captured.  A change of a key the net was built with (S, reparam, precision, ...) is refused
        (VbnnError(E_INVALID), nothing changes).  self.opt (what checkpoint.save_net records) takes opt's live keys --
        B, state, meanState, varState -- and keeps every other key.  In data-parallel training set the same values on
        every rank."""
        L.check(L.lib().vbnn_mlp_set_opts(self.handle, C.byref(opts_struct(opt))))
        self.opt = with_live(self.opt, opt)
        for m in self.model:
            m.opt = self.opt

    def init_params(self, seed=4, he_means=False):
        """means per VBLinear.lua:22-29 (or He-scaled, SURVEY 8d), Linear weights N(0, 2/fan_in)
        and zero biases per mlp.lua:47-55, drawn on the device."""
        L.check(L.lib().vbnn_mlp_init_params(self.handle, C.c_uint64(seed), 1 if he_means else 0))

    def __del__(self):
        try:
            if self.handle:
                for m in self.model:
                    m.handle = None
                L.lib().vbnn_mlp_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def _io(self, inputs, targets):
        x = as_dev_f32(inputs, self.ctx.device)
        x = x.reshape(x.shape[0], -1)                                   # nn.Reshape (mlp.lua:12)
        t = as_dev_f32(targets, self.ctx.device).reshape(-1)
        if x.shape[1] != self.sizes[0] or t.shape[0] != x.shape[0]:
            raise L.VbnnError(L.E_INVALID, f"inputs must be [N x {self.sizes[0]}] with N targets")
        return x, t

    # ---- mlp.lua:62-84 ----
    def resetGradients(self):
        L.check(L.lib().vbnn_mlp_reset_gradients(self.handle))
        self._s = 0
        self._open_n = None                                             # an open forward_train step is abandoned

    def sample(self, sample_idx=None):
        if sample_idx is not None:
            self._s = int(sample_idx)
        L.check(L.lib().vbnn_mlp_sample(self.handle, self._s))
        self._cur = self._s
        self._s += 1

    def run(self, inputs, targets):
        x, t = self._io(inputs, targets)
        err, acc = C.c_float(), C.c_float()
        s = getattr(self, "_cur", 0)
        if self.opt.get("reparam", "weight") == "local":
            s = self._s
            self._s += 1
        L.check(L.lib().vbnn_mlp_run(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                     x.shape[0], s, C.byref(err), C.byref(acc)))
        return err.value, acc.value

    # ---- mlp.lua:86-107 ----
    def test(self, input, target):
        x, t = self._io(input, target)
        err, acc = C.c_float(), C.c_float()
        ns = 0 if self.opt.get("quicktest") else int(self.opt["testSamples"])
        L.check(L.lib().vbnn_mlp_test(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                      x.shape[0], ns, C.byref(err), C.byref(acc)))
        return err.value, acc.value

    def predict(self, inputs, n_samples=None, targets=None):
        """Bayesian model average over n_samples sampled forward passes (vbnn_mlp_predict); test() keeps the
        reference's averaged error / accuracy scalars, this averages the probabilities.  n_samples defaults to
        what test() uses: 0 (one MAP pass) under quicktest, else testSamples.  Returns a Prediction of device
        tensors -- logp [N x C] = log p-bar, entropy H[p-bar], expected_entropy mean_t H[p_t], mutual_info (their
        difference, clamped at 0), label (1-based argmax of p-bar) -- plus nll / accuracy floats, None without
        targets.  Parameters, optimiser state and the step counter are left as they are."""
        import torch
        x = as_dev_f32(inputs, self.ctx.device)
        x = x.reshape(x.shape[0], -1)
        if x.shape[1] != self.sizes[0]:
            raise L.VbnnError(L.E_INVALID, f"inputs must be [N x {self.sizes[0]}]")
        if n_samples is None:
            n_samples = 0 if self.opt.get("quicktest") else int(self.opt["testSamples"])
        n = x.shape[0]
        t = None
        if targets is not None:
            t = as_dev_f32(targets, self.ctx.device).reshape(-1)
            if t.shape[0] != n:
                raise L.VbnnError(L.E_INVALID, "predict needs one target per input row")
        logp = torch.empty(n, self.sizes[-1], dtype=torch.float32, device=x.device)
        unc = torch.empty(n, 4, dtype=torch.float32, device=x.device)
        nll, acc = C.c_float(), C.c_float()
        want = t is not None
        L.check(L.lib().vbnn_mlp_predict(self.handle, C.c_void_p(x.data_ptr()), n, int(n_samples),
                                         C.c_void_p(t.data_ptr()) if want else None, C.c_void_p(logp.data_ptr()),
                                         C.c_void_p(unc.data_ptr()), C.byref(nll) if want else None,
                                         C.byref(acc) if want else None))
        return Prediction(logp, unc[:, 0], unc[:, 1], unc[:, 2], unc[:, 3].long(),
                          nll.value if want else None, acc.value if want else None)

    def predict_outputs(self, inputs, n_samples=None, model="raw", targets=None, return_samples=False):
        """Model average of the raw outputs for regression heads (vbnn_mlp_predict_outputs): the sampled forward
        passes of predict(), read without LogSoftMax.  model "raw": the C outputs are the prediction (K = C);
        "gaussian": C = 2K, columns [0, K) are means and [K, 2K) log-variances of a heteroscedastic Gaussian, as
        trained under gaussian_nll_loss(Y[..., :K], y, Y[..., K:].exp()).  n_samples defaults as in predict().
        targets: [N x K] regression targets, which add rmse and, under "gaussian", the mixture's mean NLL.  Returns an
        OutputPrediction; the predictive variance is epistemic + aleatoric.  Parameters, optimiser state and the step
        counter are left as they are."""
        import torch
        if model not in L.OUTPUT_MODELS:
            raise L.VbnnError(L.E_INVALID, f"model must be 'raw' or 'gaussian', got {model!r}")
        gaussian = model == "gaussian"
        x = as_dev_f32(inputs, self.ctx.device)
        x = x.reshape(x.shape[0], -1)
        if x.shape[1] != self.sizes[0]:
            raise L.VbnnError(L.E_INVALID, f"inputs must be [N x {self.sizes[0]}]")
        if n_samples is None:
            n_samples = 0 if self.opt.get("quicktest") else int(self.opt["testSamples"])
        n, c = x.shape[0], self.sizes[-1]
        k = c // 2 if gaussian else c
        t = None
        if targets is not None:
            t = as_dev_f32(targets, self.ctx.device).reshape(n, -1)
            if t.shape[1] != k:
                raise L.VbnnError(L.E_INVALID, f"targets must be [N x {k}]")
        dev = x.device
        mean = torch.empty(n, k, dtype=torch.float32, device=dev)
        epi = torch.empty(n, k, dtype=torch.float32, device=dev)
        ale = torch.empty(n, k, dtype=torch.float32, device=dev) if gaussian else None
        smp = torch.empty(max(int(n_samples), 1), n, c, dtype=torch.float32, device=dev) if return_samples else None
        nll, rmse = C.c_float(), C.c_float()
        want_nll = t is not None and gaussian
        ptr = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None
        L.check(L.lib().vbnn_mlp_predict_outputs(self.handle, ptr(x), n, int(n_samples), L.OUTPUT_MODELS[model], ptr(t),
                                                 ptr(smp), ptr(mean), ptr(epi), ptr(ale),
                                                 C.byref(nll) if want_nll else None,
                                                 C.byref(rmse) if t is not None else None))
        return OutputPrediction(mean, epi, ale, smp, nll.value if want_nll else None,
                                rmse.value if t is not None else None)

    def calc_lc(self, opt=None):                                        # mlp.lua:109-115
        v = C.c_float()
        L.check(L.lib().vbnn_mlp_calc_lc(self.handle, C.byref(v)))
        return v.value

    def update(self, opt=None):                                         # mlp.lua:117-142
        opt = opt or self.opt
        from . import logger
        if opt.get("log") and logger.Log is not None and self.ctx.nranks == 1:
            # with logging on the reference syncs >= 13 scalars per layer anyway (VBLinear.lua:150-163): go
            # layer by layer so every VBLinear reports its 14 diagnostics -- output-layer SGD first
            # (mlp.lua:120-123), then the VB layers in index order (:138-140); all layers log to the same
            # ids, interleaved, exactly as the reference does
            if self.model[-1].kind == L.KIND_LINEAR:
                L.check(L.lib().vbnn_layer_update(self.model[-1].handle, None))
            for k in self.vb_indices:
                self.model[k].update(opt)
            self.ctx.set_step(self.ctx.get_step() + 1)
            return
        L.check(L.lib().vbnn_mlp_update(self.handle))

    # ---- fused minibatch: main.lua:28-40 in one call ----
    def train_step(self, inputs, targets, sync=True, grad_input=None):
        """inputs/targets already on the device.  Returns (error, accuracy) averaged over the S
        samples as main.lua:38-39 (or None when sync=False).

        grad_input: optional preallocated contiguous float32 CUDA tensor [N, input_size] on the context's device.
        The step is then vbnn_mlp_step_grad_input: the same minibatch, bit for bit, and grad_input is overwritten
        with sum_s d loss_s / d inputs through this minibatch's samples and the parameters before its update --
        what a feature extractor below the net receives in the reference (feats.backward(grad_input)).  Data
        parallel: the derivative of the global mean loss (a DDP extractor, which averages, must scale by nranks).
        Reuse one tensor: the step's CUDA graph is keyed on its address."""
        import torch
        x, t = self._io(inputs, targets)
        if not hasattr(self, "_res"):
            self._res = torch.zeros(2, dtype=torch.float32, device=x.device)
        if grad_input is None:
            L.check(L.lib().vbnn_mlp_step(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                          x.shape[0], C.c_void_p(self._res.data_ptr())))
        else:
            g = grad_input
            if (not isinstance(g, torch.Tensor) or g.dtype != torch.float32 or not g.is_cuda
                    or g.device != x.device or tuple(g.shape) != (x.shape[0], self.sizes[0])
                    or not g.is_contiguous()):
                raise L.VbnnError(L.E_INVALID, f"grad_input must be a contiguous float32 tensor [{x.shape[0]}, "
                                               f"{self.sizes[0]}] on {x.device}")
            L.check(L.lib().vbnn_mlp_step_grad_input(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                                     x.shape[0], C.c_void_p(self._res.data_ptr()),
                                                     C.c_void_p(g.data_ptr())))
        if not sync:
            return None
        r = self._res.cpu()
        return float(r[0]), float(r[1])

    # ---- the fused minibatch split around the caller's loss (vbnn_mlp_forward_train / vbnn_mlp_backward_update) ----
    def forward_train(self, inputs):
        """First half of train_step without its loss: sample and run the forward of the S samples at the current step.
        Returns the output layer's pre-LogSoftMax outputs Y, a float32 device tensor [S, N, C].  The tensor belongs to
        the binding and is overwritten by the next forward_train of the same N (the forward's CUDA graph is keyed on
        it): clone it to keep it.  Opens a step that backward_update closes (resetGradients abandons it)."""
        import torch
        x = as_dev_f32(inputs, self.ctx.device)
        x = x.reshape(x.shape[0], -1)
        if x.shape[1] != self.sizes[0]:
            raise L.VbnnError(L.E_INVALID, f"inputs must be [N x {self.sizes[0]}]")
        n = x.shape[0]
        if not hasattr(self, "_logits"):
            self._logits = {}
        y = self._logits.get(n)
        if y is None:
            y = torch.empty(int(self.opt["S"]), n, self.sizes[-1], dtype=torch.float32, device=x.device)
            self._logits[n] = y
        L.check(L.lib().vbnn_mlp_forward_train(self.handle, C.c_void_p(x.data_ptr()), n, C.c_void_p(y.data_ptr())))
        self._open_n = n
        return y

    def backward_update(self, grad, grad_input=None):
        """Second half: grad = dL/dY, a contiguous float32 device tensor [S, N, C] where L is the SUM over the S samples
        of the per-sample loss (train_step is the case of the batch-mean ClassNLL of LogSoftMax(Y_s) per sample).
        Runs the backward, [exchange], KL + Adam update and step-counter bump of train_step; grad_input, as in
        train_step, is overwritten with dL/d inputs.  Asynchronous."""
        import torch
        n = getattr(self, "_open_n", None)
        if n is None:
            raise L.VbnnError(L.E_STATE, "backward_update: no open step (call forward_train first)")
        dev = torch.device(f"cuda:{self.ctx.device}")
        shape = (int(self.opt["S"]), n, self.sizes[-1])
        if (not isinstance(grad, torch.Tensor) or grad.dtype != torch.float32 or not grad.is_cuda or grad.device != dev
                or tuple(grad.shape) != shape or not grad.is_contiguous()):
            raise L.VbnnError(L.E_INVALID, f"grad must be a contiguous float32 tensor {list(shape)} on {dev}")
        g = grad_input
        if g is not None and (not isinstance(g, torch.Tensor) or g.dtype != torch.float32 or not g.is_cuda
                              or g.device != dev or tuple(g.shape) != (n, self.sizes[0]) or not g.is_contiguous()):
            raise L.VbnnError(L.E_INVALID, f"grad_input must be a contiguous float32 tensor [{n}, {self.sizes[0]}] "
                                           f"on {dev}")
        self._open_n = None
        L.check(L.lib().vbnn_mlp_backward_update(self.handle, C.c_void_p(grad.data_ptr()),
                                                 C.c_void_p(g.data_ptr()) if g is not None else None))

    def train_step_loss(self, inputs, loss_fn, grad_input=None):
        """One minibatch under any torch loss: forward_train, loss = loss_fn(Y) on a detached leaf Y [S, N, C] that
        requires grad, torch.autograd.grad, backward_update.  loss_fn must return the SUM over the S samples of the
        per-sample loss to match train_step (for ClassNLL: sum_s nll_loss(log_softmax(Y[s]), t), each a batch mean).
        Returns the loss as a device tensor without synchronising.  If loss_fn or the argument checks raise, the step
        is abandoned (resetGradients; in peer mode it is closed with a zero gradient, which keeps the peers in step)."""
        import torch
        y = self.forward_train(inputs)
        try:
            leaf = y.detach().requires_grad_(True)
            with torch.enable_grad():
                loss = loss_fn(leaf)
                (g,) = torch.autograd.grad(loss, leaf)
            self.backward_update(g.contiguous(), grad_input)
        except BaseException:
            if self._open_n is not None:
                if self.peer_active:
                    self.backward_update(torch.zeros_like(y))
                else:
                    self._open_n = None
                    self.resetGradients()
            raise
        return loss.detach()

    def train_step_host(self, inputs_host, targets_host):
        """HOST buffers in, host scalars out: H2D and D2H inside the call (main.lua:23-24)."""
        x, t = self._host_io(inputs_host, targets_host)
        err, acc = C.c_float(), C.c_float()
        L.check(L.lib().vbnn_mlp_step_host(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                           x.shape[0], C.byref(err), C.byref(acc)))
        return err.value, acc.value

    def _host_io(self, inputs_host, targets_host):
        import torch
        x = torch.as_tensor(inputs_host, dtype=torch.float32)
        t = torch.as_tensor(targets_host, dtype=torch.float32)
        if x.is_cuda or t.is_cuda:
            raise L.VbnnError(L.E_INVALID, "train_step_host expects host tensors")
        x = x.reshape(x.shape[0], -1).contiguous()
        return x, t.reshape(-1).contiguous()

    def submit_host(self, inputs_host, targets_host):
        x, t = self._host_io(inputs_host, targets_host)
        self._keep = getattr(self, "_keep", [])
        self._keep.append((x, t))
        self._keep = self._keep[-4:]
        L.check(L.lib().vbnn_mlp_submit_host(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                             x.shape[0]))

    def submit_host_u8(self, pixels_host, targets_host, mean, std):
        """The dataset's native bytes (MNIST pixels before data.lua:25 u.normalize): uint8 [N x input_size] host
        tensor; (x - mean) / std is applied on the device while staging the GEMM operand."""
        import torch
        x = torch.as_tensor(pixels_host)
        if x.dtype != torch.uint8 or x.is_cuda:
            raise L.VbnnError(L.E_INVALID, "submit_host_u8 expects a uint8 host tensor")
        x = x.reshape(x.shape[0], -1).contiguous()
        t = torch.as_tensor(targets_host, dtype=torch.float32).reshape(-1).contiguous()
        self._keep = getattr(self, "_keep", [])
        self._keep.append((x, t))
        self._keep = self._keep[-4:]
        L.check(L.lib().vbnn_mlp_submit_host_u8(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                                x.shape[0], C.c_float(mean), C.c_float(1.0 / std)))

    def join_streams(self):
        L.check(L.lib().vbnn_mlp_join_streams(self.handle))

    def collect(self):
        err, acc = C.c_float(), C.c_float()
        L.check(L.lib().vbnn_mlp_collect(self.handle, C.byref(err), C.byref(acc)))
        return err.value, acc.value

    def outputs(self, sample_idx=0, n=None):
        """LogSoftMax output of the last forward (self.model.output in the reference)."""
        import torch
        n = n or self._last_n()
        out = torch.empty(n, self.sizes[-1], dtype=torch.float32)
        L.check(L.lib().vbnn_mlp_get_outputs(self.handle, sample_idx, C.c_void_p(out.data_ptr())))
        return out

    def _last_n(self):
        return self.max_batch

    # ---- checkpoint / resume (reference: u.safe_save(net) main.lua:181, utils.lua:73-80; resume
    # main.lua:146-148).  The reference torch.save()s the whole object graph; here the device state
    # is exported as a flat dict of CPU tensors (means, lvars, bias, Adam m/v/t per layer, the output
    # layer, the Philox step counter, each layer's live hyper-parameters "{k}.opts" in L.LIVE_OPTS
    # order) that torch.save / numpy can persist.
    def state_dict(self):
        import torch
        sd = {"sizes": list(self.sizes), "step": self.ctx.get_step()}
        names = [("means", L.BUF_MEANS), ("lvars", L.BUF_LVARS), ("bias", L.BUF_BIAS), ("m_mu", L.BUF_ADAM_M_MU),
                 ("v_mu", L.BUF_ADAM_V_MU), ("m_var", L.BUF_ADAM_M_VAR), ("v_var", L.BUF_ADAM_V_VAR)]
        for k, m in enumerate(self.model):
            if m.kind == L.KIND_VB:
                for n, b in names:
                    sd[f"{k}.{n}"] = m.get(b)
                if self.opt.get("strict_reference", True):
                    sd[f"{k}.stdv"] = m.get(L.BUF_STDV)
                    sd[f"{k}.mu_sqe"] = m.get(L.BUF_MU_SQE)
                kind, mean, var = m.prior
                sd[f"{k}.prior"] = L.PRIOR_KINDS[kind]
                if kind == "fixed":
                    sd[f"{k}.prior_mean"], sd[f"{k}.prior_var"] = mean, var
                if kind == "per_weight":
                    sd[f"{k}.prior_means"] = m.get(L.BUF_PRIOR_MEANS)
                    sd[f"{k}.prior_lvars"] = m.get(L.BUF_PRIOR_LVARS)
            else:
                sd[f"{k}.weight"] = m.get(L.BUF_WEIGHT)
                sd[f"{k}.bias"] = m.get(L.BUF_BIAS)
            sd[f"{k}.t"] = m.t
            live = m.opts
            sd[f"{k}.opts"] = torch.tensor([live[f] for f in L.LIVE_OPTS], dtype=torch.float32)
        return sd

    def load_state_dict(self, sd):
        if list(sd["sizes"]) != list(self.sizes):
            raise L.VbnnError(L.E_INVALID, f"checkpoint is for sizes {sd['sizes']}, net has {self.sizes}")
        codes = dict(means=L.BUF_MEANS, lvars=L.BUF_LVARS, bias=L.BUF_BIAS, m_mu=L.BUF_ADAM_M_MU, v_mu=L.BUF_ADAM_V_MU,
                     m_var=L.BUF_ADAM_M_VAR, v_var=L.BUF_ADAM_V_VAR, weight=L.BUF_WEIGHT, stdv=L.BUF_STDV,
                     mu_sqe=L.BUF_MU_SQE)
        kinds = {c: n for n, c in L.PRIOR_KINDS.items()}
        for k, m in enumerate(self.model):
            L.check(L.lib().vbnn_layer_set_t(m.handle, int(sd[f"{k}.t"])))
            if f"{k}.opts" in sd:                                        # older checkpoints keep the net's values
                o = m._get_opts()
                live = dict(zip(L.LIVE_OPTS, [float(v) for v in sd[f"{k}.opts"]]))
                for f, v in live.items():
                    setattr(o, f, v)
                L.check(L.lib().vbnn_layer_set_opts(m.handle, C.byref(o)))
                m.opt = with_live(self.opt, m.opts)
            if m.kind == L.KIND_VB:
                # before the parameters: a per_weight prior snapshots them, then takes its own arrays below.  A
                # checkpoint without prior keys (older files) is the empirical prior.
                kind = kinds[int(sd.get(f"{k}.prior", L.PRIOR_EMPIRICAL))]
                m.set_prior(kind, float(sd.get(f"{k}.prior_mean", 0.0)), sd.get(f"{k}.prior_var"))
                if kind == "per_weight":
                    m.set(L.BUF_PRIOR_MEANS, sd[f"{k}.prior_means"])
                    m.set(L.BUF_PRIOR_LVARS, sd[f"{k}.prior_lvars"])
            for n, b in codes.items():
                if f"{k}.{n}" in sd:
                    m.set(b, sd[f"{k}.{n}"])
            if m.kind == L.KIND_VB and f"{k}.stdv" not in sd:
                m.compute_prior()
        if "0.opts" in sd:
            # the net's opt (what save_net records) follows the first layer, as MLP.set_opt sets every layer alike
            self.opt = with_live(self.opt, self.model[0].opts)
        self.ctx.set_step(int(sd["step"]))

    # ---- data parallel over NVLink peer memory (new; include/vbnn.h "peer mode") ----
    def enable_peer(self, all_gather_bytes):
        """all_gather_bytes(blob: bytes) -> list[bytes] in rank order (e.g. over torch.distributed).
        After this, train_step / submit_host exchange gradients through the fused dW-epilogue
        reduce-scatter + sharded update + copy-engine all-gather instead of an NCCL allreduce."""
        n = C.c_size_t()
        L.check(L.lib().vbnn_mlp_peer_export(self.handle, None, 0, C.byref(n)))
        buf = (C.c_char * n.value)()
        L.check(L.lib().vbnn_mlp_peer_export(self.handle, buf, n.value, C.byref(n)))
        blobs = all_gather_bytes(bytes(buf))
        if len(blobs) != self.ctx.nranks or any(len(b) != n.value for b in blobs):
            raise L.VbnnError(L.E_INVALID, "enable_peer: all_gather_bytes must return one blob per rank")
        joined = b"".join(blobs)
        L.check(L.lib().vbnn_mlp_peer_import(self.handle, joined, n.value))

    @property
    def peer_active(self):
        return bool(L.lib().vbnn_mlp_peer_active(self.handle))

    def sync_replicas(self):
        """Collective: call on every rank between two host barriers (see vbnn_mlp_sync_replicas)."""
        L.check(L.lib().vbnn_mlp_sync_replicas(self.handle))

    def launch_count(self):
        v = C.c_longlong()
        L.check(L.lib().vbnn_mlp_launch_count(self.handle, C.byref(v)))
        return v.value

    def graph_captures(self):
        """CUDA graphs this net has captured (vbnn_mlp_graph_captures)."""
        v = C.c_longlong()
        L.check(L.lib().vbnn_mlp_graph_captures(self.handle, C.byref(v)))
        return v.value

    def grad_arena(self):
        import torch
        from .context import DevView
        p, n = C.c_void_p(), C.c_size_t()
        L.check(L.lib().vbnn_mlp_grad_arena(self.handle, C.byref(p), C.byref(n)))
        return torch.as_tensor(DevView(p.value, (n.value,)), device=f"cuda:{self.ctx.device}")
