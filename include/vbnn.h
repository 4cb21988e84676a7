/*
 * vbnn.h -- C ABI of libvbnn.so: the B200-native (sm_100a) VBLinear hot path of louissmit/VBNN.
 *
 * This is the drop-in boundary.  Every entry point replaces one call the reference makes
 * through Torch7's nn.Module protocol on class nn.VBLinear (reference VBLinear.lua:7) or through
 * the mlp.lua net object; the reference interface each one replaces is cited as file:line.
 * The reference-side binding (LuaJIT ffi.cdef over this header) is lua/VBLinear.lua; see
 * INTEGRATION.md.
 *
 * Conventions
 *   - plain C, opaque handles, plain pointers and sizes; no C++/torch types cross the ABI;
 *   - every function returns int: 0 = VBNN_OK, negative = VBNN_E_*; vbnn_last_error() gives a
 *     thread-local message; nothing throws or exits across the ABI;
 *   - all tensors are fp32, row-major, dense, exactly as the reference's torch.FloatTensor /
 *     CudaTensor (main.lua:10): weights are [outputSize x inputSize] (VBLinear.lua:18-23),
 *     activations are [N x features]; class targets are 1-based floats (data.lua:16);
 *   - pointers named *_dev are device pointers on the context's GPU, borrowed for the call;
 *     pointers named *_host are host pointers (pinned memory makes the copies asynchronous);
 *   - work is enqueued on the context's stream; a function that returns a host scalar
 *     synchronises that stream, nothing else does;
 *   - there is no CPU fallback: without a CUDA device every compute entry returns VBNN_E_CUDA.
 */
#ifndef VBNN_H
#define VBNN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VBNN_ABI_VERSION 2

typedef struct vbnn_ctx vbnn_ctx;     /* one per (GPU, host thread)                         */
typedef struct vbnn_layer vbnn_layer; /* one nn.VBLinear (VBLinear.lua:7) or plain nn.Linear */
typedef struct vbnn_mlp vbnn_mlp;     /* the mlp.lua net object (mlp.lua:5-143)              */

enum vbnn_status {
  VBNN_OK = 0,
  VBNN_E_INVALID = -1,     /* bad argument / shape mismatch (Torch would raise a Lua error) */
  VBNN_E_CUDA = -2,        /* CUDA runtime/driver error, or no device                       */
  VBNN_E_NOMEM = -3,
  VBNN_E_UNSUPPORTED = -4,
  VBNN_E_NCCL = -5,
  VBNN_E_STATE = -6        /* call order violated (e.g. backward before forward)            */
};

enum vbnn_reparam {
  VBNN_REPARAM_WEIGHT = 0, /* W = mu + sigma*eps per MC sample -- the reference (VBLinear.lua:59)  */
  VBNN_REPARAM_LOCAL = 1   /* local reparameterisation: Y = X mu^T + sqrt(X^2 s2^T)*zeta (new)    */
};
/* Local reparameterisation keeps R = zeta / (2 sqrt(V)), V = X^2 s2^T, for the backward.  Where V == 0 (an all-zero
 * input row: zero-padded minibatch rows, or a hidden row whose units are all dead after ReLU) R := 0, so the variance
 * term adds nothing to gradInput or gradSum for that row; the row's output is X mu^T + b.  Any V > 0, subnormal ones
 * included, gets the finite zeta / (2 sqrt(V)). */

enum vbnn_precision {
  VBNN_PREC_FP32 = 0,      /* fp32 operands, fp32 accumulate, CUDA-core GEMM (exact-parity mode)   */
  VBNN_PREC_BF16 = 1       /* bf16 operands, fp32 accumulate, tcgen05/TMEM tensor-core GEMM        */
};

enum vbnn_kind { VBNN_KIND_VB = 0, VBNN_KIND_LINEAR = 1 };

/* names for vbnn_layer_get / vbnn_layer_set; all fp32, [O x I] unless noted */
enum vbnn_buf {
  VBNN_BUF_MEANS = 0,      /* self.means      VBLinear.lua:23                  */
  VBNN_BUF_LVARS = 1,      /* self.lvars      VBLinear.lua:18                  */
  VBNN_BUF_BIAS = 2,       /* self.bias [O]   VBLinear.lua:13                  */
  VBNN_BUF_WEIGHT = 3,     /* self.weight (last sampled W)   VBLinear.lua:63   */
  VBNN_BUF_GRAD_WEIGHT = 4,/* self.gradWeight VBLinear.lua:113                 */
  VBNN_BUF_GRAD_SUM = 5,   /* self.gradSum    VBLinear.lua:20,115              */
  VBNN_BUF_GRAD_BIAS = 6,  /* self.gradBias [O]                                */
  VBNN_BUF_ADAM_M_MU = 7,  /* meanState.m     VBLinear.lua:32,135              */
  VBNN_BUF_ADAM_V_MU = 8,
  VBNN_BUF_ADAM_M_VAR = 9, /* varState.m      VBLinear.lua:33,140              */
  VBNN_BUF_ADAM_V_VAR = 10,
  VBNN_BUF_EPS = 11,       /* self.e (last epsilon)  VBLinear.lua:37,55        */
  VBNN_BUF_STDV = 12,      /* self.stdv cached by compute_prior  VBLinear.lua:79 */
  VBNN_BUF_MU_SQE = 13,    /* self.mu_sqe cached by compute_prior VBLinear.lua:82 */
  VBNN_BUF_PRIOR_MEANS = 14, /* prior means mu0 [O x I]        (VBNN_PRIOR_PER_WEIGHT only) */
  VBNN_BUF_PRIOR_LVARS = 15, /* prior log-variances l0 [O x I] (VBNN_PRIOR_PER_WEIGHT only) */
  VBNN_BUF__COUNT = 16
};

/* The prior N(mu_hat, var_hat) of the KL ("complexity") terms of a VB layer (vbnn_layer_set_prior). */
enum vbnn_prior {
  VBNN_PRIOR_EMPIRICAL = 0,  /* Graves' empirical Bayes, the reference: mu_hat = 0 (VBLinear.lua:81),
                                var_hat = mean(sigma^2 + mu^2) re-estimated at every update (:86)         */
  VBNN_PRIOR_FIXED = 1,      /* scalars mu_hat = mu0, var_hat = var0 > 0                                  */
  VBNN_PRIOR_PER_WEIGHT = 2  /* per-weight arrays mu_hat = mu0[o,i], var_hat = exp(l0[o,i]): the buffers
                                VBNN_BUF_PRIOR_MEANS / _LVARS, same parameterisation as means / lvars     */
};

/* config.lua restated; vbnn_opts_default() fills the reference's shipped values. */
typedef struct vbnn_opts {
  float var_init;          /* config.lua:44 (0.001)                                        */
  int msr_init;            /* config.lua:45: var_init = 2/inputSize (VBLinear.lua:14-16)   */
  float mu_init;           /* config.lua:43: 0 -> means = 0, else means ~ N(0, var_init)   */
  float B;                 /* config.lua:30 (1e6): number of minibatches, scales the KL    */
  int S;                   /* config.lua:32: Monte-Carlo weight samples per minibatch      */
  float lr_bias;           /* opt.state.learningRate      config.lua:51-54 (1e-3)          */
  float lr_mu;             /* opt.meanState.learningRate  config.lua:60-64 (1e-4)          */
  float lr_var;            /* opt.varState.learningRate   config.lua:55-59 (0.05)          */
  float adam_beta1, adam_beta2, adam_eps; /* optim.adam defaults 0.9, 0.999, 1e-8         */
  int reparam;             /* enum vbnn_reparam                                            */
  int precision;           /* enum vbnn_precision                                          */
  int strict_reference;    /* 1: reproduce quirks Q1/Q6 (sample() and calc_lc() use the
                              sigma / mu^2 cached by the last compute_prior)               */
} vbnn_opts;

/* the 14 diagnostics VBLinear.lua:150-163 logs, in file order */
typedef struct vbnn_stats {
  float vlc_grad, vle_grad, mlc_grad, mle_grad;
  float min_variance, max_variance, mean_variance, var_hat;
  float mean_means, std_means, min_means, max_means;
  float mu_normratio, var_normratio;
} vbnn_stats;

/* ---------------------------------------------------------------- library ------------ */
int vbnn_abi_version(void);
const char* vbnn_last_error(void);
void vbnn_opts_default(vbnn_opts* opts);

/* ---------------------------------------------------------------- context ------------
 * replaces: require 'cunn' + the implicit cutorch default stream (VBLinear.lua:2, main.lua:1),
 * torch.manualSeed (config.lua:40).  `stream` is a cudaStream_t (NULL = a private stream). */
int vbnn_ctx_create(int device, void* stream, uint64_t seed, vbnn_ctx** out);
/* Which stream the context enqueues on.  The reference's other modules (nn.ReLU, nn.LogSoftMax, the
 * criterion: mlp.lua:19,27,30,32) run on cutorch's LEGACY DEFAULT stream (stream 0), with which a
 * non-blocking private stream does not synchronise -- a layer-level drop-in must therefore share it:
 *   VBNN_CTX_STREAM_GIVEN           `stream` as passed (NULL = private non-blocking stream: the net-level
 *                                   entry points, which own the whole minibatch; = vbnn_ctx_create)
 *   VBNN_CTX_STREAM_LEGACY_DEFAULT  stream 0 itself (`stream` must be NULL): every call is ordered with
 *                                   the caller's default-stream work exactly like a cunn module.  CUDA
 *                                   graphs cannot capture stream 0, so vbnn_mlp_step launches eagerly.
 *   VBNN_CTX_STREAM_PRIVATE_BLOCKING a private stream created without cudaStreamNonBlocking: it keeps
 *                                   graph replay and still synchronises implicitly with stream 0. */
enum vbnn_ctx_stream {
  VBNN_CTX_STREAM_GIVEN = 0,
  VBNN_CTX_STREAM_LEGACY_DEFAULT = 1,
  VBNN_CTX_STREAM_PRIVATE_BLOCKING = 2
};
int vbnn_ctx_create_ex(int device, void* stream, int stream_mode, uint64_t seed, vbnn_ctx** out);
int vbnn_ctx_destroy(vbnn_ctx* ctx);
int vbnn_ctx_synchronize(vbnn_ctx* ctx);
/* Per-launch device timing of the tensor-core GEMM: CUDA events on the context's stream around
 * every launch, summed per epilogue class (0 store, 1 fwd, 2 fwd-lrt, 3 dx, 4 dx-lrt, 5 dw,
 * 6 dw-lrt) together with the algorithmic flops; class 7 is the fused KL + Adam update, whose
 * "flops" slot holds its algorithmic HBM bytes (56 B per weight, 64 under VBNN_PRIOR_PER_WEIGHT); class 8 is vbnn_mlp_predict's averaging
 * kernel and vbnn_mlp_predict_outputs' moments kernel, whose "flops" slot likewise holds bytes (20 B per (row,
 * class, sample) for predict; for predict_outputs, per (row, sample), 28 B per mean column and 12 B per
 * log-variance column: zc * N * 28 * C under RAW, zc * N * 40 * K under GAUSSIAN, per chunk of zc samples).
 * Enabling it disables graph replay.  This is
 * what bench.py's roofline object is computed from. */
int vbnn_ctx_profile(vbnn_ctx* ctx, int enable);
int vbnn_ctx_profile_read(vbnn_ctx* ctx, int cls, double* total_ms, long long* launches, double* flops);
/* same switch: time between phase marks of the minibatch (1 start..params ready, 2 sample, 3 forward,
 * 4 loss, 5 backward (per layer), 6 exchange + update, 7 finalise) */
int vbnn_ctx_phase_read(vbnn_ctx* ctx, int id, double* total_ms, long long* count);
int vbnn_ctx_set_step(vbnn_ctx* ctx, uint32_t step);   /* Philox "minibatch" counter */
int vbnn_ctx_get_step(vbnn_ctx* ctx, uint32_t* step);

/* ---------------------------------------------------------------- nn.VBLinear --------- */
/* nn.VBLinear(inputSize, outputSize, opt)  VBLinear.lua:9-47 (kind VB) or nn.Linear (mlp.lua:29) */
int vbnn_layer_create(vbnn_ctx* ctx, int inputSize, int outputSize, int kind,
                      const vbnn_opts* opts, vbnn_layer** out);
int vbnn_layer_destroy(vbnn_layer* layer);
int vbnn_layer_dims(const vbnn_layer* layer, int* inputSize, int* outputSize);

/* VBLinear:sample(opt)  VBLinear.lua:49-64.  eps_dev == NULL: epsilon is drawn on the device
 * (Philox4x32-10, counter = (element, layer, sample_idx, step)); otherwise the [O x I] tensor
 * eps_dev is injected (parity mode) and kept as self.e. */
int vbnn_layer_sample(vbnn_layer* layer, int sample_idx, const float* eps_dev);
/* VBLinear:clamp_to_map()  VBLinear.lua:105-107 */
int vbnn_layer_clamp_to_map(vbnn_layer* layer);

/* nn.Linear:updateOutput(input)  (inherited; invoked via mlp.lua:77).  Y_dev [N x O].
 * In VBNN_REPARAM_LOCAL mode zeta_dev ([N x O], nullable) injects the activation noise. */
int vbnn_layer_forward(vbnn_layer* layer, const float* X_dev, int N, float* Y_dev,
                       const float* zeta_dev);
/* nn.Linear:updateGradInput(input, gradOutput)  (inherited; via mlp.lua:79).  dX_dev [N x I]. */
int vbnn_layer_backward_data(vbnn_layer* layer, const float* X_dev, const float* G_dev, int N,
                             float* dX_dev);
/* VBLinear:accGradParameters(input, gradOutput, scale)  VBLinear.lua:112-118
 * (one GEMM, not the reference's two -- quirk Q2 -- with the same result). */
int vbnn_layer_acc_grad(vbnn_layer* layer, const float* X_dev, const float* G_dev, int N,
                        float scale);
/* VBLinear:resetAcc() VBLinear.lua:120-122 plus gradParameters:zero() (mlp.lua:63) */
int vbnn_layer_reset_acc(vbnn_layer* layer);

/* VBLinear:compute_prior()  VBLinear.lua:77-88 -> mu_hat, var_hat (host scalars, synchronises); under a
 * non-empirical prior see vbnn_layer_set_prior */
int vbnn_layer_compute_prior(vbnn_layer* layer, float* mu_hat, float* var_hat);
/* VBLinear:compute_mugrads / compute_vargrads  VBLinear.lua:90-98.  Each out pointer is a
 * nullable [O x I] device buffer: mleg/vleg likelihood terms, mlcg/vlcg complexity terms.
 * Like the reference this divides gradWeight / gradSum in place. */
int vbnn_layer_grads(vbnn_layer* layer, float* mleg_dev, float* mlcg_dev, float* vleg_dev,
                     float* vlcg_dev);
/* VBLinear:update(opt)  VBLinear.lua:124-166.  stats (nullable) receives the 14 diagnostics
 * of VBLinear.lua:150-163 and synchronises; NULL keeps the call asynchronous. */
int vbnn_layer_update(vbnn_layer* layer, vbnn_stats* stats);
/* VBLinear:calc_lc(opt)  VBLinear.lua:99-103.  lc_dev: nullable [O x I]; sum_host: nullable. */
int vbnn_layer_calc_lc(vbnn_layer* layer, float* lc_dev, float* sum_host);

/* Choose the prior of the KL terms (enum vbnn_prior; a new layer is VBNN_PRIOR_EMPIRICAL).  Per weight, divided by
 * B, the KL gradient w.r.t. mu is (mu - mu_hat) / var_hat (VBLinear.lua:91), the one w.r.t. log sigma^2 is
 * (sigma^2 / var_hat - 1) / 2 (:96-97), and calc_lc is 1/2 log var_hat - 1/2 log sigma^2 + ((mu - mu_hat)^2 +
 * sigma^2 - var_hat) / (2 var_hat) (:100-101); only where mu_hat and var_hat come from changes.
 *   - It changes the KL terms of every update path -- vbnn_layer_update, vbnn_mlp_update, vbnn_mlp_step,
 *     vbnn_mlp_step_grad_input, vbnn_mlp_backward_update, vbnn_mlp_submit_host* -- and of vbnn_layer_grads,
 *     vbnn_layer_calc_lc and vbnn_mlp_calc_lc.  The likelihood terms, the loss and the noise are unchanged.
 *   - mu0 / var0 are read for VBNN_PRIOR_FIXED only.
 *   - VBNN_PRIOR_PER_WEIGHT initialises the prior arrays with a copy of the layer's current means and lvars (the
 *     continual-learning step: the posterior becomes the next prior).  At that moment both KL gradients are exactly
 *     0 for any finite log-variance, and so is calc_lc from the log-variances.  Afterwards the arrays are ordinary
 *     buffers (vbnn_layer_get / _set / _device_ptr with VBNN_BUF_PRIOR_MEANS / _LVARS, which return VBNN_E_STATE
 *     under any other kind); an edit takes effect at the next update.  They are allocated by the first PER_WEIGHT
 *     call and kept until vbnn_layer_destroy, so a pointer from vbnn_layer_device_ptr stays valid across kind
 *     changes.  In peer mode each rank keeps its own copy: edit it on every rank (the same rule holds for the
 *     values of vbnn_layer_set_opts / vbnn_mlp_set_opts).
 *   - FIXED and PER_WEIGHT compute the KL terms from log var_hat (FIXED: log var0) without a division: they are
 *     finite wherever the exact value is representable in fp32 (for log var_hat >= -177), and the mean term is
 *     exactly 0 where mu == mu_hat.
 *   - vbnn_layer_compute_prior returns (mu0, var0) for FIXED and NaN for PER_WEIGHT, where there is no scalar
 *     prior; the var_hat diagnostic of vbnn_stats follows the same rule.  With strict_reference the mu_sqe cache
 *     keeps its reference meaning (mu - mu_hat)^2, with the prior mean.
 *   - Every update keeps writing the partial sums of the empirical var_hat, so switching back to
 *     VBNN_PRIOR_EMPIRICAL needs no extra pass and gives the reference's prior again.
 *   - Stream-ordered on the context's stream: a PER_WEIGHT snapshot sees the posterior left by everything enqueued
 *     before it, host-pipeline minibatches still in flight included.
 *   - A layer of a vbnn_mlp: each of the net's step graphs re-captures once at its next use after this call.
 *     Editing the PER_WEIGHT arrays needs no re-capture.
 * VBNN_E_INVALID: a plain nn.Linear layer, an unknown kind, or FIXED with a non-finite mu0 or a var0 that is not
 * finite and > 0.  VBNN_E_STATE: the layer's net has an open split step (vbnn_mlp_forward_train); or, in peer mode
 * with PER_WEIGHT, rows owned by other ranks are stale -- run the vbnn_mlp_sync_replicas protocol first so that
 * every rank snapshots the same posterior. */
int vbnn_layer_set_prior(vbnn_layer* layer, int kind, float mu0, float var0);
/* the current kind; mu0 / var0 (nullable) receive FIXED's scalars, NaN under the other kinds */
int vbnn_layer_get_prior(const vbnn_layer* layer, int* kind, float* mu0, float* var0);

/* Learning-rate schedules and KL annealing: the reference reads opt.B and its optimiser tables (learningRate, beta1,
 * beta2, epsilon) at every update (VBLinear.lua:31-33,90-103,125-143), so a Torch7 user decays a rate or anneals the KL
 * weight 1/B by writing them between minibatches.  The idiom here is get, modify, set.
 *   - Live fields: B, lr_bias, lr_mu, lr_var, adam_beta1, adam_beta2, adam_eps.  B must be finite and > 0, each rate
 *     finite and >= 0, each beta in [0, 1), adam_eps finite and > 0.  Every other field (var_init, msr_init, mu_init,
 *     S, reparam, precision, strict_reference) must equal the layer's current value: they size buffers, choose
 *     kernels or only matter at creation.  Otherwise VBNN_E_INVALID, naming the field.  A refused call changes
 *     nothing; vbnn_mlp_set_opts checks every layer before it writes any.
 *   - A new value applies to every update enqueued on the context's stream after the call -- vbnn_layer_update,
 *     vbnn_mlp_update, vbnn_mlp_step, vbnn_mlp_step_grad_input, vbnn_mlp_backward_update, vbnn_mlp_submit_host*,
 *     the peer-mode shard updates -- and to vbnn_layer_grads, vbnn_layer_calc_lc and vbnn_mlp_calc_lc.  lr_bias is
 *     the SGD rate of the biases and of a plain nn.Linear output layer; Adam applies lr * sqrt(1 - beta2^t) /
 *     (1 - beta1^t) with the current values and the layer's own t, as optim.adam does.
 *   - The values live in a small device block per layer that the update kernels read, written by one launch on the
 *     context's stream (counted by vbnn_mlp_launch_count).  No step graph is re-captured or dropped
 *     (vbnn_mlp_graph_captures does not move), and the call does not synchronise.
 *   - Accepted at any time outside stream capture, also while a vbnn_mlp_forward_train step is open: that step's
 *     vbnn_mlp_backward_update then uses the new values.  While the context's stream is being captured:
 *     VBNN_E_STATE (the host copy would disagree with the graph).
 *   - vbnn_layer_get_opts returns the last values set, whether or not the device has reached the write yet.
 *   - vbnn_layer_set_opts on a layer borrowed from a net gives that layer its own values (per-layer optimiser
 *     tables in Torch7); vbnn_mlp_set_opts sets every layer of the net and replaces the net's own copy.
 *   - Peer mode: the context's stream first waits for the library's side stream (as vbnn_mlp_join_streams does), so
 *     the previous minibatch's shard update still reads the old values.  Each rank keeps its own copy: set the same
 *     values on every rank.  NCCL mode needs nothing extra.
 * NULL arguments: VBNN_E_INVALID. */
int vbnn_layer_get_opts(const vbnn_layer* layer, vbnn_opts* out);
int vbnn_layer_set_opts(vbnn_layer* layer, const vbnn_opts* opts);
int vbnn_mlp_set_opts(vbnn_mlp* mlp, const vbnn_opts* opts);   /* every layer of the net */

/* parameters() / field access (mlp.lua:37,48-49; main.lua:123; checkpointing utils.lua:73-80) */
int vbnn_layer_get(vbnn_layer* layer, int which, float* dst_host);
int vbnn_layer_set(vbnn_layer* layer, int which, const float* src_host);
int vbnn_layer_device_ptr(vbnn_layer* layer, int which, float** ptr_dev, size_t* count);
/* Adopt CALLER-OWNED device storage for weight / bias / gradWeight / gradBias (which = VBNN_BUF_WEIGHT,
 * _BIAS, _GRAD_WEIGHT, _GRAD_BIAS): Torch7's getParameters() (mlp.lua:37) re-flattens these four tensors
 * of every module into one new storage, so the module must follow them there instead of the other way
 * round.  The caller's buffer is adopted AS IS (Torch copies the old values into the flat storage itself,
 * and mlp.lua:48-54 then rewrites weight / bias there: the tensor is the parameter) and must stay valid until
 * the next bind or vbnn_layer_destroy; ptr_dev == NULL hands the buffer back to the library (contents kept).
 * Layers owned by a vbnn_mlp keep their gradients in the mlp's arena and refuse. */
int vbnn_layer_bind(vbnn_layer* layer, int which, float* ptr_dev);
/* optimiser step counters (meanState.t / varState.t / biasState.evalCounter) */
int vbnn_layer_get_t(vbnn_layer* layer, int* t);
int vbnn_layer_set_t(vbnn_layer* layer, int t);
/* signal-to-noise pruning mask of mainviz.lua:20-24: counts |mu|/sigma < thresh */
int vbnn_layer_snr_count(vbnn_layer* layer, float thresh, uint8_t* mask_dev, long long* count);

/* draw the exact epsilon [O x I] (or, for local reparameterisation, zeta [N x O] with
 * rows = N) that the fused kernels generate for (step, sample_idx) -- parity tests inject it
 * into the CPU oracle. */
int vbnn_layer_draw_noise(vbnn_layer* layer, uint32_t step, int sample_idx, int rows,
                          int row0, float* out_dev);

/* ---------------------------------------------------------------- mlp.lua -------------
 * MLP:buildModel(opt)  mlp.lua:7-60.  sizes = {input_size, hidden..., #classes}; hidden layers
 * are VBLinear+ReLU, the last is nn.Linear (mlp.lua:29) or, with vb_output, a VBLinear
 * (convnet.lua:30).  Ends in LogSoftMax + ClassNLLCriterion (mlp.lua:30-32). */
int vbnn_mlp_create(vbnn_ctx* ctx, const int* sizes, int n_sizes, int vb_output, int max_batch,
                    const vbnn_opts* opts, vbnn_mlp** out);
int vbnn_mlp_destroy(vbnn_mlp* mlp);
int vbnn_mlp_num_layers(const vbnn_mlp* mlp);
int vbnn_mlp_layer(vbnn_mlp* mlp, int k, vbnn_layer** out);   /* borrowed handle */
/* parameter init on the device: means per VBLinear.lua:22-29, Linear weights ~ N(0, 2/fan_in)
 * and zero biases per mlp.lua:47-55 */
int vbnn_mlp_init_params(vbnn_mlp* mlp, uint64_t seed, int he_means);

/* the step pieces, same names and order as mlp.lua / main.lua:28-40 */
int vbnn_mlp_reset_gradients(vbnn_mlp* mlp);                               /* mlp.lua:62-67  */
int vbnn_mlp_sample(vbnn_mlp* mlp, int sample_idx);                        /* mlp.lua:69-74  */
int vbnn_mlp_run(vbnn_mlp* mlp, const float* X_dev, const float* targets_dev, int N,
                 int sample_idx, float* err_host, float* acc_host);        /* mlp.lua:76-84  */
int vbnn_mlp_update(vbnn_mlp* mlp);                                        /* mlp.lua:117-142 */
int vbnn_mlp_calc_lc(vbnn_mlp* mlp, float* lc_host);                       /* mlp.lua:109-115 */

/* One whole minibatch of main.lua:28-40 (reset, S x (sample, run), [allreduce], update) as one
 * enqueued sequence (CUDA graph when the shape repeats).  result_dev: nullable device float[2]
 * = {mean error, mean accuracy %} as main.lua:38-39.
 * Targets: a target outside 1..C (0 or C+1, e.g. a padding row) adds 0 to the error, is never counted correct and
 * gives its row the gradient softmax(Y) * scale with no -1 term; the mean still divides by N.  The predicted class is
 * the lowest index among tied maximal logits, as in vbnn_mlp_predict. */
int vbnn_mlp_step(vbnn_mlp* mlp, const float* X_dev, const float* targets_dev, int N,
                  float* result_dev);
/* vbnn_mlp_step that also returns the gradient with respect to its input, so that the net can train as the head of
 * a feature extractor (convnet.lua:23-33, whose model:backward sends the head's gradInput into the conv stack once
 * per MC sample: mlp.lua:76-84 driven by main.lua:32-37).
 * The function does exactly what vbnn_mlp_step does: it runs the same kernels on the same data and leaves the same
 * parameters, Adam state, gradients, result and step counter, bit for bit.  It also OVERWRITES dX_dev, a dense
 * fp32 [N x I0] device buffer that must be non-NULL, with
 *     dX = sum_{s < S} d l_s / dX
 * where l_s is the size-averaged ClassNLL of MC sample s over the GLOBAL batch (gradient scale 1 / (N * nranks), as
 * for the parameter gradients).  The derivative is taken through this minibatch's sampled weights (weight mode) or
 * its zeta (local reparameterisation, pathwise: G mu + 2 X .* (H sigma^2)), with the parameters BEFORE this
 * minibatch's update.  This is what Torch7 accumulates into the extractor over main.lua:32-37, so feats:backward(dX)
 * afterwards gives the extractor the reference's gradients; like the parameter gradients (quirk Q3) nothing is
 * divided by S.
 * Data parallel: each rank receives the rows it stepped, and the result is the derivative of the GLOBAL mean loss.
 * A torch DDP extractor, which averages its gradients over ranks, must therefore scale dX by nranks (or sum its
 * gradients instead of averaging them).
 * The minibatch is replayed as its own CUDA graph, keyed on (N, dX_dev): reusing one buffer captures once, and
 * vbnn_mlp_step's graph is never re-captured because of this call (nor the other way round). */
int vbnn_mlp_step_grad_input(vbnn_mlp* mlp, const float* X_dev, const float* targets_dev, int N,
                             float* result_dev, float* dX_dev);
/* The fused minibatch under ANY loss, in two halves around the caller's criterion (mlp.lua:30-32 builds the criterion
 * as a separate, swappable object: nn.MSECriterion, a soft-label or a user criterion instead of ClassNLL).
 *
 * vbnn_mlp_forward_train: the first half of vbnn_mlp_step without its loss.  Stages X_dev [N x I0], samples, and
 * runs the forward of the S samples at the current step (the noise indices of vbnn_mlp_step), writing the output
 * layer's pre-LogSoftMax outputs Y_s into logits_dev, a dense fp32 [S x N x C] device buffer (sample slowest,
 * 16-byte aligned).  Opens a step on the net.
 *
 * vbnn_mlp_backward_update: the second half.  grad_dev is a dense fp32 [S x N x C] device buffer holding dL/dY_s,
 * where L = sum_s l_s.  Runs the backward, [the data-parallel exchange], the KL + Adam update and the step-counter
 * bump exactly as vbnn_mlp_step does after its loss.  dX_dev (nullable) is overwritten with dL/dX [N x I0] as in
 * vbnn_mlp_step_grad_input.  Closes the step, also when it fails.
 *
 * Gradient convention: vbnn_mlp_step is the special case grad_dev[s] = d l_s / dY_s with l_s the mean over the
 * GLOBAL batch of ClassNLL(LogSoftMax(Y_s)).  The S samples are summed as in vbnn_mlp_step: gradWeight is divided by
 * S in the VB update, gradBias and the plain nn.Linear output layer are not (quirk Q3); nothing is rescaled.  In
 * data-parallel runs each rank passes its rows of the gradient of the global loss, so a mean divides by
 * N * nranks, as vbnn_mlp_step does.
 *
 * Ordering: both calls enqueue on the context's stream and neither synchronises.  The caller's loss must run on that
 * stream or be ordered against it with events (the Python Context makes its stream torch's current stream).
 *
 * Open step: while it is open every vbnn_mlp_* entry point that enqueues work returns VBNN_E_STATE, a second
 * vbnn_mlp_forward_train included; only vbnn_mlp_backward_update and vbnn_mlp_reset_gradients are accepted.
 * vbnn_mlp_forward_train is refused while the host pipeline (vbnn_mlp_submit_host*) has minibatches not collected.
 * vbnn_mlp_reset_gradients abandons an open step: no update, and the step counter does not move.  In peer mode it
 * refuses (the forward half has already advanced the peers' flag protocol): pass zeros to vbnn_mlp_backward_update
 * instead, which drops this minibatch's likelihood term and still applies the KL update.
 * vbnn_mlp_get_outputs returns VBNN_E_STATE after vbnn_mlp_forward_train until the next step, test or predict: this
 * minibatch's outputs are in the caller's buffer.
 *
 * Each half is replayed as its own CUDA graph where vbnn_mlp_step would be: the forward keyed on (N, logits_dev),
 * the backward on (N, grad_dev, dX_dev), with and without dX_dev in graphs of their own (each runs eagerly once
 * before it is captured, and alternating the two never re-captures).  Neither re-captures the graphs of vbnn_mlp_step or
 * vbnn_mlp_step_grad_input.  NULL X_dev / logits_dev / grad_dev and N outside 1..max_batch: VBNN_E_INVALID. */
int vbnn_mlp_forward_train(vbnn_mlp* mlp, const float* X_dev, int N, float* logits_dev);
int vbnn_mlp_backward_update(vbnn_mlp* mlp, const float* grad_dev, float* dX_dev);
/* same with HOST buffers: H2D of inputs + D2H of {error, accuracy} inside the call
 * (replaces inputs:cuda()/targets:cuda() main.lua:23-24 and the scalar reads mlp.lua:80-82). */
int vbnn_mlp_step_host(vbnn_mlp* mlp, const float* X_host, const float* targets_host, int N,
                       float* err_host, float* acc_host);
/* pipelined host-buffer variant: submit copies minibatch t+1 while minibatch t computes;
 * collect returns the {error, accuracy} of the oldest submitted minibatch. */
int vbnn_mlp_submit_host(vbnn_mlp* mlp, const float* X_host, const float* targets_host, int N);
int vbnn_mlp_collect(vbnn_mlp* mlp, float* err_host, float* acc_host);
/* The same pipeline fed with the dataset's NATIVE bytes: MNIST pixels are uint8 before data.lua:25,30
 * (u.normalize, utils.lua:29-35) turns them into (x - mean) / std floats on the host.  Here the bytes cross
 * PCIe (4x fewer than fp32) and the normalisation is fused into the operand-staging kernel on the device:
 * x = (float(byte) - mean) * inv_std, then exactly the path of vbnn_mlp_submit_host. */
int vbnn_mlp_submit_host_u8(vbnn_mlp* mlp, const uint8_t* X_host, const float* targets_host, int N,
                            float mean, float inv_std);
/* Make the context's stream wait for everything a minibatch enqueued on the library's auxiliary streams (the
 * peer-mode side stream: last shard update + operand push; the NCCL stream), so that an event recorded on the
 * context's stream afterwards covers the WHOLE minibatch.  Asynchronous; a no-op on one GPU. */
int vbnn_mlp_join_streams(vbnn_mlp* mlp);

/* net:test(input, target)  mlp.lua:86-107: n_samples == 0 -> clamp_to_map (quicktest),
 * else mean over n_samples sampled forward passes (no wasted backward). */
int vbnn_mlp_test(vbnn_mlp* mlp, const float* X_dev, const float* targets_dev, int N,
                  int n_samples, float* err_host, float* acc_host);
/* Bayesian model average over n_samples sampled forward passes (no backward, no parameter change): the
 * predictive distribution p-bar(c|x) = (1/T) sum_t softmax(f_t(x)) and its split of uncertainty.
 * vbnn_mlp_test keeps the reference's semantics (it averages the error and accuracy SCALARS of the T passes);
 * this is the average of the probabilities.
 * n_samples == 0: one MAP pass (clamp_to_map, as quicktest).  Samples use the same noise indices as
 * vbnn_mlp_test ((1 << 20) + t at the current step), so test and predict at one step see the same weights;
 * the step counter and every optimiser counter stay as they are.
 * X_dev [N x I0], N <= max_batch.  targets_dev: nullable 1-based [N]; needed when nll_host or acc_host is given.
 * logp_dev:  nullable [N x C]  log p-bar(c|x) = logsumexp_t logp_t(c|x) - log T
 * unc_dev:   nullable [N x 4]  {H[p-bar], mean_t H[p_t], max(H[p-bar] - mean_t H[p_t], 0), argmax_c p-bar (1-based)}
 *            = total, aleatoric and epistemic (mutual information, "BALD") uncertainty, predicted class
 * nll_host / acc_host: nullable; mean -log p-bar(target) and % argmax p-bar == target; synchronises only if given.
 * Targets outside 1..C add 0 to the NLL and never count as correct (as the training loss does).
 * In VBNN_REPARAM_LOCAL mode the activation noise zeta of a row depends on its row index within the call, so a
 * row's prediction depends on where it sits in X_dev.  Two calls at the same step give bit-identical outputs.
 * Afterwards vbnn_mlp_get_outputs(s) and VBNN_BUF_WEIGHT hold sample s of the LAST chunk of S samples, as after
 * vbnn_mlp_test.  In peer mode the preconditions are those of vbnn_mlp_test.  Profile class 8 ("predict") times
 * the averaging kernel; its flops slot holds 20 algorithmic bytes per (row, class, sample). */
int vbnn_mlp_predict(vbnn_mlp* mlp, const float* X_dev, int N, int n_samples, const float* targets_dev,
                     float* logp_dev, float* unc_dev, float* nll_host, float* acc_host);
/* How vbnn_mlp_predict_outputs reads the net's C raw outputs f_t(x) (no LogSoftMax anywhere). */
enum vbnn_output_model {
  VBNN_OUTPUT_RAW = 0,      /* K = C outputs m_t = f_t(x) themselves                                        */
  VBNN_OUTPUT_GAUSSIAN = 1  /* C = 2K: columns [0,K) are means m_t, [K,2K) log-variances s_t of a
                               heteroscedastic Gaussian likelihood (torch: gaussian_nll_loss(Y[..., :K],
                               y, Y[..., K:].exp()))                                                     */
};
/* Model average of the RAW outputs over n_samples sampled forward passes, for regression heads: the predictive
 * mean and the split of its variance into epistemic (weight posterior) and aleatoric (heteroscedastic head) parts.
 * Sampling is that of vbnn_mlp_predict: the same noise indices ((1 << 20) + t at the current step), the same chunks of
 * S samples, no backward, no parameter, optimiser-state or step-counter change, the same LRT caveat (a row's zeta
 * depends on its row index within the call) and the same peer-mode preconditions.  n_samples == 0: one MAP pass
 * (clamp_to_map), and T = 1 below.  Otherwise T = n_samples.
 * X_dev [N x I0], 1 <= N <= max_batch.  K = C (RAW) or C / 2 (GAUSSIAN; an odd C is VBNN_E_INVALID).
 * Every output is nullable:
 *   samples_dev   [T x N x C] dense fp32, sample slowest, 16-byte aligned: every sampled raw output, stored there by
 *                 the output layer's epilogue (no extra copy)
 *   mean_dev      [N x K] (1/T) sum_t m_t
 *   epistemic_dev [N x K] (1/T) sum_t (m_t - mean)^2: the population variance over samples, exactly 0 at T = 1 and for
 *                 MAP.  Formed from sums of deviations from the first sample, so it does not cancel when |mean| is
 *                 large against the spread.
 *   aleatoric_dev [N x K] (1/T) sum_t exp(s_t), GAUSSIAN only; +inf where exp(s) overflows fp32 (s > ~88.7).
 *                 The predictive variance of the mixture is epistemic + aleatoric.
 * targets_dev: dense fp32 [N x K] regression targets y (not 1-based labels); needed when nll_host or rmse_host is given.
 *   rmse_host  sqrt(mean over N*K of (y - mean)^2)
 *   nll_host   GAUSSIAN only: -(1/N) sum_n log p-bar(y_n | x_n), log p-bar = logsumexp_t sum_k log N(y_nk; m_tnk,
 *              e^{s_tnk}) - log T: the full density (with 1/2 log 2 pi per output) of the joint per-row mixture, not a
 *              product of per-column mixtures.  log N = -1/2 (log 2 pi + s + (y - m)^2 e^{-s}) is formed in the log
 *              domain with the product taken as 0 where y == m, so nll is finite wherever its value is, s = +-100
 *              included.
 * Either scalar synchronises only if asked for; both are sums of per-block partials added on the host in a fixed
 * order (no atomics): two calls at the same step give bit-identical results, and the result does not depend on S.
 * VBNN_E_INVALID: NULL net or X_dev, N outside 1..max_batch, n_samples < 0, an unknown output_model, aleatoric_dev or
 * nll_host under RAW, nll_host or rmse_host without targets_dev, an unaligned samples_dev.  VBNN_E_STATE while a
 * vbnn_mlp_forward_train step is open.  The first call allocates the kernel's state and cannot be captured.
 * Afterwards vbnn_mlp_get_outputs(s) returns sample s of the last chunk, as after vbnn_mlp_predict, unless
 * samples_dev was given: then it returns VBNN_E_STATE until the next step, test or predict (the outputs are in the
 * caller's buffer, as after vbnn_mlp_forward_train).  Profile class 8 ("predict") times the moments kernel. */
int vbnn_mlp_predict_outputs(vbnn_mlp* mlp, const float* X_dev, int N, int n_samples, int output_model,
                             const float* targets_dev, float* samples_dev, float* mean_dev,
                             float* epistemic_dev, float* aleatoric_dev, float* nll_host, float* rmse_host);
/* last forward's LogSoftMax output [N x C] (self.model.output, visualize.lua:97) */
int vbnn_mlp_get_outputs(vbnn_mlp* mlp, int sample_idx, float* logp_host);
/* kernels launched by this handle since creation (bench.py's gpu_launches) */
int vbnn_mlp_launch_count(vbnn_mlp* mlp, long long* count);
/* CUDA graphs this handle has captured since creation, over all its step graphs (vbnn_mlp_step,
 * vbnn_mlp_step_grad_input and the two halves of the split step): a caller that keeps its buffers and N fixed sees it
 * stop growing after the second call of each entry point */
int vbnn_mlp_graph_captures(vbnn_mlp* mlp, long long* count);
/* flat gradient arena {gW, gS, gb per layer}: what the data-parallel allreduce sums */
int vbnn_mlp_grad_arena(vbnn_mlp* mlp, float** ptr_dev, size_t* count);

/* ---------------------------------------------------------------- data parallel -------
 * New functionality (the reference is single-GPU, SURVEY.md section 2.2): one rank per GPU,
 * minibatch rows sharded, sum-allreduce of the gradient arena over NCCL/NVLink. */
int vbnn_comm_unique_id(void* id128);                       /* 128-byte ncclUniqueId       */
int vbnn_comm_init(vbnn_ctx* ctx, const void* id128, int rank, int nranks);
int vbnn_comm_destroy(vbnn_ctx* ctx);
int vbnn_comm_allreduce(vbnn_ctx* ctx, float* buf_dev, size_t count);

/* Peer mode: the same exchange without any collective call, fused into the hot path over NVLink
 * peer memory (CUDA IPC; one process per GPU of one box).  Rows [q*rpo, (q+1)*rpo) of every layer
 * belong to rank q: the dW GEMM epilogue stores each gradient tile straight into its owner's
 * receive slot (reduce-scatter), the owner's fused update sums the slots for its rows only, and
 * the copy engines push the refreshed operands to every rank (all-gather) while backward
 * continues.  Set-up: after vbnn_comm_init, every rank exports a blob (blob == NULL queries its
 * size), the host all-gathers the blobs (rank order, blob_len bytes each) and every rank imports
 * them.  vbnn_mlp_step / vbnn_mlp_submit_host then use the peer path. */
int vbnn_mlp_peer_export(vbnn_mlp* mlp, void* blob, size_t capacity, size_t* blob_len);
int vbnn_mlp_peer_import(vbnn_mlp* mlp, const void* blobs_all_ranks, size_t blob_len);
int vbnn_mlp_peer_active(const vbnn_mlp* mlp);
/* collective: refresh the fp32 state of rows owned by other ranks (Adam moments, and whatever training does
 * not push) before get / checkpoint / clamp_to_map.  Protocol, on EVERY rank: drain the device
 * (cudaDeviceSynchronize: the last minibatch's shard updates run on the library's side stream) -> host barrier
 * -> vbnn_mlp_sync_replicas -> host barrier.  A rank that pulls before its peer has drained reads rows one
 * optimiser step behind. */
int vbnn_mlp_sync_replicas(vbnn_mlp* mlp);
/* shard of an O-row matrix owned by `rank`; returns rows per owner (a multiple of 32) */
int vbnn_peer_shard(int O, int nranks, int rank, int* row0, int* rows);

/* ---------------------------------------------------------------- self-test hooks -----
 * Raw GEMM entry used by tests/profiling to exercise the tcgen05 kernel in isolation:
 * D[M x N] (fp32) = A * B with bf16 operands. a_kmajor: A is [M x K] row-major (1) or
 * [K x M] row-major (0); b_kmajor: B is [N x K] row-major (1) or [K x N] row-major (0). */
int vbnn_gemm_bf16(vbnn_ctx* ctx, const uint16_t* A_dev, int lda, int a_kmajor,
                   const uint16_t* B_dev, int ldb, int b_kmajor, float* D_dev, int ldd,
                   int M, int N, int K, int batch, long long strideA, long long strideB,
                   long long strideD);
int vbnn_philox_normal(vbnn_ctx* ctx, uint64_t seed, uint32_t step, uint32_t stream,
                       uint32_t sample, int rows, int cols, int row0, float* out_dev);
/* Experiment switches (csrc/knobs.h: "tc_bn", "tc_cg", "lrt_split", "dw_split", "no_graph", ...; the same
 * names upper-cased with a VBNN_ prefix are read from the environment once per process).  The parity
 * tests use this to force the CTA-pair 256 x 256 tiles / a GEMM form at oracle-sized problems.
 * value == INT_MIN restores the default; old_value is nullable.  Unknown name: VBNN_E_INVALID. */
int vbnn_debug_knob(const char* name, int value, int* old_value);

#ifdef __cplusplus
}
#endif
#endif /* VBNN_H */
