-- vbnn_ffi.lua -- LuaJIT FFI declarations of libvbnn.so (include/vbnn.h), the part the shim uses.
-- NOT EXECUTED IN THIS REPO'S CI: the build image and the GPU box have no Lua/LuaJIT/Torch7
-- (SURVEY.md section 8c).  The same ABI is exercised through Python ctypes (vbnn_b200/_lib.py)
-- and the tests in tests/; this file is the binding a VBNN maintainer would drop in.
local ffi = require 'ffi'

ffi.cdef[[
typedef struct vbnn_ctx vbnn_ctx;
typedef struct vbnn_layer vbnn_layer;
typedef struct vbnn_opts {
  float var_init; int msr_init; float mu_init; float B; int S;
  float lr_bias, lr_mu, lr_var; float adam_beta1, adam_beta2, adam_eps;
  int reparam; int precision; int strict_reference;
} vbnn_opts;
typedef struct vbnn_stats {
  float vlc_grad, vle_grad, mlc_grad, mle_grad, min_variance, max_variance, mean_variance, var_hat;
  float mean_means, std_means, min_means, max_means, mu_normratio, var_normratio;
} vbnn_stats;
const char* vbnn_last_error(void);
void vbnn_opts_default(vbnn_opts*);
int vbnn_ctx_create_ex(int device, void* stream, int stream_mode, uint64_t seed, vbnn_ctx** out);
int vbnn_ctx_destroy(vbnn_ctx*);
int vbnn_layer_create(vbnn_ctx*, int inputSize, int outputSize, int kind, const vbnn_opts*, vbnn_layer** out);
int vbnn_layer_destroy(vbnn_layer*);
int vbnn_layer_sample(vbnn_layer*, int sample_idx, const float* eps_dev);
int vbnn_layer_clamp_to_map(vbnn_layer*);
int vbnn_layer_forward(vbnn_layer*, const float* X_dev, int N, float* Y_dev, const float* zeta_dev);
int vbnn_layer_backward_data(vbnn_layer*, const float* X_dev, const float* G_dev, int N, float* dX_dev);
int vbnn_layer_acc_grad(vbnn_layer*, const float* X_dev, const float* G_dev, int N, float scale);
int vbnn_layer_reset_acc(vbnn_layer*);
int vbnn_layer_compute_prior(vbnn_layer*, float* mu_hat, float* var_hat);
int vbnn_layer_grads(vbnn_layer*, float* mleg, float* mlcg, float* vleg, float* vlcg);
int vbnn_layer_update(vbnn_layer*, vbnn_stats*);
int vbnn_layer_calc_lc(vbnn_layer*, float* lc_dev, float* sum_host);
int vbnn_layer_set_prior(vbnn_layer*, int kind, float mu0, float var0);
int vbnn_layer_get_prior(const vbnn_layer*, int* kind, float* mu0, float* var0);
int vbnn_layer_get_opts(const vbnn_layer*, vbnn_opts* out);
int vbnn_layer_set_opts(vbnn_layer*, const vbnn_opts*);
int vbnn_layer_device_ptr(vbnn_layer*, int which, float** ptr_dev, size_t* count);
int vbnn_layer_bind(vbnn_layer*, int which, float* ptr_dev);
/* net level (lua/mlp.lua): the mlp.lua object and the main.lua:19-51 closure */
typedef struct vbnn_mlp vbnn_mlp;
int vbnn_mlp_create(vbnn_ctx*, const int* sizes, int n_sizes, int vb_output, int max_batch, const vbnn_opts*, vbnn_mlp** out);
int vbnn_mlp_destroy(vbnn_mlp*);
int vbnn_mlp_num_layers(const vbnn_mlp*);
int vbnn_mlp_layer(vbnn_mlp*, int k, vbnn_layer** out);
int vbnn_mlp_init_params(vbnn_mlp*, uint64_t seed, int he_means);
int vbnn_mlp_reset_gradients(vbnn_mlp*);
int vbnn_mlp_sample(vbnn_mlp*, int sample_idx);
int vbnn_mlp_run(vbnn_mlp*, const float* X_dev, const float* targets_dev, int N, int sample_idx, float* err_host, float* acc_host);
int vbnn_mlp_update(vbnn_mlp*);
int vbnn_mlp_calc_lc(vbnn_mlp*, float* lc_host);
int vbnn_mlp_set_opts(vbnn_mlp*, const vbnn_opts*);
int vbnn_mlp_step(vbnn_mlp*, const float* X_dev, const float* targets_dev, int N, float* result_dev);
int vbnn_mlp_step_grad_input(vbnn_mlp*, const float* X_dev, const float* targets_dev, int N, float* result_dev, float* dX_dev);
int vbnn_mlp_forward_train(vbnn_mlp*, const float* X_dev, int N, float* logits_dev);
int vbnn_mlp_backward_update(vbnn_mlp*, const float* grad_dev, float* dX_dev);
int vbnn_mlp_submit_host(vbnn_mlp*, const float* X_host, const float* targets_host, int N);
int vbnn_mlp_collect(vbnn_mlp*, float* err_host, float* acc_host);
int vbnn_mlp_test(vbnn_mlp*, const float* X_dev, const float* targets_dev, int N, int n_samples, float* err_host, float* acc_host);
int vbnn_mlp_predict(vbnn_mlp*, const float* X_dev, int N, int n_samples, const float* targets_dev, float* logp_dev, float* unc_dev, float* nll_host, float* acc_host);
int vbnn_mlp_predict_outputs(vbnn_mlp*, const float* X_dev, int N, int n_samples, int output_model, const float* targets_dev, float* samples_dev, float* mean_dev, float* epistemic_dev, float* aleatoric_dev, float* nll_host, float* rmse_host);
/* data parallel: NCCL id, then (optionally) the peer-memory exchange */
int vbnn_comm_unique_id(void* id128);
int vbnn_comm_init(vbnn_ctx*, const void* id128, int rank, int nranks);
int vbnn_mlp_peer_export(vbnn_mlp*, void* blob, size_t capacity, size_t* blob_len);
int vbnn_mlp_peer_import(vbnn_mlp*, const void* blobs_all_ranks, size_t blob_len);
int vbnn_mlp_sync_replicas(vbnn_mlp*);
]]

local C = ffi.load('vbnn')

local M = { C = C, ffi = ffi }

function M.check(rc)
   if rc ~= 0 then error('libvbnn: ' .. ffi.string(C.vbnn_last_error()), 2) end
end

-- stream modes: the enum of include/vbnn.h next to vbnn_ctx_create_ex
M.STREAM_GIVEN, M.STREAM_LEGACY_DEFAULT, M.STREAM_PRIVATE_BLOCKING = 0, 1, 2

-- cutorch's CURRENT stream, the one nn.ReLU / nn.LogSoftMax / the criterion (mlp.lua:19,27,30,32) enqueue on:
-- THCState_getCurrentStream(cutorch.getState()) from libTHC.  cutorch's default stream -- and the only
-- stream of the early-2015 cutorch the reference was written against -- is CUDA's legacy default stream
-- (stream 0, a NULL cudaStream_t): the library is then told so explicitly, because a NULL `stream` alone
-- would mean "give me a private stream", which does not synchronise with stream 0.
local function cutorch_stream()
   local ok, s = pcall(function()
      ffi.cdef[[ typedef struct THCState THCState; void* THCState_getCurrentStream(THCState* state); ]]
      local THC = ffi.load('THC')
      return THC.THCState_getCurrentStream(ffi.cast('THCState*', cutorch.getState()))
   end)
   if ok and s ~= nil then return s end
   return nil                                   -- stream 0 (or a cutorch without streams)
end

-- one context per process, on cutorch's current device and stream.
-- layer level (lua/VBLinear.lua; default): the library runs ON cutorch's stream -- stream 0 itself when that is the
--   current one -- so every call is ordered with the neighbouring cunn modules like one of them;
-- net level (lua/mlp.lua passes net_level = true): the whole minibatch is inside the library, which then wants CUDA graph
--   replay; stream 0 cannot be captured, so it takes a private BLOCKING stream, which still synchronises implicitly with
--   stream 0 (inputs:cuda() before, scalar reads after).
function M.context(seed, net_level)
   if not M.ctx then
      local out = ffi.new('vbnn_ctx*[1]')
      local dev = cutorch.getDevice() - 1
      local stream = cutorch_stream()
      if stream ~= nil then
         M.check(C.vbnn_ctx_create_ex(dev, stream, M.STREAM_GIVEN, seed or 3, out))
      elseif net_level then
         M.check(C.vbnn_ctx_create_ex(dev, nil, M.STREAM_PRIVATE_BLOCKING, seed or 3, out))
      else
         M.check(C.vbnn_ctx_create_ex(dev, nil, M.STREAM_LEGACY_DEFAULT, seed or 3, out))
      end
      M.ctx = ffi.gc(out[0], C.vbnn_ctx_destroy)
   end
   return M.ctx
end

-- config.lua's table mapped as vbnn_b200/config.py maps it, at creation and by setOpt.  The fields the reference reads at
-- every update: opt.B, opt.state / meanState / varState learningRate, and meanState's beta1 / beta2 / epsilon (optim.adam's
-- 0.9, 0.999, 1e-8 where absent).  setOpt passes the whole table, so the library refuses a change of anything else (S,
-- reparam, precision, ...) instead of ignoring it.
function M.opts(opt)
   local o = ffi.new('vbnn_opts')
   C.vbnn_opts_default(o)
   o.var_init = opt.var_init; o.msr_init = opt.msr_init and 1 or 0; o.mu_init = opt.mu_init
   o.B = opt.B; o.S = opt.S
   o.lr_bias = opt.state.learningRate; o.lr_mu = opt.meanState.learningRate; o.lr_var = opt.varState.learningRate
   o.adam_beta1 = opt.meanState.beta1 or 0.9
   o.adam_beta2 = opt.meanState.beta2 or 0.999
   o.adam_eps = opt.meanState.epsilon or 1e-8
   o.reparam = (opt.reparam == 'local') and 1 or 0
   o.precision = (opt.precision == 'bf16') and 1 or 0
   o.strict_reference = (opt.strict_reference == false) and 0 or 1
   return o
end

-- raw device pointer of a contiguous CudaTensor: cutorch's FFI accessor tensor:data() returns a float* to
-- the first element (storage data + storageOffset), on the device
function M.ptr(t)
   assert(t:isContiguous(), 'libvbnn needs contiguous tensors')
   return ffi.cast('float*', t:data())
end

return M
