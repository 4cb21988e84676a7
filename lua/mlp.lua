-- mlp.lua -- drop-in replacement of the reference's mlp.lua net object (reference mlp.lua:5-143) on top of
-- libvbnn.so's net-level entry points: the same duck-typed interface main.lua drives
--   MLP:buildModel(opt), :resetGradients(), :sample(), :run(inputs, targets), :test(input, target),
--   :calc_lc(opt), :update(opt)
-- plus :predict(input, nsamples, target), the Bayesian model average with per-row uncertainty,
-- :predict_outputs(input, nsamples, model, target), the same over the raw outputs of a regression head,
-- and :train_minibatch(inputs, targets), the whole closure of main.lua:19-51 as ONE call that keeps the
-- minibatch, the sampled weights and the noise on the GPU, and :train_minibatch_grad(inputs, targets, gradInput),
-- the same on device tensors that also returns the gradient for a feature extractor below the net, and
-- :forward_train(inputs) / :backward_update(gradLogits, gradInput), the same minibatch split around ANY criterion.
--
-- NOT EXECUTED IN THIS REPO (no Lua/Torch7 in the image); vbnn_b200/mlp.py makes the same calls in the
-- same order and is what tests/ and bench.py drive.
local V = require 'vbnn_ffi'
local ffi, C = V.ffi, V.C

local MLP = {}
MLP.__index = MLP

function MLP:buildModel(opt)                                          -- reference mlp.lua:7-60
   local net = setmetatable({}, MLP)
   net.opt = opt
   local sizes = { opt.input_size }
   for _, h in ipairs(opt.hidden) do sizes[#sizes + 1] = h end
   -- a regression net (opt.criterion 'mse' or 'gaussian_nll') may give its output width as opt.outputs
   local crit = opt.criterion or 'class_nll'
   sizes[#sizes + 1] = (crit ~= 'class_nll' and opt.outputs) or #opt.classes
   local csizes = ffi.new('int[?]', #sizes, sizes)
   local out = ffi.new('vbnn_mlp*[1]')
   -- hidden layers: VBLinear + ReLU; output: plain nn.Linear + LogSoftMax (mlp.lua:29-30), or a VBLinear with
   -- opt.vb_output (the convnet.lua:30 head)
   V.check(C.vbnn_mlp_create(V.context(opt.seed, true), csizes, #sizes, opt.vb_output and 1 or 0, opt.batchSize,
                             V.opts(opt), out))
   net.h = ffi.gc(out[0], C.vbnn_mlp_destroy)
   V.check(C.vbnn_mlp_init_params(net.h, opt.param_seed or 4, opt.msr_init and 1 or 0))     -- mlp.lua:47-55
   net.s = 0
   net.err, net.acc = ffi.new('float[1]'), ffi.new('float[1]')
   assert(opt.prior == nil or opt.prior == 'empirical' or opt.prior == 'fixed',
          "opt.prior must be 'empirical' or 'fixed'")
   if opt.prior == 'fixed' then net:set_prior('fixed', opt.prior_mean, opt.prior_var) end
   net.C = sizes[#sizes]
   net:set_criterion(crit)
   return net
end

-- The criterion of the fused minibatch (vbnn_mlp_set_criterion), the swap of mlp.lua:30-32's criterion object:
-- 'class_nll' (LogSoftMax + ClassNLL), 'mse' (nn.MSECriterion, targets [N x C]) or 'gaussian_nll' (C = 2K outputs:
-- K means, K log-variances; targets [N x K]).  Under a regression criterion run / test / train_minibatch return
-- (mean loss, MSE of the means) instead of (error, accuracy %).
local CRITERION = { class_nll = 0, mse = 1, gaussian_nll = 2 }
function MLP:set_criterion(name)
   assert(CRITERION[name], "set_criterion: 'class_nll', 'mse' or 'gaussian_nll'")
   V.check(C.vbnn_mlp_set_criterion(self.h, CRITERION[name]))
   self.criterion = name
end

-- VBLinear:set_prior on every VB layer of the net (the hidden layers and a vb_output layer)
local PRIOR = { empirical = 0, fixed = 1, per_weight = 2 }
function MLP:set_prior(kind, mean, var)
   assert(PRIOR[kind], "set_prior: kind must be 'empirical', 'fixed' or 'per_weight'")
   local n = C.vbnn_mlp_num_layers(self.h)
   local layer = ffi.new('vbnn_layer*[1]')
   for k = 0, n - 1 do
      if k < n - 1 or self.opt.vb_output then
         V.check(C.vbnn_mlp_layer(self.h, k, layer))
         V.check(C.vbnn_layer_set_prior(layer[0], PRIOR[kind], mean or 0, var or 0))
      end
   end
end

-- VBLinear:setOpt on every layer of the net in one call (vbnn_mlp_set_opts); no step graph is re-captured
function MLP:setOpt(opt)
   V.check(C.vbnn_mlp_set_opts(self.h, V.opts(opt)))
   self.opt = opt
end

function MLP:resetGradients()                                         -- mlp.lua:62-67
   self.s = 0
   V.check(C.vbnn_mlp_reset_gradients(self.h))
end

function MLP:sample()                                                 -- mlp.lua:69-74 (epsilon drawn on the device)
   V.check(C.vbnn_mlp_sample(self.h, self.s))
   self.s = self.s + 1
end

function MLP:run(inputs, targets)                                     -- mlp.lua:76-84; inputs/targets: CudaTensors
   local n = inputs:size(1)
   V.check(C.vbnn_mlp_run(self.h, V.ptr(inputs), V.ptr(targets), n, self.s - 1, self.err, self.acc))
   return self.err[0], self.acc[0]
end

function MLP:test(input, target)                                      -- mlp.lua:86-107
   local samples = self.opt.quicktest and 0 or self.opt.testSamples
   V.check(C.vbnn_mlp_test(self.h, V.ptr(input), V.ptr(target), input:size(1), samples, self.err, self.acc))
   return self.err[0], self.acc[0]
end

-- Bayesian model average over nsamples sampled forward passes (default: test's count, 0 = one MAP pass under
-- quicktest).  input / target: CudaTensors, target optional.  Returns logp [N x C] = log p-bar, unc [N x 4] =
-- {H[p-bar], mean_t H[p_t], mutual information, 1-based argmax} as CudaTensors, then nll and accuracy (nil
-- without a target).  :test keeps the reference's averaged-scalar semantics; this averages the probabilities.
function MLP:predict(input, nsamples, target)
   local n = input:size(1)
   if nsamples == nil then nsamples = self.opt.quicktest and 0 or self.opt.testSamples end
   local logp = torch.CudaTensor(n, self.C)
   local unc = torch.CudaTensor(n, 4)
   if target then
      V.check(C.vbnn_mlp_predict(self.h, V.ptr(input), n, nsamples, V.ptr(target), V.ptr(logp), V.ptr(unc),
                                 self.err, self.acc))
      return logp, unc, self.err[0], self.acc[0]
   end
   V.check(C.vbnn_mlp_predict(self.h, V.ptr(input), n, nsamples, nil, V.ptr(logp), V.ptr(unc), nil, nil))
   return logp, unc
end

-- Model average of the RAW outputs for a regression head (vbnn_mlp_predict_outputs): model 'raw' (K = C outputs) or
-- 'gaussian' (C = 2K: means, then log-variances).  Returns mean and epistemic variance [n x K], the aleatoric variance
-- under 'gaussian' (else nil), and with a target [n x K] the mixture NLL ('gaussian', else nil) and the RMSE.
function MLP:predict_outputs(input, nsamples, model, target)
   local n = input:size(1)
   if nsamples == nil then nsamples = self.opt.quicktest and 0 or self.opt.testSamples end
   local gaussian = model == 'gaussian'
   local k = gaussian and self.C / 2 or self.C
   local mean, epi = torch.CudaTensor(n, k), torch.CudaTensor(n, k)
   local ale = gaussian and torch.CudaTensor(n, k) or nil
   local nll = (gaussian and target) and ffi.new('float[1]') or nil
   local rmse = target and ffi.new('float[1]') or nil
   V.check(C.vbnn_mlp_predict_outputs(self.h, V.ptr(input), n, nsamples, gaussian and 1 or 0,
                                      target and V.ptr(target) or nil, nil, V.ptr(mean), V.ptr(epi),
                                      ale and V.ptr(ale) or nil, nll, rmse))
   return mean, epi, ale, nll and nll[0] or nil, rmse and rmse[0] or nil
end

function MLP:calc_lc(opt)                                             -- mlp.lua:109-115
   local lc = ffi.new('float[1]')
   V.check(C.vbnn_mlp_calc_lc(self.h, lc))
   return lc[0]
end

function MLP:update(opt)                                              -- mlp.lua:117-142
   V.check(C.vbnn_mlp_update(self.h))
end

-- main.lua:28-40 in one enqueue: reset, S x (sample, run), update.  inputs / targets are HOST FloatTensors
-- (pinned memory makes the copy asynchronous); returns the mean error and accuracy of main.lua:38-39.  Under a
-- regression criterion (set_criterion) targets are [N x K] and the pair is (mean loss, MSE of the means).
function MLP:train_minibatch(inputs, targets)
   V.check(C.vbnn_mlp_submit_host(self.h, inputs:data(), targets:data(), inputs:size(1)))
   V.check(C.vbnn_mlp_collect(self.h, self.err, self.acc))
   return self.err[0], self.acc[0]
end

-- The same minibatch when the net is the head of a feature extractor (convnet.lua:23-33, with opt.vb_output for its
-- VBLinear output layer): inputs / targets / gradInput are CudaTensors, and gradInput [N x input_size] is OVERWRITTEN
-- with the sum over the S samples of d loss_s / d inputs (the parameters before this minibatch's update), which is
-- what model:backward sends into the extractor over main.lua:32-37:  feats:backward(x, gradInput).
function MLP:train_minibatch_grad(inputs, targets, gradInput)
   local n = inputs:size(1)
   assert(gradInput:isContiguous() and gradInput:size(1) == n and gradInput:size(2) == self.opt.input_size,
          'gradInput must be a contiguous CudaTensor [N x input_size]')
   self.res = self.res or torch.CudaTensor(2)
   V.check(C.vbnn_mlp_step_grad_input(self.h, V.ptr(inputs), V.ptr(targets), n, V.ptr(self.res), V.ptr(gradInput)))
   local r = self.res:float()
   return r[1], r[2]
end

-- The fused minibatch under any nn criterion, in place of the ClassNLL of mlp.lua:78-79:
--   local Y = net:forward_train(inputs)                           -- S x N x C pre-LogSoftMax outputs
--   local err = 0
--   local dY = Y.new():resizeAs(Y)
--   for s = 1, S do err = err + crit:forward(Y[s], t); dY[s]:copy(crit:backward(Y[s], t)) end
--   net:backward_update(dY)                                      -- backward, KL + Adam update, step counter
-- gradLogits is the gradient of the SUM over the S samples of the per-sample loss (mlp.lua:79 accumulates the S
-- backward passes the same way); a size-averaged criterion divides by N as ClassNLL does.  inputs / gradLogits /
-- gradInput are CudaTensors on the library's stream; Y is reused from call to call (the graph is keyed on it), so copy
-- it to keep it.  gradInput (optional, [N x input_size]) is overwritten as in :train_minibatch_grad.
function MLP:forward_train(inputs)
   local n = inputs:size(1)
   assert(inputs:isContiguous() and inputs:size(2) == self.opt.input_size,
          'inputs must be a contiguous CudaTensor [N x input_size]')
   self.logits = self.logits or {}
   local Y = self.logits[n]
   if not Y then
      Y = torch.CudaTensor(self.opt.S, n, self.C)
      self.logits[n] = Y
   end
   V.check(C.vbnn_mlp_forward_train(self.h, V.ptr(inputs), n, V.ptr(Y)))
   self.open_n = n
   return Y
end

function MLP:backward_update(gradLogits, gradInput)
   local n = self.open_n
   assert(n, 'backward_update: call forward_train first')
   assert(gradLogits:isContiguous() and gradLogits:nElement() == self.opt.S * n * self.C,
          'gradLogits must be a contiguous CudaTensor [S x N x C]')
   if gradInput then
      assert(gradInput:isContiguous() and gradInput:size(1) == n and gradInput:size(2) == self.opt.input_size,
             'gradInput must be a contiguous CudaTensor [N x input_size]')
   end
   self.open_n = nil
   V.check(C.vbnn_mlp_backward_update(self.h, V.ptr(gradLogits), gradInput and V.ptr(gradInput) or nil))
end

return MLP
