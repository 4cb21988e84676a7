-- VBLinear.lua -- drop-in replacement of the reference's VBLinear.lua: the same Torch7
-- nn.Module API (torch.class 'nn.VBLinear' < 'nn.Linear', reference VBLinear.lua:7), every method
-- a thin call into libvbnn.so.  mu / log sigma^2 / Adam state live in device buffers owned by
-- the library (`means`, `lvars`, `gradSum` are exposed as CudaTensor views on them); `weight`, `bias`,
-- `gradWeight`, `gradBias` stay Torch's own tensors -- created by nn.Linear's constructor, moved by
-- model:cuda() (mlp.lua:34), re-flattened by getParameters() (mlp.lua:37) -- and the library adopts their
-- storage (vbnn_layer_bind), so mlp.lua and main.lua run unmodified.  The context runs on cutorch's
-- current stream (stream 0 unless the caller changed it), like every cunn module.
--
-- NOT EXECUTED IN THIS REPO (no Lua/Torch7 in the image); the Python mirror
-- vbnn_b200/vblinear.py makes the same calls in the same order and is what the tests drive.
require 'cunn'
local V = require 'vbnn_ffi'
local ffi, C = V.ffi, V.C

local VBLinear, parent = torch.class('nn.VBLinear', 'nn.Linear')

local BUF = { MEANS = 0, LVARS = 1, BIAS = 2, WEIGHT = 3, GRAD_WEIGHT = 4, GRAD_SUM = 5, GRAD_BIAS = 6 }

-- wrap a library-owned device buffer as a CudaTensor view (no copy)
local function view(self, which, ...)
   local p, n = ffi.new('float*[1]'), ffi.new('size_t[1]')
   V.check(C.vbnn_layer_device_ptr(self.h, which, p, n))
   local s = torch.CudaStorage(tonumber(n[0]), tonumber(ffi.cast('intptr_t', p[0])))
   return torch.CudaTensor(s, 1, torch.LongStorage{...})
end

function VBLinear:__init(inputSize, outputSize, opt)                 -- reference VBLinear.lua:9-47
   parent.__init(self, inputSize, outputSize)                        -- :10  nn.Linear: weight, bias, gradWeight, gradBias
   self.opt = opt
   self.bias:zero()                                                  -- :13
   local out = ffi.new('vbnn_layer*[1]')
   V.check(C.vbnn_layer_create(V.context(), inputSize, outputSize, 0, V.opts(opt), out))
   self.h = ffi.gc(out[0], C.vbnn_layer_destroy)
   self.W = outputSize * inputSize
   -- library-owned state, exposed as CudaTensor views (main.lua:123 reads lvars; torch.save sees them)
   self.means = view(self, BUF.MEANS, outputSize, inputSize)
   self.lvars = view(self, BUF.LVARS, outputSize, inputSize)
   self.gradSum = view(self, BUF.GRAD_SUM, outputSize, inputSize)
   -- weight / bias / gradWeight / gradBias stay ORDINARY Torch tensors of the usual shapes in every mode, so the
   -- unmodified mlp.lua:34 (model:cuda()), :37 (getParameters() re-flattens exactly these four) and :48-54
   -- (weight:size(2), weight:copy, bias:zero) work; the library follows them (vbnn_layer_bind) wherever Torch
   -- puts them.  In bf16 / local-reparameterisation mode the sampled weights exist only as tensor-core
   -- operands, so `weight` is then just Torch's tensor (the compute never reads it).
   self.has_weight = (opt.precision ~= 'bf16') and (opt.reparam ~= 'local')
   self.bound = {}
   self.s = 0
   self:compute_prior()                                              -- :46
end

-- Follow the four nn.Linear tensors to wherever Torch moved them.  Called at the top of every method that
-- touches them; a pointer comparison per tensor when nothing moved.
function VBLinear:bind()
   if torch.type(self.bias) ~= 'torch.CudaTensor' then
      error('nn.VBLinear (libvbnn) needs model:cuda() (mlp.lua:34) before use: there is no CPU path')
   end
   local function follow(which, t)
      local p = V.ptr(t)
      if self.bound[which] ~= p then
         V.check(C.vbnn_layer_bind(self.h, which, p))
         self.bound[which] = p
      end
   end
   if self.has_weight then follow(BUF.WEIGHT, self.weight) end
   follow(BUF.BIAS, self.bias)
   follow(BUF.GRAD_WEIGHT, self.gradWeight)
   follow(BUF.GRAD_BIAS, self.gradBias)
end

-- model:cuda() / :float() (nn.Module:type) converts every tensor field of the module; the library-owned views
-- must not be converted (they ARE device memory), only the four nn.Linear tensors and output / gradInput
function VBLinear:type(type)
   assert(type == 'torch.CudaTensor', 'nn.VBLinear (libvbnn) is CUDA-only')
   for _, k in ipairs{'weight', 'bias', 'gradWeight', 'gradBias', 'output', 'gradInput'} do
      self[k] = self[k]:type(type)
   end
   return self
end

function VBLinear:sample(opt)                                        -- :49-64 (epsilon drawn on the device)
   self:bind()
   V.check(C.vbnn_layer_sample(self.h, self.s, nil))
   self.s = self.s + 1
end

function VBLinear:updateOutput(input)                                -- nn.Linear:updateOutput
   self:bind()
   local n = input:dim() == 1 and 1 or input:size(1)
   self.output:resize(n, self.bias:size(1))
   V.check(C.vbnn_layer_forward(self.h, V.ptr(input), n, V.ptr(self.output), nil))
   return self.output
end

function VBLinear:updateGradInput(input, gradOutput)                 -- nn.Linear:updateGradInput
   self:bind()
   local n = input:dim() == 1 and 1 or input:size(1)
   self.gradInput:resizeAs(input)
   V.check(C.vbnn_layer_backward_data(self.h, V.ptr(input), V.ptr(gradOutput), n, V.ptr(self.gradInput)))
   return self.gradInput
end

function VBLinear:accGradParameters(input, gradOutput, scale)        -- :112-118, one GEMM instead of two
   self:bind()
   local n = input:dim() == 1 and 1 or input:size(1)
   V.check(C.vbnn_layer_acc_grad(self.h, V.ptr(input), V.ptr(gradOutput), n, scale or 1))
end

function VBLinear:resetAcc()                                         -- :120-122
   self:bind()
   V.check(C.vbnn_layer_reset_acc(self.h))
   self.s = 0
end

function VBLinear:compute_prior()                                    -- :77-88
   local mu, var = ffi.new('float[1]'), ffi.new('float[1]')
   V.check(C.vbnn_layer_compute_prior(self.h, mu, var))
   self.mu_hat, self.var_hat = mu[0], var[0]
   return self.mu_hat, self.var_hat
end

function VBLinear:compute_mugrads(opt)                               -- :90-93
   local leg, lcg = self.means:clone(), self.means:clone()
   V.check(C.vbnn_layer_grads(self.h, V.ptr(leg), V.ptr(lcg), nil, nil))
   return leg, lcg
end

function VBLinear:compute_vargrads(opt)                              -- :95-98
   local leg, lcg = self.lvars:clone(), self.lvars:clone()
   V.check(C.vbnn_layer_grads(self.h, nil, nil, V.ptr(leg), V.ptr(lcg)))
   return leg, lcg
end

function VBLinear:calc_lc(opt)                                       -- :99-103
   local lc = self.means:clone()
   V.check(C.vbnn_layer_calc_lc(self.h, V.ptr(lc), nil))
   return lc
end

-- The prior of the KL terms (vbnn_layer_set_prior): 'empirical' (the reference's, the default), 'fixed'
-- N(mean, var) or 'per_weight' (this layer's current posterior becomes its prior)
local PRIOR = { empirical = 0, fixed = 1, per_weight = 2 }
function VBLinear:set_prior(kind, mean, var)
   assert(PRIOR[kind], "set_prior: kind must be 'empirical', 'fixed' or 'per_weight'")
   V.check(C.vbnn_layer_set_prior(self.h, PRIOR[kind], mean or 0, var or 0))
end

-- Learning-rate schedules and KL annealing (vbnn_layer_set_opts): the reference reads opt.B and its optimiser tables at
-- every update, so decay a rate or anneal opt.B, then call setOpt(opt) before the next minibatch
function VBLinear:setOpt(opt)
   V.check(C.vbnn_layer_set_opts(self.h, V.opts(opt)))
end

function VBLinear:clamp_to_map()                                     -- :105-107
   self:bind()
   V.check(C.vbnn_layer_clamp_to_map(self.h))
end

local STAT = { 'vlc grad', 'vle grad', 'mlc grad', 'mle grad', 'min variance', 'max variance', 'mean variance',
               'var hat', 'mean means', 'std means', 'min. means', 'max. means', 'mu normratio', 'var normratio' }

function VBLinear:update(opt)                                        -- :124-166
   self:bind()
   if opt.log then
      local st = ffi.new('vbnn_stats')
      V.check(C.vbnn_layer_update(self.h, st))
      local f = ffi.cast('float*', st)
      for i, id in ipairs(STAT) do Log:add(id, f[i - 1]) end          -- :150-163
   else
      V.check(C.vbnn_layer_update(self.h, nil))
   end
end
