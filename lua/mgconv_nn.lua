--[[ mgconv_nn.lua -- Torch7 nn.Module on top of libmgconv's plan-level C ABI (LuaJIT FFI).

   nn.MGStage is the drop-in for the module graph mgConv() assembles in the reference's model files:

     residual (models/ilsvrc/rnmg.lua:91-159; cifar/rnmg.lua:102-173; cifar/prnmg.lua:122-193)
        ReLU( BN( mg( ReLU( BN( mg(x) ) ) ) ) + Shortcut(x) )        per grid, Shortcut = Identity / nn.Padding(1, nOP-nIP, 3)
     plain    (models/cifar/nmg.lua:31-86)
        ReLU( BN( mg(x) ) )

   with mg(x)_i = conv_k( JoinTable(2){ MaxPool2x2ceil(x_{i-1}), x_i, UpSampleNearest2(x_{i+1}) } ).

   input  : Lua table of 4-D CudaTensors (NCHW), finest grid first      -- what ResampleConcat receives (rnmg.lua:41-89)
   output : Lua table of 4-D CudaTensors (NCHW), same structure; gradInput likewise.
   Parameters are ordinary Torch tensors in Torch's layout -- weight [nOP][nIP_cat][k][k] with input planes ordered
   finer | same | coarser, bias [nOP]; BatchNorm weight / bias / running_mean / running_var [nOP] -- so getParameters(),
   optim.sgd, torch.save and the init code keyed on field names work unchanged.  Raw device pointers are fetched on EVERY
   call (getParameters() re-homes the tensors, pipelines/standard/train.lua:115).  The shim's state (plan handle, workspace
   CudaTensor) is built lazily for the input sizes at hand and dropped by clearState(); it is never serialised.

   The whole stage is two C calls, mg_stage_forward / mg_stage_backward (include/mgconv.h): segment lists, pooled
   companions, fused epilogues and gradient routing live behind them (csrc/stage.cu), so nothing of the Python host
   (mgconv/lower.py, ops.py, sched.py) has to exist in Lua.  tests/cabi_unit.c makes the same calls from plain C and is
   checked against the oracle on the GPU (tests/test_cabi.py).

   NOT EXECUTED HERE: there is no LuaJIT / Torch7 in the build container nor on the GPU box (`which luajit th lua`: nothing).
]]
local mg = require 'mgconv_ffi'
local ffi, C = mg.ffi, mg.C

ffi.cdef[[ void* THCState_getCurrentStream(void* state); ]]   -- cutorch: the stream Torch's own kernels are enqueued on

-- one mg_ctx per (GPU, Lua state): DataParallelTable runs one Lua state per GPU (multigpu.lua:94-98)
local contexts = {}
local function context(precision)
   local dev = cutorch.getDevice()
   local key = dev .. ':' .. precision
   if not contexts[key] then
      contexts[key] = mg.ctx(dev - 1, nil, precision == 'fp32' and C.MG_F32 or C.MG_BF16)
   end
   local ctx = contexts[key]
   mg.check(ctx, C.mg_ctx_set_stream(ctx, ffi.C.THCState_getCurrentStream(cutorch._state)))   -- order with neighbouring Torch ops
   return ctx
end

local MGStage, parent = torch.class('nn.MGStage', 'nn.Module')

--- nIPs / nOPs: channel tables per grid (finest first); kernels: 3 or 1 per grid; residual: boolean
function MGStage:__init(nIPs, nOPs, kernels, residual, eps, precision)
   parent.__init(self)
   assert(#nIPs == #nOPs and #nIPs == #kernels, '#nInputPlanes is not consistent with #nOutputPlanes')   -- rnmg.lua:99-102
   assert(#nIPs <= 4, 'at most 4 grids per stage')
   self.nIPs, self.nOPs, self.kernels = nIPs, nOPs, kernels
   self.residual = residual and true or false
   self.eps, self.momentum, self.precision = eps or 1e-5, 0.1, precision or 'bf16'
   self.train = true
   local n, L = #nIPs, self.residual and 2 or 1
   self.convs, self.bns = {}, {}          -- index (l-1)*n + i, the order of mg_stage_params
   for l = 1, L do
      for i = 1, n do
         local cin = function(j) return l == 1 and nIPs[j] or nOPs[j] end
         local ccat = cin(i) + (i > 1 and cin(i - 1) or 0) + (i < n and cin(i + 1) or 0)
         local k = kernels[i]
         local conv = { weight = torch.Tensor(nOPs[i], ccat, k, k), bias = torch.Tensor(nOPs[i]),
                        gradWeight = torch.Tensor(nOPs[i], ccat, k, k):zero(), gradBias = torch.Tensor(nOPs[i]):zero(),
                        kW = k, kH = k, nInputPlane = ccat, nOutputPlane = nOPs[i] }
         local bn = { weight = torch.Tensor(nOPs[i]), bias = torch.Tensor(nOPs[i]):zero(),
                      gradWeight = torch.Tensor(nOPs[i]):zero(), gradBias = torch.Tensor(nOPs[i]):zero(),
                      running_mean = torch.zeros(nOPs[i]), running_var = torch.ones(nOPs[i]) }
         self.convs[#self.convs + 1] = conv
         self.bns[#self.bns + 1] = bn
      end
   end
   self:reset()
end

-- ConvInit / BNInit of models/ilsvrc/rnmg.lua:288-300: a module of a new type is invisible to model:findModules('cudnn.Spatial-
-- Convolution'), so it initialises itself the way the model file would have
function MGStage:reset()
   for _, c in ipairs(self.convs) do
      c.weight:normal(0, math.sqrt(2 / (c.kW * c.kH * c.nOutputPlane)))
      c.bias:zero()
   end
   for _, b in ipairs(self.bns) do
      b.weight:fill(1); b.bias:zero(); b.running_mean:zero(); b.running_var:fill(1)
   end
end

function MGStage:parameters()
   local w, gw = {}, {}
   for k = 1, #self.convs do
      local c, b = self.convs[k], self.bns[k]
      w[#w + 1] = c.weight;  gw[#gw + 1] = c.gradWeight
      w[#w + 1] = c.bias;    gw[#gw + 1] = c.gradBias
      w[#w + 1] = b.weight;  gw[#gw + 1] = b.gradWeight
      w[#w + 1] = b.bias;    gw[#gw + 1] = b.gradBias
   end
   return w, gw
end

function MGStage:type(t, cache)   -- :cuda() / :float(): move every tensor of the sub-tables too
   for _, tbl in ipairs{self.convs, self.bns} do
      for _, m in ipairs(tbl) do
         for name, v in pairs(m) do
            if torch.isTensor(v) then m[name] = v:type(t) end
         end
      end
   end
   self:clearState()
   return parent.type(self, t, cache)
end

local function fptr(t) return ffi.cast('float*', t:data()) end

-- plan + workspace for the sizes of `input` (rebuilt when the batch or the image size changes, e.g. the partial last batch of
-- pipelines/standard/test.lua:40-44)
function MGStage:_state(input)
   local n = #self.nIPs
   assert(#input == n, string.format('nn.MGStage: %d input grids for a %d-grid stage', #input, n))
   local key = {}
   for i = 1, n do
      assert(input[i]:dim() == 4 and input[i]:size(2) == self.nIPs[i], 'nn.MGStage: grid ' .. i .. ' must be N x ' .. self.nIPs[i] .. ' x H x W')
      key[i] = table.concat(input[i]:size():totable(), 'x')
   end
   key = table.concat(key, '|')
   if self._key ~= key then
      local ctx = context(self.precision)
      local d = ffi.new('mg_stage_desc')
      d.n_scales = n
      for i = 1, n do
         d.C_in[i - 1], d.C_out[i - 1] = self.nIPs[i], self.nOPs[i]
         d.H[i - 1], d.W[i - 1], d.ksize[i - 1] = input[i]:size(3), input[i]:size(4), self.kernels[i]
      end
      d.residual, d.no_final_relu, d.eps, d.momentum = self.residual and 1 or 0, 0, self.eps, self.momentum
      local out = ffi.new('mg_stage_plan*[1]')
      mg.check(ctx, C.mg_plan_create(ctx, d, input[1]:size(1), out))   -- MG_ERR_SHAPE here = the size error JoinTable(2) would raise
      self._plan = ffi.gc(out[0], C.mg_plan_destroy)
      local bytes = tonumber(C.mg_plan_workspace_bytes(self._plan))
      self._ws = torch.CudaTensor(math.ceil(bytes / 4) + 64)           -- owned by Torch, like every tensor the host can see
      self._key = key
      self.output, self.gradInput = {}, {}
      for i = 1, n do
         self.output[i] = torch.CudaTensor(input[i]:size(1), self.nOPs[i], input[i]:size(3), input[i]:size(4))
         self.gradInput[i] = torch.CudaTensor():resizeAs(input[i])
      end
   end
   -- 256-byte aligned view of the workspace
   local base = ffi.cast('uintptr_t', self._ws:data())
   local aligned = ffi.cast('void*', bit.band(base + 255, bit.bnot(255ULL)))
   return context(self.precision), aligned
end

function MGStage:_params()
   local p = ffi.new('mg_stage_params')
   for k = 1, #self.convs do
      local c, b = self.convs[k], self.bns[k]
      p.conv_w[k - 1], p.conv_b[k - 1], p.conv_gw[k - 1], p.conv_gb[k - 1] = fptr(c.weight), fptr(c.bias), fptr(c.gradWeight), fptr(c.gradBias)
      p.bn_g[k - 1], p.bn_b[k - 1], p.bn_gg[k - 1], p.bn_gb[k - 1] = fptr(b.weight), fptr(b.bias), fptr(b.gradWeight), fptr(b.gradBias)
      p.bn_rm[k - 1], p.bn_rv[k - 1] = fptr(b.running_mean), fptr(b.running_var)
   end
   return p
end

local function ptr_array(tensors, n)
   local a = ffi.new('float*[4]')
   for i = 1, n do a[i - 1] = tensors[i] and fptr(tensors[i]) or nil end
   return a
end

function MGStage:updateOutput(input)
   local ctx, ws = self:_state(input)
   local n = #self.nIPs
   local x = {}
   for i = 1, n do x[i] = input[i]:contiguous() end
   mg.check(ctx, C.mg_stage_forward(self._plan, ws, ffi.cast('const float* const*', ptr_array(x, n)), self:_params(),
                                    ptr_array(self.output, n), self.train and 1 or 0))
   return self.output
end

-- nn.Module:backward = updateGradInput + accGradParameters; the stage computes both in one call
function MGStage:backward(input, gradOutput, scale)
   local ctx, ws = self:_state(input)
   local n = #self.nIPs
   local dy = {}
   for i = 1, n do dy[i] = gradOutput[i]:contiguous() end
   mg.check(ctx, C.mg_stage_backward(self._plan, ws, ffi.cast('const float* const*', ptr_array(dy, n)), self:_params(),
                                     ptr_array(self.gradInput, n), scale or 1))
   return self.gradInput
end

-- the two halves on their own (nngraph's gModule, hand-written loops, input-gradient tools): updateGradInput computes gradInput
-- and launches no weight-gradient kernel; accGradParameters adds scale * the parameter gradients of the gradOutput given to the
-- last updateGradInput (what that call left in the workspace: gradOutput itself is not read again).  Calling accGradParameters
-- without an updateGradInput since the last updateOutput is an error.
function MGStage:updateGradInput(input, gradOutput)
   local ctx, ws = self:_state(input)
   local n = #self.nIPs
   local dy = {}
   for i = 1, n do dy[i] = gradOutput[i]:contiguous() end
   mg.check(ctx, C.mg_stage_update_grad_input(self._plan, ws, ffi.cast('const float* const*', ptr_array(dy, n)), self:_params(),
                                              ptr_array(self.gradInput, n)))
   return self.gradInput
end

function MGStage:accGradParameters(input, gradOutput, scale)
   local ctx, ws = self:_state(input)
   mg.check(ctx, C.mg_stage_acc_grad_parameters(self._plan, ws, self:_params(), scale or 1))
end

function MGStage:zeroGradParameters()
   for k = 1, #self.convs do
      self.convs[k].gradWeight:zero(); self.convs[k].gradBias:zero()
      self.bns[k].gradWeight:zero(); self.bns[k].gradBias:zero()
   end
end

function MGStage:training() self.train = true; return self end
function MGStage:evaluate() self.train = false; return self end

function MGStage:clearState()
   self._plan, self._ws, self._key = nil, nil, nil    -- plans / workspaces are rebuilt lazily; never serialised
   self.output, self.gradInput = {}, {}
   return self
end

function MGStage:__tostring__()
   return string.format('nn.MGStage(%s -> %s, %s)', table.concat(self.nIPs, ','), table.concat(self.nOPs, ','), self.residual and 'residual' or 'plain')
end

-- ------------------------------------------------------------------------------------------------------------
-- builder helper with the reference's signature (models/ilsvrc/rnmg.lua:91): a model file rebinds its local `mgConv`
local M = {}
function M.mgConv(nInputPlanes, nOutputPlanes, kernels)
   return nn.MGStage(nInputPlanes, nOutputPlanes, kernels, true, 1e-5)
end
function M.plain_mgConv(nInputPlanes, nOutputPlanes, kernels)      -- models/cifar/nmg.lua:31 (BN eps 1e-3)
   return nn.MGStage(nInputPlanes, nOutputPlanes, kernels, false, 1e-3)
end
return M
