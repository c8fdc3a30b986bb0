-- Device slice sampler: the chain of bot7.samplers.slice (samplers/slice.lua:51-168), one device call per step.
--
-- step(x0, dir, log_u, u_right, u_shrink, width, max_step) runs a whole directed slice step on the device (model:device_step =
-- b7_gp_slice_step) and returns {x1 =, used =, evals =, logp =}, or nil when the shrink uniforms ran out.  The generator stays
-- on the host: every step draws what the reference would consume, in its order -- the direction (xDim normals), the slice level,
-- the bracket (xDim uniforms) and `k` shrink uniforms -- then rewinds the generator (torch.getRNGState / setRNGState) to the
-- state after the bracket and draws the shrink uniforms the step used, so for a given generator state the samples are those of
-- samplers/slice.lua, bit for bit.  When the shrink uniforms ran out the step is made again from the same draws with twice as
-- many.  Same algorithm as bot7_b200/samplers.py:slice_device.
require('bot7_b200.ffi')          -- creates the package table bot7_b200.samplers that torch.class stores the class in
local sampler = torch.class('bot7_b200.samplers.slice_device')

function sampler:__init()
  self.calls, self.evals = 0, 0
end

-- samplers/slice.lua:32-48
local function configure(opt)
  local opt = opt or {}
  opt['max_step'] = opt.max_step or 1e3
  opt['nSamples'] = opt.nSamples or 1
  if opt.step_out ~= false then opt['step_out'] = true end
  if opt.logspace ~= false then opt['logspace'] = true end
  return opt
end

function sampler:directed_slice(step, opt, x0, k)
  local xDim  = x0:size(2)
  local width = opt.width or 1.0
  local state = torch.getRNGState()
  local res, after
  while true do
    torch.setRNGState(state)
    local dir = torch.randn(1, xDim)
    dir = dir:div(dir:norm())
    local u = torch.log(torch.rand(1))[1]                       -- :108
    local u_right = torch.rand(1, xDim)                         -- :114
    after = torch.getRNGState()
    res = step(x0, dir, u, u_right, torch.rand(k), width, opt.max_step)
    self.calls = self.calls + 1
    if res then break end
    k = 2 * k
  end
  torch.setRNGState(after)
  if res.used > 0 then torch.rand(res.used) end                 -- the shrink uniforms the step consumed (:136)
  self.evals = self.evals + res.evals
  if res.logp ~= res.logp then print('Error: samplers.slice encountered a NaN') end
  return res.x1
end

-- sampler(step, X0, opt, f_args, k) -> nSamples x dim tensor (samplers/slice.lua:24-28,51-89 without the Gibbs sweep)
function sampler:__call__(step, X0, opt, f_args, k)
  local opt = configure(opt)
  assert(not opt.gibbs and not opt.widths and opt.logspace and opt.step_out,
         'bot7_b200.samplers.slice_device: the log-space directed step with step-out and a scalar width only')
  local X0 = X0:clone():repeatTensor(opt.nSamples, 1)
  local N, xDim = X0:size(1), X0:size(2)
  local samples = torch.Tensor(N, xDim)
  for n = 1, N do
    samples[n] = self:directed_slice(step, opt, X0[{{n}, {}}], math.max(k or 16, 1))
  end
  return samples
end

return sampler
