-- gp_regressor protocol over the C ABI: every method bot7 calls on `bot7.models.gp_regressor`
--   bots/abstract.lua:148                     model:init(X, Y)
--   bots/bayesopt.lua:68,74                   model:sample_hypers(X, Y [, _, _, single])
--   bots/bayesopt.lua:75                      model:parse_hypers(hyp)
--   bots/bayesopt.lua:65                      model:class()
--   scores/expected_improvement.lua:57,63     model:fantasize(n, X0, Y0, Xp, hyp), model:predict(X0, Y0, X1, hyp, req)
--   models/abstract.lua:32-41                 model:cache()
-- The arithmetic (kernels, hyper layout [log l_1..log l_d, log sigma_f, log sigma_n, m], N(0, prior_std^2) prior on
-- every entry, initial values) is the declared spec of oracle/SPEC.md: gpTorch7 is not available (parity unpinned).
-- Same defaults, control flow and guards as the Python twin bot7_b200/models.py, which is what the tests drive.
local B   = require('bot7_b200.ffi')
local ffi = require('ffi')

local kernels = { ardse = B.C.B7_KERNEL_ARDSE, matern52 = B.C.B7_KERNEL_MATERN52, matern_52 = B.C.B7_KERNEL_MATERN52 }
local model, parent = torch.class('bot7_b200.models.gp_regressor', 'bot7.models.abstract')

function model:__init(config)
  parent.__init(self)
  local config = config or {}
  config['kernel']     = config.kernel    or 'ardse'
  config['nzModel']    = config.nzModel   or 'GaussianNoise_iso'
  config['mean']       = config.mean      or 'constant'
  config['sampler']    = config.sampler   or 'slice'
  config['nSamples']   = config.nSamples  or 1
  config['prior_std']  = config.prior_std or 2.0     -- declared: independent N(0, prior_std^2) on every hyp entry
  config['spec_width'] = config.spec_width or 8      -- density evaluations per batched device call
  -- batched density evaluations through sampler_spec.lua: the chain of bot7.samplers.slice from the same generator state,
  -- in fewer device calls (false: the reference sampler, one evaluation per call)
  if config.speculative == nil then config['speculative'] = true end
  -- one device call per slice step through sampler_device.lua (b7_gp_slice_step) for fits of up to 128 observations; the
  -- same chain, larger fits keep the route above
  if config.device_step == nil then config['device_step'] = false end
  -- declared initial state of the chain (model:init); gpTorch7's own values are unknown
  config['init_lengthscale'] = config.init_lengthscale or 0.5
  config['init_sigma_f']     = config.init_sigma_f or 1.0
  self.config = config
  self.hyp    = nil
end

function model:class() return 'gp.models.gp_regressor' end

function model:cache()
  return {config = self.config, hyp = self.hyp}
end

---------------- bots/abstract.lua:148: initial hyper-parameter state from the data
function model:init(X, Y)
  local d = X:size(2)
  local h = torch.zeros(1, d + 3)
  h:narrow(2, 1, d):fill(math.log(self.config.init_lengthscale))
  h[1][d + 1] = math.log(self.config.init_sigma_f)
  h[1][d + 2] = 0.5 * math.log(self.config.init_noise or (self.config.noiseless and 1e-6 or 1e-2))
  h[1][d + 3] = Y:mean()
  self.hyp = h
  return self
end

function model:parse_hypers(h)
  if h:dim() == 1 then return h:view(1, -1) end
  return h
end

-- S x H hyper draws -> device factors (handle freed by the GC); returns handle, logml (S), info (int[S])
function model:fit(X, Y, hyp, flags)
  local X, Y, hyp = X:contiguous():double(), Y:contiguous():double(), self:parse_hypers(hyp):contiguous():double()
  local S, H = hyp:size(1), hyp:size(2)
  local box   = ffi.new('b7_gp*[1]')
  local info  = ffi.new('int[?]', S)
  local logml = torch.DoubleTensor(S)
  local jit   = torch.DoubleTensor(S)
  B.check(B.C.b7_gp_fit(B.context(), kernels[self.config.kernel], X:data(), Y:data(), X:size(1), X:size(2),
                        hyp:data(), S, H, self.config.noiseless and 1 or 0, flags or B.C.B7_FIT_PREDICT,
                        box, info, logml:data(), jit:data()), 'b7_gp_fit')
  for s = 1, S do
    if jit[s] == math.huge then -- utils/math.lua:204-215
      print('Warning: utils.math.chol failed to find a PSD version\nof the input matrix; returning chol(I).')
    elseif jit[s] > 0 then
      print(string.format('Warning: utils.math.chol succeeded in factorizing the\ninput matrix after applying a jitter of %.2e', jit[s]))
    end
  end
  return ffi.gc(box[0], B.C.b7_gp_free), logml, info
end

---------------- scores/expected_improvement.lua:63: {mean=, var=} (M x 1 each) for one hyper-parameter vector
function model:predict(X0, Y0, X1, hyp, req)
  local gp   = self:fit(X0, Y0, hyp or self.hyp)
  local X1   = X1:contiguous():double()
  if X1:dim() == 1 then X1 = X1:view(1, -1) end
  local M    = X1:size(1)
  local mean = torch.DoubleTensor(M, 1)
  local var  = torch.DoubleTensor(M, 1)
  B.check(B.C.b7_gp_predict(gp, 0, X1:data(), M, mean:data(), var:data()), 'b7_gp_predict')
  local req, out = req or {mean = true, var = true}, {}
  if req.mean then out.mean = mean end
  if req.var  then out.var  = var end
  return out
end

---------------- log p(y | h) + log p(h): the density the slice sampler evaluates (samplers/slice.lua:100-103).
-- X and y stay resident between evaluations (b7_gp_refit on one handle of `spec_width` slots); a failed
-- factorisation or a non-finite likelihood is -inf, so the sampler rejects the point.
function model:log_density_batch(H, X, Y, W)
  local H = self:parse_hypers(H):contiguous():double()
  local k = H:size(1)
  local W = W or math.max(self.config.spec_width, 1)           -- slots of the resident handle (one handle per width)
  local sd   = self.config.prior_std
  local out  = torch.DoubleTensor(k)
  local pad  = torch.DoubleTensor(W, H:size(2))
  local info, logml, jit = ffi.new('int[?]', W), torch.DoubleTensor(W), torch.DoubleTensor(W)
  self._density = self._density or {}
  for c0 = 1, k, W do
    local n = math.min(W, k - c0 + 1)
    pad:narrow(1, 1, n):copy(H:narrow(1, c0, n))
    for r = n + 1, W do pad[r]:copy(H[c0 + n - 1]) end       -- short batches repeat their last row
    local slot = self._density[W]
    if slot == nil or slot.X ~= X or slot.Y ~= Y then
      local gp, lm, inf = self:fit(X, Y, pad, B.C.B7_FIT_LOGML_ONLY)
      self._density[W] = {gp = gp, X = X, Y = Y}
      logml:copy(lm); ffi.copy(info, inf, W * ffi.sizeof('int'))
    else
      B.check(B.C.b7_gp_refit(slot.gp, pad:data(), B.C.B7_FIT_LOGML_ONLY, info, logml:data(), jit:data()), 'b7_gp_refit')
    end
    for i = 1, n do
      local lp = logml[i]
      if info[i - 1] ~= 0 or lp ~= lp or lp == math.huge or lp == -math.huge then lp = -math.huge end
      out[c0 + i - 1] = lp - 0.5 * H[c0 + i - 1]:clone():div(sd):pow(2):sum()
    end
  end
  return out
end

-- one evaluation at a time (what bot7.samplers.slice asks for): a handle with a single slot, 2.0 ms at N = 4096
function model:log_density(h, X, Y)
  return self:log_density_batch(self:parse_hypers(h), X, Y, 1)[1]
end

-- one slice step in one device call on the single-slot handle of log_density (X, y resident); Torch7's sequential order for
-- the prior's sum.  Returns {x1, used, evals, logp}, or nil when the shrink uniforms ran out.
function model:device_step(X, Y, x0, dir, log_u, u_right, u_shrink, width, max_step)
  local slot = self._density and self._density[1]
  if slot == nil or slot.X ~= X or slot.Y ~= Y then
    self:log_density(x0, X, Y)
    slot = self._density[1]
  end
  local H = x0:nElement()
  local x1 = torch.DoubleTensor(1, H)
  local used, evals, logp = ffi.new('int[1]'), ffi.new('int[1]'), ffi.new('double[1]')
  local x0c, dirc, urc, usc = x0:contiguous():double(), dir:contiguous():double(), u_right:contiguous():double(), u_shrink:contiguous():double()
  local rc = B.C.b7_gp_slice_step(slot.gp, x0c:data(), dirc:data(), log_u, urc:data(), usc:data(), usc:nElement(), width, max_step,
                                  self.config.prior_std, 0, x1:data(), used, evals, logp)
  if rc == B.C.B7_ERR_STATE then return nil end
  B.check(rc, 'b7_gp_slice_step')
  return {x1 = x1, used = used[0], evals = evals[0], logp = logp[0]}
end

---------------- bots/bayesopt.lua:68,74: slice-sample the hyper-parameter posterior, keep the chain state.
-- bot7.samplers.slice (samplers/slice.lua, unchanged) drives the chain; each f(x) is one density evaluation on the GPU.
function model:sample_hypers(X, Y, _, _, single)
  if self.hyp == nil then self:init(X, Y) end
  local n    = single and 1 or self.config.nSamples
  local dev  = self.config.device_step and self.config.sampler == 'slice' and X:size(1) <= 128
  local spec = not dev and self.config.speculative and self.config.sampler == 'slice'
  local sampler, f
  if dev then
    sampler = require('bot7_b200.sampler_device')()
    f       = function(...) return self:device_step(X, Y, ...) end
  elseif spec then
    sampler = require('bot7_b200.sampler_spec')()
    f       = function(V, args) return self:log_density_batch(V, X, Y) end
  else
    sampler = bot7.samplers[self.config.sampler]()
    f       = function(x, args) return self:log_density(x, X, Y) end
  end
  local out = torch.DoubleTensor(n, self.hyp:nElement())
  local x   = self.hyp:view(1, -1):clone()
  for i = 1, n do
    if dev then
      x = sampler(f, x, {nSamples = 1}, nil)
    elseif spec then
      x = sampler(f, x, {nSamples = 1}, nil, self.config.spec_width)
    else
      x = sampler(f, x, {nSamples = 1}, nil)
    end
    out[i]:copy(x[1])
  end
  self.hyp = out[n]:view(1, -1):clone()
  if single then return out[1]:view(1, -1) end
  return out
end

---------------- scores/expected_improvement.lua:57: Y_pend ~ N(mean, var) at the pending points (independent marginals)
function model:fantasize(n, X0, Y0, Xp, hyp)
  local p = self:predict(X0, Y0, Xp, hyp, {mean = true, var = true})
  local z = torch.randn(p.mean:size(1), n)
  return z:cmul(p.var:sqrt():expand(p.mean:size(1), n)):add(p.mean:expand(p.mean:size(1), n))
end

return model
