-- bot7.models.dngo with the hand-off of models/dngo.lua:155-174 routed to the GPU: the network update (trainer,
-- :126-153) and every other method stay the parent's; what changes is how Z1 = basis(X_hid) and
-- predictor:predict(Z0, Y0, Z1, nil, hyp, req) are evaluated for the candidate grid:
--   * the Linear / ReLU / Tanh stack below the basis layer is read out of self.network and applied to the device grid by
--     b7_mlp_features (b7_mlp_features_act when it has Tanh or no-activation inner layers; no 32-row minibatch loop, no host
--     copy of Z1), the head is b7_blr_fit + b7_blr_predict;
--   * bots.bayesopt (bayesopt.lua) calls model:acquire(...), which fuses basis + head + score + argmax in one pass
--     over the grid (b7_dngo_score) and never stores Z1; with config.bot.nGPU > 1 it calls model:acquire_multi(...), the
--     same pass over the grid's shards (b7_blr_fit_multi + b7_dngo_score_multi).
-- BLR hyper rows [log alpha_p, log beta, m] follow oracle/SPEC.md (gpTorch7's bayes_linear is not available).
-- With config.predictor.sampler == 'slice' the rows that 'marginalize' averages over are nSamples successive states of a slice
-- sampling chain on the BLR log evidence + the N(0, prior_std^2) prior (dngo:sample_blr_hypers, b7_blr_refit on a resident
-- handle); without it the head uses the one fixed row [log alpha_p, log beta, mean(Y0)], as it always has.
local B   = require('bot7_b200.ffi')
local ffi = require('ffi')

local dngo, parent = torch.class('bot7_b200.models.dngo', 'bot7.models.dngo')

function dngo:__init(config, cache, X, Y)
  parent.__init(self, config, cache, X, Y)
end

function dngo:class() return 'bot7.models.dngo' end

-- weights of the nn.Linear modules up to (and including) the basis layer, with the activation that follows each one: arrays for
-- b7_mlp_features(_act) / b7_dngo_score(_act).  Recognised: nn.Linear, nn.ReLU, nn.Tanh, and what is the identity in evaluation
-- mode (nn.Identity; nn.Dropout in its v2 form, Torch7's default, or with p = 0).  Anything else -- another module, two
-- activations after one Linear, an activation before the first Linear -- is an error naming the module and its position:
-- the device would otherwise evaluate a different network than the host basis the head is fitted on.
-- relu_last is set when the codes are the relu_last form (ReLU after every Linear but the last, ReLU or nothing after the
-- last): such stacks keep calling the entries without _act.
local ACT = {['nn.ReLU'] = 1, ['nn.Tanh'] = 2}                   -- B7_ACT_RELU, B7_ACT_TANH (B7_ACT_NONE = 0)

function dngo:basis_stack()
  local Ws, bs, dims, codes = {}, {}, {}, {}
  local acted = false                                            -- an activation already follows the last Linear
  for idx = 1, self.network:size() do
    local mod = self.network:get(idx)
    local t   = torch.type(mod)
    local where = string.format("module %d of the network (%s)", idx, t)
    if t == 'nn.Linear' then
      Ws[#Ws + 1] = mod.weight:contiguous():double()         -- h_out x h_in, like torch nn.Linear.weight
      bs[#bs + 1] = mod.bias:contiguous():double()
      if #dims == 0 then dims[1] = mod.weight:size(2) end
      dims[#dims + 1] = mod.weight:size(1)
      codes[#codes + 1] = 0
      acted = false
    elseif ACT[t] then
      if #Ws == 0 then error('bot7_b200.models.dngo: ' .. where .. ' comes before the first nn.Linear of the basis', 2) end
      if acted then error('bot7_b200.models.dngo: ' .. where .. ' is a second activation after one nn.Linear', 2) end
      codes[#codes] = ACT[t]
      acted = true
    elseif t == 'nn.Identity' or (t == 'nn.Dropout' and (mod.v2 or (mod.p or 0) == 0)) then
      -- the identity in evaluation mode (host_basis runs the network after :evaluate())
    elseif t == 'nn.Dropout' then
      error('bot7_b200.models.dngo: ' .. where .. ' is a v1 Dropout with p > 0, which scales by 1 - p in evaluation mode; ' ..
            'the basis takes nn.Linear, nn.ReLU, nn.Tanh, nn.Identity and v2 nn.Dropout', 2)
    else
      error('bot7_b200.models.dngo: ' .. where .. ' is not supported in the basis; it takes nn.Linear, nn.ReLU, nn.Tanh, ' ..
            'nn.Identity and v2 nn.Dropout', 2)
    end
    if mod == self.basis then break end
  end
  local n   = #Ws
  local relu_form = n > 0 and codes[n] ~= 2
  for l = 1, n - 1 do relu_form = relu_form and codes[l] == 1 end
  local cd  = ffi.new('int[?]', n + 1, dims)
  local cW  = ffi.new('const double*[?]', n)
  local cb  = ffi.new('const double*[?]', n)
  for l = 1, n do cW[l - 1] = Ws[l]:data(); cb[l - 1] = bs[l]:data() end
  return {n = n, dims = cd, W = cW, b = cb, relu_last = (codes[n] == 1) and 1 or 0, act = ffi.new('int[?]', n, codes),
          relu_form = relu_form, codes = codes, keep = {Ws, bs}, zDim = dims[#dims]}
end

-- Z = basis(X) on the host for the (few) observations, through the network itself (models/dngo.lua:155-162)
function dngo:host_basis(X)
  local bsz = self.config.update.schedule.batchsize
  local N   = X:size(1)
  local Z   = torch.DoubleTensor(N, self.config.zDim)
  self.network:evaluate()
  for tail = 1, N, bsz do
    local head = math.min(tail + bsz - 1, N)
    self.network:forward(X:sub(tail, head))
    Z:sub(tail, head):copy(self.basis.output)
  end
  return Z
end

function dngo:blr_hyp(Y0, hyp)
  if torch.isTensor(hyp) then return hyp:contiguous():double() end
  local p = self.config.predictor or {}
  return torch.DoubleTensor{{math.log(p.alpha_p or 1.0), math.log(p.beta or 1e2), Y0:mean()}}
end

-- settings of the hyper-parameter chain (config.predictor, read with the defaults of the Python twin bayes_linear)
local function chain_config(self)
  local p = self.config.predictor or {}
  return {sampler = p.sampler, nSamples = p.nSamples or 10, prior_std = p.prior_std or 2.0, speculative = p.speculative ~= false,
          spec_width = math.max(p.spec_width or 8, 1), burnin = p.burnin or 0}
end

-- the S x 3 rows the head is fitted with: `hyp` if given, else the chain's next nSamples states (sampler = 'slice', evaluated
-- on B.context() also when the head is fitted on several devices) or the one fixed row
function dngo:blr_rows_for(Z0, Y0, hyp)
  if not torch.isTensor(hyp) and chain_config(self).sampler == 'slice' then hyp = self:sample_blr_hypers(Z0, Y0) end
  return self:blr_hyp(Y0, hyp)
end

function dngo:blr_fit(Z0, Y0, hyp)
  local hyp    = self:blr_rows_for(Z0, Y0, hyp)
  local Z0, Y0 = Z0:contiguous():double(), Y0:contiguous():double()
  local box, info = ffi.new('b7_blr*[1]'), ffi.new('int[?]', hyp:size(1))
  B.check(B.C.b7_blr_fit(B.context(), Z0:data(), Y0:data(), Z0:size(1), Z0:size(2), hyp:data(), hyp:size(1), box, info), 'b7_blr_fit')
  self.blr_rows = hyp
  return ffi.gc(box[0], B.C.b7_blr_free), hyp:size(1)
end

---------------- log p(y | h) + log p(h) of the BLR head for the rows of H: the density the slice sampler evaluates.
-- Z0 and y stay resident between evaluations (b7_blr_refit on one handle of W slots); a failed factorisation or a
-- non-finite evidence is -inf, so the sampler rejects the point.
function dngo:blr_log_density_batch(H, Z0, Y0, W)
  local c    = chain_config(self)
  local H    = H:contiguous():double():view(-1, 3)
  local k    = H:size(1)
  local W    = W or c.spec_width
  local out  = torch.DoubleTensor(k)
  local pad  = torch.DoubleTensor(W, 3)
  local info, logev = ffi.new('int[?]', W), torch.DoubleTensor(W)
  self._blr_density = self._blr_density or {}
  for c0 = 1, k, W do
    local n = math.min(W, k - c0 + 1)
    pad:narrow(1, 1, n):copy(H:narrow(1, c0, n))
    for r = n + 1, W do pad[r]:copy(H[c0 + n - 1]) end       -- short batches repeat their last row
    local slot = self._blr_density[W]
    if slot == nil or slot.Z ~= Z0 or slot.Y ~= Y0 then
      local box, finfo = ffi.new('b7_blr*[1]'), ffi.new('int[?]', W)
      B.check(B.C.b7_blr_fit(B.context(), Z0:data(), Y0:data(), Z0:size(1), Z0:size(2), pad:data(), W, box, finfo), 'b7_blr_fit')
      slot = {blr = ffi.gc(box[0], B.C.b7_blr_free), Z = Z0, Y = Y0}
      self._blr_density[W] = slot
    end
    B.check(B.C.b7_blr_refit(slot.blr, pad:data(), B.C.B7_FIT_LOGML_ONLY, info, logev:data()), 'b7_blr_refit')
    for i = 1, n do
      local lp = logev[i]
      if info[i - 1] ~= 0 or lp ~= lp or lp == math.huge or lp == -math.huge then lp = -math.huge end
      out[c0 + i - 1] = lp - 0.5 * H[c0 + i - 1]:clone():div(c.prior_std):pow(2):sum()
    end
  end
  return out
end

---------------- the (alpha_p, beta, m) rows 'marginalize' averages over: nSamples successive states of the chain, which starts
-- at the fixed row of blr_hyp (after `burnin` discarded steps) and is kept across calls, like gp_regressor:sample_hypers.
-- sampler_spec.lua batches spec_width evaluations per device call; speculative = false uses bot7.samplers.slice.
function dngo:sample_blr_hypers(Z0, Y0, single)
  local c = chain_config(self)
  local Z0, Y0 = Z0:contiguous():double(), Y0:contiguous():double()
  local sampler, f
  if c.speculative then
    sampler = require('bot7_b200.sampler_spec')()
    f       = function(V, args) return self:blr_log_density_batch(V, Z0, Y0) end
  else
    sampler = bot7.samplers.slice()
    f       = function(x, args) return self:blr_log_density_batch(x, Z0, Y0, 1)[1] end
  end
  local function step(x)
    if c.speculative then return sampler(f, x, {nSamples = 1}, nil, c.spec_width) end
    return sampler(f, x, {nSamples = 1}, nil)
  end
  if self.blr_state == nil then
    local x = self:blr_hyp(Y0, nil)
    for _ = 1, c.burnin do x = step(x) end
    self.blr_state = x:view(1, -1):clone()
  end
  local n   = single and 1 or c.nSamples
  local out = torch.DoubleTensor(n, 3)
  local x   = self.blr_state:view(1, -1):clone()
  for i = 1, n do
    x = step(x)
    out[i]:copy(x[1])
  end
  self.blr_state = out[n]:view(1, -1):clone()
  if single then return out[1]:view(1, -1) end
  return out
end

---------------- models/dngo.lua:108-175: same signature and return value
function dngo:predict(X0, Y0, X1, hyp, req, skip)
  if not skip then parent.update_network(self, X0, Y0) end       -- the network update of :126-153 (see install())
  local Z0      = self:host_basis(X0)
  local blr, S  = self:blr_fit(Z0, Y0, hyp)
  local st      = self:basis_stack()
  local X1      = X1:contiguous():double()
  local M       = X1:size(1)
  local gbox, fbox = ffi.new('b7_grid*[1]'), ffi.new('b7_grid*[1]')
  B.check(B.C.b7_grid_from_host(B.context(), X1:data(), M, X1:size(2), gbox), 'b7_grid_from_host')
  local grid = ffi.gc(gbox[0], B.C.b7_grid_free)
  if st.relu_form then
    B.check(B.C.b7_mlp_features(B.context(), grid, st.n, st.dims, st.W, st.b, st.relu_last, fbox), 'b7_mlp_features')
  else
    B.check(B.C.b7_mlp_features_act(B.context(), grid, st.n, st.dims, st.W, st.b, st.act, fbox), 'b7_mlp_features_act')
  end
  local feats = ffi.gc(fbox[0], B.C.b7_grid_free)
  local Z1 = torch.DoubleTensor(M, st.zDim)
  B.check(B.C.b7_grid_read(feats, 0, M, Z1:data()), 'b7_grid_read')
  local mean, var = torch.zeros(M, 1), torch.zeros(M, 1)
  local m_s, v_s  = torch.DoubleTensor(M, 1), torch.DoubleTensor(M, 1)
  for s = 0, S - 1 do                                            -- 'marginalize': average over the (alpha_p, beta) rows
    B.check(B.C.b7_blr_predict(blr, s, Z1:data(), M, m_s:data(), v_s:data()), 'b7_blr_predict')
    mean:add(m_s); var:add(v_s)
  end
  collectgarbage()
  return {mean = mean:div(S), var = var:div(S)}
end

---------------- device body of bot:eval + bot:nominate for DNGO (bots/bayesopt.lua:65-66,96): one pass over the grid
function dngo:acquire(X0, Y0, grid_dev, kind, tradeoff, bound, sign, skip)
  if not skip then parent.update_network(self, X0, Y0) end
  local blr = self:blr_fit(self:host_basis(X0), Y0, nil)
  local st  = self:basis_stack()
  local argmax, orig = ffi.new('int64_t[1]'), ffi.new('int64_t[1]')
  local best, nans   = ffi.new('double[1]'), ffi.new('int64_t[1]')
  if st.relu_form then
    B.check(B.C.b7_dngo_score(blr, grid_dev, st.n, st.dims, st.W, st.b, st.relu_last, kind, tradeoff, bound, sign, Y0:min(),
                              nil, argmax, orig, best, nans), 'b7_dngo_score')
  else
    B.check(B.C.b7_dngo_score_act(blr, grid_dev, st.n, st.dims, st.W, st.b, st.act, kind, tradeoff, bound, sign, Y0:min(),
                                  nil, argmax, orig, best, nans), 'b7_dngo_score_act')
  end
  return tonumber(argmax[0]), best[0], tonumber(nans[0])
end

---------------- the same over the nGPU devices of a communicator (bots.bayesopt with config.bot.nGPU > 1): the head is fitted on
-- every device (b7_blr_fit_multi), each device scores its shard of the grid and the library combines the argmax
-- (b7_dngo_score_multi); the result equals acquire's on one device over the whole grid
function dngo:acquire_multi(X0, Y0, comm, grids, nGPU, kind, tradeoff, bound, sign, skip)
  if not skip then parent.update_network(self, X0, Y0) end
  local Z0   = self:host_basis(X0)
  local hyp  = self:blr_rows_for(Z0, Y0, nil)
  local Yc   = Y0:contiguous():double()
  local blrs = ffi.new('b7_blr*[?]', nGPU)
  B.check(B.C.b7_blr_fit_multi(comm, Z0:data(), Yc:data(), Z0:size(1), Z0:size(2), hyp:data(), hyp:size(1), blrs, nil), 'b7_blr_fit_multi')
  self.blr_rows = hyp
  local st = self:basis_stack()
  local argmax, orig = ffi.new('int64_t[1]'), ffi.new('int64_t[1]')
  local best, nans   = ffi.new('double[1]'), ffi.new('int64_t[1]')
  local rc, what
  if st.relu_form then
    rc, what = B.C.b7_dngo_score_multi(comm, blrs, grids, st.n, st.dims, st.W, st.b, st.relu_last, kind, tradeoff, bound, sign,
                                       Y0:min(), nil, argmax, orig, best, nans), 'b7_dngo_score_multi'
  else
    rc, what = B.C.b7_dngo_score_multi_act(comm, blrs, grids, st.n, st.dims, st.W, st.b, st.act, kind, tradeoff, bound, sign,
                                           Y0:min(), nil, argmax, orig, best, nans), 'b7_dngo_score_multi_act'
  end
  for g = 0, nGPU - 1 do B.C.b7_blr_free(blrs[g]) end
  B.check(rc, what)
  return tonumber(argmax[0]), best[0], tonumber(nans[0])
end

return dngo
