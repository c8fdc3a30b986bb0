-- bots.bayesopt with the body of eval / nominate (bots/bayesopt.lua:56-99) routed to batched device calls:
--   S draws -> S factors -> posterior + score + average + argmax over the device-resident grid.
-- config.bot.nGPU > 1 spreads the same work over the GPUs of the box through the multi-GPU block of the C ABI
-- (b7_comm_init_all, b7_gp_fit_sharded, b7_acq_score_multi): candidate shards per device, the S factorisations split
-- over the devices and exchanged once per fit with NCCL, the per-device (best, index) triples combined in the library.
-- A DNGO model does the same through dngo:acquire_multi (b7_blr_fit_multi: the small BLR head is fitted on every device;
-- b7_dngo_score_multi: basis + head + score on each shard, same combine).
local B   = require('bot7_b200.ffi')
local ffi = require('ffi')

local title  = 'bot7_b200.bots.bayesopt'
local parent = 'bot7.bots.bayesopt'
local bot, parent = torch.class(title, parent)

local kernels = { ardse = B.C.B7_KERNEL_ARDSE, matern52 = B.C.B7_KERNEL_MATERN52, matern_52 = B.C.B7_KERNEL_MATERN52 }

function bot:__init(objective, hypers, config, cache)
  parent.__init(self, objective, hypers, config, cache)
  self.nGPU = (self.config.bot.nGPU or 1)
  -- keep the grid on the device(s) as well; self.candidates stays for callers that read it
  local X = self.candidates:contiguous():double()
  if self.nGPU > 1 then
    local cbox = ffi.new('b7_comm*[1]')
    B.check(B.C.b7_comm_init_all(self.nGPU, nil, cbox), 'b7_comm_init_all')
    self.comm  = ffi.gc(cbox[0], B.C.b7_comm_free)
    self.grids = ffi.new('b7_grid*[?]', self.nGPU)
    B.check(B.C.b7_grid_from_host_sharded(self.comm, X:data(), X:size(1), X:size(2), self.grids), 'b7_grid_from_host_sharded')
  else
    local box = ffi.new('b7_grid*[1]')
    B.check(B.C.b7_grid_from_host(B.context(), X:data(), X:size(1), X:size(2), box), 'b7_grid_from_host')
    self.grid_dev = ffi.gc(box[0], B.C.b7_grid_free)
  end
end

-- utils.tensor.steal on the device grid (bots/abstract.lua:118): same compacted numbering as self.candidates
function bot:remove_dev(idx)
  if self.nGPU > 1 then
    B.check(B.C.b7_grid_remove_sharded(self.comm, self.grids, idx, nil), 'b7_grid_remove_sharded')
  else
    B.check(B.C.b7_grid_remove(self.grid_dev, idx, nil), 'b7_grid_remove')
  end
end

function bot:score_args()
  local sc    = self.score.config
  local kind  = (torch.type(self.score):find('confidence_bound')) and B.C.B7_SCORE_CB or B.C.B7_SCORE_EI
  local bound = (sc.bound and sc.bound:lower() == 'upper') and B.C.B7_BOUND_UPPER or B.C.B7_BOUND_LOWER
  return kind, sc.tradeoff, bound, sc.sign or -1.0
end

function bot:nominate(candidates)
  if self.nTrials <= self.config.bot.nInitial then             -- bots/bayesopt.lua:90-91
    local idx = torch.rand(1):mul(self.candidates:size(1)):long():add(1)
    self:remove_dev(idx[1])
    return idx
  end
  local X_obs, Y_obs = self.observed, self.responses
  local kind, tradeoff, bound, sign = self:score_args()
  local argmax, orig = ffi.new('int64_t[1]'), ffi.new('int64_t[1]')
  local best, nans   = ffi.new('double[1]'), ffi.new('int64_t[1]')
  if self.model:class() == 'bot7.models.dngo' then             -- :65-66
    if self.nGPU > 1 then
      argmax[0] = self.model:acquire_multi(X_obs, Y_obs, self.comm, self.grids, self.nGPU, kind, tradeoff, bound, sign)
    else
      argmax[0] = self.model:acquire(X_obs, Y_obs, self.grid_dev, kind, tradeoff, bound, sign)
    end
  else
    local nSamples = self.config.bot.nSamples
    self.model:sample_hypers(X_obs, Y_obs)                      -- :68 priming draw (result unused)
    local hyps = {}
    for s = 1, nSamples do                                      -- :73-75
      hyps[s] = self.model:parse_hypers(self.model:sample_hypers(X_obs, Y_obs, nil, nil, true)):view(1, -1)
    end
    local hyp = torch.cat(hyps, 1):contiguous():double()
    if self.nGPU > 1 then
      local Xc, Yc = X_obs:contiguous():double(), Y_obs:contiguous():double()
      local gps  = ffi.new('b7_gp*[?]', self.nGPU)
      local info = ffi.new('int[?]', nSamples)
      B.check(B.C.b7_gp_fit_sharded(self.comm, kernels[self.model.config.kernel], Xc:data(), Yc:data(), Xc:size(1), Xc:size(2),
                                    hyp:data(), nSamples, hyp:size(2), self.model.config.noiseless and 1 or 0, gps, info,
                                    nil, nil, nil), 'b7_gp_fit_sharded')
      local rc = B.C.b7_acq_score_multi(self.comm, gps, self.grids, kind, tradeoff, bound, sign, Y_obs:min(),
                                        nil, argmax, orig, best, nans)
      for g = 0, self.nGPU - 1 do B.C.b7_gp_free(gps[g]) end
      B.check(rc, 'b7_acq_score_multi')
    else
      local gp = self.model:fit(X_obs, Y_obs, hyp)
      B.check(B.C.b7_acq_score(gp, self.grid_dev, kind, tradeoff, bound, sign, Y_obs:min(),
                               nil, argmax, orig, best, nans), 'b7_acq_score')
    end
  end
  assert(tonumber(argmax[0]) > 0, string.format('acquisition returned no finite score (%d NaN)', tonumber(nans[0])))
  local idx = torch.LongTensor{tonumber(argmax[0])}             -- compacted numbering, as score:max(1) (:96)
  self:remove_dev(idx[1])
  return idx
end

return bot
