"""Parity of the BENCHMARKED tier (fp16 operands on tcgen05, fp32 accumulation / master weights) at the
benchmark's minibatch size, against the CPU oracle and the live-reference golden vectors.

North star: action logits, values, GAE returns and losses within 1e-2 of the reference's torch path on
identical rollout tensors for the reduced-precision tier.  Three levels:

 (1) ONE update from identical weights (`test_tc_tier_step_all_keys`): all 18 logged statistics
     (reference ppo.py:76-92,122-123,141-145), the values / action means of the minibatch and the
     gradient of each optimiser bucket, at RTOL = 1e-2.
 (2) A WHOLE EPOCH along the reference trajectory (`test_tc_tier_epoch_teacher_forced`): 8 minibatches x
     2 opt-epochs at B = 1024; before every minibatch the engine's parameters and Adam moments are set to
     the oracle's, so each of the 16 updates is compared on identical weights / optimiser state at the
     point of the trajectory where the reference would evaluate it (stepped encoders, ratio != 1, clipping
     active).  All 18 statistics of EVERY minibatch, GAE returns and held-out outputs at RTOL = 1e-2.
 (3) The FREE-RUNNING epoch (`test_tc_tier_epoch_free_running`, and the T=8, E=4 case of tests/golden
     written by the live reference): two trajectories that start identical drift apart, because a ReLU
     gate whose pre-activation lies within the fp16 rounding error of 0 flips, and Adam's first steps are
     sign-like (|dw| = lr whatever |g|), so a gradient component within the noise of 0 moves its weight by
     2 lr the other way.  This is a property of 16-bit STORAGE, not of these kernels:
     tools/probe_storage_rounding.py reproduces it on the CPU with the oracle's own fp32 arithmetic and
     straight-through fp16 rounding of the stored tensors and drifts by the same amounts (policy_loss 10 %,
     ratio extremes 9-10 %, grad_norm/pf 9 %, held-out means 5 % after 16 steps; profiles/r2_storage_drift.txt).
     The drift saturates at that level for ANY perturbation, down to 1e-6 relative noise (the size of an fp32
     summation-order change: policy_loss 9 %, ratio 7-10 %, held-out 3-4 %): the 16-step trajectory is chaotic at
     the fp32 rounding level, so the exact fp32 tier drifts just the same (`test_exact_tier_epoch_free_running`).
     Asserted here:
     GAE at 1e-2, every statistic within FREE_RTOL of the fp32 trajectory, held-out outputs within
     FREE_RTOL_OUT (measured numbers are printed and kept in profiles/).

Absolute floors: a statistic that is a difference of nearly equal numbers is compared on the scale of its
operands — advs/mean on the scale of advs/std, logprob/* on the scale of logprob/std (log-probabilities
are O(10) with extremes near 0), everything else 1e-4.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as po, synth
from tests import _golden as g
from tests._harness import build_nets, load_np_sd, fill_buffer, make_ppo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-2
FREE_RTOL = 0.15          # free-running drift of the logged statistics over 16 optimiser steps (see module doc)
FREE_RTOL_OUT = 6e-2      # ... of held-out action means / values after those steps
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _agent(family, buf, B, frames, opt_epochs, graph=True):
  S, A = g.FAMILIES[family]
  pf, vf = build_nets(family, S, A)
  pf_np, vf_np = g.family_weights(family)
  load_np_sd(pf, pf_np); load_np_sd(vf, vf_np)
  pf, vf = pf.to(DEV), vf.to(DEV)
  agent, logger = make_ppo(pf, vf, buf, A, B, frames, opt_epochs, device=DEV)
  agent.precision = "f16"
  agent.use_cuda_graph = graph
  return agent, logger, pf, vf, pf_np, vf_np


def _atol(k, ref, rtol):
  if k == "advs/mean":
    return rtol * abs(ref["advs/std"])
  if k.startswith("logprob/"):
    return rtol * abs(ref["logprob/std"])
  return 1e-4


def info_errors(infos, refs, rtol=RTOL, rtol_grad_norm=None):
  """[(minibatch, key, got, want, err / allowed)] with allowed = rtol*|want| + atol(key)"""
  rows = []
  for i, (a, b) in enumerate(zip(infos, refs)):
    for k in g.INFO_KEYS:
      rt = rtol_grad_norm if (rtol_grad_norm and k.startswith("grad_norm/")) else rtol
      rows.append((i, k, float(a[k]), float(b[k]), abs(a[k] - b[k]) / (rt * abs(b[k]) + _atol(k, b, rt))))
  return rows


def _report(name, rows, extra, rtol):
  worst = {}
  for i, k, a, b, e in rows:
    if e >= worst.get(k, (-1, 0, 0, 0))[0]:
      worst[k] = (e, i, a, b)
  print("\n%s: worst error per statistic, in units of the allowed deviation (rtol %.0e)" % (name, rtol))
  for k in g.INFO_KEYS:
    e, i, a, b = worst.get(k, (0, 0, 0, 0))
    print("  %-22s %6.3f   (minibatch %2d: got %.6g want %.6g)" % (k, e, i, a, b))
  for k, v in extra.items():
    print("  %-22s %.3e" % (k, v))
  out = os.path.join(ROOT, "gpurun_out")
  if os.path.isdir(out):
    with open(os.path.join(out, "tc_parity_%s.json" % name), "w") as f:
      json.dump({"rtol": rtol, "worst_in_units_of_allowed": {k: list(v) for k, v in worst.items()}, "extra": extra},
                f, indent=1)


def _epoch_case(family, n_mb=8, opt_epochs=2, B=1024, E=8):
  S, A = g.FAMILIES[family]
  T = n_mb * B // E
  roll = synth.make_rollout(31, T, E, S, A, p_term=1.0 / 200)
  np.random.seed(77)
  perms = np.stack([np.random.permutation(T) for _ in range(opt_epochs)])
  return S, A, T, roll, perms


def _heldout(agent, orc, S):
  held = synth.make_obs(np.random.default_rng(5), 256, S)
  mean, value = agent.engine.infer(held)
  held = torch.tensor(held, dtype=orc.dtype)
  return {"heldout/mean": g.rel_err(mean.cpu().numpy(), orc.policy(held).numpy()),
          "heldout/value": g.rel_err(value.cpu().numpy(), orc.values(held).numpy())}


def _bucket_grad_err(eng, orc, info_ref):
  """norm-wise error of the whole gradient of each optimiser (the quantity clip + Adam consume); the
  oracle keeps its gradients AFTER clip_grad_norm_ scaled them in place"""
  out = {}
  for name, G, ref, key in (("vf", eng.G_vf, orc._last["vgrads"], "grad_norm/vf"),
                            ("pf", eng.G_pf, orc._last["pgrads"], "grad_norm/pf")):
    c = min(1.0, 0.5 / (info_ref[key] + 1e-6))
    num = sum(float((G[k].double().cpu() * c - r.double()).pow(2).sum()) for k, r in ref.items())
    den = sum(float(r.double().pow(2).sum()) for r in ref.values())
    out["grad_bucket_err/" + name] = (num / den) ** 0.5
  return out


# -------------------------------------------------------------------------------------------------
# (1) one update from identical weights
# -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["loco", "nature", "vit", "nvo"])
def test_tc_tier_step_all_keys(family):
  S, A = g.FAMILIES[family]
  B = 1024
  agent, _, pf, vf, pf_np, vf_np = _agent(family, None, B, B, 1, graph=False)
  agent.current_epoch = 0
  opf, ovf = po.sd_to_torch(pf_np, vf_np)
  orc = po.PPOOracle(family, opf, ovf, S, batch_size=B, opt_epochs=1)
  rng = np.random.default_rng(21)
  roll = synth.make_rollout(21, B // 8, 8, S, A, p_term=0.01)
  batch = {"obs": roll["obs"].reshape(B, -1), "acts": roll["acts"].reshape(B, -1),
           "advs": rng.standard_normal((B, 1)), "estimate_returns": rng.standard_normal((B, 1)),
           "values": roll["values"].reshape(B, 1)}
  ref = orc.update(batch)
  info = agent.update(batch)
  eng = agent.engine
  extra = {"step/values": g.rel_err(eng._bufs(B)["values"].cpu().numpy(), orc._last["values"].numpy()),
           "step/mean": g.rel_err(eng._bufs(B)["mean"].cpu().numpy(), orc._last["mean"].numpy())}
  extra.update(_bucket_grad_err(eng, orc, ref))
  rows = info_errors([info], [ref])
  _report("step_" + family, rows, extra, RTOL)
  assert extra["step/values"] < RTOL and extra["step/mean"] < RTOL, extra
  bad = [(k, a, b, round(e, 2)) for _, k, a, b, e in rows if not e <= 1.0]
  assert not bad, bad
  # whole-bucket gradients (what the clip + Adam step consumes); individual encoder tensors with small
  # gradients deviate by up to ~8 % (ReLU gates within the fp16 rounding error of 0, see the module doc)
  assert extra["grad_bucket_err/vf"] < 2e-2 and extra["grad_bucket_err/pf"] < 2e-2, extra


# -------------------------------------------------------------------------------------------------
# (2) a whole epoch along the reference trajectory
# -------------------------------------------------------------------------------------------------
def _sync_from_oracle(agent, orc):
  """engine parameters + Adam moments + step counts <- the oracle's (the reference trajectory)"""
  eng = agent.engine
  agent.pf.load_state_dict({k: v.detach().clone() for k, v in orc.pf.items()})
  agent.vf.load_state_dict({k: v.detach().clone() for k, v in orc.vf.items()})
  for net, keys, opt, m_flat, v_flat, rng, hyper in (
      (agent.pf, orc.pf_keys, orc.pf_opt, eng.m_pf, eng.v_pf, eng.pf_range, eng.hyper_pf),
      (agent.vf, orc.vf_keys, orc.vf_opt, eng.m_vf, eng.v_vf, eng.vf_range, eng.hyper_vf)):
    named = dict(net.named_parameters())
    for k, m, v in zip(keys, opt.m, opt.v):
      eng.bucket.view_of(m_flat, named[k], rng[0]).copy_(m)
      eng.bucket.view_of(v_flat, named[k], rng[0]).copy_(v)
    hyper[5] = float(opt.t)
  eng.check_views()


@pytest.mark.parametrize("family", ["loco", "nature"])
def test_tc_tier_epoch_teacher_forced(family):
  """The oracle runs in float64: the 16-step trajectory is chaotic at the fp32 rounding level (module doc, (3)), so an
  fp32 oracle's trajectory, and with it the points at which the tier is compared, would depend on the host's CPU
  kernels and thread count.  In float64 every host follows the same trajectory."""
  S, A, T, roll, perms = _epoch_case(family)
  B, E = 1024, 8
  agent, _, pf, vf, pf_np, vf_np = _agent(family, None, B, B, 1, graph=False)
  agent.current_epoch = 0
  opf, ovf = po.sd_to_torch(pf_np, vf_np, dtype=torch.float64)
  orc = po.PPOOracle(family, opf, ovf, S, batch_size=B, opt_epochs=len(perms), dtype=torch.float64)
  advs, rets = orc.process_epoch_samples(roll)
  # GAE on the device (the bootstrap value runs on the fp16 tier) through the engine's own entry points
  eng = agent.engine
  eng.load_rollout_arrays(roll)
  eng.compute_advantages(roll["last_obs"], roll["last_terminals"], 0.99, 0.95, True, True)
  gae = {"gae/advs": g.rel_err(eng._roll["advs"].cpu().numpy().reshape(advs.shape), advs),
         "gae/returns": g.rel_err(eng._roll["rets"].cpu().numpy().reshape(rets.shape), rets)}
  infos, refs = [], []
  rows_mb = B // E
  for ep in range(len(perms)):
    for pos in range(0, T, rows_mb):
      idx = perms[ep][pos:pos + rows_mb]
      batch = {"obs": roll["obs"][idx].reshape(B, -1), "acts": roll["acts"][idx].reshape(B, -1),
               "advs": advs[idx].reshape(B, 1), "estimate_returns": rets[idx].reshape(B, 1),
               "values": roll["values"][idx].reshape(B, 1)}
      _sync_from_oracle(agent, orc)
      infos.append(agent.update(batch))
      refs.append(orc.update(batch))
  extra = dict(gae)
  _sync_from_oracle(agent, orc)
  extra.update(_heldout(agent, orc, S))
  # grad_norm/*: 3e-2.  The surrogate's gradient is discontinuous in the ratio (a sample whose ratio is within
  # the 3e-3 forward error of 1 +- clip switches between "contributes" and "clipped"), so along the trajectory,
  # where ~1 % of the 1024 samples sit that close to the boundary, the logged gradient NORM moves by ~1 %;
  # on the first minibatch (ratio ~ 1, nothing near the boundary) it is within 1e-3 (step test above).
  rows = info_errors(infos, refs, rtol_grad_norm=3e-2)
  _report("forced_" + family, rows, extra, RTOL)
  assert extra["gae/advs"] < RTOL and extra["gae/returns"] < RTOL
  bad = [(i, k, a, b, round(e, 2)) for i, k, a, b, e in rows if not e <= 1.0]
  assert not bad, bad[:10]
  assert extra["heldout/mean"] < RTOL and extra["heldout/value"] < RTOL, extra


# -------------------------------------------------------------------------------------------------
# (3) free-running epochs
# -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family,precision", [("loco", "f16"), ("nature", "f16"), ("loco", "fp32")],
                         ids=["loco", "nature", "exact_tier_loco"])
def test_tc_tier_epoch_free_running(family, precision):
  """precision fp32 = the exact tier (1e-5 per-step parity with the reference's goldens): it drifts from the
  oracle's trajectory by the same few percent over these 16 steps — the drift is not a reduced-precision effect."""
  S, A, T, roll, perms = _epoch_case(family)
  B, E = 1024, 8
  buf = fill_buffer(roll, T, E)
  agent, logger, pf, vf, pf_np, vf_np = _agent(family, buf, B, T * E, len(perms))
  agent.precision = precision
  agent.current_epoch = 7
  np.random.seed(77)
  agent.update_per_epoch()
  torch.cuda.synchronize()
  assert agent.engine.ops.opt_tail_error() == 0
  opf, ovf = po.sd_to_torch(pf_np, vf_np)
  orc = po.PPOOracle(family, opf, ovf, S, batch_size=B, opt_epochs=len(perms))
  orc.current_epoch = 7
  advs, rets, refs = orc.update_per_epoch(roll, perms)
  extra = {"gae/advs": g.rel_err(buf._advs, advs), "gae/returns": g.rel_err(buf._estimate_returns, rets)}
  assert len(logger.infos) == len(refs) == len(perms) * T * E // B
  extra.update(_heldout(agent, orc, S))
  extra["params/pf_max_rel_drift"] = max(g.rel_err(v.cpu().numpy(), orc.pf[k].numpy()) for k, v in pf.state_dict().items())
  extra["params/vf_max_rel_drift"] = max(g.rel_err(v.cpu().numpy(), orc.vf[k].numpy()) for k, v in vf.state_dict().items())
  rows = info_errors(logger.infos, refs, FREE_RTOL)
  _report("free_" + family + ("" if precision == "f16" else "_exact_tier"), rows, extra, FREE_RTOL)
  assert extra["gae/advs"] < RTOL and extra["gae/returns"] < RTOL
  bad = [(i, k, a, b, round(e, 2)) for i, k, a, b, e in rows if not e <= 1.0]
  assert not bad, bad[:10]
  assert extra["heldout/mean"] < FREE_RTOL_OUT and extra["heldout/value"] < FREE_RTOL_OUT, extra
  # the first minibatch starts from identical weights: 1e-2 on everything
  first = [(k, a, b, round(e, 2)) for i, k, a, b, e in info_errors(logger.infos[:1], refs[:1]) if not e <= 1.0]
  assert not first, first


@pytest.mark.parametrize("family", ["loco", "nature"])
def test_tc_tier_epoch_vs_reference_golden(family):
  """The T=8, E=4 epoch of tests/golden (outputs of the LIVE reference): GAE at 1e-2, the first
  minibatch at 1e-2, the free-running 2 opt-epochs x 2 minibatches of 16 within FREE_RTOL."""
  G = g.load(family)
  roll = g.epoch_inputs(family)
  buf = fill_buffer(roll, 8, 4)
  agent, logger, pf, vf, _, _ = _agent(family, buf, 16, 32, 2)
  agent.current_epoch = 30
  np.random.seed(1234)
  agent.update_per_epoch()
  assert g.rel_err(buf._advs, G["epoch/advs"]) < RTOL
  assert g.rel_err(buf._estimate_returns, G["epoch/rets"]) < RTOL
  assert len(logger.infos) == int(G["epoch/n_infos"])
  refs = [{k: float(G["epoch/info%d/%s" % (i, k)]) for k in g.INFO_KEYS} for i in range(len(logger.infos))]
  first = [(k, a, b, round(e, 2)) for _, k, a, b, e in info_errors(logger.infos[:1], refs[:1]) if not e <= 1.0]
  assert not first, first
  rows = info_errors(logger.infos, refs, FREE_RTOL)
  _report("golden_" + family, rows, {}, FREE_RTOL)
  bad = [(i, k, a, b, round(e, 2)) for i, k, a, b, e in rows if not e <= 1.0]
  assert not bad, bad
  g.check_summary(G, "epoch/pf", [(k, v.cpu().numpy()) for k, v in pf.state_dict().items()], 5e-2)
  g.check_summary(G, "epoch/vf", [(k, v.cpu().numpy()) for k, v in vf.state_dict().items()], 5e-2)
