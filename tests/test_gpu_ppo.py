"""End-to-end parity of the CUDA path against (a) the golden vectors produced by the live
reference and (b) the CPU oracle on the same seeded inputs.  Everything goes through the
public classes (networks / policies / PPO / OnPolicyReplayBuffer), i.e. through the C ABI.

Tolerance (north star): 1e-3 relative for the fp32 tier on action means, values, log-probs,
GAE returns and losses.  Measured errors are ~1e-5; a few quantities get documented looser
bounds because the reference computation itself amplifies fp32 noise (see comments).
"""
import numpy as np
import pytest
import torch

from oracle import ppo_oracle as po, synth
from tests import _golden as g
from tests._harness import build_nets, load_np_sd, fill_buffer, make_ppo

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3


def _nets(family):
  S, A = g.FAMILIES[family]
  pf, vf = build_nets(family, S, A)
  pf_np, vf_np = g.family_weights(family)
  load_np_sd(pf, pf_np); load_np_sd(vf, vf_np)
  return pf.to(DEV), vf.to(DEV), S, A


ALL = ["loco", "nature", "mlp", "vit", "nvo"]


@pytest.mark.parametrize("family", ALL)
def test_forward_matches_reference_golden(family):
  G = g.load(family)
  pf, vf, S, A = _nets(family)
  obs, acts = g.fwd_inputs(family)
  obs_t, acts_t = torch.tensor(obs, device=DEV), torch.tensor(acts, device=DEV)
  with torch.no_grad():
    out = pf.update(obs_t, acts_t)
    value = vf(obs_t)
    v1 = vf(obs_t[0])                      # 1-D input path (SURVEY B13)
  assert g.rel_err(out["mean"].cpu().numpy(), G["fwd/mean"]) < TOL
  assert g.rel_err(value.cpu().numpy(), G["fwd/value"]) < TOL
  assert g.rel_err(out["log_prob"].cpu().numpy(), G["fwd/log_prob"]) < TOL
  assert g.rel_err(out["ent"].cpu().numpy(), G["fwd/ent"]) < TOL
  assert v1.shape == (1,)
  if "fwd/value_1d" in G:
    assert g.rel_err(v1.cpu().numpy(), G["fwd/value_1d"]) < TOL
  assert g.rel_err(pf.eval_act(obs_t), G["fwd/eval_act"]) < TOL
  ex = pf.explore(obs_t, return_log_probs=True)
  assert ex["action"].shape == (8, A) and ex["log_prob"].shape == (8, 1)


@pytest.mark.parametrize("family", ALL)
def test_autograd_through_modules_matches_oracle(family):
  """d(sum of outputs * random cotangent)/d(every parameter) through torch.autograd on the CUDA
  modules vs torch autograd on the CPU oracle."""
  pf, vf, S, A = _nets(family)
  pf_np, vf_np = g.family_weights(family)
  opf, ovf = po.sd_to_torch(pf_np, vf_np)
  roll = synth.make_rollout(77, 3, 4, S, A, with_img=family != "mlp")
  obs = roll["obs"].reshape(12, -1)
  rng = np.random.default_rng(3)
  for net, sd, out_dim in ((pf, opf, A), (vf, ovf, 1)):
    cot = rng.standard_normal((12, out_dim)).astype(np.float32)
    names = [n for n, _ in net.named_parameters() if n != "logstd"]
    # oracle
    ps = [sd[n].requires_grad_(True) for n in names]
    ref = po.FORWARD[family](sd, torch.tensor(obs), S)
    gref = torch.autograd.grad((ref * torch.tensor(cot)).sum(), ps)
    for p in ps:
      p.requires_grad_(False)
    # product
    out = net(torch.tensor(obs, device=DEV))
    out = out[0] if isinstance(out, tuple) else out
    assert g.rel_err(out.detach().cpu().numpy(), ref.detach().numpy()) < TOL
    (out * torch.tensor(cot, device=DEV)).sum().backward()
    params = dict(net.named_parameters())
    for n, gr in zip(names, gref):
      e = g.rel_err(params[n].grad.cpu().numpy(), gr.numpy())
      assert e < TOL, (family, n, e)
    net.zero_grad()


@pytest.mark.parametrize("family", ALL)
@pytest.mark.parametrize("clipped", [False, True])
def test_one_update_matches_reference_golden(family, clipped):
  G = g.load(family)
  pf, vf, S, A = _nets(family)
  agent, _ = make_ppo(pf, vf, None, A, 16, 16, 1, device=DEV, clipped_value_loss=clipped)
  agent.current_epoch = 0
  info = agent.update(g.update_inputs(family))
  prefix = "updclip" if clipped else "upd"
  g.check_info(G, prefix + "/info", info, rtol=TOL, atol=1e-5)
  g.check_summary(G, prefix + "/vf", [(k, v.cpu().numpy()) for k, v in vf.state_dict().items()], TOL)
  if not clipped:
    g.check_summary(G, "upd/pf", [(k, v.cpu().numpy()) for k, v in pf.state_dict().items()], TOL)
    eng = agent.engine
    # gradients: the golden .grad are post-clip (clip_grad_norm_ scales in place)
    pn, vn = info["grad_norm/pf"], info["grad_norm/vf"]
    pc, vc = min(1.0, 0.5 / (pn + 1e-6)), min(1.0, 0.5 / (vn + 1e-6))
    g.check_summary(G, "upd/pgrad", [(k, v.cpu().numpy() * pc) for k, v in eng.G_pf.items()], 2e-3)
    g.check_summary(G, "upd/vgrad", [(k, v.cpu().numpy() * vc) for k, v in eng.G_vf.items()
                                     if k not in eng.G_pf], 2e-3)


@pytest.mark.parametrize("family", ALL)
@pytest.mark.parametrize("graph", [False, True])
def test_update_per_epoch_matches_reference_golden(family, graph):
  """GAE + LR schedule + target copy + 2 opt-epochs x 2 minibatches, through the replay buffer
  API and PPO.update_per_epoch(), eager and CUDA-graph replay."""
  G = g.load(family)
  pf, vf, S, A = _nets(family)
  roll = g.epoch_inputs(family)
  buf = fill_buffer(roll, 8, 4)
  agent, logger = make_ppo(pf, vf, buf, A, 16, 32, 2, device=DEV)
  agent.use_cuda_graph = graph
  agent.current_epoch = 30
  np.random.seed(1234)
  agent.update_per_epoch()
  assert g.rel_err(buf._advs, G["epoch/advs"]) < TOL
  assert g.rel_err(buf._estimate_returns, G["epoch/rets"]) < TOL
  assert len(logger.infos) == int(G["epoch/n_infos"]) == agent.training_update_num
  for i, info in enumerate(logger.infos):
    # ratio extremes: exp() of a difference of log-probs that is itself ~64x the parameter noise
    g.check_info(G, "epoch/info%d" % i, info, rtol=2e-3, atol=1e-4)
  g.check_summary(G, "epoch/pf", [(k, v.cpu().numpy()) for k, v in pf.state_dict().items()], TOL)
  g.check_summary(G, "epoch/vf", [(k, v.cpu().numpy()) for k, v in vf.state_dict().items()], TOL)
  g.check_summary(G, "epoch/target", [(k, v.cpu().numpy()) for k, v in agent.target_pf.state_dict().items()], TOL)
  np.testing.assert_allclose(G["epoch/lr"], [agent.pf_optimizer.param_groups[0]["lr"],
                                             agent.vf_optimizer.param_groups[0]["lr"]], rtol=1e-12)


def test_graph_and_eager_epochs_are_bit_identical():
  """Idempotence of the execution mode: replaying the captured graph must give exactly the
  bits of the eager kernel sequence (same kernels, deterministic reductions)."""
  outs = []
  for graph in (False, True):
    pf, vf, S, A = _nets("loco")
    roll = synth.make_rollout(5, 16, 4, S, A, p_term=0.1)
    buf = fill_buffer(roll, 16, 4)
    agent, logger = make_ppo(pf, vf, buf, A, 16, 64, 2, device=DEV)
    agent.use_cuda_graph = graph
    agent.current_epoch = 3
    np.random.seed(9)
    agent.update_per_epoch()
    agent.current_epoch = 4
    agent.update_per_epoch()
    outs.append((agent.engine.bucket.flat.clone(), [tuple(i.values()) for i in logger.infos]))
  assert torch.equal(outs[0][0], outs[1][0])
  assert outs[0][1] == outs[1][1]


def test_full_minibatch_matches_oracle():
  """BASELINE minibatch size (B=1024, LocoTransformer, S=93, A=12): one PPO.update against
  the CPU oracle on the same 1024 samples."""
  family = "loco"
  pf, vf, S, A = _nets(family)
  pf_np, vf_np = g.family_weights(family)
  opf, ovf = po.sd_to_torch(pf_np, vf_np)
  orc = po.PPOOracle(family, opf, ovf, S, batch_size=1024, opt_epochs=1)
  rng = np.random.default_rng(21)
  roll = synth.make_rollout(21, 128, 8, S, A, p_term=0.01)
  batch = {"obs": roll["obs"].reshape(1024, -1), "acts": roll["acts"].reshape(1024, -1),
           "advs": rng.standard_normal((1024, 1)), "estimate_returns": rng.standard_normal((1024, 1)),
           "values": roll["values"].reshape(1024, 1)}
  ref = orc.update(batch)
  agent, _ = make_ppo(pf, vf, None, A, 1024, 1024, 1, device=DEV)
  agent.current_epoch = 0
  info = agent.update(batch)
  for k in g.INFO_KEYS:
    assert abs(info[k] - ref[k]) <= 1e-5 + TOL * abs(ref[k]), (k, info[k], ref[k])
  for k, v in pf.state_dict().items():
    assert g.rel_err(v.cpu().numpy(), orc.pf[k].numpy()) < TOL, k
  for k, v in vf.state_dict().items():
    assert g.rel_err(v.cpu().numpy(), orc.vf[k].numpy()) < TOL, k


def test_ragged_last_minibatch():
  """T not divisible by the minibatch rows: the reference yields a short last batch
  (on_policy.py:81-92)."""
  pf, vf, S, A = _nets("mlp")
  pf_np, vf_np = g.family_weights("mlp")
  opf, ovf = po.sd_to_torch(pf_np, vf_np)
  orc = po.PPOOracle("mlp", opf, ovf, S, batch_size=12, opt_epochs=1)
  orc.current_epoch = 0
  T, E = 7, 4
  roll = synth.make_rollout(8, T, E, S, A, with_img=False, p_term=0.2)
  buf = fill_buffer(roll, T, E)
  agent, logger = make_ppo(pf, vf, buf, A, 12, T * E, 1, device=DEV)
  agent.current_epoch = 0
  np.random.seed(4)
  perm = np.random.permutation(T)
  np.random.seed(4)
  agent.update_per_epoch()
  _, _, infos = orc.update_per_epoch(roll, perm[None])
  assert len(logger.infos) == len(infos) == 3
  for a, b in zip(logger.infos, infos):
    for k in g.INFO_KEYS:
      assert abs(a[k] - b[k]) <= 1e-5 + 2e-3 * abs(b[k]), (k, a[k], b[k])


def test_state_dict_roundtrip_and_snapshot(tmp_path):
  pf, vf, S, A = _nets("loco")
  agent, _ = make_ppo(pf, vf, None, A, 16, 16, 1, device=DEV)
  agent.engine                                   # flatten parameters into the bucket
  sd = {k: v.clone() for k, v in pf.state_dict().items()}
  agent.snapshot(str(tmp_path), "t")
  loaded = torch.load(str(tmp_path / "model_pf_t.pth"))
  assert list(loaded.keys()) == list(sd.keys())
  pf2, _ = build_nets("loco", S, A)
  pf2.load_state_dict(loaded)                    # loads into a fresh (CPU) module: plain tensors
  for k in sd:
    assert torch.equal(loaded[k].cpu(), sd[k].cpu())
  # loading INTO the flattened module keeps the views
  pf.load_state_dict({k: v * 0 + 1 for k, v in sd.items()})
  agent.engine.check_views()
  assert float(agent.engine.pf_flat.sum()) > 0
