"""CPU checks of the host-side mirror of the reference classes: state_dict keys / parameter
order / seeded initial weights identical to the live reference (golden `init/*` fingerprints),
deepcopy, replay-buffer bookkeeping, minibatch index construction."""
import copy

import numpy as np
import pytest
import torch

from tests import _golden as g
from tests._harness import build_nets, fill_buffer
from oracle import synth


GOLDEN_THREADS = 8       # torch threads oracle/make_golden.py wrote the init fingerprints with


@pytest.mark.parametrize("family", ["loco", "nature", "mlp", "vit", "nvo"])
def test_init_parity_with_reference(family):
  G = g.load(family)
  S, A = g.FAMILIES[family]
  # nn.init.orthogonal_ runs a LAPACK QR whose last bits depend on the thread count: use the golden's count
  threads = torch.get_num_threads()
  torch.set_num_threads(GOLDEN_THREADS)
  try:
    torch.manual_seed(0)
    pf, vf = build_nets(family, S, A)
  finally:
    torch.set_num_threads(threads)
  assert list(pf.state_dict().keys()) == list(G["init/pf_keys"])
  assert list(vf.state_dict().keys()) == list(G["init/vf_keys"])
  assert [k for k, _ in pf.named_parameters()] == list(G["init/pf_param_order"])
  assert [k for k, _ in vf.named_parameters()] == list(G["init/vf_param_order"])
  # bit-identical seeded initialisation (same construction order + same init rules)
  g.check_summary(G, "init/pf", [(k, v.numpy()) for k, v in pf.state_dict().items()], 0.0)
  g.check_summary(G, "init/vf", [(k, v.numpy()) for k, v in vf.state_dict().items()], 0.0)


def test_shared_encoder_and_deepcopy():
  pf, vf = build_nets("loco", 93, 12)
  shared = {id(p) for p in pf.parameters()} & {id(p) for p in vf.parameters()}
  assert len(shared) == len(list(pf.encoder.parameters())) == 14
  t = copy.deepcopy(pf)
  assert type(t) is type(pf)
  assert not ({id(p) for p in t.parameters()} & {id(p) for p in pf.parameters()})
  assert pf.encoder.visual_dim == 64 and pf.encoder.per_modal_tokens == 16
  assert pf.encoder.base.output_shape == 256 and pf.continuous and not pf.tanh_action


def test_unsupported_variants_fail_loudly():
  import vision4leg_b200.networks as networks
  with pytest.raises(NotImplementedError):
    networks.LocoTransformerEncoder(in_channels=16, state_input_dim=8, hidden_shapes=[16])
  enc = networks.LocoTransformerEncoder(in_channels=4, state_input_dim=8, hidden_shapes=[16])
  with pytest.raises(NotImplementedError):
    networks.LocoTransformer(encoder=enc, output_shape=1, state_input_shape=8,
                             visual_input_shape=(4, 64, 64), max_pool=True)


def test_replay_buffer_bookkeeping():
  T, E, S, A = 6, 3, 5, 2
  roll = synth.make_rollout(5, T, E, S, A, with_img=False)
  buf = fill_buffer(roll, T, E)
  assert buf.num_steps_can_sample() == T and buf._top == 0
  assert buf._obs.shape == (T, E, S) and buf._obs.dtype == np.float32
  np.testing.assert_array_equal(buf._obs, roll["obs"])
  last = buf.last_sample(["next_obs", "terminals", "time_limits"])
  np.testing.assert_array_equal(last["next_obs"], roll["last_obs"])
  np.testing.assert_array_equal(last["terminals"], roll["terminals"][-1])
  buf._advs = np.zeros((T, E, 1), np.float32)
  np.random.seed(3)
  perm = np.random.permutation(T)
  np.random.seed(3)
  batches = list(buf.one_iteration(6, ["obs", "acts", "advs"], True))
  assert len(batches) == 3 and batches[0]["obs"].shape == (6, S)
  np.testing.assert_array_equal(batches[0]["acts"], roll["acts"][perm[:2]].reshape(6, A))
  with pytest.raises(AssertionError):
    next(buf.one_iteration(4, ["obs"], False))


def test_replay_buffer_half_image_staging_tracks_add_sample():
  """enable_half_image_staging: rows already stored are converted once, later add_sample calls keep
  the fp16 image copy and the packed proprio copy in step with the fp32 rows (ring overwrite too)."""
  import numpy as np
  from vision4leg_b200.replay_buffers import OnPolicyReplayBuffer
  rng = np.random.default_rng(0)
  T, E, S, I = 5, 2, 3, 8
  buf = OnPolicyReplayBuffer(env_nums=E, max_replay_buffer_size=T * E)
  def sample():
    return {"obs": rng.standard_normal((E, S + I)).astype(np.float32), "next_obs": rng.standard_normal((E, S + I)),
            "acts": rng.standard_normal((E, 2)), "rewards": rng.standard_normal((E, 1))}
  for _ in range(3):
    buf.add_sample(sample())
  buf.enable_half_image_staging(S)
  for _ in range(4):                    # wraps around the ring
    buf.add_sample(sample())
  n = buf.num_steps_can_sample()
  assert n == T
  np.testing.assert_array_equal(buf._obs_img16[:n], buf._obs[:n, :, S:].astype(np.float16))
  np.testing.assert_array_equal(buf._obs_state[:n, :, :S], buf._obs[:n, :, :S])
  assert buf._obs_img16.dtype == np.float16
