"""Checkpoint wire format (SURVEY 8(f) N2): what RLAlgo.snapshot writes must stay loadable by the untouched
reference (viewers, TensorRT export): `model_{pf,vf}_{epoch}.pth` = plain state_dicts with the reference's keys,
`_obs_normalizer_{epoch}.pkl` = a pickled torchrl.env.base_wrapper.Normalizer (reference rl_algo.py:84-95).

The fixture tests/golden/obs_normalizer_ref.pkl was written by the live reference (oracle/make_golden_obs.py).
tests/golden/checkpoint_wire.npz records what the live reference did with OUR files (oracle/make_golden_wire.py):
the bytes of our normaliser pickle it loaded and what it computed from them, the key order / shapes / dtypes of its
modules after a strict load of our state_dicts and their forward outputs."""
import io
import os
import pickle

import numpy as np
import pytest
import torch

from tests import _golden as g
from vision4leg_b200 import obs_pipeline as op

WIRE = os.path.join(g.GOLDEN_DIR, "checkpoint_wire.npz")


def _globals(stream):
  """(module, name) of every class / function a pickle names, as the unpickler resolves them"""
  seen = []

  class Rec(op._WireUnpickler):
    def find_class(self, module, name):
      seen.append((module, name))
      return super().find_class(module, name)
  Rec(io.BytesIO(stream)).load()
  return seen


class _DeviceStandIn:
  """the device Normalizer's pickling hook without a device: same __reduce__, statistics from the fixture"""
  __reduce__ = op.Normalizer.__reduce__

  def __init__(self, st):
    self.st = st

  def to_reference(self):
    return op.reference_normalizer_object(**{k.lstrip("_") if k in ("_mean", "_var", "_count") else k: v
                                             for k, v in self.st.items()})


def test_reference_pickle_fixture_loads_without_the_reference():
  G = np.load(os.path.join(g.GOLDEN_DIR, "obs_normalizer.npz"))
  with open(os.path.join(g.GOLDEN_DIR, "obs_normalizer_ref.pkl"), "rb") as f:
    st = op.load_reference_normalizer(f)
  assert list(st.keys()) == ["shape", "_mean", "_var", "_count", "clip", "should_estimate"]
  assert np.array_equal(st["_mean"], G["mean"]) and np.array_equal(st["_var"], G["var"])
  assert st["_count"] == float(G["count"]) and st["clip"] == 10.0 and st["should_estimate"] is False


def test_our_pickle_names_only_the_reference_class():
  with open(os.path.join(g.GOLDEN_DIR, "obs_normalizer_ref.pkl"), "rb") as f:
    raw = f.read()
  st = op.load_reference_normalizer(io.BytesIO(raw))
  for obj in (op.reference_normalizer_object(st["shape"], st["_mean"], st["_var"], st["_count"], st["clip"],
                                             st["should_estimate"]), _DeviceStandIn(st)):
    mine = pickle.dumps(obj)
    assert b"vision4leg_b200" not in mine
    names = _globals(mine)
    assert op.REFERENCE_NORMALIZER in names
    assert {m.split(".")[0] for m, _ in names} <= {"torchrl", "numpy", "copyreg", "builtins"}, names
    back = op.load_reference_normalizer(io.BytesIO(mine))
    assert list(back.keys()) == list(st.keys())
    for k in st:
      assert np.array_equal(back[k], st[k]), k
  # the plain object pickles to the very bytes the reference wrote (same class path, attribute order, protocol)
  assert pickle.dumps(op.reference_normalizer_object(st["shape"], st["_mean"], st["_var"], st["_count"], st["clip"],
                                                     st["should_estimate"])) == raw


def normalizer_case():
  """(bytes of the `_obs_normalizer_7.pkl` we write for a device normaliser with these statistics, filter input)"""
  rng = np.random.RandomState(3)
  mean, var = rng.randn(37), rng.rand(37) + 0.5
  raw = pickle.dumps(_DeviceStandIn(dict(shape=(37,), _mean=mean, _var=var, _count=123.0001, clip=10.,
                                         should_estimate=True)))
  return raw, rng.randn(4, 37)


def save_state_dicts(family, d):
  """model_{pf,vf}_3.pth the way RLAlgo.snapshot writes them, for the family's fixture weights"""
  from benchutil.harness import build_nets, load_np_sd
  S, A = g.FAMILIES[family]
  pf, vf = build_nets(family, S, A)
  pf_np, vf_np = g.family_weights(family)
  load_np_sd(pf, pf_np); load_np_sd(vf, vf_np)
  for name, net in (("pf", pf), ("vf", vf)):
    torch.save({k: v.detach().clone() for k, v in net.state_dict().items()}, os.path.join(d, "model_%s_3.pth" % name))
  return pf_np, vf_np


def test_live_reference_loads_our_normalizer_pickle():
  """the reference unpickled these very bytes as its own Normalizer and filtered with the statistics they carry"""
  W = np.load(WIRE)
  raw, x = normalizer_case()
  assert raw == W["norm/pickle"].tobytes()
  rng = np.random.RandomState(3)
  mean, var = rng.randn(37), rng.rand(37) + 0.5
  assert float(W["norm/count"]) == 123.0001
  want = np.clip((x - mean) / (np.sqrt(var) + 1e-4), -10, 10)
  assert np.array_equal(W["norm/filt"], want)


@pytest.mark.parametrize("family", ["loco", "mlp"])
def test_live_reference_loads_our_state_dicts(tmp_path, family):
  """model_{pf,vf}_{epoch}.pth written the way RLAlgo.snapshot writes them carry the reference's keys, in its order,
  with its shapes and dtypes (what its strict load_state_dict took), holding the fixture weights under those keys; the
  reference's modules loaded from them reproduce the reference's forward fixture"""
  W = np.load(WIRE)
  G = g.load(family)
  weights = dict(zip(("pf", "vf"), save_state_dicts(family, str(tmp_path))))
  for name in ("pf", "vf"):
    sd = torch.load(str(tmp_path / ("model_%s_3.pth" % name)), map_location="cpu")
    assert list(sd.keys()) == list(W["sd/%s/%s/keys" % (family, name)])
    assert [",".join(map(str, v.shape)) for v in sd.values()] == list(W["sd/%s/%s/shapes" % (family, name)])
    assert [str(v.dtype) for v in sd.values()] == list(W["sd/%s/%s/dtypes" % (family, name)])
    for k, v in sd.items():
      assert np.array_equal(v.numpy(), weights[name][k]), (name, k)
  assert np.allclose(W["sd/%s/value" % family], G["fwd/value"], rtol=1e-5, atol=1e-6)
  assert np.allclose(W["sd/%s/mean" % family], G["fwd/mean"], rtol=1e-5, atol=1e-6)
