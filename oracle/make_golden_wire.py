"""Generate tests/golden/checkpoint_wire.npz: what the LIVE reference does with the checkpoint files this package
writes (build container only).

  PYTHONDONTWRITEBYTECODE=1 python -m oracle.make_golden_wire

Our files are written first, exactly as tests/test_checkpoint_wire_cpu.py writes them; the reference then loads them:
  normaliser : `_obs_normalizer_{epoch}.pkl` unpickled by the reference (torchrl/env/base_wrapper.py loaded on its
               own with a stub `gym`), its class checked, `_count` and `filt(x)` recorded, together with the bytes it
               loaded (the test asserts that we still write those bytes);
  state_dicts: `model_{pf,vf}_{epoch}.pth` loaded with strict=True into the reference's own modules; the reference's
               key order and shapes and its forward outputs on the fixture inputs are recorded.
TEST INFRASTRUCTURE — not imported by the product.
"""
import importlib.util
import os
import pickle
import shutil
import sys
import tempfile
import types

import numpy as np
import torch

from oracle import make_golden as mg
from tests import _golden as g
from tests import test_checkpoint_wire_cpu as wire

FAMILIES = ("loco", "mlp")


def main():
  torch.set_num_threads(8)
  out = {}
  tmp = tempfile.mkdtemp()
  # ---- our files (before the reference takes over sys.path / torchrl.*)
  raw, x = wire.normalizer_case()
  out["norm/pickle"] = np.frombuffer(raw, np.uint8)
  inputs = {}
  for family in FAMILIES:
    os.makedirs(os.path.join(tmp, family))
    wire.save_state_dicts(family, os.path.join(tmp, family))
    inputs[family] = g.fwd_inputs(family)

  # ---- the reference loads them
  gym = types.ModuleType("gym")
  for n in ("Wrapper", "RewardWrapper", "ObservationWrapper"):
    setattr(gym, n, type(n, (), {}))
  sys.modules["gym"] = gym
  spec = importlib.util.spec_from_file_location("torchrl.env.base_wrapper",
                                                os.path.join(mg.REF, "torchrl/env/base_wrapper.py"))
  mod = importlib.util.module_from_spec(spec)
  sys.modules["torchrl.env.base_wrapper"] = mod
  spec.loader.exec_module(mod)
  nz = pickle.loads(raw)
  assert type(nz) is mod.Normalizer, type(nz)
  out["norm/count"] = np.float64(nz._count)
  out["norm/filt"] = nz.filt(x)
  del sys.modules["torchrl.env.base_wrapper"]

  networks, policies, _, _, _ = mg.import_reference()
  for family in FAMILIES:
    S, A = mg.FAMILIES[family]
    pf, vf = mg.build_reference_nets(networks, policies, family, S, A)
    for name, net in (("pf", pf), ("vf", vf)):
      net.load_state_dict(torch.load(os.path.join(tmp, family, "model_%s_3.pth" % name), map_location="cpu"), strict=True)
      sd = net.state_dict()
      out["sd/%s/%s/keys" % (family, name)] = np.array(list(sd.keys()))
      out["sd/%s/%s/shapes" % (family, name)] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
      out["sd/%s/%s/dtypes" % (family, name)] = np.array([str(v.dtype) for v in sd.values()])
    obs, acts = inputs[family]
    with torch.no_grad():
      out["sd/%s/value" % family] = vf(torch.tensor(obs)).numpy()
      out["sd/%s/mean" % family] = pf.update(torch.tensor(obs), torch.tensor(acts))["mean"].numpy()
  shutil.rmtree(tmp)
  np.savez_compressed(os.path.join(mg.OUT, "checkpoint_wire.npz"), **out)
  print("checkpoint_wire.npz", len(out), "arrays")


if __name__ == "__main__":
  main()
