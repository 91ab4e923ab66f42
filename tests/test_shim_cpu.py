"""The `torchrl/` drop-in shim (SURVEY 8(b): the boundary is "whatever starter/ppo_*.py import"): with this
repo BEFORE a reference checkout on the path, the hot-path names resolve to vision4leg_b200 and everything
else falls through to the reference.  The checkout is a stand-in written by the test: a `torchrl/` tree with the
reference's package layout, whose fall-through modules use the same kinds of imports (a relative import of a
sibling the shim does not re-author, an absolute import of a shim-served module).  `gym` need not be installed:
the ten-line stub the oracle tooling uses stands in for it."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# path relative to the checkout -> source
STAND_IN = {
  "torchrl/__init__.py": "",
  "torchrl/algo/__init__.py": "from .on_policy import *\nfrom .off_policy import *\n",
  "torchrl/algo/on_policy/__init__.py": "from .a2c import A2C\nfrom .v_mpo import VMPO\n",
  "torchrl/algo/on_policy/a2c.py": "class A2C:\n  pass\n",
  "torchrl/algo/on_policy/v_mpo.py": "from .a2c import A2C\nimport torchrl.algo.utils as atu\n\n\n"
                                     "class VMPO(A2C):\n  schedule = atu.update_linear_schedule\n",
  "torchrl/algo/off_policy/__init__.py": "class SAC:\n  pass\n",
  "torchrl/algo/utils.py": "",
  "torchrl/networks/__init__.py": "",
  "torchrl/policies/__init__.py": "",
  "torchrl/replay_buffers/__init__.py": "",
  "torchrl/replay_buffers/on_policy.py": "",
}


SCRIPT = r'''
import sys, types
gym = types.ModuleType("gym"); spaces = types.ModuleType("gym.spaces")
class Box:                      # only isinstance(..., gym.spaces.Box) is used (reference rl_algo.py:36)
  def __init__(self, *a, **k): self.shape = k.get("shape", ())
spaces.Box = Box; gym.spaces = spaces
sys.modules["gym"] = gym; sys.modules["gym.spaces"] = spaces
import torchrl, torchrl.algo, torchrl.networks, torchrl.policies
from torchrl.replay_buffers.on_policy import OnPolicyReplayBuffer
ours = lambda o: o.__module__.startswith("vision4leg_b200")
assert ours(torchrl.algo.PPO) and ours(torchrl.algo.A2C), torchrl.algo.PPO.__module__
for n in ("LocoTransformer", "LocoTransformerEncoder", "NatureFuseEncoder", "ImpalaEncoderProjNet", "Net", "MLPBase",
          "NatureEncoder", "TransformerEncoder", "Transformer", "NatureEncoderProjNet"):
  assert ours(getattr(torchrl.networks, n)), n
for n in ("GaussianContPolicyLocoTransformer", "GaussianContPolicyImpalaEncoderProj", "GaussianContPolicyBasicBias"):
  assert ours(getattr(torchrl.policies, n)), n
assert ours(OnPolicyReplayBuffer)
# outside the hot path: served by the reference checkout
VMPO = torchrl.algo.VMPO
assert not ours(VMPO) and REF in sys.modules[VMPO.__module__].__file__, VMPO.__module__
import torchrl.algo.off_policy as off
assert REF in off.__file__
import torchrl.algo.utils as atu
assert hasattr(atu, "update_linear_schedule")
print("shim ok")
'''


def test_torchrl_shim_resolution(tmp_path):
  for rel, src in STAND_IN.items():
    (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
    (tmp_path / rel).write_text(src)
  REF = str(tmp_path)
  env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + REF, V4L_REFERENCE_ROOT=REF, PYTHONDONTWRITEBYTECODE="1")
  out = subprocess.run([sys.executable, "-c", SCRIPT.replace("REF", repr(REF))], env=env, capture_output=True, text=True,
                       timeout=300)
  assert out.returncode == 0 and "shim ok" in out.stdout, out.stdout + out.stderr
