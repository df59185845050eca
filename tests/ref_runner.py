"""Run test files of the reference (unmodified, under oracle/_ref/tests) against this repo's
stand-ins: ``mujoco`` / ``mujoco_warp`` / ``warp`` from mjlab_b200.compat, ``mjlab`` from oracle/_ref (tests/refload.py),
and - there being no GPU in the container - the engine compiled for the host (tests/emul/engine.py) behind the
``mujoco_warp`` stand-in.  Used by tests/test_reference_own_tests.py:  python tests/ref_runner.py <pytest args>
On a GPU box `B2_REF_DEVICE=cuda:0 python tests/ref_runner.py tests/ref_env_cases.py` runs the env cases on libb2sim.so
(tools/gpu_round.sh does; not part of `-m gpu` until it has been seen green there)."""
import os
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
sys.path[:0] = [str(HERE.parent), str(HERE), str(HERE / "emul"), str(HERE / "stubs")]  # stubs: prettytable stand-in
if not os.environ.get("B2_REF_DEVICE", "cpu").startswith("cuda"):
  # the host-emulated engine takes host tensors; the reference's tests pick cuda:0 whenever torch sees a GPU
  os.environ["CUDA_VISIBLE_DEVICES"] = ""

import mjlab_b200.compat as compat  # noqa: E402
import refload  # noqa: E402

compat.install()
sys.path.insert(0, str(refload.REF))
# Packages of the image-less RL / viewer stack that mjlab.envs and mjlab.tasks import at module level: empty modules
# whose attributes are placeholder types (nothing of them is called by the tests); tests/stubs holds the two that
# are used for real (gymnasium base classes / spaces / registry, prettytable).  The viewer package is entered as a
# namespace stub (its __init__ pulls in the interactive viewers) with the one config class the task configs need.
import types  # noqa: E402

mj = sys.modules["mujoco"]
mj.__path__ = []
mj.__getattr__ = lambda k: type(k, (), {})  # annotations such as `mujoco.Renderer` in viewer/offscreen_renderer.py
for name in ("mujoco.viewer", "viser", "viser.transforms", "trimesh", "tyro", "tyro.conf", "moviepy", "wandb", "rsl_rl",
             "rsl_rl.env", "rsl_rl.env.vec_env", "rsl_rl.runners", "onnx", "tensordict", "tqdm", "mediapy"):
  if name not in sys.modules:
    try:
      __import__(name)
    except Exception:  # noqa: BLE001
      m = types.ModuleType(name)
      m.__path__ = []
      m.__getattr__ = lambda k: type(k, (), {})
      sys.modules[name] = m
vw = types.ModuleType("mjlab.viewer")
vw.__path__ = [str(refload.REF / "mjlab" / "viewer")]
sys.modules["mjlab.viewer"] = vw
from mjlab.viewer.viewer_config import ViewerConfig  # noqa: E402

vw.ViewerConfig = ViewerConfig
for pkg in ("mjlab.managers", "mjlab.scene", "mjlab.envs"):  # real packages where they import (refload stubs the rest)
  try:
    __import__(pkg)
  except Exception:  # noqa: BLE001
    for k in [k for k in sys.modules if k == pkg or k.startswith(pkg + ".")]:
      sys.modules.pop(k, None)
refload.load()

import mjlab_b200.compat.mujoco_warp_shim as mw  # noqa: E402
from engine import EmulEngine  # noqa: E402
from mjlab_b200.sim import native  # noqa: E402

if not os.environ.get("B2_REF_DEVICE", "cpu").startswith("cuda"):  # (on a GPU box: the real engine, libb2sim.so)
  mw._Engine = EmulEngine


def _check(rc):
  if rc:
    raise RuntimeError("b2sim call failed")


if not os.environ.get("B2_REF_DEVICE", "cpu").startswith("cuda"):
  native.check = _check

import pytest  # noqa: E402

# confcutdir: collection starts at the repository, not at the filesystem root (whose directories may be unreadable)
sys.exit(pytest.main(["-q", "-c", "/dev/null", "--confcutdir", str(HERE.parent), "-p", "no:cacheprovider", *sys.argv[1:]]))
