"""Host-side logic of mjlab_b200.compat (no GPU): the stand-in modules register only when the real ones are
absent, the reference's own sim-layer files import and run against them (oracle/_ref, unmodified), and the
pieces that need no engine — wp.array views, the vectorised wp.launch, TorchArray/WarpBridge over CPU tensors,
the MjModel accessors and the entity spec view — behave as the reference code expects."""

import types

import numpy as np
import pytest
import torch

import refload

pytestmark = pytest.mark.skipif(not refload.available(), reason="oracle/_ref not installed (oracle/install_reference.py)")


@pytest.fixture(scope="module")
def ref():
  return refload.load()


def test_reference_modules_load_from_their_own_files(ref):
  import mujoco, mujoco_warp, warp

  for mod in (mujoco, mujoco_warp, warp):
    assert getattr(mod, "__b2_compat__", False) or mod.__name__ in ("mujoco", "mujoco_warp", "warp")
  assert ref.sim.Simulation.__module__ == "mjlab.sim.sim"
  assert "oracle/_ref/mjlab/envs/mdp/events.py" in ref.events.__file__.replace("\\", "/")
  assert mujoco.mjtJoint.mjJNT_FREE == 0 and mujoco.mjtGeom.mjGEOM_BOX == 6 and mujoco.mjtObj.mjOBJ_XBODY == 2


def test_expand_model_fields_runs_the_reference_kernel(ref):
  """sim/randomization.py: tile() + wp.launch(repeat_array_kernel) on shared [nworld, n, k] arrays (stride 0)."""
  import warp as wp

  nworld = 3
  base = torch.arange(12, dtype=torch.float32).reshape(1, 4, 3)
  shared = wp.array(base.expand(nworld, 4, 3))
  assert shared.strides[0] == 0 and shared.shape == (nworld, 4, 3)

  class FakeModel:
    __dataclass_fields__ = {"geom_friction": None, "body_mass": None}

  m = FakeModel()
  m.geom_friction = shared
  m.body_mass = wp.array(torch.ones(1, 5).expand(nworld, 5))
  ref.randomization.expand_model_fields(m, nworld, ["geom_friction"])
  out = wp.to_torch(m.geom_friction)
  assert out.shape == (nworld, 4, 3) and out.stride(0) == 12 and torch.equal(out, base.expand(nworld, 4, 3))
  assert m.body_mass.strides[0] == 0  # untouched


def test_torcharray_and_bridge_over_cpu_arrays(ref):
  import warp as wp

  t = torch.zeros(4, 6)
  arr = ref.sim_data.TorchArray(wp.array(t))
  arr[:, 1] = 2.0
  assert t[:, 1].eq(2).all() and torch.sum(arr).item() == 8.0 and (arr + 1)[0, 0] == 1
  struct = types.SimpleNamespace(qpos=wp.array(t), nworld=4, opt=types.SimpleNamespace(ls_parallel=True))
  br = ref.sim_data.WarpBridge(struct)
  assert br.qpos is br.qpos and br.nworld == 4 and br.opt.ls_parallel is True
  with pytest.raises(AttributeError, match="read-only"):
    br.qpos = 1


def test_mjmodel_accessors_and_spec_view(g1_model):
  import mujoco

  m = g1_model
  j = m.joint("robot/left_knee_joint")
  assert j.type[0] == mujoco.mjtJoint.mjJNT_HINGE and j.qposadr[0] == j.dofadr[0] + 1
  s = m.sensor("robot/left_foot_ground_contact")
  assert s.dim[0] >= 1 and s.adr[0] == 0
  assert hasattr(m, "geom_friction") and not hasattr(m, "no_such_field") and m.na == 0
  v = mujoco.EntitySpecView(m, "robot/")
  assert len(v.bodies) == 31 and len(v.joints) == 30 and len(v.geoms) == 68 and len(v.actuators) == 29
  assert v.bodies[1].name == "robot/pelvis" and v.bodies[1].id == 2
  assert v.joints[0].type == mujoco.mjtJoint.mjJNT_FREE


def test_reference_simulation_refuses_to_run_without_cuda(ref, g1_model):
  if torch.cuda.is_available():
    pytest.skip("CUDA present")
  with pytest.raises(RuntimeError, match="no CUDA device"):
    ref.sim.Simulation(2, ref.sim.SimulationCfg(), g1_model, "cpu")
