"""The reference's own code on the B200 engine (VERDICT r01 item 2, SURVEY.md §7 step 3).

``oracle/_ref`` holds the UNMODIFIED reference package (oracle/install_reference.py); ``mjlab_b200.compat``
supplies ``mujoco_warp`` / ``warp`` / ``mujoco`` over libb2sim.so.  Executed from the reference's files:
``mjlab.sim.sim.Simulation`` + ``WarpBridge``/``TorchArray`` (sim/sim.py, sim/sim_data.py), ``expand_model_fields``
(sim/randomization.py), ``Entity.initialize`` / ``_compute_indexing`` / ``EntityData`` (entity/entity.py,
entity/data.py), the event functions of envs/mdp/events.py and ``NanGuard`` (utils/nan_guard.py).
Restated reference tests: tests/test_entity.py:269-388 (root velocity frames), tests/test_domain_randomization.py
(per-world fields reach the engine), tests/test_sim_data / test_nan_guard semantics.
"""

import sys
import types
from pathlib import Path

import numpy as np
import pytest
import torch

import refload
from util import load_oracle, make_states, relerr

pytestmark = [pytest.mark.skipif(not refload.available(), reason="oracle/_ref not installed")]

N = 16


@pytest.fixture(scope="module")
def ref():
  return refload.load()


@pytest.fixture(scope="module", params=[pytest.param("cuda", marks=pytest.mark.gpu), "emul"])
def DEV(request, ref):
  """"cuda": libb2sim.so on the GPU.  "emul": the same sources compiled for the host (tests/emul) behind the same
  compat modules, so the CPU suite runs the reference's code against the product's kernels too."""
  if request.param == "cuda":
    yield "cuda:0"
    return
  import mjlab_b200.compat.mujoco_warp_shim as mw
  from mjlab_b200.sim import native

  sys.path.insert(0, str(Path(__file__).parent / "emul"))
  from engine import EmulEngine

  mp = pytest.MonkeyPatch()
  mp.setattr(mw, "_Engine", EmulEngine)
  mp.setattr(native, "check", lambda rc: (_ for _ in ()).throw(RuntimeError("b2sim call failed")) if rc else None)
  yield "cpu"
  mp.undo()


def _sync(dev):
  if dev != "cpu":
    torch.cuda.synchronize()


@pytest.fixture(scope="module")
def world(ref, g1_model, DEV):
  """Reference Simulation + reference Entity (initialised by the reference's own code) on the G1 flat scene."""
  import mujoco  # the compat stand-in (or the real module where it exists)

  m = g1_model
  sim = ref.sim.Simulation(N, ref.sim.SimulationCfg(nconmax=140_000 * N // 4096 + 64 * N, njmax=300), m, DEV)
  E = ref.entity
  key = m.keys["robot/init_state"]
  ent = E.Entity.__new__(E.Entity)  # Entity.__init__ edits an MjSpec; the scene here is already compiled
  jn = [n.split("/")[-1] for n in m.names["joint"][1:]]
  ent.cfg = E.EntityCfg(
    init_state=E.EntityCfg.InitialStateCfg(
      pos=tuple(key["qpos"][0:3]), rot=tuple(key["qpos"][3:7]),
      joint_pos={n: float(v) for n, v in zip(jn, key["qpos"][7:])}),
    articulation=E.EntityArticulationInfoCfg(soft_joint_pos_limit_factor=0.9))
  ent._spec = mujoco.EntitySpecView(m, "robot/")
  ent._free_joint = ent._spec.joints[0]
  ent._non_free_joints = tuple(ent._spec.joints[1:])
  ent.initialize(sim.mj_model, sim.model, sim.data, DEV)  # reference code: indexing + EntityData

  class SceneStub:  # what events.py reads from `env.scene`: entity lookup and the env origins
    env_origins = torch.zeros(N, 3, device=DEV)
    entities = {"robot": ent}

    def __getitem__(self, k):
      return self.entities[k]

  env = types.SimpleNamespace(sim=sim, device=DEV, num_envs=N, scene=SceneStub())
  return types.SimpleNamespace(sim=sim, ent=ent, env=env, model=m)


def _load_state(sim, st, DEV):
  for k, v in st.items():
    getattr(sim.data, k)[:] = torch.as_tensor(v, dtype=torch.float32, device=DEV)


def test_reference_simulation_steps_the_engine(ref, world, DEV):
  """reference Simulation.step()/forward() (CUDA-graph path included) == oracle and == this repo's Simulation."""
  from mjlab_b200.sim import Simulation, SimulationCfg
  from oracle.oracle import Oracle

  sim, m = world.sim, world.model
  assert type(sim).__module__ == "mjlab.sim.sim" and type(sim.data).__module__ == "mjlab.sim.sim_data"
  gpu = DEV != "cpu"
  if gpu:
    assert sim.use_cuda_graph and sim.step_graph is not None  # wp.ScopedCapture -> torch CUDA graph of b2_step
  else:
    assert not sim.use_cuda_graph and sim.step_graph is None
  st = make_states(m, N, seed=77)
  mine = Simulation(N, SimulationCfg(nconmax=140_000 * N // 4096 + 64 * N, njmax=300), m, DEV) if gpu else None
  maxcon = int(mine.get_option("maxcon")) if gpu else max(16, min(96, -(-(140_000 * N // 4096 + 64 * N) // N)))
  o = Oracle(m, nworld=N, maxcon=maxcon)
  load_oracle(o, st)
  _load_state(sim, st, DEV)
  if gpu:
    for k, v in st.items():
      getattr(mine.data, k)[:] = torch.as_tensor(v, dtype=torch.float32, device=DEV)
    mine.forward()
  sim.forward()
  o.forward()
  _sync(DEV)
  if gpu:
    assert torch.equal(sim.data.xpos[:], mine.data.xpos[:]) and torch.equal(sim.data.qacc[:], mine.data.qacc[:])
  assert relerr(sim.data.xpos[:].cpu().numpy().reshape(N, -1), o.xpos).max() < 1e-5
  for _ in range(3):
    sim.step()
    if gpu:
      mine.step()
    o.step()
  _sync(DEV)
  if gpu:
    assert torch.equal(sim.data.qpos[:], mine.data.qpos[:]) and torch.equal(sim.data.qvel[:], mine.data.qvel[:])
    mine.close()
  assert relerr(sim.data.qpos[:].cpu().numpy(), o.qpos).max() < 1e-4
  assert np.median(relerr(sim.data.qvel[:].cpu().numpy(), o.qvel)) < 1e-4
  assert float(sim.data.time[0]) == pytest.approx(3 * float(m.opt_timestep))


def test_reference_bridge_semantics(ref, world, DEV):
  """sim/sim_data.py behaviour on engine memory: zero-copy views, cache, read-only bridge, torch functions."""
  sim = world.sim
  TorchArray = ref.sim_data.TorchArray
  q = sim.data.qpos
  assert isinstance(q, TorchArray) and q is sim.data.qpos  # cached wrapper
  assert q.shape == (N, 36) and q._tensor.data_ptr() == sim.wp_data.qpos.ptr  # shares engine memory
  q[:, 2] = 1.25
  assert torch.all(sim.data.qpos[:, 2] == 1.25)
  assert torch.allclose(torch.sum(q, dim=1), q[:].sum(dim=1))  # __torch_function__
  assert (q * 2.0)[0, 2].item() == 2.5 and (q > 100).sum().item() == 0
  with pytest.raises(AttributeError, match="read-only"):
    sim.data.qpos = torch.zeros(N, 36, device=DEV)
  with pytest.raises(ValueError, match="Fields not found in model"):
    sim.expand_model_fields(["no_such_field"])
  # model fields are shared by all worlds (leading stride 0) until expanded
  assert sim.wp_model.body_mass.strides[0] == 0 and sim.model.body_mass.shape[0] == N


def test_reference_entity_indexing_and_data(ref, world, DEV):
  """Entity._compute_indexing / initialize / EntityData (reference code) against this repo's EntityData and the
  qualitative checks of the reference's tests/test_entity.py:269-388."""
  from mjlab_b200.entity_data import EntityData as Mine
  from mjlab_b200.entity_data import EntityIndexing as MyIndexing

  sim, ent, m = world.sim, world.ent, world.model
  ix = ent.indexing
  assert ix.root_body_id == m.names["body"].index("robot/pelvis")
  assert ix.joint_q_adr.tolist() == list(range(7, 36)) and ix.free_joint_v_adr.tolist() == list(range(6))
  assert ix.ctrl_ids.tolist() == list(range(29)) and len(ix.geom_ids) == 68 and len(ix.body_ids) == 30
  assert set(ix.sensor_adr) == {"left_foot_ground_contact", "right_foot_ground_contact"}
  st = make_states(m, N, seed=78)
  _load_state(sim, st, DEV)
  sim.forward()
  d = ent.data
  mine = Mine(MyIndexing.from_model(m, "robot", DEV), sim.data, sim.model, DEV, N)
  broken = []
  for name in ("root_link_pose_w", "root_link_vel_w", "root_com_pose_w", "root_com_vel_w", "body_link_pose_w",
               "body_link_vel_w", "body_com_pose_w", "body_com_vel_w", "joint_pos", "joint_vel", "projected_gravity_b",
               "heading_w", "root_link_lin_vel_b", "root_link_ang_vel_b", "root_com_lin_vel_b", "geom_pos_w", "site_pos_w",
               "root_link_pos_w", "root_com_pos_w", "body_link_quat_w", "body_com_lin_vel_w", "geom_quat_w"):
    try:
      a = getattr(d, name)
    except Exception as e:  # noqa: BLE001
      broken.append((name, type(e).__name__))
      continue
    b = getattr(mine, name)
    if name.endswith("quat_w"):  # q and -q are the same rotation (the two quat_from_matrix branches differ in sign)
      b = torch.where((a * b).sum(-1, keepdim=True) < 0, -b, b)
    assert a.shape == b.shape and torch.allclose(a, b, atol=1e-5), name
  # entity/data.py:211-219 multiplies a (N, 4) by a (1, N, 4) quaternion batch, which its own quat_mul rejects for
  # every model layout: root_com_pose_w (and the slices taken from it) cannot be evaluated upstream either
  assert {n for n, _ in broken} <= {"root_com_pose_w", "root_com_pos_w", "root_com_quat_w"}, broken
  # test_entity.py:292-298 — a spinning, translating base: link velocity differs from com velocity by w x r
  qv = torch.zeros(N, 35, device=DEV)
  qv[:, 0:3] = torch.tensor([1.0, 0.0, 0.0], device=DEV)
  qv[:, 3:6] = torch.tensor([0.0, 0.0, 2.0], device=DEV)  # body-frame angular velocity (events.py:87,142)
  sim.data.qvel[:] = qv
  sim.forward()
  lin_link, lin_com = d.root_link_lin_vel_w, d.root_com_lin_vel_w
  off = sim.data.xipos[:, ix.root_body_id] - d.root_link_pos_w
  ang = d.root_link_ang_vel_w
  assert torch.allclose(lin_com, lin_link + torch.cross(ang, off, dim=-1), atol=1e-4)
  assert torch.allclose(d.root_link_lin_vel_w[:, :], sim.data.qvel[:, 0:3], atol=1e-5)  # free-joint lin vel is world frame
  # write -> read round trip through the reference writers (test_entity.py:317-330)
  pose = d.root_link_pose_w.clone()
  pose[:, 0] += 0.5
  ent.write_root_link_pose_to_sim(pose, env_ids=torch.arange(N, device=DEV))
  sim.forward()
  assert torch.allclose(d.root_link_pose_w, pose, atol=1e-6)


def test_reference_events_drive_the_engine(ref, world, DEV):
  """envs/mdp/events.py: reset_root_state_uniform, reset_joints_by_scale, push_by_setting_velocity,
  apply_external_force_torque run unmodified against sim.data through the reference Entity."""
  ev, sim, ent, env = ref.events, world.sim, world.ent, world.env
  SceneEntityCfg = ref.scene_entity_config.SceneEntityCfg
  ids = torch.tensor([1, 3, 5], device=DEV)
  before = sim.data.qpos[:].clone()
  torch.manual_seed(0)
  ev.reset_root_state_uniform(env, ids, pose_range={"x": (-0.5, 0.5), "y": (-0.5, 0.5), "yaw": (-3.14, 3.14)},
                              velocity_range={})
  ev.reset_joints_by_scale(env, ids, position_range=(1.0, 1.0), velocity_range=(0.0, 0.0))
  sim.forward()
  key = world.model.keys["robot/init_state"]["qpos"]
  q = sim.data.qpos[:]
  assert torch.allclose(q[ids, 2], torch.full((3,), float(key[2]), device=DEV), atol=1e-6)
  assert ((q[ids, 0:2] - torch.tensor(key[0:2], device=DEV, dtype=torch.float32)).abs() <= 0.5).all()
  assert torch.allclose(q[ids, 3:7].norm(dim=1), torch.ones(3, device=DEV), atol=1e-5)
  lo, hi = ent.data.soft_joint_pos_limits[ids, :, 0], ent.data.soft_joint_pos_limits[ids, :, 1]
  assert ((q[ids, 7:] >= lo - 1e-6) & (q[ids, 7:] <= hi + 1e-6)).all()
  others = torch.tensor([i for i in range(N) if i not in (1, 3, 5)], device=DEV)
  assert torch.equal(q[others], before[others])
  assert (sim.data.qvel[ids] == 0).all()
  # push: world-frame velocity delta, written back in the free joint's mixed frame
  ev.push_by_setting_velocity(env, ids, velocity_range={"x": (0.5, 0.5), "y": (-0.25, -0.25)})
  sim.forward()
  assert torch.allclose(ent.data.root_link_lin_vel_w[ids, 0:2], torch.tensor([0.5, -0.25], device=DEV).expand(3, 2), atol=1e-5)
  # external wrench on two bodies reaches xfrc_applied and changes the engine's accelerations
  sim.forward()
  a0 = sim.data.qacc[:].clone()
  cfg = SceneEntityCfg("robot", body_names=["torso_link", "pelvis"])
  cfg.resolve(env.scene)
  ev.apply_external_force_torque(env, ids, force_range=(50.0, 50.0), torque_range=(0.0, 0.0), asset_cfg=cfg)
  gid = [world.model.names["body"].index(f"robot/{b}") for b in ("pelvis", "torso_link")]
  assert torch.allclose(sim.data.xfrc_applied[ids][:, gid, 0:3], torch.full((3, 2, 3), 50.0, device=DEV))
  sim.forward()
  assert (sim.data.qacc[ids] - a0[ids]).abs().max() > 1.0 and torch.equal(sim.data.qacc[others], a0[others])
  ent.clear_state()
  assert (sim.data.xfrc_applied[:] == 0).all()


def test_reference_domain_randomization_reaches_the_engine(ref, world, DEV):
  """tests/test_domain_randomization.py restated: expand_model_fields (repeat_array_kernel via wp.launch) +
  randomize_field write per-world friction that the physics then uses."""
  ev, sim, ent, env, m = ref.events, world.sim, world.ent, world.env, world.model
  SceneEntityCfg = ref.scene_entity_config.SceneEntityCfg
  # (read through the struct: the bridge caches wrappers by name, and a wrapper made before the expansion would
  # keep pointing at the shared array — the reference expands before anything reads the field, for the same reason)
  import warp as wp

  shared = wp.to_torch(sim.wp_model.geom_friction).clone()
  sim.expand_model_fields(["geom_friction"])
  sim.create_graph()  # the reference re-captures after expansion (model arrays moved)
  gf = sim.model.geom_friction
  assert sim.wp_model.geom_friction.strides[0] > 0 and gf.shape == (N, int(m.ngeom), 3)
  assert torch.equal(gf[:], shared)  # tiled copy of the shared values
  cfg = SceneEntityCfg("robot", geom_names=[".*_foot[1-7]_collision"])
  cfg.resolve(env.scene)
  assert len(cfg.geom_ids) == 14
  torch.manual_seed(1)
  ev.randomize_field(env, None, "geom_friction", ranges=(0.3, 1.2), operation="abs", asset_cfg=cfg)
  feet = ent.indexing.geom_ids[cfg.geom_ids].long()
  mu = sim.model.geom_friction[:, feet, 0]
  assert mu.min() >= 0.3 and mu.max() <= 1.2 and mu.std() > 0.05
  assert torch.equal(sim.model.geom_friction[:, feet, 1:], shared[:, feet, 1:])  # only axis 0 was touched
  # the engine reads the per-world values: same sliding state, friction 0.05 vs 1.5 -> different tangential decel
  key = m.keys["robot/init_state"]
  q = torch.tensor(key["qpos"], dtype=torch.float32, device=DEV).repeat(N, 1)
  q[:, 2] -= 0.005
  sim.data.qpos[:] = q
  v = torch.zeros(N, 35, device=DEV)
  v[:, 0] = 1.0
  sim.data.qvel[:] = v
  sim.data.ctrl[:] = torch.tensor(key["ctrl"], dtype=torch.float32, device=DEV)
  sim.model.geom_friction[0, feet, 0] = 0.05
  sim.model.geom_friction[1, feet, 0] = 1.5
  sim.forward()
  assert int(sim.data.ncon[0]) >= 4
  # same state, friction 0.05 vs 1.5: the sliding feet pull on the base very differently
  assert abs(float(sim.data.qacc[0, 0]) - float(sim.data.qacc[1, 0])) > 1.0


def test_reference_nan_guard_on_engine_state(ref, world, DEV, tmp_path):
  """utils/nan_guard.py (reference) watches Simulation.step through the bridge and dumps on the first NaN."""
  m = world.model
  cfg = ref.sim.SimulationCfg(nan_guard=ref.nan_guard.NanGuardCfg(enabled=True, buffer_size=4, output_dir=str(tmp_path)))
  sim = ref.sim.Simulation(4, cfg, m, DEV)
  sim.step()
  sim.data.qvel[2, 7] = float("nan")
  sim.step()
  _sync(DEV)
  dumps = list(tmp_path.glob("nan_dump_*.npz"))
  assert len(dumps) == 1
  z = np.load(dumps[0], allow_pickle=True)
  meta = z["_metadata"].item()
  assert meta["nan_env_ids"] == [2] and meta["state_size"] == 36 + 35
  assert z["states_step_000001"].shape == (4, 71)
