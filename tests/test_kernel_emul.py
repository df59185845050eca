"""The whole product library (b2sim.cu + the fused step kernel) compiled for the host (tests/emul/build.py:
g++ against cuda_emul.h, one warp per CTA, the 32 lanes as fibers on one host thread) and driven through its C ABI —
the same parity checks as tests/test_parity_gpu.py, without a GPU; tolerances are the GPU tests' (fp32 engine vs
fp64 oracle)."""

import ctypes
import sys
from pathlib import Path

import numpy as np
import pytest

from mjlab_b200.sim import native
from oracle.oracle import Oracle
from util import load_oracle, make_states, relerr, terrain_states

sys.path.insert(0, str(Path(__file__).parent / "emul"))


def _load(defines=()):
  from engine import load_emul_library

  return load_emul_library(defines)


@pytest.fixture(scope="module")
def lib():
  return _load()


class EmulSim:
  """ctypes + numpy views over the emulated library ("device" memory is host memory)."""

  def __init__(self, lib, model, nworld, ncon=0):
    self.lib, self.n = lib, nworld
    self.desc, self._keep = native.make_model_desc(model)
    self.h = ctypes.c_void_p()
    rc = lib.b2_create(ctypes.byref(self.desc), nworld, ncon, 0, 0, ctypes.byref(self.h))
    assert rc == 0, lib.b2_last_error(None).decode()
    lib.b2_set_option(self.h, b"debug_outputs", 1.0)
    lib.b2_set_option(self.h, b"sorted_dispatch", 0.0)  # (the 1024-thread sort kernel works but is slow to emulate)

  def field(self, name, which=0):
    t = native.B2Tensor()
    rc = self.lib.b2_get_field(self.h, which, name.encode(), ctypes.byref(t))
    assert rc == 0, name
    dt = {0: np.float32, 1: np.int32}[t.dtype] if t.dtype in (0, 1) else np.float32
    shape = tuple(t.shape[i] for i in range(t.ndim))
    strides = tuple(t.stride[i] * 4 for i in range(t.ndim))
    total = 1 + sum((s - 1) * st for s, st in zip(shape, (t.stride[i] for i in range(t.ndim))))
    buf = (ctypes.c_byte * (total * 4)).from_address(t.ptr)
    return np.ndarray(shape, dtype=dt, buffer=buf, strides=strides)

  def load(self, st):
    for k, v in st.items():
      self.field(k)[...] = v

  def option(self, key):
    v = ctypes.c_double()
    self.lib.b2_get_option(self.h, key.encode(), ctypes.byref(v))
    return v.value

  def forward(self):
    assert self.lib.b2_forward(self.h, None) == 0

  def step(self, n=1):
    assert self.lib.b2_step_n(self.h, n, None) == 0

  def close(self):
    self.lib.b2_destroy(self.h)


def _check_forward(sim, o, n, acc_tol=1e-3):
  nc = o.ncon.ravel()
  assert (sim.field("ncon").ravel() == nc).all() and (sim.field("nefc").ravel() == o.nefc.ravel()).all()
  cg, og = sim.field("contact_geom"), o.contact_geom.reshape(n, -1, 2)
  for w in range(n):
    assert (cg[w, : nc[w]] == og[w, : nc[w]]).all()
    if nc[w]:
      assert np.abs(sim.field("contact_dist")[w, : nc[w]] - o.contact_dist[w, : nc[w]]).max() < 1e-5
  for f in ["xpos", "xquat", "xmat", "xipos", "subtree_com", "cvel", "geom_xpos", "geom_xmat", "site_xpos",
            "actuator_force", "qfrc_bias", "qfrc_smooth", "qM"]:
    e = relerr(np.asarray(sim.field(f)).reshape(n, -1), o.field(f).reshape(n, -1)).max()
    assert e < 1e-5, (f, e)
  assert relerr(sim.field("qacc_smooth"), o.qacc_smooth).max() < 1e-4
  e = relerr(sim.field("qacc"), o.qacc, floor=10.0)
  assert e.max() < acc_tol, e
  assert np.abs(sim.field("sensordata") - o.sensordata).max() < 1e-3


@pytest.mark.parametrize("name,n", [("go1_flat", 4), ("g1_flat", 3)])
def test_emulated_kernel_forward_and_step_parity(lib, name, n):
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled(name)
  sim = EmulSim(lib, m, n)
  # derived fields are valid right after construction (b2_create ran one forward at qpos0)
  assert np.isfinite(sim.field("xpos")).all() and (sim.field("time") == 0).all()
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  st = make_states(m, n, seed=5)
  load_oracle(o, st)
  sim.load(st)
  o.forward()
  sim.forward()
  _check_forward(sim, o, n)
  for _ in range(2):
    o.step()
  sim.step(2)
  assert relerr(sim.field("qpos"), o.qpos).max() < 1e-4
  assert relerr(sim.field("qvel"), o.qvel).max() < 5e-3
  assert sim.field("time").ravel() == pytest.approx(2 * float(m.opt_timestep))
  sim.close()


def test_emulated_kernel_on_stairs_and_masked_forward(lib):
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled("go1_stairs_small")
  n = 4
  sim = EmulSim(lib, m, n)
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  st = terrain_states(m, n, 104, 1.4)
  load_oracle(o, st)
  sim.load(st)
  o.forward()
  sim.forward()
  _check_forward(sim, o, n, acc_tol=2e-3)
  assert int(o.ncon.max()) >= 5  # box terrain contacts through the grid broadphase
  # masked forward: only the selected worlds are recomputed
  before = sim.field("xpos").copy()
  sim.field("qpos")[:, 2] += 1.0
  mask = np.array([0, 1, 0, 1], dtype=np.uint8)
  assert lib.b2_forward_masked(sim.h, mask.ctypes.data_as(ctypes.c_void_p), None) == 0
  after = sim.field("xpos")
  assert (after[0] == before[0]).all() and (after[2] == before[2]).all()
  assert np.abs(after[1, 2:, 2] - before[1, 2:, 2] - 1.0).max() < 1e-5  # (body 1 is the static terrain)
  sim.close()


def test_emulated_kernel_dense_and_tree_schedules_agree(lib):
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled("go1_flat")
  n = 3
  a, b = EmulSim(lib, m, n), EmulSim(lib, m, n)
  lib.b2_set_option(b.h, b"dense_factor", 1.0)
  st = make_states(m, n, seed=9)
  a.load(st)
  b.load(st)
  a.step(1)
  b.step(1)
  assert relerr(a.field("qvel"), b.field("qvel")).max() < 1e-4
  a.close()
  b.close()


def test_emulated_kernel_obstacle_course(lib):
  """Pair table + static grid + all six primitive pair types inside the emulated kernel, a few resynchronised steps."""
  from test_boxes_terrain import obstacle_course_xml

  from mjlab_b200.compiler import Spec

  m = Spec.from_string(obstacle_course_xml()).compile()
  n = 2
  sim = EmulSim(lib, m, n, ncon=96)
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  rng = np.random.default_rng(1)
  q = np.tile(m.qpos0, (n, 1))
  q += rng.uniform(-0.08, 0.08, q.shape) * (np.arange(q.shape[1]) % 7 < 3)
  q[:, 2::7] -= 0.42  # start near the ground so that contacts exist from the first step
  st = dict(qpos=q, qvel=rng.uniform(-0.3, 0.3, (n, int(m.nv))))
  load_oracle(o, st)
  sim.load(st)
  seen = 0
  for it in range(8):
    o.forward()
    sim.forward()
    nc = o.ncon.ravel()
    assert (sim.field("ncon").ravel() == nc).all()
    cg, og = sim.field("contact_geom"), o.contact_geom.reshape(n, -1, 2)
    for w in range(n):
      a = sorted(zip(map(tuple, cg[w, : nc[w]].tolist()), sim.field("contact_dist")[w, : nc[w]].tolist()))
      b = sorted(zip(map(tuple, og[w, : nc[w]].tolist()), o.contact_dist[w, : nc[w]].tolist()))
      assert [x[0] for x in a] == [x[0] for x in b]
      if nc[w]:
        assert np.abs(np.array([x[1] for x in a]) - np.array([x[1] for x in b])).max() < 2e-5
    assert relerr(sim.field("qacc"), o.qacc, floor=10.0).max() < 1e-2
    seen = max(seen, int(nc.max()))
    o.step()
    sim.step(1)
    for f in ("qpos", "qvel", "qacc_warmstart"):
      sim.field(f)[...] = getattr(o, f)
  assert seen >= 6
  sim.close()


def test_emulated_host_entry_and_field_expansion(lib):
  """Two host paths no CPU test could reach before: b2_step_host (host buffers in/out) equals b2_step_n, and an
  expanded per-world model field (geom_friction) is what the kernel reads."""
  from mjlab_b200.asset_zoo import load_compiled

  lib.b2_step_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
  lib.b2_expand_model_field.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.POINTER(native.B2Tensor)]
  m = load_compiled("go1_flat")
  n, nq, nv, nu = 3, int(m.nq), int(m.nv), int(m.nu)
  st = make_states(m, n, seed=21)
  ref, host = EmulSim(lib, m, n), EmulSim(lib, m, n)
  for s in (ref, host):
    s.load(st)
  ref.step(2)
  # host-buffer entry: ctrl from a dense host array, qpos/qvel back into dense host arrays
  ctrl = np.ascontiguousarray(st["ctrl"], dtype=np.float32)
  qpos_out, qvel_out = np.zeros((n, nq), dtype=np.float32), np.zeros((n, nv), dtype=np.float32)
  assert lib.b2_step_host(host.h, ctrl.ctypes.data, 2, qpos_out.ctypes.data, qvel_out.ctypes.data, None) == 0
  assert (qpos_out == ref.field("qpos")).all() and (qvel_out == ref.field("qvel")).all()
  # per-world friction: world 0 keeps the model's value, the others get ice under their feet
  t = native.B2Tensor()
  assert lib.b2_expand_model_field(ref.h, b"geom_friction", None, ctypes.byref(t)) == 0
  fr = ref.field("geom_friction", which=1)
  assert fr.shape[0] == n and fr.strides[0] > 0  # a real leading world dimension now
  st2 = make_states(m, n, seed=22, vel=1.5)
  ref.load(st2)
  ref.forward()
  qa = ref.field("qacc").copy()
  fr[1:, :, 0] = 1e-3
  ref.forward()
  qb = ref.field("qacc")
  assert np.abs(qa[0] - qb[0]).max() == 0.0  # the untouched world: bit-identical
  # (only the feet have condim 3; a world whose contacts are all frictionless would not notice)
  assert max(np.abs(qa[w] - qb[w]).max() for w in range(1, n)) > 1e-3
  for s in (ref, host):
    s.close()


class EmulSimulation:
  """Test double with the slice of `mjlab_b200.sim.Simulation` that VelocityFlatEnv uses, backed by the emulated
  library: fields are torch CPU tensors aliasing the library's (host) memory."""

  def __init__(self, num_envs, cfg, model, device):
    import torch

    self._torch = torch
    self._lib = _load()
    vp = ctypes.c_void_p
    self._lib.b2_velenv_pre.argtypes = [vp, vp, vp, vp, vp]
    self._lib.b2_velenv_post.argtypes = [vp, ctypes.POINTER(native.B2VelEnvArgs), vp]
    self._lib.b2_expand_model_field.argtypes = [vp, ctypes.c_char_p, vp, ctypes.POINTER(native.B2Tensor)]
    self._lib.b2_trackenv_post1.argtypes = [vp, ctypes.POINTER(native.B2TrackEnvArgs), vp]
    self._lib.b2_trackenv_post2.argtypes = [vp, ctypes.POINTER(native.B2TrackEnvArgs), vp]
    self._e = EmulSim(self._lib, model, num_envs, ncon=max(16, min(96, -(-cfg.nconmax // num_envs))) if cfg.nconmax else 0)
    self._h = self._e.h
    self.device = device
    outer = self

    class _Fields:
      def __init__(self, which):
        object.__setattr__(self, "_which", which)

      def __getattr__(self, name):
        try:
          return outer._torch.from_numpy(outer._e.field(name, which=self._which))
        except AssertionError:
          raise AttributeError(name) from None

    self.data, self.model = _Fields(0), _Fields(1)

  def _stream(self):
    return ctypes.c_void_p(0)

  def expand_model_fields(self, fields):
    for f in fields:
      assert self._lib.b2_expand_model_field(self._h, f.encode(), None, None) == 0

  def step_n(self, n):
    self._e.step(n)

  def forward(self, env_mask=None):
    if env_mask is None:
      self._e.forward()
    else:
      assert self._lib.b2_forward_masked(self._h, ctypes.c_void_p(env_mask.data_ptr()), None) == 0

  def close(self):
    self._e.close()


def test_emulated_env_native_mdp_kernels_match_torch_reference(monkeypatch):
  """The velocity env on the emulated library: the fused MDP kernels (b2_velenv_pre / b2_velenv_post) against the
  torch implementation of the same step - terminations, rewards, masked resets, pushes, observations - on CPU."""
  import torch

  import mjlab_b200.envs.velocity_env as ve

  monkeypatch.setattr(ve, "Simulation", EmulSimulation)
  monkeypatch.setattr(native, "check", lambda rc: (_ for _ in ()).throw(RuntimeError("b2sim call failed")) if rc else None)
  cfg = dict(robot="go1", num_envs=6, decimation=2, fall_angle=0.2, push_interval_s=(0.01, 0.03), episode_length_s=0.03)
  a = ve.VelocityFlatEnv(ve.VelocityEnvCfg(**cfg), device="cpu", native_mdp=False)
  b = ve.VelocityFlatEnv(ve.VelocityEnvCfg(**cfg), device="cpu", native_mdp=True)
  assert torch.equal(a.sim.data.qpos[:], b.sim.data.qpos[:])
  g = torch.Generator()
  g.manual_seed(3)
  resets = 0
  for k in range(10):
    act = torch.rand((6, 12), generator=g) * 2 - 1
    oa, ra, ta, ua, _ = a.step(act)
    ob, rb, tb, ub, _ = b.step(act)
    assert torch.equal(ua, ub)
    assert torch.equal(ta, tb)
    assert torch.allclose(ra, rb, atol=1e-4)
    assert torch.allclose(oa, ob, atol=2e-3)
    assert torch.allclose(a.command, b.command, atol=1e-6) and torch.allclose(a.push_time_left, b.push_time_left, atol=1e-6)
    assert torch.equal(a.episode_length_buf, b.episode_length_buf)
    for f in ("qpos", "qvel", "qacc_warmstart", "ctrl"):  # resynchronise: the MDP logic is what is under test
      getattr(b.sim.data, f)[:] = getattr(a.sim.data, f)[:]
    resets += int((ta | ua).sum())
  assert resets >= 6  # time-outs (every 2 steps) exercised the masked reset path
  a.close()
  b.close()


def test_emulated_tracking_env_native_mdp_kernels_match_torch_reference(monkeypatch):
  """The tracking env (config C) on the emulated library: the fused MDP kernels (csrc/b2_trackenv.cuh) against the
  torch implementation of the same step - terminations, rewards, RSI resets, clip restarts, anchor-relative targets,
  pushes, policy and critic observations - on CPU, consuming the same uniforms."""
  import torch

  import mjlab_b200.envs.tracking_env as te

  monkeypatch.setattr(te, "Simulation", EmulSimulation)
  monkeypatch.setattr(native, "check", lambda rc: (_ for _ in ()).throw(RuntimeError("b2sim call failed")) if rc else None)
  cfg = dict(num_envs=4, decimation=1, episode_length_s=0.015, clip_frames=4, push_interval_s=(0.004, 0.012))
  a = te.TrackingFlatEnv(te.TrackingEnvCfg(**cfg), device="cpu", native_mdp=False)
  b = te.TrackingFlatEnv(te.TrackingEnvCfg(**cfg), device="cpu", native_mdp=True)
  assert torch.equal(a.sim.data.qpos[:], b.sim.data.qpos[:])
  g = torch.Generator()
  g.manual_seed(5)
  events = dict(term=0, trunc=0, ended=0, push=0)
  for k in range(8):
    act = torch.rand((4, a.nu), generator=g) * 2 - 1
    if k == 2:  # a fall: the anchor drops below the clip's by more than 0.25 m
      for e in (a, b):
        e.sim.data.qpos[1, 2] -= 0.4
    ts0, ptl0 = a.time_steps.clone(), a.push_time_left.clone()
    oa, ra, ta, ua, xa = a.step(act)
    ob, rb, tb, ub, xb = b.step(act)
    assert torch.equal(ta, tb) and torch.equal(ua, ub), (k, ta, tb, ua, ub)
    assert torch.allclose(ra, rb, atol=2e-5), (k, ra, rb)
    assert torch.equal(a.time_steps, b.time_steps) and torch.equal(a.episode_length_buf, b.episode_length_buf)
    assert torch.allclose(a.push_time_left, b.push_time_left, atol=1e-6)
    assert torch.allclose(a.last_action, b.last_action)
    assert torch.equal(a._done_buf, b._done_buf)
    assert torch.allclose(a.body_pos_relative_w, b.body_pos_relative_w, atol=1e-5)
    assert torch.allclose(a.body_quat_relative_w, b.body_quat_relative_w, atol=1e-5)
    assert torch.allclose(a.log_row, b.log_row, atol=2e-5)
    for f in ("qpos", "qvel", "ctrl"):
      assert torch.allclose(getattr(a.sim.data, f)[:], getattr(b.sim.data, f)[:], atol=1e-5), (k, f)
    assert oa.shape == ob.shape == (4, 160) and xa["critic"].shape == xb["critic"].shape == (4, 286)
    assert torch.allclose(oa, ob, atol=1e-4), (k, (oa - ob).abs().max())
    assert torch.allclose(xa["critic"], xb["critic"], atol=1e-4), (k, (xa["critic"] - xb["critic"]).abs().max())
    events["term"] += int(ta.sum()); events["trunc"] += int(ua.sum())
    events["ended"] += int(((ts0 + 1 >= 4) & ~(ta | ua)).sum()); events["push"] += int((ptl0 - a.step_dt <= 0).sum())
    for f in ("qpos", "qvel", "qacc_warmstart", "ctrl"):  # resynchronise: the MDP logic is what is under test
      getattr(b.sim.data, f)[:] = getattr(a.sim.data, f)[:]
  assert all(v > 0 for v in events.values()), events
  a.close()
  b.close()


def _limb(name, n, pos, axes):
  s, close = "", ""
  for k in range(n):
    p = pos if k == 0 else "0 0 -0.12"
    s += (f'<body name="{name}{k}" pos="{p}"><joint name="{name}j{k}" axis="{axes[k % len(axes)]}" range="-1.2 1.2" '
          f'limited="true" damping="0.2" armature="0.01"/><geom type="capsule" fromto="0 0 0 0 0 -0.12" size="0.03" mass="0.4"/>')
    close += "</body>"
  return s + close


def test_emulated_kernel_synthetic_45dof_robot(lib):
  """Sizes no GPU test reaches: a 45-dof, 41-body floating base with five 7-8 joint limbs, 781 collision pairs,
  self-collisions (dense factorisation schedule), ~40 contacts / ~160 constraint rows per world."""
  from mjlab_b200.compiler import Spec

  xml = f"""<mujoco><compiler angle="radian"/><option timestep="0.004" integrator="implicitfast"/>
  <worldbody><geom name="floor" type="plane" size="0 0 1"/>
  <body name="base" pos="0 0 0.55"><freejoint/><geom type="box" size="0.2 0.15 0.06" mass="4"/>
  {_limb("a", 8, "0.18 0.12 -0.06", ["1 0 0", "0 1 0"])}{_limb("b", 8, "0.18 -0.12 -0.06", ["0 1 0", "1 0 0"])}
  {_limb("c", 8, "-0.18 0.12 -0.06", ["1 0 0", "0 1 0", "0 0 1"])}{_limb("d", 8, "-0.18 -0.12 -0.06", ["0 1 0", "0 0 1"])}
  {_limb("e", 7, "0 0 0.06", ["0 1 0", "1 0 0"])}
  </body></worldbody></mujoco>"""
  m = Spec.from_string(xml).compile()
  assert int(m.nv) == 45 and int(m.nbody) == 41 and int(m.npair) > 500
  n = 2
  sim = EmulSim(lib, m, n, ncon=64)
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  rng = np.random.default_rng(0)
  q = np.tile(m.qpos0, (n, 1))
  q[:, 2] += rng.uniform(-0.25, 0.0, n)
  q[:, 7:] += rng.uniform(-0.9, 0.9, (n, int(m.nq) - 7))
  st = dict(qpos=q, qvel=rng.uniform(-1, 1, (n, 45)), qacc_warmstart=rng.uniform(-1, 1, (n, 45)))
  load_oracle(o, st)
  sim.load(st)
  o.forward()
  sim.forward()
  assert (sim.field("ncon").ravel() == o.ncon.ravel()).all() and int(o.ncon.min()) >= 20
  assert (sim.field("nefc").ravel() == o.nefc.ravel()).all()
  for f in ["xpos", "cvel", "qfrc_bias", "qM"]:
    assert relerr(np.asarray(sim.field(f)).reshape(n, -1), o.field(f).reshape(n, -1)).max() < 1e-5, f
  assert relerr(sim.field("qacc"), o.qacc, floor=10.0).max() < 1e-3
  o.step()
  sim.step(1)
  assert relerr(sim.field("qvel"), o.qvel).max() < 1e-3
  sim.close()


def test_emulated_reduced_solver_matches_full_solver(lib):
  """The Newton solver on the constrained leading block (Schur complement of M onto the dofs any constraint
  touches, the rest by back-substitution) gives the full-size solver's answer."""
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled("g1_flat")
  n = 5
  sim = EmulSim(lib, m, n)
  assert sim.option("reduced_block_cap") == 19
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  st = make_states(m, n, seed=5)
  load_oracle(o, st)
  o.forward()
  res = {}
  for mode, full in (("reduced", 0), ("full", 1)):
    lib.b2_set_option(sim.h, b"full_solver", float(full))
    sim.load(st)
    sim.field("qacc")[...] = 0
    sim.forward()
    res[mode] = (np.array(sim.field("qacc")), np.array(sim.field("qfrc_constraint")))
    assert relerr(res[mode][0], o.qacc).max() < 1e-4, mode
    assert relerr(res[mode][1], o.qfrc_constraint).max() < 1e-4, mode
  assert (o.nefc.ravel() > 0).sum() >= 3
  assert relerr(res["reduced"][0], res["full"][0]).max() < 1e-4
  lib.b2_set_option(sim.h, b"full_solver", 0.0)
  load_oracle(o, st)
  sim.load(st)
  o.step()
  sim.step(1)
  for f in ("qpos", "qvel", "qacc_warmstart"):
    assert relerr(sim.field(f), o.field(f)).max() < 1e-4, f
  sim.close()


def test_emulated_cg_solver_reaches_the_newton_minimiser(lib):
  """opt.solver = CG (mujoco_warp's second solver, `MujocoCfg.solver="cg"`): Polak-Ribiere directions
  preconditioned by the factor of M, same cost / update pass / exact line search - same minimiser as the fp64
  Newton oracle once it is given enough iterations (CG needs tens where Newton needs a handful)."""
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled("go1_flat")
  n = 3
  sim = EmulSim(lib, m, n)
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  o.set_option("iterations", 50)
  st = make_states(m, n, seed=5)
  load_oracle(o, st)
  o.forward()
  lib.b2_set_option(sim.h, b"solver", 1.0)
  lib.b2_set_option(sim.h, b"iterations", 200.0)
  assert sim.option("solver") == 1
  sim.load(st)
  sim.forward()
  assert relerr(sim.field("qacc"), o.qacc).max() < 2e-3 and relerr(sim.field("qfrc_constraint"), o.qfrc_constraint).max() < 2e-3
  it = sim.field("solver_niter").ravel()
  assert it.max() > 10 and it.max() < 200  # converged by its own criterion, not by the cap
  assert lib.b2_set_option(sim.h, b"solver", 0.0) != 0  # PGS is refused
  sim.close()


def test_emulated_sorted_dispatch_changes_scheduling_only(lib):
  """b2_order_kernel (heavy-first counting sort of the worlds, one 1024-thread CTA) on the host emulation: with the
  sorted dispatch on, every world is still stepped exactly once - the states after three steps are bit-identical
  to the unsorted run (a lost or duplicated world would leave its state behind or step it twice)."""
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled("go1_flat")
  n = 520  # (the sort is used from 512 worlds up)
  st = make_states(m, n, seed=3)
  out = []
  for sd in (0.0, 1.0):
    sim = EmulSim(lib, m, n)
    lib.b2_set_option(sim.h, b"sorted_dispatch", sd)
    sim.load(st)
    sim.step(3)
    out.append((sim.field("qpos").copy(), sim.field("qvel").copy(), sim.field("solver_niter").copy()))
    sim.close()
  assert len(np.unique(out[0][2])) > 2  # the sort key (Newton iterations) takes several values
  assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
