"""Per-world model fields (domain randomisation) against the fp64 oracle.

Every expandable float model array the step kernel reads is expanded, perturbed differently in every world but the
first, and given to the oracle with the same per-world values; forward and one step must then agree world by world.
A sensitivity check keeps each case honest: the perturbed run must differ from an unperturbed run of the same states
by at least 10x the parity tolerance, so a kernel that read the field with the wrong world index, or not at all in
some phase, fails.  The CPU cases run the product library on the host emulation (tests/emul, Go1); the GPU cases
cover G1 at 1024 worlds and the reordered, two-partition dispatch at 2048.
"""

import numpy as np
import pytest

from oracle.oracle import Oracle
from test_kernel_emul import EmulSim, _load
from util import _quat_mul, load_oracle, make_states, relerr

# The library's float model fields (B2_MODEL_FARRAYS in b2_types.h) minus geom_rgba (never read) and dof_frictionloss
# (the compiler refuses friction loss and the kernel has no friction-loss rows); test_fields_are_the_float_model_fields
# holds the two lists together.
FIELDS = [
  "body_pos", "body_quat", "body_ipos", "body_iquat", "body_mass", "body_subtreemass", "body_inertia",
  "body_invweight0", "jnt_pos", "jnt_axis", "jnt_range", "jnt_solref", "jnt_solimp", "jnt_margin", "jnt_stiffness",
  "dof_armature", "dof_damping", "dof_invweight0", "geom_size", "geom_pos", "geom_quat", "geom_friction",
  "geom_solref", "geom_solimp", "geom_solmix", "geom_margin", "geom_gap", "geom_rbound", "site_pos", "site_quat",
  "actuator_gainprm", "actuator_biasprm", "actuator_ctrlrange", "actuator_forcerange", "actuator_gear", "qpos0",
]
# the arrays the compact kinematic records (kinrec) copy at create time
KINREC = ["body_pos", "body_quat", "jnt_pos", "jnt_axis", "qpos0"]
# the states a field needs to matter (see states()); the fields not listed use "ground"
KIND = dict(jnt_range="air", jnt_solref="air", jnt_solimp="air", jnt_margin="air", dof_invweight0="air",
            body_invweight0="shallow", geom_solimp="shallow", geom_rbound="shallow",
            geom_solmix="deep")
GAP_MARGIN = 0.02  # geom_gap is only meaningful below a margin: its cases run with this margin on every geom
# geom_solmix only weighs two geoms' solref / solimp when they differ: its cases give the ground this solref
FLOOR_SOLREF = (0.05, 1.5)

_TIGHT = ["xpos", "xquat", "xmat", "xipos", "subtree_com", "cvel", "geom_xpos", "geom_xmat", "site_xpos", "site_xmat",
          "actuator_force", "qfrc_bias", "qfrc_smooth", "qM"]
# compared quantity -> (tolerance, relerr floor; None = absolute error): test_kernel_emul._check_forward's, plus the
# state after one step at the emulated step tolerances
TOL = {**{f: (1e-5, 1e-9) for f in _TIGHT}, "qacc_smooth": (1e-4, 1e-9), "qacc": (1e-3, 10.0),
       "sensordata": (1e-3, None), "qpos": (1e-4, 1e-9), "qvel": (5e-3, 1e-9)}
_FWD = [f for f in TOL if f not in ("qpos", "qvel")]


def _movable(m):
  """Bodies and geoms that the kinematics poses every step (the world body and jointless children of the world are
  posed once from world 0's values, INTEGRATION.md "Terrains")."""
  parent, dofnum = np.asarray(m.body_parentid), np.asarray(m.body_dofnum)
  body = np.array([b != 0 and not (parent[b] == 0 and dofnum[b] == 0) for b in range(int(m.nbody))])
  return body, body[np.asarray(m.geom_bodyid)]


def _rotate_quat(q, rng, lo=0.05, hi=0.25):
  ax = rng.normal(size=q.shape[:-1] + (3,))
  ax /= np.linalg.norm(ax, axis=-1, keepdims=True)
  ang = rng.uniform(lo, hi, q.shape[:-1])[..., None]
  r = _quat_mul(q, np.concatenate([np.cos(ang / 2), ax * np.sin(ang / 2)], axis=-1))
  return r / np.linalg.norm(r, axis=-1, keepdims=True)


def _rotate_vec(v, rng, lo=0.05, hi=0.25):
  k = rng.normal(size=v.shape)
  k /= np.linalg.norm(k, axis=-1, keepdims=True)
  a = rng.uniform(lo, hi, v.shape[:-1])[..., None]
  r = v * np.cos(a) + np.cross(k, v) * np.sin(a) + k * (k * v).sum(-1, keepdims=True) * (1 - np.cos(a))
  return r / np.linalg.norm(r, axis=-1, keepdims=True)


def perturbed(m, name, n, rng, keep0=True, margin=None):
  """Values of model field ``name`` for ``n`` worlds, shape (n, *model shape), fp32-exact: world 0 keeps the model's
  values when ``keep0``, every other world gets its own perturbation.  Each field keeps its invariants: unit
  quaternions and joint axes; positive masses, inertias, armature, invweight0 and sizes; lo < hi for ranges;
  positive solref time constants / damping ratios; solimp inside (0, 1) with a positive width; gap <= ``margin``."""
  base = np.asarray(getattr(m, name), dtype=np.float64)
  a = np.repeat(base[None], n, axis=0)

  def U(lo, hi, shape=None):
    return rng.uniform(lo, hi, a.shape if shape is None else shape)

  mb, mg = _movable(m)
  row = dict(body_pos=mb, body_quat=mb, body_ipos=mb, body_iquat=mb, geom_pos=mg, geom_quat=mg, geom_size=mg,
             geom_rbound=mg).get(name)
  if name in ("body_pos", "body_ipos", "jnt_pos", "geom_pos", "site_pos"):
    a += U(-0.02, 0.02) * (1.0 if row is None else row[:, None])
  elif name in ("body_quat", "body_iquat", "geom_quat", "site_quat"):
    a = np.where((np.ones(len(base), bool) if row is None else row)[:, None], _rotate_quat(a, rng), a)
  elif name == "jnt_axis":
    a = _rotate_vec(a, rng)
  elif name in ("body_invweight0", "dof_invweight0"):
    a *= U(0.2, 5.0)
  elif name in ("body_mass", "body_subtreemass", "body_inertia"):
    a *= U(0.6, 1.6)
  elif name == "dof_armature":
    a += U(0.005, 0.03)
  elif name == "dof_damping":
    a += U(0.5, 3.0)
  elif name == "jnt_stiffness":
    a += U(2.0, 20.0) * (np.asarray(m.jnt_type) != 0)  # (the kernel and MuJoCo skip free joints)
  elif name in ("jnt_range", "actuator_ctrlrange"):
    a += U(-0.1, 0.1) * (base[:, 0] < base[:, 1])[:, None]  # (every range is wider than 0.2)
  elif name in ("jnt_solref", "geom_solref"):
    a *= np.stack([U(1.2, 2.5, a.shape[:-1]), U(0.6, 1.5, a.shape[:-1])], axis=-1)  # time constant stays > 2 dt
  elif name in ("jnt_solimp", "geom_solimp"):
    s = a.shape[:-1]
    a = np.stack([U(0.7, 0.9, s), U(0.91, 0.99, s), U(0.002, 0.03, s), U(0.3, 0.7, s), U(1.5, 3.0, s)], axis=-1)
  elif name == "jnt_margin":
    a += U(0.01, 0.04)
  elif name == "geom_margin":
    a += U(0.005, 0.02)
  elif name == "geom_gap":
    a = U(0.2, 0.8) * margin
  elif name in ("geom_size", "geom_rbound"):
    lo, hi = (0.85, 1.2) if name == "geom_size" else (0.05, 0.5)  # (a smaller bound drops contacts in the broadphase)
    a *= np.where((a > 0) & (row[:, None] if a.ndim == 3 else row), U(lo, hi), 1.0)
  elif name == "geom_friction":
    a *= U(0.3, 1.5)
  elif name == "geom_solmix":
    a = np.exp(U(-3.0, 3.0))
  elif name == "actuator_gainprm":
    a[..., 0] *= U(0.6, 1.5, a.shape[:-1])
  elif name == "actuator_biasprm":
    a[..., 1:3] *= U(0.6, 1.5, a.shape[:-1] + (2,))
  elif name == "actuator_forcerange":
    a *= U(0.2, 0.6, a.shape[:-1] + (1,))  # (symmetric ranges: the forces of the stretched actuators saturate)
  elif name == "actuator_gear":
    a *= U(0.7, 1.4)
  elif name == "qpos0":
    jt, adr = np.asarray(m.jnt_type), np.asarray(m.jnt_qposadr)
    scalar = adr[(jt == 2) | (jt == 3)]  # slide and hinge joints (free and ball joints carry no reference pose)
    a[:, scalar] += U(-0.2, 0.2, (n, len(scalar)))
  else:
    raise KeyError(name)
  if keep0:
    a[0] = base
  return a.astype(np.float32)


def states(m, n, seed, kind="ground"):
  """make_states() made to exercise the fields.  ``kind``:
  "ground": trunks low enough for foot contacts (condim 3, inside a margin), joints past their limits and moving
    further in, controls outside their ranges (the stretched position actuators then also exceed a reduced force
    range);
  "air": the same joints, trunks lifted clear of the ground and controls at the joint positions, so that the limit
    rows are the only constraints and nothing else dominates the accelerations;
  "shallow": level, slow trunks whose feet and shins just touch the ground, controls at the joint positions
    (contact softness and the broadphase bound decide there);
  "deep": trunks pressed into the ground, so that shins and trunks bear load too (the feet's contacts take the
    feet's parameters by priority; only these contacts mix two geoms' solref / solimp)."""
  z, tilt, noise, vel = dict(ground=((-0.05, -0.01), 0.15, 0.25, 0.5), shallow=((-0.012, -0.006), 0.03, 0.1, 0.05),
                             air=((0.3, 0.35), 0.15, 0.25, 0.5), deep=((-0.14, -0.12), 0.3, 0.25, 0.5))[kind]
  st = make_states(m, n, seed=seed, z_range=z, tilt=tilt, joint_noise=noise, vel=vel)
  rng = np.random.default_rng(seed + 1)
  jr, adr, dadr = np.asarray(m.jnt_range), np.asarray(m.jnt_qposadr), np.asarray(m.jnt_dofadr)
  hinge = np.nonzero(np.asarray(m.jnt_type) == 3)[0]
  if kind in ("ground", "air"):
    for w in range(n):  # two joints past a limit, one just inside it, all moving towards the limit
      j = rng.choice(hinge, 3, replace=False)
      st["qpos"][w, adr[j]] = [jr[j[0], 0] - 0.01, jr[j[1], 1] + 0.01, jr[j[2], 1] - 0.02]
      st["qvel"][w, dadr[j]] = [-1.0, 1.0, 1.0]
  if kind == "ground":
    cr = np.asarray(m.actuator_ctrlrange)
    st["ctrl"][:, 0::3] = cr[0::3, 1] + 0.3
    st["ctrl"][:, 2::3] = cr[2::3, 0] - 0.3
  else:
    st["ctrl"][:] = st["qpos"][:, adr[np.asarray(m.actuator_trnid)]]
  return st


def snapshot(get, n):
  """Forward outputs (``get`` called after a forward) as float64 rows per world, plus contacts."""
  out = {f: np.array(get(f), dtype=np.float64).reshape(n, -1) for f in _FWD}
  out["ncon"] = np.array(get("ncon")).reshape(n)
  out["nefc"] = np.array(get("nefc")).reshape(n)
  out["contact_geom"] = np.array(get("contact_geom")).reshape(n, -1, 2)
  out["contact_dist"] = np.array(get("contact_dist"), dtype=np.float64).reshape(n, -1)
  return out


def errors(a, b):
  """Per-world error of every compared quantity of ``a`` against ``b``, in units of its tolerance."""
  out = {}
  for f, (tol, floor) in TOL.items():
    if f in a:
      out[f] = (relerr(a[f], b[f], floor) if floor else np.abs(a[f] - b[f]).max(axis=1)) / tol
  return out


def assert_parity(a, o):
  """``a`` (engine) matches ``o`` (oracle) within TOL, with identical contacts."""
  for w in range(len(a["ncon"])):
    k = int(o["ncon"][w])
    assert a["ncon"][w] == k and a["nefc"][w] == o["nefc"][w], (w, a["ncon"][w], k)
    assert (a["contact_geom"][w, :k] == o["contact_geom"][w, :k]).all(), w
    if k:
      assert np.abs(a["contact_dist"][w, :k] - o["contact_dist"][w, :k]).max() < 1e-5, w
  for f, e in errors(a, o).items():
    assert e.max() < 1.0, (f, e.max() * TOL[f][0])


def sensitivity(a, b, worlds):
  """Largest difference between two runs over the compared quantities, in units of the parity tolerance."""
  return max(e[list(worlds)].max() for e in errors(a, b).values())


# ---- host emulation ---------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def lib():
  return _load()


@pytest.fixture(scope="module")
def go1():
  from mjlab_b200.asset_zoo import load_compiled

  return load_compiled("go1_flat")


def _expand(sim, name):
  """b2_expand_model_field, then a numpy view of the (now per-world) array, shape (n, *model shape)."""
  assert sim.lib.b2_expand_model_field(sim.h, name.encode(), None, None) == 0
  return sim.field(name, which=1)


def _emul_run(sim, st):
  """Forward, snapshot, one step: outputs of the forward plus qpos / qvel after the step."""
  sim.load(st)
  sim.forward()
  out = snapshot(lambda f: sim.field(f), sim.n)
  sim.step(1)
  out["qpos"], out["qvel"] = np.array(sim.field("qpos"), np.float64), np.array(sim.field("qvel"), np.float64)
  return out


def _oracle_run(o, st):
  load_oracle(o, st)
  o.forward()
  out = snapshot(o.field, o.nworld)
  o.step()
  out["qpos"], out["qvel"] = o.qpos.copy(), o.qvel.copy()
  return out


def _shared_setting(m, name):
  """Values of other (shared) fields that a field's cases need, identical in every world: a margin on every geom
  for geom_gap, a distinct solref on the ground for geom_solmix."""
  if name == "geom_gap":
    return {"geom_margin": np.full(int(m.ngeom), GAP_MARGIN, np.float32)}
  if name == "geom_solmix":
    sr = np.asarray(m.geom_solref, np.float32).copy()
    sr[~_movable(m)[1]] = FLOOR_SOLREF
    return {"geom_solref": sr}
  return {}


def _write_shared(sim, o, setting):
  """Write through the shared (unexpanded) views: every world sees the values."""
  for f, v in setting.items():
    sim.field(f, which=1)[0] = v
    if o is not None:
      o.model_field(f)[:] = v.reshape(1, -1)


_baselines = {}


def _baseline(lib, m, n, seed, kind, name):
  """Outputs of a sim whose field ``name`` was never expanded or written (cached per state set)."""
  setting = _shared_setting(m, name)
  key = (n, seed, kind, tuple(setting))
  if key not in _baselines:
    sim = EmulSim(lib, m, n)
    _write_shared(sim, None, setting)
    _baselines[key] = _emul_run(sim, states(m, n, seed, kind))
    sim.close()
  return _baselines[key]


def test_fields_are_the_float_model_fields(lib, go1):
  """FIELDS plus the two arrays the kernel does not read are exactly the float model fields the library lists."""
  import ctypes

  from mjlab_b200.sim import native

  sim = EmulSim(lib, go1, 1)
  names = [lib.b2_field_name(sim.h, 1, i).decode() for i in range(lib.b2_num_fields(sim.h, 1))]
  t = native.B2Tensor()
  floats = []
  for name in names:
    assert lib.b2_get_field(sim.h, 1, name.encode(), ctypes.byref(t)) == 0
    if t.dtype == 2:  # B2_F32
      floats.append(name)
  sim.close()
  assert sorted(FIELDS + ["geom_rgba", "dof_frictionloss"]) == sorted(floats)


@pytest.mark.parametrize("name", FIELDS)
def test_per_world_field_matches_oracle(lib, go1, name):
  """One field expanded and perturbed per world (world 0 at the model's values) on 3 worlds: forward and one step
  match the oracle world by world, every perturbed world moves away from the unperturbed run, and world 0 (outside
  the kinematic records) is bit-identical to a sim that never expanded the field."""
  m, n, seed, kind = go1, 3, 41, KIND.get(name, "ground")
  rng = np.random.default_rng(FIELDS.index(name))
  sim = EmulSim(lib, m, n)
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  setting = _shared_setting(m, name)
  _write_shared(sim, o, setting)
  margin = setting["geom_margin"][None] if "geom_margin" in setting else None
  vals = perturbed(m, name, n, rng, margin=margin)
  view = _expand(sim, name)
  assert view.shape == vals.shape and view.strides[0] > 0
  view[...] = vals
  o.model_field(name)[:] = vals.reshape(n, -1)
  st = states(m, n, seed, kind)
  got = _emul_run(sim, st)
  sim.close()
  assert_parity(got, _oracle_run(o, st))
  base = _baseline(lib, m, n, seed, kind, name)
  s = sensitivity(got, base, range(1, n))
  assert s >= 10.0, (name, s)
  if name not in KINREC:
    for f in TOL:
      assert np.array_equal(got[f][0], base[f][0]), (name, f)


@pytest.mark.parametrize("name", KINREC)
def test_kinematic_record_field_written_at_one_world(lib, go1, name):
  """At one world expansion tiles nothing and the caller writes the shared array itself (the reference's
  expand_model_fields returns early at nworld == 1): the kinematics must still see the new values."""
  m, seed = go1, 43
  rng = np.random.default_rng(100 + KINREC.index(name))
  sim = EmulSim(lib, m, 1)
  o = Oracle(m, nworld=1, maxcon=int(sim.option("maxcon")))
  vals = perturbed(m, name, 1, rng, keep0=False)
  view = _expand(sim, name)
  view[...] = vals
  o.model_field(name)[:] = vals.reshape(1, -1)
  st = states(m, 1, seed)
  got = _emul_run(sim, st)
  sim.close()
  assert_parity(got, _oracle_run(o, st))
  assert sensitivity(got, _baseline(lib, m, 1, seed, "ground", name), [0]) >= 10.0


@pytest.mark.parametrize("name", KINREC)
def test_kinematic_record_field_written_through_shared_view(lib, go1, name):
  """A write through the shared (stride-0, never expanded) view changes the field in every world."""
  m, n, seed = go1, 3, 41
  rng = np.random.default_rng(200 + KINREC.index(name))
  sim = EmulSim(lib, m, n)
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  vals = perturbed(m, name, 1, rng, keep0=False)[0]
  view = sim.field(name, which=1)
  assert view.strides[0] == 0
  view[0] = vals
  o.model_field(name)[:] = vals.reshape(1, -1)
  st = states(m, n, seed)
  got = _emul_run(sim, st)
  sim.close()
  assert_parity(got, _oracle_run(o, st))
  assert sensitivity(got, _baseline(lib, m, n, seed, "ground", name), range(n)) >= 10.0


def _perturb_all(m, n, rng):
  out = {}
  for name in FIELDS:  # (geom_margin comes before geom_gap)
    out[name] = perturbed(m, name, n, rng, margin=out.get("geom_margin"))
  return out


def test_all_fields_perturbed_together(lib, go1):
  """Every field expanded and perturbed at once on 3 worlds: forward, then two steps, against the oracle."""
  m, n = go1, 3
  vals = _perturb_all(m, n, np.random.default_rng(7))
  sim = EmulSim(lib, m, n)
  o = Oracle(m, nworld=n, maxcon=int(sim.option("maxcon")))
  for name, v in vals.items():
    _expand(sim, name)[...] = v
    o.model_field(name)[:] = v.reshape(n, -1)
  st = states(m, n, 47)
  sim.load(st)
  load_oracle(o, st)
  sim.forward()
  o.forward()
  assert_parity(snapshot(lambda f: sim.field(f), n), snapshot(o.field, n))
  sim.step(2)
  o.step()
  o.step()
  assert relerr(sim.field("qpos"), o.qpos).max() < 1e-4
  assert relerr(sim.field("qvel"), o.qvel).max() < 5e-3
  sim.close()


# ---- GPU --------------------------------------------------------------------------------------------------------

def _T(x):
  return x[:].detach().cpu().numpy()


def _gpu_pair(m, n, vals, st):
  """A Simulation and an oracle with the same per-world model fields (expanded through Simulation.expand_model_fields
  and written through sim.model) and the same states."""
  import torch

  from mjlab_b200.sim import Simulation, SimulationCfg
  from util import load_sim

  sim = Simulation(n, SimulationCfg(), m, "cuda:0")
  sim.set_option("debug_outputs", 1)
  o = Oracle(m, nworld=n, maxcon=int(sim.get_option("maxcon")))
  sim.expand_model_fields(list(vals))
  for name, v in vals.items():
    t = getattr(sim.model, name)
    t[:] = torch.as_tensor(v, device="cuda:0").reshape(t[:].shape)
    o.model_field(name)[:] = v.reshape(n, -1)
  load_sim(sim, st)
  load_oracle(o, st)
  return sim, o


def _comparable(sim, o, vals, n):
  """Worlds where fp32 and fp64 take the same discrete decisions: the contact count matches, and no contact lies
  within the contact-distance tolerance (1e-5) of its row-inclusion threshold margin - gap (a contact at
  dist < margin - gap gets constraint rows).  On either side of such a tie the two legitimately solve different
  problems, as they do for a contact at the margin itself."""
  same = _T(sim.data.ncon).ravel() == o.ncon.ravel()
  mg, gp = vals["geom_margin"].reshape(n, -1), vals["geom_gap"].reshape(n, -1)
  cg = o.contact_geom.reshape(n, -1, 2)
  for w in np.nonzero(same)[0]:
    g = cg[w, : int(o.ncon[w, 0])]
    inc = np.maximum(mg[w, g[:, 0]], mg[w, g[:, 1]]) - np.maximum(gp[w, g[:, 0]], gp[w, g[:, 1]])
    same[w] = (np.abs(o.contact_dist[w, : len(g)] - inc) >= 1e-5).all()
  return same


@pytest.mark.gpu
def test_gpu_g1_per_world_fields_1024_worlds():
  """G1 (35 dofs: reduced-Newton block, dense schedule) with every field perturbed per world at 1024 worlds, 50
  solver iterations on both sides: qacc, and qvel after one step, meet the parity table's thresholds over the worlds
  whose contacts the two sides decide alike (_comparable)."""
  import torch

  from mjlab_b200.asset_zoo import load_compiled

  m, n = load_compiled("g1_flat"), 1024
  vals = _perturb_all(m, n, np.random.default_rng(11))
  st = states(m, n, 51)
  sim, o = _gpu_pair(m, n, vals, st)
  sim.set_option("iterations", 50)
  o.set_option("iterations", 50)
  sim.forward()
  o.forward()
  torch.cuda.synchronize()
  same = _comparable(sim, o, vals, n)
  assert same.mean() > 0.99
  got = snapshot(lambda f: _T(getattr(sim.data, f)), n)
  ref = snapshot(o.field, n)
  for f in _TIGHT:
    assert relerr(got[f], ref[f]).max() < 1e-5, f
  e = relerr(got["qacc"][same], ref["qacc"][same])
  assert np.percentile(e, 99) <= 1e-4 and e.max() <= 3e-4, ("qacc", np.percentile(e, 99), e.max())
  sim.step()
  o.step()
  torch.cuda.synchronize()
  e = relerr(_T(sim.data.qvel)[same], o.qvel[same])
  assert np.percentile(e, 99) <= 1e-4 and e.max() <= 3e-4, ("qvel", np.percentile(e, 99), e.max())
  assert relerr(_T(sim.data.qpos)[same], o.qpos[same]).max() <= 1e-5
  sim.close()


@pytest.mark.gpu
def test_gpu_per_world_fields_under_reordered_dispatch():
  """2048 worlds: the heavy-first reorder and the two partitions put worlds on other warps and streams than their
  index.  With per-world fields, step_n(4) equals four step() calls bit for bit, and step_n(1) matches the oracle
  world by world (a model row read by launch slot rather than by world would fail here)."""
  import torch

  from mjlab_b200.asset_zoo import load_compiled
  from util import load_sim

  m, n = load_compiled("g1_flat"), 2048
  vals = _perturb_all(m, n, np.random.default_rng(13))
  st = states(m, n, 53)
  a, o = _gpu_pair(m, n, vals, st)
  b, _ = _gpu_pair(m, n, vals, st)
  for _ in range(4):
    a.step()
  b.step_n(4)
  torch.cuda.synchronize()
  for f in ("qpos", "qvel", "qacc", "qacc_warmstart", "xpos", "sensordata", "contact_force"):
    assert (getattr(a.data, f)[:] == getattr(b.data, f)[:]).all(), f
  b.close()
  a.set_option("iterations", 50)
  o.set_option("iterations", 50)
  load_sim(a, st)
  a.step_n(1)
  o.step()
  torch.cuda.synchronize()
  assert relerr(_T(a.data.qpos), o.qpos).max() <= 1e-5
  same = _comparable(a, o, vals, n)
  assert same.mean() > 0.99
  e = relerr(_T(a.data.qvel)[same], o.qvel[same])
  assert np.percentile(e, 99) <= 1e-4 and e.max() <= 3e-4, ("qvel", np.percentile(e, 99), e.max())
  a.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", KINREC)
def test_gpu_kinematic_record_field_written_at_one_world(go1, name):
  """The one-world case of the emulated test on the GPU, through Simulation.expand_model_fields and sim.model."""
  import torch

  m = go1
  vals = {name: perturbed(m, name, 1, np.random.default_rng(100 + KINREC.index(name)), keep0=False)}
  st = states(m, 1, 43)
  sim, o = _gpu_pair(m, 1, vals, st)
  sim.forward()
  o.forward()
  torch.cuda.synchronize()
  got, ref = snapshot(lambda f: _T(getattr(sim.data, f)), 1), snapshot(o.field, 1)
  sim.step()
  o.step()
  torch.cuda.synchronize()
  got["qpos"], got["qvel"] = _T(sim.data.qpos).astype(np.float64), _T(sim.data.qvel).astype(np.float64)
  ref["qpos"], ref["qvel"] = o.qpos.copy(), o.qvel.copy()
  assert_parity(got, ref)
  sim.close()
