"""Shared helpers for the parity tests (seeded states, oracle/engine state transfer)."""

from __future__ import annotations

from pathlib import Path

import numpy as np


def golden_xml(robot: str) -> str:
  """MJCF text of a zoo robot (``g1``, ``go1``): the reference's asset_zoo file, stored as a fixture in tests/golden."""
  return (Path(__file__).parent / "golden" / f"{robot}.xml").read_text()


def _quat_mul(a, b):
  w = a[..., 0] * b[..., 0] - a[..., 1] * b[..., 1] - a[..., 2] * b[..., 2] - a[..., 3] * b[..., 3]
  x = a[..., 0] * b[..., 1] + a[..., 1] * b[..., 0] + a[..., 2] * b[..., 3] - a[..., 3] * b[..., 2]
  y = a[..., 0] * b[..., 2] - a[..., 1] * b[..., 3] + a[..., 2] * b[..., 0] + a[..., 3] * b[..., 1]
  z = a[..., 0] * b[..., 3] + a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1] + a[..., 3] * b[..., 0]
  return np.stack([w, x, y, z], axis=-1)


def make_states(model, n: int, seed: int = 0, key: str = "robot/init_state", z_range=(-0.06, 0.03),
                tilt: float = 0.15, joint_noise: float = 0.25, vel: float = 0.5):
  """Seeded batch of states around the init keyframe: some envs penetrate the ground, joints are
  perturbed (a few hit their limits), velocities are non-zero, controls are perturbed."""
  rng = np.random.default_rng(seed)
  k = model.keys[key]
  nq, nv, nu = int(model.nq), int(model.nv), int(model.nu)
  qpos = np.tile(k["qpos"], (n, 1))
  qpos[:, 0:2] += rng.uniform(-0.5, 0.5, (n, 2))
  qpos[:, 2] += rng.uniform(*z_range, n)
  ax = rng.normal(size=(n, 3))
  ax /= np.linalg.norm(ax, axis=1, keepdims=True)
  ang = rng.uniform(-tilt, tilt, n)
  dq = np.concatenate([np.cos(ang / 2)[:, None], ax * np.sin(ang / 2)[:, None]], axis=1)
  qpos[:, 3:7] = _quat_mul(qpos[:, 3:7], dq)
  qpos[:, 7:] += rng.uniform(-joint_noise, joint_noise, (n, nq - 7))
  # clamp hinge joints slightly beyond their range for a subset so limit rows get exercised
  lo = model.jnt_range[1:, 0] - 0.02
  hi = model.jnt_range[1:, 1] + 0.02
  qpos[:, 7:] = np.clip(qpos[:, 7:], lo, hi)
  qvel = rng.uniform(-vel, vel, (n, nv))
  ctrl = np.tile(k["ctrl"], (n, 1)) + rng.uniform(-0.3, 0.3, (n, nu))
  warm = rng.uniform(-1.0, 1.0, (n, nv))
  return dict(qpos=qpos, qvel=qvel, ctrl=ctrl, qacc_warmstart=warm)


def terrain_states(model, n: int, seed: int, spread: float):
  """make_states() moved onto random sub-terrain origins of a box-terrain scene (xy spread around them)."""
  rng = np.random.default_rng(seed)
  st = make_states(model, n, seed=seed, z_range=(-0.05, 0.04))
  org = np.asarray(model.arrays["terrain_origins"]).reshape(-1, 3)
  spot = org[rng.integers(0, len(org), n)]
  st["qpos"][:, 0:2] = spot[:, 0:2] + rng.uniform(-spread, spread, (n, 2))
  st["qpos"][:, 2] += spot[:, 2]
  return st


def load_oracle(o, st):
  for k, v in st.items():
    o.field(k)[:] = v


def load_sim(sim, st):
  import torch

  for k, v in st.items():
    getattr(sim.data, k)[:] = torch.as_tensor(v, dtype=torch.float32, device=sim.device)


def relerr(a, b, floor=1e-9):
  """True norm-wise relative error per env: max|a-b| / max|b| (``floor`` only guards an all-zero reference)."""
  a = np.asarray(a, dtype=np.float64).reshape(len(a), -1)
  b = np.asarray(b, dtype=np.float64).reshape(len(b), -1)
  return np.abs(a - b).max(axis=1) / np.maximum(np.abs(b).max(axis=1), floor)


def convex_scene():
  """Scene that exercises every mesh / height-field pair type of csrc/b2_convex.h: a ground plane, a wavy height
  field, and free bodies carrying mesh, box, sphere and capsule geoms — one cluster over the plane (plane-mesh,
  mesh-mesh, box-mesh, sphere-mesh, capsule-mesh) and one over the field (hfield-sphere/capsule/box/mesh)."""
  from mjlab_b200.compiler.spec import Spec

  rng = np.random.default_rng(7)
  spec = Spec()
  spec.option.timestep = 0.005
  v1 = rng.normal(size=(14, 3)) * np.array([0.16, 0.12, 0.09])
  v2 = rng.normal(size=(9, 3)) * np.array([0.1, 0.1, 0.14])
  spec.add_mesh("poly1", vertex=v1)
  spec.add_mesh("poly2", vertex=v2)
  nrow, ncol = 14, 18
  ii, jj = np.meshgrid(np.arange(nrow), np.arange(ncol), indexing="ij")
  elev = 0.5 + 0.3 * np.sin(0.8 * ii + 0.3) * np.cos(0.6 * jj) + rng.uniform(-0.05, 0.05, size=(nrow, ncol))
  spec.add_hfield("waves", size=[1.6, 1.2, 0.25, 0.1], nrow=nrow, ncol=ncol, userdata=np.clip(elev, 0, 1))
  wb = spec.worldbody
  wb.add_geom(name="floor", type="plane", size=[0, 0, 0.05])
  wb.add_geom(name="terrain", type="hfield", hfieldname="waves", pos=[4.0, 0.0, 0.0])
  anchors = {}

  def body(name, pos, **geom):
    b = wb.add_body(name=name, pos=pos)
    b.add_freejoint(name=name + "_j")
    b.add_geom(name=name + "_g", density=600.0, **geom)
    anchors[name] = np.array(pos, dtype=float)

  body("m1", [0.0, 0.0, 0.22], type="mesh", meshname="poly1")
  body("m2", [0.12, 0.05, 0.42], type="mesh", meshname="poly2")
  body("bx", [-0.3, 0.05, 0.18], type="box", size=[0.1, 0.07, 0.12])
  body("sp", [0.05, -0.28, 0.2], type="sphere", size=[0.09])
  body("cp", [0.16, 0.14, 0.2], type="capsule", size=[0.05, 0.12])
  body("hs", [3.6, -0.3, 0.0], type="sphere", size=[0.08])
  body("hc", [4.3, 0.4, 0.0], type="capsule", size=[0.05, 0.15])
  body("hb", [4.5, -0.5, 0.0], type="box", size=[0.12, 0.09, 0.06])
  body("hm", [3.5, 0.5, 0.0], type="mesh", meshname="poly1")
  m = spec.compile()
  hf = dict(pos=np.array([4.0, 0.0, 0.0]), size=np.array([1.6, 1.2, 0.25, 0.1]), data=np.clip(elev, 0, 1))
  return m, anchors, hf


def convex_states(model, anchors, hf, n: int, seed: int, drop: bool = False):
  """Generic (untied) poses: every body near its anchor with a random orientation; the bodies over the height field
  sit at the local surface height minus a small random penetration.  ``drop``: bodies at rest, spread apart and
  lifted clear of every surface (a settling run; the interpenetrating parity states produce impacts that spin the
  capsules up to hundreds of rad/s, where no fixed-step integrator of free bodies is stable)."""
  rng = np.random.default_rng(seed)
  nq, nv = int(model.nq), int(model.nv)
  qpos = np.zeros((n, nq))
  qvel = rng.normal(size=(n, nv)) * 0.2
  names = list(anchors)
  nrow, ncol = hf["data"].shape
  dx, dy = 2 * hf["size"][0] / (ncol - 1), 2 * hf["size"][1] / (nrow - 1)
  for w in range(n):
    for k, name in enumerate(names):
      p = anchors[name] + rng.normal(size=3) * np.array([0.04, 0.04, 0.02])
      if drop and not name.startswith("h"):
        p[0:2] = anchors[name][0:2] * 3.0
        p[2] += 0.25
      if name.startswith("h"):
        lx, ly = p[0] - hf["pos"][0] + hf["size"][0], p[1] - hf["pos"][1] + hf["size"][1]
        c, r = int(lx / dx), int(ly / dy)
        p[2] = hf["data"][r:r + 2, c:c + 2].mean() * hf["size"][2] + rng.uniform(0.03, 0.1) + (0.3 if drop else 0.0)
      q = rng.normal(size=4)
      qpos[w, 7 * k:7 * k + 3] = p
      qpos[w, 7 * k + 3:7 * k + 7] = q / np.linalg.norm(q)
  if drop:
    qvel[:] = 0.0
  return dict(qpos=qpos, qvel=qvel, ctrl=np.zeros((n, int(model.nu))), qacc_warmstart=np.zeros((n, nv)))


def surface_height(model, x: float, y: float) -> float:
  """Height of the topmost height-field surface at world (x, y) (0 when no field covers the point); fields are
  assumed unrotated, as the terrain generator places them."""
  gt = np.asarray(model.geom_type)
  best = 0.0
  for g in np.nonzero(gt == 1)[0]:
    hid = int(model.geom_dataid[g])
    size = np.asarray(model.hfield_size)[hid]
    nr, nc = int(model.hfield_nrow[hid]), int(model.hfield_ncol[hid])
    data = np.asarray(model.hfield_data)[int(model.hfield_adr[hid]):int(model.hfield_adr[hid]) + nr * nc].reshape(nr, nc)
    p = np.asarray(model.geom_pos)[g] + np.asarray(model.body_pos)[int(model.geom_bodyid[g])]
    lx, ly = x - p[0] + size[0], y - p[1] + size[1]
    if not (0 <= lx <= 2 * size[0] and 0 <= ly <= 2 * size[1]):
      continue
    c = min(int(lx / (2 * size[0] / (nc - 1))), nc - 2)
    r = min(int(ly / (2 * size[1] / (nr - 1))), nr - 2)
    best = p[2] + data[r:r + 2, c:c + 2].max() * size[2]
  return best


def hfield_states(model, n: int, seed: int, spread: float, clearance=(-0.03, 0.05)):
  """terrain_states() with the trunk height taken from the height field under the robot (the reference's spawn
  origins of the pyramid fields sit at the level of the base, heightfield_terrains.py:245-249)."""
  rng = np.random.default_rng(seed + 1000)
  st = terrain_states(model, n, seed, spread)
  key = make_states(model, 1, seed=0, z_range=(0.0, 0.0))["qpos"][0, 2]
  for w in range(n):
    st["qpos"][w, 2] = surface_height(model, st["qpos"][w, 0], st["qpos"][w, 1]) + key + rng.uniform(*clearance)
  return st
