"""Box primitives and grid-static broadphase in the oracle + terrain generator (BASELINE config E groundwork).

The box routines are own restatements (MuJoCo's sources for mjc_SphereBox / mjc_CapsuleBox / mjc_BoxBox are not
available here; box-box is the textbook separating-axis test + face clipping / edge-edge contact), so they are
pinned by statics and by cross-checking the grid broadphase against the exhaustive pair table."""

import sys
from pathlib import Path

import numpy as np
import pytest

from mjlab_b200.compiler import Spec
from mjlab_b200.compiler import compile as C
from mjlab_b200.compiler import spec as S
from mjlab_b200.terrains import RoughTerrainCfg, generate_terrain, pyramid_stairs, terrain_spec
from oracle.oracle import Oracle

ON_BOX = """
<mujoco><option timestep="0.002"/>
  <worldbody>
    <body name="table" pos="0 0 0.25"><geom name="top" type="box" size="0.5 0.5 0.25"/></body>
    <body name="obj" pos="0 0 {z}" {quat}><freejoint/>{geom}</body>
  </worldbody></mujoco>
"""


@pytest.mark.parametrize("geom,z,quat,ncon", [
  ('<geom type="sphere" size="0.1" mass="2"/>', 0.599, "", 1),
  ('<geom type="capsule" size="0.05 0.2" mass="2"/>', 0.549, 'quat="0.7071068 0 0.7071068 0"', 2),
  ('<geom type="box" size="0.1 0.15 0.05" mass="2"/>', 0.549, "", 4),
])
def test_objects_rest_on_a_box(geom, z, quat, ncon):
  m = Spec.from_string(ON_BOX.format(geom=geom, z=z, quat=quat)).compile()
  assert int(m.npair) == 1 and int(m.nstatic) == 0  # one static box: pair-table route
  o = Oracle(m)
  for _ in range(1500):
    o.step()
  n = int(o.ncon[0, 0])
  assert n == ncon
  assert abs(o.qvel[0]).max() < 1e-4
  assert o.contact_force[0, 0 : 3 * n : 3].sum() == pytest.approx(2 * 9.81, rel=1e-4)
  fr = o.contact_frame[0, :9].reshape(3, 3)
  # normal points from geom1 to geom2 (mjtGeom order: sphere < capsule < box; box-box by id)
  g1 = int(o.contact_geom[0, 0])
  assert fr[0] == pytest.approx([0, 0, 1.0 if g1 == 0 else -1.0], abs=1e-6)
  assert o.qpos[0, 2] == pytest.approx(z, abs=2e-3)


def _prim_box_box(p1, R1, h1, p2, R2, h2, margin=0.0):
  import ctypes

  from oracle.oracle import build
  build()
  L = ctypes.CDLL(str(Path(__file__).parents[1] / "oracle" / "libb2oracle64.so"))
  dp = ctypes.POINTER(ctypes.c_double)
  L.b2o_prim_box_box.argtypes = [dp] * 6 + [ctypes.c_double, dp]
  out = np.zeros(56)
  P = lambda a: np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(dp)
  arrs = [np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel()) for a in (p1, R1, h1, p2, R2, h2)]
  n = L.b2o_prim_box_box(*[a.ctypes.data_as(dp) for a in arrs], margin, out.ctypes.data_as(dp))
  return n, out[: 7 * n].reshape(n, 7)


def test_box_box_face_clipping_and_edge_edge_cases():
  """box-box = SAT + clipping: a cube on a slab (4 contacts at its bottom corners), the same cube overhanging the
  slab's edge (the incident face is clipped at the slab's side plane), rotated 45 deg (4), two crossed beams
  turned edge-up / edge-down (one edge-edge contact at the crossing, depth = overlap of the edges), separation
  beyond the margin (none), and symmetry under swapping the two boxes (normal flips)."""
  I = np.eye(3)
  n, c = _prim_box_box([0, 0, 0], I, [2, 2, .5], [0.3, 0.2, 0.999], I, [.5, .5, .5])
  assert n == 4 and c[:, 0] == pytest.approx(-0.001) and np.allclose(c[:, 4:7], [0, 0, 1])
  assert sorted(map(tuple, np.round(c[:, 1:3], 6))) == [(-0.2, -0.3), (-0.2, 0.7), (0.8, -0.3), (0.8, 0.7)]
  assert c[:, 3] == pytest.approx(0.4995)  # midway between the two surfaces
  n, c = _prim_box_box([0, 0, 0], I, [2, 2, .5], [1.8, 0, 0.999], I, [.5, .5, .5])  # overhang: x in [1.3, 2.3] clipped at 2
  assert n == 4 and c[:, 1].max() == pytest.approx(2.0, abs=1e-5) and c[:, 1].min() == pytest.approx(1.3)
  a = np.pi / 4
  Rz = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
  n, c = _prim_box_box([0, 0, 0], I, [2, 2, .5], [0, 0, 0.99], Rz, [.5, .5, .5])
  assert n == 4 and c[:, 0] == pytest.approx(-0.01) and np.hypot(c[:, 1], c[:, 2]) == pytest.approx(np.sqrt(0.5))
  Rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
  Ry = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
  n, c = _prim_box_box([0, 0, 0], Rx, [1, .1, .1], [0, 0, 0.27], Ry, [.1, 1, .1])
  assert n == 1 and c[0, 0] == pytest.approx(0.27 - 2 * 0.1 * np.sqrt(2), abs=2e-6) and np.allclose(c[0, 4:7], [0, 0, 1])
  assert np.allclose(c[0, 1:4], [0, 0, 0.135], atol=1e-9)
  assert _prim_box_box([0, 0, 0], I, [1, 1, 1], [0, 0, 2.05], I, [1, 1, 1])[0] == 0
  assert _prim_box_box([0, 0, 0], I, [1, 1, 1], [0, 0, 2.05], I, [1, 1, 1], margin=0.1)[0] == 4  # within the margin
  n1, c1 = _prim_box_box([0, 0, 0], Rx, [1, .1, .1], [0, 0, 0.27], Ry, [.1, 1, .1])
  n2, c2 = _prim_box_box([0, 0, 0.27], Ry, [.1, 1, .1], [0, 0, 0], Rx, [1, .1, .1])
  assert n1 == n2 == 1 and np.allclose(c1[0, :4], c2[0, :4]) and np.allclose(c1[0, 4:7], -c2[0, 4:7])


def test_box_resting_on_an_edge_of_a_box():
  """A flat box lying across the table's edge (half of it overhangs): it rests on the clipped contact patch, the
  contact forces carry its weight and the net moment about its centre vanishes (it does not tip: com is over the table)."""
  xml = ON_BOX.format(geom='<geom type="box" size="0.2 0.1 0.02" mass="3"/>', z=0.5199, quat="").replace('pos="0 0 0.5199"', 'pos="0.4 0 0.5199"')
  m = Spec.from_string(xml).compile()
  o = Oracle(m)
  fz = []
  for i in range(3000):
    o.step()
    if i >= 2000:
      fz.append(o.contact_force[0, 0 : 3 * int(o.ncon[0, 0]) : 3].sum())
  n = int(o.ncon[0, 0])
  assert n == 4 and abs(o.qvel[0]).max() < 0.05  # (a lightly damped rocking mode of the soft contacts remains)
  assert np.mean(fz) == pytest.approx(3 * 9.81, rel=5e-3)
  assert abs(o.qpos[0, 2] - 0.5199) < 2e-3 and abs(o.qpos[0, 0] - 0.4) < 5e-3  # it neither sinks, tips nor slides
  pos = o.contact_pos[0, : 3 * n].reshape(n, 3)
  assert pos[:, 0].max() == pytest.approx(0.5, abs=1e-4) and pos[:, 0].min() == pytest.approx(0.2, abs=1e-3)  # patch ends at the table's edge


def test_sphere_inside_box_is_pushed_out_through_the_nearest_face():
  m = Spec.from_string(ON_BOX.format(geom='<geom type="sphere" size="0.05" mass="1"/>', z=0.47, quat="")).compile()
  o = Oracle(m)
  o.forward()
  assert int(o.ncon[0, 0]) == 1
  assert o.contact_dist[0, 0] == pytest.approx(-(0.03 + 0.05))  # depth to the top face + radius
  assert o.contact_frame[0, :3] == pytest.approx([0, 0, -1])
  assert o.qacc[0, 2] > 0  # pushed upwards


def test_terrain_census_and_geometry():
  boxes, origins = generate_terrain(RoughTerrainCfg())
  assert len(boxes) == 3564 and origins.shape == (10, 20, 3)  # SURVEY.md Appendix B
  bx, org = pyramid_stairs((8.0, 8.0), 1.0)
  assert len(bx) == 29 and org == pytest.approx([4, 4, 0.7])
  tops = sorted({round(float(p[2] + h[2]), 6) for h, p in bx})
  assert tops == pytest.approx([0.1 * k for k in range(8)])  # border at 0, steps 0.1 .. 0.6, platform 0.7
  bx, org = pyramid_stairs((8.0, 8.0), 0.5, inverted=True)
  assert org[2] == pytest.approx(-0.35) and max(p[2] + h[2] for h, p in bx) == pytest.approx(0.0)
  # difficulty grows with the row (curriculum), the first 8 columns are flat
  assert (origins[:, :8, 2] == 0).all() and origins[9, 10, 2] > origins[0, 10, 2] > 0 > origins[9, 19, 2]


def _go1_on(cfg, threshold=None):
  from util import golden_xml

  from mjlab_b200.asset_zoo import go1

  old = C.STATIC_GRID_THRESHOLD
  if threshold is not None:
    C.STATIC_GRID_THRESHOLD = threshold
  try:
    tsp, origins = terrain_spec(cfg)
    sp = S.Spec()
    sp.attach(tsp, prefix="")
    sp.attach(go1.robot_cfg(golden_xml("go1"), go1.velocity_sensors()).build_spec(), prefix="robot/")
    sp.option.timestep = 0.005
    sp.option.integrator = S.INT_IMPLICITFAST
    sp.option.iterations, sp.option.ls_iterations = 10, 20
    return sp.compile(), origins
  finally:
    C.STATIC_GRID_THRESHOLD = old


@pytest.fixture(scope="module")
def go1_stairs():
  from mjlab_b200.asset_zoo import load_compiled

  m = load_compiled("go1_stairs_small")
  return m, np.asarray(m.arrays["terrain_origins"])


def test_grid_broadphase_equals_exhaustive_pairs(go1_stairs):
  sys.path.insert(0, str(Path(__file__).resolve().parents[1] / "tools"))
  from compile_assets import SMALL_STAIRS

  mg, origins = go1_stairs
  mp, _ = _go1_on(SMALL_STAIRS, threshold=10**9)  # same scene, every static box in the pair table
  assert (mp.geom_size == mg.geom_size).all()
  assert int(mg.nstatic) > 100 and int(mg.npair) == 0 and int(mp.nstatic) == 0 and int(mp.npair) == 30 * int(mg.nstatic)
  n = 12
  rng = np.random.default_rng(5)
  key = mg.keys["robot/init_state"]
  qpos = np.tile(key["qpos"], (n, 1))
  spots = origins.reshape(-1, 3)[rng.integers(0, origins.shape[0] * origins.shape[1], n)]
  qpos[:, 0:3] = spots + np.stack([rng.uniform(-2.5, 2.5, n), rng.uniform(-2.5, 2.5, n), rng.uniform(0.15, 0.35, n)], 1)
  ang = rng.uniform(-0.6, 0.6, n)
  qpos[:, 3], qpos[:, 4] = np.cos(ang / 2), np.sin(ang / 2)
  a, b = Oracle(mg, nworld=n, maxcon=64), Oracle(mp, nworld=n, maxcon=64)
  for o in (a, b):
    o.qpos[:] = qpos
    o.forward()
  assert (a.ncon == b.ncon).all() and int(a.ncon.max()) >= 4
  for w in range(n):
    k = int(a.ncon[w, 0])
    sa = sorted(zip(map(tuple, a.contact_geom[w].reshape(-1, 2)[:k]), np.round(a.contact_dist[w][:k], 9)))
    sb = sorted(zip(map(tuple, b.contact_geom[w].reshape(-1, 2)[:k]), np.round(b.contact_dist[w][:k], 9)))
    assert sa == sb
  assert np.abs(a.qacc - b.qacc).max() < 1e-6 * max(1.0, np.abs(b.qacc).max())


def test_go1_stands_on_stairs(go1_stairs):
  m, origins = go1_stairs
  o = Oracle(m, nworld=2, maxcon=64)
  key = m.keys["robot/init_state"]
  for w, (r, c) in enumerate([(1, 2), (1, 3)]):  # a pyramid platform and an inverted one
    o.qpos[w] = key["qpos"]
    o.qpos[w, 0:3] = origins[r, c] + [0, 0, 0.3]
  o.ctrl[:] = key["ctrl"]
  for _ in range(400):
    o.step()
  assert np.isfinite(o.qpos).all()
  for w, (r, c) in enumerate([(1, 2), (1, 3)]):
    assert 0.2 < o.qpos[w, 2] - origins[r, c, 2] < 0.33  # standing on its feet on the platform
    assert int(o.ncon[w, 0]) >= 4
  assert (o.sensordata > 0).all()  # all four feet report ground contact (geom1 vs body "terrain")


NARROW = """
<mujoco><option timestep="0.002"/>
  <worldbody>
    <body name="beam" pos="0 0 0.25"><geom type="box" size="0.08 0.5 0.25"/></body>
    <body name="obj" pos="{x} 0 {z}" quat="{quat}"><freejoint/><geom type="capsule" size="0.05 0.2" mass="2"/></body>
  </worldbody></mujoco>
"""


def test_capsule_box_contact_set():
  # lying across a narrow beam: the two contacts sit on the beam's edges, not on the capsule's end caps
  m = Spec.from_string(NARROW.format(x=0.02, z=0.549, quat="0.7071068 0 0.7071068 0")).compile()
  o = Oracle(m)
  o.forward()
  assert int(o.ncon[0, 0]) == 2
  xs = sorted(o.contact_pos[0, 0:6:3])
  assert xs == pytest.approx([-0.08, 0.08], abs=3e-3)
  assert o.contact_dist[0, :2] == pytest.approx([-0.001, -0.001], abs=1e-4)
  # tilted by 45 degrees: a single contact under the lower end cap
  m = Spec.from_string(NARROW.format(x=0.1414, z=0.549 + 0.2 * 0.7071, quat="0.9238795 0 0.3826834 0")).compile()
  o = Oracle(m)
  o.forward()
  assert int(o.ncon[0, 0]) == 1
  assert o.contact_frame[0, :3] == pytest.approx([0, 0, -1], abs=1e-6)


def obstacle_course_xml(seed=0, nobst=24, nobj=9):
  """A plane, `nobst` static boxes / spheres / capsules (some rotated) and `nobj` free spheres / capsules /
  boxes dropped among them: exercises the pair table and the static grid in one scene."""
  rng = np.random.default_rng(seed)
  obst, objs = [], []
  for i in range(nobst):
    x, y = rng.uniform(-2, 2, 2)
    kind = ("box", "box", "box", "sphere", "capsule")[i % 5]
    yaw = rng.uniform(-1.5, 1.5)
    quat = f"{np.cos(yaw / 2):.6f} 0 0 {np.sin(yaw / 2):.6f}"
    if kind == "box":
      sx, sy, sz = rng.uniform(0.2, 0.6), rng.uniform(0.1, 0.5), rng.uniform(0.05, 0.2)
      obst.append(f'<geom name="ob{i}" type="box" size="{sx:.3f} {sy:.3f} {sz:.3f}" pos="{x:.3f} {y:.3f} {sz:.3f}" quat="{quat}"/>')
    elif kind == "sphere":
      obst.append(f'<geom name="ob{i}" type="sphere" size="0.2" pos="{x:.3f} {y:.3f} 0.1"/>')
    else:
      obst.append(f'<geom name="ob{i}" type="capsule" size="0.1 0.4" pos="{x:.3f} {y:.3f} 0.1" quat="0.7071068 0.7071068 0 0"/>')
  for i in range(nobj):
    kind = ("sphere", "capsule", "box")[i % 3]
    g = {"sphere": '<geom type="sphere" size="0.12" mass="1"/>',
         "capsule": '<geom type="capsule" size="0.06 0.2" mass="1"/>',
         "box": '<geom type="box" size="0.15 0.1 0.08" mass="1"/>'}[kind]
    x, y = rng.uniform(-1.8, 1.8, 2)
    objs.append(f'<body name="obj{i}" pos="{x:.3f} {y:.3f} 0.6"><freejoint/>{g}</body>')
  return f"""<mujoco><option timestep="0.004"/>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 0.01"/>
    <body name="course">{''.join(obst)}</body>
    {''.join(objs)}
  </worldbody></mujoco>"""


def test_mixed_pair_table_and_grid_scene():
  xml = obstacle_course_xml()
  mg = Spec.from_string(xml).compile()
  old = C.STATIC_GRID_THRESHOLD
  C.STATIC_GRID_THRESHOLD = 10**9
  try:
    mp = Spec.from_string(xml).compile()
  finally:
    C.STATIC_GRID_THRESHOLD = old
  assert int(mg.nstatic) == 24 and int(mg.npair) > 0 and int(mp.nstatic) == 0
  n = 6
  rng = np.random.default_rng(1)
  a, b = Oracle(mg, nworld=n, maxcon=96), Oracle(mp, nworld=n, maxcon=96)
  q = np.tile(mg.qpos0, (n, 1))
  q += rng.uniform(-0.05, 0.05, q.shape) * (np.arange(q.shape[1]) % 7 < 3)  # jitter positions only
  for o in (a, b):
    o.qpos[:] = q
  seen = 0
  for it in range(150):
    for o in (a, b):
      o.step()
    assert (a.ncon == b.ncon).all()
    for w in range(n):
      k = int(a.ncon[w, 0])
      sa = sorted(zip(map(tuple, a.contact_geom[w].reshape(-1, 2)[:k]), np.round(a.contact_dist[w][:k], 8)))
      sb = sorted(zip(map(tuple, b.contact_geom[w].reshape(-1, 2)[:k]), np.round(b.contact_dist[w][:k], 8)))
      assert sa == sb
    seen = max(seen, int(a.ncon.max()))
    # different contact order -> different summation order only
    assert np.abs(a.qpos - b.qpos).max() < 1e-6
    b.qpos[:], b.qvel[:], b.qacc_warmstart[:] = a.qpos, a.qvel, a.qacc_warmstart
  assert seen >= 8 and np.isfinite(a.qpos).all()
  assert a.qpos[:, 2::7].min() > 0.0  # nothing fell through the floor
