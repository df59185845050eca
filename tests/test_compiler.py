"""Model compiler checks (restates the reference's tests/test_g1_constants.py and
tests/test_go1_constants.py, which run against C MuJoCo's compiler)."""

import re

import numpy as np
import pytest

from mjlab_b200.compiler import Spec
from mjlab_b200.compiler import spec as S
from mjlab_b200.compiler.spec_cfg import ActuatorCfg, ActuatorSetCfg, CollisionCfg, ContactSensorCfg


def test_g1_sizes_and_ordering(g1_model):
  m = g1_model
  # tests/test_g1_constants.py:120-124 and SURVEY.md Appendix B / D
  assert (int(m.nq), int(m.nv), int(m.nu), int(m.njnt)) == (36, 35, 29, 30)
  assert int(m.nbody) == 32 and int(m.ngeom) == 69 and int(m.npair) == 502
  assert m.names["body"][:3] == ["world", "terrain", "robot/pelvis"]
  assert m.names["geom"][0] == "terrain" and int(m.geom_type[0]) == S.GEOM_PLANE
  assert m.names["joint"][0] == "robot/floating_base_joint" and int(m.jnt_type[0]) == S.JNT_FREE
  # actuators in joint order (spec_config.py:429-430)
  assert m.names["actuator"] == m.names["joint"][1:]
  assert (m.actuator_trnid == np.arange(1, 30)).all()


def test_g1_actuator_gains(g1_model):
  # tests/test_g1_constants.py:37-49: gainprm[0]=kp, biasprm=[0,-kp,-kd], forcerange=+-effort
  m = g1_model
  table = {"elbow": (14.25, 0.907, 25.0), "hip_pitch": (40.18, 2.558, 88.0), "knee": (99.10, 6.309, 139.0),
           "wrist_pitch": (16.78, 1.068, 5.0), "ankle_roll": (28.50, 1.814, 50.0)}
  for key, (kp, kd, eff) in table.items():
    i = next(k for k, n in enumerate(m.names["actuator"]) if key in n)
    assert m.actuator_gainprm[i, 0] == pytest.approx(kp, rel=2e-3)
    assert m.actuator_biasprm[i, 1] == pytest.approx(-kp, rel=2e-3)
    assert m.actuator_biasprm[i, 2] == pytest.approx(-kd, rel=2e-3)
    assert tuple(m.actuator_forcerange[i]) == (-eff, eff)
    j = int(m.actuator_trnid[i])
    assert tuple(m.actuator_ctrlrange[i]) == pytest.approx(tuple(m.jnt_range[j]))  # inheritrange=1
    assert int(m.actuator_ctrllimited[i]) == 1 and int(m.actuator_forcelimited[i]) == 1


def test_g1_collision_config(g1_model):
  # tests/test_g1_constants.py:80-117
  m = g1_model
  foot = [i for i, n in enumerate(m.names["geom"]) if re.search(r"(left|right)_foot[1-7]_collision$", n)]
  assert len(foot) == 14
  for i in foot:
    assert int(m.geom_condim[i]) == 3 and int(m.geom_priority[i]) == 1
    assert m.geom_friction[i, 0] == pytest.approx(0.6)
  others = [i for i, n in enumerate(m.names["geom"]) if n.endswith("_collision") and i not in foot]
  assert others and all(int(m.geom_condim[i]) == 1 and int(m.geom_priority[i]) == 0 for i in others)
  visual = [i for i, n in enumerate(m.names["geom"]) if not n.endswith("_collision") and n != "terrain"]
  assert all(int(m.geom_contype[i]) == 0 and int(m.geom_conaffinity[i]) == 0 for i in visual)
  # pair census of SURVEY.md Appendix B: 33 vs plane, 469 self pairs
  t1, t2 = m.geom_type[m.pair_geom1], m.geom_type[m.pair_geom2]
  assert int((t1 == S.GEOM_PLANE).sum()) == 33
  assert int(((t1 == S.GEOM_CAPSULE) & (t2 == S.GEOM_CAPSULE)).sum()) == 409
  assert int(((t1 == S.GEOM_SPHERE) & (t2 == S.GEOM_CAPSULE)).sum()) == 59
  assert int(((t1 == S.GEOM_SPHERE) & (t2 == S.GEOM_SPHERE)).sum()) == 1


def test_g1_keyframe(g1_model):
  # tests/test_g1_constants.py:52-77
  k = g1_model.keys["robot/init_state"]
  assert tuple(k["qpos"][:7]) == (0, 0, 0.76, 1, 0, 0, 0)
  names = [n.split("/")[-1] for n in g1_model.names["joint"][1:]]
  q = dict(zip(names, k["qpos"][7:]))
  assert q["left_knee_joint"] == pytest.approx(0.669) and q["right_hip_pitch_joint"] == pytest.approx(-0.312)
  assert q["right_shoulder_roll_joint"] == pytest.approx(-0.2) and q["waist_yaw_joint"] == 0.0
  assert (k["ctrl"] == k["qpos"][7:]).all()


def test_go1_model(go1_model):
  m = go1_model
  assert (int(m.nq), int(m.nv), int(m.nu)) == (19, 18, 12)  # tests/test_go1_constants.py:89-94
  feet = [i for i, n in enumerate(m.names["geom"]) if re.search(r"[FR][LR]_foot_collision$", n)]
  assert len(feet) == 4
  for i in feet:
    assert int(m.geom_condim[i]) == 3 and int(m.geom_priority[i]) == 1
    assert tuple(m.geom_solimp[i][:3]) == pytest.approx((0.9, 0.95, 0.023))
  assert int(m.npair) == 30  # no self collision (contype 1 / conaffinity 0)
  assert int(m.nsensordata) == 4


def test_derived_constants_are_consistent(g1_model):
  m = g1_model
  assert m.body_subtreemass[0] == pytest.approx(m.body_mass.sum())
  assert m.body_subtreemass[2] == pytest.approx(m.body_mass[2:].sum())
  assert (m.dof_invweight0 > 0).all() and (m.body_invweight0[2:] > 0).all()
  assert m.dof_invweight0[0] == pytest.approx(m.dof_invweight0[2])  # free-joint averaging
  assert float(m.stat_meaninertia) > 0
  # translational invweight of the root body ~ 1/total mass at the com
  assert m.body_invweight0[2, 0] < 1.0 / m.body_mass[2]


INLINE = """
<mujoco>
  <compiler angle="degree"/>
  <default><default class="c"><geom type="capsule" size="0.05"/></default></default>
  <worldbody>
    <geom name="floor" type="plane" size="0 0 1"/>
    <body name="a" pos="0 0 1">
      <freejoint name="root"/>
      <geom name="ga" type="box" size="0.1 0.2 0.3" mass="2"/>
      <body name="b" pos="0 0 -0.4" childclass="c">
        <joint name="h" axis="0 1 0" range="-90 90"/>
        <geom name="gb" fromto="0 0 0 0 0 -0.3"/>
      </body>
    </body>
  </worldbody>
  <actuator><position name="act" joint="h" kp="10" kv="1" ctrlrange="-1 1"/></actuator>
</mujoco>
"""


def test_inline_mjcf_and_geometry_inertia():
  m = Spec.from_string(INLINE).compile()
  assert (int(m.nq), int(m.nv), int(m.nu), int(m.nbody)) == (8, 7, 1, 3)
  assert m.jnt_range[1] == pytest.approx(np.radians([-90, 90]))
  assert int(m.jnt_limited[1]) == 1
  # box inertia: m/3 * (b^2+c^2) ..., sorted decreasing in the principal frame
  assert m.body_mass[1] == pytest.approx(2.0)
  assert sorted(m.body_inertia[1], reverse=True) == pytest.approx(
    sorted([2 / 3 * (0.04 + 0.09), 2 / 3 * (0.01 + 0.09), 2 / 3 * (0.01 + 0.04)], reverse=True))
  # capsule from fromto: half length 0.15, centred at -0.15, mass = density * volume
  g = m.names["geom"].index("gb")
  assert m.geom_size[g, 1] == pytest.approx(0.15) and m.geom_pos[g, 2] == pytest.approx(-0.15)
  vol = np.pi * 0.05**2 * 0.3 + 4 / 3 * np.pi * 0.05**3
  assert m.body_mass[2] == pytest.approx(1000 * vol)
  assert m.actuator_biasprm[0, 1] == -10 and m.actuator_biasprm[0, 2] == -1
  # floor collides with both moving geoms; parent-child pair (a,b) is filtered
  assert int(m.npair) == 2


def test_spec_cfg_semantics():
  sp = Spec.from_string(INLINE)
  with pytest.raises(ValueError, match="condim must be one of"):
    CollisionCfg(geom_names_expr=[".*"], condim=2).edit_spec(sp)
  CollisionCfg(geom_names_expr=["gb"], condim=1, friction=(0.3,), disable_other_geoms=True).edit_spec(sp)
  assert sp.geom("gb").condim == 1 and sp.geom("gb").friction[0] == 0.3
  assert sp.geom("ga").contype == 0 and sp.geom("ga").conaffinity == 0
  with pytest.raises(ValueError, match="effort_limit must be positive"):
    ActuatorSetCfg((ActuatorCfg(["h"], effort_limit=0, stiffness=1, damping=1),)).edit_spec(sp)
  with pytest.raises(ValueError, match="Exactly one of"):
    ContactSensorCfg(name="s").validate()
  with pytest.raises(ValueError, match="must be in order"):
    ContactSensorCfg(name="s", body1="a", data=("force", "found"))._intprm()
  assert ContactSensorCfg(name="s", body1="a", data=("found", "force"), reduce="netforce", num=2)._intprm() == (3, 3, 2)


def test_attach_prefix_and_sensor_references(g1_model):
  m = g1_model
  i = m.names["sensor"].index("robot/left_foot_ground_contact")
  assert m.names["body"][int(m.sensor_objid[i])] == "robot/left_ankle_roll_link"
  assert m.names["body"][int(m.sensor_refid[i])] == "terrain"  # un-prefixed global reference
  assert int(m.sensor_dim[i]) == 1


def test_unsupported_features_fail_loudly():
  base = '<mujoco><worldbody><geom name="f" type="plane" size="0 0 1"/><body name="b" pos="0 0 1"><freejoint/>{geom}{extra}</body></worldbody>{top}</mujoco>'
  ok = base.format(geom='<geom name="g" type="sphere" size="0.1"/>', extra="", top="")
  Spec.from_string(ok).compile()
  with pytest.raises(NotImplementedError, match="tendon"):
    Spec.from_string(base.format(geom='<geom type="sphere" size="0.1"/>', extra="", top="<tendon/>"))
  with pytest.raises(NotImplementedError, match="composite"):
    Spec.from_string(base.format(geom='<geom type="sphere" size="0.1"/>', extra="<composite/>", top=""))
  with pytest.raises(NotImplementedError, match="condim 4"):
    Spec.from_string(base.format(geom='<geom name="g" type="sphere" size="0.1" condim="4"/>', extra="", top="")).compile()
  # (cylinders and ellipsoids were refused until the convex routines learned their support points)
  mc = Spec.from_string(base.format(geom='<geom name="g" type="cylinder" size="0.1 0.1"/>', extra="", top="")).compile()
  assert int(mc.npair) == 1 and [int(mc.geom_type[int(mc.pair_geom1[0])]), int(mc.geom_type[int(mc.pair_geom2[0])])] == [0, 5]
  with pytest.raises(NotImplementedError, match="ball"):
    Spec.from_string('<mujoco><worldbody><body name="b"><joint type="ball"/><geom type="sphere" size="0.1"/></body></worldbody></mujoco>').compile()
  sp = Spec.from_string(ok)
  sp.worldbody.children[0].add_joint(name="h", type="hinge", frictionloss=0.1)
  with pytest.raises(NotImplementedError, match="frictionloss"):
    sp.compile()


def test_compiled_blobs_are_reproducible_from_the_reference_xml():
  """The model blobs shipped in asset_zoo/compiled (what every GPU test and the bench load) are exactly what the
  compiler produces today from the reference's MJCF: arrays, names and keyframes, bit for bit."""
  import sys

  from util import golden_xml

  from mjlab_b200.asset_zoo import g1, go1, load_compiled
  from mjlab_b200.asset_zoo.scene import compile_scene

  g1_xml, go1_xml = golden_xml("g1"), golden_xml("go1")
  sys.path.insert(0, str(__import__("pathlib").Path(__file__).resolve().parents[1] / "tools"))
  import compile_assets as ca

  fresh = {
    "g1_flat": compile_scene(g1.robot_cfg(g1_xml, g1.velocity_sensors()), ca.TASK),
    "g1_tracking_flat": compile_scene(g1.robot_cfg(g1_xml, g1.tracking_sensors()), ca.TASK),
    "go1_flat": compile_scene(go1.robot_cfg(go1_xml, go1.velocity_sensors()), ca.TASK),
    "go1_hf_small": compile_scene(go1.robot_cfg(go1_xml, go1.velocity_sensors()), ca.TASK, ca.SMALL_HF),
  }
  for name, m in fresh.items():
    old = load_compiled(name)
    assert old.names == m.names, name
    assert set(old.arrays) == set(m.arrays), (name, set(old.arrays) ^ set(m.arrays))
    for k in old.arrays:
      assert np.array_equal(np.asarray(old.arrays[k]), np.asarray(m.arrays[k])), (name, k)
    for k in old.keys:
      for f in ("qpos", "qvel", "ctrl"):
        assert np.array_equal(old.keys[k][f], m.keys[k][f]), (name, k, f)
