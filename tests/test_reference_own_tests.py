"""The reference's OWN test files, unmodified (copied into oracle/_ref/tests by the build), executed against this
repo's drop-in: ``mjlab`` is the unmodified package under oracle/_ref, ``mujoco`` / ``mujoco_warp`` / ``warp`` are
mjlab_b200.compat, and the engine behind them is the product's CUDA source compiled for the host (tests/ref_runner.py).
Only files whose subject is on the boundary of SURVEY.md §8(b) are run; the few cases that need what this image
lacks are deselected by name, everything else must pass.
With stand-ins for the absent RL / viewer wheels (tests/stubs, tests/ref_runner.py) the reference's task configs and
``ManagerBasedRlEnv`` import too: its smoke test passes and its hot loop is stepped on the engine (ref_env_cases.py).
Where no reference checkout was found at build time there is no oracle/_ref and the module skips."""

import re
import subprocess
import sys
from pathlib import Path

import pytest

import refload

REF_TESTS = refload.REF / "tests"
pytestmark = pytest.mark.skipif(not (REF_TESTS.is_dir() and refload.available()),
                                reason="oracle/_ref not installed (no reference checkout at build time)")

CASES = [
  # file, deselect expression, minimum number of passing tests
  ("test_sim_data.py", None, 6),             # TorchArray / WarpBridge on the warp stand-in's arrays
  ("test_scene_entity_config.py", None, 12),  # name -> id resolution used by every MDP term
  ("test_nan_guard.py", "not complex_model", 4),  # Simulation.step on the engine under NanGuard, dump + model blob
  ("smoke_test.py", None, 1),                # ManagerBasedRlEnv(UnitreeGo1FlatEnvCfg) constructs: every manager of the task on the engine
  ("test_rewards.py", None, 10),             # reward terms of the velocity / tracking tasks on entity data
  ("test_scene.py", None, 14),               # Scene: entities + terrain attached into one spec, compiled, initialised on the engine
  ("test_domain_randomization.py", None, 5),  # events.randomize_field on a Scene: per-world model fields reach the engine
  ("test_observation_history.py", None, 14),  # ObservationManager (history buffers, flattening) with the real managers package
  # the model compiler (SURVEY.md §8 f-4) against the reference's expectations on its own robot XMLs and spec editors:
  ("test_spec_config.py", None, 27),    # utils/spec_config.py editors (actuators, collisions, sensors, visuals) on the MjSpec stand-in
  ("test_g1_constants.py", None, 12),   # asset_zoo G1: gains, armature, effort limits, keyframe, collision pairs
  ("test_go1_constants.py", None, 6),
  ("test_asset_zoo.py", None, 2),       # every robot of the zoo compiles
  # (one case compiles a model with a <jointpos> sensor: the engine evaluates contact sensors only and compile() says so)
  ("test_entity.py", "not test_force_on_specific_body", 8),
]


def test_reference_test_files_pass_on_the_drop_in(tmp_path):
  """One pytest run (one interpreter start) over all files; per-file pass counts from the junit report."""
  import xml.etree.ElementTree as ET

  deselect = " and ".join(c[1] for c in CASES if c[1])
  report = tmp_path / "report.xml"
  cmd = [sys.executable, str(Path(__file__).with_name("ref_runner.py")), "--rootdir", str(tmp_path), "-k", deselect,
         f"--junitxml={report}", "-o", "junit_family=xunit1", *[str(REF_TESTS / c[0]) for c in CASES]]
  r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp_path, timeout=900)
  tail = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-500:]
  assert r.returncode == 0 and "failed" not in tail and "error" not in tail, r.stdout[-3000:] + r.stderr[-2000:]
  passed = {c[0]: 0 for c in CASES}
  for tc in ET.parse(report).getroot().iter("testcase"):
    if any(ch.tag in ("failure", "error", "skipped") for ch in tc):
      continue
    f = Path(tc.get("file", "")).name or tc.get("classname", "").split(".")[0] + ".py"
    for name in passed:
      if f == name or tc.get("classname", "").split(".")[-1] == name[:-3] or name[:-3] in tc.get("classname", ""):
        passed[name] += 1
        break
  short = {n: (passed[n], c[2]) for n, c in zip(passed, CASES) if passed[n] < c[2]}
  assert not short, (short, tail)
  assert sum(passed.values()) >= 121, (passed, tail)


@pytest.mark.parametrize("task", ["go1", "g1", "go1_rough", "g1_tracking"])
def test_reference_env_hot_loop_runs_on_the_engine(tmp_path, task):
  """tests/ref_env_cases.py (own cases, run in the runner's interpreter): the reference's ``ManagerBasedRlEnv.step`` -
  action manager -> ctrl, 4 x ``Simulation.step``, terminations, rewards, resets, commands, observations (SURVEY.md
  §3.2) - for its Go1 and G1 flat velocity tasks (G1 flat = BASELINE config B) and Go1 on the generated rough terrain
  (config E: the reference's TerrainImporter builds the boxes, this repo's compiler bins them) and the G1 tracking task
  (config C, synthetic static clip), and the states it reaches against
  the oracle."""
  import os

  cmd = [sys.executable, str(Path(__file__).with_name("ref_runner.py")), "--rootdir", str(tmp_path),
         str(Path(__file__).with_name("ref_env_cases.py"))]
  r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp_path, timeout=900, env=dict(os.environ, B2_REF_TASK=task))
  tail = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-500:]
  assert r.returncode == 0 and re.search(r"2 passed", tail), r.stdout[-3000:] + r.stderr[-2000:]
