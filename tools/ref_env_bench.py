"""Throughput of the REFERENCE's own env layer on this engine: ``ManagerBasedRlEnv.step`` (unmodified mjlab from
oracle/_ref, its managers and task config) over libb2sim.so through mjlab_b200.compat - BASELINE's metric in the
reference's formulation of the caller, next to bench.py's fused MDP kernels.

  B2_REF_DEVICE=cuda:0 python tools/ref_env_bench.py [task=g1|go1|go1_rough] [num_envs=4096] [steps=50]
(on the CPU container: B2_REF_DEVICE unset -> the host-emulated engine, small num_envs only)"""
import os
import runpy
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
task = sys.argv[1] if len(sys.argv) > 1 else "g1"
n = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 50
dev = os.environ.get("B2_REF_DEVICE", "cpu")

# tests/ref_runner.py installs the stand-ins and then calls pytest.main: reuse its set-up, not its exit
sys.argv = [sys.argv[0], "--collect-only", "-q", str(ROOT / "tests" / "ref_env_cases.py")]
try:
  runpy.run_path(str(ROOT / "tests" / "ref_runner.py"), run_name="__main__")
except SystemExit:
  pass

import torch  # noqa: E402
from mjlab.envs.manager_based_rl_env import ManagerBasedRlEnv  # noqa: E402

if task == "g1":
  from mjlab.tasks.velocity.config.g1.flat_env_cfg import UnitreeG1FlatEnvCfg as Cfg
elif task == "go1_rough":
  from mjlab.tasks.velocity.config.go1.rough_env_cfg import UnitreeGo1RoughEnvCfg as Cfg
else:
  from mjlab.tasks.velocity.config.go1.flat_env_cfg import UnitreeGo1FlatEnvCfg as Cfg
cfg = Cfg()
cfg.scene.num_envs = n
env = ManagerBasedRlEnv(cfg, device=dev)
env.reset()
nact = env.action_manager.total_action_dim
g = torch.Generator(device=dev).manual_seed(0)
act = lambda: torch.rand((n, nact), generator=g, device=dev) * 2 - 1  # noqa: E731
for _ in range(5):
  env.step(act())
if dev.startswith("cuda"):
  torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(steps):
  env.step(act())
if dev.startswith("cuda"):
  torch.cuda.synchronize()
dt = time.perf_counter() - t0
print(f"reference ManagerBasedRlEnv ({Cfg.__name__}) on {dev}: {n} envs, {steps} steps, "
      f"{dt / steps * 1e3:.2f} ms/step, {n * steps / dt:.3e} env-steps/s")
