"""Time the physics sub-step of a compiled scene under standing PD control.

  python tools/time_scene.py go1_flat go1_rough [--n 4096] [--iters 50]

Robots are spawned on the terrain's curriculum origins when the scene has them.  Prints us per sub-step
(CUDA events around step_n(4) x iters, after a 100-step pre-roll), mean contacts and Newton iterations."""
import argparse
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mjlab_b200.asset_zoo import load_compiled  # noqa: E402
from mjlab_b200.sim import Simulation, SimulationCfg  # noqa: E402
from mjlab_b200.terrains import env_origins_curriculum  # noqa: E402


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("scenes", nargs="+")
  ap.add_argument("--n", type=int, default=4096)
  ap.add_argument("--iters", type=int, default=50)
  ap.add_argument("--ncon", type=int, default=0, help="contact capacity per world (0: engine default)")
  a = ap.parse_args()
  for name in a.scenes:
    m = load_compiled(name)
    sim = Simulation(a.n, SimulationCfg(nconmax=a.ncon * a.n if a.ncon else None), m, "cuda:0")
    key = m.keys["robot/init_state"]
    qpos = np.tile(key["qpos"], (a.n, 1))
    if "terrain_origins" in m.arrays:
      org, _, _ = env_origins_curriculum(a.n, np.asarray(m.arrays["terrain_origins"]), max_init_level=9)
      qpos[:, 0:3] += org
    rng = np.random.default_rng(0)
    qpos[:, 0:2] += rng.uniform(-1.0, 1.0, (a.n, 2))
    sim.data.qpos[:] = torch.as_tensor(qpos, dtype=torch.float32, device="cuda:0")
    sim.data.qvel[:] = 0
    ctrl = torch.as_tensor(np.tile(key["ctrl"], (a.n, 1)), dtype=torch.float32, device="cuda:0")
    sim.data.ctrl[:] = ctrl
    sim.step_n(100)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(a.iters):
      sim.data.ctrl[:] = ctrl + 0.2 * np.sin(0.3 * i)
      sim.step_n(4)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (4 * a.iters)
    nc = sim.data.ncon[:].float().mean().item()
    ni = sim.data.solver_niter[:].float().mean().item()
    ov = int(sim.data.overflow[:].sum().item())
    print(f"{name}: n={a.n} {us:.1f} us/sub-step  {a.n / us:.2f} M env-substeps/s  ncon={nc:.1f} niter={ni:.2f} overflow={ov} "
          f"smem/env={int(sim.get_option('smem_bytes_per_env'))}")
    sim.close()


if __name__ == "__main__":
  main()
