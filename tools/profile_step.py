"""Profiling driver: bring 4096 G1 envs into the steady-state workload distribution (random
actions with resets), then run a few physics steps for ncu / timing experiments."""
import sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch
from mjlab_b200.envs import VelocityEnvCfg, VelocityFlatEnv

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
mode = sys.argv[2] if len(sys.argv) > 2 else "time"
import os
_wl = os.environ.get("B2_WORKLOAD", "B")  # B: G1 flat, E: Go1 rough boxes, F: Go1 rough boxes + height fields
_kw = dict(B={}, E=dict(robot="go1", terrain="rough"), F=dict(robot="go1", terrain="rough_hf"))[_wl]
env = VelocityFlatEnv(VelocityEnvCfg(num_envs=n, **_kw), device="cuda:0")
_nu = 29 if _wl == "B" else 12
g = torch.Generator(device="cuda:0"); g.manual_seed(0)
for _ in range(int(sys.argv[3]) if len(sys.argv) > 3 else 60):
  env.step(torch.rand((n, _nu), generator=g, device="cuda:0") * 2 - 1)
torch.cuda.synchronize()
sim = env.sim
def timeit(label, k=20):
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  state = (sim.data.qpos[:].clone(), sim.data.qvel[:].clone(), sim.data.qacc_warmstart[:].clone())
  a.record()
  for _ in range(k): sim.step()
  b.record(); torch.cuda.synchronize()
  st = sim.stats()
  print(f"{label:40s} {a.elapsed_time(b)/k*1e3:9.1f} us/step  ncon {st.ncon_mean:.1f} nefc {st.nefc_mean:.1f} iters {st.niter_mean:.2f} max {st.niter_max}")
  sim.data.qpos[:] = state[0]; sim.data.qvel[:] = state[1]; sim.data.qacc_warmstart[:] = state[2]
def timeit4(label, k=10):
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  state = (sim.data.qpos[:].clone(), sim.data.qvel[:].clone(), sim.data.qacc_warmstart[:].clone())
  a.record()
  for _ in range(k): sim.step_n(4)
  b.record(); torch.cuda.synchronize()
  print(f"{label:40s} {a.elapsed_time(b)/k/4*1e3:9.1f} us/sub-step")
  sim.data.qpos[:] = state[0]; sim.data.qvel[:] = state[1]; sim.data.qacc_warmstart[:] = state[2]
if mode == "time":
  timeit("steady state (random actions)")
  timeit4("step_n(4)")
  sim.set_option("iterations", 1); timeit("iterations=1")
  sim.set_option("iterations", 0); timeit("iterations=0")
  sim.set_option("iterations", 10)
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(20): sim.forward()
  b.record(); torch.cuda.synchronize()
  print(f"{'forward':40s} {a.elapsed_time(b)/20*1e3:9.1f} us")
  sim.data.qpos[:, 2] += 5.0  # lift everyone: no contacts
  timeit("airborne (no contacts)")
else:
  for _ in range(6): sim.step_n(1) if hasattr(sim, "step_n") else sim.step()
  torch.cuda.synchronize()
