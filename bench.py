"""bench.py — env-steps/s of the B200-native physics step on BASELINE.json's headline workload.

Workload (BASELINE.json configs[1], SURVEY.md §8d config B): Unitree G1 velocity-tracking on flat
terrain, 4096 envs per GPU, random-action agent (``2*U(0,1)-1``, reference ``scripts/play.py:167-169``),
dt 0.005 s, decimation 4, Newton <=10 iterations / <=20 line-search iterations, implicitfast,
pyramidal cones, foot-friction domain randomisation, resets on fall (>70 deg) or time-out, pushes.

One "step" = one environment step = ctrl write + 4 physics sub-steps (4 launches of the fused step
kernel) + mask-based partial reset + one forward pass + the (torch) MDP glue of
``VelocityFlatEnv.step``.  ``value`` uses device-resident actions; ``e2e`` feeds actions from pinned
host memory and reads reward/done/obs back every step.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--envs E] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...      (one rank per GPU, weak scaling)

``--dump-outputs DIR`` writes what the last timed env step returned (rank 0's envs) as float32 ``DIR/<name>.npy``,
so that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# Rank 0 logs (reward, done) of every env; the rows travel in batches: one all-gather per LOG_EVERY env steps (each is a
# rendezvous of the ranks, so the faster rank idles for the skew accumulated since the last one: 2 GPUs, every 16 steps:
# +3.7 % per env step over the 1-GPU run of the same box)
LOG_EVERY = 64
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
WORKLOADS = {
  # BASELINE.json configs[1] (the headline), configs[2], configs[4] (per-GPU share): SURVEY.md §8d B / C / E
  "B": dict(desc="Unitree G1 velocity-tracking flat, {envs} envs/GPU, random-action agent, decimation 4, "
                 "dt 0.005, Newton<=10 it / ls<=20, implicitfast, pyramidal, foot-friction DR, resets+pushes",
            model="g1_flat", robot="g1"),
  "C": dict(desc="Unitree G1 motion-tracking flat (synthetic static clip, self-collision sensor num=10), {envs} envs/GPU, "
                 "random-action agent, decimation 4, dt 0.005, Newton<=10 it / ls<=20, implicitfast, pyramidal, "
                 "DR body_ipos/qpos0/foot friction, RSI resets + pushes, policy obs noise + critic group",
            model="g1_tracking_flat", robot="g1"),
  "E": dict(desc="Unitree Go1 velocity-tracking on the rough box terrain (3564 boxes, curriculum spawn levels <= 5), "
                 "{envs} envs/GPU, random-action agent, decimation 4, dt 0.005, Newton<=10 it / ls<=20, implicitfast, "
                 "pyramidal, foot-friction DR, resets+pushes",
            model="go1_rough", robot="go1"),
  # not a BASELINE config: config E's terrain with the four height-field sub-terrains the reference keeps commented
  # out of ROUGH_TERRAINS_CFG (terrains/config.py:28-55) switched on — exercises csrc/b2_convex.h
  "F": dict(desc="Unitree Go1 velocity-tracking on the rough terrain with height fields (2374 boxes + 70 hfields of 80x80 "
                 "samples: pyramid slopes, random rough, waves), {envs} envs/GPU, random-action agent, decimation 4, "
                 "dt 0.005, Newton<=10 it / ls<=20, implicitfast, pyramidal, foot-friction DR, resets+pushes",
            model="go1_rough_hf", robot="go1"),
}
WORKLOAD = WORKLOADS["B"]["desc"]


def make_env(workload: str, envs: int, seed: int, dev: str):
  from mjlab_b200.envs import TrackingEnvCfg, TrackingFlatEnv, VelocityEnvCfg, VelocityFlatEnv

  if workload == "C":
    return TrackingFlatEnv(TrackingEnvCfg(num_envs=envs, seed=seed), device=dev)
  if workload in ("E", "F"):
    return VelocityFlatEnv(VelocityEnvCfg(robot="go1", terrain="rough" if workload == "E" else "rough_hf",
                                          num_envs=envs, seed=seed), device=dev)
  return VelocityFlatEnv(VelocityEnvCfg(num_envs=envs, seed=seed), device=dev)


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, out) -> None:
  """obs, reward, terminated, truncated and the extras' tensors of one env step, as float32 .npy files.  Above
  DUMP_MAX_BYTES in all, a fixed seeded sample of env rows is written, with its indices as env_ids.npy."""
  import numpy as np

  obs, reward, terminated, truncated, extras = out
  arrays = {"obs": obs, "reward": reward, "terminated": terminated, "truncated": truncated, **extras}
  arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
  n = len(reward)
  row_bytes = sum(a.nbytes for a in arrays.values()) // n
  if row_bytes * n > DUMP_MAX_BYTES:
    rows = (DUMP_MAX_BYTES - 128 * (len(arrays) + 1)) // (row_bytes + 8)  # (128: a .npy header)
    ids = np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    arrays = {k: a[ids] for k, a in arrays.items()}
    arrays["env_ids"] = ids.astype(np.float64)
  d = Path(out_dir)
  d.mkdir(parents=True, exist_ok=True)
  for k, a in arrays.items():
    np.save(d / f"{k}.npy", a)


def _peaks():
  p = ROOT / "MEASURED_PEAKS.json"
  if p.exists():
    return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
  return 6650.0, "fallback"


def _issue_roofline(kern_ms: float, envs: int, clocks) -> dict:
  """The roofline that actually binds this kernel: warp-instruction issue slots (4 schedulers per SM, one warp
  instruction per cycle each).  Instructions per environment come from the committed ncu capture of the same
  kernel and workload (profiles/step_kernel_traffic.json: smsp__inst_executed.sum / envs); time is this run's."""
  tp = ROOT / "profiles" / "step_kernel_traffic.json"
  try:
    t = json.loads(tp.read_text())
    ipe, sms = float(t["warp_inst_per_env"]), int(t.get("sms", 148))
  except Exception:
    return {"bound": "issue", "frac": None, "note": "no warp_inst_per_env in profiles/step_kernel_traffic.json"}
  mhz = (clocks or {}).get("sm_mhz") or 1965.0
  achieved = ipe * envs / (kern_ms * 1e-3)
  peak = sms * 4 * mhz * 1e6
  return {"bound": "issue", "achieved": achieved, "peak": peak, "unit": "warp-inst/s", "frac": achieved / peak,
          "warp_inst_per_env": ipe, "source": t.get("source", "profiles/")}


class ClockSampler:
  """SM clock / throttle-reason sampling during the timed region (B200_PROFILING.md clocks line).

  NVML is polled from a thread every 5 ms (the timed region of the default run is ~150 ms, shorter than the
  start-up time of an `nvidia-smi -lms` child process, which remains the fallback)."""

  Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
       "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
       "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

  def __init__(self, index: int):
    self.index = index
    self.proc = None
    self.path = None
    self.thread = None
    self.samples = []      # (sm_mhz, reasons bit mask)
    self.smax = None
    self._stop = False

  def _nvml_handle(self):
    import pynvml
    import torch

    pynvml.nvmlInit()
    try:
      uuid = str(torch.cuda.get_device_properties(self.index).uuid)
      if not uuid.startswith("GPU-"):
        uuid = "GPU-" + uuid
      return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
    except Exception:
      return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

  def start(self):
    try:
      nv, h = self._nvml_handle()
      self.smax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
      nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
      get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons

      def loop():
        while not self._stop:
          try:
            self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(get_reasons(h))))
          except Exception:
            pass
          time.sleep(0.005)

      self.thread = threading.Thread(target=loop, daemon=True)
      self.thread.start()
      return
    except Exception:
      self.thread = None
    try:
      self.path = tempfile.mktemp(suffix=".csv")
      self.proc = subprocess.Popen(
        ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
         "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
    except Exception:
      self.proc = None

  def stop(self):
    if self.thread is not None:
      self._stop = True
      self.thread.join(timeout=2)
      if not self.samples:
        return {"sm_mhz": None, "sm_max_mhz": self.smax, "reasons": ["no samples"]}
      sm = sorted(x[0] for x in self.samples)
      bits = 0
      for _, r in self.samples:
        bits |= r
      # nvml.h: SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
      names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
      return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.smax,
              "reasons": sorted(v for k, v in names.items() if bits & k), "samples": len(sm), "source": "nvml"}
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except Exception:
      self.proc.kill()
    sm, smax, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    try:
      for line in open(self.path):
        f = [x.strip() for x in line.split(",")]
        if len(f) < 9:
          continue
        sm.append(float(f[1]))
        smax.append(float(f[2]))
        for k, nm in enumerate(names):
          if f[5 + k].lower().startswith("active"):
            reasons.add(nm)
    except Exception:
      pass
    if not sm:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
    sm.sort()
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "reasons": sorted(reasons),
            "samples": len(sm), "source": "nvidia-smi"}


def physical_cores() -> list[int]:
  """One logical CPU per physical core among those this process may run on (hyper-thread siblings dropped)."""
  try:
    allowed = sorted(os.sched_getaffinity(0))
  except AttributeError:
    allowed = list(range(os.cpu_count() or 1))
  seen, out = set(), []
  for c in allowed:
    try:
      sib = Path(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read_text().strip()
    except OSError:
      sib = str(c)
    if sib not in seen:
      seen.add(sib)
      out.append(c)
  return out


def _pinned_env(ncores: int) -> dict:
  """Environment of the CPU arm's process: one OpenMP thread per physical core, pinned (torchrun exports
  OMP_NUM_THREADS=1 to its workers and torch's own OpenMP runtime is already initialised in this process, so the
  arm runs in a child whose runtime starts with these settings)."""
  env = dict(os.environ)
  # (the core count travels with it: once the runtime has bound the main thread to its place, the child's own
  # affinity mask no longer shows the other cores)
  env.update(OMP_NUM_THREADS=str(ncores), OMP_PROC_BIND="close", OMP_PLACES="cores", OMP_DYNAMIC="false",
             B2_CPU_ARM_PINNED="1", B2_CPU_ARM_CORES=str(ncores))
  return env


class CpuPort:
  """The CPU port of the hot path (oracle, fp32, OpenMP static over envs) on a bounded sample of the
  same workload: keyframe + reset noise, settled onto the ground, random actions, 4 sub-steps per
  env step.  Test infrastructure used here only as the *measured baseline*, never by the product."""

  def __init__(self, envs_per_thread: int = 128, nthreads: int | None = None, workload: str = "B"):
    import re

    import numpy as np

    from mjlab_b200.asset_zoo import g1, go1, load_compiled
    from oracle.oracle import Oracle

    self.np = np
    wl = WORKLOADS[workload]
    zoo = g1 if wl["robot"] == "g1" else go1
    m = load_compiled(wl["model"])
    self.cores = nthreads or int(os.environ.get("B2_CPU_ARM_CORES", 0)) or len(physical_cores())
    self.pinned = os.environ.get("B2_CPU_ARM_PINNED") == "1"
    self.n = max(self.cores * envs_per_thread, 8)
    self.o = Oracle(m, nworld=self.n, maxcon=48, precision="f32")
    self.rng = np.random.default_rng(42)
    self.key = m.keys["robot/init_state"]
    qpos = np.tile(self.key["qpos"], (self.n, 1))
    qpos[:, 0:2] += self.rng.uniform(-0.5, 0.5, (self.n, 2))
    if "terrain_origins" in m.arrays:  # rough terrain: spawn on sub-terrain origins of the lower levels
      org = np.asarray(m.arrays["terrain_origins"])[:6].reshape(-1, 3)
      qpos[:, 0:3] += org[self.rng.integers(0, len(org), self.n)]
    yaw = self.rng.uniform(-3.14, 3.14, self.n)
    qpos[:, 3], qpos[:, 6] = np.cos(yaw / 2), np.sin(yaw / 2)
    self.o.qpos[:] = qpos
    names = [x.split("/")[-1] for x in m.names["joint"][1:]]
    self.scale = np.array(
      [next((v for p, v in zoo.ACTION_SCALE.items() if re.match(p, nm)), 0.5) for nm in names])
    self.o.ctrl[:] = self.key["ctrl"]
    for _ in range(40):  # settle onto the ground (untimed) so the sample carries the contact load
      self.o.step(self.cores)

  def env_step(self) -> float:
    t0 = time.perf_counter()
    self.o.ctrl[:] = self.key["ctrl"] + self.scale * self.rng.uniform(-1, 1, (self.n, len(self.scale)))
    for _ in range(4):
      self.o.step(self.cores)
    return time.perf_counter() - t0

  def measure(self, env_steps: int, repeats: int = 3, min_seconds: float = 4.0) -> dict:
    """`repeats` timed blocks of at least `env_steps` env steps and `min_seconds` each (10-30 s of CPU work in
    all): value = median block, spread = (max - min) / median."""
    self.env_step()  # warm caches / thread pool
    vals, secs, total_steps = [], 0.0, 0
    for _ in range(repeats):
      dt, k = 0.0, 0
      while k < env_steps or dt < min_seconds:
        dt += self.env_step()
        k += 1
      secs += dt
      total_steps += k
      vals.append(self.n * k / dt)
    vals.sort()
    v = vals[len(vals) // 2]
    return {
      "value": v, "unit": UNIT, "cores": self.cores, "kind": "port",
      "per_core": v / self.cores, "repeats": vals, "spread": (vals[-1] - vals[0]) / v,
      "threads": f"{self.cores} OpenMP threads, one per physical core, " +
                 ("pinned (OMP_PROC_BIND=close, OMP_PLACES=cores)" if self.pinned else "NOT pinned"),
      "sample": f"{self.n} envs ({self.n // self.cores} per thread) x {total_steps} env-steps in {repeats} blocks (x4 sub-steps), fp32 "
                f"restated CPU oracle (not C-MuJoCo, not mujoco_warp-CPU), OpenMP static over envs, {secs:.1f} s",
    }


def cpu_reference_throughput(env_steps: int = 4, workload: str = "B"):
  """The cpu_baseline leg: the pinned CPU arm in a child process (see _pinned_env); returns its description."""
  cores = len(physical_cores())
  r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", workload,
                      "--steps", str(3 * env_steps), "--warmup", "1"],
                     capture_output=True, text=True, env={**_pinned_env(cores), "RANK": "0", "WORLD_SIZE": "1"}, timeout=900)
  for line in reversed(r.stdout.splitlines()):
    if line.startswith("{"):
      return json.loads(line)["cpu_baseline"]
  raise RuntimeError(f"cpu arm produced no line: {r.stderr[-300:]}")


def run_reference(args):
  """--impl reference: the reference's physics cannot be installed here (mujoco / mujoco_warp /
  warp wheels absent, no network; DESIGN.md §7), so this arm times the CPU port of the same path on
  all physical host cores (pinned); each step is one env step of a bounded sample of the workload.  Rank 0 only."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  if os.environ.get("B2_CPU_ARM_PINNED") != "1":
    # re-run in a child whose OpenMP runtime starts pinned with one thread per physical core
    r = subprocess.run([sys.executable, str(ROOT / "bench.py")] + sys.argv[1:], env=_pinned_env(len(physical_cores())))
    sys.exit(r.returncode)
  t0 = time.perf_counter()
  port = CpuPort(workload=args.workload)
  K = max(1, min(args.steps, 36) // 3)  # three timed blocks; bounded so the whole arm ends within a few minutes
  cb = port.measure(K, repeats=3)
  v = cb["value"]
  line = {
    "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
    "steps": 3 * K, "warmup": args.warmup, "ms_per_step": 1e3 * port.n / v,
    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
    "data": "synthetic", "config": {"workload": WORKLOADS[args.workload]["desc"].format(envs=args.envs),
                                     "config_id": args.workload,
                                     "note": "CPU port of the hot path on host cores (the reference's mujoco_warp / C-MuJoCo "
                                             "cannot be installed in this image); each step = one env step of a "
                                             f"bounded sample ({port.n} envs)"},
    "reference_runnable": False, "impl_detail": "cpu_port (restated oracle, fp32, OpenMP)", "gpus_used": 0,
    "cpu_baseline": cb,
    "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    "wall_s": time.perf_counter() - t0,
  }
  print(json.dumps(line))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=50)
  ap.add_argument("--warmup", type=int, default=10)
  ap.add_argument("--impl", default="b200")
  ap.add_argument("--envs", type=int, default=4096)
  ap.add_argument("--workload", default="B", choices=sorted(WORKLOADS), help="SURVEY.md §8d config: B (headline), C, E")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-flush", action="store_true")
  ap.add_argument("--preroll", type=int, default=100, help="untimed env steps before warm-up")
  ap.add_argument("--no-graph", action="store_true", help="do not capture the env step in a CUDA graph")
  ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
  args = ap.parse_args()
  if args.impl == "reference":
    return run_reference(args)

  import ctypes

  import torch
  import torch.distributed as dist

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  torch.cuda.set_device(local)
  dev = f"cuda:{local}"
  if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device(dev))
  W = max(args.warmup, 3)
  K = args.steps
  env = make_env(args.workload, args.envs, 42 + rank, dev)
  n, nu = env.num_envs, env.nu
  gen = torch.Generator(device=dev)
  gen.manual_seed(1234 + rank)
  flush_buf = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)
  from mjlab_b200.dist import EnvLogGather

  # the one collective of the data-parallel path: per-env (reward, done) to rank 0 for logging
  gathers = {"device": EnvLogGather(n, dev, every=LOG_EVERY), "host": EnvLogGather(n, dev, every=LOG_EVERY)}

  def run(kind: str, steps: int, timed: bool):
    """kind: 'device' (actions resident) or 'host' (pinned host actions, results read back)."""
    ev = []
    phys_ms = 0.0
    host_actions = None
    # stream-ordered when steps are enqueued back to back, side stream when the host syncs every step
    gather_logs = gathers[kind]
    if kind == "host":
      host_actions = [(torch.rand((n, nu)) * 2 - 1).pin_memory() for _ in range(steps)]
      out_r = torch.empty(n, pin_memory=True)
      out_d = torch.empty((n, 2), dtype=torch.bool).pin_memory()
      out_o = None
    for k in range(steps):
      if flush_buf is not None:
        flush_buf.zero_()
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      if kind == "host":
        action = host_actions[k].to(dev, non_blocking=True)
      else:
        action = torch.rand((n, nu), generator=gen, device=dev) * 2 - 1
      out = env.step(action)
      obs, reward, terminated, truncated, _ = out
      gather_logs(env.log_row)  # packed (reward, terminated, truncated), written by the env step itself
      if kind == "host":
        out_r.copy_(reward, non_blocking=True)
        out_d.copy_(torch.stack([terminated, truncated], dim=1), non_blocking=True)
        if out_o is None:
          out_o = torch.empty(obs.shape, pin_memory=True)
        out_o.copy_(obs, non_blocking=True)
        e1.record()
        e1.synchronize()  # the caller consumes the result before issuing the next action
      else:
        e1.record()
      ev.append((e0, e1))
    # the log gather runs on a side stream; its tail after the last step belongs to the timed region
    j0, j1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    j0.record()
    gather_logs.join()
    j1.record()
    torch.cuda.synchronize()
    total = sum(a.elapsed_time(b) for a, b in ev) + j0.elapsed_time(j1)
    # (with the CUDA graph the returned tensors are its static outputs: the next step overwrites them)
    return total, (n * nu * 4, n * 4 + n * 2 + (obs.numel() * 4)) if kind == "host" else None, out

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def maxr(x: float) -> float:
    if world == 1:
      return x
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  # launches of OUR kernels per env step (counted eagerly; graph replays do not pass through Python)
  l0 = env.sim.launch_count()
  run("device", 1, False)
  launches_per_step = env.sim.launch_count() - l0

  # Pre-roll to the steady-state mix of standing / falling / freshly reset robots (all envs start
  # standing at t=0, so without it the timed window would measure a transient), then W warm-up steps.
  run("device", args.preroll, False)
  # ---- kernel-only timing: the decimation's sub-step launches replayed from their own CUDA graph (no launch
  # gaps, like inside the env-step graph), one replay after every env step of a short pass so that the states
  # keep the workload's distribution.  Feeds the roofline; 4 x kernel_ms <= ms_per_step by construction.
  dec = env.cfg.decimation
  side = torch.cuda.Stream(dev)
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    env.sim.step_n(dec)
    g_phys = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_phys, stream=side):
      env.sim.step_n(dec)
  torch.cuda.current_stream().wait_stream(side)
  phys_ms, reps = 0.0, max(W, 8)
  for _ in range(reps):
    env.step(torch.rand((n, nu), generator=gen, device=dev) * 2 - 1)
    if flush_buf is not None:
      flush_buf.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    g_phys.replay()
    b.record()
    torch.cuda.synchronize()
    phys_ms += a.elapsed_time(b)
  kern_ms = maxr(phys_ms / (reps * dec))
  if not args.no_graph:
    env.enable_cuda_graph()
  run("device", W, False)  # warm-up (untimed)
  sampler = ClockSampler(local)
  barrier()
  if rank == 0:
    sampler.start()
  wall0 = time.perf_counter()
  total_ms, _, out = run("device", K, True)
  barrier()
  wall = time.perf_counter() - wall0
  clocks = sampler.stop() if rank == 0 else None
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, out)
  launches = launches_per_step * K
  total_ms = maxr(total_ms)
  st = env.sim.stats()
  import ctypes
  sb, wb = ctypes.c_double(), ctypes.c_double()
  env.sim._lib.b2_algorithmic_bytes(env.sim._h, env.sim._stream(), ctypes.byref(sb), ctypes.byref(wb))

  # ---- end-to-end through host buffers -----------------------------------------------------------
  run("host", W, False)
  barrier()
  e2e_ms, (h2d, d2h), _ = run("host", K, True)
  barrier()
  e2e_ms = maxr(e2e_ms)

  # ---- the plugin call itself: b2_step_host (C ABI, HOST buffers in and out, copies inside the call) -------
  import numpy as np

  ctrl_h = torch.empty((n, nu), pin_memory=True)
  qpos_h = torch.empty((n, env.nq), pin_memory=True)
  qvel_h = torch.empty((n, env.nv), pin_memory=True)
  base_ctrl = env.sim.data.ctrl[:].cpu()
  cabi_ev = []
  for k in range(W + K):
    ctrl_h.copy_(base_ctrl + 0.1 * (torch.rand((n, nu)) * 2 - 1))
    if flush_buf is not None:
      flush_buf.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = env.sim._lib.b2_step_host(env.sim._h, ctypes.c_void_p(ctrl_h.data_ptr()), dec, ctypes.c_void_p(qpos_h.data_ptr()),
                                   ctypes.c_void_p(qvel_h.data_ptr()), env.sim._stream())
    assert rc == 0
    e1.record()
    e1.synchronize()
    if k >= W:
      cabi_ev.append(e0.elapsed_time(e1))
  cabi_ms = maxr(sum(cabi_ev))
  assert np.isfinite(qpos_h.numpy()).all()

  if rank == 0:
    peak, which = _peaks()
    value = world * n * K / (total_ms * 1e-3)
    e2e = world * n * K / (e2e_ms * 1e-3)
    achieved = wb.value / (kern_ms * 1e-3) / 1e9
    traffic = None
    tp = ROOT / "profiles" / "step_kernel_traffic.json"
    if tp.exists():
      traffic = json.loads(tp.read_text()).get("dram_bytes_per_launch")
    line = {
      "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
      "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "f32", "data": "synthetic",
      "config": {
        "workload": WORKLOADS[args.workload]["desc"].format(envs=n), "config_id": args.workload,
        "envs_per_gpu": n, "decimation": 4,
        "parallelism": f"dp{world} (envs sharded, no physics coupling; (reward, done) rows all-gathered to every rank "
                       f"once per {LOG_EVERY} env steps, same packing at 1 GPU)",
        "env_step": "one CUDA-graph replay per env step" if not args.no_graph else "eager",
        "l2": "flushed between timed steps (256 MiB memset, untimed)" if flush_buf is not None else "not flushed",
        "preroll_env_steps": args.preroll,
        "mean_ncon": st.ncon_mean, "mean_nefc": st.nefc_mean, "mean_newton_iters": st.niter_mean,
        "overflow_worlds": st.overflow_worlds,
      },
      "clocks": clocks,
      "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
              "ms_per_step": e2e_ms / K,
              "path": "env.step through the public Python API: pinned host actions in, reward/done/obs out every step"},
      "e2e_cabi": {"value": world * n * K / (cabi_ms * 1e-3), "unit": UNIT, "ms_per_step": cabi_ms / K,
                   "h2d_bytes_per_step": n * nu * 4, "d2h_bytes_per_step": n * (env.nq + env.nv) * 4,
                   "path": "b2_step_host (include/b2sim.h): host ctrl in, 4 sub-steps, host qpos/qvel out; physics only, no MDP terms"},
      "gpu_launches": int(launches),
      "roofline": {
        "kernel": "b2_step_kernel<true> (fused physics sub-step)", "bound": "hbm",
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "peak_source": which, "traffic": traffic, "kernel_ms": kern_ms,
        "algorithmic_bytes_per_launch": wb.value,
        "note": "whole-step minimal traffic (state in/out + consumer-visible kinematics); the kernel is "
                "latency/ALU bound, the constraint Jacobian never exists in HBM",
        "solver_formula_gbs": sb.value / (kern_ms * 1e-3) / 1e9,
      },
      "roofline_issue": _issue_roofline(kern_ms, n, clocks),
      "physics_only_env_steps_per_sec": world * n / (4 * kern_ms * 1e-3),
      "wall_s": wall,
    }
    if not args.no_cpu_baseline and world == 1:
      try:
        line["cpu_baseline"] = cpu_reference_throughput(workload=args.workload)
      except Exception as e:  # the oracle is test infrastructure; never fail the bench on it
        line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                "sample": f"failed: {e}"}
    print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


if __name__ == "__main__":
  main()
