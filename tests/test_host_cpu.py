"""Host-side logic that needs no GPU: C-ABI symbol surface, bridge/TorchArray semantics (the
reference's tests/test_sim_data.py on plain tensors), product-has-no-CPU-path, gloo collectives."""

import ctypes
import os
import re
from pathlib import Path
from types import SimpleNamespace

import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


def test_c_abi_exports_every_declared_symbol():
  import __graft_entry__ as g

  g.build()
  hdr = (ROOT / "include" / "b2sim.h").read_text()
  declared = set(re.findall(r"\b(b2_[a-z_0-9]+)\s*\(", hdr))
  assert {"b2_create", "b2_step", "b2_forward", "b2_get_field", "b2_expand_model_field",
          "b2_step_host", "b2_forward_masked"} <= declared
  lib = ctypes.CDLL(str(ROOT / "mjlab_b200" / "csrc" / "libb2sim.so"))
  for sym in declared:
    assert hasattr(lib, sym), f"{sym} declared in include/b2sim.h but not exported"
  lib.b2_version.restype = ctypes.c_char_p
  assert b"sm_100a" in lib.b2_version()


def test_library_is_built_for_sm_100a_with_tma():
  import subprocess

  so = ROOT / "mjlab_b200" / "csrc" / "libb2sim.so"
  out = subprocess.run(["cuobjdump", "-sass", str(so)], capture_output=True, text=True).stdout
  assert "sm_100a" in out
  assert "UBLKCP" in out  # cp.async.bulk (TMA 1-D) staging of the env state


def test_product_has_no_cpu_fallback(g1_model):
  from mjlab_b200.sim import Simulation, SimulationCfg

  with pytest.raises(RuntimeError, match="no CPU path"):
    Simulation(2, SimulationCfg(), g1_model, "cpu")
  if not torch.cuda.is_available():
    with pytest.raises(RuntimeError):
      Simulation(2, SimulationCfg(), g1_model, "cuda:0")
  # the product package never imports the oracle
  for p in (ROOT / "mjlab_b200").rglob("*.py"):
    assert "oracle" not in p.read_text().replace("# oracle", ""), p


def test_missing_extension_fails_loudly(monkeypatch, tmp_path):
  from mjlab_b200.sim import native

  monkeypatch.setattr(native, "_lib", None)
  monkeypatch.setattr(native, "LIB_PATH", tmp_path / "nope.so")
  with pytest.raises(RuntimeError, match="There is no CPU fallback"):
    native.load_library()


def test_torch_array_and_bridge_semantics():
  from mjlab_b200.sim.sim_data import Bridge, TorchArray

  struct = SimpleNamespace(qpos=torch.zeros(3, 5), nworld=3, nested=7)
  br = Bridge(struct)
  q = br.qpos
  assert isinstance(q, TorchArray) and q is br.qpos  # cached wrapper (test_sim_data.py:84-89)
  assert br.nworld == 3
  q[:, 1] = 2.0
  assert struct.qpos[0, 1] == 2.0  # shares memory (:37-43)
  ptr = q.data_ptr()
  q[:] = 5.0
  assert q.data_ptr() == ptr  # slice assignment keeps the address (:62-70)
  assert torch.sum(q).item() == 75.0 and torch.cat([q, q]).shape == (6, 5)  # torch functions (:46-52)
  assert ((q * 2 - 1) == 9).all() and ((2 + q) / 7 == 1).all() and (-q < 0).all()
  assert q.shape == (3, 5) and q.numpy().shape == (3, 5)
  with pytest.raises(AttributeError, match=r"Cannot set attribute 'qpos' on WarpBridge.*obj.qpos\[:\] = value"):
    br.qpos = torch.ones(3, 5)  # (:73-81)
  # advanced indexing with (N,1) int64 env ids and int32 column ids on a strided view (entity/data.py:86-87)
  base = torch.arange(3 * 8, dtype=torch.float32).reshape(3, 8)
  view = TorchArray(base.as_strided((3, 5), (8, 1)))
  env_ids = torch.tensor([[0], [2]])
  cols = torch.tensor([1, 3], dtype=torch.int32)
  view[env_ids, cols] = -1.0
  assert base[2, 3] == -1.0 and base[1, 3] == 11.0
  assert view[env_ids, cols].shape == (2, 2)


def test_model_desc_roundtrip(g1_model):
  from mjlab_b200.sim.native import make_model_desc

  desc, keep = make_model_desc(g1_model)
  names = {desc.arrays[i].name.decode(): desc.arrays[i] for i in range(desc.narray)}
  assert names["nq"].n == 1 and names["body_pos"].n == 3 * int(g1_model.nbody)
  assert names["pair_geom1"].dtype == 1 and names["geom_friction"].dtype == 0
  assert tuple(desc.gravity) == (0.0, 0.0, -9.81)


def _gloo_worker(rank, world, port, q):
  os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
  import torch.distributed as dist

  from mjlab_b200 import dist as b2dist

  r, w = b2dist.init(backend="gloo")
  n = 16
  lo, hi = b2dist.shard_range(world * n, r, w)
  g = b2dist.EnvLogGather(n, "cpu", every=4)
  reward = torch.arange(lo, hi, dtype=torch.float32)
  # six env steps: one gather after the 4th row (ring full), join() flushes the 2 rows of the next round
  for k in range(4):
    out = g(reward + 100.0 * k, reward % 2 == 0, reward % 3 == 0)
  assert g.flushes == 1
  first = out.clone()
  packed = torch.stack([reward + 400.0, (reward % 2 == 0).float(), (reward % 3 == 0).float()], dim=1)
  g(packed)  # a row the env packed itself (b2_velenv_post writes env.log_row)
  g(packed + 0.0)
  assert g.flushes == 1
  out = g.join()
  assert g.flushes == 2 and g.join() is out and g.flushes == 2
  q.put((r, first[:, 0, :, 0].flatten().tolist(), first[:, 3, :, 0].flatten().tolist(), out[:, 0, :, 0].flatten().tolist(),
         b2dist.EnvLogGather.summarize(first[:, 0])))
  dist.destroy_process_group()


def test_env_log_gather_world_size_2_gloo():
  import torch.multiprocessing as mp

  ctx = mp.get_context("spawn")
  q = ctx.Queue()
  port = 29611
  procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
  for p in procs:
    p.start()
  res = sorted(q.get(timeout=120) for _ in procs)
  for p in procs:
    p.join(timeout=60)
    assert p.exitcode == 0
  for _, row0, row3, row4, summ in res:
    assert row0 == [float(i) for i in range(32)]  # every rank sees the whole job, rank order, step order
    assert row3 == [float(i) + 300.0 for i in range(32)] and row4 == [float(i) + 400.0 for i in range(32)]
    assert summ["terminated"] == 16 and summ["truncated"] == 11


def test_shard_range():
  from mjlab_b200.dist import shard_range

  assert shard_range(32768, 3, 8) == (12288, 16384)
  with pytest.raises(ValueError):
    shard_range(10, 0, 3)


def test_b2_create_rejects_malformed_model_tables(g1_model):
  """The descriptor is checked on the host before any device work: wrong sizes, out-of-range indices and models the
  engine does not support are refused with a message (no compute happens here; on a CPU box a valid table ends at
  'no CUDA device')."""
  import copy
  import ctypes

  import numpy as np

  from mjlab_b200.asset_zoo import load_compiled
  from mjlab_b200.sim import native

  lib = native.load_library()
  lib.b2_last_error.restype = ctypes.c_char_p

  def create(model):
    desc, keep = native.make_model_desc(model)
    h = ctypes.c_void_p()
    rc = lib.b2_create(ctypes.byref(desc), 2, 0, 0, 0, ctypes.byref(h))
    msg = lib.b2_last_error(None).decode() if rc else ""
    if rc == 0:
      lib.b2_destroy(h)
    return rc, msg

  def set_at(index, value):
    def mod(a):
      a = a.copy()
      a[index] = value
      return a
    return mod

  terrain = load_compiled("go1_rough")
  for model in (g1_model, terrain):
    rc, msg = create(model)
    assert rc == 0 or "no CUDA device" in msg  # the unmodified table passes validation
  # a terrain geom moved onto the first body with a joint (the trunk)
  trunk = int(np.flatnonzero(np.asarray(terrain.arrays["body_jntnum"]))[0])
  static_on_trunk = set_at(int(np.asarray(terrain.arrays["static_geom"])[0]), trunk)
  cases = [
    (g1_model, "dof_parentid", lambda a: a[:-1], "has 34 elements, expected 35"),
    (g1_model, "pair_geom1", lambda a: np.where(np.arange(len(a)) == 3, 999, a).astype(np.int32), "index out of range"),
    (g1_model, "geom_size", lambda a: a[:-1], "'geom_size' has"),
    (g1_model, "body_parentid", lambda a: np.where(np.arange(len(a)) == 2, 5, a).astype(np.int32), "parents must precede children"),
    # the checks below follow the table checks; none of them needs a device
    (g1_model, "pair_geom2", set_at(0, 0), "unsupported geom type combination"),  # the floor (geom 0) against itself
    (g1_model, "opt_solver", lambda a: np.zeros_like(a), "solver must be Newton or CG"),
    (g1_model, "opt_cone", lambda a: np.ones_like(a), "only pyramidal cones are supported"),
    (g1_model, "sensor_intprm", set_at((0, 0), 1 | 4), "contact sensor data/reduce combination not implemented"),
    (terrain, "geom_bodyid", static_on_trunk, "grid-static geoms must sit on a jointless child of the world body"),
  ]
  for model, field, mod, expect in cases:
    m2 = copy.deepcopy(model)
    m2.arrays[field] = np.ascontiguousarray(mod(np.asarray(model.arrays[field])))
    rc, msg = create(m2)
    assert rc != 0 and expect in msg, (field, msg)


def test_bench_reference_arm_prints_one_contract_line():
  """`bench.py --impl reference` (the CPU arm the driver launches, also under torchrun where OMP_NUM_THREADS=1):
  one JSON line with the contract's keys, all available cores in use."""
  import json
  import os
  import subprocess
  import sys

  root = Path(__file__).resolve().parents[1]
  env = dict(os.environ, OMP_NUM_THREADS="1")
  out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=600)
  assert out.returncode == 0, out.stderr[-500:]
  lines = [l for l in out.stdout.splitlines() if l.strip()]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
  assert d["higher_is_better"] is True and d["value"] > 0 and d["e2e"]["value"] == d["value"]
  assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
  assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
  # rank != 0 of a torchrun launch exits quietly
  env["RANK"] = "1"
  out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=120)
  assert out.returncode == 0 and out.stdout.strip() == ""
