"""Load the reference's own modules (installed unmodified under oracle/_ref by oracle/install_reference.py)
on top of mjlab_b200.compat, for the drop-in tests.

Only the packages whose ``__init__`` drags in viewers / RL / terrain tooling that the image lacks (viser,
trimesh, prettytable, gymnasium, tyro ...) are entered as *namespace stubs*: ``mjlab.envs``, ``mjlab.envs.mdp``,
``mjlab.managers`` (and ``mjlab.scene`` if its real import fails) get an empty module object whose ``__path__`` points at the real
directory, so their submodules (``envs/mdp/events.py``, ``managers/scene_entity_config.py`` ...) are executed
from the reference's files, byte for byte, without running the package ``__init__``.
"""

from __future__ import annotations

import sys
import types
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
REF = ROOT / "oracle" / "_ref"


def available() -> bool:
  return (REF / "mjlab" / "entity" / "data.py").exists()


def load():
  """Returns the namespace of reference modules used by the tests (idempotent)."""
  import mjlab_b200.compat as compat

  shimmed = compat.install()
  if str(REF) not in sys.path:
    sys.path.insert(0, str(REF))
  try:  # the scene package imports cleanly on the stand-ins (its terrain generators only need numpy here)
    import mjlab.scene  # noqa: F401
  except Exception:  # noqa: BLE001
    sys.modules.pop("mjlab.scene", None)
  for name in ("mjlab.envs", "mjlab.envs.mdp", "mjlab.managers", "mjlab.scene"):
    if name not in sys.modules:
      mod = types.ModuleType(name)
      mod.__path__ = [str(REF / Path(*name.split(".")))]
      mod.__b2_stub__ = True
      sys.modules[name] = mod
  if not hasattr(sys.modules["mjlab.scene"], "Scene"):
    sys.modules["mjlab.scene"].Scene = type("Scene", (), {})  # only a type annotation in scene_entity_config.py
  import mjlab  # noqa: F401  (configure_warp() runs against the stand-in)
  import mjlab.entity.data as entity_data
  import mjlab.entity.entity as entity
  import mjlab.envs.mdp.events as events
  import mjlab.managers.scene_entity_config as scene_entity_config
  import mjlab.sim.randomization as randomization
  import mjlab.sim.sim as sim
  import mjlab.sim.sim_data as sim_data
  import mjlab.utils.nan_guard as nan_guard

  for mod in (entity_data, entity, events, sim, sim_data, randomization, nan_guard, scene_entity_config):
    assert Path(mod.__file__).resolve().is_relative_to(REF.resolve()), mod.__file__
  return types.SimpleNamespace(
    shimmed=shimmed, entity_data=entity_data, entity=entity, events=events, sim=sim, sim_data=sim_data,
    randomization=randomization, nan_guard=nan_guard, scene_entity_config=scene_entity_config)
