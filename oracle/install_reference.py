"""Install the UNMODIFIED reference package (mujocolab/mjlab, pure Python) and its own test files into oracle/_ref,
so that the drop-in tests can import its modules (entity/data.py, envs/mdp/events.py, sim/sim_data.py ...) and run
its tests against mjlab_b200.compat.  oracle/_ref is a build product: git-ignored, so no reference source enters the
history, and made from a checkout of the reference named ``reference`` beside this repository or beside one of its
parent directories (or the one ``MJLAB_REFERENCE`` names).  Without such a checkout nothing is installed and the tests
that need oracle/_ref skip.

The install is a file copy of ``src/mjlab`` (the layout pip gives a src-layout package) without the mesh files
(29 MB of STL that nothing here reads), plus ``tests/*.py``.  No file is edited.
"""
import os
import shutil
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
TARGET = ROOT / "oracle" / "_ref"
SKIP = (".stl", ".pyc")


def find_reference() -> Path | None:
  env = os.environ.get("MJLAB_REFERENCE")
  cands = [Path(env)] if env else [d / "reference" for d in ROOT.parents]
  for c in cands:
    if os.path.isdir(c / "src" / "mjlab") and os.path.isdir(c / "tests"):  # (isdir: unreadable parents are absent)
      return c
  return None


def _copy(src: Path, dst: Path, top_only: bool = False) -> None:
  for d, dirs, files in os.walk(src):
    if top_only:
      dirs.clear()
    dirs[:] = [x for x in dirs if x != "__pycache__"]
    out = dst / Path(d).relative_to(src)
    out.mkdir(parents=True, exist_ok=True)
    for f in files:
      if not f.lower().endswith(SKIP):
        shutil.copyfile(Path(d) / f, out / f)  # contents only: the checkout may be read-only


def install(force: bool = False) -> bool:
  done = TARGET / "mjlab" / "entity" / "data.py"
  if done.exists() and not force:
    return True
  ref = find_reference()
  if ref is None:
    return done.exists()
  TARGET.parent.mkdir(exist_ok=True)
  tmp = Path(tempfile.mkdtemp(prefix="_ref.", dir=TARGET.parent))
  try:
    tmp.chmod(0o755)
    _copy(ref / "src" / "mjlab", tmp / "mjlab")
    _copy(ref / "tests", tmp / "tests", top_only=True)
    shutil.rmtree(TARGET, ignore_errors=True)
    tmp.rename(TARGET)
  finally:
    shutil.rmtree(tmp, ignore_errors=True)
  return done.exists()


if __name__ == "__main__":
  ok = install(force="--force" in sys.argv)
  print("oracle/_ref:", "installed" if ok else "NOT installed (no reference checkout found)")
