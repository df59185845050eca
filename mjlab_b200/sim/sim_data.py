"""Zero-copy torch views of engine memory with the semantics of the reference's
``TorchArray`` / ``WarpBridge`` (``src/mjlab/sim/sim_data.py:15-229``).

Differences by design: there is no Warp array underneath — a field is a (possibly strided)
``torch.Tensor`` created over the device pointer returned by ``b2_get_field`` — and physics is
enqueued on torch's *current* stream, so writes through ``__setitem__`` need no stream switch
(SURVEY.md §8b "Threading").
"""

from __future__ import annotations

import ctypes
from typing import Any, Dict, Optional, Tuple

import torch

from mjlab_b200.sim import native


class _RawCudaBuffer:
  """Minimal ``__cuda_array_interface__`` carrier for a device pointer owned by libb2sim."""

  def __init__(self, ptr: int, nbytes: int, owner: Any):
    self._owner = owner  # keeps the simulation (and therefore the allocation) alive
    self.__cuda_array_interface__ = {
      "shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2, "strides": None,
    }


def tensor_from_b2(t: native.B2Tensor, owner: Any) -> torch.Tensor:
  """Wrap a ``B2Tensor`` as a torch tensor sharing the engine's memory."""
  shape = tuple(int(t.shape[k]) for k in range(t.ndim))
  stride = tuple(int(t.stride[k]) for k in range(t.ndim))
  dtype = torch.int32 if t.dtype == 1 else torch.float32
  span = 1 + sum((s - 1) * st for s, st in zip(shape, stride) if s > 0)
  if any(s == 0 for s in shape) or not t.ptr:
    return torch.empty(shape, dtype=dtype, device=f"cuda:{t.device}")
  raw = torch.as_tensor(_RawCudaBuffer(int(t.ptr), span * 4, owner), device=f"cuda:{t.device}")
  return raw.view(dtype).as_strided(shape, stride)


class TorchArray:
  """Engine array that behaves like a ``torch.Tensor`` sharing its memory."""

  def __init__(self, tensor: torch.Tensor) -> None:
    self._tensor = tensor

  def __repr__(self) -> str:
    return repr(self._tensor)

  def __getitem__(self, idx: Any) -> Any:
    return self._tensor[idx]

  def __setitem__(self, idx: Any, value: Any) -> None:
    self._tensor[idx] = value

  def __getattr__(self, name: str) -> Any:
    return getattr(self._tensor, name)

  def __len__(self) -> int:
    return len(self._tensor)

  def numpy(self):
    """Host copy (the reference's viewers call ``wp_array.numpy()``, ``viewer/viser.py:557``)."""
    return self._tensor.detach().cpu().numpy()

  @classmethod
  def __torch_function__(
    cls, func: Any, types: Tuple[type, ...], args: Tuple[Any, ...] = (),
    kwargs: Optional[Dict[str, Any]] = None,
  ) -> Any:
    kwargs = kwargs or {}
    if not any(issubclass(t, cls) for t in types):
      return NotImplemented

    def unwrap(x: Any) -> Any:
      if isinstance(x, cls):
        return x._tensor
      if isinstance(x, (list, tuple)):
        return type(x)(unwrap(y) for y in x)
      return x

    return func(*tuple(unwrap(a) for a in args), **{k: unwrap(v) for k, v in kwargs.items()})

  # arithmetic / comparison dunders delegate to the tensor
  def __add__(self, o): return self._tensor + o
  def __radd__(self, o): return o + self._tensor
  def __sub__(self, o): return self._tensor - o
  def __rsub__(self, o): return o - self._tensor
  def __mul__(self, o): return self._tensor * o
  def __rmul__(self, o): return o * self._tensor
  def __truediv__(self, o): return self._tensor / o
  def __rtruediv__(self, o): return o / self._tensor
  def __pow__(self, o): return self._tensor ** o
  def __rpow__(self, o): return o ** self._tensor
  def __neg__(self): return -self._tensor
  def __pos__(self): return +self._tensor
  def __abs__(self): return abs(self._tensor)
  def __eq__(self, o): return self._tensor == o
  def __ne__(self, o): return self._tensor != o
  def __lt__(self, o): return self._tensor < o
  def __le__(self, o): return self._tensor <= o
  def __gt__(self, o): return self._tensor > o
  def __ge__(self, o): return self._tensor >= o
  __hash__ = None  # type: ignore[assignment]


class Bridge:
  """Attribute view of the engine's Data or Model struct (the reference's ``WarpBridge``).

  Array attributes come back as cached :class:`TorchArray` objects; assignment is refused so
  addresses captured by CUDA graphs never change (``sim_data.py:214-220``)."""

  def __init__(self, struct: Any) -> None:
    object.__setattr__(self, "_struct", struct)
    object.__setattr__(self, "_wrapped_cache", {})

  def __getattr__(self, name: str) -> Any:
    cache = object.__getattribute__(self, "_wrapped_cache")
    if name in cache:
      return cache[name]
    val = getattr(object.__getattribute__(self, "_struct"), name)
    if isinstance(val, torch.Tensor):
      val = TorchArray(val)
      cache[name] = val
    return val

  def __setattr__(self, name: str, value: Any) -> None:
    raise AttributeError(
      f"Cannot set attribute '{name}' on WarpBridge. "
      f"This wrapper is read-only to preserve memory addresses for CUDA graphs. "
      f"Use in-place operations instead: obj.{name}[:] = value"
    )

  def _invalidate(self, name: str) -> None:
    object.__getattribute__(self, "_wrapped_cache").pop(name, None)

  def __repr__(self) -> str:
    return f"WarpBridge({object.__getattribute__(self, '_struct')!r})"

  @property
  def struct(self) -> Any:
    return object.__getattribute__(self, "_struct")


WarpBridge = Bridge


class EngineStruct:
  """Lazily materialised tensors of one side (Data or Model) of a ``b2_sim``."""

  def __init__(self, sim: Any, which: int, extra: Optional[dict] = None) -> None:
    self._sim = sim
    self._which = which
    self._tensors: dict[str, torch.Tensor] = {}
    self._extra = extra or {}
    lib = sim._lib
    self._names = [
      lib.b2_field_name(sim._h, which, i).decode() for i in range(lib.b2_num_fields(sim._h, which))
    ]

  def __getattr__(self, name: str) -> Any:
    if name.startswith("_"):
      raise AttributeError(name)
    if name in self._extra:
      return self._extra[name]
    if self.__dict__.get("_closed"):
      raise RuntimeError(f"Simulation is closed: field '{name}' no longer exists (engine memory was freed)")
    if name in self._tensors:
      return self._tensors[name]
    if name not in self._names:
      raise AttributeError(f"engine struct has no field '{name}'")
    t = native.B2Tensor()
    native.check(self._sim._lib.b2_get_field(self._sim._h, self._which, name.encode(), ctypes.byref(t)))
    tensor = tensor_from_b2(t, self._sim)
    self._tensors[name] = tensor
    if self._which == 1:
      # a writable model view can switch the engine off its cached kinematic records, which a captured graph holds
      # by value: re-capture before the next replay
      self._sim._graph_dirty = True
    return tensor

  def _drop(self, name: str) -> None:
    self._tensors.pop(name, None)

  def __dir__(self):
    return list(self._names) + list(self._extra)
