"""One cache for values derived from tensors: packed weights, composite matrices, catalogue tables, propagated embeddings, graph indices."""
from __future__ import annotations

import weakref

import torch


def _stamp(s):
    if isinstance(s, torch.Tensor):
        return id(s), s.data_ptr(), s.shape, s.dtype, s.device, s._version
    return None if s is None else id(s)


class Derived:
    """Up to `capacity` values, each derived from a tuple of sources (tensors, `None`s or other weak-referenceable objects such as a
    `GraphIndex`).  An entry hits only while every source is the SAME live object (checked through a weak reference, so a new object at a
    freed address or `id` misses) and a tensor source keeps its address, shape, dtype, device and `_version` (an in-place op, `.to()` or
    `p.data = ...` misses).  An edit through `.data` (`p.data.copy_()`) bumps nothing: such code calls `invalidate_caches()`.
    Nothing is stored while grad mode is on and a source requires grad; the value is still returned.  A full store is emptied."""

    def __init__(self, capacity: int = 1):
        self.capacity = capacity
        self._entries = {}

    def get(self, sources: tuple, build, *extra):
        """The value stored for `sources` and the hashable key parts `extra`, else `build()` (stored as described above)."""
        key = tuple(map(_stamp, sources)) + extra
        hit = self._entries.get(key)
        if hit is not None and all(s is None or r() is s for r, s in zip(hit[0], sources)):
            return hit[1]
        value = build()
        if not (torch.is_grad_enabled() and any(getattr(s, 'requires_grad', False) for s in sources)):
            if len(self._entries) >= self.capacity:
                self._entries.clear()
            self._entries[key] = (tuple(None if s is None else weakref.ref(s) for s in sources), value)
        return value

    def clear(self):
        self._entries.clear()

    def values(self):
        return [v for _, v in self._entries.values()]

    def __len__(self):
        return len(self._entries)

    def __reduce__(self):                        # a pickled / deep-copied model starts empty (weak references do not pickle)
        return Derived, (self.capacity,)
