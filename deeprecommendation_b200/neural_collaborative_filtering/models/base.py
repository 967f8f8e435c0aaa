"""Model base classes: the reference's plugin API (neural_collaborative_filtering/models/base.py:6-42)."""
from __future__ import annotations

import torch
from torch import nn

from ...derived import Derived


def _named_like(dataset_class, *names) -> bool:
    """True if the class (ours or the reference's own) derives from a dataset class with one of these names, so the
    reference's `train.py:40` compatibility check passes with either package's datasets."""
    return any(c.__name__ in names for c in getattr(dataset_class, '__mro__', ()))


class NCF(nn.Module):
    """forward / get_model_parameters / save_model / is_dataset_compatible / important_hypeparams + `.kwargs`."""

    kwargs: dict

    def forward(self, *args):
        raise NotImplementedError

    def get_model_parameters(self) -> dict:
        return self.kwargs

    def save_model(self, file):
        # same on-disk format as the reference: [state_dict, constructor kwargs]
        torch.save([self.state_dict(), self.get_model_parameters()], file)

    def is_dataset_compatible(self, dataset_class) -> bool:
        raise NotImplementedError

    def important_hypeparams(self) -> str:
        return ''

    # ---- derived copies of the weights (packed MMA tiles, composite / transposed matrices, cached embeddings) -----------------------
    # They are kept in `derived.Derived` stores (the model's own are attributes of it) and reused only while every source is the same live
    # tensor at the same address with the same `_version`.  Loading a state dict, moving / casting the module, or editing parameters through
    # `.data` (which does NOT bump `_version`) must drop them: the first two are hooked here, the third is what `invalidate_caches()` is for.
    def invalidate_caches(self):
        from ... import ops
        ops.invalidate_caches()
        for v in self.__dict__.values():
            if isinstance(v, Derived):
                v.clear()

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.invalidate_caches()
        return out

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self.invalidate_caches()
        return out


class GNN_NCF(NCF):
    """forward(graph, userIds, itemIds, device, ...) -> (B, 1); ids are NODE ids (items first)."""
