"""MLP builder and checkpoint loader with the reference's parameter layout (neural_collaborative_filtering/util.py)."""
from __future__ import annotations

import torch
from torch import nn

from .. import ops


def build_MLP_layers(input_size, layer_sizes, dropout_rate, output_size=1) -> nn.Sequential:
    """Parameter container laid out exactly like the reference's (util.py:5-18): Linear, then per further layer
    ReLU, [Dropout when dropout_rate is not None], Linear; the last Linear has `output_size` outputs.  This fixes the
    state_dict keys (`MLP.0`, `MLP.3`, `MLP.6`, ... or `MLP.0`, `MLP.2`, ... without dropout).  The modules are never
    called: `run_mlp` feeds their weights to the fused CUDA tower."""
    widths = [input_size, *layer_sizes, output_size]
    mods = []
    for n, (fan_in, fan_out) in enumerate(zip(widths[:-1], widths[1:])):
        if n:
            mods.append(nn.ReLU())
            if dropout_rate is not None:
                mods.append(nn.Dropout(dropout_rate))
        mods.append(nn.Linear(fan_in, fan_out))
    return nn.Sequential(*mods)


def mlp_parameters(mlp: nn.Sequential):
    lin = [m for m in mlp if isinstance(m, nn.Linear)]
    drops = [m.p for m in mlp if isinstance(m, nn.Dropout)]
    return [m.weight for m in lin], [m.bias for m in lin], (drops[0] if drops else 0.0)


def run_mlp(mlp: nn.Sequential, in0, in1, idx0=None, idx1=None, training=False, generator=None):
    """MLP([in0[idx0], in1[idx1]]) -> (B, 1).  Eval (or inert dropout): one fused kernel, activations stay in shared
    memory.  Training with dropout p > 0: layer-by-layer through the CUDA linear kernel with torch's Bernoulli mask in
    between (the reference's Philox stream cannot be bit-matched anyway, SURVEY.md §7.3).  `generator`: draw the masks from
    it instead of torch's default generator (partitioned training: the same masks on every rank)."""
    weights, biases, p = mlp_parameters(mlp)
    if not (training and p > 0.0):
        return ops.mlp_tower(in0, in1, weights, biases, idx0, idx1)
    xa = in0[idx0] if idx0 is not None else in0
    x = torch.cat((xa, in1[idx1] if idx1 is not None else in1), dim=1) if in1 is not None else xa
    last = len(weights) - 1
    for n, (w, b) in enumerate(zip(weights, biases)):
        x = ops.linear(x, w, b, relu=n < last)
        if n < last:
            if generator is None:
                x = torch.nn.functional.dropout(x, p, training=True)
            else:
                x = x * torch.empty_like(x).bernoulli_(1.0 - p, generator=generator).div_(1.0 - p)
    return x


def load_model(file, ModelClass=None, map_location=None, **kargs):
    """Reads a `[state_dict, kwargs]` checkpoint (models/base.py:18-19 of the reference).  `map_location` is new: the
    reference's loader (util.py:27) cannot open its own CUDA-saved checkpoints on another device."""
    state, kwargs = torch.load(file, map_location=map_location, weights_only=False)
    kwargs = dict(kwargs, **kargs)
    if ModelClass is None:
        return state, kwargs
    model = ModelClass(**kwargs)
    model.load_state_dict(state)
    return model
