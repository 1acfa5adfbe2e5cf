"""
Config-driven sequential x-vector network with the reference's surface
(/root/reference/kaldi_tflite/lib/models/kaldi/sequential.py:29-143):
`cfg2layers`, `SequentialFromConfig(cfg, nnet3Path, name)`.

The returned `Sequential` keeps the reference's one-object-per-layer view (`.layers`,
`get_layer`, `set_weights` per layer) but executes a FUSED plan: every
affine [-> relu] [-> batchnorm] run becomes one kernel (bias/ReLU/BN in the epilogue), and a
following reduce-all StatsPooling consumes per-utterance sums produced by that kernel's
epilogue when the engine provides them.
"""

from typing import Iterable

import numpy as np
import torch

from .. import _tensor as T
from ..io import KaldiNnet3Reader
from ..layers import TDNN, BatchNorm, ReLU, StatsPooling
from ..layers.base import Layer


def cfg2layers(layerCfg: dict) -> Iterable[Layer]:
    layerTypes = layerCfg.get("type", [])
    if isinstance(layerTypes, str):
        layerTypes = [layerTypes]
    if len(layerTypes) == 0:
        raise KeyError("layer config does not define layer 'type'")
    name = layerCfg.get("name", None)
    layers = []
    for layerType in layerTypes:
        t = layerType.lower()
        cfg = dict(layerCfg.get("cfg", {}))
        if t in ["affine", "tdnn"]:
            cfg["name"] = f"{name}.affine"
            layer = TDNN(**cfg)
        elif t in ["relu"]:
            layer = ReLU(name=f"{name}.relu")
        elif t in ["batchnorm", "bn"]:
            layer = BatchNorm(name=f"{name}.batchnorm")
        elif t in ["stats", "stats_extraction", "stats_pooling"]:
            cfg["name"] = name
            layer = StatsPooling(**cfg)
        else:
            raise ValueError(f"unsupported layer type '{t}'")
        layers.append(layer)
    return layers


class Sequential:

    def __init__(self, layers, input_shape=None, name=None, precision=None):
        self.layers = list(layers)
        self.name = name
        self.input_shape = input_shape          # (batch, timesteps, featDim), entries may be None
        self.precision = precision
        self.dtype = "float32"
        self._plan = None
        self._stack = None
        self._plan_version = None
        if input_shape is not None and input_shape[-1] is not None:
            self._build_layers(input_shape[-1])

    def _build_layers(self, feat_dim):
        dim = feat_dim
        for l in self.layers:
            if isinstance(l, (TDNN, BatchNorm)):
                l._maybe_build((None, None, dim))
            if isinstance(l, TDNN):
                dim = l.units
            elif isinstance(l, StatsPooling):
                dim = dim * 2 if l.includeStd else dim

    def get_layer(self, name):
        for l in self.layers:
            if l.name == name:
                return l
        raise ValueError(f"No such layer: {name}")

    def invalidate(self):
        """Drop the fused plan.  Not needed after `layer.set_weights(...)`: every forward compares the layers' weight
        versions with the ones the plan was built from (keras applies set_weights immediately; so does this)."""
        self._plan = None

    def _weights_version(self):
        return tuple(l._weights_version for l in self.layers)

    def _resolved_precision(self):
        from ..layers import tdnn as _t
        return (self.precision or _t.DEFAULT_PRECISION).lower()

    def _try_stack(self, plan):
        """bf16: run the whole [affine]* -> stats(reduce) -> [affine]* network as ONE tcgen05 stack."""
        from ..layers.tdnn import _Stack
        affines, stats_after, stats = [], -1, None
        for kind, obj, st in plan:
            if kind != "affine" or not obj.same or not obj.bf16:
                return None
            affines.append(obj)
            if st is not None:
                if stats is not None:
                    return None
                stats, stats_after = st, len(affines) - 1
        if stats_after >= 0:
            for a in affines[stats_after + 1:]:
                if a.context != [0]:
                    return None
        return _Stack(affines, stats_after, stats.includeStd if stats else True,
                      stats.epsilon if stats else 1e-10)

    def _make_plan(self):
        plan, i, L = [], 0, self.layers
        while i < len(L):
            l = L[i]
            if isinstance(l, TDNN):
                relu, bn, j = False, None, i + 1
                if j < len(L) and isinstance(L[j], ReLU):
                    relu, j = True, j + 1
                if j < len(L) and isinstance(L[j], BatchNorm):
                    bn, j = L[j], j + 1
                scale = offset = None
                if bn is not None:
                    scale, offset = bn.scale_offset()
                aff = l.make_affine(relu=relu, bn_scale=scale, bn_offset=offset, precision=self.precision)
                stats = None
                if j < len(L) and isinstance(L[j], StatsPooling) and L[j].reduce and L[j].inputPeriod == 1:
                    stats, j = L[j], j + 1
                plan.append(("affine", aff, stats))
                i = j
            elif isinstance(l, StatsPooling):
                plan.append(("stats", l, None))
                i += 1
            else:
                plan.append(("layer", l, None))
                i += 1
        return plan

    def _ensure_plan(self, feat_dim):
        if self._plan is None or self._plan_version != self._weights_version():
            self._build_layers(feat_dim)
            self._plan = self._make_plan()
            self._plan_version = self._weights_version()
            self._stack = self._try_stack(self._plan)       # None unless every layer runs on the tcgen05 engine

    def fused_vad_cmvn_stack(self, feat_dim, cmvn_window=None, max_frames=None):
        """The tcgen05 stack if it can take un-normalised features + a VAD index list directly (fused pre-pass).  With
        `cmvn_window` and `max_frames` (an upper bound on the longest utterance), only if the pre-pass fits them."""
        self._ensure_plan(feat_dim)
        if self._stack is None or not self._stack.can_fuse_vad_cmvn(cmvn_window, max_frames):
            return None
        return self._stack

    def forward_ragged(self, x2d, offsets):
        """x2d CUDA (rows, D); utterance b = rows offsets[b]..offsets[b+1].  Returns (y2d, offsets)."""
        self._ensure_plan(x2d.shape[-1])
        B = offsets.numel() - 1
        if self._stack is not None:
            y = self._stack.forward_ragged(x2d, offsets)
            return y, (T.uniform_offsets(B, 1) if self._stack.pools else offsets)
        for kind, obj, stats in self._plan:
            if kind == "affine":
                if stats is not None:
                    _, sums, out_offs = obj.forward_ragged(x2d, offsets, want_y=False, want_stats=True)
                    x2d = stats.finalize_sums(sums, out_offs)
                    offsets = T.uniform_offsets(B, 1)
                else:
                    x2d, _, offsets = obj.forward_ragged(x2d, offsets)
            elif kind == "stats":
                if not obj.reduce:
                    raise NotImplementedError("windowed StatsPooling is only supported on uniform batches "
                                              "(call the model with a (batch, T, D) tensor)")
                x2d = obj.reduce_ragged(x2d, offsets)
                offsets = T.uniform_offsets(B, 1)
            else:
                rows = x2d.shape[0]
                x2d = T.as_device(obj(x2d[None]))[0]
                assert x2d.shape[0] == rows
        return x2d, offsets

    def __call__(self, inputs, training=False):
        x = T.as_device(inputs)
        if x.dim() != 3:
            raise ValueError(f"expected input of shape (batch, timesteps, feats), got {tuple(x.shape)}")
        B, Tn, D = x.shape
        windowed = any(isinstance(l, StatsPooling) and not l.reduce for l in self.layers)
        if windowed:                                   # generic layer-by-layer path
            y = x
            for l in self.layers:
                y = T.as_device(l(y))
            return T.like_input(y, inputs)
        y, offs = self.forward_ragged(x.reshape(B * Tn, D), T.uniform_offsets(B, Tn))
        return T.like_input(y.reshape(B, -1, y.shape[-1]), inputs)

    def summary(self):
        for l in self.layers:
            print(f"{l.name:32s} {type(l).__name__}")


def SequentialFromConfig(cfg: dict, nnet3Path: str = None, name: str = None, precision: str = None,
                         seed: int = None) -> Sequential:
    layersConfig = cfg.get("layers", [])
    if len(layersConfig) == 0:
        raise ValueError("no layers defined in config")
    inputCfg = layersConfig[0]
    if inputCfg.get("type", "") != "input":
        raise ValueError("first layer in sequential model needs to be of type 'input'")
    batchSize, timesteps, featDim = inputCfg["shape"]

    layers = []
    for lCfg in cfg["layers"][1:]:
        layers.extend(cfg2layers(lCfg))
    if seed is not None:                               # reproducible random init (weights absent)
        for i, l in enumerate(layers):
            if isinstance(l, TDNN):
                l._seed = seed + i
    mdl = Sequential(layers, input_shape=(batchSize, timesteps, featDim), name=name, precision=precision)

    if nnet3Path is not None:
        nnet3Mdl = KaldiNnet3Reader(nnet3Path, True)
        for layer in mdl.layers:
            try:
                layer.set_weights(nnet3Mdl.getWeights(layer.name))
            except KeyError:
                print(f"component with name '{layer.name}' not found in nnet3 model, "
                      "skipping initialization")
    return mdl
