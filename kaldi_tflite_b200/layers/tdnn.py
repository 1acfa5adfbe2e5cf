"""
TDNN affine layer and ReLU with the reference's constructor surface
(/root/reference/kaldi_tflite/lib/layers/tdnn/{tdnn,utils}.py; keras ReLU as used by
models/kaldi/sequential.py:71-72).
"""

import ctypes

import numpy as np
import torch

from .. import _native as N
from .. import _tensor as T
from .base import Layer

PRECISIONS = {"f32": N.KTF_PREC_F32, "fp32": N.KTF_PREC_F32, "float32": N.KTF_PREC_F32,
              "bf16": N.KTF_PREC_BF16, "bfloat16": N.KTF_PREC_BF16}

# Operand precision of TDNN contractions when a layer does not say otherwise: bf16 operands with fp32 accumulation on the
# tcgen05 engine (BASELINE.json north_star: "x-vectors with cosine >= 0.9999 at TF32/bf16 TDNN precision").  "f32" selects
# the exact fp32 SIMT tiles (the precision reference of the tests).
DEFAULT_PRECISION = "bf16"


def reshapeKaldiTdnnWeights(weights, units, kernel_width):
    """Kaldi (U, K*D) -> TF kernel (1, K, D, U): kernel[0,k,d,u] = W[u, k*D+d] (utils.py:22-28)."""
    w = np.asarray(weights)
    if w.ndim != 2 or w.shape[0] != units or w.shape[1] % kernel_width != 0:
        raise ValueError(f"cannot reshape weights of shape {w.shape} for units={units}, "
                         f"kernel width={kernel_width}")
    D = w.shape[1] // kernel_width
    return np.ascontiguousarray(w.reshape(units, kernel_width, D).transpose(1, 2, 0)[None])


def kernelToKaldi(kernel):
    """Inverse of reshapeKaldiTdnnWeights: (1, K, D, U) -> (U, K*D)."""
    k = np.asarray(kernel)
    _, K, D, U = k.shape
    return np.ascontiguousarray(k[0].transpose(2, 0, 1).reshape(U, K * D))


class _Affine:
    """Owns one ktf_affine handle: splice + contraction + bias + activation + BN scale/offset."""

    def __init__(self, w_kaldi, bias, context, subsampling=1, padding="SAME", relu=False,
                 bn_scale=None, bn_offset=None, precision=None):
        N.require_cuda()
        w = np.ascontiguousarray(w_kaldi, dtype=np.float32)
        K = len(context)
        U, KD = w.shape
        assert KD % K == 0
        self.in_dim, self.out_dim, self.context = KD // K, U, list(context)
        prec = PRECISIONS[(precision or DEFAULT_PRECISION).lower()]
        self.bf16 = prec == N.KTF_PREC_BF16
        cfg = N.AffineCfg(in_dim=self.in_dim, out_dim=U, num_context=K, subsampling_factor=subsampling,
                          padding_valid=int(padding.upper() == "VALID"),
                          activation=N.KTF_ACT_RELU if relu else N.KTF_ACT_NONE, precision=prec)
        for i, c in enumerate(context):
            cfg.context[i] = int(c)
        b = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
        s = None if bn_scale is None else np.ascontiguousarray(bn_scale, dtype=np.float32)
        o = None if bn_offset is None else np.ascontiguousarray(bn_offset, dtype=np.float32)
        self.handle = ctypes.c_void_p()
        N.check(N.lib().ktf_affine_create(ctypes.byref(cfg), T.host_ptr(w), T.host_ptr(b), T.host_ptr(s),
                                          T.host_ptr(o), ctypes.byref(self.handle)))
        self.same = padding.upper() == "SAME" and subsampling == 1

    def __del__(self):
        try:
            if self.handle:
                N.lib().ktf_affine_destroy(self.handle)
        except Exception:
            pass

    def out_rows(self, T_in):
        return int(N.lib().ktf_affine_out_rows(self.handle, T_in))

    def forward_ragged(self, x2d, in_offsets, out_offsets=None, out_rows=None, want_y=True,
                       want_stats=False):
        """x2d (rows, D) -> y (out_rows, U) and/or per-utterance sums (B, 2, U)."""
        rows, D = x2d.shape
        if D != self.in_dim:
            raise ValueError(f"expected input feature dimension {self.in_dim}, got {D}")
        B = in_offsets.numel() - 1
        if out_offsets is None:
            if self.same:
                out_offsets, out_rows = in_offsets, rows
            else:
                lens = (in_offsets[1:] - in_offsets[:-1]).cpu().tolist()
                oo = np.zeros(B + 1, dtype=np.int64)
                oo[1:] = np.cumsum([self.out_rows(int(l)) for l in lens])
                out_offsets, out_rows = torch.from_numpy(oo).to(x2d.device), int(oo[-1])
        y = torch.empty((out_rows, self.out_dim), device=x2d.device, dtype=torch.float32) if want_y else None
        stats = torch.empty((B, 2, self.out_dim), device=x2d.device, dtype=torch.float32) if want_stats else None
        N.check(N.lib().ktf_affine_forward(self.handle, T.ptr(x2d), T.ptr(in_offsets), T.ptr(out_offsets),
                                           B, rows, out_rows, T.ptr(y), T.ptr(stats), T.stream_ptr()))
        return y, stats, out_offsets

    def forward_uniform(self, x):
        B, Tn, D = x.shape
        To = self.out_rows(Tn)
        y, _, _ = self.forward_ragged(x.reshape(B * Tn, D), T.uniform_offsets(B, Tn),
                                      T.uniform_offsets(B, To), B * To)
        return y.reshape(B, To, self.out_dim)


class _Stack:
    """Owns one ktf_tdnn_stack: the whole affine/ReLU/BN (+ reduce-all stats) network on the tcgen05 engine."""

    def __init__(self, affines, stats_after=-1, include_std=True, epsilon=1e-10):
        N.require_cuda()
        self.affines = list(affines)                 # keep the borrowed handles alive
        arr = (ctypes.c_void_p * len(affines))(*[a.handle for a in affines])
        self.handle = ctypes.c_void_p()
        N.check(N.lib().ktf_tdnn_stack_create(arr, len(affines), stats_after, int(include_std),
                                              float(epsilon), ctypes.byref(self.handle)))
        self.out_dim = int(N.lib().ktf_tdnn_stack_out_dim(self.handle))
        self.pools = stats_after >= 0

    def __del__(self):
        try:
            if self.handle:
                N.lib().ktf_tdnn_stack_destroy(self.handle)
        except Exception:
            pass

    def forward_ragged(self, x2d, offsets):
        rows, _ = x2d.shape
        B = offsets.numel() - 1
        out = torch.empty((B if self.pools else rows, self.out_dim), device=x2d.device, dtype=torch.float32)
        N.check(N.lib().ktf_tdnn_stack_forward(self.handle, T.ptr(x2d), T.ptr(offsets), B, rows, T.ptr(out),
                                               T.stream_ptr()))
        return out

    def can_fuse_vad_cmvn(self, cmvn_window=None, max_frames=None):
        """First layer with consecutive contexts: the VAD gather + CMVN + splice pre-pass applies.  Given the CMVN window
        and the longest utterance, also whether the pre-pass tile fits in shared memory (ktf_tdnn_stack_vad_prepass_fits)."""
        ctx = self.affines[0].context
        if not (all(c == ctx[0] + k for k, c in enumerate(ctx)) and max(abs(c) for c in ctx) <= 4):
            return False
        if cmvn_window is None:
            return True
        return bool(N.lib().ktf_tdnn_stack_vad_prepass_fits(self.handle, int(cmvn_window), int(max_frames)))

    def forward_vad(self, feats2d, index, offsets, max_frames, cmvn_window):
        """Un-normalised features + VAD index list + compacted offsets -> stack output (ktf_tdnn_stack_forward_vad)."""
        rows, _ = feats2d.shape
        B = offsets.numel() - 1
        out = torch.empty((B if self.pools else rows, self.out_dim), device=feats2d.device, dtype=torch.float32)
        N.check(N.lib().ktf_tdnn_stack_forward_vad(self.handle, T.ptr(feats2d), T.ptr(index), T.ptr(offsets), B, rows,
                                                   int(max_frames), int(cmvn_window), T.ptr(out), T.stream_ptr()))
        return out


def glorot_uniform(shape, rng):
    """keras GlorotUniform: U(-l, l), l = sqrt(6 / (fan_in + fan_out)) (tdnn.py:50-51)."""
    if len(shape) == 1:
        fan_in = fan_out = shape[0]
    else:
        receptive = int(np.prod(shape[:-2]))
        fan_in, fan_out = shape[-2] * receptive, shape[-1] * receptive
    limit = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-limit, limit, size=shape).astype(np.float32)


class TDNN(Layer):
    """tdnn.py:44-280."""

    def __init__(self, units, context=[0], subsampling_factor=1, padding="SAME", use_bias=True,
                 kernel_initializer=None, bias_initializer=None, activation=None, name=None,
                 precision=None, seed=None, **kwargs):
        super().__init__(name=name, trainable=True, **kwargs)
        self.units = units
        self.useBias = use_bias
        self.subsamplingFactor = subsampling_factor
        if self.subsamplingFactor <= 0:
            raise ValueError("subsampling_factor should be > 0")
        self.padding = padding.upper()
        if self.padding not in ["VALID", "SAME"]:
            raise ValueError("padding should be either 'VALID' or 'SAME'")
        if context is None:
            ctx = [0]
        elif isinstance(context, int):
            ctx = [context]
        elif isinstance(context, (list, tuple)):
            ctx = list(context) if len(context) > 0 else [0]
        else:
            raise ValueError("context should be None, a list or an integer")
        self.context = sorted(ctx)
        self.kernelWidth = len(self.context)
        self.activation = activation
        if activation not in (None, "relu", "linear"):
            raise NotImplementedError(f"activation '{activation}' is not supported")
        self.precision = precision
        self._seed = seed
        self.kernel = None          # TF layout (1, K, D, U)
        self.bias = None
        self._affine = None

    def build(self, input_shape):
        D = input_shape[-1]
        if self.kernel is None:
            rng = np.random.default_rng(self._seed)
            self.kernel = glorot_uniform((1, self.kernelWidth, D, self.units), rng)
            self.bias = glorot_uniform((self.units,), rng) if self.useBias else None
        elif self.kernel.shape[2] != D:
            raise ValueError(f"kernel expects feature dimension {self.kernel.shape[2]}, input has {D}")
        super().build(input_shape)

    def getStartEndSteps(self, inputTimesteps):
        start, end = 0, inputTimesteps
        if self.padding == "VALID":
            if self.context[0] < 0:
                start = -self.context[0]
            if self.context[-1] > 0:
                end = inputTimesteps - self.context[-1]
        return start, end

    def compute_output_shape(self, input_shape):
        batch, steps = input_shape[0], input_shape[1]
        if steps is None:
            return (batch, None, self.units)
        start, end = self.getStartEndSteps(steps)
        n = max(0, end - start)
        return (batch, (n + self.subsamplingFactor - 1) // self.subsamplingFactor, self.units)

    def get_config(self):
        config = super().get_config()
        config.pop("trainable", None)
        config.update({"units": self.units, "context": self.context,
                       "subsampling_factor": self.subsamplingFactor, "padding": self.padding,
                       "use_bias": self.useBias, "activation": self.activation})
        return config

    def get_weights(self):
        return [self.kernel, self.bias] if self.useBias else [self.kernel]

    def set_weights(self, weights, fmt="kaldi"):
        fmt = fmt.lower()
        if fmt not in ["kaldi", "tensorflow"]:
            raise ValueError(f"expected 'fmt' to be either 'kaldi' or 'tensorflow', got {fmt}")
        if len(weights) == 0:
            raise ValueError("expected a weight list of at least length 2, got 0")
        if self.useBias and len(weights) != 2:
            raise ValueError(f"expected a weight list of length 2, got {len(weights)}")
        kernel = np.asarray(weights[0], dtype=np.float32)
        if fmt == "kaldi":
            kernel = reshapeKaldiTdnnWeights(kernel, self.units, self.kernelWidth)
        if kernel.ndim != 4 or kernel.shape[0] != 1 or kernel.shape[1] != self.kernelWidth \
                or kernel.shape[3] != self.units:
            raise ValueError(f"unexpected kernel shape {kernel.shape}")
        if self.built and self._build_shape[-1] != kernel.shape[2]:
            raise ValueError(f"kernel feature dimension {kernel.shape[2]} != input {self._build_shape[-1]}")
        self.kernel = np.ascontiguousarray(kernel)
        if self.useBias:
            bias = np.asarray(weights[1], dtype=np.float32).reshape(-1)
            if bias.shape[0] != self.units:
                raise ValueError(f"unexpected bias shape {bias.shape}")
            self.bias = bias
        self._affine = None
        self._weights_version += 1

    def kaldi_weights(self):
        return kernelToKaldi(self.kernel), self.bias

    def make_affine(self, relu=False, bn_scale=None, bn_offset=None, precision=None):
        w, b = self.kaldi_weights()
        return _Affine(w, b, self.context, self.subsamplingFactor, self.padding,
                       relu=relu or self.activation == "relu", bn_scale=bn_scale, bn_offset=bn_offset,
                       precision=precision or self.precision)

    def call(self, inputs):
        x = T.as_device(inputs)
        if x.dim() != 3:
            raise ValueError(f"expected input of shape (batch, timesteps, feats), got {tuple(x.shape)}")
        self._maybe_build(x.shape)
        if self._affine is None:
            self._affine = self.make_affine()
        return T.like_input(self._affine.forward_uniform(x), inputs)


class ReLU(Layer):
    """keras.layers.ReLU stand-in."""

    def __init__(self, name=None, **kwargs):
        super().__init__(name=name, trainable=False, **kwargs)

    def call(self, inputs, training=False):
        x = T.as_device(inputs)
        y = torch.empty_like(x)
        N.check(N.lib().ktf_relu_forward(T.ptr(x), x.numel(), T.ptr(y), T.stream_ptr()))
        return T.like_input(y, inputs)
