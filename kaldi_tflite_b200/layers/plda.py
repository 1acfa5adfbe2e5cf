"""
PLDA scoring layer with the reference's constructor surface
(/root/reference/kaldi_tflite/lib/layers/plda/plda.py:41-263).
"""

import ctypes

import numpy as np
import torch

from .. import _native as N
from .. import _tensor as T
from .base import Layer


def _np_dtype(dtype):
    if isinstance(dtype, torch.dtype):
        return {torch.float32: np.float32, torch.float64: np.float64}[dtype]
    name = getattr(dtype, "name", None) or str(dtype)
    if "64" in name or name in ("double", "float"):
        return np.float64
    if "32" in name:
        return np.float32
    return np.dtype(dtype).type


class PLDA(Layer):

    def __init__(self, dim, plda_mean, plda_transform, plda_psi, normalize_length=True,
                 simple_length_norm=False, dtype=np.float64, return_transformed=True, name=None):
        super().__init__(name=name, trainable=False)
        self.dim = int(dim)
        self.normalizeLength = normalize_length
        self.simpleLengthNorm = simple_length_norm
        self.paramDtype = _np_dtype(dtype)
        if self.paramDtype not in (np.float32, np.float64):
            raise ValueError("dtype must be float32 or float64")
        self.returnTransformed = return_transformed
        self.mean = np.ascontiguousarray(plda_mean, dtype=np.float64)
        self.transformMat = np.ascontiguousarray(plda_transform, dtype=np.float64)
        self.psi = np.ascontiguousarray(plda_psi, dtype=np.float64)
        self.assertParamShapes()
        self.inputRank = 3
        self._handles = {}          # one ktf_plda handle per num_examples value

    def assertParamShapes(self):
        assert self.mean.ndim == 1, f"plda_mean must be a vector, got dimension={self.mean.ndim}"
        assert self.psi.ndim == 1, f"plda_psi must be a vector, got dimension={self.psi.ndim}"
        assert self.transformMat.ndim == 2, \
            f"plda_transform_mat must be a matrix, got dimension={self.transformMat.ndim}"
        assert self.mean.shape[0] == self.dim, \
            f"plda_mean dimension size ({self.mean.shape[0]}) != input dim ({self.dim})"
        assert self.psi.shape[0] == self.dim, \
            f"plda_psi dimension size ({self.psi.shape[0]}) != input dim ({self.dim})"
        assert self.transformMat.shape[0] == self.dim, \
            f"plda_transform_mat dimension size ({self.transformMat.shape[0]}) != input dim ({self.dim})"
        assert self.transformMat.shape[0] == self.transformMat.shape[1], \
            f"plda_transform_mat ({self.transformMat.shape[0]} x {self.transformMat.shape[1]}) is not a square matrix"

    def build(self, input_shape):
        if input_shape[-1] != self.dim:
            raise ValueError(f"expected input vector dimension to be {self.dim}, got {input_shape[-1]}")
        self.inputRank = len(input_shape)
        if self.inputRank not in [2, 3]:
            raise ValueError(f"expected input tensor rank to be 2 or 3, got {len(input_shape)}")
        super().build(input_shape)

    def get_config(self):
        config = super().get_config()
        config.update({"dim": self.dim, "normalize_length": self.normalizeLength,
                       "simple_length_norm": self.simpleLengthNorm,
                       "return_transformed": self.returnTransformed})
        return config

    def handle_for(self, num_examples=1.0):
        """The constants of the score depend on how many utterances an enrolled vector averages
        (plda.py:163-182, 215-231), so handles are cached per `num_examples`."""
        key = float(num_examples)
        assert key > 0, "num_examples must be greater than 1"          # plda.py:164
        if key not in self._handles:
            N.require_cuda()
            h = ctypes.c_void_p()
            N.check(N.lib().ktf_plda_create_ex(self.dim, T.host_ptr(self.mean), T.host_ptr(self.transformMat),
                                               T.host_ptr(self.psi), int(self.normalizeLength),
                                               int(self.simpleLengthNorm),
                                               8 if self.paramDtype == np.float64 else 4, key, ctypes.byref(h)))
            self._handles[key] = h
        return self._handles[key]

    @property
    def handle(self):
        return self.handle_for(1.0)

    def __del__(self):
        try:
            for h in self._handles.values():
                N.lib().ktf_plda_destroy(h)
        except Exception:
            pass

    @property
    def torchDtype(self):
        return torch.float64 if self.paramDtype == np.float64 else torch.float32

    def transformVector(self, x2d, num_examples=1.0):
        """(n, dim) float32 CUDA -> (n, dim) in the layer dtype: plda.py:184-196."""
        n = x2d.shape[0]
        u = torch.empty((n, self.dim), device=x2d.device, dtype=self.torchDtype)
        N.check(N.lib().ktf_plda_transform(self.handle_for(num_examples), T.ptr(x2d), n, T.ptr(u), T.stream_ptr()))
        return u

    def logLikelihoodRatio(self, u_test, u_enroll=None, out=None, num_examples=1.0, score_dtype=None):
        """scores[i, j] = LLR(test i | enrolled j): plda.py:215-245 (all-pairs); `num_examples` = utterances averaged
        into each enrolled vector.  `score_dtype=torch.bfloat16` (float32 layers only) writes the compact score matrix
        of SURVEY 8f rank 3: the same fp32-equivalent value, rounded once to bfloat16 -- half the HBM write that bounds
        all-vs-all scoring at dim 128."""
        u_enroll = u_test if u_enroll is None else u_enroll
        nt, ne = u_test.shape[0], u_enroll.shape[0]
        compact = score_dtype is torch.bfloat16 or (out is not None and out.dtype is torch.bfloat16)
        if score_dtype is not None and not compact and score_dtype != self.torchDtype:
            raise ValueError(f"score_dtype must be {self.torchDtype} or torch.bfloat16")
        if compact and self.paramDtype != np.float32:
            raise ValueError("bfloat16 scores need a float32 PLDA layer")
        if out is None:
            out = torch.empty((nt, ne), device=u_test.device, dtype=torch.bfloat16 if compact else self.torchDtype)
        N.check(N.lib().ktf_plda_score_ex(self.handle_for(num_examples), T.ptr(u_test), nt, T.ptr(u_enroll), ne,
                                          T.ptr(out), out.stride(0),
                                          N.KTF_SCORES_BF16 if compact else N.KTF_SCORES_NATIVE, T.stream_ptr()))
        return out

    def bestMatch(self, u_test, u_enroll=None, num_examples=1.0):
        """Best enrolled vector per test vector: (scores (n_test,) float32, indexes (n_test,) int64) with
        scores[i] = max_j LLR(test i | enrolled j) -- the entry of `logLikelihoodRatio` (plda.py:215-245), same
        arithmetic -- without writing the (n_test, n_enroll) matrix (SURVEY 8f rank 3, top-k = 1; float32 layers only).
        The lowest index wins a tie."""
        if self.paramDtype != np.float32:
            raise ValueError("bestMatch needs a float32 PLDA layer")
        u_enroll = u_test if u_enroll is None else u_enroll
        nt, ne = u_test.shape[0], u_enroll.shape[0]
        best = torch.empty((nt,), device=u_test.device, dtype=torch.float32)
        index = torch.empty((nt,), device=u_test.device, dtype=torch.int64)
        N.check(N.lib().ktf_plda_score_top1(self.handle_for(num_examples), T.ptr(u_test), nt, T.ptr(u_enroll), ne,
                                            T.ptr(best), T.ptr(index), T.stream_ptr()))
        return best, index

    def bestMatches(self, u_test, u_enroll=None, *, k, num_examples=1.0):
        """The k best enrolled vectors per test vector, 1 <= k <= 32: (scores (n_test, k) float32, indexes (n_test, k)
        int64), row i = the k largest entries of row i of `logLikelihoodRatio` (same arithmetic, bit for bit) and their
        columns, best first, the lower index first on equal scores -- the first k of a stable descending sort of the row
        -- without writing the (n_test, n_enroll) matrix (float32 layers only).  Past the last enrolled vector the
        entries are (-inf, -1).  `u_enroll=None` scores the set against itself."""
        if self.paramDtype != np.float32:
            raise ValueError("bestMatches needs a float32 PLDA layer")
        k = int(k)
        u_enroll = u_test if u_enroll is None else u_enroll
        nt, ne = u_test.shape[0], u_enroll.shape[0]
        scores = torch.empty((nt, max(k, 0)), device=u_test.device, dtype=torch.float32)
        index = torch.empty((nt, max(k, 0)), device=u_test.device, dtype=torch.int64)
        N.check(N.lib().ktf_plda_score_topk(self.handle_for(num_examples), T.ptr(u_test), nt, T.ptr(u_enroll), ne, k,
                                            T.ptr(scores), T.ptr(index), T.stream_ptr()))
        return scores, index

    def call(self, inputs):
        x = T.as_device(inputs)
        self._maybe_build(x.shape)
        if x.dim() == 3:
            if x.shape[1] != 1:
                raise ValueError(f"expected input of shape (batch, 1, dim), got {tuple(x.shape)}")
            x = x[:, 0, :]
        x = x.contiguous()
        u = self.transformVector(x)
        scores = self.logLikelihoodRatio(u)
        if self.returnTransformed:
            return T.like_input(scores, inputs), T.like_input(u[:, :, None], inputs)
        return T.like_input(scores, inputs)
