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

    def _need_float32(self, caller):
        if self.paramDtype != np.float32:
            raise ValueError(f"{caller} needs a float32 PLDA layer")

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
        self._need_float32("bestMatch")
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
        return self._bestMatches("bestMatches", N.lib().ktf_plda_score_topk, N.KTF_PLDA_TOPK_MAX, u_test, u_enroll, k,
                                 None, num_examples)

    def bestMatchesLarge(self, u_test, u_enroll=None, *, k, num_examples=1.0):
        """`bestMatches` for 1 <= k <= 1024 (shortlists, recall@100, neighbour graphs): (scores (n_test, k) float32,
        indexes (n_test, k) int64), row i = the first k entries of a stable descending sort of row i of
        `logLikelihoodRatio` (same values, bit for bit) and their columns, padded with (-inf, -1) past the last enrolled
        vector, without the (n_test, n_enroll) matrix in memory: k <= 32 runs `bestMatches`, larger k scores row chunks
        of at most 128 MB and selects each while it is in L2.  `u_enroll=None` scores the set against itself.  float32
        layers only."""
        return self._bestMatches("bestMatchesLarge", N.lib().ktf_plda_score_topk_large, N.KTF_PLDA_TOPK_LARGE_MAX,
                                 u_test, u_enroll, k, None, num_examples)

    def _bestMatches(self, caller, c_fn, k_max, u_test, u_enroll, k, stats, num_examples):
        """The k best enrolled vectors per test vector from the native k-best call `c_fn` (1 <= k <= `k_max`): of the
        raw scores, or with `stats` = (u_cohort, top_n, test_stats, enroll_stats) of the AS-norm scores, the statistics
        resolved as in `asNorm`."""
        self._need_float32(caller)
        k = int(k)
        if not 1 <= k <= k_max:
            raise ValueError(f"k = {k}, must be 1 .. {k_max}")
        u_enroll = u_test if u_enroll is None else u_enroll
        nt, ne = u_test.shape[0], u_enroll.shape[0]
        if stats is not None:
            stats = self._asNormStats(u_test, u_enroll, *stats, num_examples, caller)
        scores = torch.empty((nt, k), device=u_test.device, dtype=torch.float32)
        index = torch.empty((nt, k), device=u_test.device, dtype=torch.int64)
        N.check(c_fn(self.handle_for(num_examples), T.ptr(u_test), nt, T.ptr(u_enroll), ne,
                     *(T.ptr(t) for t in (stats or ())), k, T.ptr(scores), T.ptr(index), T.stream_ptr()))
        return scores, index

    def cohortStats(self, u, u_cohort, *, top_n, role="test", num_examples=1.0):
        """AS-norm statistics of every vector of `u` against an imposter cohort: (mean (n,), std (n,)) float32, the
        mean and population std (ddof 0) of its `top_n` largest cohort scores.  role="test": the scores are row i of
        `logLikelihoodRatio(u, u_cohort)` (num_examples 1); role="enrolled": column i of
        `logLikelihoodRatio(u_cohort, u, num_examples=num_examples)`.  The selection is exact (bit-equal scores) and
        the statistics are evaluated in float64 and rounded once; a vector's statistics do not depend on the other
        vectors of the call.  2 <= top_n <= len(u_cohort); float32 layers only."""
        self._need_float32("cohortStats")
        if role not in ("test", "enrolled"):
            raise ValueError(f"role must be 'test' or 'enrolled', got {role!r}")
        n = u.shape[0]
        mean = torch.empty((n,), device=u.device, dtype=torch.float32)
        std = torch.empty((n,), device=u.device, dtype=torch.float32)
        h = self.handle_for(1.0) if role == "test" else self.handle_for(num_examples)
        N.check(N.lib().ktf_plda_cohort_stats(h, T.ptr(u), n, T.ptr(u_cohort), u_cohort.shape[0], int(top_n),
                                              N.KTF_COHORT_AS_TEST if role == "test" else N.KTF_COHORT_AS_ENROLLED,
                                              T.ptr(mean), T.ptr(std), None, T.stream_ptr()))
        return mean, std

    def _asNormStats(self, u_test, u_enroll, u_cohort, top_n, test_stats, enroll_stats, num_examples, caller):
        """The four (mean, std) statistics tensors of an AS-norm call, test side first: those given, checked, and the
        others computed from `u_cohort` and `top_n` (test role for u_test, enrolled role with `num_examples` for
        u_enroll)."""
        nt, ne = u_test.shape[0], u_enroll.shape[0]
        if (test_stats is None or enroll_stats is None) and (u_cohort is None or top_n is None):
            raise ValueError(f"{caller} needs u_cohort and top_n for the statistics it is not given")
        if test_stats is None:
            test_stats = self.cohortStats(u_test, u_cohort, top_n=top_n, role="test")
        if enroll_stats is None:
            enroll_stats = self.cohortStats(u_enroll, u_cohort, top_n=top_n, role="enrolled", num_examples=num_examples)
        stats = []
        for (m, s), n, side in ((test_stats, nt, "test"), (enroll_stats, ne, "enroll")):
            for t in (m, s):
                if t.dtype != torch.float32 or t.shape != (n,) or not t.is_contiguous():
                    raise ValueError(f"{side}_stats must be two contiguous float32 tensors of shape ({n},)")
                stats.append(t)
        return stats

    def asNorm(self, u_test, u_enroll=None, u_cohort=None, *, top_n=None, test_stats=None, enroll_stats=None,
               num_examples=1.0, out=None, score_dtype=None):
        """Adaptive symmetric normalisation (AS-norm1) of the `logLikelihoodRatio` matrix:
        s'[i, j] = 0.5 ((s[i, j] - mu_e[j]) / sigma_e[j] + (s[i, j] - mu_t[i]) / sigma_t[i]), float32 (n_test, n_enroll),
        normalised in the score kernel (the raw matrix is never written).  `test_stats` / `enroll_stats` are
        (mean, std) pairs from `cohortStats`; whichever is not given is computed from `u_cohort` and `top_n`
        (test role for u_test, enrolled role with `num_examples` for u_enroll).  `u_enroll=None` scores the set against
        itself.  `score_dtype=torch.bfloat16` (or a bfloat16 `out`) writes the same float32 value rounded once to
        bfloat16: half the bytes of the matrix.  float32 layers only."""
        self._need_float32("asNorm")
        compact = score_dtype is torch.bfloat16 or (out is not None and out.dtype is torch.bfloat16)
        if score_dtype is not None and not compact and score_dtype != torch.float32:
            raise ValueError("score_dtype must be torch.float32 or torch.bfloat16")
        dtype = torch.bfloat16 if compact else torch.float32
        u_enroll = u_test if u_enroll is None else u_enroll
        nt, ne = u_test.shape[0], u_enroll.shape[0]
        stats = self._asNormStats(u_test, u_enroll, u_cohort, top_n, test_stats, enroll_stats, num_examples, "asNorm")
        if out is None:
            out = torch.empty((nt, ne), device=u_test.device, dtype=dtype)
        elif out.dtype != dtype or tuple(out.shape) != (nt, ne) or out.stride(1) != 1:
            raise ValueError(f"out must be a {dtype} ({nt}, {ne}) tensor with unit column stride")
        N.check(N.lib().ktf_plda_score_asnorm_ex(self.handle_for(num_examples), T.ptr(u_test), nt, T.ptr(u_enroll), ne,
                                                 *(T.ptr(t) for t in stats), T.ptr(out), out.stride(0),
                                                 N.KTF_SCORES_BF16 if compact else N.KTF_SCORES_NATIVE, T.stream_ptr()))
        return out

    def asNormBestMatches(self, u_test, u_enroll=None, u_cohort=None, *, k, top_n=None, test_stats=None,
                          enroll_stats=None, num_examples=1.0):
        """The k best enrolled vectors per test vector by AS-norm score, 1 <= k <= 32: (scores (n_test, k) float32,
        indexes (n_test, k) int64), row i = the first k entries of a stable descending sort of row i of `asNorm` (same
        statistics, same values bit for bit) and their columns, without writing the matrix.  NaN and -inf scores (a
        deviation of 0 can give them) are never listed; past the last listed column the entries are (-inf, -1).  The
        statistics are given or computed as in `asNorm`; `u_enroll=None` scores the set against itself.  float32 layers
        only."""
        return self._bestMatches("asNormBestMatches", N.lib().ktf_plda_score_asnorm_topk, N.KTF_PLDA_TOPK_MAX, u_test,
                                 u_enroll, k, (u_cohort, top_n, test_stats, enroll_stats), num_examples)

    def asNormBestMatchesLarge(self, u_test, u_enroll=None, u_cohort=None, *, k, top_n=None, test_stats=None,
                               enroll_stats=None, num_examples=1.0):
        """`asNormBestMatches` for 1 <= k <= 1024: (scores (n_test, k) float32, indexes (n_test, k) int64), row i = the
        first k entries of a stable descending sort of row i of `asNorm` (same statistics, same values bit for bit) and
        their columns, NaN and -inf scores never listed (+inf is), padded with (-inf, -1), without the matrix in memory:
        k <= 32 runs `asNormBestMatches`, larger k normalises row chunks of at most 128 MB and selects each while it is in
        L2.  The statistics are given or computed as in `asNorm`; `u_enroll=None` scores the set against itself.  float32
        layers only."""
        return self._bestMatches("asNormBestMatchesLarge", N.lib().ktf_plda_score_asnorm_topk_large,
                                 N.KTF_PLDA_TOPK_LARGE_MAX, u_test, u_enroll, k, (u_cohort, top_n, test_stats,
                                                                                  enroll_stats), num_examples)

    def withinScores(self, u, lengths):
        """Within-recording scores for diarization (Kaldi's ivector-plda-scoring-dense without its PCA): recording r is
        the next `lengths[r]` rows of the transformed vectors `u` (float32 CUDA, from `transformVector`), and its
        (n_r, n_r) float32 matrix S_r[i, j] = LLR(enrolled u_i | test u_j), each entry bit-equal to
        `logLikelihoodRatio(u_r)[j, i]`.  Returns one view per recording into a single buffer that packs the matrices
        one after another (the layout `diarization.agglomerative_cluster` takes without a copy); one score launch for
        the whole batch.  float32 layers only."""
        self._need_float32("withinScores")
        lengths = [int(n) for n in lengths]
        if any(n < 0 for n in lengths):
            raise ValueError("lengths must be >= 0")
        offsets = np.concatenate(([0], np.cumsum(lengths, dtype=np.int64))).astype(np.int64)
        if u.dtype != torch.float32 or u.dim() != 2 or u.shape[1] != self.dim or not u.is_contiguous():
            raise ValueError(f"u must be a contiguous float32 (n, {self.dim}) tensor")
        if int(offsets[-1]) != u.shape[0]:
            raise ValueError(f"lengths sum to {int(offsets[-1])}, u has {u.shape[0]} rows")
        sizes = [n * n for n in lengths]
        buf = torch.empty((sum(sizes),), device=u.device, dtype=torch.float32)
        N.check(N.lib().ktf_plda_score_within(self.handle, T.ptr(u), T.host_ptr(offsets), len(lengths), T.ptr(buf),
                                              T.stream_ptr()))
        starts = np.concatenate(([0], np.cumsum(sizes)))
        return [buf[int(a):int(a) + n * n].view(n, n) for a, n in zip(starts[:-1], lengths)]

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
