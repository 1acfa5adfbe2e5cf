"""
Diarization back-end: Kaldi's agglomerative-cluster (average-linkage AHC, single pass) for a batch of recordings on the
GPU, on the within-recording PLDA scores of `layers.PLDA.withinScores`.

    scores = plda.withinScores(u, lengths)                      # one (n_r, n_r) matrix per recording
    labels = agglomerative_cluster(scores, threshold=0.0)       # Kaldi cost units: cost = -score
    labels = agglomerative_cluster(scores, num_speakers=[2, 3, ...])
"""

import ctypes

import numpy as np
import torch

from . import _native as N
from . import _tensor as T


def _packed_base(scores, sizes):
    """The address of a packed buffer that `scores` are consecutive views of (the `withinScores` layout), or None."""
    base = None
    at = 0
    for s, n in zip(scores, sizes):
        if n > 0:
            if not s.is_contiguous():
                return None
            b = s.data_ptr() - 4 * at
            if base is None:
                base, storage = b, s.untyped_storage().data_ptr()
                if b < storage:
                    return None
            elif b != base or s.untyped_storage().data_ptr() != storage:
                return None
        at += n * n
    return base


def agglomerative_cluster(scores, *, threshold=None, num_speakers=None, return_merges=False):
    """Average-linkage clustering of every recording's square float32 CUDA score matrix in `scores`, exactly Kaldi's
    AgglomerativeClusterer: the cost of two segments is -S[min][max] (the upper triangle), a cluster pair's cost is the
    float32 sum of its segment costs over the product of the sizes, and each step merges the cheapest pair (ties: the
    lower cluster ids) while its cost is <= `threshold`.  With `num_speakers` (an int, or one per recording) the
    threshold is FLT_MAX and clustering stops at that many clusters -- Kaldi's reco2num_spk.  Pass exactly one of the
    two.

    Returns a list of (n_r,) int32 label views (labels 1 .. C_r, in the order of the clusters' ids), and with
    `return_merges` also a list of (ids (max(n_r - 1, 0), 2) int32, costs (max(n_r - 1, 0),) float32) merge lists: the
    merges in order as (lower id, higher id, cost), point ids 0 .. n_r - 1 and the k-th merge's cluster n_r + k, then
    (-1, -1, NaN).  A thresholded run's merges are the prefix of the num_speakers=1 run's merges up to the first cost
    above the threshold, so one run serves a threshold sweep.  Outputs of `withinScores` are read in place; any other
    list is packed once.  At most KTF_AHC_MAX_POINTS (16384) segments per recording."""
    if (threshold is None) == (num_speakers is None):
        raise ValueError("pass exactly one of threshold and num_speakers")
    scores = list(scores)
    sizes = []
    for s in scores:
        if not isinstance(s, torch.Tensor) or not s.is_cuda or s.dtype != torch.float32 or s.dim() != 2 \
                or s.shape[0] != s.shape[1]:
            raise ValueError("scores must be square float32 CUDA tensors")
        sizes.append(int(s.shape[0]))
    g = len(sizes)
    offsets = np.concatenate(([0], np.cumsum(sizes, dtype=np.int64))).astype(np.int64)
    num_clusters = None
    if num_speakers is not None:
        per = [num_speakers] * g if np.isscalar(num_speakers) else list(num_speakers)
        if len(per) != g:
            raise ValueError(f"num_speakers has {len(per)} entries for {g} recordings")
        num_clusters = np.ascontiguousarray(per, dtype=np.int32)
    dev = scores[0].device if scores else torch.device("cuda")
    base = _packed_base(scores, sizes)
    packed = None
    if base is None and sum(sizes) > 0:
        packed = torch.cat([s.reshape(-1) for s in scores])
        base = packed.data_ptr()
    total = int(offsets[-1])
    n_merges = [max(n - 1, 0) for n in sizes]
    labels = torch.empty((total,), device=dev, dtype=torch.int32)
    merge_ids = torch.empty((sum(n_merges), 2), device=dev, dtype=torch.int32) if return_merges else None
    merge_costs = torch.empty((sum(n_merges),), device=dev, dtype=torch.float32) if return_merges else None
    counts = torch.empty((g,), device=dev, dtype=torch.int32)
    N.check(N.lib().ktf_ahc_cluster(ctypes.c_void_p(base or 0), T.host_ptr(offsets), g,
                                    float(threshold) if threshold is not None else 0.0, T.host_ptr(num_clusters),
                                    T.ptr(labels), T.ptr(merge_ids), T.ptr(merge_costs), T.ptr(counts),
                                    T.stream_ptr()))
    out = [labels[int(a):int(b)] for a, b in zip(offsets[:-1], offsets[1:])]
    if not return_merges:
        return out
    m_offs = np.concatenate(([0], np.cumsum(n_merges)))
    merges = [(merge_ids[int(a):int(b)], merge_costs[int(a):int(b)]) for a, b in zip(m_offs[:-1], m_offs[1:])]
    return out, merges
