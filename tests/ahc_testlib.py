"""
Helpers of the clustering tests at scale (test_diarization_ref.py, test_gpu_diarization_limits.py): the compiled
reference tests/ahc_ref.cc (Kaldi's AgglomerativeClusterer in C++, the contract of ahc_oracle.py) as a module fixture,
and the structured score matrices that stress the GPU clusterer.
"""

import ctypes
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import ROOT

F32_MAX = np.float32(np.finfo(np.float32).max)


class AhcRef:
    """ctypes binding of ahc_ref.cc.  The call releases the GIL, so `submit` runs several references in threads."""

    def __init__(self, path):
        self._lib = ctypes.CDLL(path)
        P = ctypes.c_void_p
        self._lib.ahc_ref.restype = ctypes.c_int
        self._lib.ahc_ref.argtypes = [P, ctypes.c_int, ctypes.c_float, ctypes.c_int, P, P, P]
        self._pool = ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1))

    def cluster(self, scores, threshold=None, num_clusters=None):
        """ahc_oracle.agglomerative_cluster's contract: exactly one of threshold and num_clusters.  Returns (labels (n,)
        int32, ids (k, 2) int32, costs (k,) float32) for the k merges."""
        assert (threshold is None) != (num_clusters is None)
        S = np.ascontiguousarray(scores, dtype=np.float32)
        n = S.shape[0]
        assert S.shape == (n, n)
        thr = F32_MAX if num_clusters is not None else np.float32(threshold)
        labels = np.zeros(n, dtype=np.int32)
        ids = np.zeros((max(n - 1, 0), 2), dtype=np.int32)
        costs = np.zeros(max(n - 1, 0), dtype=np.float32)
        P = ctypes.c_void_p
        k = self._lib.ahc_ref(P(S.ctypes.data), n, ctypes.c_float(thr), int(num_clusters or 1), P(labels.ctypes.data),
                              P(ids.ctypes.data), P(costs.ctypes.data))
        assert k >= 0, n
        return labels, ids[:k], costs[:k]

    def submit(self, scores, threshold=None, num_clusters=None):
        """`cluster` in a worker thread: a Future of its result."""
        return self._pool.submit(self.cluster, scores, threshold, num_clusters)

    def close(self):
        self._pool.shutdown(wait=True, cancel_futures=True)


@pytest.fixture(scope="module")
def ahc_ref(tmp_path_factory):
    """ahc_ref.cc compiled with the system C++ compiler (strict IEEE float32: no contraction, no fast-math)."""
    cxx = shutil.which(os.environ.get("CXX", "c++")) or shutil.which("g++") or shutil.which("clang++")
    if cxx is None:
        pytest.skip("no C++ compiler to build the clustering reference tests/ahc_ref.cc")
    out = str(tmp_path_factory.mktemp("ahc_ref") / "libahc_ref.so")
    cmd = [cxx, "-O2", "-ffp-contract=off", "-shared", "-fPIC", os.path.join(ROOT, "tests", "ahc_ref.cc"), "-o", out]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0, p.stdout
    ref = AhcRef(out)
    yield ref
    ref.close()


def oracle_arrays(result):
    """ahc_oracle.agglomerative_cluster's (labels, merges) as (labels, ids (k, 2) int32, costs (k,) float32)."""
    labels, merges = result
    ids = np.array([m[:2] for m in merges], dtype=np.int32).reshape(-1, 2)
    costs = np.array([m[2] for m in merges], dtype=np.float32)
    return labels, ids, costs


def bits(costs, signed_zero=True):
    """float32 bit patterns of `costs`; without `signed_zero` -0.0 is taken as +0.0."""
    c = np.asarray(costs, dtype=np.float32)
    if not signed_zero:
        c = np.where(c == 0, np.float32(0), c)
    return c.view(np.int32)


# Structured score matrices (float32, n x n).  Only the upper triangle matters; they are built symmetric.

def _sym(upper):
    return np.triu(upper, 1) + np.triu(upper, 1).T


def star(n, rng):
    """One hub every point prefers: after each merge the new cluster is almost every row's best partner, so nearly every
    row's cached partner was merged and is rescanned (more rows than the kernel's rescan list holds)."""
    S = _sym(rng.standard_normal((n, n)).astype(np.float32))
    if n:
        h = int(rng.integers(0, n))
        S[h, :] = S[:, h] = (10.0 + 0.01 * rng.standard_normal(n)).astype(np.float32)
    return S


def chain(n, rng, shuffled):
    """1-D points at random gaps, scores -distance: every merge extends a nearest-neighbour chain.  In point order, or
    shuffled."""
    x = np.cumsum(rng.random(n) + 0.01)
    if shuffled:
        x = x[rng.permutation(n)]
    return (-np.abs(x[:, None] - x[None, :])).astype(np.float32)


def blocks(n, rng, inside=None):
    """Block-diagonal: random block sizes up to 63, -1 outside.  Inside, `inside(rng, (b, b))`, by default one value per
    block from {1, 2, 3}: ties inside and across blocks, and every cost sum an exact integer."""
    S = np.full((n, n), -1.0, dtype=np.float32)
    at = 0
    while at < n:
        b = int(rng.integers(1, 64))
        S[at:at + b, at:at + b] = inside(rng, S[at:at + b, at:at + b].shape) if inside else float(rng.integers(1, 4))
        at += b
    return S


def signed_zeros(rng, shape):
    """Only +0.0 and -0.0: every avg between them is a zero of either sign, and the ids decide the order."""
    return np.where(rng.random(shape) < 0.5, np.float32(0.0), np.float32(-0.0)).astype(np.float32)


def structured(n, seed):
    """(name, scores, clustering arguments) of the structured cases, at any size up to KTF_AHC_MAX_POINTS: a star, chains,
    tied blocks, all NaN (no merge), all -inf with num_clusters (cost +inf is above FLT_MAX: no merge), blocks of +inf
    (costs and sums -inf, merged by ids) and blocks of +-0."""
    rng = np.random.default_rng(seed)
    return [("star", star(n, rng), {"num_clusters": 1}),
            ("chain", chain(n, rng, False), {"num_clusters": 1}),
            ("chain_shuffled", chain(n, rng, True), {"num_clusters": 1}),
            ("blocks", blocks(n, rng), {"threshold": -0.5}),
            ("nan", np.full((n, n), np.nan, dtype=np.float32), {"threshold": np.inf}),
            ("neg_inf", np.full((n, n), -np.inf, dtype=np.float32), {"num_clusters": 1}),
            ("inf_blocks", blocks(n, rng, lambda r, shape: np.inf), {"num_clusters": 1}),
            ("zero_blocks", blocks(n, rng, signed_zeros), {"threshold": 0.0})]


def dense_ties(n, seed):
    """(name, scores, clustering arguments) of the cases where every pair ties at every step: all equal, all +inf (costs
    -inf) and all +-0.  The ids alone decide, so every merge replaces the lowest active id, every row's best partner, and
    the GPU kernel rescans every row: O(n^3) work for one CTA, so these are tested up to a few thousand points."""
    rng = np.random.default_rng(seed)
    return [("equal", np.full((n, n), -1.0, dtype=np.float32), {"num_clusters": 1}),
            ("pos_inf", np.full((n, n), np.inf, dtype=np.float32), {"num_clusters": 1}),
            ("zeros", signed_zeros(rng, (n, n)), {"threshold": 0.0})]
