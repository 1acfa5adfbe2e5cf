"""
The compiled clustering reference (tests/ahc_ref.cc) against the pinned oracle (tests/ahc_oracle.py): the same merge
lists, ids and float32 cost bits, and the same labels, on random, tie-heavy, NaN / +-inf and structured scores at every
kind of threshold.  The GPU tests at KTF_AHC_MAX_POINTS (test_gpu_diarization_limits.py) rest on this.  CPU only.
"""

import numpy as np
import pytest

import ahc_oracle as O
from ahc_testlib import ahc_ref, bits, dense_ties, oracle_arrays, structured  # noqa: F401  (ahc_ref: fixture)
from test_gpu_diarization import _scores

THRESHOLDS = (-np.inf, -0.5, -0.0, 0.0, 0.7, np.inf, np.nan)


def _assert_same(got, want, what):
    # the oracle builds its symmetric costs as -S + 0 (a score of 0.0 becomes the cost +0.0), Kaldi and the reference
    # as -S (-0.0): the sign of a zero cost is the only difference, and the contract takes -0 and +0 as equal
    gl, gi, gc = got
    wl, wi, wc = want
    assert gi.shape == wi.shape and np.array_equal(gi, wi), what
    assert np.array_equal(bits(gc, signed_zero=False), bits(wc, signed_zero=False)), what
    assert np.array_equal(gl, wl), what


def _check(ahc_ref, S, what, **kw):
    _assert_same(ahc_ref.cluster(S, **kw), oracle_arrays(O.agglomerative_cluster(S, **kw)), (what, kw))


@pytest.mark.parametrize("kind", ["normal", "integer", "special"])
def test_reference_matches_oracle(ahc_ref, kind):
    rng = np.random.default_rng({"normal": 11, "integer": 12, "special": 13}[kind])
    for n in (0, 1, 2, 3, 5, 17, 64, 150, 300):
        S = _scores(kind, n, rng)
        for t in THRESHOLDS:
            _check(ahc_ref, S, (kind, n), threshold=t)
        for c in (1, 3, n, n + 5):
            _check(ahc_ref, S, (kind, n), num_clusters=max(c, 1))


@pytest.mark.parametrize("n", [2, 40, 257])
def test_reference_matches_oracle_structured(ahc_ref, n):
    for name, S, kw in structured(n, seed=n) + dense_ties(n, seed=n):
        _check(ahc_ref, S, (name, n), **kw)
        _check(ahc_ref, S, (name, n), threshold=0.0)


def test_reference_reads_only_the_upper_triangle(ahc_ref):
    S = np.random.default_rng(14).standard_normal((60, 60)).astype(np.float32)
    bad = S.copy()
    bad[np.tril_indices(60)] = np.nan
    for kw in ({"threshold": 0.0}, {"num_clusters": 1}):
        _assert_same(ahc_ref.cluster(bad, **kw), ahc_ref.cluster(S, **kw), kw)


def test_reference_ties_and_signed_zeros(ahc_ref):
    # every pair ties: the ids alone decide, and the last merges join the clusters with the highest ids
    labels, ids, costs = ahc_ref.cluster(np.full((4, 4), -1.0, dtype=np.float32), num_clusters=1)
    assert ids.tolist() == [[0, 1], [2, 3], [4, 5]] and costs.tolist() == [1.0, 1.0, 1.0]
    assert labels.tolist() == [1, 1, 1, 1]
    # -0.0 and +0.0 are one cost: (0, 1) goes first though its cost is +0.0 and (0, 2)'s is -0.0
    S = np.zeros((3, 3), dtype=np.float32)
    S[0, 1], S[0, 2] = -0.0, 0.0
    _, ids, costs = ahc_ref.cluster(S, num_clusters=1)
    assert ids[0].tolist() == [0, 1] and bits(costs)[0] == bits([0.0])[0]
    # labels follow the final clusters' ids
    S = np.full((4, 4), -10.0, dtype=np.float32)
    S[2, 3], S[0, 1] = 5.0, 4.0
    labels, ids, _ = ahc_ref.cluster(S, threshold=0.0)
    assert ids.tolist() == [[2, 3], [0, 1]] and labels.tolist() == [2, 2, 1, 1]


def test_reference_threads_agree(ahc_ref):
    rng = np.random.default_rng(15)
    mats = [_scores("integer", 200, rng) for _ in range(6)]
    futures = [ahc_ref.submit(S, threshold=0.5) for S in mats]
    for S, f in zip(mats, futures):
        _assert_same(f.result(), ahc_ref.cluster(S, threshold=0.5), "threads")
