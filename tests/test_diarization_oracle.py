"""
The AHC oracle (tests/ahc_oracle.py, Kaldi's AgglomerativeClusterer restated) against scipy's average linkage, and
the properties the GPU clustering is held to: threshold runs are prefixes of the full run, ties go to the lower ids,
the lower triangle is never read.  CPU only.
"""

import numpy as np
import pytest

import ahc_oracle as O


def _points_scores(n, seed, dim=3):
    """Scores -distance of random points: costs are Euclidean distances, with no ties."""
    x = np.random.default_rng(seed).standard_normal((n, dim))
    d = np.sqrt(((x[:, None, :] - x[None, :, :]) ** 2).sum(-1))
    return (-d).astype(np.float32)


def _partition(labels):
    groups = {}
    for i, lab in enumerate(labels):
        groups.setdefault(int(lab), []).append(i)
    return sorted(tuple(g) for g in groups.values())


@pytest.mark.parametrize("n,seed", [(2, 0), (7, 1), (60, 2), (300, 3)])
def test_oracle_matches_scipy_average_linkage(n, seed):
    from scipy.cluster.hierarchy import fcluster, linkage
    from scipy.spatial.distance import squareform
    S = _points_scores(n, seed)
    cost = -S.astype(np.float64)
    np.fill_diagonal(cost, 0.0)
    Z = linkage(squareform(cost, checks=False), method="average")
    _, merges = O.agglomerative_cluster(S, num_clusters=1)
    heights = np.array([m[2] for m in merges])
    assert len(merges) == n - 1
    np.testing.assert_allclose(np.sort(heights), np.sort(Z[:, 2]), rtol=1e-4)
    for q in (0.1, 0.3, 0.5, 0.8):
        t = float(np.quantile(Z[:, 2], q))
        if np.min(np.abs(Z[:, 2] - t)) <= 1e-4 * abs(t):
            continue
        labels, _ = O.agglomerative_cluster(S, threshold=t)
        assert _partition(labels) == _partition(fcluster(Z, t, criterion="distance")), (n, q)


@pytest.mark.parametrize("integer", [False, True])
def test_oracle_threshold_runs_are_prefixes(integer):
    rng = np.random.default_rng(5)
    n = 80
    S = rng.integers(-4, 5, size=(n, n)).astype(np.float32) if integer else rng.standard_normal((n, n)).astype(np.float32)
    _, full = O.agglomerative_cluster(S, num_clusters=1)
    for t in (-10.0, -2.0, -0.5, 0.0, 0.5, 3.0, 1e30):
        labels, part = O.agglomerative_cluster(S, threshold=t)
        stop = next((i for i, m in enumerate(full) if m[2] > t), len(full))
        assert part == full[:stop], t
        assert labels.max() == n - len(part)


def test_oracle_ties_go_to_lower_ids():
    S = np.full((4, 4), -1.0, dtype=np.float32)
    labels, merges = O.agglomerative_cluster(S, num_clusters=1)
    assert merges == [(0, 1, 1.0), (2, 3, 1.0), (4, 5, 1.0)]
    assert labels.tolist() == [1, 1, 1, 1]
    # -0.0 and +0.0 are the same cost: the ids decide
    S = np.zeros((3, 3), dtype=np.float32)
    S[0, 2] = -0.0
    S[0, 1] = 0.0
    _, merges = O.agglomerative_cluster(S, num_clusters=1)
    assert merges[0][:2] == (0, 1)


def test_oracle_ignores_the_lower_triangle():
    S = np.random.default_rng(8).standard_normal((40, 40)).astype(np.float32)
    bad = S.copy()
    bad[np.tril_indices(40)] = np.nan
    for kw in ({"threshold": 0.0}, {"num_clusters": 3}, {"num_clusters": 1}):
        a, ma = O.agglomerative_cluster(S, **kw)
        b, mb = O.agglomerative_cluster(bad, **kw)
        assert np.array_equal(a, b) and ma == mb


def test_oracle_labels_follow_cluster_ids():
    # two clear groups: the group whose final cluster has the lower id gets label 1
    S = np.full((4, 4), -10.0, dtype=np.float32)
    S[2, 3] = 5.0          # 2 + 3 merge first (id 4)
    S[0, 1] = 4.0          # then 0 + 1 (id 5)
    labels, merges = O.agglomerative_cluster(S, threshold=0.0)
    assert merges == [(2, 3, -5.0), (0, 1, -4.0)]
    assert labels.tolist() == [2, 2, 1, 1]
