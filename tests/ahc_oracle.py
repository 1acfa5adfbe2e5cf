"""
CPU oracle of the diarization back-end's clustering: Kaldi's single-pass AgglomerativeClusterer
(ivector/agglomerative-clustering.cc, the agglomerative-cluster binary) restated literally, with a heapq priority queue
and lazy deletion, in float32 NumPy arithmetic.  Test infrastructure: tests/test_diarization_oracle.py pins it against
scipy's average linkage and the properties of the contract; tests/test_gpu_diarization.py holds ktf_ahc_cluster to it
exactly.
"""

import numpy as np

F32 = np.float32


def agglomerative_cluster(scores, threshold=None, num_clusters=None):
    """Kaldi's AgglomerativeClusterer on one score matrix, restated literally:
    - cost(a, b) = -S[min(a, b)][max(a, b)] (only the upper triangle is read); points get ids 0 .. n-1 and every merge
      creates a cluster with the next id n, n+1, ...;
    - W(a, b), the cost sum of two active clusters, is the cost for two points; merging i and j into m gives every other
      active cluster k W(k, m) = W(k, i) + W(k, j) in float32, and avg(k, m) = W(k, m) / float32(size_k * size_m);
    - a priority queue (heapq, lazy deletion) holds (avg, lower id, higher id) of the pairs with avg <= threshold (NaN
      never; Python compares -0.0 and +0.0 as equal); each step pops the smallest entry whose clusters are both active
      and merges them, until the queue is empty or min_clusters clusters are left;
    - min_clusters is 1, or num_clusters, which also makes the threshold FLT_MAX (Kaldi's reco2num_spk).
    Returns (labels (n,) int32: the final clusters in increasing id order are 1 .. C, merges: list of (lo, hi, avg))."""
    import heapq

    S = np.asarray(scores, dtype=F32)
    n = S.shape[0]
    min_clusters = 1
    thr = F32(threshold) if threshold is not None else None
    if num_clusters is not None:
        min_clusters = int(num_clusters)
        thr = F32(np.finfo(np.float32).max)
    iu = np.triu_indices(n, 1)
    cost = np.zeros((n, n), dtype=F32)
    cost[iu] = -S[iu]
    cost = cost + cost.T                                   # (exact: one of the two terms is 0)
    W = cost                                               # by slot: slot s holds cluster ids[s]
    ids = np.arange(n, dtype=np.int64)
    size = np.ones(n, dtype=np.int64)
    alive = np.ones(n, dtype=bool)                         # by slot
    active = set(range(n))                                 # active cluster ids
    slot = {i: i for i in range(n)}
    members = {i: [i] for i in range(n)}
    keep = W[iu] <= thr                                    # (NaN compares false)
    heap = list(zip(W[iu][keep].tolist(), iu[0][keep].tolist(), iu[1][keep].tolist()))
    heapq.heapify(heap)
    merges = []
    next_id = n
    while len(active) > min_clusters and heap:
        avg, lo, hi = heapq.heappop(heap)
        if lo not in active or hi not in active:
            continue
        si, sj = slot.pop(lo), slot.pop(hi)
        active.discard(lo)
        active.discard(hi)
        alive[si] = alive[sj] = False
        m = next_id
        next_id += 1
        merges.append((lo, hi, avg))
        size_m = size[si] + size[sj]
        row = W[si] + W[sj]                                # float32 add, elementwise
        W[si, :] = row
        W[:, si] = row
        others = np.nonzero(alive)[0]
        avg_k = row[others] / (size[others] * size_m).astype(F32)
        ok = avg_k <= thr
        for a_k, id_k in zip(avg_k[ok].tolist(), ids[others[ok]].tolist()):
            heapq.heappush(heap, (a_k, id_k, m))           # (id_k < m)
        ids[si], size[si], alive[si] = m, size_m, True
        slot[m] = si
        members[m] = members.pop(lo) + members.pop(hi)
        active.add(m)
    labels = np.zeros(n, dtype=np.int32)
    for lab, c in enumerate(sorted(active), start=1):
        labels[members[c]] = lab
    return labels, merges
