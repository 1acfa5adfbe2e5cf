"""
The diarization back-end at its limits, held exactly to the compiled reference (tests/ahc_ref.cc, pinned to the oracle
by test_diarization_ref.py):
- clustering at KTF_AHC_MAX_POINTS (cluster ids up to 32 766), at 8 193 points (the first size whose ids need the 15th
  bit of the merge key) and a last merge whose size product float32 cannot hold exactly;
- structures that stress the kernel's row caches: a hub every point prefers (its merges overflow the rescan list),
  chains, tied blocks, NaN / +-inf / +-0 scores, and scores where every pair ties;
- batches whose packed scores, W scratch and withinScores output pass 2^31 elements;
- the C entry points' optional outputs, offsets_host[0] > 0 and every output's end (sentinel tails);
- withinScores groups of 16 384 rows, clustered in place, and the list forms agglomerative_cluster copies.
Every comparison is exact: labels, merge ids, merge costs as float32 bits (the kernel reports a zero cost as +0.0),
the (-1, -1, NaN) padding and cluster_counts_dev.  The references run in threads, started when the module starts.
"""

import ctypes

import numpy as np
import pytest

from ahc_testlib import ahc_ref, bits, blocks, dense_ties, structured  # noqa: F401  (ahc_ref: fixture)
from plda_testlib import ktf, plda_vectors  # noqa: F401  (ktf: fixture)
from test_gpu_diarization import _scores

pytestmark = pytest.mark.gpu

LIMIT = 16384                  # KTF_AHC_MAX_POINTS
ABOVE = 8200                   # a size whose cluster ids need the 15th bit
SMALL = [0, 1, 2, 33, 600]     # groups interleaved with the large ones
SENTINEL = 0x5A5A5A5A
TAIL = 256                     # sentinel elements after every output
P = ctypes.c_void_p


def _two_groups(a, b, rng):
    """Two groups of a and b points in a shuffled order, close inside and far apart: the last merge joins them, and
    a * b (odd, above 2^24) is the first size product float32 cannot hold exactly."""
    side = rng.permutation(np.arange(a + b) < a)
    S = rng.standard_normal((a + b, a + b)).astype(np.float32)
    return S + np.where(side[:, None] == side[None, :], np.float32(5), np.float32(-5))


def _limit_cases():
    """name -> (scores, clustering arguments) of the cases whose references are computed once per module."""
    rng = np.random.default_rng(101)
    cases = {
        "normal": (rng.standard_normal((LIMIT, LIMIT)).astype(np.float32), {"num_clusters": 1}),
        # tied blocks: ids up to 32 766 decide every tie (all scores equal would do so too, but makes every merge
        # rescan every row: see ahc_testlib.dense_ties)
        "blocks": (blocks(LIMIT, rng), {"num_clusters": 1}),
        "integer_8193": (_scores("integer", 8193, rng), {"threshold": 0.5}),
        "two_groups": (_two_groups(5001, 4099, rng), {"num_clusters": 1}),
    }
    for name, S, kw in structured(ABOVE, seed=102):
        cases["above_" + name] = (S, kw)
    return cases


@pytest.fixture(scope="module")
def within_limit(ktf):
    """One withinScores group of LIMIT rows: (layer, u, scores)."""
    layer, (u,), _, _ = plda_vectors(ktf, [LIMIT], seed=103, cuda_rng=True)
    (S,) = layer.withinScores(u, [LIMIT])
    return layer, u, S


@pytest.fixture(scope="module")
def refs(ahc_ref, within_limit):
    """name -> (scores, clustering arguments, Future of the reference result), the largest submitted first."""
    out = {"within": (within_limit[2].cpu().numpy(), {"num_clusters": 1})}
    out.update(_limit_cases())
    return {name: (S, kw, ahc_ref.submit(S, **kw)) for name, (S, kw) in out.items()}


def _sentinel_buffer(n):
    import torch
    return torch.full((n + TAIL,), SENTINEL, device="cuda", dtype=torch.int32)


def _tail_intact(buf, n):
    import torch
    return bool(torch.all(buf[n:] == SENTINEL))


def run_ahc(ktf, scores, offsets, *, threshold=None, num_clusters=None, ids=True, costs=True):
    """ktf_ahc_cluster through the C ABI on the packed score matrices from scores.data_ptr(), every output followed by a
    sentinel tail that must be intact afterwards.  num_clusters: one int for every group, or None.  Returns
    (counts (g,), [(labels, ids (n - 1, 2) or None, costs (n - 1,) or None)] per group) as numpy arrays."""
    import torch
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    sizes = np.diff(offsets)
    g, points = len(sizes), int(offsets[-1] - offsets[0])
    m_offs = np.concatenate(([0], np.cumsum(np.maximum(sizes - 1, 0))))
    lab, cnt = _sentinel_buffer(points), _sentinel_buffer(g)
    mid = _sentinel_buffer(2 * int(m_offs[-1])) if ids else None
    mc = _sentinel_buffer(int(m_offs[-1])) if costs else None
    nc = np.full(g, num_clusters, dtype=np.int32) if num_clusters is not None else None
    lib = ktf._native.lib()
    rc = lib.ktf_ahc_cluster(P(scores.data_ptr()), P(offsets.ctypes.data), g,
                             threshold if threshold is not None else 0.0, P(nc.ctypes.data) if nc is not None else P(0),
                             P(lab.data_ptr()), P(mid.data_ptr()) if ids else P(0), P(mc.data_ptr()) if costs else P(0),
                             P(cnt.data_ptr()), P(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, ktf._native.last_error()
    torch.cuda.synchronize()
    assert _tail_intact(lab, points) and _tail_intact(cnt, g)
    assert mid is None or _tail_intact(mid, 2 * int(m_offs[-1]))
    assert mc is None or _tail_intact(mc, int(m_offs[-1]))
    lab, cnt = lab[:points].cpu().numpy(), cnt[:g].cpu().numpy()
    mid = mid[:2 * int(m_offs[-1])].cpu().numpy().reshape(-1, 2) if ids else None
    mc = mc[:int(m_offs[-1])].view(torch.float32).cpu().numpy() if costs else None
    out = []
    for r in range(g):
        a, b = int(offsets[r] - offsets[0]), int(offsets[r + 1] - offsets[0])
        m0, m1 = int(m_offs[r]), int(m_offs[r + 1])
        out.append((lab[a:b], mid[m0:m1] if ids else None, mc[m0:m1] if costs else None))
    return cnt, out


def assert_matches(got, count, want, what):
    """One group's GPU result (labels, ids or None, costs or None) and cluster count equal the reference's, padding
    included."""
    labels, ids, costs = got
    wl, wi, wc = want
    n, k = len(wl), len(wc)
    assert np.array_equal(labels, wl), what
    assert count == n - k, what
    if ids is not None:
        assert ids.shape == (max(n - 1, 0), 2), what
        assert np.array_equal(ids[:k], wi), what
        assert (ids[k:] == -1).all(), what
    if costs is not None:
        assert costs.shape == (max(n - 1, 0),), what
        assert np.array_equal(bits(costs[:k], signed_zero=False), bits(wc, signed_zero=False)), what
        assert np.isnan(costs[k:]).all(), what


def _cluster_kwargs(kw):
    return {"threshold": kw.get("threshold"), "num_clusters": kw.get("num_clusters")}


def _packed(mats):
    import torch
    return torch.cat([torch.from_numpy(np.ascontiguousarray(S)).reshape(-1) for S in mats]).cuda()


@pytest.mark.parametrize("name", ["normal", "blocks", "integer_8193", "two_groups"])
def test_ahc_at_the_limit(ktf, refs, name):
    S, kw, want = refs[name]
    counts, (got,) = run_ahc(ktf, _packed([S]), [0, S.shape[0]], **_cluster_kwargs(kw))
    assert_matches(got, counts[0], want.result(), name)


STRUCTURED = ["star", "chain", "chain_shuffled", "blocks", "nan", "neg_inf", "inf_blocks", "zero_blocks"]


@pytest.mark.parametrize("name", STRUCTURED + ["equal", "pos_inf", "zeros"])
def test_ahc_structured(ktf, ahc_ref, refs, name):
    # at 33 and 3000 points in one batch, then (all but the dense ties) above 8192
    small = [dict((c[0], c) for c in structured(n, seed=n) + dense_ties(n, seed=n))[name] for n in (33, 3000)]
    kw = small[0][2]
    futures = [ahc_ref.submit(S, **kw) for _, S, _ in small]
    counts, got = run_ahc(ktf, _packed([S for _, S, _ in small]), [0, 33, 3033], **_cluster_kwargs(kw))
    for r, f in enumerate(futures):
        assert_matches(got[r], counts[r], f.result(), (name, small[r][1].shape[0]))
    if name in STRUCTURED:
        S, kw, want = refs["above_" + name]
        counts, (got,) = run_ahc(ktf, _packed([S]), [0, ABOVE], **_cluster_kwargs(kw))
        assert_matches(got, counts[0], want.result(), (name, ABOVE))


def _need_free_gb(gb):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < gb * 2 ** 30:
        pytest.skip(f"needs about {gb} GB of free device memory, {free / 2 ** 30:.1f} GB free")


def _interleaved(large, copies, seed):
    """Group sizes: `copies` groups of `large` and the SMALL groups, in a shuffled order (so large groups sit at
    offsets past 2^31 elements)."""
    sizes = [large] * copies + SMALL
    return [int(n) for n in np.random.default_rng(seed).permutation(sizes)]


def test_ahc_batch_past_2_31_elements(ktf, ahc_ref, refs):
    import torch
    _need_free_gb(24)
    S, kw, want = refs["normal"]
    rng = np.random.default_rng(104)
    small = {n: _scores("normal", n, rng) for n in SMALL}
    small_want = {n: ahc_ref.submit(small[n], num_clusters=1) for n in SMALL}
    sizes = _interleaved(LIMIT, 9, seed=105)
    total = sum(n * n for n in sizes)
    assert total > 2 ** 31
    buf = torch.empty(total, device="cuda", dtype=torch.float32)
    big = torch.from_numpy(S).cuda().reshape(-1)
    at = 0
    for n in sizes:
        buf[at:at + n * n] = big if n == LIMIT else torch.from_numpy(small[n]).cuda().reshape(-1)
        at += n * n
    del big
    offsets = np.concatenate(([0], np.cumsum(sizes)))
    counts, got = run_ahc(ktf, buf, offsets, num_clusters=1)
    del buf
    torch.cuda.empty_cache()
    for r, n in enumerate(sizes):
        assert_matches(got[r], counts[r], want.result() if n == LIMIT else small_want[n].result(), (r, n))


def test_ahc_c_abi_edges(ktf, ahc_ref):
    rng = np.random.default_rng(106)
    sizes = [5, 0, 300, 1, 64, 2]
    mats = [_scores("integer", n, rng) for n in sizes]
    scores = _packed(mats)
    offsets = np.concatenate(([0], np.cumsum(sizes)))
    for kw in ({"threshold": 0.5}, {"num_clusters": 2}):
        want = [ahc_ref.cluster(S, **kw) for S in mats]
        counts, full = run_ahc(ktf, scores, offsets, **_cluster_kwargs(kw))
        for r in range(len(sizes)):
            assert_matches(full[r], counts[r], want[r], (kw, r))
        # offsets_host[0] > 0: the scores still start at scores_dev, labels go to offsets[r] - offsets[0]
        c, got = run_ahc(ktf, scores, offsets + 1000, **_cluster_kwargs(kw))
        assert np.array_equal(c, counts)
        for r in range(len(sizes)):
            assert_matches(got[r], c[r], want[r], (kw, r, "offset"))
        # the merge outputs are optional, each on its own
        for ids, costs in ((True, False), (False, True), (False, False)):
            c, got = run_ahc(ktf, scores, offsets, ids=ids, costs=costs, **_cluster_kwargs(kw))
            assert np.array_equal(c, counts)
            for r in range(len(sizes)):
                assert_matches(got[r], c[r], want[r], (kw, r, ids, costs))


def _within_call(ktf, layer, u, offsets, out):
    import torch
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    rc = ktf._native.lib().ktf_plda_score_within(layer.handle, P(u.data_ptr()), P(offsets.ctypes.data),
                                                 len(offsets) - 1, P(out.data_ptr()),
                                                 P(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, ktf._native.last_error()


def _within_vs_llr(layer, u, sizes, packed):
    """Every group of the packed within scores is bit-equal to the transposed logLikelihoodRatio of its rows (one
    group's reference live at a time)."""
    import torch
    at = row = 0
    for n in sizes:
        if n:
            want = layer.logLikelihoodRatio(u[row:row + n].contiguous()).t()
            assert torch.equal(packed[at:at + n * n].view(n, n), want), (row, n)
            del want
        at += n * n
        row += n


def test_within_scores_one_group_at_the_limit(within_limit):
    layer, u, S = within_limit
    _within_vs_llr(layer, u, [LIMIT], S.reshape(-1))


def test_within_scores_batch_past_2_31_elements(ktf):
    import torch
    _need_free_gb(14)
    sizes = _interleaved(LIMIT, 9, seed=107)
    layer, (u,), _, _ = plda_vectors(ktf, [sum(sizes)], seed=108, cuda_rng=True)
    total = sum(n * n for n in sizes)
    assert total > 2 ** 31
    buf = _sentinel_buffer(total).view(torch.float32)
    _within_call(ktf, layer, u, np.concatenate(([0], np.cumsum(sizes))), buf)
    torch.cuda.synchronize()
    assert _tail_intact(buf.view(torch.int32), total)
    _within_vs_llr(layer, u, sizes, buf)
    del buf
    torch.cuda.empty_cache()


def test_within_scores_offset_rows(ktf):
    import torch
    sizes, skip = [5, 300, 0, 257, 1], 37
    layer, (u,), _, _ = plda_vectors(ktf, [skip + sum(sizes)], seed=109)
    total = sum(n * n for n in sizes)
    buf = _sentinel_buffer(total).view(torch.float32)
    _within_call(ktf, layer, u, skip + np.concatenate(([0], np.cumsum(sizes))), buf)
    torch.cuda.synchronize()
    assert _tail_intact(buf.view(torch.int32), total)
    want = torch.cat([m.reshape(-1) for m in layer.withinScores(u[skip:].contiguous(), sizes)])
    assert torch.equal(buf[:total], want)


def test_within_then_cluster_in_place_at_the_limit(ktf, refs, within_limit):
    _, _, S = within_limit
    _, kw, want = refs["within"]
    labels, merges = ktf.diarization.agglomerative_cluster([S], num_speakers=kw["num_clusters"], return_merges=True)
    ids, costs = merges[0]
    got = (labels[0].cpu().numpy(), ids.cpu().numpy(), costs.cpu().numpy())
    assert_matches(got, got[0].max(), want.result(), "within")


def test_list_forms_match_the_packed_list(ktf, ahc_ref):
    import torch
    sizes = [300, 0, 1, 1000, 64]
    layer, (u,), _, _ = plda_vectors(ktf, [sum(sizes)], seed=110)
    mats = layer.withinScores(u, sizes)
    assert ktf.diarization._packed_base(mats, sizes) is not None
    for kw in ({"threshold": 0.0}, {"num_speakers": 2}):
        ref_kw = {"threshold": 0.0} if "threshold" in kw else {"num_clusters": 2}
        want = [ahc_ref.cluster(m.cpu().numpy(), **ref_kw) for m in mats]

        def check(lst, expect, what):
            labels, merges = ktf.diarization.agglomerative_cluster(lst, return_merges=True, **kw)
            assert len(labels) == len(expect), what
            for r, (lab, (ids, costs), w) in enumerate(zip(labels, merges, expect)):
                got = (lab.cpu().numpy(), ids.cpu().numpy(), costs.cpu().numpy())
                assert_matches(got, got[0].max() if len(got[0]) else 0, w, (what, kw, r))

        check(mats, want, "packed")
        check(mats[::-1], want[::-1], "reversed")
        check(mats[1:4], want[1:4], "sub-list")
        check([mats[3], mats[3]], [want[3], want[3]], "twice")
        wide = torch.full((1000, 1003), float("nan"), device="cuda")
        wide[:, :1000] = mats[3]
        view = wide[:, :1000]
        assert not view.is_contiguous()
        check([mats[0], view], [want[0], want[3]], "non-contiguous")
