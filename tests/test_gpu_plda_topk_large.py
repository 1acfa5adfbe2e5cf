"""
PLDA.bestMatchesLarge / asNormBestMatchesLarge / ktf_plda_score_topk_large / ktf_plda_score_asnorm_topk_large /
ktf_topk_merge_large: the k best enrolled vectors of every test vector for 1 <= k <= 1024, without the score matrix.
The contract: row i equals the first k entries of a stable descending sort of row i of the float32
`logLikelihoodRatio` / `asNorm` matrix, bit for bit, with NaN and -inf entries left out and the row padded with
(-inf, -1).  k <= 32 runs the top-k epilogue of bestMatches; larger k scores row chunks into the workspace and selects
each one (radix select, ordered emit, bitonic sort).

The argument checks that need no device run everywhere; the rest is marked gpu.
"""

import ctypes

import numpy as np
import pytest

from oracle import ktf_oracle as O
from plda_testlib import DIM, check_equal, expected_listed, ktf, listed_sort, plda_vectors  # noqa: F401
from plda_testlib import run_two_ranks, stats
from test_gpu_tdnn_plda import synthetic_plda

gpu = pytest.mark.gpu

KS = (33, 64, 100, 255, 256, 257, 1000, 1024)
N_TEST, N_ENROLL, N_COHORT = 1037, 49153, 1500


# ---- argument checks (no device) ----

def test_c_entry_points_reject_bad_arguments():
    from kaldi_tflite_b200 import _native as N
    lib = N.lib()
    p = ctypes.c_void_p(0)
    assert N.KTF_PLDA_TOPK_LARGE_MAX == 1024
    for k in (0, 1025, -1):
        rc = lib.ktf_plda_score_topk_large(None, p, 10, p, 10, k, p, p, None)
        assert rc == N.KTF_EINVAL and "KTF_PLDA_TOPK_LARGE_MAX" in N.last_error()
        rc = lib.ktf_plda_score_asnorm_topk_large(None, p, 10, p, 10, p, p, p, p, k, p, p, None)
        assert rc == N.KTF_EINVAL and "KTF_PLDA_TOPK_LARGE_MAX" in N.last_error()
        rc = lib.ktf_topk_merge_large(p, p, 2, 10, 5, k, p, p, None)
        assert rc == N.KTF_EINVAL and "KTF_PLDA_TOPK_LARGE_MAX" in N.last_error()
    for k in (33, 1024):
        assert lib.ktf_plda_score_topk_large(None, p, 10, p, 10, k, p, p, None) == N.KTF_EINVAL
        assert "null handle" in N.last_error()
        assert lib.ktf_plda_score_asnorm_topk_large(None, p, 10, p, 10, p, p, p, p, k, p, p, None) == N.KTF_EINVAL
        assert "null handle" in N.last_error()
    assert lib.ktf_topk_merge_large(p, p, 2, 10, 0, 5, p, p, None) == N.KTF_EINVAL
    assert lib.ktf_topk_merge_large(p, p, 1 << 16, 10, 1 << 15, 5, p, p, None) == N.KTF_EINVAL
    assert lib.ktf_topk_merge_large(None, None, 2, 0, 5, 5, None, None, None) == 0       # no rows: a no-op


def test_python_argument_validation():
    import torch
    import kaldi_tflite_b200 as ktf
    mean, Tm, psi = synthetic_plda(DIM)
    l32 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32)
    l64 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float64)
    ut, ue = torch.zeros((6, DIM)), torch.zeros((5, DIM))
    ts, es = (torch.zeros(6), torch.ones(6)), (torch.zeros(5), torch.ones(5))
    with pytest.raises(ValueError, match="float32"):
        l64.bestMatchesLarge(ut.double(), ue.double(), k=100)
    with pytest.raises(ValueError, match="float32"):
        l64.asNormBestMatchesLarge(ut.double(), ue.double(), k=100, test_stats=ts, enroll_stats=es)
    for k in (0, 1025):
        with pytest.raises(ValueError, match="1024"):
            l32.bestMatchesLarge(ut, ue, k=k)
        with pytest.raises(ValueError, match="1024"):
            l32.asNormBestMatchesLarge(ut, ue, k=k, test_stats=ts, enroll_stats=es)
    with pytest.raises(ValueError, match="u_cohort and top_n"):
        l32.asNormBestMatchesLarge(ut, ue, k=100, test_stats=ts)


# ---- on the GPU ----

@pytest.fixture(scope="module")
def setup(ktf):
    """A float32 layer and transformed vectors: 1037 test, 49 153 enrolled (one past the shared-memory row limit), a
    1500-vector cohort."""
    layer, (ut, ue, uc), _, _ = plda_vectors(ktf, (N_TEST, N_ENROLL, N_COHORT), 2026, cuda_rng=True)
    return layer, ut, ue, uc


def both_forms(layer, ut, ue, uc, num_examples=1.0, top_n=100):
    """(name, full matrix, k -> (scores, indexes)) of the raw and the AS-norm form on the same vectors."""
    ts, es = stats(layer, ut, ue, uc, top_n, num_examples)
    yield ("raw", layer.logLikelihoodRatio(ut, ue, num_examples=num_examples),
           lambda k: layer.bestMatchesLarge(ut, ue, k=k, num_examples=num_examples))
    yield ("asnorm", layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, num_examples=num_examples),
           lambda k: layer.asNormBestMatchesLarge(ut, ue, k=k, test_stats=ts, enroll_stats=es,
                                                  num_examples=num_examples))


@gpu
@pytest.mark.parametrize("num_examples", [1.0, 3.0])
@pytest.mark.parametrize("nt", [1, 255, 257, 1037])
@pytest.mark.parametrize("ne", [1, 31, 255, 257, 700, 4099, 49152, 49153])
def test_equals_stable_sort_of_matrix(setup, nt, ne, num_examples):
    layer, ut, ue, uc = setup
    for name, full, run in both_forms(layer, ut[:nt], ue[:ne], uc, num_examples):
        srt = listed_sort(full)
        del full
        for k in KS:
            check_equal(run(k), expected_listed(srt, k))
    # AS-norm statistics computed inside the call
    ts, es = stats(layer, ut[:nt], ue[:ne], uc, 100, num_examples)
    want = expected_listed(listed_sort(layer.asNorm(ut[:nt], ue[:ne], test_stats=ts, enroll_stats=es,
                                             num_examples=num_examples)), 100)
    check_equal(layer.asNormBestMatchesLarge(ut[:nt], ue[:ne], uc, k=100, top_n=100, num_examples=num_examples), want)


@gpu
def test_large_shapes(ktf):
    """20 000 x 60 000: many row chunks, rows past the shared-memory limit; compared in blocks of 2000 rows."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    g = torch.Generator(device="cuda").manual_seed(17)
    x = torch.randn((85000, DIM), generator=g, device="cuda")
    u = layer.transformVector((x / x.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
    ut, ue, uc = u[:20000], u[20000:80000], u[80000:]
    ts, es = stats(layer, ut, ue, uc, 300)
    for k in (100, 1024):
        raw = layer.bestMatchesLarge(ut, ue, k=k)
        norm = layer.asNormBestMatchesLarge(ut, ue, k=k, test_stats=ts, enroll_stats=es)
        for r0 in range(0, 20000, 2000):
            rows = slice(r0, r0 + 2000)
            want = expected_listed(listed_sort(layer.logLikelihoodRatio(ut[rows], ue)), k)
            check_equal((raw[0][rows], raw[1][rows]), want)
            full = layer.asNorm(ut[rows], ue, test_stats=(ts[0][rows], ts[1][rows]), enroll_stats=es)
            check_equal((norm[0][rows], norm[1][rows]), expected_listed(listed_sort(full), k))


@gpu
def test_ties_come_back_lowest_column_first(setup):
    """One enrolled vector copied to 700 columns spread over the row (copies get equal statistics); the test rows
    include that vector at positions in different row chunks (4099 columns: 3840 rows per chunk), where the 700
    equal scores are at or near the top and straddle rank k for k < 700."""
    import torch
    layer, ut, ue, uc = setup
    ne = 4099
    cols = torch.from_numpy(np.sort(np.random.default_rng(5).choice(ne, size=700, replace=False))).cuda()
    ue2 = ue[:ne].clone()
    ue2[cols] = ue[int(cols[0])]
    ut2 = torch.cat([ut] * 5)[:4500].clone()
    at = [0, 3839, 3840, 4499]
    ut2[at] = ue[int(cols[0])]
    for name, full, run in both_forms(layer, ut2, ue2, uc):
        tie = full[at][:, cols[:1]]
        assert torch.equal(full[at][:, cols], tie.expand(len(at), len(cols))), name
        srt = listed_sort(full)
        del full
        for k in (33, 256, 699, 700, 701, 1024):
            s, i = run(k)
            check_equal((s, i), expected_listed(srt, k))
            for j, r in enumerate(at):
                listed = i[r][s[r] == tie[j, 0]]
                assert len(listed) > 0 and torch.equal(listed, cols[:len(listed)]), (name, k, r)


def _order_keys(v):
    """The radix select's unsigned order keys of float32 scores, as int64."""
    import torch
    b = v.contiguous().view(torch.int32).to(torch.int64) & 0xffffffff
    return torch.where(b >= 0x80000000, 0xffffffff - b, b | 0x80000000)


@gpu
@pytest.mark.parametrize("bit", [20, 10])
def test_ties_across_radix_digit_boundaries(setup, bit):
    """Two enrolled vectors whose scores against test row 0 are neighbours in the row whose order keys sit on either
    side of a digit boundary of the radix select (bit 20: the first 12-bit digit differs; bit 10: only the middle 10-bit
    digit differs), each copied to 200 columns: rank k falls on the first, inside and at the end of either group of equal
    scores, and between them."""
    import torch
    layer, ut, ue, uc = setup
    ne = 4099
    row = layer.logLikelihoodRatio(ut[:1], ue[:ne])[0]
    s, order = torch.sort(row, descending=True, stable=True)
    keys = _order_keys(s)
    hi_same = (keys[1:] >> (bit + 10 if bit == 10 else 32)) == (keys[:-1] >> (bit + 10 if bit == 10 else 32))
    cross = ((keys[1:] >> bit) != (keys[:-1] >> bit)) & hi_same
    pos = [p for p in torch.nonzero(cross).flatten().tolist() if 60 <= p < 600]
    assert pos, f"no neighbouring scores across bit {bit} in row 0"
    a, b = int(order[pos[0]]), int(order[pos[0] + 1])
    rng = np.random.default_rng(bit)
    cols = torch.from_numpy(rng.choice(ne, size=400, replace=False)).cuda()
    ue2 = ue[:ne].clone()
    ue2[cols[:200]] = ue[a]
    ue2[cols[200:]] = ue[b]
    ut2 = ut[:257].contiguous()
    full = layer.logLikelihoodRatio(ut2, ue2)
    va, vb = full[0, cols[0]], full[0, cols[200]]
    assert bool((full[0, cols[:200]] == va).all()) and bool((full[0, cols[200:]] == vb).all())
    ka, kb = _order_keys(va.reshape(1)), _order_keys(vb.reshape(1))
    assert bool(ka > kb) and bool((ka >> bit) != (kb >> bit))
    m = int((full[0] > va).sum())                              # rank of the first score of the upper group
    srt = listed_sort(full)
    ks = sorted({min(max(k, 33), 1024) for k in (m + 1, m + 100, m + 201, m + 202, m + 300, m + 402)})
    for k in ks:
        got = layer.bestMatchesLarge(ut2, ue2, k=k)
        check_equal(got, expected_listed(srt, k))
        s0, i0 = got[0][0], got[1][0]
        for v in (va, vb):
            listed = i0[s0 == v]
            group = torch.sort(torch.nonzero(full[0] == v).flatten()).values
            assert torch.equal(listed, group[:len(listed)]), (bit, k)


@gpu
def test_row_independence(setup):
    """The same rows alone, in other batches and in calls whose row count moves the chunk boundaries (49 153 columns:
    256 rows per chunk) give the same bits."""
    import torch
    layer, ut, ue, uc = setup
    ts, es = stats(layer, ut, ue, uc, 100)
    for k in (100, 1024):
        ref = (layer.bestMatchesLarge(ut, ue, k=k),
               layer.asNormBestMatchesLarge(ut, ue, k=k, test_stats=ts, enroll_stats=es))
        perm = torch.from_numpy(np.random.default_rng(9).permutation(N_TEST)).cuda()
        for rows in (perm[:1], perm[:300], perm[300:813], perm):
            sub = ut[rows].contiguous()
            sub_ts = (ts[0][rows].contiguous(), ts[1][rows].contiguous())
            got = (layer.bestMatchesLarge(sub, ue, k=k),
                   layer.asNormBestMatchesLarge(sub, ue, k=k, test_stats=sub_ts, enroll_stats=es))
            for (gs, gi), (rs, ri) in zip(got, ref):
                assert torch.equal(gs, rs[rows]) and torch.equal(gi, ri[rows])


@gpu
def test_sigma_zero_lists_plus_inf_only(setup):
    """Zero deviations on some rows and columns (given statistics), and on all of them (a cohort of one vector repeated:
    computed statistics): +inf entries are listed, NaN and -inf entries never."""
    import torch
    layer, ut, ue, uc = setup
    nt, ne = 300, 4099
    ts, es = stats(layer, ut[:nt], ue[:ne], uc, 100)
    t_std, e_std = ts[1].clone(), es[1].clone()
    t_std[::3] = 0.0
    e_std[::5] = 0.0
    ts, es = (ts[0], t_std), (es[0], e_std)
    full = layer.asNorm(ut[:nt], ue[:ne], test_stats=ts, enroll_stats=es)
    assert bool((full == float("inf")).any()) and bool((full == float("-inf")).any()) and bool(torch.isnan(full).any())
    srt = listed_sort(full)
    for k in (33, 100, 1024):
        s, i = layer.asNormBestMatchesLarge(ut[:nt], ue[:ne], k=k, test_stats=ts, enroll_stats=es)
        check_equal((s, i), expected_listed(srt, k))
        assert not bool(torch.isnan(s).any()) and bool((s == float("inf")).any())
        assert not bool((s[i >= 0] == float("-inf")).any())
    flat = uc[:1].expand(200, DIM).contiguous()
    full = layer.asNorm(ut[:nt], ue[:ne], flat, top_n=100)
    srt = listed_sort(full)
    for k in (33, 1024):
        check_equal(layer.asNormBestMatchesLarge(ut[:nt], ue[:ne], flat, k=k, top_n=100), expected_listed(srt, k))


@gpu
def test_consistent_with_small_k_path(setup):
    import torch
    layer, ut, ue, uc = setup
    for ne in (700, 49153):
        ts, es = stats(layer, ut, ue[:ne], uc, 100)
        small = (lambda k: layer.bestMatches(ut, ue[:ne], k=k),
                 lambda k: layer.asNormBestMatches(ut, ue[:ne], k=k, test_stats=ts, enroll_stats=es))
        large = (lambda k: layer.bestMatchesLarge(ut, ue[:ne], k=k),
                 lambda k: layer.asNormBestMatchesLarge(ut, ue[:ne], k=k, test_stats=ts, enroll_stats=es))
        for sm, lg in zip(small, large):
            for k in (1, 32):
                check_equal(lg(k), sm(k))
            s, i = lg(33)
            check_equal((s[:, :32].contiguous(), i[:, :32].contiguous()), sm(32))


@gpu
def test_edges(setup, ktf):
    import torch
    from kaldi_tflite_b200 import _native as N
    layer, ut, ue, uc = setup
    ts, es = stats(layer, ut[:40], ue[:5], uc, 100)
    # fewer enrolled vectors than k: (-inf, -1) after the last one
    for name, full, run in both_forms(layer, ut[:40], ue[:5], uc):
        s, i = run(100)
        check_equal((s, i), expected_listed(listed_sort(full), 100))
        assert bool((i[:, 5:] == -1).all()) and bool((s[:, 5:] == float("-inf")).all())
    # no enrolled vector at all
    for s, i in (layer.bestMatchesLarge(ut[:33], ue[:0], k=100),
                 layer.asNormBestMatchesLarge(ut[:33], ue[:0], uc, k=100, top_n=100)):
        assert s.shape == (33, 100) and bool((i == -1).all()) and bool((s == float("-inf")).all())
    # no test vector: nothing to do
    for s, i in (layer.bestMatchesLarge(ut[:0], ue, k=100), layer.asNormBestMatchesLarge(ut[:0], ue, uc, k=100,
                                                                                            top_n=100)):
        assert s.shape == (0, 100) and i.shape == (0, 100)
    # k outside 1 .. 1024, from Python and through the C-ABI with a real handle
    out_s = torch.empty((40, 1025), device="cuda")
    out_i = torch.empty((40, 1025), device="cuda", dtype=torch.int64)
    ptrs = [ctypes.c_void_p(t.data_ptr()) for t in (ts[0], ts[1], es[0], es[1])]
    vp = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    for k in (0, 1025):
        with pytest.raises(ValueError, match="1024"):
            layer.bestMatchesLarge(ut[:40], ue[:5], k=k)
        with pytest.raises(ValueError, match="1024"):
            layer.asNormBestMatchesLarge(ut[:40], ue[:5], k=k, test_stats=ts, enroll_stats=es)
        rc = N.lib().ktf_plda_score_topk_large(layer.handle, vp(ut), 40, vp(ue), 5, k, vp(out_s), vp(out_i), None)
        assert rc == N.KTF_EINVAL and "1024" in N.last_error()
        rc = N.lib().ktf_plda_score_asnorm_topk_large(layer.handle, vp(ut), 40, vp(ue), 5, *ptrs, k, vp(out_s),
                                                      vp(out_i), None)
        assert rc == N.KTF_EINVAL and "1024" in N.last_error()
    # the k <= 32 entry points still stop at 32
    rc = N.lib().ktf_plda_score_topk(layer.handle, vp(ut), 40, vp(ue), 5, 33, vp(out_s), vp(out_i), None)
    assert rc == N.KTF_EINVAL
    # float64 layers have no tcgen05 score path
    mean, Tm, psi = synthetic_plda(DIM)
    l64 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float64)
    with pytest.raises(ValueError):
        l64.bestMatchesLarge(ut.double()[:10], k=100)
    with pytest.raises(ValueError):
        l64.asNormBestMatchesLarge(ut.double()[:10], u_cohort=uc.double(), k=100, top_n=10)
    with pytest.raises(ValueError):
        N.check(N.lib().ktf_plda_score_topk_large(l64.handle, vp(ut), 10, vp(ue), 5, 100, vp(out_s), vp(out_i), None))
    # the set against itself
    st = layer.cohortStats(ut, uc, top_n=100)
    ss = layer.cohortStats(ut, uc, top_n=100, role="enrolled", num_examples=3.0)
    check_equal(layer.bestMatchesLarge(ut, k=300, num_examples=3.0),
                expected_listed(listed_sort(layer.logLikelihoodRatio(ut, num_examples=3.0)), 300))
    check_equal(layer.asNormBestMatchesLarge(ut, k=300, test_stats=st, enroll_stats=ss, num_examples=3.0),
                expected_listed(listed_sort(layer.asNorm(ut, test_stats=st, enroll_stats=ss, num_examples=3.0)), 300))


@gpu
def test_against_float64_oracle(ktf):
    """257 x 700 from raw x-vectors (AS-norm: 1500-vector cohort, top_n 100): every listed score is within
    1e-3 max(|s|, 1) of the float64 oracle's score of the same rank."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    rng = np.random.default_rng(78)
    x = rng.standard_normal((257 + 700 + 1500, DIM))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(DIM)).astype(np.float32)
    u = layer.transformVector(torch.from_numpy(x).cuda())
    ut, ue, uc = u[:257], u[257:957], u[957:]
    uo = O.plda_transform(x, mean, Tm, psi, dtype=np.float64)
    llr = O.plda_llr(uo, psi)
    t, e, c = slice(0, 257), slice(257, 957), slice(957, None)
    top_t = -np.sort(-llr[t, c], axis=1)[:, :100]
    top_e = -np.sort(-llr[c, e], axis=0)[:100, :]
    s = llr[t, e]
    norm = 0.5 * ((s - top_e.mean(axis=0)[None, :]) / top_e.std(axis=0)[None, :]
                  + (s - top_t.mean(axis=1)[:, None]) / top_t.std(axis=1)[:, None])
    for ref, run in ((s, lambda k: layer.bestMatchesLarge(ut, ue, k=k)),
                     (norm, lambda k: layer.asNormBestMatchesLarge(ut, ue, uc, k=k, top_n=100))):
        ref_sorted = -np.sort(-ref, axis=1)
        for k in (33, 100, 700):
            got_s, got_i = run(k)
            idx = got_i.cpu().numpy()
            assert idx.min() >= 0 and idx.max() < 700 and all(len(set(r)) == k for r in idx)
            listed = got_s.cpu().numpy().astype(np.float64)
            want = ref_sorted[:, :k]
            assert np.all(np.abs(listed - want) <= 1e-3 * np.maximum(np.abs(want), 1.0))


@gpu
def test_cuda_graph_capture_and_replay(setup):
    import torch
    layer, ut, ue, uc = setup
    st, se = ut[:700].clone(), ue[:6000].clone()
    ts, es = stats(layer, st, se, uc, 100)
    gts, ges = (ts[0].clone(), ts[1].clone()), (es[0].clone(), es[1].clone())

    def run():
        return (layer.bestMatchesLarge(st, se, k=100),
                layer.asNormBestMatchesLarge(st, se, k=1024, test_stats=gts, enroll_stats=ges))

    run()                                               # grows the workspace for these shapes
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed = run()
    nts, nes = stats(layer, ut[300:1000], ue[7000:13000], uc, 100)
    st.copy_(ut[300:1000])
    se.copy_(ue[7000:13000])
    for dst, src in zip(gts + ges, nts + nes):
        dst.copy_(src)
    g.replay()
    torch.cuda.synchronize()
    nt, ne = ut[300:1000].contiguous(), ue[7000:13000].contiguous()
    check_equal(graphed[0], layer.bestMatchesLarge(nt, ne, k=100))
    check_equal(graphed[1], layer.asNormBestMatchesLarge(nt, ne, k=1024, test_stats=nts, enroll_stats=nes))


def _numpy_stable_merge(s_in, i_in, k):
    """First k of a stable descending sort by score of every row's concatenated lists, without index < 0, NaN and
    -inf entries, padded with (-inf, -1)."""
    L, n, _ = s_in.shape
    out_s = np.full((n, k), -np.inf, np.float32)
    out_i = np.full((n, k), -1, np.int64)
    for r in range(n):
        s, i = s_in[:, r].ravel(), i_in[:, r].ravel()
        keep = (i >= 0) & ~np.isnan(s) & (s != -np.inf)
        s, i = s[keep], i[keep]
        order = np.argsort(-s.astype(np.float64), kind="stable")[:k]
        out_s[r, :len(order)] = s[order]
        out_i[r, :len(order)] = i[order]
    return out_s, out_i


@gpu
def test_topk_merge_large_against_numpy(ktf):
    """Many ties, on values next to the radix digit boundaries of the order keys (bits 20 and 10) and one ulp apart,
    with +inf, -inf, NaN and empty entries; lists long enough for both the shared-memory and the L2 form of a row."""
    import torch
    from kaldi_tflite_b200 import _native as N
    rng = np.random.default_rng(11)
    base = np.float32([-3.5, 0.25, 2.0, 7.5]).view(np.uint32)
    vals = np.concatenate([(base[:, None] + np.uint32([0, 1, 1023, 1024, 1025, (1 << 20) - 1, 1 << 20])).ravel()
                           .view(np.float32), np.float32([np.inf, -np.inf, np.nan])])
    for L, n, k_in in ((5, 300, 300), (3, 40, 20000)):
        s_in = rng.choice(vals, size=(L, n, k_in)).astype(np.float32)
        i_in = rng.integers(0, 1 << 40, size=(L, n, k_in)).astype(np.int64)
        i_in[rng.random(i_in.shape) < 0.2] = -1                                                     # empty entries
        i_in[:, :7] = -1                                                                             # rows with nothing
        ds, di = torch.from_numpy(s_in).cuda(), torch.from_numpy(i_in).cuda()
        for k in (1, 32, 33, 500, 1024):
            os_, oi = torch.empty((n, k), device="cuda"), torch.empty((n, k), device="cuda", dtype=torch.int64)
            N.check(N.lib().ktf_topk_merge_large(ctypes.c_void_p(ds.data_ptr()), ctypes.c_void_p(di.data_ptr()), L, n,
                                                 k_in, k, ctypes.c_void_p(os_.data_ptr()),
                                                 ctypes.c_void_p(oi.data_ptr()), None))
            torch.cuda.synchronize()
            ws, wi = _numpy_stable_merge(s_in, i_in, k)
            assert np.array_equal(oi.cpu().numpy(), wi), (L, k_in, k)
            assert np.array_equal(os_.cpu().numpy().view(np.uint32), ws.view(np.uint32)), (L, k_in, k)


@gpu
def test_sharded_two_ranks_gloo(tmp_path):
    for r in run_two_ranks(tmp_path, "topk_large", "gloo"):
        assert r["ok"], r


@gpu
def test_sharded_two_gpus_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    for r in run_two_ranks(tmp_path, "topk_large", "nccl"):
        assert r["ok"], r
