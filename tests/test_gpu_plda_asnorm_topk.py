"""
PLDA.asNormBestMatches / ktf_plda_score_asnorm_topk: the k best enrolled vectors of every test vector by AS-norm score,
from the tcgen05 score GEMM's normalising top-k epilogue, without the matrix.  The contract: row i equals the first k
entries of a stable descending sort of row i of the float32 `asNorm` matrix (same statistics), bit for bit, with NaN and
-inf entries left out and the row padded with (-inf, -1).

PLDA.asNorm(score_dtype=torch.bfloat16) / ktf_plda_score_asnorm_ex(KTF_SCORES_BF16): the float32 normalised matrix
rounded once to bfloat16, bit-equal to `asNorm(...).to(torch.bfloat16)`.

The argument checks that need no device run everywhere; the rest is marked gpu.
"""

import ctypes

import numpy as np
import pytest

from oracle import ktf_oracle as O
from plda_testlib import DIM, check_equal, epilogue_warp_runs, expected_listed, ktf, listed_sort  # noqa: F401
from plda_testlib import plda_vectors, run_two_ranks, stats
from test_gpu_tdnn_plda import synthetic_plda

gpu = pytest.mark.gpu

KS = (1, 2, 7, 10, 16, 31, 32)


# ---- argument checks (no device) ----

def test_c_entry_points_reject_bad_arguments():
    from kaldi_tflite_b200 import _native as N
    lib = N.lib()
    p = ctypes.c_void_p(0)
    for k in (0, 33, -1):
        rc = lib.ktf_plda_score_asnorm_topk(None, p, 10, p, 10, p, p, p, p, k, p, p, None)
        assert rc == N.KTF_EINVAL and "KTF_PLDA_TOPK_MAX" in N.last_error()
    rc = lib.ktf_plda_score_asnorm_topk(None, p, 10, p, 10, p, p, p, p, 5, p, p, None)
    assert rc == N.KTF_EINVAL and "null handle" in N.last_error()
    for fmt in (2, -1, 7):
        rc = lib.ktf_plda_score_asnorm_ex(None, p, 10, p, 10, p, p, p, p, p, 10, fmt, None)
        assert rc == N.KTF_EINVAL and "score_format" in N.last_error()
    for fmt in (N.KTF_SCORES_NATIVE, N.KTF_SCORES_BF16):
        rc = lib.ktf_plda_score_asnorm_ex(None, p, 10, p, 10, p, p, p, p, p, 10, fmt, None)
        assert rc == N.KTF_EINVAL and "null handle" in N.last_error()


def test_python_argument_validation():
    import torch
    import kaldi_tflite_b200 as ktf
    mean, Tm, psi = synthetic_plda(DIM)
    l32 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32)
    l64 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float64)
    ut, ue = torch.zeros((6, DIM)), torch.zeros((5, DIM))
    ts = (torch.zeros(6), torch.ones(6))
    es = (torch.zeros(5), torch.ones(5))
    with pytest.raises(ValueError, match="float32"):
        l64.asNormBestMatches(ut.double(), ue.double(), k=3, test_stats=ts, enroll_stats=es)
    with pytest.raises(ValueError, match="float32"):
        l64.asNorm(ut.double(), ue.double(), test_stats=ts, enroll_stats=es, score_dtype=torch.bfloat16)
    for k in (0, 33):
        with pytest.raises(ValueError, match="32"):
            l32.asNormBestMatches(ut, ue, k=k, test_stats=ts, enroll_stats=es)
    with pytest.raises(ValueError, match="u_cohort and top_n"):
        l32.asNormBestMatches(ut, ue, k=3, test_stats=ts)
    with pytest.raises(ValueError, match="enroll_stats"):
        l32.asNormBestMatches(ut, ue, k=3, test_stats=ts, enroll_stats=(torch.zeros(4), torch.ones(4)))
    with pytest.raises(ValueError, match="test_stats"):
        l32.asNormBestMatches(ut, ue, k=3, test_stats=(ts[0].double(), ts[1]), enroll_stats=es)
    with pytest.raises(ValueError, match="score_dtype"):
        l32.asNorm(ut, ue, test_stats=ts, enroll_stats=es, score_dtype=torch.float16)
    with pytest.raises(ValueError, match="out must be"):
        l32.asNorm(ut, ue, test_stats=ts, enroll_stats=es, score_dtype=torch.bfloat16, out=torch.empty((6, 5)))
    with pytest.raises(ValueError, match="out must be"):
        l32.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=torch.empty((6, 4), dtype=torch.bfloat16))


# ---- on the GPU ----

@pytest.fixture(scope="module")
def setup(ktf):
    """A float32 layer, transformed vectors (1037 test, 4099 enrolled, a 2000-vector cohort) and the raw x-vectors."""
    layer, (ut, ue, uc), _, _ = plda_vectors(ktf, (1037, 4099, 2000), 2025)
    return layer, ut, ue, uc


@gpu
@pytest.mark.parametrize("num_examples", [1.0, 3.0])
@pytest.mark.parametrize("nt", [1, 255, 257, 1037])
@pytest.mark.parametrize("ne", [1, 31, 255, 257, 700, 4099])
def test_topk_equals_stable_sort_of_asnorm_matrix(setup, nt, ne, num_examples):
    layer, ut, ue, uc = setup
    ts, es = stats(layer, ut[:nt], ue[:ne], uc, 100, num_examples)
    full = layer.asNorm(ut[:nt], ue[:ne], test_stats=ts, enroll_stats=es, num_examples=num_examples)
    for k in KS:
        got = layer.asNormBestMatches(ut[:nt], ue[:ne], k=k, test_stats=ts, enroll_stats=es, num_examples=num_examples)
        check_equal(got, expected_listed(listed_sort(full), k))
    # statistics computed from the cohort inside the call
    got = layer.asNormBestMatches(ut[:nt], ue[:ne], uc, k=10, top_n=100, num_examples=num_examples)
    check_equal(got, expected_listed(listed_sort(full), 10))


@gpu
@pytest.mark.parametrize("k", [10, 32])
def test_topk_large(ktf, k):
    """20 000 x 60 000: many units per cluster and several n-ranges, against the asNorm matrix."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    g = torch.Generator(device="cuda").manual_seed(17)
    x = torch.randn((85000, DIM), generator=g, device="cuda")
    u = layer.transformVector((x / x.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
    ut, ue, uc = u[:20000], u[20000:80000], u[80000:]
    ts, es = stats(layer, ut, ue, uc, 300)
    got = layer.asNormBestMatches(ut, ue, k=k, test_stats=ts, enroll_stats=es)
    full = layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es)
    want = expected_listed(listed_sort(full), k)
    del full
    check_equal(got, want)


@gpu
def test_ties_come_back_lowest_column_first(setup):
    """One enrolled vector copied to columns in different column quarters, n-tiles and n-ranges (copies get equal
    statistics); the test rows include that vector itself, so the copies tie near the top of its row."""
    import torch
    layer, ut, ue, uc = setup
    cols = [5, 200, 300, 1000, 2100, 3333, 4000]
    ue2 = ue.clone()
    ue2[cols] = ue[cols[0]]
    ut2 = torch.cat([ue[cols[0]:cols[0] + 1], ut[:300]]).contiguous()
    ts, es = stats(layer, ut2, ue2, uc, 100)
    assert torch.equal(es[0][cols], es[0][cols[:1]].expand(len(cols)))
    full = layer.asNorm(ut2, ue2, test_stats=ts, enroll_stats=es)
    row = full[0, cols]
    assert torch.equal(row, row[:1].expand(len(cols))), "copies of one vector must score equal"
    for k in (7, 16, 32):
        check_equal(layer.asNormBestMatches(ut2, ue2, k=k, test_stats=ts, enroll_stats=es),
                    expected_listed(listed_sort(full), k))
    s, i = layer.asNormBestMatches(ut2, ue2, k=32, test_stats=ts, enroll_stats=es)
    tied = [int(c) for c, v in zip(i[0].tolist(), s[0].tolist()) if v == float(row[0])]
    assert tied == cols


@gpu
def test_sigma_zero_lists_plus_inf_only(setup):
    """Zero deviations on some rows and columns: +inf entries are listed, NaN and -inf entries never."""
    import torch
    layer, ut, ue, uc = setup
    nt, ne = 300, 700
    ts, es = stats(layer, ut[:nt], ue[:ne], uc, 100)
    t_std, e_std = ts[1].clone(), es[1].clone()
    t_std[::3] = 0.0
    e_std[::5] = 0.0
    ts, es = (ts[0], t_std), (es[0], e_std)
    full = layer.asNorm(ut[:nt], ue[:ne], test_stats=ts, enroll_stats=es)
    assert bool((full == float("inf")).any()) and bool((full == float("-inf")).any()) and bool(torch.isnan(full).any())
    for k in (1, 10, 32):
        s, i = layer.asNormBestMatches(ut[:nt], ue[:ne], k=k, test_stats=ts, enroll_stats=es)
        check_equal((s, i), expected_listed(listed_sort(full), k))
        assert not bool(torch.isnan(s).any()) and bool((s == float("inf")).any())
        listed = i >= 0
        assert not bool((s[listed] == float("-inf")).any())


@gpu
def test_edges(setup, ktf):
    import torch
    from kaldi_tflite_b200 import _native as N
    layer, ut, ue, uc = setup
    ts, es = stats(layer, ut[:40], ue[:5], uc, 100)
    # fewer enrolled vectors than k: (-inf, -1) after the last one
    s, i = layer.asNormBestMatches(ut[:40], ue[:5], k=9, test_stats=ts, enroll_stats=es)
    check_equal((s, i), expected_listed(listed_sort(layer.asNorm(ut[:40], ue[:5], test_stats=ts, enroll_stats=es)), 9))
    assert bool((i[:, 5:] == -1).all()) and bool((s[:, 5:] == float("-inf")).all())
    # no enrolled vector at all
    s, i = layer.asNormBestMatches(ut[:33], ue[:0], uc, k=4, top_n=100)
    assert s.shape == (33, 4) and bool((i == -1).all()) and bool((s == float("-inf")).all())
    # no test vector: nothing to do
    s, i = layer.asNormBestMatches(ut[:0], ue, uc, k=4, top_n=100)
    assert s.shape == (0, 4) and i.shape == (0, 4)
    # k outside 1 .. 32, from Python and through the C-ABI with a real handle
    for k in (0, 33):
        with pytest.raises(ValueError, match="32"):
            layer.asNormBestMatches(ut[:40], ue[:5], k=k, test_stats=ts, enroll_stats=es)
        out_s = torch.empty((40, 33), device="cuda")
        out_i = torch.empty((40, 33), device="cuda", dtype=torch.int64)
        ptrs = [ctypes.c_void_p(t.data_ptr()) for t in (ts[0], ts[1], es[0], es[1])]
        rc = N.lib().ktf_plda_score_asnorm_topk(layer.handle, ctypes.c_void_p(ut.data_ptr()), 40,
                                                ctypes.c_void_p(ue.data_ptr()), 5, *ptrs, k,
                                                ctypes.c_void_p(out_s.data_ptr()), ctypes.c_void_p(out_i.data_ptr()),
                                                None)
        assert rc == N.KTF_EINVAL and "32" in N.last_error()
    # float64 layers have no tcgen05 score path
    mean, Tm, psi = synthetic_plda(DIM)
    l64 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float64)
    with pytest.raises(ValueError):
        l64.asNormBestMatches(ut.double()[:10], u_cohort=uc.double(), k=3, top_n=10)
    with pytest.raises(ValueError):
        h = l64.handle
        rc = N.lib().ktf_plda_score_asnorm_topk(h, ctypes.c_void_p(ut.data_ptr()), 10, ctypes.c_void_p(ue.data_ptr()),
                                                5, *ptrs, 3, ctypes.c_void_p(out_s.data_ptr()),
                                                ctypes.c_void_p(out_i.data_ptr()), None)
        N.check(rc)
    # the set against itself
    ss = layer.cohortStats(ut, uc, top_n=100, role="enrolled", num_examples=3.0)
    st = layer.cohortStats(ut, uc, top_n=100)
    full = layer.asNorm(ut, test_stats=st, enroll_stats=ss, num_examples=3.0)
    check_equal(layer.asNormBestMatches(ut, k=16, test_stats=st, enroll_stats=ss, num_examples=3.0),
                expected_listed(listed_sort(full), 16))


@gpu
def test_against_float64_oracle(ktf):
    """257 x 700 from raw x-vectors, 1500-vector cohort, top_n 100: every listed s' is within 1e-3 max(|s'|, 1) of the
    float64 oracle's AS-norm k-th best (or above it)."""
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
    mt, st = top_t.mean(axis=1)[:, None], top_t.std(axis=1)[:, None]
    me, se = top_e.mean(axis=0)[None, :], top_e.std(axis=0)[None, :]
    s = llr[t, e]
    ref = 0.5 * ((s - me) / se + (s - mt) / st)
    ref_sorted = -np.sort(-ref, axis=1)
    for k in (1, 10, 32):
        got_s, got_i = layer.asNormBestMatches(ut, ue, uc, k=k, top_n=100)
        idx = got_i.cpu().numpy()
        assert idx.min() >= 0 and idx.max() < 700 and all(len(set(r)) == k for r in idx)
        at = np.take_along_axis(ref, idx, axis=1)
        kth = ref_sorted[:, k - 1:k]
        assert np.all(kth - at <= 1e-3 * np.maximum(np.abs(kth), 1.0))
        listed = got_s.cpu().numpy().astype(np.float64)
        assert np.all(np.abs(listed - at) <= 1e-3 * np.maximum(np.abs(at), 1.0))


_EW_CHILD = r"""
rng = np.random.default_rng(6)
x = rng.standard_normal((1037 + 4099 + 3000, 128)).astype(np.float32)
u = layer.transformVector(torch.from_numpy(x).cuda())
ut, ue, uc = u[:1037].contiguous(), u[1037:5136].contiguous(), u[5136:].contiguous()
out = {{}}
for k in (1, 7, 16, 32):
    s, i = layer.asNormBestMatches(ut, ue, uc, k=k, top_n=300, num_examples=3.0)
    out[f"s{{k}}"], out[f"i{{k}}"] = s.cpu().numpy(), i.cpu().numpy()
out["bf16"] = layer.asNorm(ut, ue, uc, top_n=300, score_dtype=torch.bfloat16).view(torch.int16).cpu().numpy()
np.savez({path!r}, **out)
"""


@gpu
def test_independent_of_epilogue_warp_count(tmp_path):
    res = epilogue_warp_runs(tmp_path, _EW_CHILD)
    for key in res["8"].files:
        assert np.array_equal(res["8"][key], res["16"][key]), key


@gpu
def test_cuda_graph_capture_and_replay(setup):
    import torch
    layer, ut, ue, uc = setup
    st, se = ut[:700].clone(), ue[:1500].clone()
    ts, es = stats(layer, st, se, uc, 100)
    gts, ges = (ts[0].clone(), ts[1].clone()), (es[0].clone(), es[1].clone())

    def run():
        return (layer.asNormBestMatches(st, se, k=10, test_stats=gts, enroll_stats=ges),
                layer.asNorm(st, se, test_stats=gts, enroll_stats=ges, score_dtype=torch.bfloat16))

    run()                                               # grows the workspace for these shapes
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        (gs, gi), gb = run()
    nts, nes = stats(layer, ut[300:1000], ue[2000:3500], uc, 100)
    st.copy_(ut[300:1000])
    se.copy_(ue[2000:3500])
    for dst, src in zip(gts + ges, nts + nes):
        dst.copy_(src)
    g.replay()
    torch.cuda.synchronize()
    want = layer.asNormBestMatches(ut[300:1000].contiguous(), ue[2000:3500].contiguous(), k=10, test_stats=nts,
                                   enroll_stats=nes)
    check_equal((gs, gi), want)
    assert torch.equal(gb, layer.asNorm(ut[300:1000].contiguous(), ue[2000:3500].contiguous(), test_stats=nts,
                                        enroll_stats=nes, score_dtype=torch.bfloat16))


@gpu
@pytest.mark.parametrize("ne", [4099, 4096, 257, 31, 1])
def test_bf16_matrix_equals_rounded_float32(setup, ne):
    """n_enroll not a multiple of 8 puts the row ends on the ragged store path."""
    import torch
    layer, ut, ue, uc = setup
    ts, es = stats(layer, ut, ue[:ne], uc, 300, 3.0)
    want = layer.asNorm(ut, ue[:ne], test_stats=ts, enroll_stats=es, num_examples=3.0).to(torch.bfloat16)
    got = layer.asNorm(ut, ue[:ne], test_stats=ts, enroll_stats=es, num_examples=3.0, score_dtype=torch.bfloat16)
    assert got.dtype is torch.bfloat16 and torch.equal(got.view(torch.int16), want.view(torch.int16))
    computed = layer.asNorm(ut, ue[:ne], uc, top_n=300, num_examples=3.0, score_dtype=torch.bfloat16)
    assert torch.equal(computed.view(torch.int16), want.view(torch.int16))
    # a sliced bfloat16 `out`: a 16-byte-aligned pitch, and one that is not (per-row stores)
    for pad in (16 - ne % 8, 3):
        pitch = ne + pad
        buf = torch.full((ut.shape[0], pitch), 7.0, device="cuda", dtype=torch.bfloat16)
        out = layer.asNorm(ut, ue[:ne], test_stats=ts, enroll_stats=es, num_examples=3.0, out=buf[:, :ne])
        assert out.data_ptr() == buf.data_ptr()
        assert torch.equal(out.view(torch.int16), want.view(torch.int16)) and bool((buf[:, ne:] == 7.0).all())


@gpu
def test_sharded_two_ranks_gloo(tmp_path):
    for r in run_two_ranks(tmp_path, "asnorm_topk", "gloo"):
        assert r["ok"], r


@gpu
def test_sharded_two_gpus_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    for r in run_two_ranks(tmp_path, "asnorm_topk", "nccl"):
        assert r["ok"], r
