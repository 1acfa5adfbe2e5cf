"""
PLDA.cohortStats / PLDA.asNorm / ktf_plda_cohort_stats / ktf_plda_score_asnorm: adaptive symmetric score normalisation
(AS-norm1) on the tcgen05 score kernel.  The contract: the top_n-th largest cohort score is bit-equal to entry
top_n - 1 of a descending sort of the logLikelihoodRatio row (test role) or column (enrolled role); mean and std are
within 1 float32 ulp of the float64 statistics of that exact top_n; the normalised matrix matches the float64 formula
applied to the fp32 logLikelihoodRatio matrix and the returned statistics within 2e-6 max(|s'|, 1).
"""

import ctypes

import numpy as np
import pytest

from oracle import ktf_oracle as O
from plda_testlib import DIM, epilogue_warp_runs, ktf, plda_vectors, run_two_ranks  # noqa: F401
from test_gpu_tdnn_plda import synthetic_plda

pytestmark = pytest.mark.gpu

NS = (1, 255, 257, 1037)
TOP_NS = (2, 7, 100, 300, 1000)


@pytest.fixture(scope="module")
def setup(ktf):
    """A float32 layer, 1037 transformed test vectors and a 60 000-vector transformed cohort."""
    layer, (ut, uc), _, _ = plda_vectors(ktf, (1037, 60000), 99, cuda_rng=True)
    return layer, ut, uc


def stats_with_nth(layer, u, uc, top_n, role, num_examples=1.0):
    """ktf_plda_cohort_stats through the C-ABI, with the top_n-th largest score."""
    import torch
    from kaldi_tflite_b200 import _native as N
    n = u.shape[0]
    out = [torch.empty((n,), device="cuda", dtype=torch.float32) for _ in range(3)]
    h = layer.handle_for(1.0 if role == "test" else num_examples)
    N.check(N.lib().ktf_plda_cohort_stats(h, ctypes.c_void_p(u.data_ptr()), n, ctypes.c_void_p(uc.data_ptr()),
                                          uc.shape[0], top_n,
                                          N.KTF_COHORT_AS_TEST if role == "test" else N.KTF_COHORT_AS_ENROLLED,
                                          *(ctypes.c_void_p(t.data_ptr()) for t in out),
                                          ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out


def cohort_scores(layer, u, uc, role, num_examples=1.0):
    """(n, n_cohort) fp32 cohort scores of every vector: rows of LLR(u, uc) or columns of LLR(uc, u, num_examples)."""
    if role == "test":
        return layer.logLikelihoodRatio(u, uc)
    return layer.logLikelihoodRatio(uc, u, num_examples=num_examples).t()


def check_stats(got, s, top_n):
    """got = (mean, std, nth) against `s`, the descending sort of every row of the cohort scores."""
    import torch
    mean, std, nth = got
    assert torch.equal(nth, s[:, top_n - 1]), f"{int((nth != s[:, top_n - 1]).sum())} thresholds differ"
    top = s[:, :top_n].double()
    w_mean = top.mean(dim=1)
    w_std = top.std(dim=1, unbiased=False)
    for g, w, name in ((mean, w_mean, "mean"), (std, w_std, "std")):
        wf = w.float().abs()
        ulp = torch.nextafter(wf, torch.full_like(wf, float("inf"))) - wf
        err = (g.double() - w).abs()
        bad = err > ulp.double()
        assert not bool(bad.any()), f"{name}: {int(bad.sum())} rows beyond 1 ulp, worst {float((err / ulp).max()):.2f} ulp"


def sorted_desc(full):
    import torch
    return torch.sort(full, dim=1, descending=True).values


@pytest.mark.parametrize("nc", [2, 31, 257, 4099, 60000])
@pytest.mark.parametrize("role,num_examples", [("test", 1.0), ("enrolled", 1.0), ("enrolled", 3.0)])
def test_selection_is_exact(setup, nc, role, num_examples):
    layer, ut, uc = setup
    for n in NS:
        s = sorted_desc(cohort_scores(layer, ut[:n], uc[:nc], role, num_examples))
        for top_n in sorted({t for t in TOP_NS if t <= nc} | {nc}):
            check_stats(stats_with_nth(layer, ut[:n], uc[:nc], top_n, role, num_examples), s, top_n)
        m, s = layer.cohortStats(ut[:n], uc[:nc], top_n=min(7, nc), role=role, num_examples=num_examples)
        want = stats_with_nth(layer, ut[:n], uc[:nc], min(7, nc), role, num_examples)
        assert np.array_equal(m.cpu().numpy(), want[0].cpu().numpy())
        assert np.array_equal(s.cpu().numpy(), want[1].cpu().numpy())


@pytest.mark.parametrize("role", ["test", "enrolled"])
def test_ties_straddle_the_threshold(setup, role):
    """Copies of one cohort vector occupy 20 ranks around rank 99 of vector 0's cohort scores (top_n = 100), and the
    cohort holds vector 0 itself."""
    import torch
    layer, ut, uc = setup
    u = ut[:300]
    base = uc[:3000]
    order = torch.argsort(cohort_scores(layer, u[:1], base, role)[0], descending=True)
    dup = base[order[90]][None].expand(20, DIM)
    cohort = torch.cat([base[order[:90]], dup, base[order[110:]], u[:1]]).contiguous()
    s = sorted_desc(cohort_scores(layer, u, cohort, role))
    at = (s[0] == cohort_scores(layer, u[:1], dup[:1].contiguous(), role)[0, 0]).nonzero()[:, 0]
    assert len(at) >= 20 and int(at.min()) < 99 < int(at.max()), "copies of one vector must score equal around rank 99"
    for top_n in (7, 100, 1000):
        check_stats(stats_with_nth(layer, u, cohort, top_n, role), s, top_n)


def test_edges(setup, ktf):
    import torch
    from kaldi_tflite_b200 import _native as N
    layer, ut, uc = setup
    for top_n, nc in ((1, 100), (101, 100), (2, 0)):
        for role in ("test", "enrolled"):
            with pytest.raises(ValueError, match="top_n"):
                layer.cohortStats(ut[:10], uc[:nc], top_n=top_n, role=role)
        buf = torch.empty((10,), device="cuda")
        p = ctypes.c_void_p(buf.data_ptr())
        rc = N.lib().ktf_plda_cohort_stats(layer.handle, ctypes.c_void_p(ut.data_ptr()), 10,
                                           ctypes.c_void_p(uc.data_ptr()), nc, top_n, N.KTF_COHORT_AS_TEST, p, p, None,
                                           None)
        assert rc == N.KTF_EINVAL
    with pytest.raises(ValueError, match="role"):
        layer.cohortStats(ut[:10], uc[:100], top_n=10, role="cohort")
    m, s = layer.cohortStats(ut[:0], uc[:100], top_n=10)
    assert m.shape == (0,) and s.shape == (0,)
    out = layer.asNorm(ut[:0], uc[:50], uc[:100], top_n=10)
    assert out.shape == (0, 50)
    with pytest.raises(ValueError):
        layer.asNorm(ut[:10], uc[:10])                          # no statistics and no cohort
    mean, Tm, psi = synthetic_plda(DIM)
    l64 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float64)
    with pytest.raises(ValueError):
        l64.cohortStats(ut.double()[:10], uc.double()[:100], top_n=10)
    with pytest.raises(ValueError):
        l64.asNorm(ut.double()[:10], u_cohort=uc.double()[:100], top_n=10)


def test_statistics_do_not_depend_on_batch_or_chunk(setup):
    """A vector's statistics alone, inside ragged batches and across chunk boundaries (60 000-long rows: 256-row chunks)."""
    import torch
    layer, ut, uc = setup
    for nc, top_n in ((4099, 300), (60000, 1000)):
        for role in ("test", "enrolled"):
            whole = layer.cohortStats(ut, uc[:nc], top_n=top_n, role=role, num_examples=3.0)
            for lo, hi in ((0, 1), (255, 256), (256, 513), (700, 1037), (5, 6)):
                part = layer.cohortStats(ut[lo:hi].contiguous(), uc[:nc], top_n=top_n, role=role, num_examples=3.0)
                assert torch.equal(part[0], whole[0][lo:hi]) and torch.equal(part[1], whole[1][lo:hi])
            again = layer.cohortStats(ut, uc[:nc], top_n=top_n, role=role, num_examples=3.0)
            assert torch.equal(again[0], whole[0]) and torch.equal(again[1], whole[1])


def asnorm_reference(full, ts, es):
    """float64 AS-norm of the fp32 matrix `full` with the statistics ts / es."""
    s = full.double()
    tm, tsd = (t.double()[:, None] for t in ts)
    em, esd = (t.double()[None, :] for t in es)
    return 0.5 * ((s - em) / esd + (s - tm) / tsd)


def check_asnorm(got, full, ts, es, rows=4096):
    for r0 in range(0, full.shape[0], rows):
        want = asnorm_reference(full[r0:r0 + rows], (ts[0][r0:r0 + rows], ts[1][r0:r0 + rows]), es)
        err = (got[r0:r0 + rows].double() - want).abs()
        tol = 2e-6 * want.abs().clamp(min=1.0)
        assert not bool((err > tol).any()), f"rows {r0}..: worst {float((err / tol).max()):.3f} of the tolerance"


@pytest.mark.parametrize("num_examples", [1.0, 3.0])
def test_normalised_matrix(setup, num_examples):
    import torch
    layer, ut, uc = setup
    ue, cohort = uc[:4099], uc[10000:12000]
    ts = layer.cohortStats(ut, cohort, top_n=300)
    es = layer.cohortStats(ue, cohort, top_n=300, role="enrolled", num_examples=num_examples)
    full = layer.logLikelihoodRatio(ut, ue, num_examples=num_examples)
    got = layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, num_examples=num_examples)
    check_asnorm(got, full, ts, es)
    computed = layer.asNorm(ut, ue, cohort, top_n=300, num_examples=num_examples)
    assert torch.equal(computed, got)
    # sliced output with a padded pitch, and a pitch that is not a multiple of 16 bytes (per-row stores)
    for pitch in (4104, 4101):
        buf = torch.full((1037, pitch), 7.0, device="cuda")
        out = layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, num_examples=num_examples, out=buf[:, :4099])
        assert torch.equal(out, got) and bool((buf[:, 4099:] == 7.0).all())
    # the set against itself
    ss = layer.cohortStats(ut, cohort, top_n=100, role="enrolled", num_examples=num_examples)
    self_scores = layer.asNorm(ut, test_stats=layer.cohortStats(ut, cohort, top_n=100), enroll_stats=ss,
                               num_examples=num_examples)
    check_asnorm(self_scores, layer.logLikelihoodRatio(ut, num_examples=num_examples),
                 layer.cohortStats(ut, cohort, top_n=100), ss)


def test_normalised_matrix_large(ktf):
    """20 000 x 60 000 (4.8 GB), statistics from a 10 000-vector cohort."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.randn((90000, DIM), generator=g, device="cuda")
    u = layer.transformVector((x / x.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
    ut, ue, cohort = u[:20000], u[20000:80000], u[80000:]
    ts = layer.cohortStats(ut, cohort, top_n=300)
    es = layer.cohortStats(ue, cohort, top_n=300, role="enrolled")
    got = layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es)
    full = layer.logLikelihoodRatio(ut, ue)
    check_asnorm(got, full, ts, es, rows=2048)
    del full
    assert torch.equal(layer.asNorm(ut, ue, cohort, top_n=300, out=got), got)


def test_sigma_zero_gives_ieee_division(setup):
    import torch
    layer, ut, uc = setup
    ue = uc[:64]
    ts = (torch.zeros(40, device="cuda"), torch.ones(40, device="cuda"))
    es = (torch.zeros(64, device="cuda"), torch.zeros(64, device="cuda"))
    got = layer.asNorm(ut[:40], ue, test_stats=ts, enroll_stats=es)
    full = layer.logLikelihoodRatio(ut[:40], ue)
    assert torch.equal(torch.isinf(got), full != 0) and torch.equal(torch.sign(got), torch.sign(full))


def test_against_float64_oracle(ktf):
    """257 x 700 from raw x-vectors, 1500-vector cohort, top_n 100, against the float64 broadcast-form oracle."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    rng = np.random.default_rng(77)
    x = rng.standard_normal((257 + 700 + 1500, DIM))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(DIM)).astype(np.float32)
    u = layer.transformVector(torch.from_numpy(x).cuda())
    ut, ue, uc = u[:257], u[257:957], u[957:]
    got = layer.asNorm(ut, ue, uc, top_n=100).cpu().numpy().astype(np.float64)
    uo = O.plda_transform(x, mean, Tm, psi, dtype=np.float64)
    llr = O.plda_llr(uo, psi)
    t, e, c = slice(0, 257), slice(257, 957), slice(957, None)
    top_t = -np.sort(-llr[t, c], axis=1)[:, :100]
    top_e = -np.sort(-llr[c, e], axis=0)[:100, :]
    mt, st = top_t.mean(axis=1)[:, None], top_t.std(axis=1)[:, None]
    me, se = top_e.mean(axis=0)[None, :], top_e.std(axis=0)[None, :]
    s = llr[t, e]
    want = 0.5 * ((s - me) / se + (s - mt) / st)
    assert np.all(np.abs(got - want) <= 1e-3 * np.maximum(np.abs(want), 1.0))


def test_cuda_graph_capture_and_replay(setup):
    import torch
    layer, ut, uc = setup
    st, se, sc = ut[:700].clone(), uc[:1500].clone(), uc[20000:23000].clone()

    def run():
        ts = layer.cohortStats(st, sc, top_n=100)
        es = layer.cohortStats(se, sc, top_n=100, role="enrolled")
        return ts, es, layer.asNorm(st, se, test_stats=ts, enroll_stats=es)

    run()                                               # grows the workspace for these shapes
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        gts, ges, gout = run()
    st.copy_(ut[300:1000])
    se.copy_(uc[5000:6500])
    sc.copy_(uc[30000:33000])
    g.replay()
    torch.cuda.synchronize()
    ts, es, out = run()
    for a, b in ((gts, ts), (ges, es)):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(gout, out)


_EW_CHILD = r"""
rng = np.random.default_rng(5)
x = rng.standard_normal((1037 + 4099 + 5000, 128)).astype(np.float32)
u = layer.transformVector(torch.from_numpy(x).cuda())
ut, ue, uc = u[:1037].contiguous(), u[1037:5136].contiguous(), u[5136:].contiguous()
ts = layer.cohortStats(ut, uc, top_n=300)
es = layer.cohortStats(ue, uc, top_n=300, role="enrolled", num_examples=3.0)
out = layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, num_examples=3.0)
np.savez({path!r}, tm=ts[0].cpu().numpy(), ts=ts[1].cpu().numpy(), em=es[0].cpu().numpy(), es=es[1].cpu().numpy(),
         out=out.cpu().numpy())
"""


def test_independent_of_epilogue_warp_count(tmp_path):
    res = epilogue_warp_runs(tmp_path, _EW_CHILD)
    for key in res["8"].files:
        assert np.array_equal(res["8"][key], res["16"][key]), key


def test_sharded_two_ranks_gloo(tmp_path):
    for r in run_two_ranks(tmp_path, "asnorm", "gloo"):
        assert r["ok"], r


def test_sharded_two_gpus_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    for r in run_two_ranks(tmp_path, "asnorm", "nccl"):
        assert r["ok"], r
