"""
Diarization back-end on the GPU: PLDA.withinScores (bit-equal to the transposed per-recording logLikelihoodRatio, and
against Kaldi's dense scores) and diarization.agglomerative_cluster (exactly the oracle's labels, merge lists and
counts), with the argument checks of both C entry points.
"""

import ctypes

import numpy as np
import pytest

from conftest import golden_path, load_golden, rmse
import ahc_oracle as O
from plda_testlib import DIM, ktf, plda_vectors  # noqa: F401  (ktf: fixture)

pytestmark = pytest.mark.gpu


def _within_vs_llr(layer, u, sizes):
    import torch
    mats = layer.withinScores(u, sizes)
    assert len(mats) == len(sizes)
    at = 0
    for m, n in zip(mats, sizes):
        assert m.shape == (n, n) and m.dtype == torch.float32
        if n:
            want = layer.logLikelihoodRatio(u[at:at + n].contiguous()).t()
            assert torch.equal(m, want), n
        at += n


@pytest.mark.parametrize("order", ["sorted", "unsorted"])
def test_within_scores_bit_equal(ktf, order):
    import torch
    sizes = [0, 1, 2, 255, 256, 257, 511, 513, 1000]
    if order == "unsorted":
        sizes = [513, 0, 256, 1000, 2, 255, 1, 511, 257]
    layer, blocks, _, _ = plda_vectors(ktf, sizes, seed=21)
    u = torch.cat([b for b in blocks if b.shape[0]]).contiguous()
    _within_vs_llr(layer, u, sizes)
    # the buffer is packed: group r at sum_{q<r} n_q^2
    mats = layer.withinScores(u, sizes)
    base = mats[0].untyped_storage().data_ptr()
    at = 0
    for m, n in zip(mats, sizes):
        if n:
            assert m.data_ptr() == base + 4 * at
        at += n * n


def test_within_scores_many_recordings(ktf):
    import torch
    sizes = np.random.default_rng(3).integers(0, 60, size=2000).tolist()
    layer, blocks, _, _ = plda_vectors(ktf, [sum(sizes)], seed=22)
    _within_vs_llr(layer, blocks[0], sizes)


def test_within_scores_vs_kaldi(ktf):
    import torch
    g = load_golden("plda.npz")
    rd = ktf.io.KaldiPldaReader(golden_path("plda.bin"), True)
    layer = ktf.layers.PLDA(int(g["dim"]), rd.mean, rd.transformMat, rd.psi, dtype=np.float32)
    x = np.ascontiguousarray(g["plda_input"][:, 0, :], dtype=np.float32)
    u = layer.transformVector(torch.from_numpy(x).cuda())
    kaldi = g["scores"].T                       # dense scoring orientation: S[i, j] = LLR(enrolled i | test j)
    (one,) = layer.withinScores(u, [29])
    assert rmse(kaldi, one.cpu().numpy()) <= 2e-4
    a, b = layer.withinScores(u, [10, 19])
    assert rmse(kaldi[:10, :10], a.cpu().numpy()) <= 2e-4
    assert rmse(kaldi[10:, 10:], b.cpu().numpy()) <= 2e-4


def _scores(kind, n, rng):
    if kind == "normal":
        return rng.standard_normal((n, n)).astype(np.float32)
    if kind == "integer":                      # many ties
        return rng.integers(-3, 4, size=(n, n)).astype(np.float32)
    S = rng.standard_normal((n, n)).astype(np.float32)
    if n == 0:
        return S
    flat = S.reshape(-1)
    k = max(1, n * n // 50)
    flat[rng.integers(0, n * n, size=k)] = np.nan
    flat[rng.integers(0, n * n, size=k)] = np.inf
    flat[rng.integers(0, n * n, size=k)] = -np.inf
    return S


def _check_vs_oracle(ktf, mats, **kw):
    import torch
    per = kw.get("num_speakers")
    labels, merges = ktf.diarization.agglomerative_cluster([torch.from_numpy(m).cuda() for m in mats],
                                                           return_merges=True, **kw)
    for r, S in enumerate(mats):
        n = S.shape[0]
        if per is not None:
            want_l, want_m = O.agglomerative_cluster(S, num_clusters=per if np.isscalar(per) else per[r])
        else:
            want_l, want_m = O.agglomerative_cluster(S, threshold=kw["threshold"])
        assert np.array_equal(labels[r].cpu().numpy(), want_l), (r, n)
        ids, costs = merges[r]
        ids, costs = ids.cpu().numpy(), costs.cpu().numpy()
        k = len(want_m)
        assert ids.shape == (max(n - 1, 0), 2)
        assert ids[:k].tolist() == [[m[0], m[1]] for m in want_m], (r, n)
        np.testing.assert_array_equal(costs[:k], np.array([m[2] for m in want_m], dtype=np.float32))
        assert (ids[k:] == -1).all() and np.isnan(costs[k:]).all()
        assert (want_l.max() if n else 0) == n - k


@pytest.mark.parametrize("kind", ["normal", "integer", "special"])
def test_ahc_matches_oracle(ktf, kind):
    rng = np.random.default_rng({"normal": 1, "integer": 2, "special": 3}[kind])
    sizes = [0, 1, 2, 3, 31, 32, 33, 100, 257, 600]
    mats = [_scores(kind, n, rng) for n in sizes]
    for t in (-1e30, -0.5, 0.0, 0.7, 1e30):    # nothing, some, everything
        _check_vs_oracle(ktf, mats, threshold=t)
    _check_vs_oracle(ktf, mats, num_speakers=1)
    _check_vs_oracle(ktf, mats, num_speakers=1000)              # >= n: no merge
    _check_vs_oracle(ktf, mats, num_speakers=[1, 1, 2, 1, 4, 5, 6, 3, 10, 7])


def test_ahc_matches_oracle_large(ktf):
    rng = np.random.default_rng(9)
    _check_vs_oracle(ktf, [_scores("integer", 3000, rng)], threshold=0.5)


def test_ahc_threshold_runs_are_prefixes(ktf):
    import torch
    rng = np.random.default_rng(4)
    mats = [torch.from_numpy(_scores("normal", n, rng)).cuda() for n in (50, 400, 1200)]
    _, full = ktf.diarization.agglomerative_cluster(mats, num_speakers=1, return_merges=True)
    for t in (-1.0, 0.0, 0.3, 1.0):
        _, part = ktf.diarization.agglomerative_cluster(mats, threshold=t, return_merges=True)
        for (fi, fc), (pi, pc) in zip(full, part):
            fc, pc = fc.cpu().numpy(), pc.cpu().numpy()
            stop = int(np.argmax(fc > t)) if (fc > t).any() else len(fc)
            assert np.array_equal(pi.cpu().numpy()[:stop], fi.cpu().numpy()[:stop])
            assert np.array_equal(pc[:stop], fc[:stop]) and np.isnan(pc[stop:]).all()


def test_diarization_recovers_speakers(ktf):
    import torch
    from test_gpu_tdnn_plda import synthetic_plda
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    rng = np.random.default_rng(17)
    Tinv = np.linalg.inv(Tm)
    xs, truth, sizes, speakers = [], [], [], []
    for rec, (spk, n) in enumerate([(2, 120), (3, 300), (4, 500), (1, 40)]):
        centres = rng.standard_normal((spk, DIM)) * 3.0 * np.sqrt(psi)
        who = rng.integers(0, spk, size=n)
        y = centres[who] + rng.standard_normal((n, DIM)) * 0.3
        xs.append(y @ Tinv.T + mean)           # transform(x) ~ y before length normalisation
        truth.append(who)
        sizes.append(n)
        speakers.append(spk)
    x = torch.from_numpy(np.concatenate(xs).astype(np.float32)).cuda()
    mats = layer.withinScores(layer.transformVector(x), sizes)
    for kw in ({"num_speakers": speakers}, {"threshold": 0.0}):
        labels = ktf.diarization.agglomerative_cluster(mats, **kw)
        for lab, who, spk in zip(labels, truth, speakers):
            lab = lab.cpu().numpy()
            pairs = {(int(a), int(b)) for a, b in zip(who, lab)}
            assert len(pairs) == spk and len({b for _, b in pairs}) == spk, kw


def test_argument_errors(ktf):
    import torch
    lib, N = ktf._native.lib(), ktf._native
    layer, blocks, _, (mean, Tm, psi) = plda_vectors(ktf, [8], seed=5)
    u = blocks[0]
    out = torch.empty(64, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = ctypes.c_void_p

    def offs(*v):
        return np.ascontiguousarray(v, dtype=np.int64)

    def within(h, uu, o, g, s):
        return lib.ktf_plda_score_within(h, P(uu), P(o.ctypes.data) if o is not None else P(0), g, P(s), st)
    h = layer.handle
    assert within(h, u.data_ptr(), offs(0, 8), 1, out.data_ptr()) == 0
    assert within(h, u.data_ptr(), offs(0, 5, 3), 2, out.data_ptr()) == N.KTF_EINVAL       # negative length
    assert within(h, u.data_ptr(), offs(-1, 8), 1, out.data_ptr()) == N.KTF_EINVAL
    assert within(h, u.data_ptr(), None, 1, out.data_ptr()) == N.KTF_EINVAL
    assert within(h, 0, offs(0, 8), 1, out.data_ptr()) == N.KTF_EINVAL
    assert within(h, u.data_ptr(), offs(0, 8), 1, 0) == N.KTF_EINVAL
    assert within(None, u.data_ptr(), offs(0, 8), 1, out.data_ptr()) == N.KTF_EINVAL
    f64 = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float64)
    assert within(f64.handle, u.data_ptr(), offs(0, 8), 1, out.data_ptr()) == N.KTF_EINVAL
    with pytest.raises(ValueError):
        f64.withinScores(u, [8])
    with pytest.raises(ValueError):
        layer.withinScores(u, [4, 5])

    lab = torch.empty(20000, device="cuda", dtype=torch.int32)
    cnt = torch.empty(4, device="cuda", dtype=torch.int32)
    big = N.KTF_AHC_MAX_POINTS + 1

    def ahc(o, g, s=out.data_ptr(), nc=None, labels=lab.data_ptr(), counts=cnt.data_ptr()):
        return lib.ktf_ahc_cluster(P(s), P(o.ctypes.data), g, 0.0, P(nc.ctypes.data) if nc is not None else P(0),
                                   P(labels), P(0), P(0), P(counts), st)
    assert ahc(offs(0, 8), 1) == 0
    assert ahc(offs(0, big), 1) == N.KTF_EINVAL                                         # oversize group
    assert ahc(offs(0, 5, 3), 2) == N.KTF_EINVAL                                        # negative length
    assert ahc(offs(0, 8), 1, s=0) == N.KTF_EINVAL
    assert ahc(offs(0, 8), 1, labels=0) == N.KTF_EINVAL
    assert ahc(offs(0, 8), 1, counts=0) == N.KTF_EINVAL
    assert ahc(offs(0, 8), 1, nc=np.zeros(1, dtype=np.int32)) == N.KTF_EINVAL           # num_clusters < 1
    assert lib.ktf_ahc_cluster(P(out.data_ptr()), P(0), 1, 0.0, P(0), P(lab.data_ptr()), P(0), P(0),
                               P(cnt.data_ptr()), st) == N.KTF_EINVAL                  # null offsets
    with pytest.raises(ValueError):
        ktf.diarization.agglomerative_cluster([torch.zeros(3, 3, device="cuda")], threshold=0.0, num_speakers=2)
    torch.cuda.synchronize()
