"""
PLDA.bestMatches / ktf_plda_score_topk / ktf_topk_merge: the k best enrolled vectors of every test vector from the
tcgen05 score GEMM's top-k epilogue, without the score matrix.  The contract: row i equals the first k entries of a
stable descending sort of row i of the logLikelihoodRatio matrix, bit for bit, padded with (-inf, -1).
"""

import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import ktf_oracle as O
from test_gpu_tdnn_plda import synthetic_plda

pytestmark = pytest.mark.gpu

DIM = 128
KS = (1, 2, 7, 10, 16, 31, 32)


@pytest.fixture(scope="module")
def ktf():
    import kaldi_tflite_b200 as k
    return k


@pytest.fixture(scope="module")
def setup(ktf):
    """A float32 layer and transformed vectors: 1037 test rows, 4099 enrolled rows."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    rng = np.random.default_rng(2024)
    x = rng.standard_normal((1037 + 4099, DIM))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(DIM)).astype(np.float32)
    u = layer.transformVector(torch.from_numpy(x).cuda())
    return layer, u[:1037].contiguous(), u[1037:].contiguous(), x, (mean, Tm, psi)


def expected(full, k):
    """First k entries of a stable descending sort of every row, padded with (-inf, -1)."""
    import torch
    s, i = torch.sort(full, dim=1, descending=True, stable=True)
    nt, ne = full.shape
    want_s = torch.full((nt, k), float("-inf"), device=full.device, dtype=torch.float32)
    want_i = torch.full((nt, k), -1, device=full.device, dtype=torch.int64)
    m = min(k, ne)
    want_s[:, :m] = s[:, :m]
    want_i[:, :m] = i[:, :m]
    return want_s, want_i


def check_equal(got, want):
    import torch
    gs, gi = got
    ws, wi = want
    assert gs.dtype is torch.float32 and gi.dtype is torch.int64 and gs.shape == ws.shape and gi.shape == wi.shape
    assert torch.equal(gi, wi), f"{int((gi != wi).sum())} of {gi.numel()} indexes differ"
    assert torch.equal(gs, ws)


@pytest.mark.parametrize("nt", [1, 255, 257, 1037])
@pytest.mark.parametrize("ne", [1, 31, 255, 257, 700, 4099])
def test_topk_equals_stable_sort_of_score_matrix(setup, nt, ne):
    layer, ut, ue, _, _ = setup
    full = layer.logLikelihoodRatio(ut[:nt], ue[:ne])
    for k in KS:
        check_equal(layer.bestMatches(ut[:nt], ue[:ne], k=k), expected(full, k))


@pytest.mark.parametrize("k", [10, 32])
def test_topk_large_many_units_and_splits(ktf, k):
    """20 000 x 60 000: 79 row blocks x 235 n-tiles, cut into several n-ranges -- many units per cluster."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.randn((80000, DIM), generator=g, device="cuda")
    u = layer.transformVector((x / x.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
    ut, ue = u[:20000], u[20000:]
    got = layer.bestMatches(ut, ue, k=k)
    full = layer.logLikelihoodRatio(ut, ue)
    want = expected(full, k)
    del full
    check_equal(got, want)


def test_topk_against_float64_oracle(setup):
    """Every returned column's float64 score is the oracle's k-th best or within the PLDA tolerance of it."""
    layer, ut, ue, x, (mean, Tm, psi) = setup
    nt, ne = 257, 700
    uo = O.plda_transform(np.concatenate([x[:nt], x[1037:1037 + ne]]), mean, Tm, psi, dtype=np.float64)
    ref = O.plda_llr(uo, psi)[:nt, nt:]
    kth_sorted = -np.sort(-ref, axis=1)
    for k in (1, 10, 32):
        _, index = layer.bestMatches(ut[:nt], ue[:ne], k=k)
        idx = index.cpu().numpy()
        assert idx.min() >= 0 and idx.max() < ne
        assert all(len(set(r)) == k for r in idx)
        at = np.take_along_axis(ref, idx, axis=1)
        kth = kth_sorted[:, k - 1:k]
        assert np.all(kth - at <= 1e-3 * np.maximum(np.abs(kth), 1.0))


@pytest.mark.parametrize("num_examples", [1.0, 3.0])
def test_k1_equals_best_match(setup, num_examples):
    layer, ut, ue, _, _ = setup
    s, i = layer.bestMatches(ut, ue, k=1, num_examples=num_examples)
    bs, bi = layer.bestMatch(ut, ue, num_examples=num_examples)
    check_equal((s, i), (bs[:, None], bi[:, None]))
    s, i = layer.bestMatches(ut, k=1, num_examples=num_examples)
    bs, bi = layer.bestMatch(ut, num_examples=num_examples)
    check_equal((s, i), (bs[:, None], bi[:, None]))


def test_ties_come_back_lowest_column_first(setup):
    """One enrolled vector copied to columns in different column quarters, n-tiles and n-ranges; the test rows include
    that vector itself, so the copies tie near the top of its row."""
    import torch
    layer, ut, ue, _, _ = setup
    cols = [5, 200, 300, 1000, 2100, 3333, 4000]
    ue2 = ue.clone()
    ue2[cols] = ue[cols[0]]
    ut2 = torch.cat([ue[cols[0]:cols[0] + 1], ut[:300]]).contiguous()
    full = layer.logLikelihoodRatio(ut2, ue2)
    row = full[0, cols]
    assert torch.equal(row, row[:1].expand(len(cols))), "copies of one vector must score equal"
    for k in (7, 16, 32):
        got = layer.bestMatches(ut2, ue2, k=k)
        check_equal(got, expected(full, k))
    s, i = layer.bestMatches(ut2, ue2, k=32)
    tied = [int(c) for c, v in zip(i[0].tolist(), s[0].tolist()) if v == float(row[0])]
    assert tied == cols


def test_edges(setup, ktf):
    import torch
    from kaldi_tflite_b200 import _native as N
    layer, ut, ue, _, _ = setup
    # fewer enrolled vectors than k: (-inf, -1) after the last one
    s, i = layer.bestMatches(ut[:40], ue[:5], k=9)
    check_equal((s, i), expected(layer.logLikelihoodRatio(ut[:40], ue[:5]), 9))
    assert bool((i[:, 5:] == -1).all()) and bool(torch.isinf(s[:, 5:]).all()) and float(s[:, 5:].max()) < 0
    # no enrolled vector at all
    s, i = layer.bestMatches(ut[:33], ue[:0], k=4)
    assert s.shape == (33, 4) and bool((i == -1).all()) and bool((s == float("-inf")).all())
    # no test vector: nothing to do
    s, i = layer.bestMatches(ut[:0], ue, k=4)
    assert s.shape == (0, 4) and i.shape == (0, 4)
    # k outside 1 .. 32
    for k in (0, 33):
        with pytest.raises(ValueError, match="32"):
            layer.bestMatches(ut[:10], ue[:10], k=k)
    out_s = torch.empty((10, 33), device="cuda")
    out_i = torch.empty((10, 33), device="cuda", dtype=torch.int64)
    rc = N.lib().ktf_plda_score_topk(layer.handle, ctypes.c_void_p(ut.data_ptr()), 10, ctypes.c_void_p(ue.data_ptr()),
                                     10, 33, ctypes.c_void_p(out_s.data_ptr()), ctypes.c_void_p(out_i.data_ptr()), None)
    assert rc == N.KTF_EINVAL and "32" in N.last_error()
    # float64 layers have no tcgen05 score path
    mean, Tm, psi = synthetic_plda(DIM)
    with pytest.raises(ValueError):
        ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float64).bestMatches(ut.double(), k=3)


_EW_CHILD = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch
import kaldi_tflite_b200 as ktf
from test_gpu_tdnn_plda import synthetic_plda
mean, Tm, psi = synthetic_plda(128)
layer = ktf.layers.PLDA(128, mean, Tm, psi, dtype=np.float32, return_transformed=False)
rng = np.random.default_rng(5)
x = rng.standard_normal((1037 + 4099, 128)).astype(np.float32)
u = layer.transformVector(torch.from_numpy(x).cuda())
out = {{}}
for k in (1, 7, 16, 32):
    s, i = layer.bestMatches(u[:1037].contiguous(), u[1037:].contiguous(), k=k)
    out[f"s{{k}}"], out[f"i{{k}}"] = s.cpu().numpy(), i.cpu().numpy()
np.savez({path!r}, **out)
"""


def test_independent_of_epilogue_warp_count(tmp_path):
    res = {}
    for ew in ("8", "16"):
        path = str(tmp_path / f"ew{ew}.npz")
        env = dict(os.environ, KTF_TC_PAIR_EPI_WARPS=ew)
        p = subprocess.run([sys.executable, "-c", _EW_CHILD.format(root=ROOT, path=path)], env=env,
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
        assert p.returncode == 0, p.stdout
        res[ew] = np.load(path)
    for key in res["8"].files:
        assert np.array_equal(res["8"][key], res["16"][key]), key


def test_cuda_graph_capture_and_replay(setup):
    import torch
    layer, ut, ue, _, _ = setup
    st, se = ut[:700].clone(), ue[:1500].clone()
    layer.bestMatches(st, se, k=10)                      # grows the workspace for this shape
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        gs, gi = layer.bestMatches(st, se, k=10)
    st.copy_(ut[300:1000])
    se.copy_(ue[2000:3500])
    g.replay()
    torch.cuda.synchronize()
    check_equal((gs, gi), layer.bestMatches(ut[300:1000].contiguous(), ue[2000:3500].contiguous(), k=10))


def _run_topk_shard_workers(tmp_path, backend):
    worker = os.path.join(ROOT, "tests", "plda_topk_shard_worker.py")
    port = 31500 + (os.getpid() % 2000) + (7 if backend == "nccl" else 0)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, worker, str(tmp_path), backend], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for rank, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {rank} failed:\n{o}"
    for rank in range(2):
        with open(os.path.join(str(tmp_path), f"topk_rank{rank}.json")) as f:
            r = json.load(f)
        assert r["ok"], r


def test_sharded_two_ranks_gloo(tmp_path):
    _run_topk_shard_workers(tmp_path, "gloo")


def test_sharded_two_gpus_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _run_topk_shard_workers(tmp_path, "nccl")


def _numpy_merge(s_in, i_in, k):
    L, n, _ = s_in.shape
    out_s = np.full((n, k), -np.inf, np.float32)
    out_i = np.full((n, k), -1, np.int64)
    for r in range(n):
        s, i = s_in[:, r].ravel(), i_in[:, r].ravel()
        keep = i >= 0
        s, i = s[keep], i[keep]
        order = np.lexsort((i, -s.astype(np.float64)))[:k]
        out_s[r, :len(order)] = s[order]
        out_i[r, :len(order)] = i[order]
    return out_s, out_i


def test_topk_merge_against_numpy(ktf):
    import torch
    from kaldi_tflite_b200 import _native as N
    rng = np.random.default_rng(11)
    L, n, k_in = 5, 300, 12
    s_in = rng.choice(np.float32([-3.5, -1.0, 0.25, 2.0, 7.5]), size=(L, n, k_in)).astype(np.float32)   # many ties
    s_in += rng.integers(0, 2, size=s_in.shape).astype(np.float32) * np.float32(1e-3)
    i_in = np.stack([rng.permutation(L * k_in * 3)[:L * k_in].reshape(L, k_in) for _ in range(n)], axis=1)
    i_in[rng.random(i_in.shape) < 0.2] = -1                                                         # empty entries
    i_in[:, :7] = -1                                                                                 # rows with nothing
    ds, di = torch.from_numpy(s_in).cuda(), torch.from_numpy(i_in.astype(np.int64)).cuda()
    for k in (1, 10, 32):
        os_, oi = torch.empty((n, k), device="cuda"), torch.empty((n, k), device="cuda", dtype=torch.int64)
        N.check(N.lib().ktf_topk_merge(ctypes.c_void_p(ds.data_ptr()), ctypes.c_void_p(di.data_ptr()), L, n, k_in, k,
                                       ctypes.c_void_p(os_.data_ptr()), ctypes.c_void_p(oi.data_ptr()), None))
        torch.cuda.synchronize()
        ws, wi = _numpy_merge(s_in, i_in, k)
        assert np.array_equal(oi.cpu().numpy(), wi)
        assert np.array_equal(os_.cpu().numpy(), ws)
    with pytest.raises(ValueError, match="32"):
        N.check(N.lib().ktf_topk_merge(ctypes.c_void_p(ds.data_ptr()), ctypes.c_void_p(di.data_ptr()), L, n, k_in, 33,
                                       ctypes.c_void_p(os_.data_ptr()), ctypes.c_void_p(oi.data_ptr()), None))
