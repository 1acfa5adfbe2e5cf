"""
Helpers shared by the PLDA score-form tests (test_gpu_plda_*.py, test_gpu_round2.py): the layer and vector setup, the
expected k-best lists, the comparisons, the epilogue warp-count children and the two-rank launcher of
plda_shard_worker.py.
"""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_tdnn_plda import synthetic_plda

DIM = 128


@pytest.fixture(scope="module")
def ktf():
    import kaldi_tflite_b200 as k
    return k


def plda_vectors(ktf, sizes, seed, *, cuda_rng=False):
    """A float32 layer on synthetic_plda(DIM) and one contiguous block of transformed vectors per entry of `sizes`,
    from raw vectors of norm sqrt(DIM): drawn by numpy's generator and rounded to float32, or with `cuda_rng` by torch's
    CUDA generator.  Returns (layer, blocks, x, (mean, Tm, psi)); x is the raw numpy matrix, None with `cuda_rng`."""
    import torch
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    if cuda_rng:
        g = torch.Generator(device="cuda").manual_seed(seed)
        xc = torch.randn((sum(sizes), DIM), generator=g, device="cuda")
        x, u = None, layer.transformVector((xc / xc.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
    else:
        x = np.random.default_rng(seed).standard_normal((sum(sizes), DIM))
        x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(DIM)).astype(np.float32)
        u = layer.transformVector(torch.from_numpy(x).cuda())
    offs = np.cumsum((0,) + tuple(sizes))
    return layer, [u[a:b].contiguous() for a, b in zip(offs[:-1], offs[1:])], x, (mean, Tm, psi)


def stats(layer, ut, ue, uc, top_n, num_examples=1.0):
    return (layer.cohortStats(ut, uc, top_n=top_n),
            layer.cohortStats(ue, uc, top_n=top_n, role="enrolled", num_examples=num_examples))


def _first_k(s, i, k):
    import torch
    nt, ne = s.shape
    m = min(k, ne)
    want_s = torch.full((nt, k), float("-inf"), device=s.device, dtype=torch.float32)
    want_i = torch.full((nt, k), -1, device=s.device, dtype=torch.int64)
    want_s[:, :m] = s[:, :m]
    want_i[:, :m] = i[:, :m]
    return want_s, want_i


def expected_sorted(full, k):
    """First k entries of a stable descending sort of every row, padded with (-inf, -1)."""
    import torch
    s, i = torch.sort(full, dim=1, descending=True, stable=True)
    return _first_k(s, i, k)


def listed_sort(full):
    """Stable descending sort of every row with NaN and -inf entries moved last, and the number of listed entries."""
    import torch
    dropped = torch.isnan(full) | (full == float("-inf"))
    s, i = torch.sort(full.masked_fill(dropped, float("-inf")), dim=1, descending=True, stable=True)
    return s, i, (~dropped).sum(dim=1, keepdim=True)


def expected_listed(srt, k):
    """First k of `listed_sort` (NaN and -inf entries never listed), padded with (-inf, -1) past the listed entries."""
    import torch
    s, i, kept = srt
    want_s, want_i = _first_k(s, i, k)
    pad = torch.arange(k, device=s.device)[None, :] >= kept
    want_s[pad] = float("-inf")
    want_i[pad] = -1
    return want_s, want_i


def check_equal(got, want):
    import torch
    gs, gi = got
    ws, wi = want
    assert gs.dtype is torch.float32 and gi.dtype is torch.int64 and gs.shape == ws.shape and gi.shape == wi.shape
    assert torch.equal(gi, wi), f"{int((gi != wi).sum())} of {gi.numel()} indexes differ"
    assert torch.equal(gs, ws)


_EW_PREAMBLE = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch
import kaldi_tflite_b200 as ktf
from test_gpu_tdnn_plda import synthetic_plda
mean, Tm, psi = synthetic_plda(128)
layer = ktf.layers.PLDA(128, mean, Tm, psi, dtype=np.float32, return_transformed=False)
"""


def epilogue_warp_runs(tmp_path, body):
    """Runs `body` in a child process at 8 and at 16 epilogue warps (KTF_TC_PAIR_EPI_WARPS) and returns
    {"8": arrays, "16": arrays}.  `body` is a str.format template (`{path}`: where it saves its arrays) run after
    imports of np, torch and ktf and a float32 `layer` on synthetic_plda(128)."""
    res = {}
    for ew in ("8", "16"):
        path = str(tmp_path / f"ew{ew}.npz")
        env = dict(os.environ, KTF_TC_PAIR_EPI_WARPS=ew)
        p = subprocess.run([sys.executable, "-c", (_EW_PREAMBLE + body).format(root=ROOT, path=path)], env=env,
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
        assert p.returncode == 0, p.stdout
        res[ew] = np.load(path)
    return res


_PORTS = {"llr": 29500, "topk": 31500, "asnorm": 33600, "asnorm_topk": 35700, "topk_large": 36900}


def run_two_ranks(tmp_path, scenario, *args):
    """Runs `scenario` of plda_shard_worker.py on two ranks (args: [backend] [n_test]) and returns the ranks' JSON
    results."""
    worker = os.path.join(ROOT, "tests", "plda_shard_worker.py")
    port = _PORTS[scenario] + (os.getpid() % 2000) + (7 if "nccl" in args else 0)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, worker, scenario, str(tmp_path), *args], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for rank, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {rank} failed:\n{o}"
    prefix = "" if scenario == "llr" else scenario + "_"
    results = []
    for rank in range(2):
        with open(os.path.join(str(tmp_path), f"{prefix}rank{rank}.json")) as f:
            results.append(json.load(f))
    return results
