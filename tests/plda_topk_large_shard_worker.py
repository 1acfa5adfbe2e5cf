"""
One rank of the two-rank sharded k > 32 top-k test (tests/test_gpu_plda_topk_large.py).  `gloo`: both ranks share cuda:0
and gloo carries the CUDA tensors; `nccl`: every rank takes its own GPU.  Test and enrolled vectors are split unevenly
between the ranks, the cohort is replicated.  Every rank checks, against single-device results on the whole set computed
on its own device, that kaldi_tflite_b200.parallel.plda_best_matches_large_sharded equals PLDA.bestMatchesLarge and
plda_asnorm_best_matches_large_sharded equals PLDA.asNormBestMatchesLarge, bit for bit.
"""

import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch
import torch.distributed as dist


def main(out_dir, backend="gloo"):
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=world)
    import kaldi_tflite_b200 as ktf
    from kaldi_tflite_b200 import parallel
    from test_gpu_tdnn_plda import synthetic_plda

    dim, n_test, n_enroll, n_cohort = 128, 1500, 3101, 2001
    t_split, e_split = 601, 1743                       # rank 0 holds [0, split), rank 1 the rest
    mean, Tm, psi = synthetic_plda(dim)
    rng = np.random.default_rng(45)
    x = rng.standard_normal((n_test + n_enroll + n_cohort, dim))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(dim)).astype(np.float32)
    xt, xe, xc = x[:n_test], x[n_test:n_test + n_enroll], x[n_test + n_enroll:]
    t0, t1 = (0, t_split) if rank == 0 else (t_split, n_test)
    e0, e1 = (0, e_split) if rank == 0 else (e_split, n_enroll)
    layer = ktf.layers.PLDA(dim, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    ut_all = layer.transformVector(torch.from_numpy(xt).cuda())
    ue_all = layer.transformVector(torch.from_numpy(xe).cuda())
    uc = layer.transformVector(torch.from_numpy(xc).cuda())
    xt_l, xe_l = torch.from_numpy(xt[t0:t1]).cuda(), torch.from_numpy(xe[e0:e1]).cuda()
    res = {}
    ok = True
    for k, counts in ((100, [t_split, n_test - t_split]), (1024, None), (33, None), (8, None)):
        s, i = parallel.plda_best_matches_large_sharded(layer, xt_l, xe_l, k, test_counts=counts)
        ws, wi = layer.bestMatchesLarge(ut_all, ue_all, k=k)
        same = bool(torch.equal(s, ws) and torch.equal(i, wi))
        res[f"raw_k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum())}
        ok = ok and same
        s, i = parallel.plda_asnorm_best_matches_large_sharded(layer, xt_l, xe_l, uc, 300, k, test_counts=counts)
        ws, wi = layer.asNormBestMatchesLarge(ut_all, ue_all, uc, k=k, top_n=300)
        same = bool(torch.equal(s, ws) and torch.equal(i, wi))
        res[f"asnorm_k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum())}
        ok = ok and same
    with open(os.path.join(out_dir, f"topk_large_rank{rank}.json"), "w") as f:
        json.dump({"ok": ok, **res}, f)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1], *(sys.argv[2:3]))
