"""
One rank of the two-rank sharded AS-norm top-k test (tests/test_gpu_plda_asnorm_topk.py).  `gloo`: both ranks share
cuda:0 and gloo carries the CUDA tensors; `nccl`: every rank takes its own GPU.  Test and enrolled vectors are split
unevenly between the ranks, the cohort is replicated.  Every rank checks, against single-device results on the whole set
computed on its own device:
- kaldi_tflite_b200.parallel.plda_asnorm_best_matches_sharded equals PLDA.asNormBestMatches, bit for bit;
- the bfloat16 block of plda_asnorm_sharded(score_dtype=torch.bfloat16) equals its columns of the bfloat16 PLDA.asNorm.
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

    dim, n_test, n_enroll, n_cohort = 128, 1500, 1101, 3001
    t_split, e_split = 601, 743                        # rank 0 holds [0, split), rank 1 the rest
    mean, Tm, psi = synthetic_plda(dim)
    rng = np.random.default_rng(44)
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
    for top_n, k, counts in ((100, 10, [t_split, n_test - t_split]), (300, 32, None), (100, 1, None)):
        s, i = parallel.plda_asnorm_best_matches_sharded(layer, xt_l, xe_l, uc, top_n, k, test_counts=counts)
        ws, wi = layer.asNormBestMatches(ut_all, ue_all, uc, k=k, top_n=top_n)
        same = bool(torch.equal(s, ws) and torch.equal(i, wi))
        res[f"top{top_n}_k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum())}
        ok = ok and same
    block, _ = parallel.plda_asnorm_sharded(layer, xt_l, xe_l, uc, 300, score_dtype=torch.bfloat16)
    whole = layer.asNorm(ut_all, ue_all, uc, top_n=300, score_dtype=torch.bfloat16)
    same = block.dtype is torch.bfloat16 and bool(torch.equal(block.view(torch.int16), whole[:, e0:e1].view(torch.int16)))
    aligned = (block.stride(0) * 2) % 16 == 0
    res["bf16_block"] = {"equal": same, "pitch_aligned": aligned, "shape": list(block.shape)}
    ok = ok and same and aligned
    with open(os.path.join(out_dir, f"asnorm_topk_rank{rank}.json"), "w") as f:
        json.dump({"ok": ok, **res}, f)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1], *(sys.argv[2:3]))
