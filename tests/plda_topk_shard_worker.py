"""
One rank of the two-rank sharded k-best test (tests/test_gpu_plda_topk.py).  `gloo`: both ranks share cuda:0 and gloo
carries the CUDA tensors; `nccl`: every rank takes its own GPU.  Test and enrolled vectors are split unevenly between
the ranks; every rank runs kaldi_tflite_b200.parallel.plda_best_matches_sharded and checks that the merged lists equal
PLDA.bestMatches of the whole set computed on its own device.
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

    dim, n_test, n_enroll = 128, 1500, 1100
    t_split, e_split = 601, 743                        # rank 0 holds [0, split), rank 1 the rest
    mean, Tm, psi = synthetic_plda(dim)
    rng = np.random.default_rng(41)
    x = rng.standard_normal((n_test + n_enroll, dim))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(dim)).astype(np.float32)
    xt, xe = x[:n_test], x[n_test:]
    t0, t1 = (0, t_split) if rank == 0 else (t_split, n_test)
    e0, e1 = (0, e_split) if rank == 0 else (e_split, n_enroll)
    layer = ktf.layers.PLDA(dim, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    ut_all = layer.transformVector(torch.from_numpy(xt).cuda())
    ue_all = layer.transformVector(torch.from_numpy(xe).cuda())
    res = {}
    ok = True
    for k, counts in ((10, [t_split, n_test - t_split]), (32, None), (1, None)):
        s, i = parallel.plda_best_matches_sharded(layer, torch.from_numpy(xt[t0:t1]).cuda(),
                                                  torch.from_numpy(xe[e0:e1]).cuda(), k, test_counts=counts)
        ws, wi = layer.bestMatches(ut_all, ue_all, k=k)
        same = bool(torch.equal(i, wi) and torch.equal(s, ws))
        res[f"k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum()), "shape": list(s.shape)}
        ok = ok and same
    with open(os.path.join(out_dir, f"topk_rank{rank}.json"), "w") as f:
        json.dump({"ok": ok, **res}, f)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1], *(sys.argv[2:3]))
