"""
One rank of a two-rank sharded PLDA test: `plda_shard_worker.py <scenario> <out_dir> [backend] [n_test]`.  `gloo`
(default): both ranks share cuda:0 (NCCL refuses two ranks on one device, so gloo carries the CUDA tensors of the
exchange); `nccl`: every rank takes its own GPU and the exchange is the asynchronous NCCL all-gather.  Every rank writes
its results, with "ok", to <out_dir>/<scenario>_rank<r>.json (llr: rank<r>.json).  Scenarios:
- llr (test_gpu_round2.py): parallel.plda_score_sharded on shards from shard_range (n_test test vectors, default 1500:
  an odd count makes the shards ragged); each rank checks its (n_test x n_enroll / G) block against the float64 oracle,
  |delta| <= 1e-3 * max(|s|, 1).
In the others the test and enrolled vectors are split unevenly between the ranks and the cohort is replicated; every rank
checks the sharded result against the single-device one on the whole set, computed on its own device, bit for bit:
- topk (test_gpu_plda_topk.py): plda_best_matches_sharded against PLDA.bestMatches;
- asnorm (test_gpu_plda_asnorm.py): the plda_asnorm_sharded block against its columns of PLDA.asNorm;
- asnorm_topk (test_gpu_plda_asnorm_topk.py): plda_asnorm_best_matches_sharded against PLDA.asNormBestMatches, and the
  bfloat16 block of plda_asnorm_sharded(score_dtype=torch.bfloat16) against its columns of the bfloat16 PLDA.asNorm;
- topk_large (test_gpu_plda_topk_large.py): plda_best_matches_large_sharded against PLDA.bestMatchesLarge and
  plda_asnorm_best_matches_large_sharded against PLDA.asNormBestMatchesLarge.
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

# scenario: (seed, n_enroll, n_cohort, test split, enrolled split); rank 0 holds [0, split), rank 1 the rest
SETS = {
    "llr": (31, 1100, 0, None, None),               # ragged against the 128 x 256 tiles and against the ranks
    "topk": (41, 1100, 0, 601, 743),
    "asnorm": (43, 1101, 3001, 601, 743),
    "asnorm_topk": (44, 1101, 3001, 601, 743),
    "topk_large": (45, 3101, 2001, 601, 1743),
}


def llr(ktf, parallel, layer, x, plda, n_test, rank, world):
    from oracle import ktf_oracle as O
    mean, Tm, psi = plda
    n_enroll = x.shape[0] - n_test
    xt, xe = x[:n_test], x[n_test:]
    t0, t1 = parallel.shard_range(n_test, rank, world)
    e0, e1 = parallel.shard_range(n_enroll, rank, world)
    counts = [parallel.shard_range(n_test, r, world)[1] - parallel.shard_range(n_test, r, world)[0] for r in range(world)]
    n0 = ktf.launch_count()
    scores, u_all = parallel.plda_score_sharded(layer, torch.from_numpy(xt[t0:t1]).cuda(),
                                                torch.from_numpy(xe[e0:e1]).cuda(), test_counts=counts)
    torch.cuda.synchronize()
    launches = ktf.launch_count() - n0
    got = scores.cpu().numpy()

    uo = O.plda_transform(x, mean, Tm, psi, dtype=np.float64)
    want = O.plda_llr(uo, psi)[:n_test, n_test + e0:n_test + e1]
    ok = got.shape == want.shape
    rel = float(np.max(np.abs(got - want) / np.maximum(np.abs(want), 1.0))) if ok else float("inf")
    gathered_ok = bool(np.allclose(u_all.cpu().numpy(), uo[:n_test], atol=1e-4))
    return {"ok": bool(ok and gathered_ok), "max_rel": rel, "launches": int(launches), "shape": list(got.shape)}


def topk(parallel, layer, v):
    res, ok = {}, True
    for k, counts in ((10, v["counts"]), (32, None), (1, None)):
        s, i = parallel.plda_best_matches_sharded(layer, v["xt_l"], v["xe_l"], k, test_counts=counts)
        ws, wi = layer.bestMatches(v["ut"], v["ue"], k=k)
        same = bool(torch.equal(i, wi) and torch.equal(s, ws))
        res[f"k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum()), "shape": list(s.shape)}
        ok = ok and same
    return {"ok": ok, **res}


def asnorm(parallel, layer, v):
    res, ok = {}, True
    e0, e1 = v["e"]
    for top_n, counts in ((100, v["counts"]), (1000, None)):
        block, _ = parallel.plda_asnorm_sharded(layer, v["xt_l"], v["xe_l"], v["uc"], top_n, test_counts=counts)
        whole = layer.asNorm(v["ut"], v["ue"], v["uc"], top_n=top_n)
        same = bool(torch.equal(block, whole[:, e0:e1]))
        aligned = (block.stride(0) * 4) % 16 == 0
        res[f"top{top_n}"] = {"equal": same, "pitch_aligned": aligned, "shape": list(block.shape),
                              "mismatches": int((block != whole[:, e0:e1]).sum())}
        ok = ok and same and aligned
    return {"ok": ok, **res}


def asnorm_topk(parallel, layer, v):
    res, ok = {}, True
    e0, e1 = v["e"]
    for top_n, k, counts in ((100, 10, v["counts"]), (300, 32, None), (100, 1, None)):
        s, i = parallel.plda_asnorm_best_matches_sharded(layer, v["xt_l"], v["xe_l"], v["uc"], top_n, k,
                                                         test_counts=counts)
        ws, wi = layer.asNormBestMatches(v["ut"], v["ue"], v["uc"], k=k, top_n=top_n)
        same = bool(torch.equal(s, ws) and torch.equal(i, wi))
        res[f"top{top_n}_k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum())}
        ok = ok and same
    block, _ = parallel.plda_asnorm_sharded(layer, v["xt_l"], v["xe_l"], v["uc"], 300, score_dtype=torch.bfloat16)
    whole = layer.asNorm(v["ut"], v["ue"], v["uc"], top_n=300, score_dtype=torch.bfloat16)
    same = block.dtype is torch.bfloat16 and bool(torch.equal(block.view(torch.int16), whole[:, e0:e1].view(torch.int16)))
    aligned = (block.stride(0) * 2) % 16 == 0
    res["bf16_block"] = {"equal": same, "pitch_aligned": aligned, "shape": list(block.shape)}
    return {"ok": ok and same and aligned, **res}


def topk_large(parallel, layer, v):
    res, ok = {}, True
    for k, counts in ((100, v["counts"]), (1024, None), (33, None), (8, None)):
        s, i = parallel.plda_best_matches_large_sharded(layer, v["xt_l"], v["xe_l"], k, test_counts=counts)
        ws, wi = layer.bestMatchesLarge(v["ut"], v["ue"], k=k)
        same = bool(torch.equal(s, ws) and torch.equal(i, wi))
        res[f"raw_k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum())}
        ok = ok and same
        s, i = parallel.plda_asnorm_best_matches_large_sharded(layer, v["xt_l"], v["xe_l"], v["uc"], 300, k,
                                                               test_counts=counts)
        ws, wi = layer.asNormBestMatchesLarge(v["ut"], v["ue"], v["uc"], k=k, top_n=300)
        same = bool(torch.equal(s, ws) and torch.equal(i, wi))
        res[f"asnorm_k{k}"] = {"equal": same, "index_mismatches": int((i != wi).sum())}
        ok = ok and same
    return {"ok": ok, **res}


def main(scenario, out_dir, backend="gloo", n_test=1500):
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, rank=rank, world_size=world)
    import kaldi_tflite_b200 as ktf
    from kaldi_tflite_b200 import parallel
    from test_gpu_tdnn_plda import synthetic_plda

    dim = 128
    seed, n_enroll, n_cohort, t_split, e_split = SETS[scenario]
    mean, Tm, psi = synthetic_plda(dim)
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n_test + n_enroll + n_cohort, dim))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(dim)).astype(np.float32)
    layer = ktf.layers.PLDA(dim, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    if scenario == "llr":
        result = llr(ktf, parallel, layer, x, (mean, Tm, psi), n_test, rank, world)
    else:
        xt, xe, xc = x[:n_test], x[n_test:n_test + n_enroll], x[n_test + n_enroll:]
        t0, t1 = (0, t_split) if rank == 0 else (t_split, n_test)
        e0, e1 = (0, e_split) if rank == 0 else (e_split, n_enroll)
        v = {"e": (e0, e1), "counts": [t_split, n_test - t_split],
             "xt_l": torch.from_numpy(xt[t0:t1]).cuda(), "xe_l": torch.from_numpy(xe[e0:e1]).cuda(),
             "ut": layer.transformVector(torch.from_numpy(xt).cuda()),
             "ue": layer.transformVector(torch.from_numpy(xe).cuda()),
             "uc": layer.transformVector(torch.from_numpy(xc).cuda()) if n_cohort else None}
        result = {"topk": topk, "asnorm": asnorm, "asnorm_topk": asnorm_topk, "topk_large": topk_large}[scenario](
            parallel, layer, v)
    prefix = "" if scenario == "llr" else scenario + "_"
    with open(os.path.join(out_dir, f"{prefix}rank{rank}.json"), "w") as f:
        json.dump(result, f)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2], *(sys.argv[3:4]), *(int(a) for a in sys.argv[4:5]))
