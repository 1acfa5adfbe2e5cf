"""
Normalised top-k at scale: PLDA.asNormBestMatches (the k best enrolled vectors by AS-norm score, selected in the score
kernel's epilogue) against PLDA.bestMatches (raw scores) at the same k, PLDA.asNorm as float32 and as bfloat16, and the
route asNormBestMatches replaces -- the float32 asNorm matrix followed by torch.topk -- all in one run, with
precomputed cohort statistics.

    python scripts/bench_plda_asnorm_topk.py [--n 50000] [--cohort 10000] [--top-n 300] [--steps 10] [--warmup 2]
                                             [--out profiles/plda_asnorm_topk_bench.json]

Event-timed ms per call after warm-up.  Records the device name and power limit read in the same run, and checks 256
sampled test rows against the contracts of tests/test_gpu_plda_asnorm_topk.py: the lists bit-equal to the first k of a
stable descending sort of the float32 asNorm row (NaN and -inf left out), the bfloat16 matrix bit-equal to the float32
one rounded to bfloat16.
"""

import argparse
import json
import os

import numpy as np
import torch

from plda_bench_common import DIM, ROOT, gpu_info, plda_setup, time_ms
KS = (1, 10, 32)


def expected(full, k):
    """First k of a stable descending sort of every row without NaN and -inf, padded with (-inf, -1)."""
    dropped = torch.isnan(full) | (full == float("-inf"))
    s, i = torch.sort(full.masked_fill(dropped, float("-inf")), dim=1, descending=True, stable=True)
    s, i = s[:, :k].clone(), i[:, :k].clone()
    pad = torch.arange(k, device=full.device)[None, :] >= (~dropped).sum(dim=1, keepdim=True)
    s[pad] = float("-inf")
    i[pad] = -1
    return s, i


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--cohort", type=int, default=10000)
    ap.add_argument("--top-n", type=int, default=300)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plda_asnorm_topk_bench.json"))
    args = ap.parse_args()
    n, nc, top_n = args.n, args.cohort, args.top_n
    layer, ut, ue, uc = plda_setup("bench_plda_asnorm_topk.py", n, nc)
    ts = layer.cohortStats(ut, uc, top_n=top_n)
    es = layer.cohortStats(ue, uc, top_n=top_n, role="enrolled")
    normed = torch.empty((n, n), device="cuda", dtype=torch.float32)
    normed16 = torch.empty((n, n), device="cuda", dtype=torch.bfloat16)

    result = {"device": gpu_info(), "n_test": n, "n_enroll": n, "n_cohort": nc, "top_n": top_n, "dim": DIM,
              "steps": args.steps, "warmup": args.warmup}
    result["asnorm_f32_ms"] = time_ms(lambda: layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=normed),
                                      args.steps, args.warmup)
    result["asnorm_bf16_ms"] = time_ms(lambda: layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=normed16),
                                       args.steps, args.warmup)
    result["asnorm_bf16_over_f32"] = result["asnorm_bf16_ms"] / result["asnorm_f32_ms"]
    for k in KS:
        r = {}
        r["asnorm_best_matches_ms"] = time_ms(
            lambda: layer.asNormBestMatches(ut, ue, k=k, test_stats=ts, enroll_stats=es), args.steps, args.warmup)
        r["best_matches_ms"] = time_ms(lambda: layer.bestMatches(ut, ue, k=k), args.steps, args.warmup)

        def matrix_route():
            layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=normed)
            return torch.topk(normed, k, dim=1)

        r["asnorm_matrix_plus_topk_ms"] = time_ms(matrix_route, max(2, args.steps // 2), 1)
        r["over_best_matches"] = r["asnorm_best_matches_ms"] / r["best_matches_ms"]
        r["speedup_vs_matrix_route"] = r["asnorm_matrix_plus_topk_ms"] / r["asnorm_best_matches_ms"]
        result[f"k{k}"] = r

    # sampled contract checks: 256 test rows
    rows = torch.from_numpy(np.sort(np.random.default_rng(3).choice(n, size=256, replace=False))).cuda()
    layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=normed)
    layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=normed16)
    sample = normed[rows]
    ok_lists = True
    for k in KS:
        s, i = layer.asNormBestMatches(ut[rows].contiguous(), ue, k=k, test_stats=(ts[0][rows], ts[1][rows]),
                                       enroll_stats=es)
        ws, wi = expected(sample, k)
        ok_lists = ok_lists and bool(torch.equal(s, ws) and torch.equal(i, wi))
    result["sample_lists_bit_equal"] = ok_lists
    result["sample_bf16_bit_equal"] = bool(torch.equal(normed16[rows].view(torch.int16),
                                                       sample.to(torch.bfloat16).view(torch.int16)))
    result["sample_ok"] = result["sample_lists_bit_equal"] and result["sample_bf16_bit_equal"]
    print(json.dumps(result), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
