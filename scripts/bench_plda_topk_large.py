"""
k > 32 best trials per test vector at scale: PLDA.bestMatchesLarge / asNormBestMatchesLarge (score or AS-norm row
chunks selected in L2, no score matrix) against what a user would otherwise write -- the float32 logLikelihoodRatio /
asNorm matrix followed by torch.topk -- on the same transformed vectors, and bestMatches at k = 32, where the path
changes.

    python scripts/bench_plda_topk_large.py [--n 50000] [--steps 5] [--warmup 2] [--out profiles/plda_topk_large_bench.json]

Event-timed ms per call (warm-up first).  AS-norm statistics (cohort 10 000, top_n 300) are computed once and passed to
both sides, so both time the normalised scoring alone.  Records the device name and power limit read in the same run,
and checks every k against the stable sort of the float32 matrix on a sample of rows.
"""

import argparse
import json
import os

import numpy as np
import torch

from plda_bench_common import DIM, ROOT, gpu_info, plda_setup, time_ms
KS = (33, 64, 100, 256, 1024)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--cohort", type=int, default=10000)
    ap.add_argument("--top-n", type=int, default=300)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plda_topk_large_bench.json"))
    args = ap.parse_args()
    n = args.n
    layer, ut, ue, uc = plda_setup("bench_plda_topk_large.py", n, args.cohort)
    ts = layer.cohortStats(ut, uc, top_n=args.top_n)
    es = layer.cohortStats(ue, uc, top_n=args.top_n, role="enrolled")
    st = (args.steps, args.warmup)

    result = {"device": gpu_info(), "n_test": n, "n_enroll": n, "dim": DIM, "cohort": args.cohort, "top_n": args.top_n,
              "steps": args.steps, "warmup": args.warmup}
    result["best_matches_k32_ms"] = time_ms(lambda: layer.bestMatches(ut, ue, k=32), *st)
    result["asnorm_best_matches_k32_ms"] = time_ms(
        lambda: layer.asNormBestMatches(ut, ue, k=32, test_stats=ts, enroll_stats=es), *st)
    for k in KS:
        result[f"large_k{k}_ms"] = time_ms(lambda: layer.bestMatchesLarge(ut, ue, k=k), *st)
        result[f"asnorm_large_k{k}_ms"] = time_ms(
            lambda: layer.asNormBestMatchesLarge(ut, ue, k=k, test_stats=ts, enroll_stats=es), *st)
    full = torch.empty((n, n), device="cuda", dtype=torch.float32)
    result["matrix_ms"] = time_ms(lambda: layer.logLikelihoodRatio(ut, ue, out=full), *st)
    result["asnorm_matrix_ms"] = time_ms(lambda: layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=full), *st)
    for k in KS:
        def raw():
            layer.logLikelihoodRatio(ut, ue, out=full)
            return torch.topk(full, k, dim=1)

        def norm():
            layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=full)
            return torch.topk(full, k, dim=1)
        result[f"matrix_topk_k{k}_ms"] = time_ms(raw, *st)
        result[f"asnorm_matrix_topk_k{k}_ms"] = time_ms(norm, *st)
        result[f"speedup_k{k}"] = result[f"matrix_topk_k{k}_ms"] / result[f"large_k{k}_ms"]
        result[f"asnorm_speedup_k{k}"] = result[f"asnorm_matrix_topk_k{k}_ms"] / result[f"asnorm_large_k{k}_ms"]
    del full

    # parity on a sample of rows: the first k of a stable descending sort of the fp32 matrix, bit for bit
    rows = torch.from_numpy(np.sort(np.random.default_rng(3).choice(n, size=256, replace=False))).cuda()
    fulls = {"raw": layer.logLikelihoodRatio(ut[rows].contiguous(), ue),
             "asnorm": layer.asNorm(ut[rows].contiguous(), ue, test_stats=(ts[0][rows].contiguous(),
                                                                           ts[1][rows].contiguous()), enroll_stats=es)}
    for name, f in fulls.items():
        s_sorted, i_sorted = torch.sort(f, dim=1, descending=True, stable=True)
        for k in KS:
            s, i = (layer.bestMatchesLarge(ut, ue, k=k) if name == "raw" else
                    layer.asNormBestMatchesLarge(ut, ue, k=k, test_stats=ts, enroll_stats=es))
            result[f"parity_{name}_k{k}_bit_equal"] = bool(torch.equal(s[rows], s_sorted[:, :k])
                                                          and torch.equal(i[rows], i_sorted[:, :k]))
    print(json.dumps(result), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
