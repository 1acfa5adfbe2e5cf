"""
AS-norm at scale: PLDA.cohortStats (both sides) and PLDA.asNorm with precomputed statistics (normalised in the score
kernel's epilogue) against PLDA.logLikelihoodRatio in the same run, and against what a user would otherwise write --
the fp32 cohort matrices, torch.topk and an elementwise normalisation of the raw score matrix.

    python scripts/bench_plda_asnorm.py [--n 50000] [--cohort 10000] [--steps 10] [--warmup 2]
                                        [--out profiles/plda_asnorm_bench.json]

Event-timed ms per call after warm-up.  Records the device name and power limit read in the same run, and checks a
sampled sub-block against the contract of tests/test_gpu_plda_asnorm.py: statistics within 1 float32 ulp of the
float64 statistics of the exact top_n (from a sort of the fp32 cohort scores), normalised scores within
2e-6 max(|s'|, 1) of the float64 formula applied to the fp32 logLikelihoodRatio entries.
"""

import argparse
import json
import os

import numpy as np
import torch

from plda_bench_common import DIM, ROOT, gpu_info, plda_setup, time_ms
TOP_NS = (100, 300, 1000)


def within_ulp(got, want64):
    wf = want64.float().abs()
    ulp = torch.nextafter(wf, torch.full_like(wf, float("inf"))) - wf
    return bool(((got.double() - want64).abs() <= ulp.double()).all())


def stats_ok(got, scores, top_n):
    top = torch.sort(scores, dim=1, descending=True).values[:, :top_n].double()
    return within_ulp(got[0], top.mean(dim=1)) and within_ulp(got[1], top.std(dim=1, unbiased=False))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--cohort", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plda_asnorm_bench.json"))
    args = ap.parse_args()
    n, nc = args.n, args.cohort
    layer, ut, ue, uc = plda_setup("bench_plda_asnorm.py", n, nc)
    raw = torch.empty((n, n), device="cuda", dtype=torch.float32)
    normed = torch.empty((n, n), device="cuda", dtype=torch.float32)

    result = {"device": gpu_info(), "n_test": n, "n_enroll": n, "n_cohort": nc, "dim": DIM, "steps": args.steps,
              "warmup": args.warmup}
    result["llr_matrix_ms"] = time_ms(lambda: layer.logLikelihoodRatio(ut, ue, out=raw), args.steps, args.warmup)
    rows = torch.from_numpy(np.sort(np.random.default_rng(3).choice(n, size=256, replace=False))).cuda()
    for top_n in TOP_NS:
        r = {}
        r["test_stats_ms"] = time_ms(lambda: layer.cohortStats(ut, uc, top_n=top_n), args.steps, args.warmup)
        r["enroll_stats_ms"] = time_ms(lambda: layer.cohortStats(ue, uc, top_n=top_n, role="enrolled"), args.steps,
                                       args.warmup)
        ts = layer.cohortStats(ut, uc, top_n=top_n)
        es = layer.cohortStats(ue, uc, top_n=top_n, role="enrolled")
        r["asnorm_ms"] = time_ms(lambda: layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=normed), args.steps,
                                 args.warmup)
        r["llr_matrix_ms"] = time_ms(lambda: layer.logLikelihoodRatio(ut, ue, out=raw), args.steps, args.warmup)
        r["asnorm_over_llr"] = r["asnorm_ms"] / r["llr_matrix_ms"]

        def torch_stats():
            ct = layer.logLikelihoodRatio(ut, uc)
            ce = layer.logLikelihoodRatio(uc, ue)
            vt = torch.topk(ct, top_n, dim=1).values.double()
            ve = torch.topk(ce, top_n, dim=0).values.double()
            return (vt.mean(dim=1).float(), vt.std(dim=1, unbiased=False).float(),
                    ve.mean(dim=0).float(), ve.std(dim=0, unbiased=False).float())

        def torch_route():
            mt, st, me, se = torch_stats()
            layer.logLikelihoodRatio(ut, ue, out=raw)
            return 0.5 * ((raw - me[None, :]) / se[None, :] + (raw - mt[:, None]) / st[:, None])

        r["torch_stats_ms"] = time_ms(torch_stats, args.steps, args.warmup)
        r["torch_route_ms"] = time_ms(torch_route, max(2, args.steps // 2), 1)
        r["stats_speedup_vs_torch"] = r["torch_stats_ms"] / (r["test_stats_ms"] + r["enroll_stats_ms"])
        r["route_speedup_vs_torch"] = r["torch_route_ms"] / (r["test_stats_ms"] + r["enroll_stats_ms"] + r["asnorm_ms"])

        # sampled contract check: 256 test rows and 256 enrolled columns
        layer.asNorm(ut, ue, test_stats=ts, enroll_stats=es, out=normed)
        layer.logLikelihoodRatio(ut, ue, out=raw)
        s = raw[rows].double()
        want = 0.5 * ((s - es[0].double()[None, :]) / es[1].double()[None, :] +
                      (s - ts[0][rows].double()[:, None]) / ts[1][rows].double()[:, None])
        err = (normed[rows].double() - want).abs() / (2e-6 * want.abs().clamp(min=1.0))
        r["sample_asnorm_worst_over_tol"] = float(err.max())
        r["sample_stats_within_1ulp"] = (
            stats_ok((ts[0][rows], ts[1][rows]), layer.logLikelihoodRatio(ut[rows].contiguous(), uc), top_n) and
            stats_ok((es[0][rows], es[1][rows]), layer.logLikelihoodRatio(uc, ue[rows].contiguous()).t(), top_n))
        r["sample_ok"] = r["sample_stats_within_1ulp"] and r["sample_asnorm_worst_over_tol"] <= 1.0
        result[f"top{top_n}"] = r
        torch.cuda.empty_cache()
    result["bytes_written_matrix"] = 4.0 * n * n
    result["asnorm_top300_write_GBps"] = result["bytes_written_matrix"] / (result["top300"]["asnorm_ms"] * 1e-3) / 1e9
    print(json.dumps(result), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
