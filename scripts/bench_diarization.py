"""
Diarization back-end at scale: PLDA.withinScores and diarization.agglomerative_cluster (the full merge tree,
num_speakers=1, which is what a threshold sweep needs) against scipy's average linkage on the CPU cores, on three seeded
workloads at dim 128:
- callhome: 500 recordings of 50 .. 800 segments (the CALLHOME recipe's sub-segment counts);
- meetings: 8 recordings of 4800 segments;
- single: one recording of 16 384 segments (KTF_AHC_MAX_POINTS).

    python scripts/bench_diarization.py [--steps 3] [--warmup 1] [--out profiles/diarization_bench.json]

GPU times are event-timed ms per call after a warm-up; the launch count is that of one call.  scipy clusters the same
score matrices, copied to the host and converted to condensed cost arrays (shifted to be non-negative, which does not
change average linkage) before its clock starts, one recording per process over all CPU cores.  Records the device name
and power limit read in the same run, and checks that the GPU merge costs match scipy's heights (rtol 1e-3).
"""

import argparse
import json
import os
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import torch

from plda_bench_common import DIM, ROOT, gpu_info, ktf, synthetic_plda, time_ms

WORKLOADS = {
    "callhome": lambda rng: rng.integers(50, 801, size=500).tolist(),
    "meetings": lambda rng: [4800] * 8,
    "single": lambda rng: [16384],
}


def _scipy_linkage(cost):
    from scipy.cluster.hierarchy import linkage
    return linkage(cost, method="average")[:, 2]


def _condensed(S):
    """The condensed cost array of a score matrix, shifted to be non-negative, and the shift."""
    iu = np.triu_indices(S.shape[0], 1)
    c = -S[iu].astype(np.float64)
    shift = -min(0.0, float(c.min()) if c.size else 0.0)
    return c + shift, shift


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "diarization_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_diarization.py needs a CUDA device")
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    cores = os.cpu_count()
    result = {"device": gpu_info(), "dim": DIM, "cpu_cores": cores, "workloads": {}}
    for name in args.workloads.split(","):
        sizes = WORKLOADS[name](np.random.default_rng(7))
        g = torch.Generator(device="cuda").manual_seed(1234)
        x = torch.randn((sum(sizes), DIM), generator=g, device="cuda")
        u = layer.transformVector((x / x.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
        mats = layer.withinScores(u, sizes)
        t_within = time_ms(lambda: layer.withinScores(u, sizes), args.steps, args.warmup)
        c0 = ktf.launch_count()
        layer.withinScores(u, sizes)
        l_within = ktf.launch_count() - c0
        t_ahc = time_ms(lambda: ktf.diarization.agglomerative_cluster(mats, num_speakers=1), args.steps, args.warmup)
        c0 = ktf.launch_count()
        _, merges = ktf.diarization.agglomerative_cluster(mats, num_speakers=1, return_merges=True)
        l_ahc = ktf.launch_count() - c0
        torch.cuda.synchronize()
        host, shifts = zip(*[_condensed(m.cpu().numpy()) for m in mats])
        t0 = time.perf_counter()
        with ProcessPoolExecutor(max_workers=min(cores, len(host))) as ex:
            heights = list(ex.map(_scipy_linkage, host))
        t_scipy = (time.perf_counter() - t0) * 1e3
        worst = 0.0                 # largest relative difference of the sorted merge costs
        for (_, costs), h, shift in zip(merges, heights, shifts):
            if h.size:
                gpu = np.sort(costs.cpu().numpy().astype(np.float64)) + shift
                worst = max(worst, float(np.max(np.abs(gpu - np.sort(h)) / np.maximum(np.abs(np.sort(h)), 1.0))))
        result["workloads"][name] = {
            "recordings": len(sizes), "segments": int(sum(sizes)), "max_segments": int(max(sizes)),
            "score_elements": int(sum(n * n for n in sizes)),
            "within_scores_ms": round(t_within, 3), "within_scores_launches": int(l_within),
            "ahc_ms": round(t_ahc, 3), "ahc_launches": int(l_ahc),
            "scipy_average_linkage_ms": round(t_scipy, 1), "scipy_processes": min(cores, len(host)),
            "ahc_speedup_vs_scipy": round(t_scipy / t_ahc, 2), "max_rel_diff_merge_costs_vs_scipy": worst,
        }
        print(name, json.dumps(result["workloads"][name]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))
    bad = {k: w["max_rel_diff_merge_costs_vs_scipy"] for k, w in result["workloads"].items()
           if w["max_rel_diff_merge_costs_vs_scipy"] > 1e-3}
    assert not bad, f"GPU merge costs differ from scipy's heights: {bad}"


if __name__ == "__main__":
    main()
