"""
k best trials per test vector at scale: PLDA.bestMatches (tcgen05 score GEMM with the top-k epilogue, no score matrix)
against PLDA.bestMatch (k = 1) and against what a user would otherwise write -- the bfloat16 score matrix followed by
torch.topk -- on the same transformed vectors.

    python scripts/bench_plda_topk.py [--n 50000] [--steps 20] [--warmup 3] [--out profiles/plda_topk_bench.json]

Event-timed ms per call (warm-up first; the operands, 2 x 38 MB of fp16 hi/lo splits, fit in L2, as they do in every
real call).  Records the device name and power limit read in the same run, and checks bestMatches against the stable
sort of the fp32 score matrix on a sample of rows.
"""

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import kaldi_tflite_b200 as ktf                     # noqa: E402
from test_gpu_tdnn_plda import synthetic_plda       # noqa: E402

DIM = 128


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:   # still record the torch device name
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


def time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=50000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plda_topk_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_plda_topk.py needs a CUDA device")
    n = args.n
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    g = torch.Generator(device="cuda").manual_seed(1234)
    x = torch.randn((2 * n, DIM), generator=g, device="cuda")
    u = layer.transformVector((x / x.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
    ut, ue = u[:n].contiguous(), u[n:].contiguous()
    scores16 = torch.empty((n, n), device="cuda", dtype=torch.bfloat16)

    result = {"device": gpu_info(), "n_test": n, "n_enroll": n, "dim": DIM, "steps": args.steps, "warmup": args.warmup}
    result["best_match_ms"] = time_ms(lambda: layer.bestMatch(ut, ue), args.steps, args.warmup)
    for k in (1, 10, 32):
        result[f"best_matches_k{k}_ms"] = time_ms(lambda: layer.bestMatches(ut, ue, k=k), args.steps, args.warmup)
        result[f"best_matches_k{k}_over_best_match"] = result[f"best_matches_k{k}_ms"] / result["best_match_ms"]
    result["bf16_matrix_ms"] = time_ms(lambda: layer.logLikelihoodRatio(ut, ue, out=scores16), args.steps, args.warmup)
    for k in (10, 32):
        def comp():
            layer.logLikelihoodRatio(ut, ue, out=scores16)
            return torch.topk(scores16, k, dim=1)
        result[f"bf16_matrix_topk_k{k}_ms"] = time_ms(comp, args.steps, args.warmup)
        result[f"speedup_k{k}_vs_bf16_matrix_topk"] = result[f"bf16_matrix_topk_k{k}_ms"] / result[f"best_matches_k{k}_ms"]
    result["trials_per_s_k32"] = float(n) * n / (result["best_matches_k32_ms"] * 1e-3)
    del scores16

    # parity on a sample of rows: the first k of a stable descending sort of the fp32 matrix, bit for bit
    rows = torch.from_numpy(np.sort(np.random.default_rng(3).choice(n, size=512, replace=False))).cuda()
    full = layer.logLikelihoodRatio(ut[rows].contiguous(), ue)
    s_sorted, i_sorted = torch.sort(full, dim=1, descending=True, stable=True)
    for k in (1, 10, 32):
        s, i = layer.bestMatches(ut, ue, k=k)
        result[f"parity_k{k}_bit_equal"] = bool(torch.equal(s[rows], s_sorted[:, :k]) and torch.equal(i[rows], i_sorted[:, :k]))
    print(json.dumps(result), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
