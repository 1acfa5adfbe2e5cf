"""
What the PLDA score-form benchmarks (scripts/bench_plda_*.py) share: the device record, the timer and the vector setup.
"""

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


def plda_setup(script, n, n_cohort=0):
    """A float32 layer on synthetic_plda(DIM) and transformed vectors of norm sqrt(DIM) from torch's CUDA generator
    (seed 1234): (layer, n test, n enrolled, n_cohort cohort).  Exits when there is no CUDA device."""
    if not torch.cuda.is_available():
        sys.exit(f"{script} needs a CUDA device")
    mean, Tm, psi = synthetic_plda(DIM)
    layer = ktf.layers.PLDA(DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    g = torch.Generator(device="cuda").manual_seed(1234)
    x = torch.randn((2 * n + n_cohort, DIM), generator=g, device="cuda")
    u = layer.transformVector((x / x.norm(dim=1, keepdim=True) * DIM ** 0.5).contiguous())
    return layer, u[:n].contiguous(), u[n:2 * n].contiguous(), u[2 * n:].contiguous()
