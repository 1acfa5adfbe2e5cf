"""
Wide-band front-end benchmark: the fused 1024..4096-point kernel against the obvious torch composition
(unfold framing -> window -> torch.fft.rfft -> |.|^2 -> mel matmul -> log -> DCT matmul) on the same batch.

    python scripts/bench_wideband.py [--batch 256] [--seconds 10] [--steps 10] [--warmup 3] [--out profiles/...json]

Every configuration runs float32 and int16 input, 25 ms frames every 10 ms.  Reports ms/step, audio-s/s, frames/s,
the algorithmic HBM bytes (samples in once, features out once) and their fraction of 7.7 TB/s, checks both outputs
against the float64 oracle with the parity gate of the test suite on a slice of the batch, and records the device name
and power limit read in the same run.
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

import kaldi_tflite_b200 as ktf                     # noqa: E402
from kaldi_tflite_b200.layers import dsp             # noqa: E402
from oracle import ktf_oracle as O                   # noqa: E402

HBM_BPS = 7.7e12
CONFIGS = [
    dict(name="32k_mfcc", rate=32000, kind="mfcc", num_mfccs=30, num_mels=40),
    dict(name="44k1_mfcc", rate=44100, kind="mfcc", num_mfccs=30, num_mels=40),
    dict(name="48k_mfcc", rate=48000, kind="mfcc", num_mfccs=30, num_mels=40),
    dict(name="48k_fbank80", rate=48000, kind="fbank", num_mels=80),
    dict(name="96k_mfcc", rate=96000, kind="mfcc", num_mfccs=30, num_mels=40),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:   # still record the torch device name
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


class TorchComposition:
    """The same features with stock torch ops (cuFFT for the transform)."""

    def __init__(self, cfg, W, S):
        self.kind, self.W, self.S = cfg["kind"], W, S
        N, bank = dsp.mel_filterbank(W, cfg["num_mels"], float(cfg["rate"]), 20.0, cfg["rate"] / 2.0)
        self.N = N
        self.bank = torch.from_numpy(bank).cuda()
        self.window = torch.from_numpy(dsp.window_function("povey", W)).cuda()
        if self.kind == "mfcc":
            self.dct = torch.from_numpy(dsp.dct2_matrix(cfg["num_mels"], cfg["num_mfccs"])).cuda()
            self.lifter = torch.from_numpy(dsp.lifter_coefficients(cfg["num_mfccs"], 22)).cuda()

    def __call__(self, wav):
        x = wav.float().unfold(-1, self.W, self.S)                    # (B, T, W)
        if self.kind == "mfcc":
            x = x - x.mean(dim=-1, keepdim=True)
            energy = torch.log(torch.clamp((x * x).sum(-1), min=0.0) + 1e-7)
            x = torch.cat([x[..., :1] * (1.0 - 0.97), x[..., 1:] - 0.97 * x[..., :-1]], dim=-1) * self.window
        spec = torch.fft.rfft(x, n=self.N).abs() ** 2
        feats = torch.log(torch.clamp(spec @ self.bank, min=0.0) + 1e-7)
        if self.kind == "fbank":
            return feats
        out = (feats @ self.dct) * self.lifter
        out[..., 0] = energy
        return out


def fused_layer(cfg):
    if cfg["kind"] == "mfcc":
        m = ktf.layers.MFCC(num_mfccs=cfg["num_mfccs"], num_mels=cfg["num_mels"], sample_frequency=float(cfg["rate"]))
        return lambda W, S: m.frontend(W, S)
    fb = ktf.layers.FilterBank(num_bins=cfg["num_mels"], sample_frequency=float(cfg["rate"]))
    return lambda W, S: fb._frontend(W, S)


def oracle(cfg, frames, precise):
    if cfg["kind"] == "mfcc":
        return O.mfcc(frames, num_mfccs=cfg["num_mfccs"], num_mels=cfg["num_mels"], sample_frequency=cfg["rate"],
                      precise=precise)
    return O.filterbank(frames, num_bins=cfg["num_mels"], sample_frequency=cfg["rate"], precise=precise)


def gate(got, truth, ora):
    e = np.abs(np.asarray(got, np.float64) - truth)
    f = np.abs(np.asarray(ora, np.float64) - truth)
    max_ok, p_ok = max(1e-3, 1.25 * float(f.max())), max(1e-3, float(np.quantile(f, 0.999)))
    return {"max_abs": float(e.max()), "max_abs_bound": max_ok, "p999": float(np.quantile(e, 0.999)),
            "p999_bound": p_ok, "pass": bool(e.max() <= max_ok and np.quantile(e, 0.999) <= p_ok)}


def time_steps(fn, steps, warmup):
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
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wideband_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_wideband.py needs a CUDA device")

    result = {"device": gpu_info(), "batch": args.batch, "seconds_per_utt": args.seconds, "steps": args.steps,
              "warmup": args.warmup, "hbm_peak_bytes_per_s": HBM_BPS, "configs": []}
    for cfg in CONFIGS:
        rate = cfg["rate"]
        fr = ktf.layers.Framing(25.0, 10.0, rate, dynamic_input_shape=True)
        W, S = fr.frameWidth, fr.frameShift
        n = int(rate * args.seconds)
        g = torch.Generator(device="cuda").manual_seed(1234)
        wav32 = torch.round(torch.randn((args.batch, n), device="cuda", generator=g) * 2000.0).clamp(-32768, 32767)
        fe = fused_layer(cfg)(W, S)
        comp = TorchComposition(cfg, W, S)
        T = fe.num_frames(n)
        for dtype in ("float32", "int16"):
            wav = wav32 if dtype == "float32" else wav32.to(torch.int16)
            fused_ms = time_steps(lambda: fe.forward(wav), args.steps, args.warmup)
            torch_ms = time_steps(lambda: comp(wav), args.steps, args.warmup)
            in_bytes = args.batch * n * (4 if dtype == "float32" else 2)
            out_bytes = 4 * args.batch * T * fe.out_dim
            algo = in_bytes + out_bytes
            # parity on a slice: both implementations against the float64 oracle
            k = 2
            got = fe.forward(wav[:k, : rate])[0].cpu().numpy()
            ref = comp(wav[:k, : rate]).cpu().numpy()
            frames = O.framing(wav32[:k, : rate].cpu().numpy(), 25.0, 10.0, rate)
            truth, ora = oracle(cfg, frames, True), oracle(cfg, frames, False)
            row = {"config": cfg["name"], "rate": rate, "frame_width": W, "frame_shift": S, "fft_length": comp.N,
                   "kind": cfg["kind"], "out_dim": fe.out_dim, "input": dtype, "frames_per_step": args.batch * T,
                   "fused_ms_per_step": fused_ms, "torch_ms_per_step": torch_ms,
                   "speedup_vs_torch": torch_ms / fused_ms,
                   "fused_audio_s_per_s": args.batch * args.seconds / (fused_ms * 1e-3),
                   "fused_frames_per_s": args.batch * T / (fused_ms * 1e-3),
                   "algorithmic_bytes": algo, "fused_bytes_per_s": algo / (fused_ms * 1e-3),
                   "fused_fraction_of_hbm": algo / (fused_ms * 1e-3) / HBM_BPS,
                   "fused_gate": gate(got, truth, ora), "torch_gate": gate(ref, truth, ora)}
            result["configs"].append(row)
            print(json.dumps(row), flush=True)
        del wav32, fe, comp
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"device": result["device"], "written": args.out}))


if __name__ == "__main__":
    main()
