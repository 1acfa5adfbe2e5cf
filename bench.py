#!/usr/bin/env python
"""
bench.py -- headline benchmark of the wav -> x-vector hot path (BASELINE.json: "wav2xvec audio-sec/sec at 1/2/4/8
B200; MFCC GB/s vs HBM peak").

    python bench.py --gpus N --steps K --warmup W [--impl reference]
                    [--workload wav2xvec|frontend|tdnn|plda] [--no-stages] [--no-cpu-baseline] [--dump-outputs DIR]

Default workload (N = 1 and under torchrun): the BASELINE config 4 shard -- full wav2xvec (fused MFCC -> VAD mask +
compaction -> CMVN(300) -> SITW TDNN on the tcgen05 stack -> statistics -> LDA / length-norm) on 1024 gated-noise
utterances x 10 s of synthetic 16 kHz audio per GPU, through models.XvectorExtractor (the reference's
models/kaldi/xvector_extractor.py:137-186).  One "step" = one pass of the hot path over one batch.  Utterances are
sharded, there is NO data-path collective ("weak" scaling); value = all ranks' audio seconds / max-over-ranks device time.

One JSON line is printed by rank 0 (DESIGN.md section 6 explains every field):
  value        audio-seconds per second with the batch already resident in HBM (CUDA events)
  e2e          the same metric through the public model API with HOST (pinned) buffers: H2D of the audio and D2H of the
               x-vectors are inside the timed region every step; with the achieved H2D rate per rank and the box's
               measured concurrent pinned-memcpy ceiling beside it
  roofline     the dominant kernels (the tcgen05 TDNN stack): algorithmic FLOPs per step / their own device time vs the
               measured bf16 peaks in MEASURED_PEAKS.json (sustained = `frac`, burst = `frac_of_burst`)
  cpu_baseline the CPU oracle (oracle/ktf_oracle.py, an op-for-op NumPy port of the reference's layers; the reference
               itself needs TensorFlow 2.8, not installable here) on a bounded sample (N = 1 only)
  stages       the other BASELINE configs measured in the same run, each with its own roofline:
                 frontend  config 2, MFCC(30/30) + CMVN(200) on 1024 x 10 s, HBM roofline of the fused kernel
                 tdnn      config 3, SITW stack on 512 x 300 frames (N = 1 only)
                 plda      config 5, 50 000 x 50 000 trials, enrolled columns sharded over the N ranks, the all-gather of
                           the transformed test vectors (NCCL) timed separately, `parity_max_rel` of a sampled
                           sub-block against the float64 oracle

`--workload X` makes one of the stages the headline line with the same schema.

`--dump-outputs DIR` writes what the last timed step of the headline workload returned, as DIR/<name>.npy: `xvectors`
(wav2xvec), `features` (frontend, CMVN output), `embeddings` (tdnn), `scores` and `transformed_test` (plda).  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the CPU port with all host threads on a bounded sample of the same workload (rank 0 only); it
is the only other place allowed to execute oracle/.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

SR = 16000
UTT_SECONDS = 10
UTT_SAMPLES = SR * UTT_SECONDS
BATCH = 1024
FRAMES = 1 + (UTT_SAMPLES - 400) // 160          # 998
NUM_CEPS = 30
CMVN_WINDOW = 200
ALGO_BYTES_PER_UTT = UTT_SAMPLES * 4 + FRAMES * NUM_CEPS * 4      # wav once + features once (SURVEY 8d)

TDNN_FLOP_PER_FRAME = 2 * (150 * 512 + 1536 * 512 + 1536 * 512 + 512 * 512 + 512 * 1500)   # 5 359 616
TDNN_FLOP_PER_UTT = 2 * 3000 * 512                                                          # tdnn6
PLDA_DIM = 128


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "tf_burst": float(d["bf16_tflops"]),
                "tf_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        clocks, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                clocks.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(clocks)) if clocks else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(clocks)}


# ----------------------------------------------------------------------------------------------
# shared model / data builders
# ----------------------------------------------------------------------------------------------

def extractor_cfg():
    import yaml
    with open(os.path.join(ROOT, "data", "tflite_models", "0008_sitw_v2_1a.yml")) as f:
        cfg = yaml.safe_load(f)["extractor"]
    g = os.path.join(ROOT, "tests", "golden")
    cfg["mfcc"]["dither"] = 0.0
    cfg["xvec"]["model_config_path"] = os.path.join(ROOT, cfg["xvec"]["model_config_path"])
    cfg["xvec"]["model_path"] = None                       # Kaldi final.raw is not vendored: seeded random init
    cfg["xvec"]["global_mean_path"] = os.path.join(g, "sitw_mean.vec")
    cfg["xvec"]["lda_matrix_path"] = os.path.join(g, "sitw_transform.mat")
    return cfg


def sitw_nnet_cfg():
    import yaml
    with open(os.path.join(ROOT, "data", "kaldi_models", "configs", "0008_sitw_v2_1a.yml")) as f:
        return yaml.safe_load(f)["model_config"]


def gated_noise_np(n_utt, seed):
    """SURVEY 8d cfg4: Gaussian noise (sigma 3000) gated by a random on/off envelope (0.2 s grain, ~70 %
    duty), 'silence' sigma 30 -- so that the VAD keeps a non-trivial, threshold-robust subset."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n_utt, UTT_SAMPLES), dtype=np.float32)
    seg = 3200
    on = (rng.random((n_utt, UTT_SAMPLES // seg)) < 0.7).astype(np.float32)
    env = np.repeat(on, seg, axis=1)
    return x * (30.0 + 2970.0 * env)


def gated_noise_cuda(n_utt, seed, dev):
    import torch
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn((n_utt, UTT_SAMPLES), generator=g, device=dev)
    seg = 3200
    on = (torch.rand((n_utt, UTT_SAMPLES // seg), generator=g, device=dev) < 0.7).float()
    return x * (30.0 + 2970.0 * on.repeat_interleave(seg, dim=1))


def synthetic_plda(dim, seed=1234):
    rng = np.random.default_rng(seed)
    psi = np.exp(np.linspace(3, -4, dim))
    q, _ = np.linalg.qr(rng.standard_normal((dim, dim)))
    Tm = q * rng.uniform(0.5, 2.0, size=(1, dim))
    mean = rng.standard_normal(dim) * 0.05
    return mean, Tm, psi


def oracle_layers(seq):
    import kaldi_tflite_b200 as ktf
    out = []
    for l in seq.layers:
        if isinstance(l, ktf.layers.TDNN):
            out.append({"type": "affine", "kernel": l.kernel, "bias": l.bias, "context": l.context})
        elif isinstance(l, ktf.layers.ReLU):
            out.append({"type": "relu"})
        elif isinstance(l, ktf.layers.BatchNorm):
            out.append({"type": "batchnorm", "gamma": l.gamma, "mean": l.moving_mean,
                        "var": l.moving_variance, "epsilon": l.epsilon})
        elif isinstance(l, ktf.layers.StatsPooling):
            out.append({"type": "stats", "left_context": l.leftContext, "right_context": l.rightContext,
                        "include_std": l.includeStd, "reduce_time_axis": l.reduce})
    return out


# ----------------------------------------------------------------------------------------------
# CPU port (oracle) -- cpu_baseline leg and --impl reference.  The only code here that touches oracle/.
# ----------------------------------------------------------------------------------------------

_POOL_JOB = None


def _pool_call(bounds):
    fn, items = _POOL_JOB
    try:                                                     # one BLAS / FFT thread per worker process
        from threadpoolctl import threadpool_limits
        with threadpool_limits(limits=1):
            fn(items[bounds[0]:bounds[1]])
    except ImportError:
        fn(items[bounds[0]:bounds[1]])
    return 0


def _threads_run(fn, items, threads):
    """Runs fn over `items` split across `threads` host workers (forked processes: NumPy's Python-level
    glue does not scale across threads under the GIL; the CPU legs never touch CUDA, so fork is safe)."""
    global _POOL_JOB
    chunks = [(int(c[0]), int(c[-1]) + 1) for c in np.array_split(np.arange(len(items)), threads) if len(c)]
    if len(chunks) <= 1:
        t0 = time.perf_counter()
        fn(items)
        return time.perf_counter() - t0
    import multiprocessing as mp
    _POOL_JOB = (fn, items)
    with mp.get_context("fork").Pool(len(chunks)) as pool:
        pool.map(_pool_call, [(0, 0)] * len(chunks))          # spin the workers up outside the timed region
        t0 = time.perf_counter()
        pool.map(_pool_call, chunks, chunksize=1)
        dt = time.perf_counter() - t0
    _POOL_JOB = None
    return dt


class CpuPort:
    """Bounded samples of each workload on the NumPy port of the reference layers."""

    def __init__(self):
        from oracle import ktf_oracle as O
        self.O = O
        self._wav2xvec = None

    def frontend(self, n_utt, threads, seed=0):
        O = self.O
        rng = np.random.default_rng(seed)
        wav = np.clip(rng.standard_normal((n_utt, UTT_SAMPLES), dtype=np.float32) * 3000.0, -32767, 32767)

        def run(w):
            for i in range(0, w.shape[0], 8):
                x = O.framing(w[i:i + 8], 25.0, 10.0, float(SR))
                x = O.mfcc(x, num_mfccs=NUM_CEPS, num_mels=30)
                O.cmvn(x, window=CMVN_WINDOW)
        return _threads_run(run, wav, threads), n_utt * UTT_SECONDS, "audio-s"

    def _model(self):
        if self._wav2xvec is None:
            # weights come from the same seeded initialisers as the GPU arm; built WITHOUT touching CUDA
            from kaldi_tflite_b200.models.sequential import SequentialFromConfig
            from kaldi_tflite_b200.io import ReadKaldiArray
            cfg = extractor_cfg()
            seq = SequentialFromConfig(sitw_nnet_cfg(), None, "cmvn2xvec", seed=0)
            seq._build_layers(30)
            mean = np.ascontiguousarray(ReadKaldiArray(cfg["xvec"]["global_mean_path"], binary=True), np.float32)
            lda = np.ascontiguousarray(ReadKaldiArray(cfg["xvec"]["lda_matrix_path"], binary=True), np.float32)
            self._wav2xvec = (cfg, oracle_layers(seq), mean, lda)
        return self._wav2xvec

    def wav2xvec(self, n_utt, threads, seed=0):
        O = self.O
        cfg, layers, mean, lda = self._model()
        wav = gated_noise_np(n_utt, seed)

        def run(w):
            for u in w:
                O.xvector_extractor(u, cfg, layers, mean, lda)
        return _threads_run(run, wav, threads), n_utt * UTT_SECONDS, "audio-s"

    def tdnn(self, n_utt, threads, seed=0):
        O = self.O
        _, layers, _, _ = self._model()
        x = np.random.default_rng(seed).standard_normal((n_utt, 300, 30)).astype(np.float32)

        def run(xx):
            for u in xx:
                O.sequential(u[None], layers)
        return _threads_run(run, x, threads), n_utt * 3.0, "audio-s"

    def plda(self, n, threads, seed=0):
        O = self.O
        mean, Tm, psi = synthetic_plda(PLDA_DIM)
        rng = np.random.default_rng(seed)
        x = rng.standard_normal((n, PLDA_DIM))
        x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(PLDA_DIM)).astype(np.float32)
        t0 = time.perf_counter()
        O.plda(x, mean, Tm, psi, dtype=np.float32)           # the reference's (B, dim, B) broadcast formulation
        return time.perf_counter() - t0, float(n) * n, "scores"


CPU_SAMPLE = {"frontend": 192, "wav2xvec": 384, "tdnn": 32, "plda": 768}
DEFAULT_WORKLOAD = "wav2xvec"        # BASELINE.json metric: wav2xvec audio-sec/sec (config 4 shard per GPU)
WORKLOAD_UNIT = {"frontend": "audio-s/s", "wav2xvec": "audio-s/s", "tdnn": "audio-s/s", "plda": "scores/s"}
WORKLOAD_METRIC = {"frontend": "audio_sec_per_sec", "wav2xvec": "audio_sec_per_sec",
                   "tdnn": "audio_sec_per_sec", "plda": "plda_scores_per_sec"}


def cpu_baseline(workload, threads):
    port = CpuPort()
    n = CPU_SAMPLE[workload] * (max(1, threads // 2) if workload != "plda" else 1)     # about 10-20 s of CPU work
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=1 if threads == 1 else None)
    except ImportError:
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        secs, units, what = getattr(port, workload)(n, threads)
    desc = {"frontend": f"{n} utterances x {UTT_SECONDS} s of the same MFCC+CMVN workload",
            "wav2xvec": f"{n} gated-noise utterances x {UTT_SECONDS} s through the whole pipeline",
            "tdnn": f"{n} x 300-frame chunks through the SITW stack (fp32)",
            "plda": f"{n} x {n} trials, (B, dim, B) broadcast formulation of the reference (fp32)"}[workload]
    return {"value": units / secs, "unit": WORKLOAD_UNIT[workload], "cores": threads, "kind": "port",
            "sample": f"{desc}; NumPy port of the reference layers (TensorFlow unavailable), {secs:.1f} s"}


def workload_config(workload, n_gpus):
    base = {"parallelism": f"utterance-sharded x{n_gpus}, no collective"}
    if workload == "frontend":
        base.update({"workload": "BASELINE config 2: Framing(25ms/10ms) -> MFCC(30 mfcc, 30 mel, povey, dither 0) -> "
                                 "CMVN(window 200), batch 1024 x 10 s synthetic 16 kHz float32 audio per GPU",
                     "batch_per_gpu": BATCH, "utt_seconds": UTT_SECONDS, "frames_per_utt": FRAMES,
                     "l2_policy": "input batch is 655 MB per step, larger than the 126 MB L2 (no explicit flush needed)"})
    elif workload == "wav2xvec":
        base.update({"workload": "BASELINE config 4 shard: full wav2xvec (MFCC -> VAD mask -> CMVN(300) -> SITW TDNN "
                                 "bf16 -> stats -> LDA/length-norm), 1024 gated-noise utterances x 10 s per GPU, "
                                 "random-init TDNN (Kaldi weights not vendored), real LDA / mean",
                     "batch_per_gpu": BATCH, "utt_seconds": UTT_SECONDS, "tdnn_precision": "bf16 operands, fp32 accumulate "
                     "(the API default)", "host_syncs_per_step": 0,
                     "l2_policy": "655 MB of audio and > 1 GB of activations per step, larger than the 126 MB L2"})
    elif workload == "tdnn":
        base.update({"workload": "BASELINE config 3: SITW x-vector TDNN (5 TDNN-512 + 1500-d stats + 512 embedding, "
                                 "random init), batch 512 x 300 frames per GPU",
                     "batch_per_gpu": 512, "frames_per_utt": 300, "tdnn_precision": "bf16 operands, fp32 accumulate",
                     "l2_policy": "L2 flushed between timed iterations (256 MB scratch write)"})
    else:
        base.update({"workload": "BASELINE config 5: PLDA all-vs-all 50k enroll x 50k test x-vectors (dim 128), enrolled "
                                 "columns sharded over the ranks, test vectors exchanged with one all-gather",
                     "parallelism": f"enrolled columns sharded x{n_gpus}, NCCL all-gather of the transformed test vectors",
                     "n_enroll": 50000, "n_test": 50000, "dim": PLDA_DIM,
                     "l2_policy": "each step writes >= 1.25 GB of scores per GPU, larger than the 126 MB L2"})
    return base


# ----------------------------------------------------------------------------------------------
# reference arm
# ----------------------------------------------------------------------------------------------

def run_reference(args):
    """The CPU port of the reference's layers on all host threads (TensorFlow 2.8, which the reference
    needs, is not installable in this image: `import tensorflow` fails, no network)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = os.cpu_count() or 1
    port = CpuPort()
    w = args.workload
    n = CPU_SAMPLE[w] * (max(1, threads // 2) if w != "plda" else 1)
    if w == "wav2xvec":
        n = 64 * threads                                      # about 2 s per step: K + W steps within a few minutes
    elif w != "frontend":
        n = max(n // 4, threads if w != "plda" else 256)
    for _ in range(args.warmup):
        getattr(port, w)(n, threads)
    t, units = 0.0, 0.0
    for s in range(args.steps):
        secs, u, _ = getattr(port, w)(n, threads, seed=s)
        t += secs
        units += u
    value = units / t
    line = {
        "impl": "reference", "metric": WORKLOAD_METRIC[w], "value": value, "unit": WORKLOAD_UNIT[w],
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(w, args.gpus),
        "cpu_baseline": {"value": value, "unit": WORKLOAD_UNIT[w], "cores": threads, "kind": "port",
                         "sample": f"{n} units of the workload per step (NumPy port of the reference layers; "
                                   f"TensorFlow unavailable)"},
        "e2e": {"value": value, "unit": WORKLOAD_UNIT[w], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_json(line)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------

class Harness:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference "
                             "for the CPU port")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.args = args
        self.flush_buf = None
        self.last_output = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def flush_l2(self):
        if self.flush_buf is None:
            self.flush_buf = self.torch.empty(64 * 1024 * 1024, dtype=self.torch.float32, device=self.dev)
        self.flush_buf.fill_(1.0)

    def max_over_ranks(self, ms):
        t = self.torch.tensor([ms], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, step, steps, warmup, flush=False, inner=None):
        """W warm-up steps, then K steps bracketed by barrier + synchronize; returns (ms total [max over
        ranks], launches, clocks, mean ms of the `inner` event pairs recorded by step()).  What the last timed
        step returned is left in `self.last_output`."""
        import kaldi_tflite_b200 as ktf
        torch = self.torch
        for _ in range(max(warmup, 3)):
            step(None)
        self.barrier()
        sampler = ClockSampler(self.local_rank)
        sampler.start()
        pairs = []
        n0 = ktf.launch_count()
        self.barrier()
        if flush:
            # per-step events so that the L2 flush writes stay outside the measured time
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for s in range(steps):
                self.flush_l2()
                self.last_output = None                       # freed before the next step, as a caller would
                evs[s][0].record()
                self.last_output = step(pairs)
                evs[s][1].record()
            self.barrier()
            ms = sum(a.elapsed_time(b) for a, b in evs)
        else:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(steps):
                self.last_output = None
                self.last_output = step(pairs)
            e1.record()
            self.barrier()
            ms = e0.elapsed_time(e1)
        clocks = sampler.stop()
        launches = ktf.launch_count() - n0
        inner_ms = float(np.mean([a.elapsed_time(b) for a, b in pairs])) if pairs else None
        return self.max_over_ranks(ms), int(launches), clocks, inner_ms


def ev_pair(torch):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


DUMP_BYTES = 60 << 20                  # under 64 MB (10^6 bytes each) with the .npy headers


def host_outputs(arrays, seed=0):
    """{name: tensor} -> {name: float32 / float64 host array} for --dump-outputs.  Every array gets an equal share of
    DUMP_BYTES; a larger one keeps a sample of its leading-axis rows drawn with a fixed seed (sorted), so that two
    builds run with the same arguments dump the same elements."""
    import torch
    out = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.dtype != torch.float64:
            t = t.float()
        row_bytes = t[0].numel() * t.element_size() if t.dim() > 1 else t.element_size()
        keep = max(1, DUMP_BYTES // len(arrays) // row_bytes)
        if t.shape[0] > keep:
            rows = np.sort(np.random.default_rng(seed).choice(t.shape[0], size=keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        out[name] = t.cpu().numpy()
    return out


def stage_tdnn(h, steps, warmup, dump=False):
    import kaldi_tflite_b200 as ktf
    torch = h.torch
    mdl = ktf.models.SequentialFromConfig(sitw_nnet_cfg(), None, "cmvn2xvec", precision="bf16", seed=0)
    g = torch.Generator(device=h.dev).manual_seed(1234 + h.rank)
    B, Tn = 512, 300
    feats = torch.randn((B * Tn, 30), generator=g, device=h.dev)
    offs = torch.arange(B + 1, device=h.dev, dtype=torch.int64) * Tn

    def step(pairs):
        return mdl.forward_ragged(feats, offs)[0]
    ms, launches, clocks, _ = h.timed(step, steps, warmup, flush=True)
    outputs = host_outputs({"embeddings": h.last_output}) if dump else None
    flops = (TDNN_FLOP_PER_FRAME * B * Tn + TDNN_FLOP_PER_UTT * B) * steps
    host_in = torch.empty((B * Tn, 30), dtype=torch.float32, pin_memory=True).copy_(feats)
    host_out = torch.empty((B, 512), dtype=torch.float32, pin_memory=True)

    def e2e(pairs):
        y, _ = mdl.forward_ragged(host_in.to(h.dev, non_blocking=True), offs)
        host_out.copy_(y, non_blocking=True)
    ms_e2e, _, _, _ = h.timed(e2e, steps, 2)
    return {"ms": ms, "steps": steps, "launches": launches, "clocks": clocks, "units": B * 3.0 * h.world * steps,
            "flops": flops, "ms_e2e": ms_e2e, "h2d": B * Tn * 30 * 4, "d2h": B * 512 * 4, "outputs": outputs}


def h2d_ceiling(h, mbytes=256, reps=6):
    """The box's pinned-memcpy H2D rate with ALL ranks copying at once (plain cudaMemcpyAsync loop, no compute): the
    ceiling any end-to-end number that ships the audio over PCIe can reach.  Returns GB/s (this rank, min over ranks,
    sum over ranks)."""
    torch = h.torch
    host = torch.empty(mbytes << 20, dtype=torch.uint8, pin_memory=True)
    dev = torch.empty(mbytes << 20, dtype=torch.uint8, device=h.dev)
    dev.copy_(host, non_blocking=True)
    h.barrier()
    a, b = ev_pair(torch)
    a.record()
    for _ in range(reps):
        dev.copy_(host, non_blocking=True)
    b.record()
    h.barrier()
    gbs = reps * (mbytes << 20) / (a.elapsed_time(b) * 1e-3) / 1e9
    t = torch.tensor([gbs, -gbs, gbs], device=h.dev, dtype=torch.float64)
    if h.world > 1:
        mx = t[:2].clone()
        h.dist.all_reduce(mx, op=h.dist.ReduceOp.MAX)
        sm = t[2:].clone()
        h.dist.all_reduce(sm, op=h.dist.ReduceOp.SUM)
        return gbs, float(-mx[1].item()), float(sm[0].item())
    return gbs, gbs, gbs


def stage_wav2xvec(h, steps, warmup, batch=BATCH, dump=False):
    import kaldi_tflite_b200 as ktf
    torch = h.torch
    # default precision of the public API: bf16 operands on the tcgen05 stack
    ext = ktf.models.XvectorExtractor(extractor_cfg(), seed=0, allow_random_init=True)
    wav = gated_noise_cuda(batch, 7 + h.rank, h.dev)
    _, inter = ext(wav, return_intermediate=True)
    kept = int(inter["voiced_offsets"][-1].item())           # outside the timed region: for the FLOP count only
    assert ext.xvec._stack is not None, "the TDNN stack is not on the tcgen05 engine"
    stack = ext.xvec.fused_vad_cmvn_stack(30)
    assert stack is not None, "the fused VAD / CMVN / splice pre-pass does not apply"
    fuse = os.environ.get("KTF_BENCH_FUSE", "1") != "0"
    ext.fusePrepass = fuse

    def step(pairs):
        if pairs is None:
            ext(wav)
            return
        # exactly ext(wav) (models/xvector_extractor.py: features -> embed -> backend), with an event pair around the
        # TDNN stack; nothing in it synchronises with the host (the kept-row count after VAD stays on the device)
        feats, offsets = ext.features(*ext._flatten(wav))
        mask = ext.vad.mask_ragged(feats, offsets)
        if fuse:
            _, voffs, index = ext.vad.compact_ragged(feats, mask, offsets, gather=False)
            a, b = ev_pair(torch)
            a.record()
            # the tcgen05 stack: VAD gather + CMVN + splice pre-pass, 6 GEMM launches, statistics finalize
            emb = stack.forward_vad(feats, index, voffs, FRAMES, ext.cmvn.N)
            b.record()
        else:                                                  # development A/B: separate gather / CMVN / splice kernels
            voiced, voffs, _ = ext.vad.compact_ragged(feats, mask, offsets, gather=True)
            normed, _ = ext.cmvn.forward_ragged(voiced, voffs, max_frames=FRAMES)
            a, b = ev_pair(torch)
            a.record()
            emb, _ = ext.xvec.forward_ragged(normed, voffs)
            b.record()
        pairs.append((a, b))
        return ext.backend(emb)
    ms, launches, clocks, tdnn_ms = h.timed(step, steps, warmup)
    outputs = host_outputs({"xvectors": h.last_output}) if dump else None
    host_in = torch.empty((batch, UTT_SAMPLES), dtype=torch.float32, pin_memory=True).copy_(wav)
    host_out = torch.empty((batch, 128), dtype=torch.float32, pin_memory=True)

    from kaldi_tflite_b200 import parallel

    def e2e(pairs):                                           # public API: model call on chunks of the host batch,
        parallel.stream_batches(ext, host_in, 128, host_out)   # copies overlapped with compute on side streams
    ms_e2e, _, _, _ = h.timed(e2e, steps, 2)
    # the same host batch as raw int16 PCM (SURVEY 8f rank 1: what a wav file holds; reported separately, the
    # API-compatible figure above is the float32 one)
    host_pcm = torch.empty((batch, UTT_SAMPLES), dtype=torch.int16, pin_memory=True).copy_(wav.round().to(torch.int16))

    def e2e_pcm(pairs):
        parallel.stream_batches(ext, host_pcm, 128, host_out)
    ms_e2e_pcm, _, _, _ = h.timed(e2e_pcm, steps, 2)
    ceil_rank, ceil_min, ceil_sum = h2d_ceiling(h)
    return {"ms": ms, "steps": steps, "launches": launches, "clocks": clocks,
            "pcm16": {"ms_e2e": ms_e2e_pcm, "h2d": batch * UTT_SAMPLES * 2},
            "units": batch * UTT_SECONDS * h.world * steps, "tdnn_ms": tdnn_ms,
            "flops": TDNN_FLOP_PER_FRAME * kept + TDNN_FLOP_PER_UTT * batch, "vad_keep": kept / (batch * FRAMES),
            "ms_e2e": ms_e2e, "h2d": batch * UTT_SAMPLES * 4, "d2h": batch * 128 * 4,
            "h2d_ceiling": {"per_rank_min_gbs": ceil_min, "aggregate_gbs": ceil_sum,
                            "how": "plain pinned cudaMemcpyAsync loop, 256 MB x 6, all ranks at once"},
            "outputs": outputs}


def plda_parity(layer, x_test_rows, x_enroll_rows, got_block):
    """Checker (outside every timed region): a sampled sub-block of the scores against the float64 oracle, evaluated in
    the reference's direct form.  Returns max |delta| / max(|s|, 1)."""
    from oracle import ktf_oracle as O
    worst = 0.0
    nt, ne = x_test_rows.shape[0], x_enroll_rows.shape[0]
    for i in range(0, nt, 256):                               # the (B, dim, B) form: keep the temporaries near 1 GB
        xs = np.concatenate([x_test_rows[i:i + 256], x_enroll_rows]).astype(np.float32)
        u = O.plda_transform(xs, layer.mean, layer.transformMat, layer.psi, dtype=np.float64)
        k = xs.shape[0] - ne
        want = O.plda_llr(u, layer.psi)[:k, k:]
        got = got_block[i:i + k]
        worst = max(worst, float(np.max(np.abs(got - want) / np.maximum(np.abs(want), 1.0))))
    return worst


def stage_plda(h, steps, warmup, n=50000, dump=False):
    import kaldi_tflite_b200 as ktf
    from kaldi_tflite_b200 import parallel
    torch = h.torch
    n = int(os.environ.get("KTF_BENCH_PLDA_N", n))          # development knob (smaller all-vs-all problems)
    mean, Tm, psi = synthetic_plda(PLDA_DIM)
    layer = ktf.layers.PLDA(PLDA_DIM, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    g = torch.Generator(device=h.dev).manual_seed(1234 + h.rank)
    lo, hi = parallel.shard_range(n, h.rank, h.world)

    def xvecs(count):
        x = torch.randn((count, PLDA_DIM), generator=g, device=h.dev)
        return x / x.norm(dim=1, keepdim=True) * PLDA_DIM ** 0.5
    x_test, x_enroll = xvecs(hi - lo), xvecs(hi - lo)
    # this rank's block (10 GB / G); the row pitch is padded to 16 bytes so that the boxed (TMA) stores apply at every G
    ld = (hi - lo + 7) // 8 * 8
    scores = torch.empty((n, ld), device=h.dev, dtype=torch.float32)[:, :hi - lo]

    counts = [parallel.shard_range(n, r, h.world)[1] - parallel.shard_range(n, r, h.world)[0] for r in range(h.world)]

    def step(pairs):
        # transforms + the only collective (ONE asynchronous NCCL all-gather of the transformed test vectors, 25.6 MB in
        # total; the local rows are scored underneath it) + the score GEMMs of the other ranks' rows
        return parallel.plda_score_sharded(layer, x_test, x_enroll, test_counts=counts, out=scores)
    ms, launches, clocks, _ = h.timed(step, steps, warmup)
    # taken now: the checks below write into the same score buffer
    outputs = host_outputs(dict(zip(("scores", "transformed_test"), h.last_output))) if dump else None

    # ---- in-run parity: sampled rows x sampled columns of THIS rank's block against the float64 oracle
    sc, u_all_chk = parallel.plda_score_sharded(layer, x_test, x_enroll, test_counts=counts, out=scores)
    rs = np.random.default_rng(5 + h.rank)
    ti = np.sort(rs.choice(hi - lo, size=min(1024, hi - lo), replace=False))       # local test rows (global = lo + ti)
    ei = np.sort(rs.choice(hi - lo, size=min(1024, hi - lo), replace=False))
    tI, eI = torch.from_numpy(ti).to(h.dev), torch.from_numpy(ei).to(h.dev)
    got_block = sc[lo:hi][tI][:, eI].cpu().numpy()
    parity = plda_parity(layer, x_test[tI].cpu().numpy(), x_enroll[eI].cpu().numpy(), got_block)
    parity = h.max_over_ranks(parity)

    # ---- the exchange alone (NCCL all-gather of the transformed test vectors), device-timed
    u_local = layer.transformVector(x_test)

    def gather_only(pairs):
        a, b = ev_pair(torch)
        if pairs is not None:
            a.record()
        if h.world > 1:
            _, _, works = parallel.exchange_test_vectors(u_local, counts)
            for wk in works:
                if wk is not None:
                    wk.wait()
        if pairs is not None:
            b.record()
            pairs.append((a, b))
    gather_ms = 0.0
    if h.world > 1:
        _, _, _, gather_ms = h.timed(gather_only, steps, 2)
        gather_ms = h.max_over_ranks(gather_ms)

    # ---- the score kernel alone (roofline): this rank's (n x n/G) block from vectors already gathered
    u_all = parallel.gather_rows(u_local)
    u_enroll = layer.transformVector(x_enroll)

    def score_only(pairs):
        a, b = ev_pair(torch)
        if pairs is not None:
            a.record()
        layer.logLikelihoodRatio(u_all, u_enroll, out=scores)
        if pairs is not None:
            b.record()
            pairs.append((a, b))
    _, _, _, score_ms = h.timed(score_only, steps, 2)
    # compact output (SURVEY 8f rank 3): the same scores rounded once to bfloat16, half the HBM write
    scores16 = torch.empty((n, ld), device=h.dev, dtype=torch.bfloat16)[:, :hi - lo]

    def score_bf16(pairs):
        a, b = ev_pair(torch)
        if pairs is not None:
            a.record()
        layer.logLikelihoodRatio(u_all, u_enroll, out=scores16)
        if pairs is not None:
            b.record()
            pairs.append((a, b))
    _, _, _, score16_ms = h.timed(score_bf16, steps, 2)
    del scores16

    # best trial per test vector (top-k = 1): no score matrix at all
    def score_top1(pairs):
        a, b = ev_pair(torch)
        if pairs is not None:
            a.record()
        layer.bestMatch(u_all, u_enroll)
        if pairs is not None:
            b.record()
            pairs.append((a, b))
    _, _, _, top1_ms = h.timed(score_top1, steps, 2)
    host_t = torch.empty_like(x_test, device="cpu").pin_memory().copy_(x_test)
    host_e = torch.empty_like(x_enroll, device="cpu").pin_memory().copy_(x_enroll)
    host_top = torch.empty((n,), dtype=torch.float32, pin_memory=True)

    def e2e(pairs):
        sc2, _ = parallel.plda_score_sharded(layer, host_t.to(h.dev, non_blocking=True),
                                             host_e.to(h.dev, non_blocking=True), test_counts=counts, out=scores)
        host_top.copy_(sc2.max(dim=1).values, non_blocking=True)        # result read back: best trial per test vector
    ms_e2e, _, _, _ = h.timed(e2e, steps, 2)
    return {"ms": ms, "steps": steps, "launches": launches, "clocks": clocks, "units": float(n) * n * steps,
            "score_ms": score_ms, "score_bytes": float(n) * (hi - lo) * 4, "flops": 2.0 * n * (hi - lo) * PLDA_DIM,
            "allgather_ms": gather_ms, "allgather_bytes": n * PLDA_DIM * 4, "parity_max_rel": parity, "n": n,
            "score16_ms": score16_ms, "top1_ms": top1_ms,
            "ms_e2e": ms_e2e, "h2d": 2 * (hi - lo) * PLDA_DIM * 4, "d2h": n * 4, "outputs": outputs}


def stage_frontend(h, steps, warmup, dump=False):
    import kaldi_tflite_b200 as ktf
    torch = h.torch
    g = torch.Generator(device=h.dev).manual_seed(1234 + h.rank)
    wav = (torch.randn((BATCH, UTT_SAMPLES), generator=g, device=h.dev) * 3000.0).clamp_(-32767, 32767)
    framing = ktf.layers.Framing(25.0, 10.0, float(SR), dynamic_input_shape=True)
    mfcc = ktf.layers.MFCC(num_mfccs=NUM_CEPS, num_mels=30)
    cmvn = ktf.layers.CMVN(center=True, window=CMVN_WINDOW, norm_vars=False)
    fe = mfcc.frontend(framing.frameWidth, framing.frameShift)

    def step(pairs):
        if pairs is None:
            cmvn(mfcc(framing(wav)))
            return
        a, b = ev_pair(torch)
        a.record()
        feats, _ = fe.forward(wav)                           # the fused front-end kernel (one launch)
        b.record()
        pairs.append((a, b))
        return cmvn(feats)
    ms, launches, clocks, k_ms = h.timed(step, steps, warmup)
    outputs = host_outputs({"features": h.last_output}) if dump else None
    host_in = torch.empty((BATCH, UTT_SAMPLES), dtype=torch.float32, pin_memory=True).copy_(wav)
    host_out = torch.empty((BATCH, FRAMES, NUM_CEPS), dtype=torch.float32, pin_memory=True)

    from kaldi_tflite_b200 import parallel

    def e2e(pairs):                                           # public layer API on chunks of the host batch,
        parallel.stream_batches(lambda x: cmvn(mfcc(framing(x))), host_in, 128, host_out)   # copies overlapped
    ms_e2e, _, _, _ = h.timed(e2e, steps, 2)
    # the same batch as raw int16 PCM (SURVEY 8f rank 1), reported separately with its own algorithmic bytes
    pcm = wav.round().to(torch.int16)

    def step_pcm(pairs):
        if pairs is None:
            cmvn(mfcc(framing(pcm)))
            return
        a, b = ev_pair(torch)
        a.record()
        feats, _ = fe.forward(pcm)
        b.record()
        pairs.append((a, b))
        cmvn(feats)
    ms_pcm, _, _, k_ms_pcm = h.timed(step_pcm, steps, warmup)
    host_pcm = torch.empty((BATCH, UTT_SAMPLES), dtype=torch.int16, pin_memory=True).copy_(pcm)

    def e2e_pcm(pairs):
        parallel.stream_batches(lambda x: cmvn(mfcc(framing(x))), host_pcm, 128, host_out)
    ms_e2e_pcm, _, _, _ = h.timed(e2e_pcm, steps, 2)
    return {"ms": ms, "steps": steps, "launches": launches, "clocks": clocks,
            "pcm16": {"ms": ms_pcm, "kernel_ms": k_ms_pcm, "ms_e2e": ms_e2e_pcm, "h2d": BATCH * UTT_SAMPLES * 2,
                      "algo_bytes": BATCH * (UTT_SAMPLES * 2 + FRAMES * NUM_CEPS * 4)},
            "units": BATCH * UTT_SECONDS * h.world * steps, "kernel_ms": k_ms,
            "ms_e2e": ms_e2e, "h2d": BATCH * UTT_SAMPLES * 4, "d2h": BATCH * FRAMES * NUM_CEPS * 4, "outputs": outputs}


def measured_traffic(kernel_key):
    """DRAM bytes per launch of a kernel from the committed `ncu --set full` capture (profiles/r02_traffic.json, written
    by scripts/summarize_profiles.py from the .ncu-rep of the same bench command); None when there is no capture."""
    tf = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(tf):
        return None, None
    with open(tf) as f:
        d = json.load(f)
    e = d.get(kernel_key)
    if not e:
        return None, None
    return e.get("dram_bytes_per_launch"), f"profiles/r02_traffic.json ({e.get('source', 'ncu --set full')})"


def roofline_for(workload, r, pk):
    if workload == "frontend":
        achieved = ALGO_BYTES_PER_UTT * BATCH / (r["kernel_ms"] * 1e-3) / 1e9
        traffic, src = measured_traffic("frontend")
        return {"bound": "hbm", "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s", "frac": achieved / pk["hbm"],
                "traffic": traffic, "traffic_source": src, "peak_source": pk["src"] + " hbm_gbs",
                "kernel": r.get("kernel_name", "frontend kernel (framing+window+FFT+mel+log+DCT)"),
                "kernel_ms": r["kernel_ms"], "algorithmic_bytes_per_launch": ALGO_BYTES_PER_UTT * BATCH}
    if workload in ("tdnn", "wav2xvec"):
        ms = r["ms"] / r["steps"] if workload == "tdnn" else r["tdnn_ms"]
        flops = r["flops"] / r["steps"] if workload == "tdnn" else r["flops"]
        achieved = flops / (ms * 1e-3) / 1e12
        traffic, src = measured_traffic("tdnn_stack")
        return {"bound": "tensor", "achieved": achieved, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                "frac": achieved / pk["tf_sustained"], "peak_burst": pk["tf_burst"],
                "frac_of_burst": achieved / pk["tf_burst"], "traffic": traffic, "traffic_source": src,
                "peak_source": pk["src"] + " bf16_tflops_sustained (kernels timed inside a long step); burst beside it",
                "kernel": "tdnn_tc_pair_kernel x5 + tdnn_tc_kernel<STATS> (tcgen05 implicit-GEMM stack incl. pre-pass / finalize launches)",
                "kernel_ms": ms, "algorithmic_flops_per_launch": flops}
    achieved = r["score_bytes"] / (r["score_ms"] * 1e-3) / 1e9
    traffic, src = measured_traffic("plda_score")
    return {"bound": "hbm", "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s", "frac": achieved / pk["hbm"],
            "traffic": traffic, "traffic_source": src, "peak_source": pk["src"] + " hbm_gbs",
            "kernel": "tdnn_tc_kernel<F32> as PLDA score GEMM (fp16 hi/lo split, K = 3*dim) + split / A_i / B_j kernels",
            "kernel_ms": r["score_ms"], "algorithmic_bytes_per_launch": r["score_bytes"],
            "tensor_tflops": r["flops"] * 3 / (r["score_ms"] * 1e-3) / 1e12}


STAGES = {"frontend": stage_frontend, "wav2xvec": stage_wav2xvec, "tdnn": stage_tdnn, "plda": stage_plda}


def pcm16_summary(r, pk, steps):
    """Extra figures for raw int16 PCM input (not the API-compatible headline: reported beside it)."""
    p = r["pcm16"]
    out = {"note": "same workload fed as int16 PCM (kernel converts); separate from the float32 headline",
           "e2e_value": r["units"] / (p["ms_e2e"] * 1e-3), "e2e_ms_per_step": p["ms_e2e"] / steps,
           "h2d_bytes_per_step": p["h2d"]}
    if "ms" in p:
        out["value"] = r["units"] / (p["ms"] * 1e-3)
        out["ms_per_step"] = p["ms"] / steps
    if "kernel_ms" in p:
        gbs = p["algo_bytes"] / (p["kernel_ms"] * 1e-3) / 1e9
        out["roofline"] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                           "kernel_ms": p["kernel_ms"], "algorithmic_bytes_per_launch": p["algo_bytes"]}
    return out


def stage_summary(name, st, pk):
    roof = roofline_for(name, st, pk)
    out = {"value": st["units"] / (st["ms"] * 1e-3), "unit": WORKLOAD_UNIT[name],
           "ms_per_step": st["ms"] / st["steps"], "launches_per_step": st["launches"] // st["steps"],
           "e2e_value": st["units"] / (st["ms_e2e"] * 1e-3),
           "roofline": {k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac", "kernel_ms", "traffic")}}
    if "frac_of_burst" in roof:
        out["roofline"]["frac_of_burst"] = roof["frac_of_burst"]
    if name == "plda":
        out.update({"n": st["n"], "allgather_ms": st["allgather_ms"], "allgather_bytes": st["allgather_bytes"],
                    "score_ms": st["score_ms"], "parity_max_rel": st["parity_max_rel"],
                    "bf16_scores": {"score_ms": st["score16_ms"],
                                    "scores_per_sec": float(st["n"]) * st["n"] / (st["score16_ms"] * 1e-3),
                                    "hbm_write_gbs": st["score_bytes"] / 2 / (st["score16_ms"] * 1e-3) / 1e9,
                                    "note": "compact output (2 bytes per trial), reported separately from the "
                                            "API-compatible float32 figure"},
                    "best_match": {"ms": st["top1_ms"],
                                   "trials_per_sec": float(st["n"]) * (st["score_bytes"] / 4 / st["n"]) / (st["top1_ms"] * 1e-3),
                                   "note": "best enrolled vector per test vector (score + index), no score matrix written; "
                                           "reported separately from the API-compatible float32 figure"},
                    "parity": "sampled 1024 x 1024 sub-block per rank vs the float64 oracle, |d| / max(|s|, 1), max over ranks"})
    if "vad_keep" in st:
        out["vad_keep_fraction"] = st["vad_keep"]
    if "pcm16" in st:
        out["int16_input"] = pcm16_summary(st, pk, st["steps"])
    return out


def run_ours(args):
    h = Harness(args)
    pk = peaks()
    w = args.workload
    r = STAGES[w](h, args.steps, args.warmup, dump=args.dump_outputs is not None)
    line = None
    if h.rank == 0 and args.dump_outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in r["outputs"].items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    if h.rank == 0:
        e2e_s = r["ms_e2e"] * 1e-3 / args.steps
        line = {
            "metric": WORKLOAD_METRIC[w], "value": r["units"] / (r["ms"] * 1e-3), "unit": WORKLOAD_UNIT[w],
            "n_gpus": h.world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": r["ms"] / args.steps, "higher_is_better": True,
            "scaling": "strong" if w == "plda" else "weak",
            "vs_baseline": None, "dtype": {"frontend": "f32", "plda": "f32 (fp16 hi/lo split products, fp32 accumulate)"}.get(
                w, "bf16 operands, fp32 accumulate (front-end f32)"),
            "data": "synthetic", "config": workload_config(w, h.world),
            "roofline": roofline_for(w, r, pk),
            "e2e": {"value": r["units"] / (r["ms_e2e"] * 1e-3), "unit": WORKLOAD_UNIT[w],
                    "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"], "ms_per_step": r["ms_e2e"] / args.steps,
                    "h2d_gbs_per_rank": r["h2d"] / e2e_s / 1e9},
            "gpu_launches": r["launches"], "clocks": r["clocks"],
        }
        if "h2d_ceiling" in r:
            line["e2e"]["h2d_ceiling"] = r["h2d_ceiling"]
            line["e2e"]["h2d_frac_of_ceiling"] = line["e2e"]["h2d_gbs_per_rank"] / r["h2d_ceiling"]["per_rank_min_gbs"]
        if "vad_keep" in r:
            line["config"]["vad_keep_fraction"] = r["vad_keep"]
        if "pcm16" in r:
            line["int16_input"] = pcm16_summary(r, pk, args.steps)
        if w == "plda":
            line.update({"allgather_ms": r["allgather_ms"], "parity_max_rel": r["parity_max_rel"]})
    # the other BASELINE configs, measured in the same run (default workload only).  Every rank runs them (the
    # PLDA stage is the sharded one: its all-gather needs all ranks); rank 0 reports.
    if w == DEFAULT_WORKLOAD and not args.no_stages:
        stages = {}
        plan = [("frontend", {}), ("plda", {"n": 50000})]
        if h.world == 1:
            plan.insert(1, ("tdnn", {}))
        for name, kw in plan:
            try:
                st = STAGES[name](h, max(3, args.steps // 4), 3, **kw)
                stages[name] = stage_summary(name, st, pk)
            except Exception as e:                              # a stage must never take the headline line down
                stages[name] = {"error": f"{type(e).__name__}: {e}"}
                if h.world > 1:
                    raise                                       # ... but ranks must not diverge inside a collective
        if h.rank == 0:
            line["stages"] = stages
    if h.rank == 0:
        if h.world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(w, 1)           # bounded sample, 1 thread, rank 0, N = 1 only
        emit_json(line)
    if h.world > 1:
        h.dist.barrier()
        h.dist.destroy_process_group()


_JSON_FD = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line.  Libraries write there too (NCCL_DEBUG=VERSION prints its banner to
    stdout and ignores NCCL_DEBUG_FILE at that level), so file descriptor 1 is pointed at stderr for the whole run
    and the JSON line goes to a private duplicate of the original stdout."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit_json(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(STAGES))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stages", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline workload computed (rank 0) as DIR/<name>.npy, "
                         "float32 / float64, at most 64 MB in all (larger outputs: a fixed, seeded sample of rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
