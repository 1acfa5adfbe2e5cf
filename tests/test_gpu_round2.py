"""
GPU parity cases added in round 2 (VERDICT r01 "next round" item 1 and the ADVICE findings), all through the
public layer / model API (C-ABI underneath) against the CPU oracle:

  * BASELINE config 4 sample: 64 gated-noise utterances as ONE batch at the default (bf16, tcgen05) precision --
    VAD mask bit-exact per utterance, x-vector cosine >= 0.9999 per utterance;
  * BASELINE config 3 shape: 512 x 300 frames through the bf16 stack, 16 rows against the oracle;
  * CALLHOME (8 kHz, 23-dim): front-end against the oracle, the stack of 0006_callhome_diarization_v2_1a.yml against
    the oracle's sequential model;
  * measured MFCC / fbank margins of every golden configuration, written as JSON (profiles/r02_parity.json is the
    committed copy of a GPU-box run);
  * the wav -> x-vector step has no host synchronisation: it is captured in a CUDA graph and replayed;
  * set_weights() after a forward is honoured (keras semantics);
  * NCCL-style sharded PLDA: two ranks on one GPU (gloo carrying the CUDA tensors), each scoring its enrolled-column
    shard with the real kernels, against the float64 oracle;
  * VAD at 1 M frames: fixed-order fp32 mean in the oracle vs fp64 in the kernel.
"""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, golden_path, load_golden, read_wav_int16, rmse
import helpers
from oracle import ktf_oracle as O
from test_gpu_tdnn_plda import cosine, extractor_cfg, sitw_layers_for_oracle, synthetic_plda

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ktf():
    import kaldi_tflite_b200 as k
    return k


def _gated_noise(n_utt, seed):
    import bench
    return bench.gated_noise_np(n_utt, seed)


# ------------------------------------------------------------------------------------------------
# BASELINE config 4 sample
# ------------------------------------------------------------------------------------------------

def test_cfg4_gated_noise_batch_default_precision(ktf):
    from kaldi_tflite_b200.layers import tdnn as _t
    assert _t.DEFAULT_PRECISION == "bf16"          # the drop-in call runs on the tcgen05 stack
    cfg = extractor_cfg()
    ext = ktf.models.XvectorExtractor(cfg, seed=0, allow_random_init=True)
    wav = _gated_noise(64, seed=4242)
    n0 = ktf.launch_count()
    got, inter = ext(wav, return_intermediate=True)
    assert ktf.launch_count() - n0 <= 24
    assert ext.xvec._stack is not None             # whole network as ONE tcgen05 stack
    assert got.shape == (64, 128)
    mask = inter["mask"].cpu().numpy().reshape(64, -1)
    layers = sitw_layers_for_oracle(ext.xvec)
    worst, keep = 1.0, []
    for b in range(64):
        want, ointer = O.xvector_extractor(wav[b], cfg, layers, ext.xvecGlobalMean, ext.ldaTransform,
                                           return_intermediate=True)
        omask = np.zeros(mask.shape[1], np.float32)
        omask[ointer["vad_idx"][:, 1]] = 1
        assert np.array_equal(mask[b], omask), b                 # bit-exact per utterance
        c = cosine(got[b], want)
        assert c >= 0.9999, (b, c)
        worst = min(worst, c)
        keep.append(float(omask.mean()))
    assert 0.4 < np.mean(keep) < 0.95                            # the gate really removes frames
    print(f"cfg4 sample: 64 utterances, mask exact, worst cosine {worst:.7f}, mean keep {np.mean(keep):.3f}")


# ------------------------------------------------------------------------------------------------
# BASELINE config 3 shape
# ------------------------------------------------------------------------------------------------

def test_cfg3_shape_stack_bf16(ktf):
    import torch
    import yaml
    with open(os.path.join(ROOT, "data", "kaldi_models", "configs", "0008_sitw_v2_1a.yml")) as f:
        cfg = yaml.safe_load(f)["model_config"]
    mdl = ktf.models.SequentialFromConfig(cfg, None, "cmvn2xvec", seed=0)       # default precision
    g = torch.Generator(device="cuda").manual_seed(1234)
    B, Tn = 512, 300
    feats = torch.randn((B, Tn, 30), generator=g, device="cuda")
    out = mdl(feats)
    assert mdl._stack is not None
    assert tuple(out.shape) == (B, 1, 512)
    assert bool(torch.isfinite(out).all())
    layers = sitw_layers_for_oracle(mdl)
    rows = [0, 1, 2, 3, 63, 64, 127, 128, 255, 256, 300, 383, 448, 509, 510, 511]
    x = feats[rows].cpu().numpy()
    want = O.sequential(x, layers)
    got = out[rows].cpu().numpy()
    for i, b in enumerate(rows):
        assert cosine(got[i], want[i]) >= 0.9999, (b, cosine(got[i], want[i]))


# ------------------------------------------------------------------------------------------------
# CALLHOME: 8 kHz / 23-dim front-end and the stack of 0006_callhome_diarization_v2_1a.yml
# ------------------------------------------------------------------------------------------------

CALLHOME_MFCC = dict(num_mfccs=23, num_mels=23, sample_frequency=8000.0, low_freq_cutoff=20.0,
                     high_freq_cutoff=3700.0)          # the recipe's conf/mfcc.conf


def _wav_8k():
    wav = read_wav_int16(golden_path("librispeech_2.wav"))
    return np.ascontiguousarray(0.5 * (wav[0:-1:2] + wav[1::2]))[:120000]    # 15 s at 8 kHz


def test_callhome_frontend_vs_oracle(ktf):
    wav = _wav_8k()[None]
    for snip in (True, False):
        fr = ktf.layers.Framing(25.0, 10.0, 8000.0, dynamic_input_shape=True, snip_edges=snip)
        assert fr.frameWidth == 200 and fr.frameShift == 80
        got = ktf.layers.MFCC(**CALLHOME_MFCC)(fr(wav))
        x = wav if snip else O.pad_waveform(wav, 200, 80)
        frames = O.framing(x, 25.0, 10.0, 8000.0)
        truth = O.mfcc(frames, precise=True, **CALLHOME_MFCC)
        ora = O.mfcc(frames, **CALLHOME_MFCC)
        assert got.shape == truth.shape and got.shape[-1] == 23
        floor = float(np.max(np.abs(ora - truth)))
        d = float(np.max(np.abs(got - truth)))
        # 200-sample frames run on the generic radix-2 kernel.  The decimated file has frames whose mel energies span
        # 78 dB (log-mel 6.7 .. 24.7): there the weakest bins carry the float32 rounding of the strongest ones and the
        # radix-2 FFT (7 butterfly levels + the real-FFT untangling) is about 1.3x noisier than pocketfft -- measured
        # max-abs 1.22e-3 / 1.18e-3 against 1.09e-3 / 0.76e-3 of the float32 oracle, p99.9 4.3e-4 / 4.7e-4
        assert d < max(1e-3, 2.0 * floor), (snip, d, floor)
        assert float(np.quantile(np.abs(got - truth), 0.999)) < 6e-4
        assert rmse(truth, got) < 5e-5
        assert rmse(ora, got) < 1e-4
    # VAD + CMVN on the 8 kHz features (the recipe's vad.conf / sliding CMVN, window 300)
    feats = ktf.layers.MFCC(**CALLHOME_MFCC)(ktf.layers.Framing(25.0, 10.0, 8000.0, dynamic_input_shape=True)(wav))
    vkw = dict(energy_mean_scale=0.5, energy_threshold=5.5, frames_context=2, proportion_threshold=0.12)
    assert np.array_equal(ktf.layers.VAD(return_indexes=False, **vkw)(feats), O.vad(feats, return_indexes=False, **vkw))
    # against the float64 evaluation of the same windows: the float32 oracle carries the rounding of a 1498-frame
    # float32 cumsum (cmvn.py:172), which alone is ~1e-5 on features of magnitude 20
    from test_gpu_frontend import _cmvn_f64
    truth = _cmvn_f64(feats, 300, False, "SAME")
    got = ktf.layers.CMVN(window=300)(feats)
    assert rmse(truth, got) < 1e-5
    assert rmse(truth, got) <= 1.5 * rmse(truth, O.cmvn(feats, window=300))


@pytest.mark.parametrize("precision,bar", [("f32", 0.99999), (None, 0.9999)])
def test_callhome_stack_vs_oracle(ktf, precision, bar):
    import yaml
    with open(os.path.join(ROOT, "data", "kaldi_models", "configs", "0006_callhome_diarization_v2_1a.yml")) as f:
        cfg = yaml.safe_load(f)
    assert cfg["sample_rate"] == 8000
    mdl = ktf.models.SequentialFromConfig(cfg["model_config"], None, "callhome", precision=precision, seed=3)
    rng = np.random.default_rng(103)
    for l in mdl.layers:
        if isinstance(l, ktf.layers.BatchNorm):
            d = l.gamma.shape[0]
            l.set_weights([np.float32(1.0), rng.standard_normal(d).astype(np.float32) * 0.1,
                           rng.random(d).astype(np.float32) + 0.5])
    layers = sitw_layers_for_oracle(mdl)
    chunk = load_golden("tdnn.npz")["callhome_chunk_mfcc"].astype(np.float32)         # (1, 150, 23), the reference's input
    feats = ktf.layers.CMVN(window=300)(ktf.layers.MFCC(**CALLHOME_MFCC)(
        ktf.layers.Framing(25.0, 10.0, 8000.0, dynamic_input_shape=True)(_wav_8k()[None])))
    for x in (chunk, feats[:, :400], feats[:, 400:1131]):
        got = mdl(x)
        want = O.sequential(x, layers)
        assert got.shape == want.shape == (1, 1, 128)
        assert cosine(got, want) >= bar, (precision, x.shape, cosine(got, want))
    if precision is None:
        assert mdl._stack is not None      # 23-dim input: materialised splice, still the tcgen05 stack


# ------------------------------------------------------------------------------------------------
# measured margins (VERDICT r01: "the measured worst case per config is recorded nowhere")
# ------------------------------------------------------------------------------------------------

def _margins(got, truth, ora):
    e = np.abs(np.asarray(got, np.float64) - truth)
    f = np.abs(np.asarray(ora, np.float64) - truth)
    return {"max_abs": float(e.max()), "p999": float(np.quantile(e, 0.999)), "rmse": rmse(truth, got),
            "f32_oracle_max_abs": float(f.max()), "f32_oracle_p999": float(np.quantile(f, 0.999))}


def test_record_parity_margins(ktf, tmp_path):
    """Every golden MFCC / fbank configuration + the BASELINE config-2 synthetic row: error of the kernel and of
    the float32 oracle against the float64 evaluation of the same formulas.  Gate (DESIGN.md section 5), per config:
    max-abs <= max(1e-3, 1.25 x the float32 oracle's own max-abs error), p99.9 <= max(1e-3, the float32 oracle's p99.9):
    1e-3 wherever a float32 evaluation of the chain stays clear of it, never more than 25 % worse than the float32
    restatement of the reference where that one touches 1e-3 itself.  Both numbers are written out per config."""
    import torch
    fe = load_golden("frontend.npz")
    wav = fe["wav_trimmed"].astype(np.float32)
    report = {"tolerance": "1e-3 absolute on log features where a float32 evaluation meets it, else 1.25 x the float32 "
                           "oracle's own max-abs error (stated per config below)", "mfcc": {}, "fbank": {}}
    for key in sorted(fe.files):
        if key.startswith("mfcc_conf_"):
            idx = key.split("_")[-1]
            cfg = helpers.mfcc_conf_to_kwargs(str(fe[key]))
            x = wav.reshape(1, -1)
            fr = cfg["framing"]
            size, shift, _ = O.frame_params(fr["frame_length_ms"], fr["frame_shift_ms"], fr["sample_frequency"])
            if not cfg["snip_edges"]:
                x = O.pad_waveform(x, size, shift)
            x = np.ascontiguousarray(x, np.float32)
            got = ktf.layers.MFCC(**cfg["mfcc"])(ktf.layers.Framing(dynamic_input_shape=True, **fr)(x))
            frames = O.framing(x, **fr)
            m = _margins(got, O.mfcc(frames, precise=True, **cfg["mfcc"]), O.mfcc(frames, **cfg["mfcc"]))
            m["rmse_vs_kaldi"] = rmse(fe[f"mfcc_{idx}"], got)
            m["frame_width"] = int(size)
            report["mfcc"][idx] = m
        elif key.startswith("fbank_conf_"):
            idx = key.split("_")[-1]
            cfg = helpers.fbank_conf_to_kwargs(str(fe[key]))
            if not cfg["fbank"].get("use_log_fbank", True):
                continue
            x = wav.reshape(1, -1)
            fr = cfg["framing"]
            size, shift, _ = O.frame_params(fr["frame_length_ms"], fr["frame_shift_ms"], fr["sample_frequency"])
            if not cfg["snip_edges"]:
                x = O.pad_waveform(x, size, shift)
            x = np.ascontiguousarray(x, np.float32)
            frames = ktf.layers.Framing(dynamic_input_shape=True, **fr)(x)
            got = ktf.layers.FilterBank(**cfg["fbank"])(ktf.layers.Windowing(return_energy=False, **cfg["windowing"])(frames))
            fnp = O.framing(x, **fr)
            truth = O.filterbank(O.windowing(fnp, return_energy=False, precise=True, **cfg["windowing"]), precise=True,
                                 **cfg["fbank"])
            ora = O.filterbank(O.windowing(fnp, return_energy=False, **cfg["windowing"]), **cfg["fbank"])
            m = _margins(got, truth, ora)
            m["rmse_vs_kaldi"] = rmse(fe[f"fbank_{idx}"], got)
            report["fbank"][idx] = m
    # BASELINE config 2 synthetic rows (seed 1234, randn * 3000), 8 utterances of the 1024
    g = torch.Generator(device="cuda").manual_seed(1234)
    syn = (torch.randn((8, 160000), generator=g, device="cuda") * 3000).clamp(-32767, 32767)
    got = ktf.layers.MFCC(num_mfccs=30, num_mels=30)(ktf.layers.Framing(dynamic_input_shape=True)(syn)).cpu().numpy()
    frames = O.framing(syn.cpu().numpy(), 25, 10, 16000)
    report["cfg2_synthetic"] = _margins(got, O.mfcc(frames, precise=True, num_mfccs=30, num_mels=30),
                                        O.mfcc(frames, num_mfccs=30, num_mels=30))
    # BASELINE config 1 file (22.5 s of speech), SITW front-end
    cfg1 = extractor_cfg()["mfcc"]
    w1 = read_wav_int16(golden_path("librispeech_2.wav"))[None]
    got = ktf.layers.MFCC(**cfg1)(ktf.layers.Framing(dynamic_input_shape=True)(w1))
    frames = O.framing(w1, 25, 10, 16000)
    report["cfg1_librispeech_2"] = _margins(got, O.mfcc(frames, precise=True, **cfg1), O.mfcc(frames, **cfg1))

    rows = list(report["mfcc"].values()) + list(report["fbank"].values()) + [report["cfg2_synthetic"],
                                                                            report["cfg1_librispeech_2"]]
    report["summary"] = {
        "configs": len(rows),
        "worst_max_abs": max(r["max_abs"] for r in rows),
        "worst_p999": max(r["p999"] for r in rows),
        "configs_where_f32_oracle_exceeds_1e-3": sorted(
            k for k, r in report["mfcc"].items() if r["f32_oracle_max_abs"] > 1e-3),
        "configs_where_kernel_exceeds_1e-3": sorted(k for k, r in report["mfcc"].items() if r["max_abs"] > 1e-3),
    }
    out_dir = str(tmp_path)
    with open(os.path.join(out_dir, "r02_parity.json"), "w") as f:
        json.dump(report, f, indent=1, sort_keys=True)
    print("parity summary:", json.dumps(report["summary"]))
    for r in rows:
        r["gate_max_abs"] = max(1e-3, 1.25 * r["f32_oracle_max_abs"])
        r["gate_p999"] = max(1e-3, r["f32_oracle_p999"])
    with open(os.path.join(out_dir, "r02_parity.json"), "w") as f:
        json.dump(report, f, indent=1, sort_keys=True)
    for kind in ("mfcc", "fbank"):
        for idx, r in report[kind].items():
            assert r["max_abs"] <= r["gate_max_abs"], (kind, idx, r)
            assert r["p999"] <= r["gate_p999"], (kind, idx, r)
    for name in ("cfg2_synthetic", "cfg1_librispeech_2"):
        r = report[name]
        assert r["max_abs"] <= r["gate_max_abs"] and r["p999"] <= r["gate_p999"], (name, r)
    # the north-star 1e-3 holds outright on the large majority of configurations, and everywhere at the 99.9th percentile
    # except where the float32 oracle itself is above it
    assert sum(r["max_abs"] <= 1e-3 for r in rows) >= 0.85 * len(rows)


# ------------------------------------------------------------------------------------------------
# no host synchronisation on the wav -> x-vector step
# ------------------------------------------------------------------------------------------------

def test_wav2xvec_step_is_cuda_graph_capturable(ktf):
    import torch
    ext = ktf.models.XvectorExtractor(extractor_cfg(), seed=0, allow_random_init=True)
    wav = torch.from_numpy(_gated_noise(16, seed=77)).cuda()
    eager = ext(wav).clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):                          # warm-up on the capture stream (workspaces reach their size)
            ext(wav)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    n0 = ktf.launch_count()
    with torch.cuda.graph(graph):                   # any host synchronisation inside would abort the capture
        out = ext(wav)
    per_step = ktf.launch_count() - n0
    assert 0 < per_step <= 24
    wav2 = torch.from_numpy(_gated_noise(16, seed=78)).cuda()
    want2 = ext(wav2).clone()
    torch.cuda.synchronize()
    wav.copy_(wav2)                                 # new audio (different VAD decisions) through the SAME graph
    graph.replay()
    torch.cuda.synchronize()
    # (the pooled statistics are accumulated with float atomics: equal up to summation order, not bit for bit)
    assert torch.allclose(out, want2, rtol=0.0, atol=1e-3)
    assert float((out - eager).abs().max()) > 20 * float((out - want2).abs().max())   # it really is the new audio


def test_fused_vad_cmvn_splice_prepass_equals_separate_kernels(ktf):
    """ktf_tdnn_stack_forward_vad (one gather + CMVN + splice kernel in front of the GEMMs) against the separate
    vad_gather / cmvn / splice kernels, on uniform and ragged batches, and against the oracle."""
    cfg = extractor_cfg()
    ext = ktf.models.XvectorExtractor(cfg, seed=0, allow_random_init=True)
    wav = read_wav_int16(golden_path("librispeech_2.wav"))
    noise = _gated_noise(6, seed=11)
    batches = [noise, [wav[:80000], wav[80000:200000], noise[0][:40000], wav[150000:], wav[:8000], noise[1]]]
    layers = sitw_layers_for_oracle(ext.xvec)
    for x in batches:
        ext.fusePrepass = True
        n0 = ktf.launch_count()
        fused = ext(x)
        n_fused = ktf.launch_count() - n0
        ext.fusePrepass = False
        n0 = ktf.launch_count()
        separate = ext(x)
        n_sep = ktf.launch_count() - n0
        assert n_fused == n_sep - 2                    # gather, CMVN and splice became one launch
        for b in range(len(x)):
            assert cosine(fused[b], separate[b]) > 0.999995, b
            want = O.xvector_extractor(x[b], cfg, layers, ext.xvecGlobalMean, ext.ldaTransform)
            assert cosine(fused[b], want) >= 0.9999, b
    ext.fusePrepass = True
    # an utterance shorter than the CMVN window (global mean branch, cmvn.py:214-222) and a batch of one
    short = ext(wav[:30000])
    want = O.xvector_extractor(wav[:30000], cfg, layers, ext.xvecGlobalMean, ext.ldaTransform)
    assert cosine(short, want) >= 0.9999


def test_set_weights_after_forward_is_applied(ktf):
    import yaml
    with open(os.path.join(ROOT, "data", "kaldi_models", "configs", "0008_sitw_v2_1a.yml")) as f:
        cfg = yaml.safe_load(f)["model_config"]
    x = load_golden("tdnn.npz")["sitw_chunk_mfcc"].astype(np.float32)
    for precision in ("f32", None):
        mdl = ktf.models.SequentialFromConfig(cfg, None, "m", precision=precision, seed=0)
        before = mdl(x)
        layer = mdl.get_layer("tdnn3.affine")
        k, b = layer.get_weights()
        layer.set_weights([k * 0.5, b + 0.25], fmt="tensorflow")
        bn = mdl.get_layer("tdnn4.batchnorm")
        d = bn.gamma.shape[0]
        bn.set_weights([np.float32(0.9), np.full(d, 0.05, np.float32), np.full(d, 1.3, np.float32)])
        after = mdl(x)                                              # no invalidate() call
        want = O.sequential(x, sitw_layers_for_oracle(mdl))
        assert cosine(after, want) >= (0.99999 if precision == "f32" else 0.9999)
        assert cosine(before, want) < 0.999


# ------------------------------------------------------------------------------------------------
# dither drawn inside the kernel (windowing.py:182-183)
# ------------------------------------------------------------------------------------------------

def test_dither_in_kernel_is_per_framed_sample(ktf):
    """The reference adds dither * N(0, 1) to the FRAMED tensor: overlapping frames do not share noise.  On silence,
    with a rectangular window and no DC removal / pre-emphasis, the windowed frames ARE the noise."""
    from kaldi_tflite_b200 import _native
    x = np.zeros((4, 16000), np.float32)
    fr = ktf.layers.Framing(dynamic_input_shape=True)
    win = ktf.layers.Windowing(window_type="rectangular", dither=2.0, remove_dc_offset=False,
                               preemphasis_coefficient=0.0, return_energy=False)
    _native.lib().ktf_set_dither_seed(1234)
    a = win(fr(x))
    assert a.shape == (4, 98, 400)
    z = a / 2.0
    assert abs(float(z.mean())) < 0.01 and abs(float(z.std()) - 1.0) < 0.01
    assert abs(float((z ** 3).mean())) < 0.03 and abs(float((z ** 4).mean()) - 3.0) < 0.1     # skewness, kurtosis
    # frames t and t + 1 overlap in 240 samples: the shared samples must carry independent draws
    shared_a, shared_b = z[:, :-1, 160:], z[:, 1:, :240]
    corr = float(np.mean(shared_a * shared_b))
    assert abs(corr) < 0.01, corr
    # neighbouring samples / lanes are uncorrelated too
    assert abs(float(np.mean(z[..., 1:] * z[..., :-1]))) < 0.01
    # a new call draws new noise; the same seed reproduces the sequence of calls
    b = win(fr(x))
    assert abs(float(np.mean(a * b))) / 4.0 < 0.01
    _native.lib().ktf_set_dither_seed(1234)
    assert np.array_equal(win(fr(x)), a)
    # pre-emphasis sees the DITHERED neighbour: y[i] = n[i] - 0.97 n[i-1] has variance (1 + 0.97^2) * dither^2
    pre = ktf.layers.Windowing(window_type="rectangular", dither=1.0, remove_dc_offset=False,
                               preemphasis_coefficient=0.97, return_energy=False)(fr(x))
    assert abs(float(pre[..., 1:].var()) - (1.0 + 0.97 ** 2)) < 0.03
    # MFCC of a loud signal barely moves with dither 1 (and the default YAML value runs end to end)
    rng = np.random.default_rng(0)
    loud = (rng.standard_normal((2, 16000)) * 3000).astype(np.float32)
    m0 = ktf.layers.MFCC(num_mfccs=30, num_mels=30)(fr(loud))
    m1 = ktf.layers.MFCC(num_mfccs=30, num_mels=30, dither=1.0)(fr(loud))
    assert 0.0 < float(np.max(np.abs(m1 - m0))) < 0.05
    m16 = ktf.layers.MFCC(num_mfccs=30, num_mels=30, dither=1.0)(fr(loud.astype(np.int16)))
    assert float(np.max(np.abs(m16 - m0))) < 0.05


# ------------------------------------------------------------------------------------------------
# sharded PLDA, two ranks on one GPU
# ------------------------------------------------------------------------------------------------

def _run_shard_workers(tmp_path, extra=()):
    worker = os.path.join(ROOT, "tests", "plda_shard_worker.py")
    port = 29500 + (os.getpid() % 2000) + len(extra)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, worker, str(tmp_path), *extra], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for rank, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {rank} failed:\n{o}"
    for rank in range(2):
        with open(os.path.join(str(tmp_path), f"rank{rank}.json")) as f:
            r = json.load(f)
        assert r["ok"], r
        assert r["max_rel"] <= 1e-3, r
        assert r["launches"] > 0


def test_plda_sharded_two_ranks_vs_oracle(tmp_path):
    _run_shard_workers(tmp_path)


def test_plda_sharded_two_gpus_nccl_async_allgather(tmp_path):
    """The NCCL path of parallel.plda_score_sharded: ONE asynchronous all-gather, the local rows scored underneath it;
    even shards (1500 test vectors) and ragged ones (1501: padded gather + compaction).  Needs two GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _run_shard_workers(tmp_path, ("nccl", "1500"))
    _run_shard_workers(tmp_path, ("nccl", "1501"))


def _run_cabi_workers(tmp_path, nranks):
    worker = os.path.join(ROOT, "tests", "cabi_plda_worker.py")
    procs = [subprocess.Popen([sys.executable, worker, str(r), str(nranks), str(r), str(tmp_path)],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(nranks)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r} failed:\n{o}"
    res = []
    for r in range(nranks):
        with open(os.path.join(str(tmp_path), f"cabi_rank{r}.json")) as f:
            res.append(json.load(f))
    return res


def test_cabi_context_and_collective_without_torch(tmp_path):
    """SURVEY 8b: ktf_ctx_* / ktf_nccl_allgather_xvec -- the sharded PLDA step driven by ctypes alone (no torch in the
    worker process).  One rank always; two ranks over NCCL when the box has two GPUs."""
    import torch
    (r,) = _run_cabi_workers(tmp_path, 1)
    assert r["max_rel"] <= 1e-3 and r["launches"] > 0 and not r["torch_loaded"], r
    if torch.cuda.device_count() >= 2:
        two = _run_cabi_workers(tmp_path, 2)
        for r in two:
            assert r["max_rel"] <= 1e-3 and r["nranks"] == 2 and not r["torch_loaded"], r


def test_plda_compact_bf16_scores(ktf):
    # SURVEY 8f rank 3: the score matrix as bfloat16 (half the HBM write): same fp32-equivalent value rounded once
    import torch
    dim, nt, ne = 128, 777, 1300
    mean, Tm, psi = synthetic_plda(dim)
    rng = np.random.default_rng(23)
    x = rng.standard_normal((nt + ne, dim))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(dim)).astype(np.float32)
    layer = ktf.layers.PLDA(dim, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    u = layer.transformVector(torch.from_numpy(x).cuda())
    full = layer.logLikelihoodRatio(u[:nt], u[nt:])
    got = layer.logLikelihoodRatio(u[:nt], u[nt:], score_dtype=torch.bfloat16)
    assert got.dtype is torch.bfloat16 and tuple(got.shape) == (nt, ne)
    assert torch.equal(got, full.to(torch.bfloat16))            # exactly the fp32 score rounded to nearest-even
    uo = O.plda_transform(x, mean, Tm, psi, dtype=np.float64)
    want = O.plda_llr(uo, psi)[:nt, nt:]
    err = np.abs(got.float().cpu().numpy() - want)
    assert np.all(err <= 2.0 ** -8 * np.abs(want) + 1e-3)
    # into a strided, preallocated block (the sharded path writes column blocks)
    big = torch.zeros((nt, ne + 40), device="cuda", dtype=torch.bfloat16)
    layer.logLikelihoodRatio(u[:nt], u[nt:], out=big[:, 8:8 + ne])
    assert torch.equal(big[:, 8:8 + ne], got) and float(big[:, :8].abs().max()) == 0.0
    with pytest.raises(ValueError):
        ktf.layers.PLDA(dim, mean, Tm, psi, dtype=np.float64).logLikelihoodRatio(u.double(), score_dtype=torch.bfloat16)


# ------------------------------------------------------------------------------------------------
# VAD at scale
# ------------------------------------------------------------------------------------------------

def test_plda_best_match_equals_score_matrix(ktf):
    """SURVEY 8f rank 3, top-k = 1: ktf_plda_score_top1 / PLDA.bestMatch returns, per test vector, the maximum of the score
    matrix row and the column that attains it -- same arithmetic as the matrix entry (bit-equal), no matrix written --
    and that column is the float64 oracle's best within the 1e-3 score tolerance."""
    import torch
    from test_gpu_tdnn_plda import synthetic_plda
    dim = 128
    mean, Tm, psi = synthetic_plda(dim)
    rng = np.random.default_rng(77)
    x = rng.standard_normal((1037 + 700, dim))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * np.sqrt(dim)).astype(np.float32)
    layer = ktf.layers.PLDA(dim, mean, Tm, psi, dtype=np.float32, return_transformed=False)
    u = layer.transformVector(torch.from_numpy(x).cuda())
    ut, ue = u[:1037].contiguous(), u[1037:].contiguous()
    n0 = ktf.launch_count()
    best, index = layer.bestMatch(ut, ue)
    assert ktf.launch_count() > n0
    full = layer.logLikelihoodRatio(ut, ue)
    torch.cuda.synchronize()
    want = full.max(dim=1).values
    assert torch.equal(best, want)
    assert int(index.min()) >= 0 and int(index.max()) < 700
    assert torch.equal(full[torch.arange(1037, device=full.device), index], want)
    uo = O.plda_transform(x, mean, Tm, psi, dtype=np.float64)
    ref = O.plda_llr(uo, psi)[:1037, 1037:]
    at = ref[np.arange(1037), index.cpu().numpy()]
    assert np.all(ref.max(axis=1) - at <= 1e-3 * np.maximum(np.abs(ref.max(axis=1)), 1.0))
    # all-vs-all on one set (the reference's call()): every vector's best match is found in the same set
    best2, index2 = layer.bestMatch(ut)
    full2 = layer.logLikelihoodRatio(ut)
    torch.cuda.synchronize()
    assert torch.equal(best2, full2.max(dim=1).values)
    assert torch.equal(full2[torch.arange(1037, device=full2.device), index2], best2)


def test_vad_exact_at_one_million_frames(ktf):
    """1024 utterances x 998 frames (BASELINE config 4 shard): the kernel accumulates the per-utterance mean in fp64,
    the oracle in pairwise fp32; the masks must still agree bit for bit on MFCCs of gated noise.  Frames within 1 ulp
    of the threshold would be the only way to differ: count them."""
    import torch
    wav = torch.from_numpy(_gated_noise(256, seed=5)).cuda()
    cfg = extractor_cfg()
    feats = ktf.layers.MFCC(**cfg["mfcc"])(ktf.layers.Framing(dynamic_input_shape=True)(wav))
    feats = feats.repeat(4, 1, 1)[torch.randperm(1024, generator=torch.Generator().manual_seed(1))]
    assert feats.shape[0] * feats.shape[1] >= 1_000_000
    vkw = {k: v for k, v in cfg["vad"].items() if k != "return_indexes"}
    got = ktf.layers.VAD(return_indexes=False, **vkw)(feats).cpu().numpy()
    f = feats.cpu().numpy()
    want = O.vad(f, return_indexes=False, **vkw)
    assert np.array_equal(got, want)
    e = f[..., 0]
    thr = np.float32(vkw["energy_threshold"]) + np.float32(vkw["energy_mean_scale"]) * e.mean(axis=1, dtype=np.float64).astype(np.float32)
    near = np.abs(e - thr[:, None]) <= 4 * np.spacing(np.abs(thr[:, None]))
    print(f"VAD at {e.size} frames: {int(near.sum())} frames within 4 ulp of the threshold; kept {got.mean():.3f}")
