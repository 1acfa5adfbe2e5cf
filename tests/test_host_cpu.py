"""CPU-side checks: Kaldi readers, config plumbing, the C-ABI surface of the built library."""

import ctypes
import json
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_golden, golden_path


def test_readers_nnet3_vs_literals():
    # io/kaldi/nnet3_reader_test.py: binary parse equals the literal fixture (1e-7)
    from kaldi_tflite_b200.io import KaldiNnet3Reader
    g = load_golden("tdnn.npz")
    r = KaldiNnet3Reader(golden_path("tdnn_narrow.final.raw"), True)
    comps = json.loads(str(g["narrow_components"]))
    assert [c["name"] for c in r.components] == [c["name"] for c in comps]
    assert [c["type"] for c in r.components] == [c["type"] for c in comps]
    assert len(r.components) == 16
    for i, c in enumerate(comps):
        for k in c:
            key = f"narrow_c{i}_{k}"
            if key in g.files:
                assert np.allclose(np.asarray(r.components[i][k]), g[key], atol=1e-7), (i, k)
    cfg_lines = [l.strip() for l in json.loads(str(g["narrow_config"]))]
    assert [l.strip() for l in r.config] == cfg_lines
    w = r.getWeights("tdnn1.affine")
    assert w[0].shape == (5, 15) and w[1].shape == (5,)
    rms, mean, var = r.getWeights("tdnn1.batchnorm")
    assert mean.shape == (5,) and float(rms) == 1.0
    assert r.getWeights("tdnn1.relu") == []
    with pytest.raises(KeyError):
        r.getWeights("nope")


def test_readers_plda_and_arrays(tmp_path):
    from kaldi_tflite_b200.io import KaldiPldaReader, ReadKaldiArray, KaldiObjReader
    g = load_golden("plda.npz")
    r = KaldiPldaReader(golden_path("plda.bin"), True)
    assert r.mean.shape == (512,) and r.transformMat.shape == (512, 512) and r.psi.shape == (512,)
    assert np.allclose(r.mean, g["mean"], atol=1e-9)
    assert np.allclose(r.transformMat, g["transform"], atol=1e-9)
    assert np.allclose(r.psi, g["psi"], atol=1e-9)
    vb = ReadKaldiArray(golden_path("sitw_mean.vec"), True)
    vt = ReadKaldiArray(golden_path("sitw_mean.vec.txt"), False)
    assert vb.dtype == np.float32 and np.allclose(vb, vt, atol=5e-8)
    m = ReadKaldiArray(golden_path("sitw_transform.mat"), True)
    assert m.shape == (128, 513)
    txt = tmp_path / "m.txt"
    txt.write_text(" [\n  1 2 3\n  4 5 6 ]\n")
    assert np.array_equal(ReadKaldiArray(str(txt), False), np.float32([[1, 2, 3], [4, 5, 6]]))
    assert np.array_equal(ReadKaldiArray(str(txt), False, np.int32), np.int32([[1, 2, 3], [4, 5, 6]]))
    with pytest.raises(ValueError):
        ReadKaldiArray(str(txt), False, np.uint8)
    with pytest.raises(NotImplementedError):
        KaldiObjReader(str(txt), False)
    # packed symmetric + bool + scalar primitives
    blob = tmp_path / "p.bin"
    blob.write_bytes(b"FP \x04" + np.int32(3).tobytes() + np.float32([1, 2, 3, 4, 5, 6]).tobytes()
                     + b"T" + b"\x08" + np.float64(2.5).tobytes())
    r = KaldiObjReader(str(blob), True)
    assert np.array_equal(r.readPackedMat(), np.float32([[1, 2, 4], [2, 3, 5], [4, 5, 6]]))
    assert r.readBool() is True and r.readDouble() == 2.5


def test_ctor_validation_without_gpu():
    import kaldi_tflite as ktf
    L = ktf.layers
    assert L.Framing(25, 10, 16000).frameWidth == 400
    assert L.Framing(25, 10, 16000).compute_output_shape([4, 160000]) == [4, 998, 400]
    for bad in (dict(frame_length_ms=-1), dict(frame_shift_ms=0), dict(sample_frequency=0)):
        with pytest.raises(ValueError):
            L.Framing(**bad)
    with pytest.raises(ValueError):
        L.MFCC(num_mfccs=31, num_mels=30)
    with pytest.raises(ValueError):
        L.FilterBank(low_freq_cutoff=9000)
    with pytest.raises(ValueError):
        L.Windowing(window_type="nope")
    with pytest.raises(NotImplementedError):
        L.DCT(10, dct_type=3)
    with pytest.raises(ValueError):
        L.VAD(frames_context=-1)
    with pytest.raises(ValueError):
        L.CMVN(window=0)
    with pytest.raises(ValueError):
        L.StatsPooling(1, 0)
    with pytest.raises(ValueError):
        L.StatsPooling(0, 4, input_period=2, output_period=3)
    with pytest.raises(AssertionError):
        L.PLDA(4, np.zeros(3), np.eye(4), np.ones(4))
    t = L.TDNN(8, context=[2, -2, 0])
    assert t.context == [-2, 0, 2] and t.compute_output_shape((1, 10, 3)) == (1, 10, 8)
    assert L.TDNN(8, context=[-2, 0, 2], padding="VALID").compute_output_shape((1, 10, 3)) == (1, 6, 8)
    assert L.CMVN(window=5, padding="VALID").compute_output_shape([1, 12, 3]) == [1, 8, 3]
    cfg = L.MFCC(num_mfccs=30, num_mels=30, high_freq_cutoff=7600.0).get_config()
    assert cfg["num_mfccs"] == 30 and cfg["window_type"] == "povey"
    w = np.arange(2 * 3 * 4, dtype=np.float32).reshape(4, 6)          # U=4, K=2, D=3
    k = L.reshapeKaldiTdnnWeights(w, 4, 2)
    assert k.shape == (1, 2, 3, 4) and k[0, 1, 2, 3] == w[3, 1 * 3 + 2]


def test_tables_match_oracle():
    from kaldi_tflite_b200.layers import dsp
    from oracle import ktf_oracle as O
    for wt in dsp.WINDOW_TYPES:
        assert np.array_equal(dsp.window_function(wt, 400), O.window_function(wt, 400))
    for (nb, lo, hi) in [(23, 20.0, 7600.0), (30, 20.0, 7600.0), (40, 0.0, 8000.0), (80, 64.0, 7936.0)]:
        n1, b1 = dsp.mel_filterbank(400, nb, 16000.0, lo, hi)
        n2, b2 = O.mel_bank(400, nb, 16000.0, hi, lo)
        assert n1 == n2 == 512 and np.array_equal(b1, b2)
    assert np.array_equal(dsp.dct2_matrix(30, 30), O.dct_matrix(30, 30))
    assert np.array_equal(dsp.lifter_coefficients(30, 22), O.lifter_coeffs(30, 22))


def test_sequential_from_config_structure():
    import yaml
    import kaldi_tflite as ktf
    with open(os.path.join(ROOT, "data/kaldi_models/configs/0008_sitw_v2_1a.yml")) as f:
        cfg = yaml.safe_load(f)
    mdl = ktf.models.SequentialFromConfig(cfg["model_config"], None, "cmvn2xvec", seed=0)
    names = [l.name for l in mdl.layers]
    assert names[:3] == ["tdnn1.affine", "tdnn1.relu", "tdnn1.batchnorm"]
    assert names[-2:] == ["stats", "tdnn6.affine"] and len(names) == 17
    assert mdl.get_layer("tdnn5.affine").kernel.shape == (1, 1, 512, 1500)
    assert mdl.get_layer("tdnn6.affine").kernel.shape == (1, 1, 3000, 512)
    with pytest.raises(ValueError):
        ktf.models.SequentialFromConfig({"layers": []})
    with pytest.raises(ValueError):
        ktf.models.SequentialFromConfig({"layers": [{"type": "affine"}]})
    narrow = {"layers": [{"name": "input", "type": "input", "shape": [None, None, 3]}] + [
        {"name": n, "type": ["affine"] + (["relu"] if r else []) + (["batchnorm"] if b else []),
         "cfg": {"units": d, "context": c}} for n, d, c, r, b in __import__("helpers").NARROW_LAYERS]}
    m2 = ktf.models.SequentialFromConfig(narrow, golden_path("tdnn_narrow.final.raw"))
    assert np.allclose(m2.get_layer("tdnn2.batchnorm").moving_mean.shape, (8,))


def test_c_abi_exports_every_declared_symbol():
    from kaldi_tflite_b200 import _native, build
    path = build.build()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "ktf_b200.h")).read()
    declared = set(re.findall(r"\b(ktf_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_native.exported_symbols())
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.ktf_version() == 101


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "kaldi_tflite_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("ktf_oracle", "oracle") or f == "__none__", f


def test_shard_range():
    from kaldi_tflite_b200.parallel import shard_range
    for n in (0, 1, 7, 8, 100000):
        for w in (1, 2, 4, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_bench_reference_arm_prints_one_json_line():
    # bench.py contract: stdout carries exactly ONE JSON line (library chatter such as NCCL's version banner is
    # diverted to stderr); the reference arm runs on the host cores only and names itself.
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["gpu_launches"] == 0
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_output_dump_is_bounded_and_seeded():
    # bench.py --dump-outputs: float32 / float64 host arrays, at most 64 MB in all; a larger output keeps the same
    # seeded, sorted sample of rows on every run
    import importlib.util
    import subprocess
    import sys
    import torch
    spec = importlib.util.spec_from_file_location("ktf_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    big = torch.arange(3000, dtype=torch.float32)[:, None].expand(3000, 8192).contiguous()     # 98 MB, row r holds r
    small = torch.rand(7, 3, dtype=torch.float64)
    a = bench.host_outputs({"big": big, "small": small, "half": torch.ones(4, 2, dtype=torch.bfloat16)})
    b = bench.host_outputs({"big": big, "small": small, "half": torch.ones(4, 2, dtype=torch.bfloat16)})
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_BYTES
    assert a["big"].dtype == np.float32 and a["half"].dtype == np.float32 and a["small"].dtype == np.float64
    assert np.array_equal(a["small"], small.numpy()) and np.array_equal(a["half"], np.ones((4, 2), np.float32))
    rows = a["big"][:, 0]
    assert 0 < len(rows) < 3000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["big"], big.numpy()[rows.astype(np.int64)]) and np.array_equal(a["big"], b["big"])
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *bad], capture_output=True, text=True,
                           timeout=120)
        assert p.returncode == 2 and not p.stdout, (bad, p.stderr)


def test_committed_traffic_summary_feeds_the_bench_roofline():
    """bench.py takes roofline.traffic (DRAM bytes per launch of the dominant kernel) from profiles/r02_traffic.json, which
    scripts/summarize_profiles.py writes from the ncu --set full captures: the file must carry the three kernels the
    bench asks for, and the per-kernel breakdown of the stack must add up."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ktf_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for key in ("frontend", "plda_score", "tdnn_stack"):
        traffic, src = bench.measured_traffic(key)
        assert traffic and traffic > 1e6, key
        assert "profiles/r02_traffic.json" in src
    with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
        d = json.load(f)
    per = d["tdnn_stack"]["per_kernel"]
    assert len(per) == 7
    assert abs(sum(k["dram_bytes"] for k in per) - d["tdnn_stack"]["dram_bytes_per_launch"]) < 1.0
    assert bench.measured_traffic("no such kernel") == (None, None)
