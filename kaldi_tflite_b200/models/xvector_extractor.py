"""
End-to-end wav -> x-vector model with the reference's surface
(/root/reference/kaldi_tflite/lib/models/kaldi/xvector_extractor.py:25-186):
`XvectorExtractorFromConfig(cfgPath, name)`, `XvectorExtractor(cfg, name, chunk_size)`.

Differences that do not change results for the reference's use (batch 1):
  * any batch is accepted: a (B, N) array, a 1-D (N,) array, or a list of 1-D arrays of
    different lengths (ragged).  Utterances are independent (the reference collapses the batch
    at tf.gather_nd, xvector_extractor.py:163-165, so it is batch-1 only).
  * no network: when the Kaldi `final.raw` named by the config is absent the constructor raises
    FileNotFoundError (the reference would download it, :55-65).  Benchmarks and tests that only need the
    ARCHITECTURE pass `allow_random_init=True` (seeded Glorot weights, recorded as `.randomInit`).
"""

import os
import warnings

import numpy as np
import torch
import yaml

from .. import _native as N
from .. import _tensor as T
from ..io import ReadKaldiArray
from ..layers import CMVN, MFCC, VAD, Framing
from .sequential import SequentialFromConfig


def _resolve(path, base_dirs):
    if path is None or os.path.isabs(path) or os.path.exists(path):
        return path
    for b in base_dirs:
        p = os.path.join(b, path)
        if os.path.exists(p):
            return p
    return path


def XvectorExtractorFromConfig(cfgPath: str, name: str = None, **kwargs):
    with open(cfgPath) as f:
        cfg = yaml.safe_load(f)
    ext = cfg["extractor"]
    # paths in the YAML are relative to the repository root (the reference runs from there)
    bases = [os.getcwd(), os.path.dirname(os.path.abspath(cfgPath)),
             os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(cfgPath)), "..", ".."))]
    for key in ("model_config_path", "model_path", "global_mean_path", "lda_matrix_path"):
        ext["xvec"][key] = _resolve(ext["xvec"].get(key), bases)
    return XvectorExtractor(ext, name=name, **kwargs)


class XvectorExtractor:

    def __init__(self, cfg: dict, name: str = None, chunk_size: int = 300, precision: str = None,
                 seed: int = 0, dither: float = None, allow_random_init: bool = False):
        """`precision`: operand precision of the TDNN contractions ("bf16" = tcgen05 engine, the default; "f32" = exact
        SIMT tiles).  `allow_random_init`: accept a missing Kaldi `final.raw` and initialise the TDNN with seeded Glorot
        weights (x-vectors are then meaningless: benchmarks / architecture tests only)."""
        self.name = name
        self.chunkSize = chunk_size
        self.fusePrepass = True      # VAD gather + CMVN + splice as one kernel when the TDNN runs on the tcgen05 stack
        fr = dict(cfg["framing"])
        mf = dict(cfg["mfcc"])
        if dither is not None:
            mf["dither"] = dither
        self.framing = Framing(**fr)
        self.mfcc = MFCC(**mf)
        self.vad = VAD(**cfg["vad"])
        self.cmvn = CMVN(**cfg["cmvn"])

        with open(cfg["xvec"]["model_config_path"], "r") as f:
            nnet3Cfg = yaml.safe_load(f)
        model_path = cfg["xvec"].get("model_path")
        if model_path is None or not os.path.exists(model_path):
            if not allow_random_init:
                raise FileNotFoundError(
                    f"Kaldi nnet3 model '{model_path}' not found (there is no network to download it, "
                    "xvector_extractor.py:55-65); pass allow_random_init=True to run the architecture with seeded "
                    "random weights")
            warnings.warn(f"Kaldi model '{model_path}' not found: the TDNN is randomly initialised (seed {seed}); "
                          "the x-vectors carry no speaker information")
            model_path = None
        self.randomInit = model_path is None
        self.xvec = SequentialFromConfig(nnet3Cfg["model_config"], model_path, "cmvn2xvec",
                                         precision=precision, seed=seed)

        globalMean = ReadKaldiArray(cfg["xvec"]["global_mean_path"], binary=_is_binary(cfg["xvec"]["global_mean_path"]))
        ldaMat = ReadKaldiArray(cfg["xvec"]["lda_matrix_path"], binary=_is_binary(cfg["xvec"]["lda_matrix_path"]))
        self.xvecGlobalMean = np.ascontiguousarray(globalMean, dtype=np.float32)
        self.ldaTransform = np.ascontiguousarray(ldaMat, dtype=np.float32)      # (lda_dim, dim + 1) = [L | o]
        self.ldaOffset = self.ldaTransform[..., -1:].T                           # xvector_extractor.py:133
        self.ldaMat = self.ldaTransform[..., :-1].T                              # :134
        self._dev = None

    # ---- stages, all on ragged (rows, dim) layouts ------------------------------------
    def features(self, wav_flat, sample_offsets):
        """Fused framing + MFCC over a ragged batch -> (rows, num_mfccs), frame offsets (CUDA int64)."""
        fe = self.mfcc.frontend(self.framing.frameWidth, self.framing.frameShift)   # dither: inside the kernel
        snip = self.framing.snipEdges
        lens = np.diff(sample_offsets)
        if len(lens) > 0 and bool(np.all(lens == lens[0])):
            # uniform batch: no offset tables to upload, nothing on this path synchronises with the host
            B, n = len(lens), int(lens[0])
            feats, _ = fe.forward(wav_flat.reshape(B, n), snip)
            return feats.reshape(-1, feats.shape[-1]), T.uniform_offsets(B, feats.shape[1])
        feats, fo = fe.forward_ragged(wav_flat, sample_offsets, snip)
        return feats, torch.from_numpy(fo).to(wav_flat.device)

    def embed(self, feats, offsets, max_frames=None):
        mask = self.vad.mask_ragged(feats, offsets)
        stack = None
        mf = feats.shape[0] if max_frames is None else max_frames
        if self.fusePrepass and self.cmvn.padding == "SAME" and not self.cmvn.normVar:
            # None when the window is too wide for the pre-pass tile: the separate kernels below take any window
            stack = self.xvec.fused_vad_cmvn_stack(feats.shape[-1], self.cmvn.N, mf)
        if stack is not None and stack.pools:
            # tcgen05 stack: gather -> CMVN -> splice is ONE pre-pass kernel in front of the GEMMs; the kept rows are
            # never written as a gathered / normalised fp32 matrix
            _, voffs, index = self.vad.compact_ragged(feats, mask, offsets, gather=False)
            self._voffs = voffs                # examined only when the result leaves as a host array (see __call__)
            emb = stack.forward_vad(feats, index, voffs, mf, self.cmvn.N)
            return emb, mask, voffs
        # `voiced` keeps the upper-bound row count; the kept-row count stays on the device (voffs[-1])
        voiced, voffs, _ = self.vad.compact_ragged(feats, mask, offsets, gather=True)
        # An utterance without voiced frames has no statistics to pool (the reference's gather_nd / reduce_mean
        # would produce NaN).  The offsets stay on the device -- checking them here would stall the launch queue --
        # and are examined when the result is handed back as a host array (see __call__).
        self._voffs = voffs
        normed, _ = self.cmvn.forward_ragged(voiced, voffs, max_frames=max_frames)
        emb, _ = self.xvec.forward_ragged(normed, voffs)
        return emb, mask, voffs

    def backend(self, emb):
        if self._dev is None:
            self._dev = (T.as_device(self.xvecGlobalMean), T.as_device(self.ldaTransform))
        mean, tr = self._dev
        B, D = emb.shape
        out_dim = tr.shape[0]
        y = torch.empty((B, out_dim), device=emb.device, dtype=torch.float32)
        N.check(N.lib().ktf_lda_forward(T.ptr(emb), B, D, out_dim, T.ptr(mean), T.ptr(tr), 1, T.ptr(y),
                                        T.stream_ptr()))
        return y

    @staticmethod
    def _audio_dtype(x):
        """int16 inputs are raw PCM and stay int16 up to the kernel (half the PCIe / HBM bytes)."""
        return torch.int16 if T.is_int16(x) else torch.float32

    def _flatten(self, inputs):
        if isinstance(inputs, (list, tuple)):
            dt = self._audio_dtype(inputs[0]) if len(inputs) else torch.float32
            arrs = [T.as_device(a, dtype=dt).reshape(-1) for a in inputs]
            lens = [int(a.numel()) for a in arrs]
            return torch.cat(arrs), np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        x = T.as_device(inputs, dtype=self._audio_dtype(inputs))
        if x.dim() == 1:
            x = x[None]
        if x.dim() != 2:
            raise ValueError(f"expected input of shape (batch, samples), got {tuple(x.shape)}")
        B, n = x.shape
        return x.reshape(-1), (np.arange(B + 1, dtype=np.int64) * n)

    def __call__(self, inputs, training: bool = False, return_intermediate: bool = False):
        wav_flat, so = self._flatten(inputs)
        feats, offsets = self.features(wav_flat, so)
        n_max = int(np.max(np.diff(so)))
        max_frames = self.framing.numFrames(n_max) if self.framing.snipEdges else \
            (n_max + self.framing.frameShift // 2) // self.framing.frameShift
        emb, mask, voffs = self.embed(feats, offsets, max_frames=max_frames)
        y = self.backend(emb)
        ref = inputs[0] if isinstance(inputs, (list, tuple)) else inputs
        out = T.like_input(y.squeeze(), ref)                      # tf.squeeze (:184)
        if not isinstance(out, torch.Tensor) and bool((self._voffs[1:] == self._voffs[:-1]).any().item()):
            raise ValueError("an utterance has no voiced frames after VAD")
        if return_intermediate:
            return out, {"mfcc": feats, "frame_offsets": offsets, "mask": mask,
                         "voiced_offsets": voffs, "embedding": emb}
        return out

    call = __call__


def _is_binary(path):
    with open(path, "rb") as f:
        return f.read(2) == b"\x00B"
