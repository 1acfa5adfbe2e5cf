"""
DSP front-end layers with the reference's constructor surface
(/root/reference/kaldi_tflite/lib/layers/dsp/{framing,windowing,filterbank,dct,mfcc,vad}.py).

All arithmetic runs in libktf_b200.so.  `Framing` does not materialise frames: it returns a
`FramedSignal` view that `Windowing`, `FilterBank` and `MFCC` consume directly with the fused
front-end kernel; frames are only written to HBM if the caller asks for them
(`.materialize()`, `.numpy()`, `np.asarray(...)`).
"""

import ctypes

import numpy as np
import torch

from .. import _native as N
from .. import _tensor as T
from .base import Layer


# ------------------------------------------------------------------------------------------
# Framing  (framing.py:49-265)
# ------------------------------------------------------------------------------------------

class FramedSignal:
    """Lazy (batch, frames, width) view over a (batch, samples) signal."""

    def __init__(self, wav, width, shift, ref, snip_edges=True):
        self.wav = wav                  # CUDA float32 (B, N), or int16 PCM (B, N)
        self.width = width
        self.shift = shift
        self.snip_edges = snip_edges    # False: Kaldi's mirror-padded framing, done inside the kernel
        self._ref = ref                 # original user object: decides numpy vs torch outputs
        self._frames = None

    @property
    def num_frames(self):
        n = self.wav.shape[-1]
        if not self.snip_edges:
            return (n + self.shift // 2) // self.shift      # kaldi_numpy/frame_extraction.py:78-80
        return 1 + (n - self.width) // self.shift

    @property
    def shape(self):
        return (self.wav.shape[0], self.num_frames, self.width)

    def materialize(self):
        if self._frames is None:
            if not self.snip_edges or self.wav.dtype != torch.float32:
                raise NotImplementedError("materialised frames need float32 input and snip_edges=True "
                                          "(the fused MFCC / FilterBank / Windowing layers take both forms)")
            B, n = self.wav.shape
            out = torch.empty(self.shape, device=self.wav.device, dtype=torch.float32)
            N.check(N.lib().ktf_framing_forward(T.ptr(self.wav), B, n, self.wav.stride(0) if B > 1 else n, self.width,
                                                self.shift, T.ptr(out), T.stream_ptr()))
            self._frames = out
        return self._frames

    def numpy(self):
        return self.materialize().cpu().numpy()

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a.astype(dtype) if dtype is not None else a

    def __dlpack__(self, *a, **k):
        return self.materialize().__dlpack__(*a, **k)

    def __dlpack_device__(self):
        return self.materialize().__dlpack_device__()


def _as_framed(inputs):
    """FramedSignal stays lazy; an explicit (B, T, W) tensor is a framing with shift == width."""
    if isinstance(inputs, FramedSignal):
        return inputs, inputs._ref
    x = T.as_device(inputs)
    if x.dim() != 3:
        raise ValueError(f"expected input of shape (batch, frames, samples), got {tuple(x.shape)}")
    B, Tn, W = x.shape
    return FramedSignal(x.reshape(B, Tn * W), W, W, inputs), inputs


class Framing(Layer):

    def __init__(self, frame_length_ms=25.0, frame_shift_ms=10.0, sample_frequency=16000.0,
                 name=None, dynamic_input_shape=False, snip_edges=True, **kwargs):
        """`snip_edges=False` (extension, SURVEY 8f): Kaldi's default framing -- the utterance is mirror-padded inside
        the kernel, replacing kaldi_numpy.PadWaveform on the host.  int16 inputs (numpy / torch) are taken as raw PCM
        and converted in the kernel; everything else is float32 in int16 scale like the reference."""
        super().__init__(name=name, trainable=False, **kwargs)
        self.snipEdges = bool(snip_edges)
        self.sampleFreq = sample_frequency
        self.frameSizeMs = frame_length_ms
        self.frameShiftMs = frame_shift_ms
        self.dynamicInputShape = dynamic_input_shape
        if self.frameSizeMs <= 0 or self.frameShiftMs <= 0 or self.sampleFreq <= 0:
            raise ValueError("frame_length, frame_shift and sample_frequency should be > 0")
        self.frameSize = int(sample_frequency * frame_length_ms / 1000.0)
        self.frameShift = int(sample_frequency * frame_shift_ms / 1000.0)
        if self.frameSize <= 0:
            raise ValueError("frame_length should be high enough to contain at least 1 sample")
        if self.frameShift <= 0:
            raise ValueError("frame_shift should be high enough to shift by at least 1 sample")
        self.halfFrameSize = self.frameSize // 2
        self.frameWidth = 2 * self.halfFrameSize      # offsets [-half, half) (framing.py:107-109)
        self.numInputSamples = None

    def build(self, input_shape):
        n = input_shape[-1]
        if n is None and not self.dynamicInputShape:
            raise ValueError("input_shape must not be unknown if dynamic_input_shape set to False")
        if n is not None:
            if n < self.frameSize:
                raise ValueError(f"input sample size (axis=-1) must be >= frame size ({self.frameSize})")
            self.numInputSamples = n
        super().build(input_shape)

    def numFrames(self, num_samples):
        # centres range(half, N - half + 1, shift) (framing.py:231-235)
        if num_samples < self.frameWidth:
            return 0
        return 1 + (num_samples - self.frameWidth) // self.frameShift

    def compute_output_shape(self, input_shape):
        shape = list(input_shape)
        n = shape[-1]
        if n is None and not self.dynamicInputShape:
            raise ValueError("input_shape must not be unknown if dynamic_input_shape set to False")
        return shape[:-1] + [None if n is None else self.numFrames(n), self.frameWidth]

    def get_config(self):
        config = super().get_config()
        config.update({"frame_length_ms": self.frameSizeMs, "frame_shift_ms": self.frameShiftMs,
                       "sample_frequency": self.sampleFreq,
                       "dynamic_input_shape": self.dynamicInputShape})
        if not self.snipEdges:
            config["snip_edges"] = False
        return config

    def call(self, inputs):
        wav = T.as_device(inputs, dtype=torch.int16 if T.is_int16(inputs) else torch.float32)
        squeeze = wav.dim() == 1
        if squeeze:
            wav = wav[None]
        if wav.dim() != 2:
            raise ValueError(f"expected input of shape (batch, samples), got {tuple(wav.shape)}")
        self._maybe_build(wav.shape)
        n = wav.shape[-1]
        if n < self.frameSize:
            raise ValueError(f"input sample size (axis=-1) must be >= frame size ({self.frameSize})")
        if not self.dynamicInputShape and self.numInputSamples is not None and n != self.numInputSamples:
            raise ValueError(f"layer was built for {self.numInputSamples} samples, got {n} "
                             "(use dynamic_input_shape=True)")
        return FramedSignal(wav, self.frameWidth, self.frameShift, inputs, snip_edges=self.snipEdges)


# ------------------------------------------------------------------------------------------
# constant tables, computed like the reference's build() methods (float64 -> float32)
# ------------------------------------------------------------------------------------------

WINDOW_TYPES = ("hamming", "hanning", "povey", "rectangular", "sine", "blackman")


def window_function(window_type, M, blackman_coeff=0.42):
    """windowing.py:130-156."""
    n = np.arange(0, M)
    if M == 1:
        w = np.ones(1, float)
    elif window_type == "hamming":
        w = np.hamming(M)
    elif window_type == "hanning":
        w = np.hanning(M)
    elif window_type == "povey":
        w = np.power(0.5 - 0.5 * np.cos(2.0 * np.pi * n / (M - 1)), 0.85)
    elif window_type == "rectangular":
        w = np.ones((M,))
    elif window_type == "sine":
        w = np.sin(np.pi * n / (M - 1))
    elif window_type == "blackman":
        w = np.blackman(M)
        if blackman_coeff != 0.42:
            w = w - 0.42 + blackman_coeff
    else:
        raise ValueError(f"window_type '{window_type}' is not recognized")
    return np.ascontiguousarray(w, dtype=np.float32)


def next_power_of_2(n):
    return n if (n & (n - 1) == 0) and n != 0 else 2 ** (n - 1).bit_length()


def mel_filterbank(window_size, num_bins, sample_freq, lower, upper):
    """filterbank.py:141-189 -> (fft_length, float32 (fft_length/2+1, num_bins))."""
    fft_length = next_power_of_2(window_size)
    fft_bins = fft_length // 2
    mel = lambda f: 1127.0 * np.log(1.0 + f / 700.0)
    mel_low, mel_high = mel(lower), mel(upper)
    delta = (mel_high - mel_low) / (num_bins + 1)
    bin_mel = mel((sample_freq / fft_length) * np.arange(fft_bins))
    bank = np.zeros((num_bins, fft_bins + 1), dtype=np.float32)
    for i in range(num_bins):
        left = mel_low + i * delta
        center = left + delta
        right = center + delta
        rising = (bin_mel > left) & (bin_mel <= center)
        falling = (bin_mel > center) & (bin_mel < right)
        bank[i, :fft_bins][rising] = (bin_mel[rising] - left) / (center - left)
        bank[i, :fft_bins][falling] = (right - bin_mel[falling]) / (right - center)
    return fft_length, np.ascontiguousarray(bank.T)


def dct2_matrix(input_length, length):
    """dct.py:98-143: ortho DCT-II (input_length, length), column 0 = sqrt(1/N)."""
    Nf = float(input_length)
    n = np.arange(input_length)
    k = np.arange(length, dtype=np.float64)[:, None]
    m = np.cos((np.pi / Nf) * (n + 0.5) * k)
    m[0] *= 1.0 / np.sqrt(2.0)
    m *= np.sqrt(2.0 / Nf)
    m = m.T.copy()
    m[:, 0] = np.sqrt(1.0 / Nf)
    return np.ascontiguousarray(m, dtype=np.float32)


def lifter_coefficients(num_mfccs, q):
    """mfcc.py:146-159."""
    n = np.arange(0, num_mfccs)
    return np.ascontiguousarray(1 + 0.5 * np.sin(np.pi * n / q) * q, dtype=np.float32)


class _Frontend:
    """Owns one ktf_frontend handle."""

    def __init__(self, cfg, window, mel_bank=None, dct=None, lifter=None):
        N.require_cuda()
        self._keep = (window, mel_bank, dct, lifter)
        self.handle = ctypes.c_void_p()
        N.check(N.lib().ktf_frontend_create(ctypes.byref(cfg), T.host_ptr(window), T.host_ptr(mel_bank),
                                            T.host_ptr(dct), T.host_ptr(lifter),
                                            ctypes.byref(self.handle)))
        self.out_dim = N.lib().ktf_frontend_out_dim(self.handle)
        self.want_energy = bool(cfg.output == N.KTF_OUT_WINDOWED and cfg.use_energy)
        self.dither = float(cfg.dither)
        self.wide = cfg.fft_length > 512      # 1024..4096 points: a kernel that reads int16 PCM in every mode

    def __del__(self):
        try:
            if self.handle:
                N.lib().ktf_frontend_destroy(self.handle)
        except Exception:
            pass

    def num_frames(self, n, snip_edges=True):
        return int(N.lib().ktf_frontend_num_frames_ex(self.handle, n, int(bool(snip_edges))))

    def _ingest(self, wav):
        # the dithering 256 / 512-point (generic) kernel takes float32 samples: raw PCM is widened first (dither != 0
        # only); the 1024..4096-point kernel converts int16 itself, dithered or not
        if self.dither != 0.0 and wav.dtype == torch.int16 and not self.wide:
            return wav.to(torch.float32)
        return wav

    @staticmethod
    def _fmt(wav):
        if wav.dtype == torch.int16:
            return N.KTF_SAMPLE_S16
        if wav.dtype != torch.float32:
            raise ValueError(f"audio must be float32 or int16, got {wav.dtype}")
        return N.KTF_SAMPLE_F32

    def forward(self, wav, snip_edges=True):
        """wav CUDA float32 / int16 (B, n) -> (B, T, out_dim) [, (B, T, 1) energy]."""
        wav = self._ingest(wav)
        B, n = wav.shape
        Tn = self.num_frames(n, snip_edges)
        out = torch.empty((B, Tn, self.out_dim), device=wav.device, dtype=torch.float32)
        energy = torch.empty((B, Tn, 1), device=wav.device, dtype=torch.float32) if self.want_energy else None
        N.check(N.lib().ktf_frontend_forward_ex(self.handle, T.ptr(wav), self._fmt(wav), int(bool(snip_edges)), B, n,
                                                wav.stride(0) if B > 1 else n, T.ptr(out), T.ptr(energy),
                                                T.stream_ptr()))
        return out, energy

    def forward_ragged(self, wav_flat, sample_offsets, snip_edges=True):
        """wav_flat CUDA (total,), sample_offsets numpy int64 (B+1) -> (total_frames, out_dim), frame offsets."""
        wav_flat = self._ingest(wav_flat)
        B = len(sample_offsets) - 1
        so = np.ascontiguousarray(sample_offsets, dtype=np.int64)
        fo = np.zeros(B + 1, dtype=np.int64)
        lens = np.diff(so)
        total = int(sum(self.num_frames(int(l), snip_edges) for l in lens))
        out = torch.empty((total, self.out_dim), device=wav_flat.device, dtype=torch.float32)
        N.check(N.lib().ktf_frontend_forward_ragged_ex(self.handle, T.ptr(wav_flat), self._fmt(wav_flat),
                                                       int(bool(snip_edges)), B, T.host_ptr(so), T.host_ptr(fo),
                                                       T.ptr(out), None, T.stream_ptr()))
        return out, fo


# ------------------------------------------------------------------------------------------
# Windowing (windowing.py:36-209)
# ------------------------------------------------------------------------------------------

class Windowing(Layer):

    def __init__(self, window_type="povey", blackman_coeff=0.42, dither=0.0, remove_dc_offset=True,
                 preemphasis_coefficient=0.97, return_energy=True, raw_energy=True, energy_floor=0.0,
                 epsilon=1e-7, name=None, **kwargs):
        super().__init__(name=name, trainable=False, **kwargs)
        self.windowType = window_type.lower()
        if self.windowType not in WINDOW_TYPES:
            raise ValueError(f"window_type '{window_type}' is not recognized")
        self.blackmanCoeff = blackman_coeff
        self.dither = dither
        self.removeDCOffset = remove_dc_offset
        self.preemphasisCoeff = preemphasis_coefficient
        self.returnEnergy = return_energy
        self.rawEnergy = raw_energy
        self.energyFloor = energy_floor
        self.eps = epsilon
        self.windowFunc = None
        self._fe = {}

    def build(self, input_shape):
        M = input_shape[-1]
        if M == 0:
            raise ValueError("window size (input shape axis = -1) needs to be > 0")
        self.windowFunc = window_function(self.windowType, M, self.blackmanCoeff)
        super().build(input_shape)

    def get_config(self):
        config = super().get_config()
        config.update({"window_type": self.windowType, "blackman_coeff": self.blackmanCoeff,
                       "dither": self.dither, "remove_dc_offset": self.removeDCOffset,
                       "preemphasis_coefficient": self.preemphasisCoeff,
                       "return_energy": self.returnEnergy, "raw_energy": self.rawEnergy,
                       "energy_floor": self.energyFloor, "epsilon": self.eps})
        return config

    def _frontend(self, width, shift):
        key = (width, shift)
        if key not in self._fe:
            cfg = N.FrontendCfg(frame_width=width, frame_shift=shift,
                                fft_length=max(256, next_power_of_2(width)), num_mels=0, num_ceps=0,
                                output=N.KTF_OUT_WINDOWED, remove_dc_offset=int(self.removeDCOffset),
                                raw_energy=int(self.rawEnergy), use_energy=int(self.returnEnergy),
                                use_power=1, use_log_fbank=1, apply_lifter=0,
                                preemphasis=float(self.preemphasisCoeff),
                                energy_floor=float(self.energyFloor), epsilon=float(self.eps),
                                dither=float(self.dither))
            self._fe[key] = _Frontend(cfg, window_function(self.windowType, width, self.blackmanCoeff))
        return self._fe[key]

    def call(self, inputs):
        fs, ref = _as_framed(inputs)
        self._maybe_build(fs.shape)
        out, energy = self._frontend(fs.width, fs.shift).forward(fs.wav, fs.snip_edges)   # dither: inside the kernel
        if self.returnEnergy:
            return T.like_input(out, ref), T.like_input(energy, ref)
        return T.like_input(out, ref)


# ------------------------------------------------------------------------------------------
# FilterBank (filterbank.py:39-242)
# ------------------------------------------------------------------------------------------

def _check_cutoffs(sample_frequency, low_freq_cutoff, high_freq_cutoff):
    nyquist = sample_frequency / 2.0
    if sample_frequency <= 0:
        raise ValueError(f"sample_frequency must be > 0, got {sample_frequency}")
    if low_freq_cutoff > nyquist or low_freq_cutoff < 0:
        raise ValueError(f"low_freq_cutoff must be > 0 and < Nyquist Rate ({nyquist} Hz)")
    upper = high_freq_cutoff
    if upper <= 0:
        upper += nyquist
    if low_freq_cutoff >= upper:
        raise ValueError("lower_freq_cutoff must be < higher_freq_cutoff")
    return upper


class FilterBank(Layer):

    def __init__(self, num_bins=23, sample_frequency=16000.0, high_freq_cutoff=0.0,
                 low_freq_cutoff=20.0, use_log_fbank=True, use_power=True, epsilon=1e-7, name=None,
                 **kwargs):
        super().__init__(name=name, trainable=False, **kwargs)
        self.numBins = num_bins
        if self.numBins <= 0:
            raise ValueError(f"num_bins must be > 0, got {num_bins}")
        self.sampleFreq = sample_frequency
        self.nyquist = sample_frequency / 2.0
        self.lowerCutoff = low_freq_cutoff
        self.upperCutoff = _check_cutoffs(sample_frequency, low_freq_cutoff, high_freq_cutoff)
        self.useLogFBank = use_log_fbank
        self.usePower = use_power
        self.eps = epsilon
        self.melBank = None
        self.fftLength = None
        self._fe = {}

    def build(self, input_shape):
        self.fftLength, self.melBank = mel_filterbank(input_shape[-1], self.numBins, self.sampleFreq,
                                                      self.lowerCutoff, self.upperCutoff)
        super().build(input_shape)

    def compute_output_shape(self, input_shape):
        return list(input_shape[:-1]) + [self.numBins]

    def get_config(self):
        config = super().get_config()
        config.update({"sample_frequency": self.sampleFreq, "num_bins": self.numBins,
                       "low_freq_cutoff": self.lowerCutoff, "high_freq_cutoff": self.upperCutoff,
                       "use_log_fbank": self.useLogFBank, "use_power": self.usePower,
                       "epsilon": self.eps})
        return config

    def _frontend(self, width, shift):
        key = (width, shift)
        if key not in self._fe:
            fft_length, bank = mel_filterbank(width, self.numBins, self.sampleFreq, self.lowerCutoff,
                                              self.upperCutoff)
            cfg = N.FrontendCfg(frame_width=width, frame_shift=shift, fft_length=fft_length,
                                num_mels=self.numBins, num_ceps=0, output=N.KTF_OUT_FBANK,
                                remove_dc_offset=0, raw_energy=1, use_energy=0,
                                use_power=int(self.usePower), use_log_fbank=int(self.useLogFBank),
                                apply_lifter=0, preemphasis=0.0, energy_floor=0.0,
                                epsilon=float(self.eps), dither=0.0)
            self._fe[key] = _Frontend(cfg, np.ones(width, dtype=np.float32), bank)
        return self._fe[key]

    def call(self, inputs):
        fs, ref = _as_framed(inputs)
        self._maybe_build(fs.shape)
        out, _ = self._frontend(fs.width, fs.shift).forward(fs.wav, fs.snip_edges)
        return T.like_input(out, ref)


# ------------------------------------------------------------------------------------------
# DCT (dct.py:41-176)
# ------------------------------------------------------------------------------------------

class DCT(Layer):

    def __init__(self, length, dct_type=2, norm="ortho", name=None, **kwargs):
        super().__init__(name=name, trainable=False, **kwargs)
        self.length = length
        if self.length <= 0:
            raise ValueError(f"DCT length must be > 0, got {length}")
        self.dctType = dct_type
        if self.dctType not in [2]:
            raise NotImplementedError(f"DCT-{dct_type} is not supported yet")
        self.norm = norm.lower()
        if self.norm not in ["ortho"]:
            raise NotImplementedError(f"{norm} normalization is not supported yet")
        self.dct = None
        self._affine = None

    def build(self, input_shape):
        feat = input_shape[-1]
        if feat < self.length:
            raise ValueError("input feature length must be >= DCT length")
        self.dct = dct2_matrix(feat, self.length)
        from .tdnn import _Affine
        # out = x @ dct  ==  affine with Kaldi-layout weights dct^T, context [0], no bias
        self._affine = _Affine(np.ascontiguousarray(self.dct.T), None, [0], precision="f32")
        super().build(input_shape)

    def compute_output_shape(self, input_shape):
        return tuple(input_shape[:-1]) + (self.length,)

    def get_config(self):
        config = super().get_config()
        config.update({"length": self.length, "dct_type": self.dctType, "norm": self.norm})
        return config

    def call(self, inputs):
        x = T.as_device(inputs)
        self._maybe_build(x.shape)
        B, Tn, D = x.shape
        y = self._affine.forward_uniform(x)
        return T.like_input(y, inputs)


# ------------------------------------------------------------------------------------------
# MFCC (mfcc.py:43-244)
# ------------------------------------------------------------------------------------------

class MFCC(Layer):

    def __init__(self, num_mfccs=23, num_mels=23, cepstral_lifter=22, use_energy=True,
                 sample_frequency=16000.0, high_freq_cutoff=0.0, low_freq_cutoff=20.0,
                 use_log_fbank=True, use_power=True, window_type="povey", dither=0.0,
                 remove_dc_offset=True, preemphasis_coefficient=0.97, raw_energy=True,
                 energy_floor=0.0, epsilon=1e-7, name=None, **kwargs):
        super().__init__(name=name, trainable=False, **kwargs)
        self.numMfccs = num_mfccs
        self.melBins = num_mels
        self.cepstralLifter = cepstral_lifter
        self.useEnergy = use_energy
        if self.numMfccs > self.melBins:
            raise ValueError("num_mfccs must be <= num_mels")
        self.eps = epsilon
        self.windowing = Windowing(window_type=window_type, dither=dither,
                                   remove_dc_offset=remove_dc_offset,
                                   preemphasis_coefficient=preemphasis_coefficient,
                                   raw_energy=raw_energy, return_energy=use_energy,
                                   energy_floor=energy_floor, epsilon=epsilon)
        self.filterbank = FilterBank(num_bins=num_mels, sample_frequency=sample_frequency,
                                     high_freq_cutoff=high_freq_cutoff, low_freq_cutoff=low_freq_cutoff,
                                     use_log_fbank=use_log_fbank, use_power=use_power, epsilon=epsilon)
        self.dct = DCT(length=num_mfccs, dct_type=2, norm="ortho")
        self.lifters = lifter_coefficients(num_mfccs, cepstral_lifter) if num_mfccs > 1 else None
        self._fe = {}

    def compute_output_shape(self, input_shape):
        return list(input_shape[:-1]) + [self.numMfccs]

    def get_config(self):
        config = super().get_config()
        for sub in (self.windowing.get_config(), self.filterbank.get_config()):
            sub.pop("name", None)
            sub.pop("trainable", None)
            config.update(sub)
        config.pop("return_energy", None)
        config.pop("blackman_coeff", None)
        config.pop("num_bins", None)
        config.update({"num_mfccs": self.numMfccs, "num_mels": self.melBins,
                       "cepstral_lifter": self.cepstralLifter, "use_energy": self.useEnergy,
                       "epsilon": self.eps})
        return config

    def frontend(self, width, shift):
        """The fused framing->MFCC handle for frames of `width` samples every `shift` samples."""
        key = (width, shift)
        if key not in self._fe:
            w, fb = self.windowing, self.filterbank
            fft_length, bank = mel_filterbank(width, fb.numBins, fb.sampleFreq, fb.lowerCutoff, fb.upperCutoff)
            lifter_on = self.cepstralLifter > 1 and self.lifters is not None
            cfg = N.FrontendCfg(frame_width=width, frame_shift=shift, fft_length=fft_length,
                                num_mels=self.melBins, num_ceps=self.numMfccs, output=N.KTF_OUT_MFCC,
                                remove_dc_offset=int(w.removeDCOffset), raw_energy=int(w.rawEnergy),
                                use_energy=int(self.useEnergy), use_power=int(fb.usePower),
                                use_log_fbank=int(fb.useLogFBank), apply_lifter=int(lifter_on),
                                preemphasis=float(w.preemphasisCoeff), energy_floor=float(w.energyFloor),
                                epsilon=float(self.eps), dither=float(w.dither))
            self._fe[key] = _Frontend(cfg, window_function(w.windowType, width, w.blackmanCoeff), bank,
                                      dct2_matrix(self.melBins, self.numMfccs),
                                      self.lifters if lifter_on else None)
        return self._fe[key]

    def call(self, inputs):
        fs, ref = _as_framed(inputs)
        self._maybe_build(fs.shape)
        # dither (windowing.py:182-183) is drawn per framed sample inside the kernel
        out, _ = self.frontend(fs.width, fs.shift).forward(fs.wav, fs.snip_edges)
        return T.like_input(out, ref)


# ------------------------------------------------------------------------------------------
# VAD (vad.py:45-203)
# ------------------------------------------------------------------------------------------

class VAD(Layer):

    def __init__(self, energy_mean_scale=0.5, energy_threshold=5, frames_context=0,
                 proportion_threshold=0.6, return_indexes=True, energy_coeff=0, name=None, **kwargs):
        super().__init__(name=name, trainable=False, **kwargs)
        if energy_mean_scale < 0:
            raise ValueError("`energy_mean_scale` must be >= 0")
        if frames_context < 0:
            raise ValueError("`frames_context` must be >= 0")
        if proportion_threshold <= 0 or proportion_threshold >= 1:
            raise ValueError("`proportion_threshold` must be between 0 and 1 (exlcusive)")
        self.energyThreshold = float(energy_threshold)
        self.energyMeanScale = float(energy_mean_scale)
        self.propThreshold = float(proportion_threshold)
        self.returnIndexes = return_indexes
        self.useEnergyMean = energy_mean_scale > 0
        self.framesContext = frames_context
        self.windowSize = self.framesContext * 2 + 1
        self.energyCoef = energy_coeff

    def get_config(self):
        config = super().get_config()
        config.update({"energy_mean_scale": self.energyMeanScale,
                       "energy_threshold": self.energyThreshold,
                       "frames_context": self.framesContext,
                       "proportion_threshold": self.propThreshold,
                       "return_indexes": self.returnIndexes, "energy_coeff": self.energyCoef})
        return config

    def _cfg(self):
        return N.VadCfg(energy_threshold=self.energyThreshold, energy_mean_scale=self.energyMeanScale,
                        proportion_threshold=self.propThreshold, frames_context=self.framesContext,
                        energy_coeff=self.energyCoef)

    def mask_ragged(self, feats2d, offsets):
        """feats2d CUDA (rows, D), offsets CUDA int64 (B+1) -> CUDA float mask (rows,)."""
        rows, D = feats2d.shape
        mask = torch.empty((rows,), device=feats2d.device, dtype=torch.float32)
        cfg = self._cfg()
        N.check(N.lib().ktf_vad_mask(ctypes.byref(cfg), T.ptr(feats2d), D, T.ptr(offsets),
                                     offsets.numel() - 1, rows, T.ptr(mask), T.stream_ptr()))
        return mask

    @staticmethod
    def compact_ragged(feats2d, mask, offsets, gather=True):
        """Stable per-utterance compaction -> (kept feats or None, new offsets, row index).

        Nothing here synchronises with the host: the number of kept rows stays on the device (`new offsets[-1]`), the
        returned `feats` / `index` buffers have the UPPER-BOUND length `rows` and only their first `new offsets[-1]`
        entries are meaningful.  Every consumer on the hot path (CMVN, the TDNN stack) takes the per-utterance
        offsets from the device, so wav -> x-vector can be captured in a CUDA graph."""
        rows, D = feats2d.shape
        B = offsets.numel() - 1
        out_offs = torch.empty((B + 1,), device=mask.device, dtype=torch.int64)
        index = torch.empty((rows,), device=mask.device, dtype=torch.int64)
        ws = torch.empty((int(N.lib().ktf_vad_compact_workspace(B, rows)),), device=mask.device,
                         dtype=torch.uint8)
        out = torch.empty((rows, D), device=mask.device, dtype=torch.float32) if gather else None
        N.check(N.lib().ktf_vad_compact(T.ptr(feats2d), D, T.ptr(mask), T.ptr(offsets), B, rows,
                                        T.ptr(out_offs), T.ptr(index), T.ptr(out), T.ptr(ws),
                                        T.stream_ptr()))
        return out, out_offs, index

    def call(self, inputs):
        x = T.as_device(inputs)
        if x.dim() != 3:
            raise ValueError(f"expected input of shape (batch, frames, feats), got {tuple(x.shape)}")
        B, Tn, D = x.shape
        offsets = T.uniform_offsets(B, Tn)
        mask = self.mask_ragged(x.reshape(B * Tn, D), offsets)
        if not self.returnIndexes:
            return T.like_input(mask.reshape(B, Tn, 1), inputs)
        _, out_offs, index = self.compact_ragged(x.reshape(B * Tn, D), mask, offsets, gather=False)
        # tf.where returns a data-dependent shape (vad.py:200-203): this API -- unlike the fused wav -> x-vector
        # path -- has to read the count back
        index = index[:int(out_offs[-1].item())]
        idx = torch.stack([index // Tn, index % Tn], dim=1)        # (n_active, 2) like tf.where
        return T.like_input(idx, inputs)
