"""
Front-end at frame widths above 512 samples (FFT lengths 1024, 2048, 4096): 25 ms frames at 32, 44.1, 48 and 96 kHz,
85 ms at 48 kHz, and raw widths that need no padding.

Gate, against the float64 evaluation of the oracle's formulas (the rule of test_record_parity_margins with the float32
oracle's share tripled, FACTOR = 3):
    max-abs <= max(1e-3, FACTOR x 1.25 x the float32 oracle's max-abs),
    p99.9   <= max(1e-3, FACTOR x the float32 oracle's p99.9).
Why the factor: the kernel computes the N-point real FFT as an N/2-point complex FFT and untangles bins k and N/2 - k.
A strong component near Nyquist then leaves its float32 rounding (about 1e-7 of its amplitude) on the mirrored low bins,
which pre-emphasis makes the weakest of the frame; the float32 library FFT of the oracle has no such mirror.  Where a
comparison sits at that floor (a chirp up to Nyquist, linear outputs of 1e6 and more) the kernel's error measured up to
2.05x the unscaled bound on a B200 (48 kHz / 20 ms MFCC on noise plus chirp); a misrouted bin or frame misses by orders
of magnitude.

CPU tests check the oracle's wide-band semantics against torchaudio's Kaldi-compatible fbank, and the layer's mel
bank against the oracle's.  GPU tests cover MFCC / fbank / Windowing against the gate, spectral isolation of
alternating tone / silence frames, ragged batches, int16 PCM, in-kernel dither, output bounds, CUDA-graph capture and
the limits of the accepted configurations.
"""

import ctypes

import numpy as np
import pytest

from conftest import golden_path, read_wav_int16
from oracle import ktf_oracle as O

RATES = [(32000, 25.0), (44100, 25.0), (48000, 20.0), (48000, 25.0), (48000, 85.0), (96000, 25.0)]
RAW_WIDTHS = [513, 1024, 2048, 4096]


def _noise(rate, seconds, seed=0, batch=1):
    """Wide-band noise plus a chirp over the whole band, int16 scale."""
    rng = np.random.default_rng(seed)
    n = int(rate * seconds)
    t = np.arange(n) / rate
    chirp = 8000.0 * np.sin(2 * np.pi * (50.0 * t + 0.5 * (rate / 2 - 100.0) / seconds * t * t))
    x = rng.standard_normal((batch, n)) * 1500.0 + chirp[None]
    return np.round(x).astype(np.float32)


def _speech(rate, seconds=2.0):
    """librispeech_2.wav (16 kHz) resampled to `rate`: nothing above 8 kHz, near-silent upper mel bands."""
    from scipy.signal import resample_poly
    from math import gcd
    wav = read_wav_int16(golden_path("librispeech_2.wav")).astype(np.float64)
    g = gcd(int(rate), 16000)
    y = resample_poly(wav[: int(16000 * (seconds + 0.5))], int(rate) // g, 16000 // g)
    return np.round(y[: int(rate * seconds)]).astype(np.float32)[None]


FACTOR = 3.0


def _gate(got, truth, ora, what="", factor=FACTOR):
    e = np.abs(np.asarray(got, np.float64) - truth)
    f = np.abs(np.asarray(ora, np.float64) - truth)
    assert got.shape == truth.shape, (what, got.shape, truth.shape)
    assert np.all(np.isfinite(got)), what
    max_ok = max(1e-3, factor * 1.25 * float(f.max()))
    p_ok = max(1e-3, factor * float(np.quantile(f, 0.999)))
    assert float(e.max()) <= max_ok, (what, float(e.max()), max_ok)
    assert float(np.quantile(e, 0.999)) <= p_ok, (what, float(np.quantile(e, 0.999)), p_ok)


def _oracle_frames(x, rate, ms, snip):
    size, shift, _ = O.frame_params(ms, 10.0, rate)
    if not snip:
        x = O.pad_waveform(x, size, shift)
    return O.framing(x, ms, 10.0, rate)


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("rate,ms", RATES)
def test_oracle_matches_torchaudio_fbank(rate, ms):
    """Independent check of the oracle's wide-band semantics: torchaudio.compliance.kaldi.fbank (snip_edges, no dither,
    power spectrum, log) against the float64 oracle, on noise plus a chirp."""
    torchaudio = pytest.importorskip("torchaudio")
    import torch
    x = _noise(rate, 0.3, seed=1)
    for bins in (40, 80, 128):
        ref = torchaudio.compliance.kaldi.fbank(
            torch.from_numpy(x.astype(np.float64)), sample_frequency=float(rate), frame_length=ms, frame_shift=10.0,
            num_mel_bins=bins, dither=0.0, snip_edges=True, window_type="povey", preemphasis_coefficient=0.97,
            remove_dc_offset=True, round_to_power_of_two=True, low_freq=20.0, high_freq=0.0, use_energy=False,
            use_log_fbank=True, use_power=True, energy_floor=0.0).numpy()
        frames = O.framing(x, ms, 10.0, rate)
        w = O.windowing(frames, return_energy=False, precise=True)
        ora = O.filterbank(w, num_bins=bins, sample_frequency=rate, precise=True)[0]
        assert ref.shape == ora.shape
        assert float(np.max(np.abs(ref - ora))) <= 1e-3, (rate, ms, bins, float(np.max(np.abs(ref - ora))))


@pytest.mark.parametrize("width", [513, 800, 1102, 1200, 2048, 2400, 4080, 4096])
def test_layer_mel_bank_equals_oracle(width):
    from kaldi_tflite_b200.layers.dsp import mel_filterbank
    for rate, bins in ((48000, 80), (96000, 128), (44100, 40)):
        n, bank = mel_filterbank(width, bins, float(rate), 20.0, rate / 2.0)
        n_o, bank_o = O.mel_bank(width, bins, float(rate), 0.0, 20.0)
        assert n == n_o == O.next_pow2(width) and n <= 4096
        assert bank.shape == bank_o.shape == (n // 2 + 1, bins)
        assert np.array_equal(bank, bank_o)


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ktf():
    import kaldi_tflite_b200 as k
    return k


def _mfcc_kw(rate, **kw):
    d = dict(num_mfccs=30, num_mels=40, sample_frequency=float(rate))
    d.update(kw)
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("rate,ms", RATES)
def test_mfcc_fbank_windowing_gate(ktf, rate, ms):
    for snip in (True, False):
        for name, x in (("speech", _speech(rate)), ("noise", _noise(rate, 1.0, seed=2))):
            fr = ktf.layers.Framing(ms, 10.0, rate, dynamic_input_shape=True, snip_edges=snip)
            frames = _oracle_frames(x, rate, ms, snip)
            assert fr.frameWidth in (800, 1102, 960, 1200, 4080, 2400)
            what = (rate, ms, snip, name)
            kw = _mfcc_kw(rate)
            got = ktf.layers.MFCC(**kw)(fr(x))
            _gate(got, O.mfcc(frames, precise=True, **kw), O.mfcc(frames, **kw), ("mfcc",) + what)
            win = ktf.layers.Windowing()
            w, e = win(fr(x))
            wt, et = O.windowing(frames, precise=True)
            wo, eo = O.windowing(frames)
            _gate(w, wt, wo, ("windowing",) + what)
            _gate(e, et, eo, ("energy",) + what)
            fb = ktf.layers.FilterBank(num_bins=80, sample_frequency=float(rate))(
                ktf.layers.Windowing(return_energy=False)(fr(x)))
            ft = O.filterbank(O.windowing(frames, return_energy=False, precise=True), num_bins=80,
                              sample_frequency=rate, precise=True)
            fo = O.filterbank(O.windowing(frames, return_energy=False), num_bins=80, sample_frequency=rate)
            _gate(fb, ft, fo, ("fbank",) + what)


VARIANTS = [
    dict(use_power=False),
    dict(use_log_fbank=False),
    dict(raw_energy=False),
    dict(remove_dc_offset=False),
    dict(window_type="hamming"),
    dict(window_type="blackman", num_mels=128, num_mfccs=13),
    dict(num_mels=128, num_mfccs=30),
    dict(num_mfccs=13, num_mels=23, use_energy=False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", range(len(VARIANTS)))
def test_mfcc_switches_gate(ktf, variant):
    rate, ms = RATES[variant % len(RATES)]
    for snip in (True, False):
        for name, x in (("speech", _speech(rate, 1.0)), ("noise", _noise(rate, 0.5, seed=3))):
            frames = _oracle_frames(x, rate, ms, snip)
            kw = _mfcc_kw(rate, **VARIANTS[variant])
            got = ktf.layers.MFCC(**kw)(ktf.layers.Framing(ms, 10.0, rate, dynamic_input_shape=True,
                                                           snip_edges=snip)(x))
            _gate(got, O.mfcc(frames, precise=True, **kw), O.mfcc(frames, **kw), (kw, snip, name))


@pytest.mark.gpu
@pytest.mark.parametrize("width", RAW_WIDTHS)
def test_raw_widths_gate(ktf, width):
    """Pre-framed (B, T, W) input with W == N (nothing padded) and W = 513 (almost all padding)."""
    rng = np.random.default_rng(width)
    frames = (rng.standard_normal((2, 24, width)) * 2000.0).astype(np.float32)
    t = np.arange(width)
    frames[1] += (6000.0 * np.sin(2 * np.pi * 0.1234 * t)).astype(np.float32)
    kw = _mfcc_kw(48000, num_mels=64)
    _gate(ktf.layers.MFCC(**kw)(frames), O.mfcc(frames, precise=True, **kw), O.mfcc(frames, **kw), ("mfcc", width))
    for kwf in (dict(), dict(use_power=False, use_log_fbank=False)):
        fb = ktf.layers.FilterBank(num_bins=80, sample_frequency=48000.0, **kwf)(frames)
        _gate(fb, O.filterbank(frames, num_bins=80, sample_frequency=48000, precise=True, **kwf),
              O.filterbank(frames, num_bins=80, sample_frequency=48000, **kwf), ("fbank", width, kwf))
    for kww in (dict(), dict(raw_energy=False, remove_dc_offset=False, window_type="sine")):
        w, e = ktf.layers.Windowing(**kww)(frames)
        wt, et = O.windowing(frames, precise=True, **kww)
        wo, eo = O.windowing(frames, **kww)
        _gate(w, wt, wo, ("windowing", width, kww))
        _gate(e, et, eo, ("energy", width, kww))


@pytest.mark.gpu
@pytest.mark.parametrize("width", [1024, 2048, 4096])
def test_spectral_isolation(ktf, width):
    """Frames alternate between low noise and a full-scale tone at DC, at the 4-bin chunk boundaries around C/4 and
    C/2, and at Nyquist: a bin or a frame routed to the wrong place misses the gate by orders of magnitude.

    A pure integer-rounded tone leaves the bands away from it at the float32 rounding floor of ANY float32 FFT (about
    1e-7 of the peak): there two float32 transforms differ by a factor of a few in error, not by orders of magnitude,
    so this test allows 4x the float32 oracle's error (measured on a B200: up to 2.4x at 2048 points)."""
    C = width // 2
    bins = [0, 1, C // 4 - 1, C // 4, C // 4 + 1, C // 2 - 1, C // 2, C // 2 + 1, C // 2 + 4, C - 1, C]
    rng = np.random.default_rng(7)
    T = 2 * len(bins)
    frames = (rng.standard_normal((1, T, width)) * 1.0).astype(np.float32)
    n = np.arange(width)
    for i, k in enumerate(bins):
        frames[0, 2 * i + 1] = np.round(30000.0 * np.cos(2 * np.pi * k * n / width + 0.3 * (k % 3)))
    for kwf in (dict(), dict(use_power=False)):
        fb = ktf.layers.FilterBank(num_bins=128, sample_frequency=48000.0, **kwf)(frames)
        _gate(fb, O.filterbank(frames, num_bins=128, sample_frequency=48000, precise=True, **kwf),
              O.filterbank(frames, num_bins=128, sample_frequency=48000, **kwf), ("fbank", width, kwf), factor=4.0)
    kw = dict(num_mfccs=30, num_mels=128, sample_frequency=48000.0, window_type="rectangular",
              preemphasis_coefficient=0.0, remove_dc_offset=False)
    _gate(ktf.layers.MFCC(**kw)(frames), O.mfcc(frames, precise=True, **kw), O.mfcc(frames, **kw), ("mfcc", width),
          factor=4.0)


def _ragged(ktf, m, width, shift, wav_flat, offs, snip):
    import torch
    fe = m.frontend(width, shift)
    out, fo = fe.forward_ragged(torch.as_tensor(wav_flat).cuda(), offs, snip)
    return out.cpu().numpy(), fo


@pytest.mark.gpu
@pytest.mark.parametrize("rate,ms", [(48000, 25.0), (96000, 25.0), (44100, 25.0)])
def test_ragged_batches(ktf, rate, ms):
    fr = ktf.layers.Framing(ms, 10.0, rate, dynamic_input_shape=True)
    W, S = fr.frameWidth, fr.frameShift
    lens = [W, W + 1, W + S - 1, W + S, 10 * rate, 3 * W + 7, W + 2 * S + 1]
    rng = np.random.default_rng(11)
    utts = [np.round(rng.standard_normal(n) * 2000.0).astype(np.float32) for n in lens]
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    flat = np.concatenate(utts)
    m = ktf.layers.MFCC(**_mfcc_kw(rate))
    for snip in (True, False):
        for layer in (m,):
            out, fo = _ragged(ktf, layer, W, S, flat, offs, snip)
            again, _ = _ragged(ktf, layer, W, S, flat, offs, snip)
            assert np.array_equal(out, again)
            for b, u in enumerate(utts):
                solo, sfo = _ragged(ktf, layer, W, S, u, np.array([0, len(u)], np.int64), snip)
                assert np.array_equal(out[fo[b]:fo[b + 1]], solo), (snip, b)
                uni = layer(ktf.layers.Framing(ms, 10.0, rate, dynamic_input_shape=True, snip_edges=snip)(u[None]))[0]
                assert np.array_equal(solo, uni), (snip, b)
        # ragged equals uniform for equal lengths
        eq = np.stack([utts[4], np.round(rng.standard_normal(10 * rate) * 100.0).astype(np.float32)])
        out, fo = _ragged(ktf, m, W, S, eq.reshape(-1), np.array([0, 10 * rate, 20 * rate], np.int64), snip)
        uni = m(ktf.layers.Framing(ms, 10.0, rate, dynamic_input_shape=True, snip_edges=snip)(eq))
        assert np.array_equal(out, uni.reshape(-1, uni.shape[-1]))
    # utterances shorter than the frame are rejected
    bad = np.array([0, W, 2 * W - 1], np.int64)
    with pytest.raises(ValueError):
        _ragged(ktf, m, W, S, flat[: 2 * W - 1], bad, True)


@pytest.mark.gpu
@pytest.mark.parametrize("rate", [32000, 48000, 96000])
def test_int16_bit_identical_to_float32(ktf, rate):
    import torch
    x = np.clip(_noise(rate, 1.0, seed=5, batch=3) * 4.0, -32768, 32767).astype(np.int16)
    x[1] = np.clip(np.round(_speech(rate, 1.0)[0]), -32768, 32767).astype(np.int16)
    for snip in (True, False):
        fr = ktf.layers.Framing(25.0, 10.0, rate, dynamic_input_shape=True, snip_edges=snip)
        for layer in (ktf.layers.MFCC(**_mfcc_kw(rate)), ktf.layers.MFCC(**_mfcc_kw(rate, dither=0.0, num_mels=80))):
            a16 = layer(fr(x))
            a32 = layer(fr(x.astype(np.float32)))
            assert a16.shape == a32.shape and np.array_equal(a16, a32)
        w16, e16 = ktf.layers.Windowing()(fr(x))
        w32, e32 = ktf.layers.Windowing()(fr(x.astype(np.float32)))
        assert np.array_equal(w16, w32) and np.array_equal(e16, e32)
        # odd offsets into the int16 buffer: ragged
        m = ktf.layers.MFCC(**_mfcc_kw(rate))
        W, S = fr.frameWidth, fr.frameShift
        offs = np.array([0, 3 * W + 1, 3 * W + 1 + 2 * W + S - 1, x.shape[1] + 5 * W], np.int64)
        flat = x.reshape(-1)[: offs[-1]]
        fe = m.frontend(W, S)
        o16, _ = fe.forward_ragged(torch.from_numpy(flat.copy()).cuda(), offs, snip)
        o32, _ = fe.forward_ragged(torch.from_numpy(flat.astype(np.float32)).cuda(), offs, snip)
        assert np.array_equal(o16.cpu().numpy(), o32.cpu().numpy())


@pytest.mark.gpu
def test_dither_48k_is_per_framed_sample(ktf):
    from kaldi_tflite_b200 import _native
    x = np.zeros((4, 48000), np.float32)
    fr = ktf.layers.Framing(25.0, 10.0, 48000.0, dynamic_input_shape=True)
    win = ktf.layers.Windowing(window_type="rectangular", dither=2.0, remove_dc_offset=False,
                               preemphasis_coefficient=0.0, return_energy=False)
    _native.lib().ktf_set_dither_seed(4321)
    a = win(fr(x))
    assert a.shape == (4, 98, 1200)
    z = a / 2.0
    assert abs(float(z.mean())) < 0.01 and abs(float(z.std()) - 1.0) < 0.01
    assert abs(float((z ** 3).mean())) < 0.03 and abs(float((z ** 4).mean()) - 3.0) < 0.1
    shared_a, shared_b = z[:, :-1, 480:], z[:, 1:, :720]     # frames t and t + 1 share 720 samples
    assert abs(float(np.mean(shared_a * shared_b))) < 0.01
    assert abs(float(np.mean(z[..., 1:] * z[..., :-1]))) < 0.01
    b = win(fr(x))
    assert abs(float(np.mean(a * b))) / 4.0 < 0.01
    _native.lib().ktf_set_dither_seed(4321)
    assert np.array_equal(win(fr(x)), a)
    # int16 input with dither goes to the kernel as PCM: the same draws as float32
    _native.lib().ktf_set_dither_seed(99)
    d16 = win(fr(x.astype(np.int16)))
    _native.lib().ktf_set_dither_seed(99)
    assert np.array_equal(d16, win(fr(x)))
    rng = np.random.default_rng(0)
    loud = np.round(rng.standard_normal((2, 48000)) * 3000).astype(np.float32)
    m0 = ktf.layers.MFCC(**_mfcc_kw(48000))(fr(loud))
    m1 = ktf.layers.MFCC(**_mfcc_kw(48000, dither=1.0))(fr(loud))
    assert 0.0 < float(np.max(np.abs(m1 - m0))) < 0.05


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mfcc", "fbank", "windowed"])
def test_ragged_output_stays_in_bounds(ktf, kind):
    import torch
    from kaldi_tflite_b200 import _native as N
    rate = 96000
    fr = ktf.layers.Framing(25.0, 10.0, rate, dynamic_input_shape=True)
    W, S = fr.frameWidth, fr.frameShift
    if kind == "mfcc":
        fe = ktf.layers.MFCC(**_mfcc_kw(rate)).frontend(W, S)
    elif kind == "fbank":
        layer = ktf.layers.FilterBank(num_bins=80, sample_frequency=float(rate))
        fe = layer._frontend(W, S)
    else:
        fe = ktf.layers.Windowing()._frontend(W, S)
    lens = [W, W + S - 1, 5 * W + 3, W + 1]
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    wav = torch.randn(int(offs[-1]), device="cuda") * 1000.0
    total = sum(fe.num_frames(n) for n in lens)
    G = 8
    buf = torch.full((G + total + G, fe.out_dim), float("nan"), device="cuda")
    energy = torch.full((G + total + G,), float("nan"), device="cuda")
    fo = np.zeros(len(lens) + 1, np.int64)
    N.check(N.lib().ktf_frontend_forward_ragged_ex(fe.handle, ctypes.c_void_p(wav.data_ptr()), N.KTF_SAMPLE_F32, 1,
                                                   len(lens), offs.ctypes.data_as(ctypes.c_void_p),
                                                   fo.ctypes.data_as(ctypes.c_void_p),
                                                   ctypes.c_void_p(buf[G:].data_ptr()),
                                                   ctypes.c_void_p(energy[G:].data_ptr()), None))
    torch.cuda.synchronize()
    b = buf.cpu().numpy()
    assert fo[-1] == total
    assert np.all(np.isnan(b[:G])) and np.all(np.isnan(b[G + total:]))
    assert np.all(np.isfinite(b[G:G + total]))
    e = energy.cpu().numpy()
    assert np.all(np.isnan(e[:G])) and np.all(np.isnan(e[G + total:]))


@pytest.mark.gpu
def test_cuda_graph_capture_48k(ktf):
    import torch
    rate = 48000
    fr = ktf.layers.Framing(25.0, 10.0, rate, dynamic_input_shape=True)
    m = ktf.layers.MFCC(**_mfcc_kw(rate))
    static = torch.from_numpy(_noise(rate, 2.0, seed=8, batch=4)).cuda()
    m(fr(static))                                   # builds the handle outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = m(fr(static))
    static.copy_(torch.from_numpy(_noise(rate, 2.0, seed=9, batch=4)).cuda())
    g.replay()
    torch.cuda.synchronize()
    eager = m(fr(static))
    assert torch.equal(out, eager)


@pytest.mark.gpu
def test_limits(ktf):
    # width 4097 needs an 8192-point FFT: rejected at build time, naming the maximum
    with pytest.raises(ValueError, match="4096"):
        ktf.layers.Windowing()(np.zeros((1, 2, 4097), np.float32))
    with pytest.raises(ValueError, match="4096"):
        ktf.layers.MFCC(**_mfcc_kw(48000))(np.zeros((1, 2, 4098), np.float32))
    # the largest accepted shift at width 4096 (2 x fft_length) runs; one more is rejected when the handle is built
    m = ktf.layers.MFCC(**_mfcc_kw(48000, num_mels=128))
    W, S = 4096, 8192
    fe = m.frontend(W, S)
    x = _noise(48000, (W + 5 * S) / 48000.0, seed=12)
    import torch
    out, _ = fe.forward(torch.from_numpy(x).cuda())
    frames = x[:, np.arange(6)[:, None] * S + np.arange(W)[None]]
    kw = _mfcc_kw(48000, num_mels=128)
    _gate(out.cpu().numpy(), O.mfcc(frames, precise=True, **kw), O.mfcc(frames, **kw), "shift 8192")
    with pytest.raises(ValueError):
        m.frontend(W, S + 1)
