"""
Element-wise parity of the stage between the MFCCs and tdnn1 on ragged batches: the VAD mask
(`vad_mask_kernel`), the stable compaction (`vad_count_kernel`, `scan_counts_kernel`, `vad_compact_kernel`,
`vad_gather_kernel`), the stand-alone sliding CMVN (`cmvn_staged_kernel` and its `cmvn_kernel` fallback, all in
csrc/vad_cmvn.cu) and the fused gather + CMVN + splice pre-pass of the tcgen05 stack (`gather_cmvn_splice_kernel`,
csrc/tdnn_tc.cu), which is the default wav -> x-vector path.

A pooled x-vector averages hundreds of frames, so a defect limited to the frames where one CTA hands over to the next,
to the clamped head and tail windows or to the edge taps of short utterances moves it less than a cosine gate allows.
These tests look at every element.

References (float64, per utterance):
  * VAD: the oracle on each utterance alone.  The kernel sums the energy mean in fp64 and rounds it once; the oracle
    sums in fp32.  A frame whose energy lies within that difference (plus 4 ulp for the kernel's own rounding) of the
    threshold may decide either way, and so may, with context, every frame whose vote window holds such a frame.
    These exceptions are counted and printed; every other frame must be equal.
  * Compaction: numpy's stable per-utterance argwhere.  Index list and offsets exact, gathered rows bit for bit.
  * CMVN: `_cmvn_f64` per utterance (VALID slicing per utterance).

CMVN gate.  u = 2^-24 is the unit roundoff of fp32, M the largest |x| of the utterance's column, so every window sum
is at most N M.  The kernels form a window sum from partial sums and then slide it, adding (x_new - x_old) once per
frame:
  * first window, worst kernel (`cmvn_kernel`: four partial sums of N / 4 rows): u M (N / 4)^2 / 2 per partial, four
    of them, u N^2 M / 8 in all, i.e. u N M / 8 <= 125 u M on the mean for N <= 1000 (the staged kernels sum 32-row
    blocks first and stay far below this);
  * sliding: at most 128 steps (`cmvn_kernel`; the staged kernels <= 33), each rounding a sum of magnitude <= N M
    (u M on the mean) and a difference of magnitude <= 2 M: 128 (1 + 2 / N) u M;
  * 1 / N, the product by it and x - mean: 4 u M more.
Altogether <= 260 u M = 1.55e-5 M on the mean and on the output: the gate is |got - ref| <= 2e-5 M.  A window that
is one frame off moves the mean by (x_new - x_old) / N, which on the data below is up to 3e-2 M / N or more: 1.5e3 / N
times the gate, 50x at N = 301 (the mutants below measure it).

With norm_vars the kernels also form v = s2 / N - mean^2.  s2 / N carries the bound above with M^2 in place of M
(2e-5 M^2); mean^2 carries 2 |mean| 2e-5 M <= 4e-5 M^2; the subtraction and the product by 1 / N u M^2 each:
E_v = 6.1e-5 M^2.  With sigma the window's standard deviation, sd = sqrt(v) has relative error
1 / sqrt(1 - E_v / sigma^2) - 1 (+ u for the square root), and y = (x - mean) / sd
  |got - y| <= 2e-5 M / sigma + |y| (1 / sqrt(1 - E_v / sigma^2) - 1 + 3 u).
The cancellation makes the bound grow with (M / sigma)^2, so the data keeps |mean| / sigma <= 10 (M / sigma <= ~15,
E_v / sigma^2 <= 0.014).  Elements with E_v > sigma^2 / 4 (a window of nearly equal values: two-frame utterances) are
outside what the arithmetic bounds; they are counted and printed.  Every gate here is derived from the operations, not
fitted to GPU results.

The fused pre-pass is read element-wise through a probe layer: one bf16 TDNN layer with U = K D, selection weights
(W[k D + d, k D + d] = 1), zero bias, no ReLU, no BatchNorm.  Each output element is then exactly one bf16 element of
the spliced operand (the products by 1.0 and the sums of zeros are exact in fp32), and must equal bf16(cmvn64) at the
clamped tap row, except where the float64 value lies within the CMVN gate of a bf16 rounding midpoint; there the bf16
value of any number within the gate is accepted (two neighbours; more only for |value| < ~5e-3 M, where the gate spans
more than one bf16 step).  Elements that took such a neighbour are counted and printed.

The CPU tests show that the references are right and that the gates catch the defects they are meant to catch; the
GPU tests hold the kernels to them.
"""

import numpy as np
import pytest

from oracle import ktf_oracle as O
from test_gpu_frontend import _cmvn_f64
from test_gpu_tc_stack_edges import bf16, build_sequential, emulate, gate, make_params, offsets_of, tap_rows, worst

F32 = np.float32
U = 2.0 ** -24

# ------------------------------------------------------------------------------------------------------------------
# Data
# ------------------------------------------------------------------------------------------------------------------


def feats_for(lengths, D, seed, energy_coeff=0):
    """Ragged (rows, D) fp32 features.  Every utterance has its own column means (|mean| / sigma <= 10, sigma in
    0.5 .. 3) so that a window reaching into a neighbour is visible; the energy column is N(u_b, 3^2) with a per
    utterance level u_b in 5 .. 15, so that the VAD threshold (and the mean it depends on) differs per utterance."""
    rng = np.random.default_rng(seed)
    out = []
    for T in lengths:
        sd = rng.uniform(0.5, 3.0, D)
        mu = rng.uniform(-10.0, 10.0, D) * sd
        x = mu + sd * rng.standard_normal((T, D))
        x[:, energy_coeff] = rng.uniform(5.0, 15.0) + 3.0 * rng.standard_normal(T)
        out.append(x)
    return (np.concatenate(out) if out else np.zeros((0, D))).astype(F32)


def shuffled(lengths, seed):
    lengths = list(lengths)
    np.random.default_rng(seed).shuffle(lengths)
    return lengths


# ------------------------------------------------------------------------------------------------------------------
# VAD reference
# ------------------------------------------------------------------------------------------------------------------

def vad_ref(x, offs, cfg, mutant=None):
    """Oracle mask of each utterance alone -> (rows,) float mask, (rows,) bool 'may differ' (see module docstring).
    mutant "batch_mean": the energy mean over the whole batch; "edge_in_range": edge divisors = taps inside the
    utterance instead of the reference's wrapped edge lists (differs for T <= 2 ctx)."""
    mask = np.zeros(len(x), F32)
    loose = np.zeros(len(x), bool)
    e_all = x[:, cfg["energy_coeff"]]
    ctx, scale, thr0 = cfg["frames_context"], F32(cfg["energy_mean_scale"]), F32(cfg["energy_threshold"])
    for b in range(len(offs) - 1):
        seg = x[offs[b]:offs[b + 1]]
        T = len(seg)
        if T == 0:
            continue
        e = seg[:, cfg["energy_coeff"]]
        if mutant == "batch_mean":
            thr = thr0 + scale * np.mean(e_all, dtype=F32) if scale > 0 else thr0
            m = vad_with_threshold(e, thr, ctx, cfg["proportion_threshold"])
        elif mutant == "edge_in_range":
            thr = thr0 + scale * np.mean(e, dtype=F32) if scale > 0 else thr0
            m = vad_with_threshold(e, thr, ctx, cfg["proportion_threshold"], in_range=True)
        else:
            m = O.vad(seg[None], return_indexes=False, **cfg)[0, :, 0]
        mask[offs[b]:offs[b + 1]] = m
        # threshold of the oracle (fp32 mean) and the exact one (what the kernel's fp64 mean rounds to)
        c = cfg["energy_coeff"]
        thr32 = thr0 + scale * np.mean(seg[None, :, c:c + 1], axis=-2, dtype=F32)[0, 0] if scale > 0 else thr0
        thr64 = float(thr0) + float(scale) * float(np.mean(e.astype(np.float64)))
        band = abs(float(thr32) - thr64) + 4 * float(np.spacing(F32(abs(thr64))))
        near = np.abs(e.astype(np.float64) - thr64) <= band
        if ctx > 0:
            near = np.convolve(near.astype(np.int64), np.ones(2 * ctx + 1, np.int64), mode="full")[ctx:ctx + T] > 0
        loose[offs[b]:offs[b + 1]] = near
    return mask, loose


def vad_with_threshold(e, thr, ctx, prop, in_range=False):
    """The oracle's decision rule (vad.py:168-199) for a given threshold, float32 like the oracle."""
    dec = (e > thr).astype(F32)
    if ctx == 0:
        return dec
    T, N = len(e), 2 * ctx + 1
    counts = np.convolve(dec, np.ones(N, F32), mode="full")[ctx:ctx + T].astype(F32)
    if in_range:
        t = np.arange(T)
        sizes = (np.minimum(t + ctx, T - 1) - np.maximum(t - ctx, 0) + 1).astype(F32)
    else:
        sizes = np.full(T, N, F32)
        for i, s in zip(list(range(0, ctx)) + list(range(-ctx, 0)),
                        list(range(ctx + 1, N)) + list(range(N - 1, ctx, -1))):
            sizes[(i + T) % T] = s
    return ((counts / sizes).astype(F32) >= F32(prop)).astype(F32)


def compact_ref(mask, offs):
    """Stable per-utterance argwhere -> (index, out_offsets)."""
    keep = mask != 0
    counts = [int(keep[offs[b]:offs[b + 1]].sum()) for b in range(len(offs) - 1)]
    return np.flatnonzero(keep).astype(np.int64), offsets_of(counts)


# ------------------------------------------------------------------------------------------------------------------
# CMVN reference and gate
# ------------------------------------------------------------------------------------------------------------------

MEAN_TOL = 2e-5                   # |error| of the mean (and, without norm_vars, of the output) over M
VAR_TOL = 6.1e-5                  # |error| of the window variance over M^2


def valid_frames(T, window):
    return np.arange(T)[window // 2: T - (window - 1) // 2]


def cmvn_windows(T, N, mutant=None):
    """(start, width) of the statistics window of every frame of a T-frame utterance (cmvn.py:172-222)."""
    t = np.arange(T)
    if T <= N or (mutant == "global_at_N_plus_1" and T == N + 1):
        return np.zeros(T, np.int64), np.full(T, max(T, 1))
    start = np.clip(t - N // 2, 0, T - N)
    if mutant == "late_clamp":                    # the start clamped at T - N + 1: the last window reads one row past
        start = np.clip(t - N // 2, 0, T - N + 1)
    if mutant == "head_shift":                    # the windows clamped at the head start one frame late
        start = np.where(t - N // 2 < 0, 1, start)
    return start, np.full(T, N)


def window_stats(src, a, w):
    """Mean and variance of src[a : a + w] per frame, from cumulative sums of the centred rows (a one-frame window has
    variance 0 exactly, as in the kernels)."""
    c = src.mean(0) if len(src) else 0.0
    z = src - c
    cs = np.concatenate([np.zeros((1, src.shape[1])), np.cumsum(z, 0)])
    cs2 = np.concatenate([np.zeros((1, src.shape[1])), np.cumsum(z * z, 0)])
    n = w[:, None].astype(np.float64)
    m = (cs[a + w] - cs[a]) / n
    return m + c, (cs2[a + w] - cs2[a]) / n - m * m


def cmvn_batch(x, offs, window, norm_vars, padding, mutant=None):
    """float64 CMVN of every utterance of a ragged batch.  Returns out (rows_out, D), out offsets, and per output
    element M (largest |x| of the utterance's column) and sigma (the window's standard deviation)."""
    x = np.asarray(x, np.float64)
    R, D = x.shape
    outs, Ms, sds, lens = [], [], [], []
    for b in range(len(offs) - 1):
        r0, T = int(offs[b]), int(offs[b + 1] - offs[b])
        if mutant == "cross_utterance":           # the batch as one sequence
            st, w = cmvn_windows(R, window)
            mean, var = window_stats(x, st[r0:r0 + T], w[r0:r0 + T])
        else:
            st, w = cmvn_windows(T, window + 1 if mutant == "window_plus_one" else window, mutant)
            # one row past the utterance: the neighbour's first row (what a late clamp reads), or zeros at the end
            src = np.concatenate([x[r0:r0 + T], x[r0 + T:r0 + T + 1] if r0 + T < R else np.zeros((1, D))])
            mean, var = window_stats(src, st, w)
        seg = x[r0:r0 + T]
        with np.errstate(invalid="ignore", divide="ignore"):
            sd = np.sqrt(np.maximum(var, 0.0))
            y = (seg - mean) / sd if norm_vars else seg - mean
        keep = np.arange(T) if padding == "SAME" else valid_frames(T, window)
        if mutant == "valid_shift" and padding == "VALID":
            keep = np.minimum(keep + 1, T - 1)
        M = np.max(np.abs(seg), axis=0) if T else np.zeros(D)
        outs.append(y[keep])
        sds.append(sd[keep])
        Ms.append(np.broadcast_to(M, (len(keep), D)))
        lens.append(len(keep))
    cat = lambda a: np.concatenate(a) if a else np.zeros((0, D))
    return cat(outs), offsets_of(lens), cat(Ms), cat(sds)


def cmvn_bound(want, M, sd, norm_vars):
    """Per-element bound of the module docstring; NaN where the arithmetic gives no bound (E_v > sigma^2 / 4)."""
    if not norm_vars:
        return MEAN_TOL * M
    with np.errstate(invalid="ignore", divide="ignore"):
        q = VAR_TOL * M * M / (sd * sd)
        b = MEAN_TOL * M / sd + np.abs(want) * (1.0 / np.sqrt(1.0 - q) - 1.0 + 3 * U)
    return np.where(q <= 0.25, b, np.nan)


def cmvn_gate(got, want, M, sd, norm_vars):
    """-> (worst |error| / bound, elements outside the bound's domain).  NaN must match NaN (0 / 0 of a one-frame
    utterance with norm_vars): a different NaN pattern is an infinite miss."""
    got = np.asarray(got, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    nan_w = np.isnan(want)
    if not np.array_equal(np.isnan(got), nan_w):
        return np.inf, 0
    bound = cmvn_bound(want, M, sd, norm_vars)
    ok = ~nan_w & np.isfinite(bound)
    if not ok.any():
        return 0.0, int((~nan_w & ~ok).sum())
    frac = np.abs(got[ok] - want[ok]) / np.maximum(bound[ok], 1e-300)
    return float(np.max(frac)), int((~nan_w & ~ok).sum())


def splice_rule(got, want, bound):
    """bf16 operand rule: got == bf16(want), or either neighbour where want is within `bound` of a rounding midpoint.
    -> number of elements that used the exception; asserts the rule."""
    lo, hi = bf16(want - bound), bf16(want + bound)
    exact = lo == hi
    bad_exact = exact & (got != lo)
    bad_mid = ~exact & ((got < lo) | (got > hi))
    assert not bad_exact.any() and not bad_mid.any(), (
        f"{int(bad_exact.sum())} exact and {int(bad_mid.sum())} midpoint elements off; first at "
        f"{np.argwhere(bad_exact | bad_mid)[:5].tolist()}")
    return int((~exact & (got != bf16(want))).sum())


# ------------------------------------------------------------------------------------------------------------------
# The pre-pass tile rule (mirrors prepass_tile / prepass_smem_bytes in csrc/tdnn_tc.cu, so the tests know which tile
# edges a batch hits; the GPU test checks this mirror against ktf_tdnn_stack_vad_prepass_fits)
# ------------------------------------------------------------------------------------------------------------------

def prepass_tc(max_frames, window, D):
    def smem(tc):
        a = ((tc + 8 + window) * D + 3) & ~3
        y = ((tc + 8) * D + 8 + 3) & ~3
        blk = (((tc + 8 + window) // 32 + 2) * D + 1) & ~1
        return (a + y + blk) * 4 + (tc + 8 + window) * 8
    for target in range(256, 31, -2):
        gys = -(-max_frames // target)
        tc = ((-(-max_frames // gys)) + 1) & ~1
        if gys <= 65535 and smem(tc) <= 113 * 1024:
            return tc
    return None


def cmvn_staged(dim, window, norm_vars, max_frames):
    """Which kernel ktf_cmvn_forward takes (the rule in csrc/vad_cmvn.cu): True = cmvn_staged_kernel."""
    gys = -(-max_frames // 256)
    tc = ((-(-max_frames // gys)) + 1) & ~1
    smem = ((((tc + window) * dim + 4 + 3) & ~3) + (2 if norm_vars else 1) * ((tc + window) // 32 + 1) * dim) * 4
    return smem <= 113 * 1024 and gys <= 65535


# ------------------------------------------------------------------------------------------------------------------
# CPU: the references are right and the gates have teeth
# ------------------------------------------------------------------------------------------------------------------

def test_cmvn_f64_is_the_oracle():
    """The oracle is fp32 and takes window sums as differences of one cumulative sum over the whole utterance: it
    agrees with the float64 reference to a few ulp of that sum, divided by the window."""
    rng = np.random.default_rng(1)
    x = (rng.standard_normal((3, 700, 23)) * 2 + rng.uniform(-10, 10, (3, 1, 23))).astype(F32)
    csmax = np.max(np.abs(np.cumsum(x.astype(np.float64), axis=1)))
    for window in (1, 2, 7, 64, 300, 301, 699, 700, 701):
        for nv in ((False, True) if window >= 64 else (False,)):
            for padding in ("SAME", "VALID"):
                want = O.cmvn(x, window=window, norm_vars=nv, padding=padding)
                got = _cmvn_f64(x, window, nv, padding)
                assert got.shape == want.shape
                if want.size == 0:
                    continue
                err = np.max(np.abs(got - want))
                tol = 16 * U * csmax / min(window, 700) + 1e-5
                assert err < (1e-3 if nv else tol), (window, nv, padding, err, tol)


CPU_LENGTHS = [0, 1, 2, 6, 7, 8, 63, 64, 65, 300, 0, 301, 302, 5]


@pytest.mark.parametrize("window,norm_vars", [(1, False), (2, False), (7, False), (7, True), (64, True),
                                              (301, False), (301, True)])
@pytest.mark.parametrize("padding", ["SAME", "VALID"])
def test_cmvn_ragged_reference_equals_solo_runs(window, norm_vars, padding):
    offs = offsets_of(CPU_LENGTHS)
    x = feats_for(CPU_LENGTHS, 7, seed=2)
    out, oo, _, _ = cmvn_batch(x, offs, window, norm_vars, padding)
    for b, T in enumerate(CPU_LENGTHS):
        part = out[oo[b]:oo[b + 1]]
        solo = _cmvn_f64(x[offs[b]:offs[b + 1]][None], window, norm_vars, padding)[0] if T else np.zeros((0, 7))
        assert part.shape == solo.shape, (b, T)
        # (norm_vars: _cmvn_f64 takes s2 / N - mean^2 from uncentred cumulative sums, which cancels in float64 too
        # for windows of two nearly equal frames)
        tol = 1e-6 if norm_vars else 1e-9
        np.testing.assert_allclose(part, solo, rtol=tol, atol=tol, equal_nan=True)


def test_vad_ragged_reference_equals_solo_runs():
    lengths = [0, 1, 2, 3, 4, 5, 6, 255, 256, 257]
    offs = offsets_of(lengths)
    x = feats_for(lengths, 5, seed=3)
    for ctx in (0, 1, 2, 5):
        cfg = dict(energy_mean_scale=0.5, energy_threshold=5.5, frames_context=ctx, proportion_threshold=0.6,
                   energy_coeff=0)
        mask, _ = vad_ref(x, offs, cfg)
        # the rule restated with the threshold is the oracle
        for b in range(len(lengths)):
            e = x[offs[b]:offs[b + 1], 0]
            if len(e):
                thr = F32(5.5) + F32(0.5) * np.mean(e, dtype=F32)
                np.testing.assert_array_equal(vad_with_threshold(e, thr, ctx, 0.6), mask[offs[b]:offs[b + 1]])
        # the per-utterance reference is the oracle on a uniform batch of those utterances
        same = [b for b, T in enumerate(lengths) if T == 256]
        uni = O.vad(np.stack([x[offs[b]:offs[b + 1]] for b in same]), return_indexes=False, **cfg)
        np.testing.assert_array_equal(uni[0, :, 0], mask[offs[same[0]]:offs[same[0] + 1]])


CMVN_MUTANTS = ["window_plus_one", "late_clamp", "head_shift", "global_at_N_plus_1", "valid_shift", "cross_utterance"]


@pytest.mark.parametrize("norm_vars", [False, True])
@pytest.mark.parametrize("mutant", CMVN_MUTANTS)
def test_cmvn_gate_rejects_mutants(mutant, norm_vars):
    window = 301
    lengths = [5, 300, 301, 302, 700, 2, 1000]
    offs = offsets_of(lengths)
    x = feats_for(lengths, 23, seed=4)
    padding = "VALID" if mutant == "valid_shift" else "SAME"
    want, _, M, sd = cmvn_batch(x, offs, window, norm_vars, padding)
    assert cmvn_gate(want, want, M, sd, norm_vars)[0] == 0.0
    bad, _, _, _ = cmvn_batch(x, offs, window, norm_vars, padding, mutant=mutant)
    # a mutant's NaN pattern matches here (only the one-frame utterance is NaN): the gate decides
    miss, _ = cmvn_gate(bad, want, M, sd, norm_vars)
    print(f"[vad-cmvn] CMVN mutant {mutant} (norm_vars={norm_vars}): misses the gate by {miss:.0f}x")
    assert miss >= 10.0, miss


def test_sliding_branch_at_T_equal_N_is_the_global_mean():
    """At T = N the only window is the whole utterance, so 'the sliding branch at T = N' computes the global mean:
    no gate can (or needs to) tell the branches apart there.  The boundary is held by the T = N + 1 mutant."""
    x = feats_for([64], 5, seed=5).astype(np.float64)
    st, w = np.clip(np.arange(64) - 32, 0, 0), 64
    sliding = x - np.stack([x[s:s + w].mean(0) for s in st])
    np.testing.assert_allclose(sliding, _cmvn_f64(x[None], 64, False, "SAME")[0], rtol=0, atol=1e-12)


VAD_MUTANT_CFG = dict(energy_mean_scale=0.5, energy_threshold=5.5, proportion_threshold=0.6, energy_coeff=0)


@pytest.mark.parametrize("mutant", ["batch_mean", "edge_in_range"])
def test_vad_reference_rejects_mutants(mutant):
    """The VAD gate is equality outside the exceptions, so a mutant's factor is its count of differing frames."""
    lengths = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 200, 3, 2, 1, 4] * 4
    offs = offsets_of(lengths)
    x = feats_for(lengths, 5, seed=6)
    cfg = dict(VAD_MUTANT_CFG, frames_context=5)
    want, loose = vad_ref(x, offs, cfg)
    bad, _ = vad_ref(x, offs, cfg, mutant=mutant)
    miss = int(((bad != want) & ~loose).sum())
    print(f"[vad-cmvn] VAD mutant {mutant}: {miss} frames differ outside the exceptions ({miss}x the gate)")
    assert miss >= 10, miss


def test_compaction_reference_rejects_reversed_chunk():
    lengths = [300, 256, 600, 7]
    offs = offsets_of(lengths)
    mask = (np.random.default_rng(7).random(sum(lengths)) < 0.5).astype(F32)
    index, oo = compact_ref(mask, offs)
    bad = index.copy()
    b = 2                                          # the second 256-frame chunk of utterance 2, reversed
    sel = (bad >= offs[b] + 256) & (bad < offs[b] + 512)
    bad[sel] = bad[sel][::-1]
    miss = int((bad != index).sum())
    print(f"[vad-cmvn] compaction mutant reversed chunk: {miss} indices differ ({miss}x the gate)")
    assert miss >= 10, miss


def test_vad_exceptions_are_rare_on_the_test_data():
    """The 'may differ' band is a few ulp wide: on the test data it holds next to no frame, so the equality gate is
    not hollowed out by it."""
    lengths = shuffled(VAD_LENGTHS_BASE + [4, 5, 6], 8)
    offs = offsets_of(lengths)
    x = feats_for(lengths, 30, seed=9)
    for ctx in (0, 5):
        _, loose = vad_ref(x, offs, dict(VAD_MUTANT_CFG, frames_context=ctx))
        assert loose.sum() <= 1e-3 * len(x), int(loose.sum())


def test_gpu_case_lists_cover_both_cmvn_kernels_and_prepass_tiles():
    for nv in (False, True):
        kinds = {(dim, w): cmvn_staged(dim, w, nv, 2000 * 3) for dim, ws in CMVN_CASES for w in ws}
        assert kinds[(30, 600)] and kinds[(23, 600)] and kinds[(80, 64)], nv
        assert not kinds[(30, 1000)] and not kinds[(80, 300)] and not kinds[(23, 1000)], nv
    # the pre-pass table: largest window per feature dim at tc = 256 (long utterances) and at the smallest tile
    for D, w256, w32 in ((23, 623, 1047), (30, 372, 800), (40, 158, 590), (80, None, 262)):
        assert (prepass_tc(4096, w256, D) == 256) if w256 else prepass_tc(4096, 1, D) < 256
        assert w256 is None or prepass_tc(4096, w256 + 1, D) < 256
        assert prepass_tc(4096, w32, D) == 32 and prepass_tc(4096, w32 + 1, D) is None
    assert prepass_tc(998, 300, 30) == 250 and prepass_tc(768, 300, 30) == 256
    assert prepass_tc(998, 300, 80) is None


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ktf():
    import kaldi_tflite_b200 as k
    return k


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


VAD_LENGTHS_BASE = [0, 1, 2, 3, 255, 256, 257, 4095, 4096, 4097, 9000]


def vad_lengths(ctx, seed):
    extra = [4, 5] + [c for c in (ctx - 1, ctx, ctx + 1) if c >= 0]
    return shuffled(VAD_LENGTHS_BASE + extra, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("dim,coeff", [(5, 0), (23, 3), (30, 0), (30, 3)])
def test_vad_mask_and_compaction_on_ragged_batches(ktf, dim, coeff):
    loose_total, n = 0, 0
    for ctx in (0, 1, 2, 5):
        lengths = vad_lengths(ctx, seed=10 + ctx)
        offs = offsets_of(lengths)
        x = feats_for(lengths, dim, seed=100 * dim + ctx, energy_coeff=coeff)
        xd, od = dev(x), dev(offs)
        for scale, thr0 in ((0.0, 10.0), (0.5, 5.5)):
            cfg = dict(energy_mean_scale=scale, energy_threshold=thr0, frames_context=ctx, proportion_threshold=0.6,
                       energy_coeff=coeff)
            vad = ktf.layers.VAD(**cfg)
            got = vad.mask_ragged(xd, od).cpu().numpy()
            want, loose = vad_ref(x, offs, cfg)
            diff = got != want
            assert not (diff & ~loose).any(), (ctx, scale, np.flatnonzero(diff & ~loose)[:10])
            loose_total += int((diff & loose).sum())
            n += len(x)
            # compaction of the library's own mask
            out, oo, index = vad.compact_ragged(xd, dev(got), od, gather=True)
            idx_ref, oo_ref = compact_ref(got, offs)
            np.testing.assert_array_equal(oo.cpu().numpy(), oo_ref)
            kept = int(oo_ref[-1])
            np.testing.assert_array_equal(index[:kept].cpu().numpy(), idx_ref)
            np.testing.assert_array_equal(out[:kept].cpu().numpy(), x[idx_ref])
    print(f"[vad-cmvn] VAD dim {dim} coeff {coeff}: {n} frames, {loose_total} threshold-tie exceptions")


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [23, 30])
def test_compaction_many_utterances_and_extremes(ktf, dim):
    """1500 and 3000 utterances (2 and 3 passes of the 1024-thread scan), zero kept rows, every row kept."""
    for B, p in ((1500, 0.5), (3000, 0.5), (40, 0.0), (40, 1.0), (1025, 0.3)):
        rng = np.random.default_rng(B + dim)
        lengths = list(rng.integers(0, 40, B))
        lengths[:3] = [257, 0, 512]
        offs = offsets_of(lengths)
        x = feats_for(lengths, dim, seed=B)
        mask = (rng.random(len(x)) < p).astype(F32)
        out, oo, index = ktf.layers.VAD.compact_ragged(dev(x), dev(mask), dev(offs), gather=True)
        idx_ref, oo_ref = compact_ref(mask, offs)
        np.testing.assert_array_equal(oo.cpu().numpy(), oo_ref, err_msg=f"B={B} p={p}")
        kept = int(oo_ref[-1])
        np.testing.assert_array_equal(index[:kept].cpu().numpy(), idx_ref)
        np.testing.assert_array_equal(out[:kept].cpu().numpy(), x[idx_ref])


# stand-alone CMVN: (dim, windows); dim 23 rows start misaligned (cp.async head / tail copies)
CMVN_CASES = [(30, [1, 2, 7, 64, 300, 301, 600, 1000]), (23, [7, 301, 600, 1000]), (80, [64, 300])]


def cmvn_lengths(N, seed):
    return shuffled([0, 1, N - 1, N, N + 1, 255, 256, 257, 513, 2000, 0], seed)


@pytest.mark.gpu
@pytest.mark.parametrize("dim,windows", CMVN_CASES, ids=[f"d{d}" for d, _ in CMVN_CASES])
def test_cmvn_forward_ragged(ktf, dim, windows):
    worst_frac = {False: 0.0, True: 0.0}
    unbounded = 0
    for N in windows:
        lengths = cmvn_lengths(N, seed=N + dim)
        offs = offsets_of(lengths)
        x = feats_for(lengths, dim, seed=N * dim)
        xd, od = dev(x), dev(offs)
        for nv in ((False, True) if N >= 64 else (False,)):
            for padding in ("SAME", "VALID"):
                want, oo, M, sd = cmvn_batch(x, offs, N, nv, padding)
                layer = ktf.layers.CMVN(window=N, norm_vars=nv, padding=padding)
                for mf in (max(lengths), len(x)):
                    got, go = layer.forward_ragged(xd, od, max_frames=mf)
                    np.testing.assert_array_equal(go.cpu().numpy(), oo)
                    frac, nb = cmvn_gate(got.cpu().numpy(), want, M, sd, nv)
                    kind = "staged" if cmvn_staged(dim, N, nv, mf) else "fallback"
                    assert frac <= 1.0, (N, nv, padding, mf, kind, frac)
                    worst_frac[nv] = max(worst_frac[nv], frac)
                    unbounded += nb
    print(f"[vad-cmvn] CMVN dim {dim}: worst {worst_frac[False]:.3f} of the gate, norm_vars "
          f"{worst_frac[True]:.3f}; {unbounded} ill-conditioned norm_vars elements")


@pytest.mark.gpu
def test_cmvn_kernel_choice_follows_the_rule(ktf):
    """The mirror of ktf_cmvn_forward's rule above is the library's: the profiler names the kernel that ran."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    lengths = [2000, 300, 1]
    od = dev(offsets_of(lengths))
    cases = [(30, 600, False), (30, 1000, False), (23, 600, True), (80, 300, False)]
    for dim, N, nv in cases:
        xx = dev(feats_for(lengths, dim, seed=dim))
        layer = ktf.layers.CMVN(window=N, norm_vars=nv)
        layer.forward_ragged(xx, od, max_frames=2000)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            layer.forward_ragged(xx, od, max_frames=2000)
            torch.cuda.synchronize()
        names = [e.key for e in prof.key_averages() if "cmvn" in e.key]
        staged = any("cmvn_staged_kernel" in k for k in names)
        assert staged == cmvn_staged(dim, N, nv, 2000), (dim, N, nv, names)
        assert names, (dim, N, nv)


# ---- fused pre-pass through a probe layer -----------------------------------------------------------------------

PROBE_CTX = [[-2, -1, 0, 1, 2], [0], [-4, -3, -2, -1, 0, 1, 2, 3, 4], [-3, -2, -1, 0], [0, 1, 2, 3]]


def probe_params(D, ctx):
    K = len(ctx)
    return [{"W": np.eye(K * D, dtype=F32), "b": np.zeros(K * D, F32), "ctx": list(ctx), "relu": False}]


def spliced(a, offs, ctx):
    """Rows of the first layer's operand: a[clamped tap row] for every tap, per utterance."""
    return a[tap_rows(offs, ctx)].reshape(len(a), -1)


def prepass_batches(D, N):
    """(mode, compacted lengths, max_frames) for one (D, window): max_frames giving tc = 256 (a multiple of 256), giving
    tc = 250 (998 frames), and a loose bound (None: the row count of the un-compacted features).  The lengths hit the
    window (N - 1, N, N + 1), the tile (tc - 1, tc, tc + 1, 2 tc + 3) and the taps (K - 1) of every probe."""
    out = []
    for mode in ("tile", "998", "loose"):
        mf = 998 if mode == "998" else 256 * (-(-max(N + 2, 515) // 256))
        if mode == "998" and N + 1 > 998:
            continue
        tc = prepass_tc(mf, N, D)
        ks = sorted({len(c) - 1 for c in PROBE_CTX})
        lengths = [0, 1, 2, 4, N - 1, N, N + 1, tc - 1, tc, tc + 1, 2 * tc + 3, 0] + ks
        lengths = shuffled([l for l in lengths if 0 <= l <= mf], seed=N + D + len(mode))
        out.append((mode, lengths, None if mode == "loose" else mf, tc))
    return out


def with_dropped_rows(lengths, D, seed):
    """Un-compacted utterances (the kept rows plus up to 40 dropped ones, at random places) and their keep mask."""
    rng = np.random.default_rng(seed)
    full = [l + int(rng.integers(0, 40)) for l in lengths]
    foffs = offsets_of(full)
    x = feats_for(full, D, seed=seed)
    mask = np.zeros(len(x), F32)
    for b, l in enumerate(lengths):
        mask[foffs[b] + rng.choice(full[b], l, replace=False)] = 1.0
    return x, foffs, mask


@pytest.mark.gpu
@pytest.mark.parametrize("D", [23, 30])
def test_fused_prepass_elementwise(ktf, D):
    largest = max(w for w in range(1, 2000) if prepass_tc(4096, w, D) is not None)
    stacks = {tuple(c): build_sequential(ktf, probe_params(D, c))._stack for c in PROBE_CTX}
    # the tile-rule mirror agrees with the library's fit test, at the tile boundaries and past the largest window
    probe = stacks[tuple(PROBE_CTX[0])]
    for mf in (1, 31, 32, 250, 998, 4096, 100000):
        for w in (1, 300, 372, 373, 623, 624, largest, largest + 1, 2000):
            assert probe.can_fuse_vad_cmvn(w, mf) == (prepass_tc(mf, w, D) is not None), (mf, w)
    beyond, mids, n_el, tiles = {"fused": 0.0, "separate": 0.0}, {"fused": 0, "separate": 0}, 0, set()
    for N in (1, 2, 300, 301, largest):
        for mode, lengths, mf, tc in prepass_batches(D, N):
            tiles.add(tc)
            x, foffs, mask = with_dropped_rows(lengths, D, seed=N + 7 * D + len(mode))
            _, voffs_d, index_d = ktf.layers.VAD.compact_ragged(dev(x), dev(mask), dev(foffs), gather=False)
            idx_ref, voffs = compact_ref(mask, foffs)
            np.testing.assert_array_equal(voffs_d.cpu().numpy(), voffs)
            kept = int(voffs[-1])
            xc = x[idx_ref]
            cm, _, M, _ = cmvn_batch(xc, voffs, N, False, "SAME")
            max_frames = len(x) if mf is None else mf
            xd, xcd = dev(x), dev(xc)
            # the separate path on the same rows: gathered rows -> CMVN -> the stack's own splice
            normed, _ = ktf.layers.CMVN(window=N).forward_ragged(xcd, voffs_d, max_frames=max_frames)
            for ctx in PROBE_CTX:
                stack = stacks[tuple(ctx)]
                want = spliced(cm, voffs, ctx)
                bound = spliced(MEAN_TOL * M, voffs, ctx)
                lo, hi, bw = bf16(want - bound), bf16(want + bound), bf16(want)
                exact = lo == hi
                runs = {"fused": [stack.forward_vad(xd, index_d, voffs_d, max_frames, N),      # through the index
                                  stack.forward_vad(xcd, None, voffs_d, max_frames, N)],       # contiguous rows
                        "separate": [stack.forward_ragged(normed, voffs_d)]}
                for path, outs in runs.items():
                    for got in outs:
                        got = got[:kept].cpu().numpy().astype(np.float64)
                        # every element is bf16(want); within the CMVN gate of a rounding midpoint either neighbour
                        off = (exact & (got != bw)) | (got < lo) | (got > hi)
                        assert not off.any(), (path, N, mode, ctx, int(off.sum()), np.argwhere(off)[:5].tolist())
                        mids[path] += int((~exact & (got != bw)).sum())
                        if kept:
                            beyond[path] = max(beyond[path], float(np.max(
                                np.maximum(np.abs(got - want) - np.abs(bw - want), 0.0) / bound)))
                n_el += want.size
    assert {256, 250, 32} <= tiles, tiles
    print(f"[vad-cmvn] pre-pass D {D}: {n_el} spliced elements per run, tiles {sorted(tiles)}, largest window "
          f"{largest}; error beyond the bf16 rounding: fused {beyond['fused']:.3f}, separate {beyond['separate']:.3f} "
          f"of the CMVN gate; elements on a neighbour of bf16(ref): fused {mids['fused']}, separate {mids['separate']}")


# ---- end to end and the extractor -------------------------------------------------------------------------------

@pytest.mark.gpu
def test_sitw_shaped_stack_through_prepass_vs_emulation(ktf):
    """The SITW-shaped pooled stack of the stack-edge tests through the pre-pass, against the float64 emulation of
    CMVN + network: an element-wise gate where the extractor tests hold a cosine."""
    from test_gpu_tc_stack_edges import POOLED_STACKS
    name, D, spec, stats_after, include_std = POOLED_STACKS[2]
    params = make_params(spec, D, 31, stats_after, include_std)
    mdl = build_sequential(ktf, params, stats_after, include_std)
    lengths = shuffled([1, 2, 3, 5, 255, 256, 257, 299, 300, 301, 600, 601, 998, 2000], 32)
    x, foffs, mask = with_dropped_rows(lengths, D, seed=34)
    _, voffs_d, index_d = ktf.layers.VAD.compact_ragged(dev(x), dev(mask), dev(foffs), gather=False)
    idx_ref, voffs = compact_ref(mask, foffs)
    U = params[stats_after]["W"].shape[0]
    for N in (300, 600):
        cm, _, _, _ = cmvn_batch(x[idx_ref], voffs, N, False, "SAME")
        got = mdl._stack.forward_vad(dev(x), index_d, voffs_d, 2000, N).cpu().numpy()
        g = gate(got, emulate(cm, voffs, params, stats_after, include_std), pooled_units=U)
        print(f"[vad-cmvn] SITW-shaped stack through the pre-pass, window {N} (tc {prepass_tc(2000, N, D)}): "
              + ", ".join(f"{k} {v:.3f} of the gate" for k, v in sorted(g.items())))
        assert worst(g) <= 1.0, (N, g)


def small_model_config(tmp_path, D):
    """An x-vector TDNN of the SITW shape for D-dim features (5-tap first layer, pooling, a 512-dim embedding)."""
    import yaml
    arb = ["affine", "relu", "batchnorm"]
    layers = [{"name": "input", "type": "input", "shape": [None, None, D]},
              {"name": "tdnn1", "type": arb, "cfg": {"units": 256, "context": [-2, -1, 0, 1, 2]}},
              {"name": "tdnn2", "type": arb, "cfg": {"units": 256, "context": [-2, 0, 2]}},
              {"name": "tdnn5", "type": arb, "cfg": {"units": 512, "context": [0]}},
              {"name": "stats", "type": "stats_pooling",
               "cfg": {"left_context": 0, "right_context": 10000, "include_std": True, "reduce_time_axis": True}},
              {"name": "tdnn6", "type": "affine", "cfg": {"units": 512, "context": [0]}}]
    path = tmp_path / f"tdnn_{D}.yml"
    path.write_text(yaml.safe_dump({"model_config": {"type": "sequential", "layers": layers}}))
    return str(path)


EXTRACTOR_CASES = {"sitw_window600": (30, 600), "d40_window300": (40, 300), "d80_window300": (80, 300),
                   "sitw_window300": (30, 300)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(EXTRACTOR_CASES))
def test_extractor_takes_any_cmvn_window(ktf, tmp_path, case):
    """The fused pre-pass takes what the separate kernels compute: a smaller tile for a wide window, and the separate
    kernels when no tile fits (D 80).  Where the pre-pass fits it is taken: gather, CMVN and splice are one launch.
    The front-end makes at most 32 cepstra, so 40- and 80-dim features enter at `embed`; the SITW cases also run
    from the waveform."""
    import torch
    from conftest import golden_path, read_wav_int16
    from test_gpu_tdnn_plda import extractor_cfg
    D, window = EXTRACTOR_CASES[case]
    cfg = extractor_cfg()
    cfg["cmvn"]["window"] = window
    if D != 30:
        cfg["xvec"]["model_config_path"] = small_model_config(tmp_path, D)
    ext = ktf.models.XvectorExtractor(cfg, seed=0, allow_random_init=True)
    fits = prepass_tc(4096, window, D) is not None
    assert fits == (case != "d80_window300")
    lengths = shuffled([1, 7, 120, 298, 301, 599, 600, 601, 998, 2000], 40)
    x = dev(feats_for(lengths, D, seed=41))
    od = dev(offsets_of(lengths))
    runs = {"features": lambda: ext.embed(x, od, max_frames=max(lengths))[0]}
    if D == 30:
        wav = read_wav_int16(golden_path("librispeech_2.wav"))
        batch = [torch.from_numpy(a.copy()).cuda() for a in (wav[:80000], wav[80000:200000], wav[:24000], wav[150000:])]
        runs["waveform"] = lambda: ext(batch)
    for src, run in runs.items():
        out, launches = {}, {}
        for fused in (True, False):
            ext.fusePrepass = fused
            run()                                      # warm-up: plans, workspaces
            n0 = ktf.launch_count()
            out[fused] = run().cpu().numpy()
            launches[fused] = ktf.launch_count() - n0
        assert launches[True] == launches[False] - (2 if fits else 0), (src, launches, fits)
        silent = np.isnan(out[False]).all(axis=1)     # no voiced frame: NaN on both paths
        assert np.array_equal(np.isnan(out[True]).any(axis=1), silent), src
        g = gate(out[True][~silent], out[False][~silent], pooled_units=out[True].shape[1])
        print(f"[vad-cmvn] extractor {case} from {src}: pre-pass {'taken' if fits else 'not taken (no tile fits)'}, "
              f"fused vs separate {g['mean']:.3f} of the pooled gate")
        assert worst(g) <= 1.0, (src, g)
