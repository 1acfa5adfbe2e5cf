"""
Element-wise parity of the tcgen05 TDNN stack (csrc/tdnn_tc.cu) at the places a pooled-x-vector cosine cannot see:
utterance edges and tiny utterances, utterances sharing a tile, padded lengths that end on a 32-row store box or a
256-row tile, materialised vs implicit splices, pooling at any depth, long utterances whose units sit far from zero,
empty utterances and an upper-bound row count.

The reference is `emulate`, a float64 evaluation that rounds exactly where the kernels round: the layer input and the
weights to bf16, every stored inter-layer activation to bf16, the last per-frame layer to fp32, the pooled vector to
bf16 when a layer follows it.  Everything else (contraction, bias, ReLU, BatchNorm, pooling) is float64.  What is left
between kernel and reference is fp32 accumulation and the occasional one-ulp bf16 flip of a stored activation, which
`gate` bounds per row.  The CPU tests show that the emulation is the oracle's network and that the gate catches the
defects it is meant to catch; the GPU tests hold the kernels to it.
"""

import numpy as np
import pytest

from oracle import ktf_oracle as O

# ------------------------------------------------------------------------------------------------------------------
# Reference
# ------------------------------------------------------------------------------------------------------------------

EPS = 1e-10          # StatsPooling epsilon of the networks below

LENGTHS_EDGES = [1, 2, 3, 4, 5, 8, 9, 23, 24, 25, 119, 120, 121, 247, 248, 249, 503, 504, 505, 5000]


def bf16(a):
    """Round to bf16 (nearest even) the way the kernels do: from the fp32 value."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    return t.to(torch.bfloat16).to(torch.float32).numpy().astype(np.float64)


def offsets_of(lengths):
    return np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)


def make_params(spec, in_dim, seed, stats_after=-1, include_std=True):
    """spec: list of {"U", "ctx", "relu", "bn"} -> per layer W (U, K*D) Kaldi layout, bias, BN (gamma, mean, var)."""
    rng = np.random.default_rng(seed)
    params, D = [], in_dim
    for i, s in enumerate(spec):
        K, U = len(s["ctx"]), s["U"]
        lim = np.sqrt(6.0 / (K * D + U))
        p = {"W": rng.uniform(-lim, lim, (U, K * D)).astype(np.float32),
             "b": rng.uniform(-0.1, 0.1, U).astype(np.float32), "ctx": list(s["ctx"]), "relu": s["relu"]}
        if s["bn"]:
            p["bn"] = (np.float32(1.0), (0.4 * rng.random(U) if s["relu"] else 0.1 * rng.standard_normal(U))
                       .astype(np.float32), (rng.random(U) + 0.5).astype(np.float32))
        params.append(p)
        D = 2 * U if (i == stats_after and include_std) else U
    return params


def scale_offset(p):
    """The fp32 scale / offset the library folds BatchNorm into (layers/normalization.py BatchNorm.scale_offset)."""
    if "bn" not in p:
        return None, None
    from kaldi_tflite_b200.layers import BatchNorm
    bn = BatchNorm()
    bn.set_weights(list(p["bn"]))
    return bn.scale_offset()


def tap_rows(offs, ctx, mutant=None):
    """(rows, K) source row of every tap of every frame: the edge clamp, per utterance."""
    lengths = np.diff(offs)
    b = np.repeat(np.arange(len(lengths)), lengths)
    start, T = offs[:-1][b], lengths[b]
    t = np.arange(offs[-1]) - start
    c = np.asarray(ctx)[None, :]
    if mutant == "zero_pad":
        src = start[:, None] + t[:, None] + c
        inside = (t[:, None] + c >= 0) & (t[:, None] + c < T[:, None])
        return np.where(inside, src, -1)
    if mutant == "cross_utterance":              # the batch clamped as one sequence
        return np.clip(np.arange(offs[-1])[:, None] + c, 0, offs[-1] - 1)
    tt = np.clip(t[:, None] + c, 0, T[:, None] - 1)
    if mutant == "edge_tap":                     # the outermost tap is one frame off on the edge frames
        k = int(np.argmax(np.abs(ctx)))
        step = np.where(t == 0, 1, np.where(t == T - 1, -1, 0))
        tt[:, k] = np.clip(tt[:, k] + step, 0, T - 1)
    return start[:, None] + tt


def affine(x, p, offs, per_frame, out, rounding, mutant=None):
    """One fused layer: splice (edge clamp) -> contraction -> bias -> ReLU -> BatchNorm, float64.  `out`: how the
    kernel leaves the result -- "bf16" (a stored activation), "f32" (the last layer) or None (pooled, never stored)."""
    W = p["W"].astype(np.float64)
    if rounding:
        W, x = bf16(W), bf16(x)
    K = len(p["ctx"])
    D = W.shape[1] // K
    if per_frame:
        rows = tap_rows(offs, p["ctx"], mutant)
        xz = np.vstack([x, np.zeros((1, D))])    # row -1: the zero row of the zero-padding mutant
        y = sum(xz[rows[:, k]] @ W[:, k * D:(k + 1) * D].T for k in range(K))
    else:
        y = x @ W.T
    y = y + p["b"]
    if p["relu"]:
        y = np.maximum(y, 0.0)
    sc, of = scale_offset(p)
    if sc is not None:
        y = y * sc + of
    if rounding and out == "bf16":
        y = bf16(y)
    elif rounding and out == "f32":
        y = y.astype(np.float32).astype(np.float64)
    return y


def pool(y, offs, include_std, mutant=None):
    out = []
    for b in range(len(offs) - 1):
        seg = y[offs[b]:offs[b + 1]]
        if mutant == "drop_last" and len(seg) > 1:
            seg = seg[:-1]
        m = seg.mean(axis=0)
        row = [m]
        if include_std:
            row.append(np.sqrt(np.maximum((seg * seg).mean(axis=0) - m * m, 0.0) + EPS))
        out.append(np.concatenate(row))
    return np.stack(out)


def emulate(x, offs, params, stats_after=-1, include_std=True, rounding=True, mutant=None):
    """Ragged (rows, D) input -> per-frame (rows, U) output, or pooled (B, dim) when stats_after >= 0."""
    y = np.asarray(x, dtype=np.float64)
    per_frame = True
    for i, p in enumerate(params):
        last = i == len(params) - 1
        if i == stats_after:
            y = pool(affine(y, p, offs, True, None, rounding, mutant), offs, include_std, mutant)
            if rounding:
                y = y.astype(np.float32).astype(np.float64) if last else bf16(y)
            per_frame = False
            continue
        y = affine(y, p, offs, per_frame, "f32" if last else "bf16", rounding, mutant)
    if mutant == "row_block" and per_frame:     # one row of every 32-row block replaced by its neighbour
        y = y.copy()
        y[31::32] = y[30::32][:len(y[31::32])]
    return y


# ------------------------------------------------------------------------------------------------------------------
# The gate: shared by the CPU and GPU tests
# ------------------------------------------------------------------------------------------------------------------

ROW_TOL = 3e-2       # max |error| of a per-frame row over the row's RMS
MEAN_TOL = 5e-3      # max |error| of a pooled mean over the utterance's activation RMS sqrt(mean^2 + std^2)
STD_TOL = 5e-3       # the same for the pooled std


def gate(got, want, pooled_units=None):
    """Worst error as a fraction of its bound (<= 1 passes).  Per-frame rows / post-pooling rows: per-row max |error|
    over the row's RMS.  Pooled rows (pooled_units = U, the layout mean || std): the mean and the std each against
    the utterance's RMS.  Returns {name: fraction}."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    if pooled_units is None:
        rms = np.sqrt(np.mean(want * want, axis=1))
        floor = 1e-3 * np.sqrt(np.mean(want * want)) + 1e-30
        return {"row": float(np.max(np.max(np.abs(got - want), axis=1) / np.maximum(rms, floor)) / ROW_TOL)}
    U = pooled_units
    m_w = want[:, :U]
    s_w = want[:, U:] if want.shape[1] > U else np.zeros_like(m_w)
    scale = np.sqrt(np.mean(m_w * m_w + s_w * s_w, axis=1, keepdims=True)) + 1e-30
    out = {"mean": float(np.max(np.abs(got[:, :U] - m_w) / scale)) / MEAN_TOL}
    if want.shape[1] > U:
        out["std"] = float(np.max(np.abs(got[:, U:] - s_w) / scale)) / STD_TOL
    return out


def worst(g):
    return max(g.values())


# ------------------------------------------------------------------------------------------------------------------
# Networks
# ------------------------------------------------------------------------------------------------------------------

def L(U, ctx, relu=True, bn=True):
    return {"U": U, "ctx": list(ctx), "relu": relu, "bn": bn}


# per-frame stacks: (name, input dim, layers)
FRAME_STACKS = [
    # splice_rows_kernel first layer; implicit mid layers (incl. +-4); 512 / 1500 wide; 24 / 12 k-blocks
    ("rows30_implicit", 30, [L(512, [-2, -1, 0, 1, 2]), L(512, [-2, 0, 2]), L(512, [-4, 0, 4]),
                             L(1500, [0], relu=True, bn=True)]),
    # splice_kernel<float> first layer; materialised mid layer (D = 200, |ctx| > 4); asymmetric implicit taps; U = 13
    ("f23_materialised", 23, [L(200, [-2, -1, 0, 1, 2]), L(256, [-6, 0, 6]), L(128, [0, 3]),
                              L(13, [-4, -3, -2, -1, 0], relu=False, bn=False)]),
    # <= 4 k-blocks everywhere (8 epilogue warps), a 13-wide bf16 activation (unaligned rows) feeding a splice
    ("narrow_kblocks", 30, [L(13, [0, 1]), L(64, [-1, 0, 1]), L(200, [-1, 0, 1], relu=False)]),
]

# pooled stacks: (name, input dim, layers, stats_after, include_std)
POOLED_STACKS = [
    ("pool_first_2after", 30, [L(200, [-2, -1, 0, 1, 2]), L(128, [0]), L(64, [0], relu=False, bn=False)], 0, True),
    ("pool_mid_1after", 23, [L(128, [-1, 0, 1]), L(256, [-2, 0, 2]), L(100, [0], relu=False, bn=False)], 1, False),
    ("pool_last_sitw", 30, [L(512, [-2, -1, 0, 1, 2]), L(1500, [-4, 0, 4])], 1, True),
    ("pool_norelu_bn", 30, [L(64, [0]), L(200, [-1, 0, 1], relu=False, bn=True)], 1, True),
    ("pool_relu_nobn", 30, [L(256, [-1, 0, 1], relu=True, bn=False)], 0, True),
    ("pool_plain_1after", 30, [L(96, [-1, 0, 1], relu=False, bn=False), L(40, [0])], 0, False),
]


def ragged_input(lengths, D, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((int(np.sum(lengths)), D)).astype(np.float32)


def shuffled_edges(seed=5):
    lengths = list(LENGTHS_EDGES)
    np.random.default_rng(seed).shuffle(lengths)
    return lengths


def tiny_lengths(seed=6):
    return list(np.random.default_rng(seed).integers(1, 4, 300))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the reference is right and the gate has teeth
# ------------------------------------------------------------------------------------------------------------------

def oracle_layers(params, stats_after, include_std):
    out = []
    for i, p in enumerate(params):
        K = len(p["ctx"])
        U = p["W"].shape[0]
        out.append({"type": "affine", "kernel": O.kaldi_to_kernel(p["W"], U, K), "bias": p["b"], "context": p["ctx"]})
        if p["relu"]:
            out.append({"type": "relu"})
        if "bn" in p:
            g, m, v = p["bn"]
            out.append({"type": "batchnorm", "gamma": np.full(U, g, np.float32), "mean": m, "var": v,
                        "epsilon": 0.001})
        if i == stats_after:
            out.append({"type": "stats", "left_context": 0, "right_context": 0, "include_std": include_std,
                        "epsilon": EPS, "reduce_time_axis": True})
    return out


@pytest.mark.parametrize("name,D,spec,stats_after,include_std",
                         [(n, D, s, -1, True) for n, D, s in FRAME_STACKS] + list(POOLED_STACKS))
def test_emulation_without_rounding_is_the_oracle(name, D, spec, stats_after, include_std):
    params = make_params(spec, D, 1, stats_after, include_std)
    B, T = 3, 41
    x = ragged_input([T] * B, D, seed=2)
    got = emulate(x, offsets_of([T] * B), params, stats_after, include_std, rounding=False)
    want = O.sequential(x.reshape(B, T, D), oracle_layers(params, stats_after, include_std))
    want = want.reshape(got.shape).astype(np.float64)
    rms = np.sqrt(np.mean(want * want, axis=1, keepdims=True))
    assert np.max(np.abs(got - want) / rms) < 1e-5


@pytest.mark.parametrize("name,D,spec,stats_after,include_std",
                         [(n, D, s, -1, True) for n, D, s in FRAME_STACKS[1:]] + list(POOLED_STACKS[:2]))
def test_emulation_of_ragged_batch_equals_solo_runs(name, D, spec, stats_after, include_std):
    params = make_params(spec, D, 1, stats_after, include_std)
    lengths = [5, 1, 24, 2, 9, 3, 33]
    offs = offsets_of(lengths)
    x = ragged_input(lengths, D, seed=3)
    batch = emulate(x, offs, params, stats_after, include_std)
    for b, T in enumerate(lengths):
        solo = emulate(x[offs[b]:offs[b + 1]], offsets_of([T]), params, stats_after, include_std)
        part = batch[b:b + 1] if stats_after >= 0 else batch[offs[b]:offs[b + 1]]
        np.testing.assert_allclose(part, solo, rtol=1e-12, atol=1e-12)


MUTANT_LENGTHS = [1, 2, 3, 4, 5, 8, 9, 23, 24, 25, 40]


@pytest.mark.parametrize("mutant", ["zero_pad", "cross_utterance", "edge_tap", "row_block"])
def test_gate_rejects_per_frame_mutants(mutant):
    name, D, spec = FRAME_STACKS[1]
    params = make_params([dict(s, U=min(s["U"], 64)) for s in spec], D, seed=1)
    offs = offsets_of(MUTANT_LENGTHS)
    x = ragged_input(MUTANT_LENGTHS, D, seed=4)
    want = emulate(x, offs, params)
    assert worst(gate(want, want)) == 0.0
    miss = worst(gate(emulate(x, offs, params, mutant=mutant), want))
    assert miss >= 10.0, miss


@pytest.mark.parametrize("mutant", ["zero_pad", "cross_utterance", "edge_tap", "drop_last"])
def test_gate_rejects_pooled_mutants(mutant):
    name, D, spec, stats_after, include_std = POOLED_STACKS[2]
    params = make_params([dict(s, U=min(s["U"], 64)) for s in spec], D, 1, stats_after, include_std)
    offs = offsets_of(MUTANT_LENGTHS)
    x = ragged_input(MUTANT_LENGTHS, D, seed=4)
    want = emulate(x, offs, params, stats_after, include_std)
    U = params[stats_after]["W"].shape[0]
    miss = worst(gate(emulate(x, offs, params, stats_after, include_std, mutant=mutant), want, pooled_units=U))
    assert miss >= 10.0, miss


def test_bf16_rounding_matters_to_the_gate():
    """The emulation's rounding is not decoration: the unrounded network misses the gate."""
    name, D, spec = FRAME_STACKS[1]
    params = make_params([dict(s, U=min(s["U"], 64)) for s in spec], D, seed=1)
    offs = offsets_of(MUTANT_LENGTHS)
    x = ragged_input(MUTANT_LENGTHS, D, seed=4)
    assert worst(gate(emulate(x, offs, params, rounding=False), emulate(x, offs, params))) > 1.0


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------

def build_sequential(ktf, params, stats_after=-1, include_std=True):
    layers = []
    for i, p in enumerate(params):
        U, K = p["W"].shape[0], len(p["ctx"])
        t = ktf.layers.TDNN(U, context=p["ctx"], precision="bf16", name=f"l{i}.affine")
        t.build((None, None, p["W"].shape[1] // K))
        t.set_weights([p["W"], p["b"]])
        layers.append(t)
        if p["relu"]:
            layers.append(ktf.layers.ReLU(name=f"l{i}.relu"))
        if "bn" in p:
            bn = ktf.layers.BatchNorm(name=f"l{i}.batchnorm")
            bn.set_weights(list(p["bn"]))
            layers.append(bn)
        if i == stats_after:
            layers.append(ktf.layers.StatsPooling(0, 0, include_std=include_std, epsilon=EPS, reduce_time_axis=True))
    D = params[0]["W"].shape[1] // len(params[0]["ctx"])
    mdl = ktf.models.Sequential(layers, input_shape=(None, None, D), precision="bf16")
    mdl._ensure_plan(D)
    assert mdl._stack is not None, "the network must run as one tcgen05 stack"
    return mdl


def run_stack(mdl, x, lengths):
    import torch
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    od = torch.from_numpy(offsets_of(lengths)).cuda()
    y, _ = mdl.forward_ragged(xd, od)
    return y.cpu().numpy()


def report(tag, g):
    print(f"[tc-edges] {tag}: " + ", ".join(f"{k} {v:.3f} of the gate" for k, v in sorted(g.items())))


@pytest.fixture(scope="module")
def ktf():
    import kaldi_tflite_b200 as k
    return k


def test_edge_lengths_cover_store_boxes_and_tiles():
    """The padded starts (halo rows included) of the shuffled batch fall on many offsets mod 32 and mod 256, and
    padded lengths 32 and 256 end exactly on a store box / pair tile."""
    lengths = shuffled_edges()
    starts = offsets_of(lengths)[:-1] + 8 * np.arange(len(lengths))
    assert len(set(starts % 32)) >= 10 and len(set(starts % 256)) >= 15
    assert {24, 248} <= set(lengths)           # 24 + 8 = 32 rows, 248 + 8 = 256 rows


@pytest.mark.gpu
@pytest.mark.parametrize("name,D,spec", FRAME_STACKS, ids=[s[0] for s in FRAME_STACKS])
def test_per_frame_stack_vs_emulation(ktf, name, D, spec):
    params = make_params(spec, D, seed=11)
    mdl = build_sequential(ktf, params)
    for tag, lengths in (("edges", shuffled_edges()), ("tiny", tiny_lengths())):
        x = ragged_input(lengths, D, seed=12)
        got = run_stack(mdl, x, lengths)
        g = gate(got, emulate(x, offsets_of(lengths), params))
        report(f"{name} {tag}", g)
        assert worst(g) <= 1.0, g
        # an utterance's rows do not depend on its batch-mates: a row's MMA and epilogue arithmetic are the same in
        # every tile, so the rows are the same bits
        offs = offsets_of(lengths)
        for b in list(range(len(lengths)))[:: 1 if tag == "edges" else 37]:
            solo = run_stack(mdl, x[offs[b]:offs[b + 1]], [lengths[b]])
            np.testing.assert_array_equal(got[offs[b]:offs[b + 1]], solo, err_msg=f"{tag} utterance {b}")


SINGLE_LAYERS = [("rows30", 30, L(512, [-2, -1, 0, 1, 2])), ("f23", 23, L(200, [-3, 0, 3], relu=False)),
                 ("f23_1500", 23, L(1500, [-1, 0, 1]))]


def single_affine(ktf, p):
    from kaldi_tflite_b200.layers.tdnn import _Affine
    sc, of = scale_offset(p)
    return _Affine(p["W"], p["b"], p["ctx"], relu=p["relu"], bn_scale=sc, bn_offset=of, precision="bf16")


def run_affine(aff, x, lengths):
    import torch
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    od = torch.from_numpy(offsets_of(lengths)).cuda()
    y, _, _ = aff.forward_ragged(xd, od)
    return y.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("name,D,spec", SINGLE_LAYERS, ids=[s[0] for s in SINGLE_LAYERS])
def test_single_layer_vs_emulation(ktf, name, D, spec):
    params = make_params([spec], D, seed=13)
    aff = single_affine(ktf, params[0])
    for tag, lengths in (("edges", shuffled_edges()), ("tiny", tiny_lengths())):
        x = ragged_input(lengths, D, seed=14)
        got = run_affine(aff, x, lengths)
        g = gate(got, emulate(x, offsets_of(lengths), params))
        report(f"single {name} {tag}", g)
        assert worst(g) <= 1.0, g


@pytest.mark.gpu
@pytest.mark.parametrize("name,D,spec,stats_after,include_std", POOLED_STACKS, ids=[s[0] for s in POOLED_STACKS])
def test_pooled_stack_vs_emulation(ktf, name, D, spec, stats_after, include_std):
    params = make_params(spec, D, 15, stats_after, include_std)
    mdl = build_sequential(ktf, params, stats_after, include_std)
    pooled_last = stats_after == len(params) - 1
    U = params[stats_after]["W"].shape[0]
    for tag, lengths in (("edges", shuffled_edges()), ("short", [1, 2, 3]), ("tiny", tiny_lengths())):
        x = ragged_input(lengths, D, seed=16)
        got = run_stack(mdl, x, lengths)
        want = emulate(x, offsets_of(lengths), params, stats_after, include_std)
        g = gate(got, want, pooled_units=U if pooled_last else None)
        report(f"{name} {tag}", g)
        assert worst(g) <= 1.0, g
        if pooled_last and include_std:
            one = np.asarray(lengths) == 1          # a single frame has no spread: std = sqrt(eps)
            np.testing.assert_allclose(got[one, U:], np.sqrt(np.float32(EPS)), rtol=1e-6)


# ---- E: long utterances, units far from zero ----------------------------------------------------------------------

@pytest.mark.gpu
def test_pooled_std_of_units_far_from_zero(ktf):
    """Units whose post-ReLU mean is 10, 50 or 200 times their std, pooled over 300 .. 20 000 frames: the std must
    keep 1e-3 relative accuracy, below half a bf16 step (the precision the pooled vector is handed on with)."""
    lengths = [300, 3000, 20000]
    offs = offsets_of(lengths)
    D = 30
    params = make_params([L(64, [-1, 0, 1]), L(48, [0])], D, seed=17)
    x = ragged_input(lengths, D, seed=18)
    # the STATS layer's pre-activation on this data (its bf16 input is the first layer's stored output)
    h = affine(x.astype(np.float64), params[0], offs, True, "bf16", True)
    z = bf16(h) @ bf16(params[1]["W"]).T
    ratio = np.repeat([10.0, 50.0, 200.0], 16)
    sd = z.std(axis=0)
    p1 = dict(params[1], relu=True)
    p1["b"] = (ratio * sd - z.mean(axis=0)).astype(np.float32)
    r = np.maximum(z + p1["b"], 0.0)
    p1["bn"] = (np.float32(1.0), r.mean(axis=0).astype(np.float32), r.var(axis=0).astype(np.float32))
    params = [params[0], p1]
    mdl = build_sequential(ktf, params, stats_after=1, include_std=True)
    got = run_stack(mdl, x, lengths)
    want = emulate(x, offs, params, 1, True)
    U = 48
    sc, of = scale_offset(p1)
    post_bn = (np.maximum(z + p1["b"], 0.0) * sc + of).astype(np.float32)   # fp32 BN-first comparator
    for b, T in enumerate(lengths):
        for m in (10.0, 50.0, 200.0):
            u = ratio == m
            rel = np.abs(got[b, U:][u] - want[b, U:][u]) / want[b, U:][u]
            bn_first = O.stats_pooling(post_bn[None, offs[b]:offs[b + 1]], 0, 0, include_std=True, epsilon=EPS,
                                       reduce_time_axis=True)[0, 0, U:]
            rel_f32 = np.abs(bn_first[u] - want[b, U:][u]) / want[b, U:][u]
            print(f"[tc-edges] far-from-zero T={T:5d} mean/std={m:5.0f}: kernel std rel err {rel.max():.2e} "
                  f"({rel.max() / 1e-3:.3f} of the gate), fp32 BN-first pooling {rel_f32.max():.2e}")
            assert rel.max() <= 1e-3, (T, m, rel.max())


# ---- F: empty utterances -------------------------------------------------------------------------------------------

EMPTY_BASE = [5, 24, 1, 120, 9]


def with_empties(base, where):
    """Inserts empty utterances 'first', 'middle' (two), 'last', or fills every slot of a 6-utterance batch but one.
    Returns (lengths, positions of the non-empty utterances, their lengths)."""
    if where == "all_but_one":
        lengths = [0, 0, 0, base[1], 0, 0]
    else:
        slot = {"first": 0, "middle": len(base) // 2, "last": len(base)}[where]
        lengths = base[:slot] + [0] * (2 if where == "middle" else 1) + base[slot:]
    kept = [i for i, l in enumerate(lengths) if l > 0]
    return lengths, kept, [lengths[i] for i in kept]


EMPTY_CASES = ["first", "middle", "last", "all_but_one"]


@pytest.mark.gpu
@pytest.mark.parametrize("stack", [0, 1], ids=["rows30", "f23"])
def test_empty_utterances_per_frame(ktf, stack):
    name, D, spec = FRAME_STACKS[stack]
    params = make_params(spec, D, seed=19)
    mdl = build_sequential(ktf, params)
    aff = single_affine(ktf, params[0])
    for where in EMPTY_CASES:
        lengths, kept, base = with_empties(EMPTY_BASE, where)
        x = ragged_input(base, D, seed=20)
        for run in (lambda xx, ll: run_stack(mdl, xx, ll), lambda xx, ll: run_affine(aff, xx, ll)):
            got = run(x, lengths)                 # empties contribute no rows: x is the same array
            ref = run(x, base)
            assert got.shape == ref.shape
            np.testing.assert_array_equal(got, ref, err_msg=where)


@pytest.mark.gpu
@pytest.mark.parametrize("stack", [0, 2], ids=["pool_first_2after", "pool_last_sitw"])
def test_empty_utterances_pooled(ktf, stack):
    name, D, spec, stats_after, include_std = POOLED_STACKS[stack]
    params = make_params(spec, D, 21, stats_after, include_std)
    mdl = build_sequential(ktf, params, stats_after, include_std)
    for where in EMPTY_CASES:
        lengths, kept, base = with_empties(EMPTY_BASE, where)
        x = ragged_input(base, D, seed=22)
        got = run_stack(mdl, x, lengths)
        ref = run_stack(mdl, x, base)
        empty = [i for i, l in enumerate(lengths) if l == 0]
        if stats_after == len(params) - 1:
            # the pooled sums are fp32 atomics whose order follows the tile layout, which the empties shift: the same
            # values up to summation order
            scale = np.sqrt(np.mean(ref * ref, axis=1, keepdims=True))
            assert np.max(np.abs(got[kept] - ref) / scale) < 1e-4, where
            assert np.isnan(got[empty]).all(), where        # the mean over zero frames
        else:
            # here the pooled vector is rounded to bf16 before the next layer, so a last-bit difference of the sums can
            # move a pooled element by one bf16 step (2^-8 relative) and the next layers' rows by ~1e-3 of their RMS:
            # both batches are held to the gate against each other and against the reference of the batch without
            # the empties
            assert not np.isnan(got[kept]).any()
            g = gate(got[kept], ref)
            report(f"{name} empties {where} vs without", g)
            assert worst(g) <= 1.0, (where, g)
            g = gate(got[kept], emulate(x, offsets_of(base), params, stats_after, include_std))
            assert worst(g) <= 1.0, (where, g)


@pytest.mark.gpu
def test_extractor_batch_with_silent_utterance(ktf):
    import torch
    from conftest import golden_path, read_wav_int16
    from test_gpu_tdnn_plda import extractor_cfg
    ext = ktf.models.XvectorExtractor(extractor_cfg(), seed=0, allow_random_init=True)
    wav = read_wav_int16(golden_path("librispeech_2.wav"))
    speech = [wav[:48000], wav[60000:140000]]
    silent = np.zeros(16000, np.float32)
    for fused in (True, False):
        ext.fusePrepass = fused
        solo = [ext(torch.from_numpy(s.copy()).cuda()).cpu().numpy() for s in speech]
        out = ext([torch.from_numpy(a.copy()).cuda() for a in (speech[0], silent, speech[1])]).cpu().numpy()
        assert out.shape == (3, 128)
        assert np.isnan(out[1]).all(), fused
        for i, s in ((0, solo[0]), (2, solo[1])):
            assert np.isfinite(out[i]).all()
            assert np.max(np.abs(out[i] - s)) < 1e-3 * max(1.0, float(np.max(np.abs(s)))), (fused, i)
        with pytest.raises(ValueError):
            ext([speech[0], silent, speech[1]])


# ---- G: an upper bound of the row count -----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("pooled", [False, True], ids=["per_frame", "pooled"])
def test_total_rows_upper_bound(ktf, pooled):
    import torch
    from kaldi_tflite_b200 import _native as N
    from kaldi_tflite_b200 import _tensor as Tn
    if pooled:
        name, D, spec, stats_after, include_std = POOLED_STACKS[2]
    else:
        (name, D, spec), stats_after, include_std = FRAME_STACKS[1], -1, True
    params = make_params(spec, D, 23, stats_after, include_std)
    mdl = build_sequential(ktf, params, stats_after, include_std)
    stack = mdl._stack
    lengths = shuffled_edges()
    rows = int(np.sum(lengths))
    B, extra = len(lengths), 777
    x = torch.full((rows + extra, D), float("nan"), device="cuda")   # rows past offsets[B] must never be read
    x[:rows] = torch.from_numpy(ragged_input(lengths, D, seed=24)).cuda()
    od = torch.from_numpy(offsets_of(lengths)).cuda()
    outs = []
    for total in (rows, rows + extra):
        out = torch.full((B if pooled else rows + extra, stack.out_dim), 12345.0, device="cuda")
        N.check(N.lib().ktf_tdnn_stack_forward(stack.handle, Tn.ptr(x), Tn.ptr(od), B, total, Tn.ptr(out),
                                               Tn.stream_ptr()))
        outs.append(out.cpu().numpy())
    exact, bound = outs
    n = B if pooled else rows
    assert np.isfinite(bound[:n]).all()
    scale = np.sqrt(np.mean(exact[:n] ** 2, axis=1, keepdims=True))
    if pooled:                                   # fp32 atomics: equal up to summation order
        assert np.max(np.abs(bound[:n] - exact[:n]) / scale) < 1e-4
    else:
        np.testing.assert_array_equal(bound[:n], exact[:n])
        assert (bound[n:] == 12345.0).all()      # nothing written past the actual rows
