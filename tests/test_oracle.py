"""CPU tests (-m "not gpu"): the oracle against the reference's known-answer generators, the committed golden
fixtures and the UNMODIFIED reference CPU backend itself, bit for bit: live where oracle/_ref is built, elsewhere its answers to the same
requests as recorded in tests/golden/reference_calls.npz (the *_live_reference tests)."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.cases import KAT_SWEEP, kat_conv, load_golden, random_modern_case

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def naive_conv_int8(x, w, bias, scale, stride, pad, dilate):
    """naiveConvInt8 + int32ToInt8 of the reference test (test/op/ConvInt8Test.cpp:35-42, 141-171):
    roundf((acc + bias) * scale) clamped to +-127.  The reference accepts |diff| <= 1 against it (:255-260)."""
    n, ic, ih, iw = x.shape
    oc, _, kh, kw = w.shape
    oh = O.conv_out_size(ih, kh, stride[0], pad[0], dilate[0])
    ow = O.conv_out_size(iw, kw, stride[1], pad[1], dilate[1])
    xp = np.zeros((n, ic, ih + 2 * pad[0], iw + 2 * pad[1]), np.int64)
    xp[:, :, pad[0]:pad[0] + ih, pad[1]:pad[1] + iw] = x
    acc = np.zeros((n, oc, oh, ow), np.int64)
    for ky in range(kh):
        for kx in range(kw):
            patch = xp[:, :, ky * dilate[0]: ky * dilate[0] + (oh - 1) * stride[0] + 1: stride[0],
                       kx * dilate[1]: kx * dilate[1] + (ow - 1) * stride[1] + 1: stride[1]]
            acc += np.einsum("nchw,oc->nohw", patch, w[:, :, ky, kx].astype(np.int64))
    v = (acc + bias[None, :, None, None]).astype(np.float32) * scale[None, :, None, None].astype(np.float32)
    v = np.sign(v) * np.floor(np.abs(v) + np.float32(0.5))   # roundf
    return np.clip(v, -127, 127).astype(np.int8)


@pytest.mark.parametrize("case", KAT_SWEEP)
def test_oracle_vs_reference_naive_kat(case):
    (ic, oc), (kh, kw), n, pad, stride, dilate, (ih, iw) = case
    x, w, bias, scale = kat_conv(n, ic, ih, iw, oc, kh, kw)
    bf, sx = O.fold_legacy(w, scale, bias)
    y = O.conv_int8(x, w, scale, sx, bf, stride=stride, pad=pad, dilate=dilate)
    ref = naive_conv_int8(x, w, bias, scale, stride, pad, dilate)
    assert y.shape == ref.shape
    assert np.abs(y.astype(int) - ref.astype(int)).max() <= 1  # the reference test's own tolerance


def test_oracle_vs_golden_fixtures():
    """tests/golden/conv_int8_golden.npz: inputs + outputs produced by the real reference (make_golden.py)."""
    path = os.path.join(GOLD, "conv_int8_golden.npz")
    g = np.load(path, allow_pickle=False)
    ncase = int(g["ncase"])
    assert ncase >= 8
    for i in range(ncase):
        p = {k[len(f"c{i}_"):]: g[k] for k in g.files if k.startswith(f"c{i}_")}
        stride, pad, dilate = tuple(p["stride"]), tuple(p["pad"]), tuple(p["dilate"])
        if int(p["mode"]) == 0:
            bf, sx = O.fold_legacy(p["w"], p["scale"], p["bias"])
            y = O.conv_int8(p["x"], p["w"], p["scale"], sx, bf, stride=stride, pad=pad, dilate=dilate)
        else:
            bf, sx = O.fold_modern(p["w"], p["scale"], p["bias"], float(p["s_in"]), int(p["z_in"]), float(p["s_out"]),
                                   int(p["z_out"]))
            y = O.conv_int8(p["x"], p["w"], p["scale"], sx, bf, stride=stride, pad=pad, dilate=dilate,
                            z_in=int(p["z_in"]), min_v=int(p["z_out"]) if int(p["relu"]) else -127, max_v=127)
        assert np.array_equal(y, p["y"]), f"golden case {i} differs"


@pytest.mark.parametrize("case", KAT_SWEEP[:5])
def test_oracle_bit_exact_vs_reference_legacy(case):
    (ic, oc), (kh, kw), n, pad, stride, dilate, (ih, iw) = case
    x, w, bias, scale = kat_conv(n, ic, ih, iw, oc, kh, kw)
    yr = O.ref_conv(0, x, w, bias, scale, stride=stride, pad=pad, dilate=dilate)
    bf, sx = O.fold_legacy(w, scale, bias)
    yo = O.conv_int8(x, w, scale, sx, bf, stride=stride, pad=pad, dilate=dilate)
    assert np.array_equal(yr, yo)


def test_oracle_bit_exact_vs_reference_modern():
    rng = np.random.default_rng(11)
    for (ic, oc, kh, kw, n, st, pad, relu) in [(3, 32, 3, 3, 2, (2, 2), (1, 1), 1), (16, 24, 1, 1, 3, (1, 1), (0, 0), 0),
                                                (17, 40, 5, 3, 1, (1, 1), (1, 1), 1), (54, 8, 3, 3, 2, (2, 2), (0, 0), 0)]:
        c = random_modern_case(rng, ic, oc, kh, kw, n, 9, 12, st, pad, relu)
        yr = O.ref_conv(1, c["x"], c["w"], c["bias"], c["ws"], stride=st, pad=pad, relu=relu, z_in=c["z_in"],
                        z_out=c["z_out"], scale_in=c["s_in"], scale_out=c["s_out"])
        bf, sx = O.fold_modern(c["w"], c["ws"], c["bias"], c["s_in"], c["z_in"], c["s_out"], c["z_out"])
        yo = O.conv_int8(c["x"], c["w"], c["ws"], sx, bf, stride=st, pad=pad, z_in=c["z_in"],
                         min_v=c["z_out"] if relu else -127, max_v=127)
        assert np.array_equal(yr, yo)


def test_casts_round_half_away_and_clamp():
    x = np.array([0.5, -0.5, 1.5, -1.5, 2.4999, 126.5, 127.5, -127.5, -300.0, 300.0, 0.0], np.float32)
    y = O.float_to_int8(x, 1.0, 0.0, -127, 127)
    assert y.tolist() == [1, -1, 2, -2, 2, 127, 127, -127, -127, 127, 0]
    back = O.int8_to_float(y, 0.25, 3.0)
    assert np.array_equal(back, (y.astype(np.float32) - 3.0) * np.float32(0.25))
    # scale == 0 must map to inv_scale 0 (CPUCast.cpp:24), not inf
    assert O.float_to_int8(np.array([5.0], np.float32), 0.0, 2.0).tolist() == [2]


def wire_wzero(wmin, alpha):
    """IDST asymmetric alpha = {min, scale}; the loader turns min into the offset of SIGNED int8 weights:
    alpha[2o] - clampMin*alpha[2o+1] with clampMin = -128 (source/core/ConvolutionCommon.cpp:757-766)."""
    return (wmin - np.float32(-128) * alpha).astype(np.float32)


def test_depthwise_and_linear_vs_golden_fixtures():
    g = load_golden("dw_linear_golden")
    for i in range(int(g["ndw"])):
        s_in, z_in, s_out, z_out = g[f"d{i}_q"]
        relu = int(g[f"d{i}_relu"])
        sc, bi = O.fold_depthwise(g[f"d{i}_w"], g[f"d{i}_ws"], g[f"d{i}_bias"], float(s_in), int(z_in), float(s_out), int(z_out))
        y = O.depthwise_int8(g[f"d{i}_x"], g[f"d{i}_w"], sc, bi, stride=tuple(int(v) for v in g[f"d{i}_stride"]),
                             pad=tuple(int(v) for v in g[f"d{i}_pad"]), z_in=int(z_in),
                             min_v=int(z_out) if relu else -127, max_v=127)
        assert np.array_equal(y, g[f"d{i}_y"]), f"depthwise golden {i}"
    for j in range(int(g["nlin"])):
        alpha, wmin, bias = g[f"l{j}_alpha"], g[f"l{j}_wmin"], g[f"l{j}_bias"]
        y = O.linear_w8_dynamic(g[f"l{j}_x"], g[f"l{j}_wq"], alpha, wire_wzero(wmin, alpha) if wmin.size else None,
                                bias if bias.size else None)
        ref = g[f"l{j}_y"]
        # fp32 output row (BASELINE north_star: 1e-3 rel); the restatement is within 1e-6 of the real reference
        # (bit-exact for symmetric weights on full 4-token groups; the x86 remainder kernel orders one add differently)
        assert np.abs(y - ref).max() / np.abs(ref).max() < 2e-6, f"linear golden {j}"


def test_block_quant_linear_vs_golden_fixtures():
    """K-blocked weight scales (MNN-LLM's default export) recorded from the real reference: the restatement is within 4e-6 relative
    for prefill (symmetric per-token input quant, blocks summed in fp32) and decode (single-quant arithmetic) alike."""
    g = np.load(os.path.join(GOLD, "block_linear_golden.npz"))
    assert int(g["n"]) >= 6
    for j in range(int(g["n"])):
        alpha, wmin, bias = g[f"b{j}_alpha"], g[f"b{j}_wmin"], g[f"b{j}_bias"]
        blocks = alpha.shape[1]
        wz = (wmin - np.float32(-128) * alpha).astype(np.float32) if wmin.size else None
        y = O.linear_w8_dynamic_blocks(g[f"b{j}_x"], g[f"b{j}_wq"], alpha, wz, bias if bias.size else None, blocks)
        ref = g[f"b{j}_y"]
        assert np.abs(y - ref).max() / np.abs(ref).max() < 4e-6, f"block linear golden {j}"
    # one block is the per-channel function, bit for bit (both token regimes)
    x, wq, alpha = g["b0_x"], g["b0_wq"], g["b0_alpha"][:, 0]
    assert np.array_equal(O.linear_w8_dynamic(x, wq, alpha), O.linear_w8_dynamic_blocks(x, wq, alpha, None, None, 1))
    assert np.array_equal(O.linear_w8_dynamic(x[:1], wq, alpha), O.linear_w8_dynamic_blocks(x[:1], wq, alpha, None, None, 1))


def test_block_quant_linear_vs_live_reference():
    rng = np.random.default_rng(12)
    for (tokens, ic, oc, blocks, asym, hb) in [(2, 128, 48, 2, True, True), (17, 640, 64, 5, False, False), (1, 320, 72, 5, True, True)]:
        x = rng.uniform(-1, 1, (tokens, ic)).astype(np.float32)
        wq = rng.integers(-128, 128, (oc, ic)).astype(np.int8)
        alpha = rng.uniform(0.001, 0.01, (oc, blocks)).astype(np.float32)
        wmin = rng.uniform(-0.05, 0.05, (oc, blocks)).astype(np.float32) if asym else None
        bias = rng.uniform(-1, 1, oc).astype(np.float32) if hb else None
        al = np.stack([wmin, alpha], 2).ravel() if asym else alpha.ravel()
        ref = O.ref_linear(x, wq, al, asym=asym, bias=bias, blocks=blocks)
        wz = (wmin - np.float32(-128) * alpha).astype(np.float32) if asym else None
        y = O.linear_w8_dynamic_blocks(x, wq, alpha, wz, bias, blocks)
        assert np.abs(y - ref).max() / np.abs(ref).max() < 4e-6


def test_single_token_linear_is_the_references_decode_arithmetic():
    """ONE token takes a different path in the reference (asymmetric single-quant with the input zero folded into the bias) than
    two or more (symmetric per-token quant): the restatement follows both, and the two differ by far more than the tolerance."""
    rng = np.random.default_rng(4)
    for (ic, oc, asym, hb, lo, hi) in [(256, 96, False, False, -1, 1), (100, 64, True, True, 0.2, 1.0), (250, 33, False, True, -2, -0.1)]:
        x = rng.uniform(lo, hi, (1, ic)).astype(np.float32)
        wq = rng.integers(-128, 128, (oc, ic)).astype(np.int8)
        alpha = rng.uniform(0.001, 0.01, oc).astype(np.float32)
        wmin = rng.uniform(-0.05, 0.05, oc).astype(np.float32) if asym else None
        bias = rng.uniform(-1, 1, oc).astype(np.float32) if hb else None
        al = np.stack([wmin, alpha], 1).ravel() if asym else alpha
        ref = O.ref_linear(x, wq, al, asym=asym, bias=bias).reshape(1, oc)
        wz = wire_wzero(wmin, alpha) if asym else None
        one = O.linear_w8_dynamic(x, wq, alpha, wz, bias)
        assert np.abs(one - ref).max() / np.abs(ref).max() < 2e-6
        # the multi-token arithmetic on the same row (the row twice -> symmetric per-token quant) is NOT what the reference does for 1
        two = O.linear_w8_dynamic(np.concatenate([x, x]), wq, alpha, wz, bias)[:1]
        assert np.abs(two - ref).max() / np.abs(ref).max() > 1e-4


def test_oracle_random_sweep_vs_live_reference():
    """A seeded random sweep of the restatement against the UNMODIFIED reference CPU backend (conv modern form through a
    real 2-op .mnn, conv legacy form, depthwise): kernel sizes, strides, pads, dilations, ragged channels, zero points."""
    rng = np.random.default_rng(20260922)
    n_ok = 0
    for t in range(24):
        kh, kw = int(rng.choice([1, 2, 3, 5])), int(rng.choice([1, 3, 4]))
        ic, oc = int(rng.integers(1, 70)), int(rng.integers(1, 50))
        st = (int(rng.integers(1, 3)), int(rng.integers(1, 3)))
        dl = (int(rng.integers(1, 3)), 1)
        pad = (int(rng.integers(0, 3)), int(rng.integers(0, 2)))
        ih, iw = int(rng.integers(5, 14)), int(rng.integers(5, 14))
        if (ih + 2 * pad[0] - (dl[0] * (kh - 1) + 1)) < 0 or (iw + 2 * pad[1] - (dl[1] * (kw - 1) + 1)) < 0:
            continue
        n, relu = int(rng.integers(1, 3)), int(rng.integers(0, 2))
        c = random_modern_case(rng, ic, oc, kh, kw, n, ih, iw, st, pad, relu, dl)
        yr = O.ref_conv(1, c["x"], c["w"], c["bias"], c["ws"], stride=st, pad=pad, dilate=dl, relu=relu, z_in=c["z_in"],
                        z_out=c["z_out"], scale_in=c["s_in"], scale_out=c["s_out"])
        bf, sx = O.fold_modern(c["w"], c["ws"], c["bias"], c["s_in"], c["z_in"], c["s_out"], c["z_out"])
        yo = O.conv_int8(c["x"], c["w"], c["ws"], sx, bf, stride=st, pad=pad, dilate=dl, z_in=c["z_in"],
                         min_v=c["z_out"] if relu else -127, max_v=127)
        assert np.array_equal(yr, yo), f"modern conv case {t}: ic={ic} oc={oc} k={kh}x{kw} s={st} p={pad} d={dl}"
        n_ok += 1
    for t in range(8):
        ch, k = int(rng.integers(1, 40)), int(rng.choice([3, 5]))
        ih, iw = int(rng.integers(k, 12)), int(rng.integers(k, 12))
        st, pad, relu = (int(rng.integers(1, 3)),) * 2, (int(rng.integers(0, 2)),) * 2, int(rng.integers(0, 2))
        x = rng.integers(-128, 128, (1, ch, ih, iw)).astype(np.int8)
        w = rng.integers(-127, 128, (ch, 1, k, k)).astype(np.int8)
        s_in, s_out = 0.043, 0.061
        z_in, z_out = int(rng.integers(-4, 5)), int(rng.integers(-4, 5))
        ws = (rng.uniform(0.003, 0.012, ch) / k * s_out / s_in).astype(np.float32)
        bias = (rng.uniform(-1, 1, ch) * 10 * s_out).astype(np.float32)
        yr = O.ref_conv(1, x, w, bias, ws, stride=st, pad=pad, group=ch, relu=relu, z_in=z_in, z_out=z_out, scale_in=s_in,
                        scale_out=s_out)
        sc, bi = O.fold_depthwise(w, ws, bias, s_in, z_in, s_out, z_out)
        yo = O.depthwise_int8(x, w, sc, bi, stride=st, pad=pad, z_in=z_in, min_v=z_out if relu else -127, max_v=127)
        assert np.array_equal(yr, yo), f"depthwise case {t}: ch={ch} k={k} s={st} p={pad}"
        n_ok += 1
    assert n_ok >= 24


POOL_CASES = [(1, 16, 8, 8, (3, 3), (2, 2), (1, 1), 1), (2, 20, 9, 7, (2, 2), (2, 2), (0, 0), 0), (1, 33, 7, 7, (7, 7), (1, 1), (0, 0), 1),
              (1, 8, 10, 10, (3, 3), (1, 1), (1, 1), 0), (1, 5, 6, 9, (3, 2), (1, 2), (1, 0), 1), (3, 64, 12, 12, (3, 3), (2, 2), (1, 1), 0)]


def test_int8_pool_oracle_vs_live_reference():
    """int8 pooling with equal in/out quant attrs (kept in int8 by the CPU's onSetQuantInfo): the restatement of the x86
    kernels -- average on the uint8 storage with a 2^24 fixed-point reciprocal, MAX comparing the stored bytes as signed --
    against the reference itself.  The max-pool quirk is real: a true maximum would differ on these inputs."""
    rng = np.random.default_rng(5)
    differs_from_true_max = False
    for (n, c, ih, iw, k, s, p, avg) in POOL_CASES:
        x = rng.integers(-128, 128, (n, c, ih, iw)).astype(np.int8)
        for z in (0, -7):
            yo = O.pool_int8_x86(x, k, s, p, avg)
            yr = O.ref_pool_int8(x, k, s, p, avg, 0.05, z)
            assert np.array_equal(yo, yr), (n, c, ih, iw, k, s, p, avg, z)
        if not avg and p == (0, 0):
            oh, ow = yo.shape[2], yo.shape[3]
            true = np.stack([x[:, :, i:i + (oh - 1) * s[0] + 1:s[0], j:j + (ow - 1) * s[1] + 1:s[1]]
                             for i in range(k[0]) for j in range(k[1])]).max(0)
            differs_from_true_max |= not np.array_equal(true, yo)
    assert differs_from_true_max


def test_scale_int8_oracle_pinned_on_live_reference():
    """The numpy restatement of CPUScaleInt8 + MNNScaleAndAddBiasInt8 against the REAL reference: the first int8 Scale ops of
    ResNet-50 int8 (oracle/_ref/r50_int8.mnn) as executed by MNN_FORWARD_CPU, recorded from the per-command dump of `refdump run`
    (tests/golden/scale_int8_golden.npz: each op's parameters and quant attrs, an 8x8 spatial crop of its int8 input and output)."""
    g = np.load(os.path.join(GOLD, "scale_int8_golden.npz"))
    assert int(g["n"]) >= 3
    for k in range(int(g["n"])):
        s_in, z_in, s_out, z_out, min_v, max_v = g[f"s{k}_q"]
        bias = g[f"s{k}_bias"]
        y = O.scale_int8(g[f"s{k}_x"], g[f"s{k}_scale"], bias if bias.size else None, s_in, int(z_in), s_out, int(z_out),
                         int(min_v), int(max_v))
        qo = g[f"s{k}_y"]
        assert np.array_equal(y, qo), (str(g[f"s{k}_name"]), np.abs(y.astype(int) - qo.astype(int)).max())
