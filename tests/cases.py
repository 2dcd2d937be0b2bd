"""Shared test-case generators.

`kat_*` restate the deterministic (non-random) data generators of the reference's own unit test,
test/op/ConvInt8Test.cpp:175-207 (x[i] = i % 255 - 127, w = (i^2+j^2+k^2) % 255 - 127,
bias = (10000 + i*i*10 - i*i*i) % 12580, scale = ((127-i)*i % 128) / 20000), so the same vectors the
reference test feeds to its CPU backend are fed to the oracle and to the CUDA path.
"""
import os

import numpy as np


def kat_conv(n, ic, ih, iw, oc, kh, kw):
    xs = n * ic * ih * iw
    x = ((np.arange(xs) % 255) - 127).astype(np.int8).reshape(n, ic, ih, iw)
    i = np.arange(oc)[:, None, None]
    j = np.arange(ic)[None, :, None]
    k = np.arange(kh * kw)[None, None, :]
    w = (((i * i + j * j + k * k) % 255) - 127).astype(np.int8).reshape(oc, ic, kh, kw)
    bias = np.array([int(np.fmod(10000 + a * a * 10 - a * a * a, 12580)) for a in range(oc)], np.int32)
    ii = np.arange(oc)
    scale = (((127 - ii) * ii % 128) / 20000.0).astype(np.float32)
    return x, w, bias, scale


# (ic, oc), (kh, kw), n, pad(h,w), stride, dilate, (ih, iw)  -- a slice of ConvInt8Im2colGemmTest's sweep
# (test/op/ConvInt8Test.cpp:298-325) plus the {17,8} 7x7 extra case (:327-333)
KAT_SWEEP = [
    ((3, 64), (3, 3), 1, (1, 1), (1, 1), (1, 1), (27, 27)),
    ((8, 32), (3, 3), 2, (0, 0), (2, 2), (1, 1), (20, 20)),
    ((1, 32), (5, 5), 5, (3, 2), (1, 1), (2, 2), (11, 11)),
    ((54, 8), (5, 5), 1, (1, 1), (2, 2), (2, 2), (11, 14)),
    ((54, 8), (3, 3), 2, (3, 2), (1, 1), (1, 1), (12, 14)),
    ((17, 8), (3, 3), 1, (1, 1), (1, 1), (1, 1), (7, 7)),
    ((8, 32), (5, 5), 5, (0, 0), (1, 1), (1, 1), (20, 20)),
    ((3, 64), (5, 5), 2, (1, 1), (2, 2), (1, 1), (27, 27)),
]


def random_modern_case(rng, ic, oc, kh, kw, n, ih, iw, stride, pad, relu, dilate=(1, 1)):
    x = rng.integers(-128, 128, (n, ic, ih, iw)).astype(np.int8)
    w = rng.integers(-127, 128, (oc, ic, kh, kw)).astype(np.int8)
    s_in = float(np.float32(rng.uniform(0.01, 0.1)))
    s_out = float(np.float32(rng.uniform(0.01, 0.1)))
    # keep |acc * ws * s_in / s_out| around 40: a saturated output would hide epilogue errors
    ws = (rng.uniform(0.003, 0.012, oc) / np.sqrt(ic * kh * kw) * s_out / s_in).astype(np.float32)
    bias = (rng.uniform(-1, 1, oc) * 10 * s_out).astype(np.float32)
    z_in = int(rng.integers(-5, 6))
    z_out = int(rng.integers(-5, 6))
    return dict(x=x, w=w, ws=ws, bias=bias, s_in=s_in, s_out=s_out, z_in=z_in, z_out=z_out, stride=stride, pad=pad,
                dilate=dilate, relu=relu)


# ---- int8 Winograd (SURVEY a5) ------------------------------------------------------------------------------------
def kat_wino(n, ic, oc, ih, iw, k=3):
    """The reference test's own generator, test/op/ConvInt8Test.cpp:566-600 (x = i % 128 quantised with the test's
    xScale/xZeroPoint, w = i % 7 - 3, wScale = (oz % 11)*0.1 + 0.5, bias = (oz % 5)*0.5 - 1; attr scales 0.9 / 1 / 1.1,
    yScale 0.5, yZeroPoint 1, relu)."""
    xf = (np.arange(n * ic * ih * iw) % 128).astype(np.float32).reshape(n, ic, ih, iw)
    xs = np.float32((127.0 - 0.0) / (2.0 * 127))
    zx = int(round((0 - 0.0) / float(xs) - 127))
    f = xf * np.float32(1.0 / float(xs)) + np.float32(zx)
    f = np.clip(f, -127, 127)
    xq = np.trunc(f + np.where(f < 0, np.float32(-0.5), np.float32(0.5))).astype(np.int8)
    ws = (np.arange(oc) % 11 * 0.1 + 0.5).astype(np.float32)
    bias = (np.arange(oc) % 5 * 0.5 - 1).astype(np.float32)
    w = ((np.arange(oc * ic * k * k) % 7) - 3).astype(np.int8).reshape(oc, ic, k, k)
    return dict(x=xq, w=w, ws=ws, bias=bias, s_in=float(xs), z_in=zx, s_out=0.5, z_out=1, in_scales=0.9, in_zeros=1,
                w_scales=1.1, relu=True, pad=1)


def random_wino_case(rng, unit, n, ic, oc, ih, iw, pad=1, relu=False):
    """Random int8 Winograd conv with CALIBRATED per-position scales (max-abs of the float transform domain / 120), so
    neither the transformed activations, the transformed weights nor the outputs saturate."""
    from oracle import oracle as O
    alpha = unit + 2
    bt, _, g = O.wino_matrices(unit)
    bt, g = bt.astype(np.float64), g.astype(np.float64)
    x = rng.integers(-128, 128, (n, ic, ih, iw)).astype(np.int8)
    w = rng.integers(-127, 128, (oc, ic, 3, 3)).astype(np.int8)
    s_in = float(np.float32(rng.uniform(0.01, 0.1)))
    z_in = int(rng.integers(-5, 6))
    ws = (rng.uniform(0.003, 0.012, oc) / np.sqrt(ic * 9)).astype(np.float32)
    bias = rng.uniform(-1, 1, oc).astype(np.float32)
    # transformed weights: [a][oc][ic]
    wf = w.astype(np.float64) * ws[:, None, None, None]
    u = np.einsum("ai,ocij,bj->aboc", g, wf, g).reshape(alpha * alpha, oc, ic)
    w_scales = (np.abs(u).max(axis=2) / 120 + 1e-12).astype(np.float32)
    # transformed activations of the worst-case window (|x - z| <= 133): bound by sum |B^T| products
    mag = np.einsum("ai,bj->ab", np.abs(bt), np.abs(bt)).reshape(-1) * 60 * s_in
    in_scales = (mag / 120 * rng.uniform(0.8, 1.2, alpha * alpha)).astype(np.float32)
    in_zeros = rng.integers(-3, 4, alpha * alpha).astype(np.int32)
    # output range from the direct float conv of a sample
    xs = (x[:1].astype(np.float64) - z_in) * s_in
    xp = np.pad(xs, ((0, 0), (0, 0), (pad, pad), (pad, pad)))
    oh, ow = ih + 2 * pad - 2, iw + 2 * pad - 2
    acc = np.zeros((oc, oh, ow))
    for ky in range(3):
        for kx in range(3):
            acc += np.einsum("oc,chw->ohw", wf[:, :, ky, kx], xp[0, :, ky:ky + oh, kx:kx + ow])
    s_out = float(np.float32(max(np.abs(acc).max(), 1e-3) / 100))
    z_out = int(rng.integers(-5, 6))
    return dict(x=x, w=w, ws=ws, bias=(bias * 10 * s_out).astype(np.float32), s_in=s_in, z_in=z_in, s_out=s_out, z_out=z_out,
                in_scales=in_scales, in_zeros=in_zeros, w_scales=w_scales, relu=relu, pad=pad)


def wino_oracle(O, c, unit, fn=None):
    fn = fn or O.wino_conv_int8
    return fn(c["x"], c["w"], c["ws"], c["bias"], c["in_scales"], c["in_zeros"], c["w_scales"], unit, c["pad"], c["s_in"],
              c["z_in"], c["s_out"], c["z_out"], -127, 127, c["relu"])


def refdump_input(shape, seed):
    """The fp32 input `refdump run` feeds a model (oracle/refdump.cpp fillInput): std::mt19937(seed) through
    uniform_real_distribution<float>(-1, 1) in NCHW order.  RandomState(seed) draws the same 32-bit words."""
    words = np.random.RandomState(seed).randint(0, 2 ** 32, int(np.prod(shape)), dtype=np.uint64)
    u = words.astype(np.float32) / np.float32(2 ** 32)
    u = np.where(u >= 1, np.nextafter(np.float32(1), np.float32(0)), u).astype(np.float32)
    return (u * np.float32(2) + np.float32(-1)).reshape(shape)


# ---- inputs of golden files that are regenerated from their seeds instead of stored (stored, they would take the files past
# 1 MB); tests/golden/make_golden.py draws them through the same functions ---------------------------------------------------
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DW_CASES = [(32, 3, 2, 16, 16, (1, 1), (1, 1), 1), (96, 3, 1, 15, 15, (2, 2), (1, 1), 1), (40, 5, 1, 9, 11, (1, 1), (2, 2), 0),
            (7, 3, 3, 6, 6, (1, 1), (0, 0), 1)]
# the last five: ONE token = the decode step, where the reference switches to its single-quant arithmetic (asymmetric input
# quantisation over the row incl. the pack padding, zero point folded into the bias; ConvInt8TiledExecutor.cpp:1033, 1432, 2016-2050)
LINEAR_CASES = [(8, 64, 48, False, True, -1, 1), (33, 256, 200, True, True, -1, 1), (5, 96, 33, False, False, -1, 1),
                (64, 512, 128, True, False, -1, 1), (1, 2048, 512, True, True, -1, 1), (1, 100, 64, False, False, 0.2, 1.0),
                (1, 250, 33, True, False, -1, -0.1), (1, 320, 200, True, True, -3, 5), (1, 64, 48, False, True, 0.25, 0.25)]


def dw_linear_inputs():
    rng = np.random.default_rng(77)
    out = {}
    for i, (ch, k, n, ih, iw, st, pad, relu) in enumerate(DW_CASES):
        x = rng.integers(-128, 128, (n, ch, ih, iw)).astype(np.int8)
        w = rng.integers(-127, 128, (ch, 1, k, k)).astype(np.int8)
        s_in, s_out = 0.043, 0.061
        z_in, z_out = int(rng.integers(-4, 5)), int(rng.integers(-4, 5))
        ws = (rng.uniform(0.003, 0.012, ch) / k * s_out / s_in).astype(np.float32)
        bias = (rng.uniform(-1, 1, ch) * 10 * s_out).astype(np.float32)
        out.update({f"d{i}_x": x, f"d{i}_w": w, f"d{i}_ws": ws, f"d{i}_bias": bias, f"d{i}_stride": np.array(st),
                    f"d{i}_pad": np.array(pad), f"d{i}_relu": np.array(relu), f"d{i}_q": np.array([s_in, z_in, s_out, z_out])})
    for j, (tokens, ic, oc, asym, hb, lo, hi) in enumerate(LINEAR_CASES):
        x = rng.uniform(lo, hi, (tokens, ic)).astype(np.float32)
        wq = rng.integers(-128, 128, (oc, ic)).astype(np.int8)
        alpha = rng.uniform(0.001, 0.01, oc).astype(np.float32)
        wmin = rng.uniform(-0.05, 0.05, oc).astype(np.float32) if asym else np.zeros(0, np.float32)
        bias = rng.uniform(-1, 1, oc).astype(np.float32) if hb else np.zeros(0, np.float32)
        out.update({f"l{j}_x": x, f"l{j}_wq": wq, f"l{j}_alpha": alpha, f"l{j}_wmin": wmin, f"l{j}_bias": bias})
    return out


def matmul_inputs():
    from tests.test_matmul import CASES, make
    rng = np.random.default_rng(808)
    out = {}
    for i, (bd, e, l, h, ta, tb) in enumerate(CASES):
        a, b = make(rng, bd, e, l, h, ta, tb)
        out.update({f"m{i}_a": a, f"m{i}_b": b, f"m{i}_ta": np.array(ta), f"m{i}_tb": np.array(tb)})
    return out


def load_golden(name):
    """tests/golden/<name>.npz (the reference's outputs) together with the inputs regenerated for it"""
    g = np.load(os.path.join(GOLD, name + ".npz"))
    inputs = {"dw_linear_golden": dw_linear_inputs, "matmul_golden": matmul_inputs,
              "mbv2_int8_checkpoints": lambda: {"input": refdump_input((1, 3, 224, 224), 7)}}[name]()
    return dict(inputs, **{k: g[k] for k in g.files})
