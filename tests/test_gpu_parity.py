"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI (via mnn_b200.backend), must equal
the oracle / the reference's golden vectors BIT FOR BIT for int8 tensors; fp32 outputs within 1e-3 relative."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.cases import KAT_SWEEP, kat_conv, load_golden, random_modern_case

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def run_conv(backend, x, w, ws, bias, stride, pad, dilate, relu, legacy, qi, qo, variant=0):
    from mnn_b200.backend import Op, QuantAttr, Tensor
    n, ic, ih, iw = x.shape
    oc, _, kh, kw = w.shape
    op = Op(type="ConvInt8", conv=dict(ic=ic, oc=oc, kernel=(kh, kw), stride=tuple(int(v) for v in stride),
                                      pad=tuple(int(v) for v in pad), dilate=tuple(int(v) for v in dilate),
                                      group=1, relu=bool(relu)),
            weight=w, wscale=ws, bias=bias, legacy=legacy)
    xin = backend.onAcquire(Tensor((n, ic, ih, iw), "int8", QuantAttr(*qi)))
    backend.onCopyBuffer(x, xin)
    yout = Tensor((n, oc, 1, 1), "int8", QuantAttr(*qo))
    ex = backend.onCreate([xin], [yout], op)
    assert ex is not None
    if variant:
        ex.set_variant(variant)
    assert ex.onResize([xin], [yout]) == 0
    backend.onAcquire(yout)
    yout.data.fill_(77)  # poison: every byte of the valid region must be overwritten
    assert ex.onExecute([xin], [yout]) == 0
    backend.onSync()
    raw = yout.data.cpu().numpy()
    assert (raw[..., oc:] == 0).all(), "NHWC16 channel padding must stay zero"
    return backend.onCopyBuffer(yout, "same")


def test_golden_fixtures_bit_exact(backend):
    """inputs/outputs recorded from the UNMODIFIED reference CPU backend (tests/golden/make_golden.py)."""
    g = np.load(os.path.join(GOLD, "conv_int8_golden.npz"))
    for i in range(int(g["ncase"])):
        p = {k[len(f"c{i}_"):]: g[k] for k in g.files if k.startswith(f"c{i}_")}
        if int(p["mode"]) == 0:
            y = run_conv(backend, p["x"], p["w"], p["scale"], p["bias"], p["stride"], p["pad"], p["dilate"], 0, True,
                         (0, 0, -127, 127), (0, 0, -127, 127))
        else:
            y = run_conv(backend, p["x"], p["w"], p["scale"], p["bias"], p["stride"], p["pad"], p["dilate"],
                         int(p["relu"]), False, (float(p["s_in"]), int(p["z_in"]), -128, 127),
                         (float(p["s_out"]), int(p["z_out"]), -127, 127))
        assert y.shape == p["y"].shape
        assert np.array_equal(y, p["y"]), f"golden case {i}: {np.abs(y.astype(int) - p['y'].astype(int)).max()}"


@pytest.mark.parametrize("case", KAT_SWEEP)
def test_kat_sweep_vs_oracle(backend, case):
    (ic, oc), (kh, kw), n, pad, stride, dilate, (ih, iw) = case
    x, w, bias, scale = kat_conv(n, ic, ih, iw, oc, kh, kw)
    bf, sx = O.fold_legacy(w, scale, bias)
    ref = O.conv_int8(x, w, scale, sx, bf, stride=stride, pad=pad, dilate=dilate)
    y = run_conv(backend, x, w, scale, bias, stride, pad, dilate, 0, True, (0, 0, -127, 127), (0, 0, -127, 127))
    assert np.array_equal(y, ref)


SHAPES = [  # ic, oc, kh, kw, n, ih, iw, stride, pad, relu, dilate  -- MobileNet-v2 / ResNet-50 layer classes + ragged
    (3, 32, 3, 3, 2, 32, 32, (2, 2), (1, 1), 1, (1, 1)),
    (32, 16, 1, 1, 2, 28, 28, (1, 1), (0, 0), 0, (1, 1)),
    (16, 96, 1, 1, 2, 28, 28, (1, 1), (0, 0), 1, (1, 1)),
    (144, 24, 1, 1, 1, 14, 14, (1, 1), (0, 0), 0, (1, 1)),
    (320, 1280, 1, 1, 2, 7, 7, (1, 1), (0, 0), 1, (1, 1)),
    (1280, 1001, 1, 1, 3, 1, 1, (1, 1), (0, 0), 0, (1, 1)),
    (64, 64, 3, 3, 2, 14, 14, (1, 1), (1, 1), 1, (1, 1)),
    (3, 64, 7, 7, 1, 40, 40, (2, 2), (3, 3), 1, (1, 1)),
    (37, 53, 3, 2, 2, 13, 9, (1, 2), (2, 1), 1, (2, 1)),
    (5, 7, 1, 1, 1, 1, 1, (1, 1), (0, 0), 0, (1, 1)),       # single pixel, tiny channels
    (200, 130, 1, 1, 1, 5, 3, (1, 1), (0, 0), 1, (1, 1)),
    (96, 24, 1, 1, 4, 56, 56, (1, 1), (0, 0), 0, (1, 1)),     # many M tiles: persistent loop, TMEM double buffering
    (576, 160, 1, 1, 4, 7, 7, (1, 1), (0, 0), 0, (1, 1)),     # 5 K blocks
    (960, 320, 1, 1, 8, 7, 7, (1, 1), (0, 0), 0, (1, 1)),     # 8 K blocks (ring wraps), 2 N chunks
    # narrow-K 1x1 convs on big maps: pixel-packed GEMM rows (P = 128 / p16(ic) pixels per row, block-diagonal weights)
    (16, 96, 1, 1, 4, 56, 56, (1, 1), (0, 0), 1, (1, 1)),     # P = 8, N' = 768 -> 3 chunks
    (32, 16, 1, 1, 2, 56, 56, (1, 1), (0, 0), 0, (1, 1)),     # P = 4, N' = 64, resident B
    (24, 144, 1, 1, 1, 64, 64, (1, 1), (0, 0), 1, (1, 1)),    # P = 4, ic padded 24 -> 32
    (64, 40, 1, 1, 1, 40, 40, (1, 1), (0, 0), 1, (1, 1)),     # P = 2, oc 40 -> 48: zero padding INSIDE every pixel block
    (10, 20, 1, 1, 3, 32, 32, (1, 1), (0, 0), 1, (1, 1)),     # P = 8, ragged ic and oc
    (130, 530, 1, 1, 2, 9, 9, (1, 1), (0, 0), 1, (1, 1)),     # ragged K and N, 3 N chunks
    # implicit GEMM on tcgen05 (variant 2 / auto): 128-byte, 64-byte and 16-byte K chunks, stride 2, dilation, ragged tiles
    (128, 128, 3, 3, 2, 14, 14, (1, 1), (1, 1), 1, (1, 1)),   # ResNet 3x3 class, cb = 128, 9 K blocks
    (256, 200, 3, 3, 1, 7, 7, (1, 1), (1, 1), 0, (1, 1)),     # cb = 128 x 2 chunks per tap, 18 K blocks, 2 N chunks, R = 16
    (64, 64, 3, 3, 3, 28, 28, (1, 1), (1, 1), 1, (1, 1)),     # cb = 64 (SWIZZLE_64B), TWp = 32, R = 4
    (192, 48, 3, 3, 2, 15, 15, (2, 2), (1, 1), 0, (1, 1)),    # cb = 64, stride 2, odd width (both column parities)
    (256, 512, 1, 1, 2, 14, 14, (2, 2), (0, 0), 0, (1, 1)),   # strided 1x1 (ResNet downsample), 3 N chunks
    (32, 32, 3, 3, 1, 150, 9, (1, 1), (1, 1), 1, (1, 1)),     # OH 150 x OW 9: TWp = 16, R = 8, ragged last tile
    (16, 24, 3, 3, 1, 6, 200, (1, 1), (1, 1), 1, (1, 1)),     # OW = 200 > 128: two row segments per output row
    (48, 80, 5, 5, 2, 12, 12, (1, 1), (2, 2), 1, (2, 2)),     # dilation 2, 16-byte chunks (Cp = 48), odd chunk count
    (20, 10, 2, 4, 1, 9, 11, (2, 1), (0, 1), 0, (1, 1)),      # asymmetric kernel / stride / pad
]


@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("shape", SHAPES)
def test_modern_conv_vs_oracle(backend, shape, variant):
    ic, oc, kh, kw, n, ih, iw, st, pad, relu, dl = shape
    if variant == 2 and st[1] > 2:
        pytest.skip("the tcgen05 implicit-GEMM kernel takes stride_w <= 2 (two column-parity TMA views)")
    rng = np.random.default_rng(ic * 1000 + oc)
    c = random_modern_case(rng, ic, oc, kh, kw, n, ih, iw, st, pad, relu, dl)
    bf, sx = O.fold_modern(c["w"], c["ws"], c["bias"], c["s_in"], c["z_in"], c["s_out"], c["z_out"])
    ref = O.conv_int8(c["x"], c["w"], c["ws"], sx, bf, stride=st, pad=pad, dilate=dl, z_in=c["z_in"],
                      min_v=c["z_out"] if relu else -127, max_v=127)
    y = run_conv(backend, c["x"], c["w"], c["ws"], c["bias"], st, pad, dl, relu, False,
                 (c["s_in"], c["z_in"], -128, 127), (c["s_out"], c["z_out"], -127, 127), variant=variant)
    assert np.array_equal(y, ref), np.abs(y.astype(int) - ref.astype(int)).max()
    sat = (np.abs(ref.astype(int)) == 127).mean()
    assert sat < 0.5, "test case saturates: it would hide epilogue errors"


def test_casts_vs_oracle(backend):
    from mnn_b200.backend import QuantAttr, Tensor
    rng = np.random.default_rng(5)
    for (n, c, h, w) in [(2, 3, 17, 19), (1, 40, 5, 7), (3, 1001, 1, 1)]:
        x = rng.uniform(-4, 4, (n, c, h, w)).astype(np.float32)
        x.flat[:8] = [0.5, -0.5, 1.5, -1.5, 2.5, -2.5, 1e9, -1e9]
        scale, zero = 0.031, 3.0
        t = backend.onAcquire(Tensor((n, c, h, w), "int8", QuantAttr(scale, zero, -127, 127)))
        backend.onCopyBuffer(x, t)          # float host -> int8 device = FloatToInt8 in the copy
        q = backend.onCopyBuffer(t, "same")
        assert np.array_equal(q, O.float_to_int8(x, scale, zero, -127, 127))
        f = backend.onCopyBuffer(t, "float")
        assert np.array_equal(f, O.int8_to_float(q, scale, zero))


def test_depthwise_vs_oracle(backend):
    from mnn_b200.backend import Op, QuantAttr, Tensor
    rng = np.random.default_rng(9)
    for (ch, k, n, ih, iw, st, pad, relu) in [(32, 3, 2, 16, 16, (1, 1), (1, 1), 1), (96, 3, 2, 15, 15, (2, 2), (1, 1), 1),
                                              (40, 5, 1, 9, 11, (1, 1), (2, 2), 0), (7, 3, 3, 6, 6, (1, 1), (0, 0), 1)]:
        x = rng.integers(-128, 128, (n, ch, ih, iw)).astype(np.int8)
        w = rng.integers(-127, 128, (ch, 1, k, k)).astype(np.int8)
        ws = (rng.uniform(0.002, 0.02, ch) / k).astype(np.float32)
        bias = rng.uniform(-1, 1, ch).astype(np.float32)
        s_in, s_out, z_in, z_out = 0.043, 0.061, int(rng.integers(-4, 5)), int(rng.integers(-4, 5))
        sc, bi = O.fold_depthwise(w, ws, bias, s_in, z_in, s_out, z_out)
        ref = O.depthwise_int8(x, w, sc, bi, stride=st, pad=pad, z_in=z_in, min_v=z_out if relu else -127, max_v=127)
        op = Op(type="DepthwiseConvInt8", conv=dict(ic=ch, oc=ch, kernel=(k, k), stride=st, pad=pad, group=ch,
                                                   relu=bool(relu)), weight=w, wscale=ws, bias=bias)
        xin = backend.onAcquire(Tensor((n, ch, ih, iw), "int8", QuantAttr(s_in, z_in, -128, 127)))
        backend.onCopyBuffer(x, xin)
        yout = Tensor((n, ch, 1, 1), "int8", QuantAttr(s_out, z_out, -127, 127))
        ex = backend.onCreate([xin], [yout], op)
        assert ex.onResize([xin], [yout]) == 0
        backend.onAcquire(yout)
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        y = backend.onCopyBuffer(yout, "same")
        assert np.array_equal(y, ref)


@pytest.mark.parametrize("variant", [1, 2])
def test_linear_w8_dynamic_vs_oracle(backend, variant):
    """fp32 output: tolerance 1e-3 relative to max|ref| (BASELINE.json north_star)."""
    import torch
    from mnn_b200.backend import Op, Tensor
    rng = np.random.default_rng(3)
    for (tokens, ic, oc, asym, has_bias) in [(8, 64, 48, False, True), (130, 256, 200, True, True),
                                             (512, 2048, 1024, True, False), (1, 96, 33, False, False)]:
        x = rng.uniform(-1, 1, (tokens, ic)).astype(np.float32)
        x[0, :] = 0  # absmax < 1e-7 branch
        wq = rng.integers(-128, 128, (oc, ic)).astype(np.int8)
        alpha = rng.uniform(0.001, 0.01, oc).astype(np.float32)
        wzero = rng.uniform(-0.05, 0.05, oc).astype(np.float32) if asym else None
        bias = rng.uniform(-1, 1, oc).astype(np.float32) if has_bias else None
        ref = O.linear_w8_dynamic(x, wq, alpha, wzero, bias)
        op = Op(type="LinearW8", conv=dict(ic=ic, oc=oc, kernel=(1, 1)), weight=wq, wscale=alpha, wzero=wzero, bias=bias)
        xin = Tensor((tokens, ic), "float", data=torch.from_numpy(x).cuda())
        yout = Tensor((tokens, oc), "float")
        ex = backend.onCreate([xin], [yout], op)
        from mnn_b200 import _capi
        _capi.check(_capi.lib().mnnb200_conv_int8_set_variant(ex._h, variant))
        assert ex.onResize([xin], [yout]) == 0
        yout.data = torch.full((tokens, oc), float("nan"), device="cuda")
        if tokens == 1:
            # one token = the reference's decode arithmetic, which only the GEMV kernel implements: a forced tensor-core variant
            # must refuse instead of computing the multi-token form
            assert ex.onExecute([xin], [yout]) == 2          # NOT_SUPPORT
            _capi.check(_capi.lib().mnnb200_conv_int8_set_variant(ex._h, 0))
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        y = yout.data.cpu().numpy()
        err = np.abs(y - ref).max() / max(np.abs(ref).max(), 1e-6)
        assert err <= 1e-3, err
        assert np.array_equal(y, ref), "dynamic-quant linear is expected to be bit-exact as well"


def test_depthwise_and_linear_golden_fixtures(backend):
    """vectors recorded from the UNMODIFIED reference CPU backend (tests/golden/make_golden.py: dw_linear_golden)."""
    import torch
    from mnn_b200.backend import Op, QuantAttr, Tensor
    from tests.test_oracle import wire_wzero
    g = load_golden("dw_linear_golden")
    for i in range(int(g["ndw"])):
        s_in, z_in, s_out, z_out = g[f"d{i}_q"]
        x, w = g[f"d{i}_x"], g[f"d{i}_w"]
        n, ch, ih, iw = x.shape
        k = w.shape[-1]
        op = Op(type="DepthwiseConvInt8", conv=dict(ic=ch, oc=ch, kernel=(k, k), stride=tuple(int(v) for v in g[f"d{i}_stride"]),
                                                   pad=tuple(int(v) for v in g[f"d{i}_pad"]), group=ch,
                                                   relu=bool(int(g[f"d{i}_relu"]))),
                weight=w, wscale=g[f"d{i}_ws"], bias=g[f"d{i}_bias"])
        xin = backend.onAcquire(Tensor((n, ch, ih, iw), "int8", QuantAttr(float(s_in), int(z_in), -128, 127)))
        backend.onCopyBuffer(x, xin)
        yout = Tensor((n, ch, 1, 1), "int8", QuantAttr(float(s_out), int(z_out), -127, 127))
        ex = backend.onCreate([xin], [yout], op)
        assert ex.onResize([xin], [yout]) == 0
        backend.onAcquire(yout)
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        assert np.array_equal(backend.onCopyBuffer(yout, "same"), g[f"d{i}_y"]), f"depthwise golden {i}"
    for j in range(int(g["nlin"])):
        x, wq, alpha, wmin, bias = g[f"l{j}_x"], g[f"l{j}_wq"], g[f"l{j}_alpha"], g[f"l{j}_wmin"], g[f"l{j}_bias"]
        tokens, ic = x.shape
        oc = wq.shape[0]
        op = Op(type="LinearW8", conv=dict(ic=ic, oc=oc, kernel=(1, 1)), weight=wq, wscale=alpha,
                wzero=wire_wzero(wmin, alpha) if wmin.size else None, bias=bias if bias.size else None)
        xin = Tensor((tokens, ic), "float", data=torch.from_numpy(x).cuda())
        yout = Tensor((tokens, oc), "float")
        ex = backend.onCreate([xin], [yout], op)
        assert ex.onResize([xin], [yout]) == 0
        yout.data = torch.zeros((tokens, oc), device="cuda")
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        ref = g[f"l{j}_y"]
        err = np.abs(yout.data.cpu().numpy() - ref).max() / np.abs(ref).max()
        assert err <= 1e-3, (j, err)      # north_star tolerance for fp32 outputs; observed ~1e-6


@pytest.mark.parametrize("tokens,ic,oc,asym,has_bias,relu", [(1, 2048, 6144, True, True, 0), (1, 5504, 2048, True, False, 0),
                                                             (1, 100, 77, False, False, 0), (1, 250, 64, True, True, 1),
                                                             (2, 520, 301, False, True, 1), (3, 96, 33, True, True, 0),
                                                             (5, 2048, 1000, True, False, 0), (8, 1040, 777, False, False, 0)])
def test_linear_w8_decode_gemv_bit_exact(backend, tokens, ic, oc, asym, has_bias, relu):
    """The decode step (<= 8 tokens) streams the weights once through the dp4a GEMV (variant 4; what auto picks there): its output
    equals the oracle and, for 2..8 tokens, the tensor-core kernel (variant 2) bit for bit -- ragged oc (301, 33, 777), K tails
    (520, 1040, 5504), every token-count template (1, 2, 4, 8 with 3 and 5 padded), an all-zero token (absmax < 1e-7 branch).
    ONE token follows the reference's single-quant decode arithmetic (asymmetric input quantisation, zero point folded into the
    bias): the oracle restates it and is pinned on the live reference (tests/test_oracle.py, dw_linear_golden.npz decode cases)."""
    import torch
    from mnn_b200 import _capi
    from mnn_b200.backend import Op, Tensor
    rng = np.random.default_rng(tokens * 131 + oc)
    x = rng.uniform(-1, 1, (tokens, ic)).astype(np.float32)
    if tokens == 1 and ic == 100:
        x = np.abs(x) + np.float32(0.2)     # one-sided row with ic % 16 != 0: the pack padding's zeros enter the row minimum
    if tokens > 1:
        x[1, :] = 0
    wq = rng.integers(-128, 128, (oc, ic)).astype(np.int8)
    alpha = rng.uniform(0.001, 0.01, oc).astype(np.float32)
    wzero = rng.uniform(-0.05, 0.05, oc).astype(np.float32) if asym else None
    bias = rng.uniform(-1, 1, oc).astype(np.float32) if has_bias else None
    ref = O.linear_w8_dynamic(x, wq, alpha, wzero, bias)
    if relu:
        ref = np.maximum(ref, 0)
    op = Op(type="LinearW8", conv=dict(ic=ic, oc=oc, kernel=(1, 1), relu=bool(relu)), weight=wq, wscale=alpha, wzero=wzero, bias=bias)
    outs = {}
    for variant in ((4, 0) if tokens == 1 else (2, 4, 0)):     # one token: the reference's decode arithmetic, GEMV only
        xin = Tensor((tokens, ic), "float", data=torch.from_numpy(x).cuda())
        yout = Tensor((tokens, oc), "float")
        ex = backend.onCreate([xin], [yout], op)
        _capi.check(_capi.lib().mnnb200_conv_int8_set_variant(ex._h, variant))
        assert ex.onResize([xin], [yout]) == 0
        yout.data = torch.full((tokens, oc), float("nan"), device="cuda")
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        outs[variant] = yout.data.cpu().numpy()
    assert not np.isnan(outs[4]).any()
    if tokens > 1:
        assert np.array_equal(outs[4], outs[2]), np.abs(outs[4] - outs[2]).max()
    assert np.array_equal(outs[0], outs[4])
    assert np.array_equal(outs[4], ref), np.abs(outs[4] - ref).max()


@pytest.mark.parametrize("tokens,ic,oc,asym,has_bias", [(512, 2048, 1024, True, False), (256, 128, 64, False, True),
                                                        (700, 520, 300, True, True), (1024, 5504, 2048, False, False)])
def test_linear_w8_cta_pair_variant_bit_exact(backend, tokens, ic, oc, asym, has_bias):
    """The cta_group::2 (UMMA M = 256) kernel must produce exactly what the single-CTA kernel and the oracle produce:
    ragged M (700 = 2 full pair tiles + 188 rows), ragged N (300 -> two 160-column chunks), K tail (520), deep K (5504)."""
    import torch
    from mnn_b200 import _capi
    from mnn_b200.backend import Op, Tensor
    rng = np.random.default_rng(tokens + oc)
    x = rng.uniform(-1, 1, (tokens, ic)).astype(np.float32)
    wq = rng.integers(-128, 128, (oc, ic)).astype(np.int8)
    alpha = rng.uniform(0.001, 0.01, oc).astype(np.float32)
    wzero = rng.uniform(-0.05, 0.05, oc).astype(np.float32) if asym else None
    bias = rng.uniform(-1, 1, oc).astype(np.float32) if has_bias else None
    op = Op(type="LinearW8", conv=dict(ic=ic, oc=oc, kernel=(1, 1)), weight=wq, wscale=alpha, wzero=wzero, bias=bias)
    outs = {}
    for variant in (2, 3):
        xin = Tensor((tokens, ic), "float", data=torch.from_numpy(x).cuda())
        yout = Tensor((tokens, oc), "float")
        ex = backend.onCreate([xin], [yout], op)
        _capi.check(_capi.lib().mnnb200_conv_int8_set_variant(ex._h, variant))
        assert ex.onResize([xin], [yout]) == 0
        yout.data = torch.full((tokens, oc), float("nan"), device="cuda")
        for _ in range(2):      # twice: barrier phases / TMEM reuse across launches
            assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        outs[variant] = yout.data.cpu().numpy()
    assert not np.isnan(outs[3]).any()
    assert np.array_equal(outs[2], outs[3]), f"{np.count_nonzero(outs[2] != outs[3])} elements differ"
    if tokens * ic * oc <= 512 * 2048 * 1024:
        assert np.array_equal(outs[3], O.linear_w8_dynamic(x, wq, alpha, wzero, bias))


def test_lite_two_ctas_per_sm_configuration_bit_exact():
    """The opt-in `MNNB200_LITE=1` configuration of the tcgen05 GEMM (384-thread CTAs, two per SM, TMEM sized to the tile)
    is selected through an environment variable read once per process: re-run the 1x1 parity cases in a child process."""
    import subprocess
    import sys
    env = dict(os.environ, MNNB200_LITE="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_parity.py"), "-m", "gpu", "-q", "-x",
                        "-k", "test_modern_conv_vs_oracle and 2-"], env=env, cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-1500:]
    assert " passed" in r.stdout


def test_error_behaviour_mirrors_mnn_error_codes(backend):
    """Status codes are numerically MNN::ErrorCode (include/MNN/ErrorCode.hpp): COMPUTE_SIZE_ERROR = 3 for an empty shape,
    NO_EXECUTION = 4 for execute before resize, NOT_SUPPORT = 2 / INVALID_VALUE = 5 for what the path does not take."""
    import ctypes as C
    from mnn_b200 import _capi
    from mnn_b200._capi import ConvDesc
    L, rt = _capi.lib(), backend.runtime._h
    w = np.ones((8, 8, 3, 3), np.int8)
    ws = np.ones(8, np.float32)
    d = ConvDesc(8, 8, 3, 3, 1, 1, 1, 1, 1, 1, 1, 0)
    h = C.c_void_p()
    assert L.mnnb200_conv_int8_create(rt, C.byref(d), w.ctypes.data_as(C.c_void_p), ws.ctypes.data_as(C.c_void_p), None, C.byref(h)) == 0
    assert L.mnnb200_conv_int8_execute(h, None, None) == 4                               # before resize
    oh, ow = C.c_int(0), C.c_int(0)
    assert L.mnnb200_conv_int8_resize(h, 0, 8, 8, 0.1, 0, 0.1, 0, -127, 127, C.byref(oh), C.byref(ow)) == 3      # empty batch
    assert L.mnnb200_conv_int8_resize(h, 1, 1, 1, 0.1, 0, 0.0, 0, -127, 127, C.byref(oh), C.byref(ow)) == 5      # zero output scale
    oh, ow = C.c_int(0), C.c_int(0)
    assert L.mnnb200_conv_int8_resize(h, 1, 1, 1, 0.1, 0, 0.1, 0, -127, 127, C.byref(oh), C.byref(ow)) == 0 and (oh.value, ow.value) == (1, 1)
    assert L.mnnb200_dwconv_int8_resize(h, 1, 4, 4, 0.1, 0, 0.1, 0, -127, 127, C.byref(oh), C.byref(ow)) == 5    # wrong execution kind
    L.mnnb200_exec_destroy(h)
    dg = ConvDesc(8, 8, 3, 3, 1, 1, 1, 1, 1, 1, 2, 0)
    assert L.mnnb200_conv_int8_create(rt, C.byref(dg), w.ctypes.data_as(C.c_void_p), ws.ctypes.data_as(C.c_void_p), None, C.byref(h)) == 2   # grouped conv
    # Winograd: malformed attr blob -> INVALID_VALUE, unsupported unit layout -> NOT_SUPPORT
    bad = np.array([1, 1, 6, 0, 0, 3, 3, 2, 2], np.int32)
    assert L.mnnb200_conv_int8_wino_create(rt, C.byref(d), w.ctypes.data_as(C.c_void_p), ws.ctypes.data_as(C.c_void_p), None,
                                           bad.ctypes.data_as(C.c_void_p), int(bad.size), C.byref(h)) == 5
    two = np.array([0, 2, 6, 0, 0, 3, 3, 2, 2], np.int32)
    assert L.mnnb200_conv_int8_wino_create(rt, C.byref(d), w.ctypes.data_as(C.c_void_p), ws.ctypes.data_as(C.c_void_p), None,
                                           two.ctypes.data_as(C.c_void_p), int(two.size), C.byref(h)) == 2
    assert b"Winograd" in L.mnnb200_last_error() or b"wino" in L.mnnb200_last_error()
    assert L.mnnb200_matmul_create(rt, 0, 4, 4, 4, 0, 0, 0, C.byref(h)) == 5


# ---- conv group: one persistent launch over a list of GEMM-shaped convs (mnnb200_conv_group_*) ------------------------
GROUP_SHAPES = [  # ic, oc, n, ih, iw, relu  -- every MobileNet-v2 1x1 class + ragged rows / K blocks / N chunks
    (32, 16, 2, 56, 56, 0), (16, 96, 2, 56, 56, 1), (96, 24, 2, 28, 28, 0), (24, 144, 1, 28, 28, 1),
    (144, 32, 2, 14, 14, 0), (192, 64, 3, 7, 7, 0), (64, 384, 2, 14, 14, 1), (384, 96, 1, 14, 14, 0),
    (576, 160, 4, 7, 7, 0), (960, 320, 3, 7, 7, 0), (320, 1280, 2, 7, 7, 1), (1280, 1001, 3, 1, 1, 0),
    (5, 7, 1, 1, 1, 0), (130, 530, 2, 9, 9, 1), (200, 130, 1, 5, 3, 1), (10, 200, 1, 33, 17, 1),
]


def test_conv_group_vs_oracle_and_single(backend):
    """All members in ONE launch: every output equals the oracle and the per-layer tcgen05 kernel bit for bit."""
    from mnn_b200.backend import ConvGroupExecution, Op, QuantAttr, Tensor
    layers = []
    for (ic, oc, n, ih, iw, relu) in GROUP_SHAPES:
        rng = np.random.default_rng(ic * 977 + oc)
        c = random_modern_case(rng, ic, oc, 1, 1, n, ih, iw, (1, 1), (0, 0), relu)
        op = Op(type="ConvInt8", conv=dict(ic=ic, oc=oc, kernel=(1, 1), stride=(1, 1), pad=(0, 0), dilate=(1, 1), group=1,
                                          relu=bool(relu)), weight=c["w"], wscale=c["ws"], bias=c["bias"])
        xin = backend.onAcquire(Tensor((n, ic, ih, iw), "int8", QuantAttr(c["s_in"], c["z_in"], -128, 127)))
        backend.onCopyBuffer(c["x"], xin)
        yout = Tensor((n, oc, 1, 1), "int8", QuantAttr(c["s_out"], c["z_out"], -127, 127))
        ex = backend.onCreate([xin], [yout], op)
        assert ex is not None and ex.onResize([xin], [yout]) == 0
        backend.onAcquire(yout)
        assert ConvGroupExecution.groupable(ex)
        layers.append((c, relu, ex, xin, yout))
    singles = []
    for c, relu, ex, xin, yout in layers:
        ex.set_variant(2)
        yout.data.fill_(77)
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        singles.append(backend.onCopyBuffer(yout, "same"))
        yout.data.fill_(77)            # poison again: the group must overwrite every valid byte
    grp = ConvGroupExecution(backend, [l[2] for l in layers])
    assert grp.bind([l[3] for l in layers], [l[4] for l in layers]) == 0
    for rep in range(2):                # second pass: barriers / TMEM of a fresh launch, same answer
        assert grp.onExecute() == 0
        backend.onSync()
        for (c, relu, ex, xin, yout), single in zip(layers, singles):
            oc = c["w"].shape[0]
            raw = yout.data.cpu().numpy()
            assert (raw[..., oc:] == 0).all(), "NHWC16 channel padding must stay zero"
            y = backend.onCopyBuffer(yout, "same")
            bf, sx = O.fold_modern(c["w"], c["ws"], c["bias"], c["s_in"], c["z_in"], c["s_out"], c["z_out"])
            ref = O.conv_int8(c["x"], c["w"], c["ws"], sx, bf, stride=(1, 1), pad=(0, 0), z_in=c["z_in"],
                              min_v=c["z_out"] if relu else -127, max_v=127)
            assert np.array_equal(y, ref), (c["w"].shape, np.abs(y.astype(int) - ref.astype(int)).max())
            assert np.array_equal(y, single)


def test_conv_group_mixed_gemm_and_implicit_members(backend):
    """1x1 convs and k > 1 / strided convs in ONE launch (layer modes 0 and 1 of the conv-group kernel)."""
    from mnn_b200.backend import ConvGroupExecution, Op, QuantAttr, Tensor
    shapes = [(32, 16, 1, 1, 2, 28, 28, (1, 1), (0, 0), 0), (8, 32, 3, 3, 2, 32, 32, (2, 2), (1, 1), 1),
              (64, 64, 3, 3, 2, 14, 14, (1, 1), (1, 1), 1), (128, 256, 3, 3, 1, 7, 7, (1, 1), (1, 1), 0),
              (96, 24, 1, 1, 1, 14, 14, (1, 1), (0, 0), 0), (256, 128, 1, 1, 2, 14, 14, (2, 2), (0, 0), 1)]
    layers = []
    for (ic, oc, kh, kw, n, ih, iw, st, pad, relu) in shapes:
        rng = np.random.default_rng(ic * 31 + oc + kh)
        c = random_modern_case(rng, ic, oc, kh, kw, n, ih, iw, st, pad, relu)
        op = Op(type="ConvInt8", conv=dict(ic=ic, oc=oc, kernel=(kh, kw), stride=st, pad=pad, dilate=(1, 1), group=1, relu=bool(relu)),
                weight=c["w"], wscale=c["ws"], bias=c["bias"])
        xin = backend.onAcquire(Tensor((n, ic, ih, iw), "int8", QuantAttr(c["s_in"], c["z_in"], -128, 127)))
        backend.onCopyBuffer(c["x"], xin)
        yout = Tensor((n, oc, 1, 1), "int8", QuantAttr(c["s_out"], c["z_out"], -127, 127))
        ex = backend.onCreate([xin], [yout], op)
        assert ex is not None and ex.onResize([xin], [yout]) == 0
        backend.onAcquire(yout)
        yout.data.fill_(77)
        assert ConvGroupExecution.groupable(ex)
        layers.append((c, relu, st, pad, ex, xin, yout))
    grp = ConvGroupExecution(backend, [l[4] for l in layers])
    assert grp.bind([l[5] for l in layers], [l[6] for l in layers]) == 0
    assert grp.onExecute() == 0
    backend.onSync()
    for c, relu, st, pad, ex, xin, yout in layers:
        oc = c["w"].shape[0]
        assert (yout.data.cpu().numpy()[..., oc:] == 0).all()
        y = backend.onCopyBuffer(yout, "same")
        bf, sx = O.fold_modern(c["w"], c["ws"], c["bias"], c["s_in"], c["z_in"], c["s_out"], c["z_out"])
        ref = O.conv_int8(c["x"], c["w"], c["ws"], sx, bf, stride=st, pad=pad, z_in=c["z_in"],
                          min_v=c["z_out"] if relu else -127, max_v=127)
        assert np.array_equal(y, ref), (c["w"].shape, np.abs(y.astype(int) - ref.astype(int)).max())


def test_conv_group_rejects_unsupported_member(backend):
    from mnn_b200.backend import ConvGroupExecution, Op, QuantAttr, Tensor
    rng = np.random.default_rng(3)
    c = random_modern_case(rng, 16, 16, 3, 3, 1, 9, 9, (1, 3), (1, 1), 0)       # stride_w = 3: not on the tcgen05 kernels
    op = Op(type="ConvInt8", conv=dict(ic=16, oc=16, kernel=(3, 3), stride=(1, 3), pad=(1, 1), dilate=(1, 1), group=1, relu=False),
            weight=c["w"], wscale=c["ws"], bias=c["bias"])
    xin = backend.onAcquire(Tensor((1, 16, 9, 9), "int8", QuantAttr(c["s_in"], c["z_in"], -128, 127)))
    backend.onCopyBuffer(c["x"], xin)
    yout = Tensor((1, 16, 1, 1), "int8", QuantAttr(c["s_out"], c["z_out"], -127, 127))
    ex = backend.onCreate([xin], [yout], op)
    assert ex.onResize([xin], [yout]) == 0
    backend.onAcquire(yout)
    assert not ConvGroupExecution.groupable(ex)
    grp = ConvGroupExecution(backend, [ex])
    assert grp.bind([xin], [yout]) == 2      # NOT_SUPPORT, as Backend::onCreate returning nullptr would signal
    # ... and the conv itself still runs (mma.sync implicit GEMM) and is right
    assert ex.onExecute([xin], [yout]) == 0
    backend.onSync()
    bf, sx = O.fold_modern(c["w"], c["ws"], c["bias"], c["s_in"], c["z_in"], c["s_out"], c["z_out"])
    ref = O.conv_int8(c["x"], c["w"], c["ws"], sx, bf, stride=(1, 3), pad=(1, 1), z_in=c["z_in"], min_v=-127, max_v=127)
    assert np.array_equal(backend.onCopyBuffer(yout, "same"), ref)


def test_scale_and_pool_int8_vs_oracle(backend):
    """int8 Scale (CPUScaleInt8 integer arithmetic) and int8 pooling with equal quant attrs (x86 semantics: uint8 storage,
    (sum * floor(2^24 / count)) >> 24; SIGNED compare of the stored bytes for max) against the oracle, bit for bit."""
    from mnn_b200.backend import Op, QuantAttr, Tensor
    rng = np.random.default_rng(21)
    for (n, c, h, w) in [(2, 64, 14, 14), (1, 37, 9, 5), (3, 256, 7, 7)]:
        x = rng.integers(-128, 128, (n, c, h, w)).astype(np.int8)
        sc = rng.uniform(0.2, 3.0, c).astype(np.float32) * rng.choice([-1, 1], c).astype(np.float32)
        bi = rng.uniform(-2, 2, c).astype(np.float32)
        qi, qo = QuantAttr(0.043, 3, -128, 127), QuantAttr(0.061, -2, -127, 127)
        xin = backend.onAcquire(Tensor((n, c, h, w), "int8", qi))
        backend.onCopyBuffer(x, xin)
        yout = Tensor((n, c, h, w), "int8", qo)
        ex = backend.onCreate([xin], [yout], Op(type="ScaleInt8", extra=dict(scale=sc, bias=bi)))
        assert ex.onResize([xin], [yout]) == 0
        backend.onAcquire(yout)
        yout.data.fill_(77)
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        assert (yout.data.cpu().numpy()[..., c:] == 0).all()
        ref = O.scale_int8(x, sc, bi, qi.scale, int(qi.zero), qo.scale, int(qo.zero), -127, 127)
        got = backend.onCopyBuffer(yout, "same")
        assert np.array_equal(got, ref), np.abs(got.astype(int) - ref.astype(int)).max()
    for (n, c, h, w, k, s, p, avg) in [(2, 64, 15, 15, 3, 2, 1, False), (2, 64, 15, 15, 3, 2, 1, True), (1, 20, 7, 7, 7, 7, 0, True),
                                       (3, 130, 8, 6, 2, 2, 0, False), (1, 16, 5, 9, 3, 1, 1, True)]:
        x = rng.integers(-128, 128, (n, c, h, w)).astype(np.int8)
        q = QuantAttr(0.05, 1, -127, 127)
        xin = backend.onAcquire(Tensor((n, c, h, w), "int8", q))
        backend.onCopyBuffer(x, xin)
        yout = Tensor((n, c, 1, 1), "int8", q)
        ex = backend.onCreate([xin], [yout], Op(type="PoolInt8", extra=dict(kernel=(k, k), stride=(s, s), pad=(p, p), pad_type=0,
                                                                           ceil_model=False, is_avg=avg)))
        assert ex.onResize([xin], [yout]) == 0
        backend.onAcquire(yout)
        assert ex.onExecute([xin], [yout]) == 0
        backend.onSync()
        ref = O.pool_int8_x86(x, (k, k), (s, s), (p, p), avg)
        got = backend.onCopyBuffer(yout, "same")
        assert got.shape == ref.shape and np.array_equal(got, ref), (k, s, p, avg)
