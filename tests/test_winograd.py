"""int8 Winograd conv (SURVEY a5/a6): the oracle against the committed real-reference fixture and (when built) the live
reference AVX2 build; the CUDA path (-m gpu) against both, BIT FOR BIT; full-size properties."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.cases import kat_wino, random_wino_case, wino_oracle

GOLD = os.path.join(os.path.dirname(__file__), "golden", "wino_int8_golden.npz")


def golden_cases():
    g = np.load(GOLD)
    for i in range(int(g["ncase"])):
        c = {k[len(f"w{i}_"):]: g[k] for k in g.files if k.startswith(f"w{i}_")}
        for k in ("s_in", "s_out"):
            c[k] = float(c[k])
        for k in ("z_in", "z_out", "pad", "unit"):
            c[k] = int(c[k])
        c["relu"] = bool(c["relu"])
        yield i, c


def test_oracle_vs_golden_reference_outputs():
    n = 0
    for i, c in golden_cases():
        y = wino_oracle(O, c, c["unit"])
        assert np.array_equal(y, c["y"]), f"wino golden {i}"
        n += 1
    assert n >= 7


def test_oracle_close_to_direct_float_conv():
    """Sanity of the whole chain (the reference test's own acceptance idea, test/op/ConvInt8Test.cpp:493-564): the
    Winograd int8 result tracks the float convolution of the dequantised tensors within a few LSB."""
    rng = np.random.default_rng(5)
    for unit in (2, 4):
        c = random_wino_case(rng, unit, 1, 16, 8, 12, 12, 1, False)
        y = wino_oracle(O, c, unit).astype(np.float64)
        xs = (c["x"].astype(np.float64) - c["z_in"]) * c["s_in"]
        wf = c["w"].astype(np.float64) * c["ws"][:, None, None, None]
        xp = np.pad(xs, ((0, 0), (0, 0), (1, 1), (1, 1)))
        acc = np.zeros((1, 8, 12, 12))
        for ky in range(3):
            for kx in range(3):
                acc += np.einsum("oc,nchw->nohw", wf[:, :, ky, kx], xp[:, :, ky:ky + 12, kx:kx + 12])
        ref = (acc + c["bias"][None, :, None, None]) / c["s_out"] + c["z_out"]
        refc = np.clip(ref, -127, 127)
        assert np.abs(y - refc).mean() < 8.0 and np.corrcoef(y.ravel(), refc.ravel())[0, 1] > 0.9


def test_oracle_bit_exact_vs_live_reference_avx2():
    rng = np.random.default_rng(99)
    c = kat_wino(3, 32, 32, 39, 47)       # the reference unit test's exact configuration, batch 3
    assert np.array_equal(wino_oracle(O, c, 2), wino_oracle(O, c, 2, O.ref_wino))
    for unit, n, ic, oc, ih, iw, pad, relu in [(2, 1, 3, 5, 3, 3, 1, False), (4, 2, 24, 17, 9, 13, 1, True),
                                               (6, 1, 16, 16, 20, 6, 1, False), (4, 1, 70, 9, 5, 5, 0, True)]:
        c = random_wino_case(rng, unit, n, ic, oc, ih, iw, pad, relu)
        assert np.array_equal(wino_oracle(O, c, unit), wino_oracle(O, c, unit, O.ref_wino)), (unit, ic, oc)


# ------------------------------------------------------------------------------------------------------------- GPU
def run_wino(backend, c, unit):
    from mnn_b200.backend import Op, QuantAttr, Tensor, encode_winograd_attr
    x, w = c["x"], c["w"]
    n, ic, ih, iw = x.shape
    oc = w.shape[0]
    a2 = (unit + 2) ** 2
    ins = np.broadcast_to(np.asarray(c["in_scales"], np.float32), (a2,))
    inz = np.broadcast_to(np.asarray(c["in_zeros"], np.int32), (a2,))
    wsc = np.broadcast_to(np.asarray(c["w_scales"], np.float32), (a2, oc))
    attr = encode_winograd_attr([(0, 0, 3, 3, unit, unit, ins, inz, wsc)])
    op = Op(type="ConvInt8", conv=dict(ic=ic, oc=oc, kernel=(3, 3), stride=(1, 1), pad=(c["pad"], c["pad"]), group=1,
                                      relu=bool(c["relu"])),
            weight=w, wscale=c["ws"], bias=c["bias"], extra=dict(winograd_attr=attr))
    xin = backend.onAcquire(Tensor((n, ic, ih, iw), "int8", QuantAttr(c["s_in"], c["z_in"], -128, 127)))
    backend.onCopyBuffer(x, xin)
    yout = Tensor((n, oc, 1, 1), "int8", QuantAttr(c["s_out"], c["z_out"], -127, 127))
    ex = backend.onCreate([xin], [yout], op)
    assert ex is not None and type(ex).__name__ == "ConvInt8WinogradExecution"
    assert ex.onResize([xin], [yout]) == 0
    backend.onAcquire(yout)
    yout.data.fill_(77)
    assert ex.onExecute([xin], [yout]) == 0
    backend.onSync()
    raw = yout.data.cpu().numpy()
    assert (raw[..., oc:] == 0).all(), "NHWC16 channel padding must stay zero"
    return backend.onCopyBuffer(yout, "same"), ex


@pytest.mark.gpu
def test_gpu_vs_golden_reference_outputs(backend):
    for i, c in golden_cases():
        y, _ = run_wino(backend, c, c["unit"])
        assert y.shape == c["y"].shape
        assert np.array_equal(y, c["y"]), f"wino golden {i}: {np.abs(y.astype(int) - c['y'].astype(int)).max()}"


@pytest.mark.gpu
@pytest.mark.parametrize("unit,n,ic,oc,ih,iw,pad,relu", [
    (2, 2, 64, 64, 14, 14, 1, True),       # ResNet 3x3 class
    (4, 1, 128, 128, 28, 28, 1, True),     # the reference speed test's shape (test/op/ConvInt8Test.cpp:677-699)
    (6, 1, 128, 128, 28, 28, 1, False),
    (2, 3, 5, 7, 3, 3, 1, False),          # one tile per image, tiny ragged channels
    (4, 2, 130, 270, 9, 10, 1, True),      # 2 K blocks, 2 N chunks, ragged tiles
    (6, 2, 48, 40, 13, 11, 0, False),
    (2, 1, 300, 24, 1, 1, 1, True),        # 1x1 image, pad only
])
def test_gpu_vs_oracle(backend, unit, n, ic, oc, ih, iw, pad, relu):
    rng = np.random.default_rng(unit * 1000 + ic)
    c = random_wino_case(rng, unit, n, ic, oc, ih, iw, pad, relu)
    y, _ = run_wino(backend, c, unit)
    ref = wino_oracle(O, c, unit)
    assert np.array_equal(y, ref), f"max diff {np.abs(y.astype(int) - ref.astype(int)).max()}, n={np.count_nonzero(y != ref)}"


@pytest.mark.gpu
def test_gpu_full_size_properties(backend):
    """BASELINE configs[2] size class (ResNet-50 3x3, C=64, 56x56, batch 64) -- too big for the scalar oracle.  Checked
    through size-independent properties: (1) batch independence: image b of the batched run == the same image run alone
    (which IS checked against the oracle); (2) determinism across two runs."""
    rng = np.random.default_rng(7)
    c = random_wino_case(rng, 2, 64, 64, 64, 56, 56, 1, True)
    y, ex = run_wino(backend, c, 2)
    y2, _ = run_wino(backend, c, 2)
    assert np.array_equal(y, y2)
    for b in (0, 37, 63):
        c1 = dict(c, x=c["x"][b:b + 1])
        y1, _ = run_wino(backend, c1, 2)
        assert np.array_equal(y1[0], y[b])
    c1 = dict(c, x=c["x"][5:6, :, :20, :20])
    y1, _ = run_wino(backend, c1, 2)
    assert np.array_equal(y1, wino_oracle(O, c1, 2))
    bytes_, macs = ex.cost()
    assert macs == 64 * 56 * 56 * 64 * 64 * 9


def test_mnn_reader_parses_winograd_attr_of_a_real_model():
    """tests/golden/wino_modern_conv.mnn = {Input, Convolution(IDST int8 weights, tensor quant info, winogradAttr)} written by the
    reference's own FlatBuffers code (oracle/refdump.cpp convModern, REFDUMP_WINO_UNIT=2); the y in the .npz is what the REFERENCE
    (AVX2 build) produced for it -- and equals the oracle.  The reader must surface the attr so that the sessions pick Winograd
    exactly when the reference does (ConvInt8Winograd::mustUse)."""
    from mnn_b200 import mnn_file
    from mnn_b200.session import conv_op_from_node
    from mnn_b200 import graph
    root = os.path.dirname(__file__)
    net = mnn_file.load(os.path.join(root, "golden", "wino_modern_conv.mnn"))
    g = np.load(os.path.join(root, "golden", "wino_modern_conv.npz"))
    node = next(o for o in net.ops if o.conv is not None)
    c = node.conv
    assert c.winograd_attr is not None and c.winograd_attr[:9].tolist() == [0, 1, 6 + 2 * 16 + 16 * 24, 0, 0, 3, 3, 2, 2]
    assert np.allclose(c.winograd_attr[9:25].view(np.float32), float(g["in_scale"]))
    assert np.allclose(c.winograd_attr[41:].view(np.float32), float(g["w_scale"]))
    assert c.sym == dict(zero_point=int(g["z_in"]), output_zero_point=int(g["z_out"]), clamp_min=-127, clamp_max=127)
    assert np.array_equal(c.weight, g["w"]) and np.allclose(c.alpha, g["ws"]) and np.allclose(c.bias, g["bias"])
    graph.infer_shapes(net, (2, 16, 11, 13))
    op = conv_op_from_node(node)
    assert op.type == "ConvInt8" and np.array_equal(op.extra["winograd_attr"], c.winograd_attr)
    # the recorded reference output equals the oracle on the decoded model
    y = O.wino_conv_int8(g["x"], c.weight, c.alpha, c.bias, np.float32(g["in_scale"]), 0, np.float32(g["w_scale"]), 2, 1,
                         float(g["s_in"]), int(g["z_in"]), float(g["s_out"]), int(g["z_out"]), -127, 127, True)
    assert np.array_equal(y, g["y"])


@pytest.mark.gpu
def test_gpu_mnn_model_with_winograd_attr_matches_reference_output():
    """A converted .mnn whose Convolution carries a winogradAttr (written by the reference's own FlatBuffers code) through the
    product path -- .mnn reader -> WholeNetSession -> FloatToInt8 / ConvInt8Winograd / Int8ToFloat executions -> C ABI --
    must reproduce, bit for bit, the int8 tensor the reference CPU backend (AVX2 build) produced for the same file."""
    from mnn_b200.session import WholeNetSession
    root = os.path.dirname(__file__)
    g = np.load(os.path.join(root, "golden", "wino_modern_conv.npz"))
    sess = WholeNetSession(os.path.join(root, "golden", "wino_modern_conv.mnn"), 2, input_hw=(11, 13))
    assert [type(s[1]).__name__ for s in sess.steps] == ["FloatToInt8Execution", "ConvInt8WinogradExecution", "Int8ToFloatExecution"]
    sess.set_input((g["x"].astype(np.float32) - np.float32(g["z_in"])) * np.float32(g["s_in"]))
    sess.run()
    got = sess.read_int8(list(sess.checkpoints)[-1])
    assert np.array_equal(got, g["y"].reshape(got.shape))
