"""GPU: the whole MobileNet-v2 int8 .mnn on the CUDA path (no CPU fallback) against the REAL reference CPU backend:
committed checkpoints at batch 1, and every op at batch 2 against the digests of the reference's own dump
(tests/golden/reference_fullsize.npz, recorded by tests/golden/make_golden.py)."""
import hashlib
import os

import numpy as np
import pytest

from tests.cases import load_golden, refdump_input

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
MODEL = os.path.join(GOLD, "mbv2_int8.mnn")
# Softmax runs an fp32 exp internally (the reference uses its own polynomial): +-1 LSB there, bit-exact elsewhere
FP_INTERNAL = ("MobilenetV2/Predictions/Softmax",)


def test_wholenet_checkpoints_vs_reference_golden():
    from mnn_b200.session import WholeNetSession
    g = load_golden("mbv2_int8_checkpoints")
    sess = WholeNetSession(MODEL, 1)
    sess.set_input(g["input"])
    sess.run()
    names = [str(n) for n in g["names"]]
    assert len(names) >= 10
    for i, name in enumerate(names):
        got = sess.read_int8(name)
        ref = g[f"t{i}"].reshape(got.shape)
        d = np.abs(got.astype(int) - ref.astype(int)).max()
        assert d <= (1 if name in FP_INTERNAL else 0), f"{name}: max |diff| = {d}"
    out = sess.get_output()
    ref = g["output"].reshape(out.shape)
    assert np.abs(out - ref).max() <= 1e-3 * max(np.abs(ref).max(), 1e-6) + 0.05   # one softmax LSB = scale ~0.03


def _check_every_op(sess, g, what=""):
    """every int8 tensor of the reference's per-command dump (batch 2, input seed 11, quantised with the tensor's own attrs)
    against the session's checkpoint of the same name: bit-exact (sha256 of the int8 codes), softmax within 1 LSB"""
    checked = 0
    for name, digest in zip(g["every_op_names"], g["every_op_sha256"]):
        name = str(name)
        if name not in sess.checkpoints:
            continue
        got = np.ascontiguousarray(sess.read_int8(name), np.int8)
        if name in FP_INTERNAL:
            ref = g[f"every_op_{name}"].reshape(got.shape)
            dmax = np.abs(got.astype(int) - ref.astype(int)).max()
            assert dmax <= 1, f"{what}{name}: max |diff| = {dmax}"
        else:
            assert hashlib.sha256(got.tobytes()).hexdigest() == str(digest), f"{what}{name}: differs from the reference"
        checked += 1
    assert checked >= 60, checked       # 36 conv + 17 depthwise + 10 add + pool + softmax


@pytest.mark.parametrize("batch", [2])
def test_wholenet_every_op_vs_live_reference(batch):
    """every int8 tensor against the reference CPU backend's own per-command dump of the same input (recorded digests)"""
    from mnn_b200.session import WholeNetSession
    g = np.load(os.path.join(GOLD, "reference_fullsize.npz"))
    x = refdump_input((batch, 3, 224, 224), 11)
    sess = WholeNetSession(MODEL, batch)
    sess.capture()                      # CUDA-graph replay is the product path
    sess.set_input(x)
    sess.run()
    _check_every_op(sess, g)


def test_wholenet_program_mode_every_op_vs_live_reference():
    """The same .mnn with its conv / depthwise / add chain fused into ONE cooperative launch (net program: dependency flags between
    tiles of consecutive layers): every checkpoint still equals the reference, twice in a row (flags are re-armed per launch)."""
    from mnn_b200.session import WholeNetSession
    batch = 2
    g = np.load(os.path.join(GOLD, "reference_fullsize.npz"))
    x = refdump_input((batch, 3, 224, 224), 11)
    sess = WholeNetSession(MODEL, batch, program=True)
    assert sess.programs and sess.launches_per_step <= 12, [s[0] for s in sess.steps]
    sess.capture()
    for rep in range(2):
        sess.set_input(x)
        sess.run()
        _check_every_op(sess, g, f"rep {rep} ")
