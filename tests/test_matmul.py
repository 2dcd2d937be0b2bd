"""Float MatMul / BatchMatMul (SURVEY a9): oracle pinned on the reference CPU backend and on a committed fixture; the
tcgen05 kind::f16 path (-m gpu) within BASELINE's 1e-3 (max|d| / max|ref|)."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.cases import load_golden

# (batch dims, e, l, h, transpose_a, transpose_b): attention QK^T / PV of Qwen-1.8B (16 heads x 128), plus ragged shapes
CASES = [((2, 4), 64, 128, 64, False, True), ((3,), 64, 64, 128, False, False), ((), 37, 53, 29, False, False),
         ((), 40, 24, 56, True, False), ((2,), 33, 72, 17, True, True), ((), 1, 200, 300, False, True)]


def make(rng, bd, e, l, h, ta, tb, positive=False):
    sa = bd + ((l, e) if ta else (e, l))
    sb = bd + ((h, l) if tb else (l, h))
    a = rng.uniform(0 if positive else -1, 1, sa).astype(np.float32)
    b = rng.uniform(-1, 1, sb).astype(np.float32)
    return a, b


def test_oracle_vs_golden_fixture():
    g = load_golden("matmul_golden")
    for i in range(int(g["ncase"])):
        y = O.matmul_f32(g[f"m{i}_a"], g[f"m{i}_b"], bool(g[f"m{i}_ta"]), bool(g[f"m{i}_tb"]))
        ref = g[f"m{i}_y"]
        assert y.shape == ref.shape and np.abs(y - ref).max() <= 1e-5 * np.abs(ref).max()


def test_oracle_vs_live_reference():
    rng = np.random.default_rng(3)
    for bd, e, l, h, ta, tb in CASES[:4]:
        a, b = make(rng, bd, e, l, h, ta, tb)
        ref = O.ref_matmul(a, b, ta, tb)
        assert np.abs(O.matmul_f32(a, b, ta, tb) - ref).max() <= 1e-5 * np.abs(ref).max()


def run_matmul(backend, a, b, ta, tb, bias=None):
    import torch
    from mnn_b200.backend import Op, Tensor
    dev = backend.runtime.device
    ta_ = Tensor(a.shape, "float", None, torch.from_numpy(a).to(dev))
    tb_ = Tensor(b.shape, "float", None, torch.from_numpy(b).to(dev))
    y = Tensor((1,), "float")
    ex = backend.onCreate([ta_, tb_], [y], Op(type="BatchMatMul" if a.ndim > 2 else "MatMul", bias=bias,
                                              extra=dict(transpose_a=ta, transpose_b=tb)))
    assert ex is not None and ex.onResize([ta_, tb_], [y]) == 0
    backend.onAcquire(y)
    y.data.fill_(float("nan"))
    assert ex.onExecute([ta_, tb_], [y]) == 0
    backend.onSync()
    return y.data.cpu().numpy()


@pytest.mark.gpu
def test_gpu_vs_golden_and_oracle(backend):
    g = load_golden("matmul_golden")
    for i in range(int(g["ncase"])):
        y = run_matmul(backend, g[f"m{i}_a"], g[f"m{i}_b"], bool(g[f"m{i}_ta"]), bool(g[f"m{i}_tb"]))
        ref = g[f"m{i}_y"]
        assert y.shape == ref.shape and not np.isnan(y).any()
        assert np.abs(y - ref).max() <= 1e-3 * np.abs(ref).max(), f"case {i}: {np.abs(y - ref).max() / np.abs(ref).max()}"


@pytest.mark.gpu
@pytest.mark.parametrize("bd,e,l,h,ta,tb", [((8, 16), 512, 128, 512, False, True), ((8, 16), 512, 512, 128, False, False),
                                            ((), 300, 1000, 260, False, False), ((2,), 130, 520, 40, True, True)])
def test_gpu_attention_shapes_vs_oracle(backend, bd, e, l, h, ta, tb):
    """BASELINE configs[3] attention BMM shapes (8 x 16 heads: [512,128]x[128,512] and [512,512]x[512,128]); the second
    with a non-negative left operand (softmax probabilities), the worst case for one-sided rounding."""
    rng = np.random.default_rng(e + l)
    a, b = make(rng, bd, e, l, h, ta, tb, positive=(l == 512))
    bias = rng.uniform(-1, 1, h).astype(np.float32) if not bd else None
    y = run_matmul(backend, a, b, ta, tb, bias)
    ref = O.matmul_f32(a, b, ta, tb, bias)
    assert np.abs(y - ref).max() <= 1e-3 * np.abs(ref).max(), np.abs(y - ref).max() / np.abs(ref).max()
