"""Parity AT THE BENCH CONFIGS THEMSELVES (-m gpu; round-1 VERDICT weak #1): the sizes BASELINE.json's configs name, checked
against what the reference produced for them (digests and samples in tests/golden/reference_fullsize.npz, recorded by
tests/golden/make_golden.py) -- not smaller stand-ins.  The plugin checks need the reference core under oracle/_ref as host.

  C2  MobileNet-v2 int8 .mnn, batch 32: every command's int8 output, plugin vs MNN_FORWARD_CPU and WholeNetSession vs
      MNN_FORWARD_CPU (position-weighted 64-bit sums of the dequantised tensors: REFDUMP_HASH=1, oracle/refdump.cpp)
  C3  ResNet-50 3x3/s1 layers at batch 64 on int8 Winograd F(6,3): C=64/56x56 and C=512/7x7 vs the AVX2 reference build
  C4  Qwen-1.8B linear shapes at 4096 tokens: 2048->6144 (+bias, asymmetric) and 5504->2048 vs `refdump linear`
  +   a .mnn whose Convolution carries a winogradAttr through the PLUGIN (reference AVX2 core + libmnn_b200_plugin.so)
"""
import hashlib
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
from tests.cases import random_wino_case, refdump_input

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGIN = O.PLUGIN
MODEL = os.path.join(ROOT, "tests", "golden", "mbv2_int8.mnn")
FULLSIZE = os.path.join(ROOT, "tests", "golden", "reference_fullsize.npz")
FP_INTERNAL = ("MobilenetV2/Predictions/Softmax",)      # expf vs the reference's polynomial: +-1 LSB (documented in DESIGN.md)
needs_ref2 = pytest.mark.skipif(not O.have_reference_avx2(), reason="oracle/_ref/refdump_avx2 not on this box")


def wsum64(a: np.ndarray) -> int:
    """the hash refdump prints under REFDUMP_HASH=1: sum_k word[k] * (k * 0x9E3779B97F4A7C15 + 1) mod 2^64 over the fp32 words"""
    w = np.ascontiguousarray(a, np.float32).view(np.uint32).ravel().astype(np.uint64)
    k = np.arange(w.size, dtype=np.uint64)
    with np.errstate(over="ignore"):
        return int((w * (k * np.uint64(0x9E3779B97F4A7C15) + np.uint64(1))).sum(dtype=np.uint64))


def _refdump_run(exe, libdir, model, batch, seed, outdir, threads, plugin, hash_only=True):
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = libdir + ":" + os.path.join(ROOT, "mnn_b200") + ":" + env.get("LD_LIBRARY_PATH", "")
    env["REFDUMP_HASH"] = "1" if hash_only else "0"
    if plugin:
        env["REFDUMP_PLUGIN"] = PLUGIN
    else:
        env.pop("REFDUMP_PLUGIN", None)
    os.makedirs(outdir, exist_ok=True)
    r = subprocess.run([exe, "run", model, str(batch), str(seed), outdir, str(threads)], env=env, capture_output=True, text=True,
                       timeout=1800)
    assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-500:]
    recs = []
    for line in open(os.path.join(outdir, "index.txt")):
        f, name, typ, dims, qs, qz, qmin, qmax, aq = line.rstrip("\n").split("|")
        recs.append(dict(file=f, name=name, type=typ.strip(), dims=[int(v) for v in dims.split(",")] if dims else [],
                         scale=float(qs), zero=float(qz), apply_quant=int(aq)))
    stats = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{\"plugin_")]
    return recs, (stats[-1] if stats else None)


def _diagnose(d, batch, threads, ncmd):
    """a hash mismatch says nothing about how many values differ: re-run both sides up to the failing command with full dumps"""
    os.environ["REFDUMP_MAX_COMMANDS"] = str(ncmd)
    try:
        cpu, _ = _refdump_run(O.REFDUMP, O.REF_DIR, MODEL, batch, 5, os.path.join(d, "dcpu"), threads, False, hash_only=False)
        gpu, _ = _refdump_run(O.REFDUMP, O.REF_DIR, MODEL, batch, 5, os.path.join(d, "dgpu"), 4, True, hash_only=False)
    finally:
        os.environ.pop("REFDUMP_MAX_COMMANDS", None)
    a = np.fromfile(os.path.join(d, "dcpu", cpu[ncmd - 1]["file"]), np.float32)
    b = np.fromfile(os.path.join(d, "dgpu", gpu[ncmd - 1]["file"]), np.float32)
    xa = np.fromfile(os.path.join(d, "dcpu", "input.f32"), np.float32)
    xb = np.fromfile(os.path.join(d, "dgpu", "input.f32"), np.float32)
    bad = np.flatnonzero(a != b)
    signed_zero = int(np.count_nonzero((a == b) & (np.signbit(a) != np.signbit(b))))
    return (f"inputs equal: {np.array_equal(xa, xb)}; {bad.size} of {a.size} values differ (first at {bad[:5].tolist()}, "
            f"cpu {a[bad[:5]].tolist()} vs plugin {b[bad[:5]].tolist()}), max |diff| {np.abs(a - b).max() if bad.size else 0}; "
            f"{signed_zero} equal values with different zero sign")


def test_c2_mbv2_batch32_every_op_plugin_and_session_vs_cpu_backend():
    """BASELINE configs[1] at its own batch: the WholeNetSession host, and (with the reference core present) the unmodified
    reference pipeline on the plugin, both against MNN_FORWARD_CPU on the same 32 x 3 x 224 x 224 input; every int8 tensor
    bit-exact (softmax +-1 LSB excluded)."""
    from mnn_b200.session import WholeNetSession
    batch = 32
    threads = min(os.cpu_count() or 1, 32)
    g = np.load(FULLSIZE)
    cpu = [dict(name=str(n), type=str(t), file=str(h), dims=[int(v) for v in str(dm).split(",")], scale=float(sc), zero=float(z),
                apply_quant=int(aq))
           for n, t, h, dm, sc, z, aq in zip(*(g["c2_" + k] for k in ("names", "types", "hashes", "dims", "scales", "zeros",
                                                                     "apply_quant")))]
    with tempfile.TemporaryDirectory() as d:
        if O.have_reference():
            assert os.path.exists(PLUGIN), "oracle/_ref/libmnn_b200_plugin.so is missing although the reference core is present"
            gpu, stats = _refdump_run(O.REFDUMP, O.REF_DIR, MODEL, batch, 5, os.path.join(d, "gpu"), 4, True)
            assert stats is not None and stats["plugin_declined"] == 0, stats
            assert [(r["name"], r["type"]) for r in cpu] == [(r["name"], r["type"]) for r in gpu]
            n_int8 = 0
            for idx, (a, b) in enumerate(zip(cpu, gpu)):
                if a["apply_quant"] and a["name"] not in FP_INTERNAL:
                    if a["file"] != b["file"]:
                        raise AssertionError(f"plugin vs CPU backend differ at batch 32: {a['name']} ({a['type']}): " +
                                             _diagnose(d, batch, threads, idx + 1))
                    n_int8 += 1
            assert n_int8 >= 60, n_int8
        # the C-ABI host on the same input
        x = refdump_input((batch, 3, 224, 224), 5)
        sess = WholeNetSession(MODEL, batch)
        sess.capture()
        sess.set_input(x)
        sess.run()
        checked = 0
        for r in cpu:
            if r["name"] not in sess.checkpoints or r["scale"] <= 0 or not r["apply_quant"] or r["name"] in FP_INTERNAL:
                continue
            q = sess.read_int8(r["name"]).reshape(r["dims"])
            f = (q.astype(np.float32) - np.float32(r["zero"])) * np.float32(r["scale"])       # MNNInt8ScaleToFloat
            assert r["file"] == "hash:%016x" % wsum64(f), f"WholeNetSession vs CPU backend differ at batch 32: {r['name']}"
            checked += 1
        assert checked >= 60, checked
        # ... and the same forward with the conv / depthwise / add chain fused into ONE cooperative launch (net program)
        prog = WholeNetSession(MODEL, batch, program=True)
        assert prog.programs and prog.launches_per_step <= 12
        prog.capture()
        prog.set_input(x)
        prog.run()
        for name in sess.checkpoints:
            a, b = sess.read_int8(name), prog.read_int8(name)
            assert np.array_equal(a, b), f"net program vs per-op kernels differ at batch 32: {name}: {np.count_nonzero(a != b)} values"


@pytest.mark.parametrize("C_,HW", [(64, 56), (512, 7)])
def test_c3_resnet_f63_batch64_vs_live_reference(backend, C_, HW):
    """BASELINE configs[2]: ResNet-50 3x3/s1, batch 64, int8 Winograd F(6,3) -- the first and the last layer class, full size,
    bit-exact against the reference's AVX2 build (ConvInt8Winograd): the sha256 of its int8 output, recorded by make_golden.py."""
    from tests.test_winograd import run_wino
    rng = np.random.default_rng(C_ + HW)
    c = random_wino_case(rng, 6, 64, C_, C_, HW, HW, 1, True)
    y, ex = run_wino(backend, c, 6)
    assert y.shape == (64, C_, HW, HW)
    y = np.ascontiguousarray(y, np.int8)
    assert hashlib.sha256(y.tobytes()).hexdigest() == str(np.load(FULLSIZE)[f"c3_{C_}_{HW}_sha256"]), "differs from the reference"
    assert (np.abs(y.astype(int)) == 127).mean() < 0.5
    assert ex.cost()[1] == 64.0 * HW * HW * C_ * C_ * 9


@pytest.mark.parametrize("ic,oc,asym,has_bias", [(2048, 6144, True, True), (5504, 2048, True, False)])
def test_c4_qwen_linear_4096_tokens_vs_live_reference(backend, ic, oc, asym, has_bias):
    """BASELINE configs[3]: the two extreme Qwen-1.8B linear shapes at the full 4096 tokens against the reference CPU backend's
    dynamic-quant W8A8 (`refdump linear`, Memory_Low), 1e-3 relative (north_star); both product kernels (single CTA / CTA pair).
    The reference output is recorded as max |y| and its values at c4_sample_positions (every row and every column several times,
    plus random positions); every output must be written."""
    from mnn_b200.backend import Op, Tensor
    import torch
    T = 4096
    x, wq, alpha, wmin, bias = c4_case(T, ic, oc, asym, has_bias)
    g = np.load(FULLSIZE)
    ref, ref_absmax = g[f"c4_{ic}_{oc}_sample"], float(g[f"c4_{ic}_{oc}_absmax"])
    at = c4_sample_positions(T, oc)
    # the reference is fed the wire form {min, scale} (make_golden.py); the C ABI takes the offset of SIGNED int8 weights (see _signed_offset)
    from mnn_b200 import _capi
    for variant in (2, 3):
        op = Op(type="LinearW8", conv=dict(ic=ic, oc=oc), weight=wq, wscale=alpha,
                wzero=None if wmin is None else _signed_offset(wmin, alpha), bias=bias)
        xt = Tensor((T, ic), "float", None, torch.from_numpy(x).cuda())
        yt = Tensor((T, oc), "float", None, torch.full((T, oc), float("nan"), dtype=torch.float32, device="cuda"))
        ex = backend.onCreate([xt], [yt], op)
        _capi.check(_capi.lib().mnnb200_conv_int8_set_variant(ex._h, variant))
        assert ex.onResize([xt], [yt]) == 0
        assert ex.onExecute([xt], [yt]) == 0
        backend.onSync()
        y = yt.data.cpu().numpy()
        assert not np.isnan(y).any(), f"variant {variant}: outputs left unwritten"
        err = np.abs(y.ravel()[at] - ref).max() / ref_absmax
        assert err <= 1e-3, f"variant {variant}: rel err {err}"


C4_PER_ROW = 16
C4_RANDOM = 16384


def c4_case(tokens, ic, oc, asym, has_bias):
    rng = np.random.default_rng(ic + oc)
    x = rng.uniform(-1, 1, (tokens, ic)).astype(np.float32)
    wq = rng.integers(-128, 128, (oc, ic), dtype=np.int8)
    alpha = rng.uniform(0.001, 0.01, oc).astype(np.float32)
    wmin = (alpha * rng.uniform(-8, 8, oc)).astype(np.float32) if asym else None
    bias = rng.uniform(-1, 1, oc).astype(np.float32) if has_bias else None
    return x, wq, alpha, wmin, bias


def c4_sample_positions(tokens, oc):
    """flat positions of the recorded reference values: C4_PER_ROW in every row, spread so that every column is hit at least
    tokens * C4_PER_ROW // oc times (an error confined to one row or one column cannot be missed), plus C4_RANDOM random ones"""
    t = np.arange(tokens)[:, None]
    cols = (t + np.arange(C4_PER_ROW)[None, :] * (oc // C4_PER_ROW)) % oc
    rand = np.random.default_rng(tokens + oc).integers(0, tokens * oc, C4_RANDOM)
    return np.concatenate([(t * oc + cols).ravel(), rand])


def _signed_offset(wmin, alpha):
    """ConvolutionCommon::load turns the wire 'min' into the offset of SIGNED int8 weights: min - clampMin * scale with
    clampMin = -128 (source/core/ConvolutionCommon.cpp:757-766)."""
    return (wmin - np.float32(-128.0) * alpha).astype(np.float32)


@needs_ref2
def test_winograd_attr_mnn_through_the_plugin():
    """INTEGRATION.md gap of round 1: a converted .mnn whose Convolution carries a winogradAttr, scheduled by the UNMODIFIED
    reference core (AVX2 build, the one whose ConvInt8Winograd is right) on MNN_FORWARD_CUDA = the plugin, equals the same
    process's MNN_FORWARD_CPU result bit for bit, with nothing declined."""
    assert os.path.exists(PLUGIN), "oracle/_ref/libmnn_b200_plugin.so is missing although the reference core is present"
    model = os.path.join(ROOT, "tests", "golden", "wino_modern_conv.mnn")
    with tempfile.TemporaryDirectory() as d:
        cpu, _ = _refdump_run(O.REFDUMP_AVX2, O.REF_DIR, model, 2, 9, os.path.join(d, "cpu"), 1, False, hash_only=False)
        gpu, stats = _refdump_run(O.REFDUMP_AVX2, O.REF_DIR, model, 2, 9, os.path.join(d, "gpu"), 1, True, hash_only=False)
        assert stats is not None and stats["plugin_declined"] == 0 and stats["plugin_created"] >= 1, stats
        assert [(r["name"], r["type"]) for r in cpu] == [(r["name"], r["type"]) for r in gpu]
        convs = 0
        for a, b in zip(cpu, gpu):
            fa = np.fromfile(os.path.join(d, "cpu", a["file"]), np.float32)
            fb = np.fromfile(os.path.join(d, "gpu", b["file"]), np.float32)
            if a["apply_quant"]:
                assert np.array_equal(fa, fb), f"{a['name']} ({a['type']}): {np.count_nonzero(fa != fb)} of {fa.size} differ"
                convs += "Convolution" in a["type"]
            else:
                assert np.abs(fa - fb).max() <= 1e-3 * max(np.abs(fa).max(), 1e-12)
        assert convs >= 1
