"""ctypes front-end for oracle/mnn_oracle.c and for the reference harness oracle/_ref/refdump.

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference leg.  mnn_b200 (the product) never imports this module.
"""
import ctypes as C
import hashlib
import os
import struct
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmnn_oracle.so")
REF_DIR = os.path.join(HERE, "_ref")
REFDUMP = os.path.join(REF_DIR, "refdump")
# the MNN_FORWARD_CUDA plugin (product code, mnn_b200/csrc/plugin) is compiled against the reference's headers, so it is built
# where the reference is and kept beside the core library that hosts it
PLUGIN = os.path.join(REF_DIR, "libmnn_b200_plugin.so")


def build(force=False):
    """Compile the C restatement.  -ffp-contract=off: the reference epilogues are unfused."""
    src = os.path.join(HERE, "mnn_oracle.c")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
                               "-fvisibility=hidden", src, "-o", LIB_PATH, "-lm"])
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(LIB_PATH)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def conv_out_size(i, k, s, p, d):
    return (i + 2 * p - (d * (k - 1) + 1)) // s + 1


def fold_modern(w, alpha, bias, s_in, z_in, s_out, z_out):
    w = np.ascontiguousarray(w, np.int8)
    oc = w.shape[0]
    kl = w.size // oc
    alpha = np.ascontiguousarray(alpha, np.float32)
    bias = None if bias is None else np.ascontiguousarray(bias, np.float32)
    bf = np.empty(oc, np.float32)
    sx = C.c_float()
    lib().mnn_oracle_fold_modern(_p(w, C.c_int8), oc, kl, _p(alpha, C.c_float), _p(bias, C.c_float),
                                 C.c_float(s_in), int(z_in), C.c_float(s_out), int(z_out),
                                 _p(bf, C.c_float), C.byref(sx))
    return bf, np.float32(sx.value)


def fold_legacy(w, scale, bias_i32):
    w = np.ascontiguousarray(w, np.int8)
    oc = w.shape[0]
    kl = w.size // oc
    scale = np.ascontiguousarray(scale, np.float32)
    bias_i32 = None if bias_i32 is None else np.ascontiguousarray(bias_i32, np.int32)
    bf = np.empty(oc, np.float32)
    sx = C.c_float()
    lib().mnn_oracle_fold_legacy(_p(w, C.c_int8), oc, kl, _p(scale, C.c_float), _p(bias_i32, C.c_int32),
                                 _p(bf, C.c_float), C.byref(sx))
    return bf, np.float32(sx.value)


def conv_int8(x, w, wscale, scale_x, bias_float, stride=(1, 1), pad=(0, 0), dilate=(1, 1),
              z_in=0, min_v=-127, max_v=127):
    """x [n,ic,ih,iw] int8, w [oc,ic,kh,kw] int8 -> y [n,oc,oh,ow] int8.  (h, w) ordered tuples."""
    x = np.ascontiguousarray(x, np.int8)
    w = np.ascontiguousarray(w, np.int8)
    stride, pad, dilate = [tuple(int(v) for v in t) for t in (stride, pad, dilate)]
    n, ic, ih, iw = x.shape
    oc, _, kh, kw = w.shape
    oh = conv_out_size(ih, kh, stride[0], pad[0], dilate[0])
    ow = conv_out_size(iw, kw, stride[1], pad[1], dilate[1])
    y = np.empty((n, oc, oh, ow), np.int8)
    wscale = np.ascontiguousarray(wscale, np.float32)
    bias_float = np.ascontiguousarray(bias_float, np.float32)
    lib().mnn_oracle_conv_int8(_p(x, C.c_int8), n, ic, ih, iw, _p(w, C.c_int8), oc, kh, kw,
                               stride[0], stride[1], pad[0], pad[1], dilate[0], dilate[1],
                               _p(wscale, C.c_float), C.c_float(float(scale_x)), _p(bias_float, C.c_float),
                               int(z_in), int(min_v), int(max_v), _p(y, C.c_int8), oh, ow)
    return y


def float_to_int8(x, scale, zero=0.0, min_v=-127, max_v=127):
    """Pipeline-inserted cast: scale is the tensor's quant scale (inverted like CPUCast.cpp:24)."""
    x = np.ascontiguousarray(x, np.float32)
    y = np.empty(x.shape, np.int8)
    L = lib()
    L.mnn_oracle_cast_inv_scale.restype = C.c_float
    inv = L.mnn_oracle_cast_inv_scale(C.c_float(scale))
    L.mnn_oracle_float_to_int8(_p(x, C.c_float), C.c_size_t(x.size), C.c_float(inv), C.c_float(zero),
                               int(min_v), int(max_v), _p(y, C.c_int8))
    return y


def int8_to_float(x, scale, zero=0.0):
    x = np.ascontiguousarray(x, np.int8)
    y = np.empty(x.shape, np.float32)
    lib().mnn_oracle_int8_to_float(_p(x, C.c_int8), C.c_size_t(x.size), C.c_float(scale), C.c_float(zero),
                                   _p(y, C.c_float))
    return y


def linear_w8_dynamic(x, wq, alpha, wzero=None, bias=None, relu=False, relu6=False):
    x = np.ascontiguousarray(x, np.float32)
    wq = np.ascontiguousarray(wq, np.int8)
    tokens, ic = x.shape
    oc = wq.shape[0]
    alpha = np.ascontiguousarray(alpha, np.float32)
    wzero = None if wzero is None else np.ascontiguousarray(wzero, np.float32)
    bias = None if bias is None else np.ascontiguousarray(bias, np.float32)
    y = np.empty((tokens, oc), np.float32)
    lib().mnn_oracle_linear_w8_dynamic(_p(x, C.c_float), tokens, ic, _p(wq, C.c_int8), oc, _p(alpha, C.c_float),
                                       _p(wzero, C.c_float), _p(bias, C.c_float), int(relu), int(relu6),
                                       _p(y, C.c_float))
    return y


def linear_w8_dynamic_blocks(x, wq, alpha, wzero=None, bias=None, blocks=1, relu=False, relu6=False):
    """K-blocked weight scales: alpha / wzero are [oc][blocks] (mnn_oracle.c: mnn_oracle_linear_w8_dynamic_blocks)."""
    x = np.ascontiguousarray(x, np.float32)
    wq = np.ascontiguousarray(wq, np.int8)
    tokens, ic = x.shape
    oc = wq.shape[0]
    assert ic % blocks == 0
    alpha = np.ascontiguousarray(alpha, np.float32).reshape(oc, blocks)
    wzero = None if wzero is None else np.ascontiguousarray(wzero, np.float32).reshape(oc, blocks)
    bias = None if bias is None else np.ascontiguousarray(bias, np.float32)
    y = np.empty((tokens, oc), np.float32)
    lib().mnn_oracle_linear_w8_dynamic_blocks(_p(x, C.c_float), tokens, ic, _p(wq, C.c_int8), oc, _p(alpha, C.c_float),
                                              _p(wzero, C.c_float), _p(bias, C.c_float), int(blocks), int(relu), int(relu6),
                                              _p(y, C.c_float))
    return y


def fold_depthwise(w, wscale, bias, s_in, z_in, s_out, z_out):
    w = np.ascontiguousarray(w, np.int8)
    c = w.shape[0]
    kl = w.size // c
    wscale = np.ascontiguousarray(wscale, np.float32)
    bias = None if bias is None else np.ascontiguousarray(bias, np.float32)
    scale = np.empty(c, np.float32)
    bi = np.empty(c, np.int32)
    lib().mnn_oracle_fold_depthwise(_p(w, C.c_int8), c, kl, _p(wscale, C.c_float), _p(bias, C.c_float),
                                    C.c_float(s_in), int(z_in), C.c_float(s_out), int(z_out),
                                    _p(scale, C.c_float), _p(bi, C.c_int32))
    return scale, bi


def depthwise_int8(x, w, scale, bias_i32, stride=(1, 1), pad=(0, 0), dilate=(1, 1), z_in=0, min_v=-127, max_v=127):
    x = np.ascontiguousarray(x, np.int8)
    w = np.ascontiguousarray(w, np.int8)
    n, c, ih, iw = x.shape
    kh, kw = w.shape[-2:]
    oh = conv_out_size(ih, kh, stride[0], pad[0], dilate[0])
    ow = conv_out_size(iw, kw, stride[1], pad[1], dilate[1])
    y = np.empty((n, c, oh, ow), np.int8)
    scale = np.ascontiguousarray(scale, np.float32)
    bias_i32 = np.ascontiguousarray(bias_i32, np.int32)
    lib().mnn_oracle_depthwise_int8(_p(x, C.c_int8), n, c, ih, iw, _p(w, C.c_int8), kh, kw, stride[0], stride[1],
                                    pad[0], pad[1], dilate[0], dilate[1], _p(scale, C.c_float),
                                    _p(bias_i32, C.c_int32), int(z_in), int(min_v), int(max_v), _p(y, C.c_int8),
                                    oh, ow)
    return y


def binary_add_int8(x0, q0, x1, q1, qo):
    """q* = (scale, zero, min, max)"""
    x0 = np.ascontiguousarray(x0, np.int8)
    x1 = np.ascontiguousarray(x1, np.int8)
    y = np.empty(x0.shape, np.int8)
    lib().mnn_oracle_binary_add_int8(_p(x0, C.c_int8), C.c_float(q0[0]), int(q0[1]), _p(x1, C.c_int8), C.c_float(q1[0]),
                                     int(q1[1]), C.c_size_t(x0.size), C.c_float(qo[0]), int(qo[1]), int(qo[2]), int(qo[3]),
                                     _p(y, C.c_int8))
    return y


def avgpool_int8_via_float(x, kernel, stride, pad, qi, qo, pad_type=1, count_type=0):
    x = np.ascontiguousarray(x, np.int8)
    n, c, ih, iw = x.shape
    kh, kw = kernel
    if pad_type == 2:
        oh, ow = -(-ih // stride[0]), -(-iw // stride[1])
    elif pad_type == 1:
        oh, ow = (ih - kh) // stride[0] + 1, (iw - kw) // stride[1] + 1
    else:
        oh, ow = -(-(ih + 2 * pad[0] - kh) // stride[0]) + 1, -(-(iw + 2 * pad[1] - kw) // stride[1]) + 1
    y = np.empty((n, c, oh, ow), np.int8)
    lib().mnn_oracle_avgpool_int8_via_float(_p(x, C.c_int8), n, c, ih, iw, kh, kw, stride[0], stride[1], pad[0], pad[1],
                                            int(pad_type), int(count_type), C.c_float(qi[0]), C.c_float(qi[1]),
                                            C.c_float(qo[0]), C.c_float(qo[1]), int(qo[2]), int(qo[3]), _p(y, C.c_int8), oh, ow)
    return y


def softmax_int8(x, qi, qo):
    x = np.ascontiguousarray(x, np.int8)
    rows, c = x.shape
    y = np.empty((rows, c), np.int8)
    lib().mnn_oracle_softmax_int8(_p(x, C.c_int8), rows, c, C.c_float(qi[0]), C.c_float(qi[1]), C.c_float(qo[0]),
                                  C.c_float(qo[1]), int(qo[2]), int(qo[3]), _p(y, C.c_int8))
    return y


# --------------------------------------------------------------------------------------------
# The real reference (oracle/_ref/refdump, built by oracle/build_ref.py).
# --------------------------------------------------------------------------------------------
def have_reference():
    return os.path.exists(REFDUMP) and os.path.exists(os.path.join(REF_DIR, "libMNN.so"))


def _run_refdump(args, timeout=600, exe=REFDUMP):
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = REF_DIR + ":" + env.get("LD_LIBRARY_PATH", "")
    return subprocess.run([exe] + [str(a) for a in args], env=env, capture_output=True, text=True,
                          timeout=timeout, check=True)


# Answers of the reference harness, recorded by tests/golden/make_golden.py and keyed by the request they answer, so that the
# comparisons with the reference hold on machines without the reference build (where it is built, it answers live).
RECORDED = os.path.join(os.path.dirname(HERE), "tests", "golden", "reference_calls.npz")
_recorded = None
recording = None     # make_golden.py sets a dict here: every answer of the live reference is kept in it under its request key


def _reference_answer(exe, args, payload):
    """The bytes `exe cmd req.bin out.bin *rest` writes for args = [cmd, *rest] and req.bin = payload: from the live reference when
    oracle/_ref holds it, else the answer recorded for the same request."""
    global _recorded
    key = hashlib.sha256(repr([os.path.basename(exe)] + [str(a) for a in args]).encode() + payload).hexdigest()[:32]
    if not os.path.exists(exe):
        if _recorded is None:
            _recorded = dict(np.load(RECORDED)) if os.path.exists(RECORDED) else {}
        if key in _recorded:
            return _recorded[key].tobytes()
        raise FileNotFoundError(f"no recorded reference answer for this '{args[0]}' request and {exe} is not built: "
                                "build the reference (oracle/build_ref.py) or re-record (tests/golden/make_golden.py calls)")
    with tempfile.TemporaryDirectory() as d:
        req, out = os.path.join(d, "req.bin"), os.path.join(d, "out.bin")
        with open(req, "wb") as f:
            f.write(payload)
        _run_refdump([args[0], req, out] + list(args[1:]), exe=exe)
        with open(out, "rb") as f:
            raw = f.read()
    if recording is not None:
        recording[key] = np.frombuffer(raw, np.uint8)
    return raw


def ref_conv(mode, x, w, bias, scale, stride=(1, 1), pad=(0, 0), dilate=(1, 1), group=1, relu=False,
             z_in=0, z_out=0, min_v=-127, max_v=127, scale_in=0.0, scale_out=0.0):
    """Run ONE ConvInt8/DepthwiseConvInt8 op through the reference CPU backend.
    mode 0: legacy (bias int32, scale = fused multiplier); mode 1: modern (bias float, scale = weight scale)."""
    x = np.ascontiguousarray(x, np.int8)
    w = np.ascontiguousarray(w, np.int8)
    n, ic, ih, iw = x.shape
    oc, kh, kw = w.shape[0], w.shape[-2], w.shape[-1]
    hdr = struct.pack("<20i2f", mode, n, ic, ih, iw, oc, kh, kw, stride[0], stride[1], pad[0], pad[1],
                      dilate[0], dilate[1], group, int(relu), z_in, z_out, min_v, max_v, scale_in, scale_out)
    b = np.ascontiguousarray(bias, np.int32 if mode == 0 else np.float32)
    s = np.ascontiguousarray(scale, np.float32)
    raw = _reference_answer(REFDUMP, ["conv"], hdr + x.tobytes() + w.tobytes() + b.tobytes() + s.tobytes())
    dims = struct.unpack("<4i", raw[:16])
    return np.frombuffer(raw[16:], np.int8).reshape(dims).copy()


def ref_linear(x, wq, alpha, asym=False, bias=None, relu=False, relu6=False, threads=1, blocks=1):
    """alpha: [oc * blocks] scales (or {min, scale} pairs when asym), K split into `blocks` equal runs per output channel."""
    x = np.ascontiguousarray(x, np.float32)
    wq = np.ascontiguousarray(wq, np.int8)
    tokens, ic = x.shape
    oc = wq.shape[0]
    hdr = struct.pack("<8i", tokens, ic, oc, int(asym), int(relu), int(relu6), int(bias is not None), int(blocks) if blocks > 1 else 0)
    payload = hdr + x.tobytes() + wq.tobytes() + np.ascontiguousarray(alpha, np.float32).tobytes()
    if bias is not None:
        payload += np.ascontiguousarray(bias, np.float32).tobytes()
    return np.frombuffer(_reference_answer(REFDUMP, ["linear", threads], payload), np.float32).reshape(tokens, oc).copy()


def ref_run_model(model, batch, seed, outdir, threads=1):
    os.makedirs(outdir, exist_ok=True)
    _run_refdump(["run", model, batch, seed, outdir, threads], timeout=3600)
    recs = []
    for line in open(os.path.join(outdir, "index.txt")):
        f, name, typ, dims, qs, qz, qmin, qmax, aq = line.rstrip("\n").split("|")
        recs.append(dict(file=f, name=name, type=typ, dims=[int(v) for v in dims.split(",")] if dims else [],
                         scale=float(qs), zero=float(qz), min=float(qmin), max=float(qmax), apply_quant=int(aq)))
    return recs


def ref_bench(model, batch, threads, warmup, iters):
    import json
    r = _run_refdump(["bench", model, batch, threads, warmup, iters], timeout=3600)
    return json.loads(r.stdout.strip().splitlines()[-1])


# --------------------------------------------------------------------------------------------
# int8 Winograd (SURVEY a5).  Oracle = mnn_oracle_wino_conv_int8; real reference = refdump_avx2
# (the AVX2 build: the AVX512 build of ConvInt8Winograd is wrong upstream, SURVEY F8).
# --------------------------------------------------------------------------------------------
REFDUMP_AVX2 = os.path.join(REF_DIR, "refdump_avx2")


def have_reference_avx2():
    return os.path.exists(REFDUMP_AVX2) and os.path.exists(os.path.join(REF_DIR, "libMNN_avx2.so"))


def _wino_args(x, w, wscale, bias, in_scales, in_zeros, w_scales, unit):
    x = np.ascontiguousarray(x, np.int8)
    w = np.ascontiguousarray(w, np.int8)
    oc, ic, r = w.shape[0], w.shape[1], w.shape[2]
    a2 = (unit + r - 1) ** 2
    wscale = np.ascontiguousarray(wscale, np.float32)
    bias = np.ascontiguousarray(bias if bias is not None else np.zeros(oc), np.float32)
    in_scales = np.ascontiguousarray(np.broadcast_to(np.asarray(in_scales, np.float32), (a2,)))
    in_zeros = np.ascontiguousarray(np.broadcast_to(np.asarray(in_zeros, np.int32), (a2,)))
    w_scales = np.ascontiguousarray(np.broadcast_to(np.asarray(w_scales, np.float32).reshape(-1, oc) if np.ndim(w_scales) else
                                                    np.asarray(w_scales, np.float32), (a2, oc)))
    return x, w, wscale, bias, in_scales, in_zeros, w_scales


def wino_weights(w, wscale, in_scales, in_zeros, w_scales, unit):
    w = np.ascontiguousarray(w, np.int8)
    oc, ic, r = w.shape[0], w.shape[1], w.shape[2]
    _, w, wscale, _, in_scales, in_zeros, w_scales = _wino_args(np.zeros(1, np.int8), w, wscale, None, in_scales, in_zeros,
                                                                w_scales, unit)
    a2 = (unit + r - 1) ** 2
    wq = np.empty((a2, oc, ic), np.int8)
    sc = np.empty((a2, oc), np.float32)
    of = np.empty((a2, oc), np.float32)
    lib().mnn_oracle_wino_weights(_p(w, C.c_int8), oc, ic, r, unit, _p(wscale, C.c_float), _p(in_scales, C.c_float),
                                  _p(in_zeros, C.c_int32), _p(w_scales, C.c_float), _p(wq, C.c_int8), _p(sc, C.c_float),
                                  _p(of, C.c_float))
    return wq, sc, of


def wino_conv_int8(x, w, wscale, bias, in_scales, in_zeros, w_scales, unit, pad=1, s_in=1.0, z_in=0, s_out=1.0, z_out=0,
                   clamp_min=-127, clamp_max=127, relu=False):
    x, w, wscale, bias, in_scales, in_zeros, w_scales = _wino_args(x, w, wscale, bias, in_scales, in_zeros, w_scales, unit)
    n, ic, ih, iw = x.shape
    oc, r = w.shape[0], w.shape[2]
    oh, ow = ih + 2 * pad - r + 1, iw + 2 * pad - r + 1
    y = np.empty((n, oc, oh, ow), np.int8)
    lib().mnn_oracle_wino_conv_int8(_p(x, C.c_int8), n, ic, ih, iw, _p(w, C.c_int8), oc, r, pad, pad, unit,
                                    _p(wscale, C.c_float), _p(bias, C.c_float), _p(in_scales, C.c_float),
                                    _p(in_zeros, C.c_int32), _p(w_scales, C.c_float), C.c_float(s_in), int(z_in),
                                    C.c_float(s_out), int(z_out), int(clamp_min), int(clamp_max), int(relu), _p(y, C.c_int8))
    return y


def ref_wino(x, w, wscale, bias, in_scales, in_zeros, w_scales, unit, pad=1, s_in=1.0, z_in=0, s_out=1.0, z_out=0,
             clamp_min=-127, clamp_max=127, relu=False):
    """ONE ConvInt8 op with a winogradAttr through the reference CPU backend (AVX2 build)."""
    x, w, wscale, bias, in_scales, in_zeros, w_scales = _wino_args(x, w, wscale, bias, in_scales, in_zeros, w_scales, unit)
    n, ic, ih, iw = x.shape
    oc, r = w.shape[0], w.shape[2]
    hdr = struct.pack("<13i2f", n, ic, ih, iw, oc, r, pad, unit, int(relu), z_in, z_out, clamp_min, clamp_max, s_in, s_out)
    payload = hdr + x.tobytes() + w.tobytes() + bias.tobytes() + wscale.tobytes() + in_scales.tobytes() + \
        in_zeros.tobytes() + w_scales.tobytes()
    raw = _reference_answer(REFDUMP_AVX2, ["wino"], payload)
    dims = struct.unpack("<4i", raw[:16])
    return np.frombuffer(raw[16:], np.int8).reshape(dims).copy()


def wino_matrices(unit, r=3):
    alpha = unit + r - 1
    bt = np.empty((alpha, alpha), np.float32)
    at = np.empty((unit, alpha), np.float32)
    g = np.empty((alpha, r), np.float32)
    lib().mnn_oracle_wino_matrices(unit, r, _p(bt, C.c_float), _p(at, C.c_float), _p(g, C.c_float))
    return bt, at, g


# --------------------------------------------------------------------------------------------
# float MatMul / BatchMatMul (SURVEY a9).  CPUMatMul / CPUBatchMatMul compute C = op(A) op(B) in fp32
# (source/backend/cpu/CPUMatMul.cpp, compute/CommonOptFunction MNNPackedMatMul); the restatement is a plain fp32
# numpy matmul -- summation order differs from the packed kernels, so it is pinned to the reference at 1e-5 relative
# (tests/test_matmul.py) and the GPU path is held to BASELINE's 1e-3.
# --------------------------------------------------------------------------------------------
def matmul_f32(a, b, transpose_a=False, transpose_b=False, bias=None):
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    if transpose_a:
        a = np.swapaxes(a, -1, -2)
    if transpose_b:
        b = np.swapaxes(b, -1, -2)
    c = np.matmul(a, b, dtype=np.float32)
    if bias is not None:
        c = c + np.asarray(bias, np.float32)
    return c.astype(np.float32)


def ref_matmul(a, b, transpose_a=False, transpose_b=False):
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    a3 = a.reshape((-1,) + a.shape[-2:])
    b3 = b.reshape((-1,) + b.shape[-2:])
    batch = a3.shape[0]
    e, l = (a3.shape[2], a3.shape[1]) if transpose_a else (a3.shape[1], a3.shape[2])
    h = b3.shape[1] if transpose_b else b3.shape[2]
    hdr = struct.pack("<8i", batch, e, l, h, int(transpose_a), int(transpose_b), 0, 0)
    raw = _reference_answer(REFDUMP, ["matmul"], hdr + a3.tobytes() + b3.tobytes())
    return np.frombuffer(raw, np.float32).reshape(a.shape[:-2] + (e, h)).copy()


# --------------------------------------------------------------------------------------------
# int8 pooling with equal in/out quant attrs (next-round row: the CPU keeps it in int8).
# --------------------------------------------------------------------------------------------
def pool_int8_x86(x, kernel, stride, pad, is_avg):
    x = np.ascontiguousarray(x, np.int8)
    n, c, ih, iw = x.shape
    (kh, kw), (sh, sw), (ph, pw) = kernel, stride, pad
    oh, ow = (ih + 2 * ph - kh) // sh + 1, (iw + 2 * pw - kw) // sw + 1
    y = np.empty((n, c, oh, ow), np.int8)
    lib().mnn_oracle_pool_int8_x86(_p(x, C.c_int8), n, c, ih, iw, kh, kw, sh, sw, ph, pw, int(is_avg), _p(y, C.c_int8), oh, ow)
    return y


def ref_pool_int8(x, kernel, stride, pad, is_avg, scale=0.05, zero=0):
    x = np.ascontiguousarray(x, np.int8)
    n, c, ih, iw = x.shape
    hdr = struct.pack("<12if", n, c, ih, iw, kernel[0], kernel[1], stride[0], stride[1], pad[0], pad[1], int(is_avg), int(zero), scale)
    raw = _reference_answer(REFDUMP, ["pool"], hdr + x.tobytes())
    dims = struct.unpack("<4i", raw[:16])
    return np.frombuffer(raw[16:], np.int8).reshape(dims).copy()


# --------------------------------------------------------------------------------------------
# int8 Scale: CPUScaleInt8::onResize + MNNScaleAndAddBiasInt8 (source/backend/cpu/CPUScaleInt8.cpp:60-90,
# compute/Int8FunctionsOpt.cpp:2207-2252), integer arithmetic restated in numpy (test infrastructure only).
# --------------------------------------------------------------------------------------------
def scale_int8(x, scale, bias, s_in, z_in, s_out, z_out, min_v=-127, max_v=127):
    x = np.ascontiguousarray(x, np.int8)
    c = x.shape[1]
    f32 = np.float32
    inv_out = f32(0) if s_out == 0 else f32(1) / f32(s_out)
    sc = np.asarray(scale, f32)
    bi = np.zeros(c, f32) if bias is None else np.asarray(bias, f32)
    t = (sc * f32(s_in)).astype(f32)
    t = (t * inv_out).astype(f32)
    t = (t * f32(1 << 15)).astype(f32)
    alpha = np.where(t >= 0, np.floor(t.astype(np.float64) + 0.5), np.ceil(t.astype(np.float64) - 0.5)).astype(np.int64)   # roundf
    b = ((bi * inv_out).astype(f32) * f32(1 << 15)).astype(f32)
    beta = np.where(b >= 0, np.floor(b.astype(np.float64) + 0.5), np.ceil(b.astype(np.float64) - 0.5)).astype(np.int64)
    sh = (1, c) + (1,) * (x.ndim - 2)
    val = (x.astype(np.int64) - int(np.int8(z_in))) * alpha.reshape(sh) + beta.reshape(sh)
    val = val.astype(np.int32).astype(np.int64)                      # the reference computes in int32
    adj = np.where(val < 0, val - (1 << 14), val + (1 << 14))
    q = np.where(adj < 0, -((-adj) >> 15), adj >> 15)               # C integer division truncates toward zero
    out = q + int(np.int8(z_out))
    return np.clip(out, min_v, max_v).astype(np.int8)
