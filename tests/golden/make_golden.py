"""Generates tests/golden/*.npz by running the UNMODIFIED reference CPU backend (oracle/_ref/refdump,
built from /root/reference by oracle/build_ref.py).  Run in the build container:  python tests/golden/make_golden.py
The fixtures are committed so the GPU box (no /root/reference, possibly no oracle/_ref) still has real-reference vectors.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
from tests.cases import DW_CASES, KAT_SWEEP, LINEAR_CASES, dw_linear_inputs, kat_conv, matmul_inputs, random_modern_case, refdump_input  # noqa: E402,E501

HERE = os.path.dirname(os.path.abspath(__file__))


def conv_golden():
    out = {}
    i = 0
    for case in KAT_SWEEP:
        (ic, oc), (kh, kw), n, pad, stride, dilate, (ih, iw) = case
        x, w, bias, scale = kat_conv(n, ic, ih, iw, oc, kh, kw)
        y = O.ref_conv(0, x, w, bias, scale, stride=stride, pad=pad, dilate=dilate)
        out.update({f"c{i}_mode": 0, f"c{i}_x": x, f"c{i}_w": w, f"c{i}_bias": bias, f"c{i}_scale": scale,
                    f"c{i}_stride": stride, f"c{i}_pad": pad, f"c{i}_dilate": dilate, f"c{i}_y": y,
                    f"c{i}_relu": 0, f"c{i}_s_in": 0.0, f"c{i}_s_out": 0.0, f"c{i}_z_in": 0, f"c{i}_z_out": 0})
        i += 1
    rng = np.random.default_rng(2024)
    for (ic, oc, kh, kw, n, ih, iw, st, pad, relu, dl) in [
            (3, 32, 3, 3, 2, 16, 16, (2, 2), (1, 1), 1, (1, 1)),      # MobileNet-v2 stem shape class
            (32, 16, 1, 1, 2, 14, 14, (1, 1), (0, 0), 0, (1, 1)),     # pointwise projection (no relu)
            (16, 96, 1, 1, 1, 14, 14, (1, 1), (0, 0), 1, (1, 1)),     # pointwise expansion
            (96, 24, 1, 1, 3, 7, 7, (1, 1), (0, 0), 0, (1, 1)),
            (160, 40, 1, 1, 2, 7, 7, (1, 1), (0, 0), 1, (1, 1)),      # ragged oc (not a multiple of 16)
            (24, 20, 3, 3, 1, 9, 11, (1, 1), (1, 1), 1, (2, 2)),      # dilation + pad with non-zero zero point
            (64, 64, 3, 3, 1, 8, 8, (1, 1), (1, 1), 1, (1, 1)),       # ResNet 3x3 class
            (20, 10, 7, 1, 2, 12, 5, (2, 1), (3, 0), 0, (1, 1))]:     # asymmetric kernel
        c = random_modern_case(rng, ic, oc, kh, kw, n, ih, iw, st, pad, relu, dl)
        y = O.ref_conv(1, c["x"], c["w"], c["bias"], c["ws"], stride=st, pad=pad, dilate=dl, relu=relu,
                       z_in=c["z_in"], z_out=c["z_out"], scale_in=c["s_in"], scale_out=c["s_out"])
        out.update({f"c{i}_mode": 1, f"c{i}_x": c["x"], f"c{i}_w": c["w"], f"c{i}_bias": c["bias"],
                    f"c{i}_scale": c["ws"], f"c{i}_stride": st, f"c{i}_pad": pad, f"c{i}_dilate": dl, f"c{i}_y": y,
                    f"c{i}_relu": relu, f"c{i}_s_in": c["s_in"], f"c{i}_s_out": c["s_out"], f"c{i}_z_in": c["z_in"],
                    f"c{i}_z_out": c["z_out"]})
        i += 1
    out["ncase"] = i
    np.savez_compressed(os.path.join(HERE, "conv_int8_golden.npz"), **out)
    print("conv_int8_golden.npz:", i, "cases")



def dw_linear_golden():
    """depthwise int8 conv + dynamic-quant linear outputs from the real reference (refdump conv mode 1 / linear); the inputs are
    regenerated from their seed by tests/cases.dw_linear_inputs and not stored."""
    g = dw_linear_inputs()
    out = {"ndw": len(DW_CASES), "nlin": len(LINEAR_CASES)}
    for i, (ch, k, n, ih, iw, st, pad, relu) in enumerate(DW_CASES):
        s_in, z_in, s_out, z_out = g[f"d{i}_q"]
        out[f"d{i}_y"] = O.ref_conv(1, g[f"d{i}_x"], g[f"d{i}_w"], g[f"d{i}_bias"], g[f"d{i}_ws"], stride=st, pad=pad, group=ch,
                                    relu=relu, z_in=int(z_in), z_out=int(z_out), scale_in=s_in, scale_out=s_out)
    for j, (tokens, ic, oc, asym, hb, lo, hi) in enumerate(LINEAR_CASES):
        alpha, wmin, bias = g[f"l{j}_alpha"], g[f"l{j}_wmin"], g[f"l{j}_bias"]
        al = np.stack([wmin, alpha], 1).ravel() if asym else alpha
        out[f"l{j}_y"] = O.ref_linear(g[f"l{j}_x"], g[f"l{j}_wq"], al, asym=asym, bias=bias if hb else None)
    np.savez_compressed(os.path.join(HERE, "dw_linear_golden.npz"), **out)
    print("dw_linear_golden.npz:", len(DW_CASES), "depthwise,", len(LINEAR_CASES), "linear cases")


def block_linear_golden():
    """K-blocked weight scales (MNN-LLM's default export, quant_block 64 / 128) through the real reference: prefill (>= 2 tokens)
    and decode (1 token) cases.  Oracle-only for now: the CUDA path declines block-wise layers (DESIGN.md section 9)."""
    rng = np.random.default_rng(78)
    out = {}
    j = 0
    for (tokens, ic, oc, blocks, asym, hb, lo, hi) in [(4, 256, 64, 4, False, False, -1, 1), (9, 512, 96, 8, True, True, -1, 1),
                                                       (33, 384, 40, 3, True, False, -1, 1), (1, 256, 64, 2, False, True, -1, 1),
                                                       (1, 512, 96, 4, True, True, 0.1, 2.0), (1, 128, 33, 2, True, False, -2, -0.5)]:
        x = rng.uniform(lo, hi, (tokens, ic)).astype(np.float32)
        wq = rng.integers(-128, 128, (oc, ic)).astype(np.int8)
        alpha = rng.uniform(0.001, 0.01, (oc, blocks)).astype(np.float32)
        wmin = rng.uniform(-0.05, 0.05, (oc, blocks)).astype(np.float32) if asym else np.zeros(0, np.float32)
        bias = rng.uniform(-1, 1, oc).astype(np.float32) if hb else np.zeros(0, np.float32)
        al = np.stack([wmin, alpha], 2).ravel() if asym else alpha.ravel()
        y = O.ref_linear(x, wq, al, asym=asym, bias=bias if hb else None, blocks=blocks)
        out.update({f"b{j}_x": x, f"b{j}_wq": wq, f"b{j}_alpha": alpha, f"b{j}_wmin": wmin, f"b{j}_bias": bias, f"b{j}_y": y})
        j += 1
    out["n"] = j
    np.savez_compressed(os.path.join(HERE, "block_linear_golden.npz"), **out)
    print("block_linear_golden.npz:", j, "cases")


def model_weight_hashes():
    """sha256 of every conv's weights/alpha as decoded BY THE REFERENCE (ConvolutionCommon::load via `refdump export`)."""
    import hashlib
    import json
    import tempfile
    model = os.path.join(HERE, "mbv2_int8.mnn")
    out = {}
    with tempfile.TemporaryDirectory() as d:
        O._run_refdump(["export", model, d])
        for line in open(os.path.join(d, "convs.txt")):
            name, opname, wsize, asize, asym = line.strip().split("|")
            idx = int(name.split("_")[1])
            w = open(os.path.join(d, name + ".w8"), "rb").read()
            a = open(os.path.join(d, name + ".alpha"), "rb").read()
            out[str(idx)] = dict(op=opname, w=hashlib.sha256(w).hexdigest(), alpha=hashlib.sha256(a).hexdigest(),
                                 n=int(wsize))
    json.dump(out, open(os.path.join(HERE, "mbv2_int8_weights_sha256.json"), "w"), indent=0)
    print("mbv2_int8_weights_sha256.json:", len(out), "convs")



def model_checkpoints():
    """Per-op outputs of the REAL reference on tests/golden/mbv2_int8.mnn (batch 1, seed 7): a subset is committed
    (the full per-op comparison runs live against oracle/_ref/refdump where it is present)."""
    import tempfile
    model = os.path.join(HERE, "mbv2_int8.mnn")
    keep = ["MobilenetV2/Conv/Conv2D", "MobilenetV2/expanded_conv/depthwise/depthwise", "MobilenetV2/expanded_conv/project/Conv2D",
            "MobilenetV2/expanded_conv_2/add", "MobilenetV2/expanded_conv_6/project/Conv2D", "MobilenetV2/expanded_conv_13/depthwise/depthwise",
            "MobilenetV2/expanded_conv_16/project/Conv2D", "MobilenetV2/Conv_1/Conv2D", "MobilenetV2/Logits/AvgPool",
            "MobilenetV2/Logits/Conv2d_1c_1x1/Conv2D", "MobilenetV2/Predictions/Softmax"]
    out = {}
    with tempfile.TemporaryDirectory() as d:
        recs = O.ref_run_model(model, 1, 7, d, 1)
        # the input is regenerated from the seed (tests/cases.refdump_input), not stored
        assert np.array_equal(np.fromfile(os.path.join(d, "input.f32"), np.float32), refdump_input((1, 3, 224, 224), 7).ravel())
        names = []
        for r in recs:
            if r["name"] in keep and r["scale"] > 0:
                f = np.fromfile(os.path.join(d, r["file"]), np.float32).reshape(r["dims"])
                q = np.rint(f / np.float32(r["scale"]) + np.float32(r["zero"])).astype(np.int8)
                out[f"t{len(names)}"] = q
                names.append(r["name"])
        last = recs[-1]
        out["output"] = np.fromfile(os.path.join(d, last["file"]), np.float32).reshape(last["dims"])
    out["names"] = np.array(names)
    np.savez_compressed(os.path.join(HERE, "mbv2_int8_checkpoints.npz"), **out)
    print("mbv2_int8_checkpoints.npz:", len(names), "tensors")



def wino_golden():
    """int8 Winograd conv outputs from the real reference, AVX2 build (oracle/_ref/refdump_avx2 wino): the reference
    test's own generator (test/op/ConvInt8Test.cpp:566-600) at F(2,3) plus calibrated random cases at F(2/4/6,3)."""
    from tests.cases import kat_wino, random_wino_case, wino_oracle
    assert O.have_reference_avx2(), "python oracle/build_ref.py --avx2"
    rng = np.random.default_rng(4242)
    cases = [(2, kat_wino(2, 32, 32, 39, 47))]
    for (unit, n, ic, oc, ih, iw, pad, relu) in [(2, 2, 16, 24, 12, 15, 1, True), (2, 1, 40, 33, 9, 7, 0, False),
                                                 (4, 2, 32, 16, 14, 14, 1, True), (4, 1, 13, 21, 11, 18, 1, False),
                                                 (6, 1, 32, 32, 19, 15, 1, True), (6, 2, 8, 20, 7, 9, 0, False)]:
        cases.append((unit, random_wino_case(rng, unit, n, ic, oc, ih, iw, pad, relu)))
    out = {"ncase": len(cases)}
    for i, (unit, c) in enumerate(cases):
        y = wino_oracle(O, c, unit, O.ref_wino)
        out[f"w{i}_unit"] = unit
        out[f"w{i}_y"] = y
        for k, v in c.items():
            out[f"w{i}_{k}"] = np.asarray(v)
    np.savez_compressed(os.path.join(HERE, "wino_int8_golden.npz"), **out)
    print("wino_int8_golden.npz:", len(cases), "cases")



def matmul_golden():
    """float MatMul / BatchMatMul outputs of the real reference CPU backend (refdump matmul)."""
    from tests.test_matmul import CASES
    g = matmul_inputs()        # regenerated from the seed, not stored
    out = {"ncase": len(CASES)}
    for i in range(len(CASES)):
        out[f"m{i}_y"] = O.ref_matmul(g[f"m{i}_a"], g[f"m{i}_b"], bool(g[f"m{i}_ta"]), bool(g[f"m{i}_tb"]))
    np.savez_compressed(os.path.join(HERE, "matmul_golden.npz"), **out)
    print("matmul_golden.npz:", len(CASES), "cases")


def reference_calls():
    """The reference's answers to every request the oracle tests send it (conv, depthwise, linear, pool, matmul, Winograd):
    tests/golden/reference_calls.npz, where oracle.py finds them by request when oracle/_ref is not built."""
    from tests import test_matmul, test_oracle, test_winograd
    O.recording = {}
    for case in KAT_SWEEP[:5]:
        test_oracle.test_oracle_bit_exact_vs_reference_legacy(case)
    test_oracle.test_oracle_bit_exact_vs_reference_modern()
    test_oracle.test_block_quant_linear_vs_live_reference()
    test_oracle.test_single_token_linear_is_the_references_decode_arithmetic()
    test_oracle.test_oracle_random_sweep_vs_live_reference()
    test_oracle.test_int8_pool_oracle_vs_live_reference()
    test_matmul.test_oracle_vs_live_reference()
    test_winograd.test_oracle_bit_exact_vs_live_reference_avx2()
    np.savez_compressed(O.RECORDED, **O.recording)
    print("reference_calls.npz:", len(O.recording), "answers")
    O.recording = None


def scale_int8_golden():
    """The first int8 Scale ops of ResNet-50 int8 (oracle/_ref/r50_int8.mnn, written by build()) as MNN_FORWARD_CPU runs them:
    parameters, quant attrs and an 8x8 spatial crop of the int8 input and output (the op is per channel: a crop is a whole case)."""
    import tempfile
    from mnn_b200 import mnn_file
    model = os.path.join(O.REF_DIR, "r50_int8.mnn")
    net = mnn_file.load(model)
    scales = [op for op in net.ops if op.type == "Scale"]
    assert len(scales) == 17 and scales[0].attrs["scale"] is not None
    out, k = {}, 0
    with tempfile.TemporaryDirectory() as d:
        by_name = {r["name"]: r for r in O.ref_run_model(model, 1, 3, d, 8)}
        producers = {op.outputs[0]: op for op in net.ops if op.outputs}
        for op in scales[:4]:
            r_out, r_in = by_name.get(op.name), by_name.get(producers[op.inputs[0]].name)
            if r_out is None or r_in is None or not r_out["apply_quant"] or not r_in["apply_quant"]:
                continue
            fi = np.fromfile(os.path.join(d, r_in["file"]), np.float32).reshape(r_in["dims"])
            fo = np.fromfile(os.path.join(d, r_out["file"]), np.float32).reshape(r_out["dims"])
            qi = np.rint(fi / np.float32(r_in["scale"]) + np.float32(r_in["zero"])).astype(np.int8)
            qo = np.rint(fo / np.float32(r_out["scale"]) + np.float32(r_out["zero"])).astype(np.int8)
            bias = op.attrs["bias"]
            out.update({f"s{k}_name": op.name, f"s{k}_x": qi[:, :, :8, :8], f"s{k}_y": qo[:, :, :8, :8],
                        f"s{k}_scale": np.asarray(op.attrs["scale"], np.float32),
                        f"s{k}_bias": np.zeros(0, np.float32) if bias is None else np.asarray(bias, np.float32),
                        f"s{k}_q": np.array([r_in["scale"], r_in["zero"], r_out["scale"], r_out["zero"], r_out["min"], r_out["max"]])})
            k += 1
    out["n"] = k
    np.savez_compressed(os.path.join(HERE, "scale_int8_golden.npz"), **out)
    print("scale_int8_golden.npz:", k, "ops")


def fullsize_golden():
    """What the reference computes at the bench configs' own sizes, as digests and samples (tests/test_gpu_wholenet.py,
    tests/test_gpu_configs.py): every int8 tensor of MobileNet-v2 at batch 2 (sha256 of the codes) and at batch 32 (the harness's
    position-weighted sums), the int8 Winograd F(6,3) outputs at batch 64 (sha256), the Qwen linear outputs at 4096 tokens
    (max |y| and a fixed sample of positions)."""
    import hashlib
    import tempfile
    from tests.cases import random_wino_case, refdump_input, wino_oracle
    from tests.test_gpu_configs import MODEL, _refdump_run, c4_case, c4_sample_positions
    from tests.test_gpu_wholenet import FP_INTERNAL
    out = {}
    with tempfile.TemporaryDirectory() as d:
        recs = O.ref_run_model(MODEL, 2, 11, d, 8)
        assert np.array_equal(np.fromfile(os.path.join(d, "input.f32"), np.float32), refdump_input((2, 3, 224, 224), 11).ravel())
        names, digests = [], []
        for r in recs:
            if r["scale"] <= 0 or not r["apply_quant"]:
                continue
            f = np.fromfile(os.path.join(d, r["file"]), np.float32).reshape(r["dims"])
            q = np.rint(f / np.float32(r["scale"]) + np.float32(r["zero"])).astype(np.int8)
            names.append(r["name"])
            digests.append(hashlib.sha256(q.tobytes()).hexdigest())
            if r["name"] in FP_INTERNAL:
                out[f"every_op_{r['name']}"] = q
        out["every_op_names"], out["every_op_sha256"] = np.array(names), np.array(digests)
    with tempfile.TemporaryDirectory() as d:
        cpu, _ = _refdump_run(O.REFDUMP, O.REF_DIR, MODEL, 32, 5, d, min(os.cpu_count() or 1, 32), False)
        assert np.array_equal(np.fromfile(os.path.join(d, "input.f32"), np.float32), refdump_input((32, 3, 224, 224), 5).ravel())
        for key, field in (("names", "name"), ("types", "type"), ("hashes", "file"), ("scales", "scale"), ("zeros", "zero"),
                           ("apply_quant", "apply_quant")):
            out["c2_" + key] = np.array([r[field] for r in cpu])
        out["c2_dims"] = np.array([",".join(str(v) for v in r["dims"]) for r in cpu])
    for C_, HW in ((64, 56), (512, 7)):
        c = random_wino_case(np.random.default_rng(C_ + HW), 6, 64, C_, C_, HW, HW, 1, True)
        ref = np.ascontiguousarray(wino_oracle(O, c, 6, O.ref_wino), np.int8)
        out[f"c3_{C_}_{HW}_sha256"] = np.array(hashlib.sha256(ref.tobytes()).hexdigest())
    for ic, oc, asym, has_bias in ((2048, 6144, True, True), (5504, 2048, True, False)):
        x, wq, alpha, wmin, bias = c4_case(4096, ic, oc, asym, has_bias)
        al = np.stack([wmin, alpha], 1).astype(np.float32).ravel() if asym else alpha
        ref = O.ref_linear(x, wq, al, asym=asym, bias=bias, threads=min(os.cpu_count() or 1, 32))
        out[f"c4_{ic}_{oc}_sample"] = ref.ravel()[c4_sample_positions(4096, oc)]
        out[f"c4_{ic}_{oc}_absmax"] = np.abs(ref).max()
    np.savez_compressed(os.path.join(HERE, "reference_fullsize.npz"), **out)
    print("reference_fullsize.npz:", len(out), "entries")


if __name__ == "__main__":
    # python tests/golden/make_golden.py [conv] [dw_linear] [block_linear] [hashes] [checkpoints] [wino] [matmul] [calls] [scale]
    #                                    [fullsize]   (default: all)
    assert O.have_reference(), "build oracle/_ref first: python oracle/build_ref.py"
    which = set(sys.argv[1:]) or {"conv", "dw_linear", "block_linear", "hashes", "checkpoints", "wino", "matmul", "calls", "scale",
                                  "fullsize"}
    if "conv" in which:
        conv_golden()
    if "dw_linear" in which:
        dw_linear_golden()
    if "block_linear" in which:
        block_linear_golden()
    if "hashes" in which:
        model_weight_hashes()
    if "checkpoints" in which:
        model_checkpoints()
    if "wino" in which:
        wino_golden()
    if "matmul" in which:
        matmul_golden()
    if "calls" in which:
        reference_calls()
    if "scale" in which:
        scale_int8_golden()
    if "fullsize" in which:
        fullsize_golden()
