"""The drop-in boundary, end to end (-m gpu): the UNMODIFIED reference core (oracle/_ref/libMNN.so: Interpreter, Session,
Pipeline, geometry, quant-cast insertion) schedules tests/golden/mbv2_int8.mnn on MNN_FORWARD_CUDA, where the only registered
RuntimeCreator is oracle/_ref/libmnn_b200_plugin.so (mnn_b200/csrc/plugin/b200_plugin.cpp -> C ABI -> sm_100a kernels).  Every
command's output tensor, read back through the plugin's onCopyBuffer, must equal what the same process produces on
MNN_FORWARD_CPU -- bit for bit for int8 tensors (compared at the dequantised boundary, SURVEY F6), and the plugin must have
created EVERY command (nothing handed back to the CPU backup backend)."""
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
from tests.cases import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGIN = O.PLUGIN
MODEL = os.path.join(ROOT, "tests", "golden", "mbv2_int8.mnn")


def test_plugin_library_is_built_and_exports_registration_hook():
    """CPU-side check: the plugin .so exists in-tree and exports its stats hook; it links the C ABI library."""
    if not O.have_reference():
        pytest.skip("the plugin is built with the reference core (oracle/_ref), which is not built here")
    assert os.path.exists(PLUGIN), "the plugin is missing although the reference core is built (mnn_b200/csrc/plugin/build_plugin.py)"
    out = subprocess.run(["nm", "-D", "--defined-only", PLUGIN], capture_output=True, text=True, check=True).stdout
    assert "mnnb200_plugin_stats" in out
    need = subprocess.run(["objdump", "-p", PLUGIN], capture_output=True, text=True, check=True).stdout
    assert "libmnn_b200.so" in need
    undef = subprocess.run(["nm", "-D", "--undefined-only", PLUGIN], capture_output=True, text=True, check=True).stdout
    assert "MNNInsertExtraRuntimeCreator" in undef      # resolved by the host's libMNN at dlopen time


def _run(outdir, batch, plugin, model=None):
    model = model or MODEL
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = O.REF_DIR + ":" + os.path.join(ROOT, "mnn_b200") + ":" + env.get("LD_LIBRARY_PATH", "")
    if plugin:
        env["REFDUMP_PLUGIN"] = PLUGIN
    else:
        env.pop("REFDUMP_PLUGIN", None)
    os.makedirs(outdir, exist_ok=True)
    r = subprocess.run([O.REFDUMP, "run", model, str(batch), "3", outdir, "4"], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-500:]
    recs = []
    for line in open(os.path.join(outdir, "index.txt")):
        f, name, typ, dims, qs, qz, qmin, qmax, aq = line.rstrip("\n").split("|")
        recs.append((f, name, typ.strip(), float(qs), int(aq)))
    stats = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{\"plugin_")]
    return recs, (stats[-1] if stats else None), r


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [1, 4])
def test_reference_pipeline_on_plugin_matches_cpu_backend(batch):
    _need_ref_and_plugin()
    with tempfile.TemporaryDirectory() as d:
        cpu, _, _ = _run(os.path.join(d, "cpu"), batch, False)
        gpu, stats, r = _run(os.path.join(d, "gpu"), batch, True)
        assert stats is not None and stats["plugin_declined"] == 0, f"commands fell back to the CPU backend: {stats}\n{r.stderr[-1500:]}\n{r.stdout[-1500:]}"
        assert stats["plugin_created"] >= len(gpu) >= 70
        assert [(n, t) for _, n, t, _, _ in cpu] == [(n, t) for _, n, t, _, _ in gpu], "command lists differ"
        worst = 0.0
        for (fc, name, typ, qs, aq), (fg, _, _, _, _) in zip(cpu, gpu):
            a = np.fromfile(os.path.join(d, "cpu", fc), np.float32)
            b = np.fromfile(os.path.join(d, "gpu", fg), np.float32)
            assert a.shape == b.shape, name
            if aq:      # int8 tensor seen through Int8ToFloat: equal floats <=> equal int8 codes
                assert np.array_equal(a, b), f"{name} ({typ}): {np.count_nonzero(a != b)} of {a.size} int8 values differ"
            else:       # fp32 tensor between casts: north_star tolerance 1e-3 relative
                den = max(np.abs(a).max(), 1e-12)
                worst = max(worst, float(np.abs(a - b).max() / den))
                assert np.abs(a - b).max() / den <= 1e-3, f"{name} ({typ}) rel err {np.abs(a - b).max() / den}"
        oc = np.fromfile(os.path.join(d, "cpu", "output.f32"), np.float32)
        og = np.fromfile(os.path.join(d, "gpu", "output.f32"), np.float32)
        assert np.abs(oc - og).max() <= 1e-3 * max(np.abs(oc).max(), 1e-12)


def _need_ref_and_plugin():
    if not O.have_reference():
        pytest.skip("the reference core (oracle/_ref, built by oracle/build_ref.py) is not built here")
    if not os.path.exists(PLUGIN):
        pytest.fail("oracle/_ref/libmnn_b200_plugin.so is missing although the reference core is present")


def _plugin_env():
    env = dict(os.environ, REFDUMP_PLUGIN=PLUGIN)
    env["LD_LIBRARY_PATH"] = O.REF_DIR + ":" + os.path.join(ROOT, "mnn_b200") + ":" + env.get("LD_LIBRARY_PATH", "")
    return env


@pytest.mark.gpu
def test_llm_linear_through_reference_executor_on_plugin():
    """The MNN-LLM linear layer (Convolution 1x1, IDST int8 weights, BackendConfig::Memory_Low => W8A8 dynamic quant) built
    with the reference's own Express API and run by its Executor on MNN_FORWARD_CUDA (= the plugin) must reproduce the
    outputs the reference CPU backend recorded in tests/golden/dw_linear_golden.npz."""
    import struct
    _need_ref_and_plugin()
    g = load_golden("dw_linear_golden")
    for j in range(int(g["nlin"])):
        x, wq, alpha, wmin, bias, ref = (g[f"l{j}_{k}"] for k in ("x", "wq", "alpha", "wmin", "bias", "y"))
        tokens, ic = x.shape
        oc = wq.shape[0]
        asym = wmin.size > 0
        al = np.stack([wmin, alpha], 1).astype(np.float32).ravel() if asym else alpha.astype(np.float32)
        payload = struct.pack("<8i", tokens, ic, oc, int(asym), 0, 0, int(bias.size > 0), 0) + x.tobytes() + wq.tobytes() + al.tobytes()
        if bias.size:
            payload += bias.astype(np.float32).tobytes()
        with tempfile.TemporaryDirectory() as d:
            req, out = os.path.join(d, "req.bin"), os.path.join(d, "out.bin")
            open(req, "wb").write(payload)
            r = subprocess.run([O.REFDUMP, "linear", req, out, "1"], env=_plugin_env(), capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stderr[-1500:]
            stats = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{\"plugin_")]
            assert stats and stats[-1]["plugin_created"] >= 1, f"the linear layer did not run on the plugin: {r.stdout[-500:]} {r.stderr[-800:]}"
            y = np.fromfile(out, np.float32).reshape(tokens, oc)
        assert np.abs(y - ref).max() <= 1e-3 * np.abs(ref).max(), f"linear {j}: {np.abs(y - ref).max() / np.abs(ref).max()}"


@pytest.mark.gpu
def test_matmul_through_reference_executor_on_plugin():
    import struct
    _need_ref_and_plugin()
    g = load_golden("matmul_golden")
    done = 0
    for i in range(int(g["ncase"])):
        a, b, ta, tb, ref = g[f"m{i}_a"], g[f"m{i}_b"], bool(g[f"m{i}_ta"]), bool(g[f"m{i}_tb"]), g[f"m{i}_y"]
        if a.ndim != 2:
            continue       # BatchMatMul is decomposed by the reference's geometry stage; the 2-D MatMul op is the plugin's unit
        e, l = (a.shape[1], a.shape[0]) if ta else a.shape
        h = b.shape[0] if tb else b.shape[1]
        with tempfile.TemporaryDirectory() as d:
            req, out = os.path.join(d, "req.bin"), os.path.join(d, "out.bin")
            open(req, "wb").write(struct.pack("<8i", 1, e, l, h, int(ta), int(tb), 0, 0) + a.tobytes() + b.tobytes())
            r = subprocess.run([O.REFDUMP, "matmul", req, out], env=_plugin_env(), capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stderr[-1500:]
            y = np.fromfile(out, np.float32).reshape(ref.shape)
        assert np.abs(y - ref).max() <= 1e-3 * np.abs(ref).max(), f"matmul {i}: {np.abs(y - ref).max() / np.abs(ref).max()}"
        done += 1
    assert done >= 3


@pytest.mark.gpu
def test_plugin_graph_replay_and_mid_run_interrupt_match_cpu_backend():
    """The plugin captures the second forward into a CUDA graph and replays it from the third on (onExecuteBegin/End); a
    forward with per-command callbacks (copyToHostTensor in the middle of the run) must flush the deferred launches and go on
    eagerly.  4 plain forwards (eager, capture, replay, replay), then the callback forward: the replayed output and every
    per-command tensor equal MNN_FORWARD_CPU's."""
    _need_ref_and_plugin()
    batch = 2
    with tempfile.TemporaryDirectory() as d:
        env_keep = os.environ.get("REFDUMP_RUN_REPEATS")
        os.environ["REFDUMP_RUN_REPEATS"] = "4"
        try:
            cpu, _, _ = _run(os.path.join(d, "cpu"), batch, False)
            gpu, stats, r = _run(os.path.join(d, "gpu"), batch, True)
        finally:
            if env_keep is None:
                os.environ.pop("REFDUMP_RUN_REPEATS", None)
            else:
                os.environ["REFDUMP_RUN_REPEATS"] = env_keep
        assert stats is not None and stats["plugin_declined"] == 0
        oc = np.fromfile(os.path.join(d, "cpu", "output_plain.f32"), np.float32)
        og = np.fromfile(os.path.join(d, "gpu", "output_plain.f32"), np.float32)
        assert np.abs(oc - og).max() <= 1e-3 * max(np.abs(oc).max(), 1e-12) + 0.05, "graph-replayed forward differs"
        n = 0
        for (fc, name, typ, qs, aq), (fg, _, _, _, _) in zip(cpu, gpu):
            if not aq or "Softmax" in name:
                continue
            a = np.fromfile(os.path.join(d, "cpu", fc), np.float32)
            b = np.fromfile(os.path.join(d, "gpu", fg), np.float32)
            assert np.array_equal(a, b), f"{name} ({typ}) after a mid-run interrupt: {np.count_nonzero(a != b)} differ"
            n += 1
        assert n >= 60


@pytest.mark.gpu
@pytest.mark.parametrize("model_name", ["r50_int8.mnn", "r50_int8_eq.mnn"])
def test_resnet50_int8_on_plugin_matches_cpu_backend(model_name):
    """BASELINE configs[2] as a MODEL: ResNet-50 (v2) int8 from the reference's weight-less benchmark graph + its own Revert tool
    (oracle/_ref/r50_int8.mnn: retuned per-tensor scales -> int8 Convolution / Scale / BinaryOp, float ReLU / Reduction / max
    pooling between casts; r50_int8_eq.mnn: Revert's equal scales -> the CPU backend's int8 Pooling too).  Every command on the
    plugin (none declined), every int8 tensor bit-exact vs MNN_FORWARD_CPU, fp32 tensors within 1e-3."""
    _need_ref_and_plugin()
    model = os.path.join(O.REF_DIR, model_name)
    if not os.path.exists(model):
        pytest.skip(f"{model_name} not generated (build() writes it where the reference sources are present)")
    batch = 2
    with tempfile.TemporaryDirectory() as d:
        cpu, _, _ = _run(os.path.join(d, "cpu"), batch, False, model)
        gpu, stats, r = _run(os.path.join(d, "gpu"), batch, True, model)
        assert stats is not None and stats["plugin_declined"] == 0, f"commands fell back to the CPU backend: {stats}\n{r.stdout[-2500:]}"
        # The two backends may place the FloatToInt8 / Int8ToFloat casts differently around Raster (the CPU keeps a Raster in int8
        # when its tensors share one scale, the plugin dequantises -> copies -> requantises, which reproduces the same int8 values):
        # compare every tensor BY NAME; every compute op of the CPU run must exist in the plugin run
        by_name = {name: (fg, typ, aq) for fg, name, typ, _, aq in gpu}
        kinds, missing, mism = {}, [], []
        for fc, name, typ, qs, aq in cpu:
            k = typ.split()[0]
            helper = k in ("FloatToInt8", "Int8ToFloat", "Raster") or "_raster_" in name     # geometry / cast helper tensors
            if name not in by_name:
                if not helper:
                    missing.append((name, typ))
                continue
            fg, typ_g, aq_g = by_name[name]
            if helper and (typ_g.split()[0] != k or bool(aq) != bool(aq_g)):
                continue          # the same helper name denotes different commands (or an int8 vs a float copy) in the two runs
            a = np.fromfile(os.path.join(d, "cpu", fc), np.float32)
            b = np.fromfile(os.path.join(d, "gpu", fg), np.float32)
            if a.shape != b.shape and k in ("FloatToInt8", "Int8ToFloat", "Raster"):
                continue          # helper tensors of differently placed casts share names, not shapes
            assert a.shape == b.shape, name
            if aq and aq_g and "Softmax" not in typ:
                if not np.array_equal(a, b):
                    bad = np.flatnonzero(a != b)
                    mism.append(f"{name} ({typ} | plugin {typ_g}): {bad.size} of {a.size} int8 values differ, scale {qs}, first idx "
                                f"{bad[:3].tolist()} cpu/scale {(a[bad[:3]] / qs).tolist()} plugin/scale {(b[bad[:3]] / qs).tolist()}")
            else:
                den = max(np.abs(a).max(), 1e-12)
                if np.abs(a - b).max() / den > 1e-3 + (0.05 if "Softmax" in typ else 0):
                    mism.append(f"{name} ({typ} | plugin {typ_g}) fp rel err {np.abs(a - b).max() / den}")
            kinds[k] = kinds.get(k, 0) + 1
        assert not mism, "\n".join(mism[:8]) + f"\n... {len(mism)} tensors differ"
        assert not missing, missing
        assert kinds.get("Convolution", 0) >= 50 and kinds.get("Scale", 0) >= 17 and kinds.get("BinaryOp", 0) >= 16, kinds
        oc = np.fromfile(os.path.join(d, "cpu", "output.f32"), np.float32)
        og = np.fromfile(os.path.join(d, "gpu", "output.f32"), np.float32)
        assert np.abs(oc - og).max() <= 1e-3 * max(np.abs(oc).max(), 1e-12) + 0.05
