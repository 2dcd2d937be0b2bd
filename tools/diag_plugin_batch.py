"""GPU-box diagnostic: where does the plugin's first int8 tensor start to differ from MNN_FORWARD_CPU as the batch grows?"""
import json, os, subprocess, sys, tempfile
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as O
PLUGIN = os.path.join(ROOT, "oracle", "_ref", "libmnn_b200_plugin.so")
MODEL = os.path.join(ROOT, "tests", "golden", "mbv2_int8.mnn")

def run(outdir, batch, plugin, extra=None, ncmd=3):
    env = dict(os.environ, REFDUMP_MAX_COMMANDS=str(ncmd), REFDUMP_HASH="0")
    env["LD_LIBRARY_PATH"] = O.REF_DIR + ":" + os.path.join(ROOT, "mnn_b200") + ":" + env.get("LD_LIBRARY_PATH", "")
    if plugin: env["REFDUMP_PLUGIN"] = PLUGIN
    env.update(extra or {})
    os.makedirs(outdir, exist_ok=True)
    r = subprocess.run([O.REFDUMP, "run", MODEL, str(batch), "5", outdir, "8"], env=env, capture_output=True, text=True, timeout=600)
    recs = [l.rstrip("\n").split("|") for l in open(os.path.join(outdir, "index.txt"))]
    return recs, r

for batch in (4, 8, 12, 16, 24, 32):
    with tempfile.TemporaryDirectory() as d:
        cpu, _ = run(os.path.join(d, "c"), batch, False)
        gpu, r = run(os.path.join(d, "g"), batch, True)
        x = np.fromfile(os.path.join(d, "c", "input.f32"), np.float32)
        out = []
        for (fc, name, typ, dims, *_), (fg, *_) in zip(cpu, gpu):
            a = np.fromfile(os.path.join(d, "c", fc), np.float32); b = np.fromfile(os.path.join(d, "g", fg), np.float32)
            nd = int(np.count_nonzero(a != b))
            info = f"{name.split('/')[-1]}[{dims}]: {nd}/{a.size} differ"
            if nd and a.size == x.size:
                info += f"; plugin==input at {int(np.count_nonzero(b == x))} positions; first diff idx {int(np.flatnonzero(a != b)[0])}, last {int(np.flatnonzero(a != b)[-1])}"
            out.append(info)
        print("batch", batch, "|", " || ".join(out), "| stderr:", r.stderr[-200:].replace("\n", " "))
