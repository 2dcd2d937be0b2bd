#!/usr/bin/env python3
"""bench.py -- MobileNet-v2-int8 hot-path throughput on B200 (driver contract in the task statement).

  python bench.py --gpus N --steps K --warmup W          # our arm (CUDA, through the C ABI)
  python bench.py --impl reference --gpus N ...           # the reference's own CPU implementation of the same path

A "step" = one pass of the hot path over one batch of synthetic input.  Workload at N=1 = BASELINE.json
configs[1]: MobileNet-v2 int8 .mnn, batch 32, the 36 dense int8 convolutions (ConvInt8 path only), every layer
on its own resident NHWC16 activation (240 MB of distinct traffic per step > 126 MB L2, so consecutive steps
cannot be served from L2).  N>1: one replica per GPU, batch 32 each (weak scaling), the model bytes broadcast once
from rank 0 over NCCL at session build, no steady-state communication.
"""
import argparse
import json
import os
import re
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL = os.path.join(ROOT, "tests", "golden", "mbv2_int8.mnn")
BATCH_PER_GPU = 32
DUMP_ELEMENTS_PER_LAYER = 1 << 18     # --dump-outputs: 36 layers x 1 MB of float32 at most
# one metric string and one workload string for BOTH arms (the driver divides the two lines only when they agree)
METRIC = "inferences/sec (MobileNet-v2-int8 224x224, batch 32 per GPU, dense int8 conv path)"
WORKLOAD = ("MobileNet-v2 int8 .mnn (reference Revert-quantised graph, retuned weights), batch 32 per GPU, the 36 dense int8 "
            "convolutions (BASELINE.json configs[1]: ConvInt8 path only), every layer on its own resident activation")


def cpu_info():
    """CPU model / core count / ISA of the host the CPU arm runs on (BASELINE.md section 3)."""
    info = {"logical_cpus": os.cpu_count()}
    try:
        txt = open("/proc/cpuinfo").read()
        for line in txt.splitlines():
            if line.startswith("model name"):
                info["model"] = line.split(":", 1)[1].strip()
                break
        flags = next((l.split(":", 1)[1].split() for l in txt.splitlines() if l.startswith("flags")), [])
        info["isa"] = [f for f in ("avx2", "fma", "avx512f", "avx512bw", "avx512_vnni", "avx_vnni", "amx_int8") if f in flags]
        cores = {(b.split("physical id")[1].split("\n")[0], b.split("core id")[1].split("\n")[0])
                 for b in txt.strip().split("\n\n") if "core id" in b and "physical id" in b}
        info["physical_cores"] = len(cores) or None
    except Exception:
        pass
    info["reference_build"] = "oracle/build_ref.py: -O3 -mavx512f/bw/vl/dq -mavx512vnni kernels enabled (MNN_AVX512), MNN_LOW_MEMORY"
    return info


def numa_bind(local_rank):
    """Pin this process (and the pinned host buffers it is about to allocate) to the NUMA node of its GPU: the e2e number is
    PCIe-bound and a remote-node staging buffer costs 2-3x in H2D bandwidth (round-1 VERDICT weak #7)."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8: "hw_slowdown",
                 getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def conv_shapes_file(path):
    from mnn_b200 import graph, mnn_file
    net = mnn_file.load(MODEL)
    graph.infer_shapes(net, (1, 3, 224, 224))
    with open(path, "w") as f:
        for i, op in enumerate(net.ops):
            if op.type == "Convolution":
                _, _, h, w = op.attrs["in_shape"]
                f.write(f"{i} {h} {w}\n")


def cpu_reference_rate(batch, iters, warmup, threads=None):
    """images/s of the reference CPU backend on the same 36 dense conv layers (oracle/_ref when present, else the
    scalar C port).  Bounded sample; returns (value, cores, kind, sample description)."""
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    if O.have_reference():
        import tempfile
        threads = threads or min(cores, 32)
        with tempfile.TemporaryDirectory() as d:
            shp = os.path.join(d, "shapes.txt")
            conv_shapes_file(shp)
            r = O._run_refdump(["convbench", MODEL, shp, batch, threads, warmup, iters], timeout=1200)
        j = json.loads(r.stdout.strip().splitlines()[-1])
        return batch / (j["ms_total"] / 1e3), threads, "reference", \
            f"MNN_FORWARD_CPU ({threads} threads) on the 36 dense convs, batch {batch}, {iters} timed runs per layer after {warmup} warm-up"
    # port: scalar C restatement, batch 1, largest layers only would bias; run every layer once at batch 1
    import numpy as np
    from mnn_b200 import graph, mnn_file
    net = mnn_file.load(MODEL)
    graph.infer_shapes(net, (1, 3, 224, 224))
    rng = np.random.default_rng(0)
    t = 0.0
    for op in graph.dense_convs(net):
        n, c, h, w = op.attrs["in_shape"]
        x = rng.integers(-127, 128, (1, c, h, w)).astype(np.int8)
        cv = op.conv
        qi, qo = net.quant[op.inputs[0]], net.quant[op.outputs[0]]
        bf, sx = O.fold_modern(cv.weight, cv.alpha, cv.bias, qi.scale, int(qi.zero), qo.scale, int(qo.zero))
        t0 = time.perf_counter()
        O.conv_int8(x, cv.weight, cv.alpha, sx, bf, stride=cv.stride, pad=op.attrs["resolved_pad"], dilate=cv.dilate,
                    z_in=int(qi.zero))
        t += time.perf_counter() - t0
    return 1.0 / t, 1, "port", "scalar C oracle, 36 dense convs, batch 1, one pass"


def plugin_e2e_rate(batch=BATCH_PER_GPU, warmup=5, iters=20, windows=9, device=None, pin_user_tensors=True):
    """The WHOLE .mnn through the reference's own Interpreter::runSession (copyFromHostTensor of the fp32 NCHW input +
    runSession + copyToHostTensor of the result per iteration, benchmark/benchmark.cpp:120-181 style) scheduled on
    MNN_FORWARD_CUDA = oracle/_ref/libmnn_b200_plugin.so: the call a user of MNN makes.  The host program is the reference core
    built under oracle/_ref (the CALLER of the plugin, not a checker).  Median of `windows` windows of `iters` iterations."""
    import subprocess
    from oracle import oracle as O
    plugin = O.PLUGIN
    if not (O.have_reference() and os.path.exists(plugin)):
        return {"value": None, "note": "reference core or plugin .so not present"}
    env = dict(os.environ, REFDUMP_PLUGIN=plugin, REFDUMP_BENCH_WINDOWS=str(windows))
    # the harness keeps its input / output host tensors alive for the whole session: the documented precondition of the plugin's
    # opt-in in-place pinning (the e2e contract asks for copies from pinned host memory); the default (pageable) is timed too
    env["MNNB200_PLUGIN_HOSTREG"] = "1" if pin_user_tensors else "0"
    if device is not None:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        env["CUDA_VISIBLE_DEVICES"] = vis.split(",")[device] if vis else str(device)
    env["LD_LIBRARY_PATH"] = O.REF_DIR + ":" + os.path.join(ROOT, "mnn_b200") + ":" + env.get("LD_LIBRARY_PATH", "")
    r = subprocess.run([O.REFDUMP, "bench", MODEL, str(batch), "4", str(warmup), str(iters)], env=env, capture_output=True,
                       text=True, timeout=600)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if not lines:
        return {"value": None, "note": ("refdump bench failed: " + r.stderr[-300:])}
    j = json.loads(lines[-1])
    if j.get("plugin_declined", 0) != 0:
        # an op handed back to MNN's CPU backup backend would make this a mixed CPU/GPU number: refuse to report it
        return {"value": None, "note": f"plugin declined {j['plugin_declined']} commands (CPU backup ran them): not reported"}
    ms = j.get("ms_median_window", j["ms_per_iter"])
    return {"value": batch / (ms / 1e3), "unit": "img/s", "ms_per_iter": ms, "ms_mean": j["ms_per_iter"], "batch": batch,
            "windows": j.get("windows", 1), "iters_per_window": iters,
            "plugin_created": j.get("plugin_created"), "plugin_declined": j.get("plugin_declined"),
            "h2d_bytes_per_step": j.get("h2d_bytes"), "d2h_bytes_per_step": j.get("d2h_bytes"),
            "host_tensors": "pinned in place (MNNB200_PLUGIN_HOSTREG=1)" if pin_user_tensors else "pageable (plugin default)",
            "note": "unmodified MNN Interpreter + libmnn_b200_plugin.so, host tensors in/out every iteration, every command on the GPU"}


def dump_outputs(sess, out_dir):
    """The int8 output of every dense conv of the session's last step, as out_dir/<layer>_<name>.npy in float32 (logical NCHW).
    A layer with more than DUMP_ELEMENTS_PER_LAYER elements is written as the elements at a fixed, seeded sample of its flat
    NCHW positions (np.random.default_rng(layer).integers(0, size, DUMP_ELEMENTS_PER_LAYER), sorted)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    sess.stream.synchronize()
    for i, (node, _, _, y) in enumerate(sess.layers):
        with torch.cuda.stream(sess.stream):
            out = sess.backend.onCopyBuffer(y, "same").astype(np.float32).ravel()
        if out.size > DUMP_ELEMENTS_PER_LAYER:
            out = out[np.sort(np.random.default_rng(i).integers(0, out.size, DUMP_ELEMENTS_PER_LAYER))]
        np.save(os.path.join(out_dir, f"{i:02d}_{re.sub(r'[^A-Za-z0-9_.-]', '_', node.name)}.npy"), out)


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref = the unmodified reference built
    here) on this box's host cores, same metric / config / batch as our arm.  A step = one pass over the 36 dense convs at
    batch 32; the run is bounded to min(steps, 20) timed passes per layer."""
    if rank != 0:
        return
    batch = BATCH_PER_GPU
    iters, warm = max(1, min(args.steps, 20)), max(1, min(args.warmup, 3))
    val, cores, kind, sample = cpu_reference_rate(batch, iters, warm)
    one = None
    try:
        v1, _, _, s1 = cpu_reference_rate(batch, 1, 1, threads=1)
        one = {"value": v1, "unit": "img/s", "cores": 1, "sample": s1}
    except Exception as e:
        one = {"error": repr(e)[:200]}
    whole = None
    try:
        from oracle import oracle as O
        if O.have_reference():
            os.environ["REFDUMP_BENCH_WINDOWS"] = "3"
            j = O.ref_bench(MODEL, batch, min(os.cpu_count() or 1, 32), 1, 3)
            whole = {"value": batch / (j["ms_median_window"] / 1e3), "unit": "img/s", "threads": j["threads"], "batch": batch,
                     "note": "whole .mnn through Interpreter::runSession incl. input/output copies (benchmark.cpp:120-181), "
                             "the same harness bench.py times on the plugin for our arm's e2e"}
    except Exception as e:
        whole = {"error": repr(e)[:200]}
    line = {
        "impl": "reference", "metric": METRIC,
        "value": val, "unit": "img/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * batch / val, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "s8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_gpu": batch,
                   "implementation": "reference CPU backend (MNN_FORWARD_CPU), host cores only", "timed_passes": iters},
        "cpu_baseline": {"value": val, "unit": "img/s", "cores": cores, "kind": kind, "sample": sample,
                         "single_thread": one, "cpu": cpu_info()},
        "e2e": {"value": val, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "whole_net": whole,
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _max_over_ranks(torch, dist, world, ms):
    t = torch.tensor([ms], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the whole-net / ResNet-Winograd / Qwen sub-objects")
    ap.add_argument("--workload", default="mbv2", choices=["mbv2", "resnet_wino", "resnet_direct", "qwen", "qwen_decode"],
                    help="mbv2 = the driver's line (BASELINE configs[1]); resnet_wino / qwen = configs[2] / configs[3] alone")
    ap.add_argument("--wino-unit", type=int, default=6, choices=[2, 4, 6])
    ap.add_argument("--qwen-layers", type=int, default=24)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (every conv's output) to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload != "mbv2"):
        ap.error("--dump-outputs writes the outputs of the CUDA arm's mbv2 workload only")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a GPU: there is no CPU fallback on the product path"
    torch.cuda.set_device(local_rank)
    numa_node = numa_bind(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.workload != "mbv2":
        import bench_workloads
        fn = {"resnet_wino": bench_workloads.run_resnet_wino, "resnet_direct": bench_workloads.run_resnet_direct,
              "qwen": bench_workloads.run_qwen, "qwen_decode": bench_workloads.run_qwen_decode}[args.workload]
        line = fn(args, ClockSampler, rank=rank, world=world, local_rank=local_rank)
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    from mnn_b200 import _capi, mnn_file
    from mnn_b200.session import ConvPathSession

    # ---- session build: rank 0 reads the model; one NCCL broadcast ships the weights to every replica
    from mnn_b200.dist_util import broadcast_model_bytes
    model_bytes = broadcast_model_bytes(MODEL, rank, world, device="cuda")
    sess = ConvPathSession(mnn_file.load(model_bytes), BATCH_PER_GPU, device_id=local_rank, seed=rank)
    if not args.no_graph:
        sess.capture()
    W = max(args.warmup, 3)
    K = args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed throughput (inputs resident in HBM): EXACTLY K steps between two events on the launching stream
    for _ in range(W):
        sess.run()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    lc0 = _capi.lib().mnnb200_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(sess.stream):
        ev0.record()
    for _ in range(K):
        sess.run()
    with torch.cuda.stream(sess.stream):
        ev1.record()
    barrier()
    my_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(sess, args.dump_outputs)
    ms_total = _max_over_ranks(torch, dist, world, my_ms)
    # a longer look at the same loop (several K-step windows, >= 0.25 s): the median window guards the short K-step region
    # against one straggling host-side graph launch (round-1 SCALE N=4 dip)
    win = []
    t_end = time.time() + 0.25
    while len(win) < 5 or (time.time() < t_end and len(win) < 40):
        with torch.cuda.stream(sess.stream):
            ev0.record()
        for _ in range(K):
            sess.run()
        with torch.cuda.stream(sess.stream):
            ev1.record()
        sess.stream.synchronize()
        win.append(ev0.elapsed_time(ev1))
    sampler.stop_flag = True
    sampler.join()
    win.sort()
    ms_median = _max_over_ranks(torch, dist, world, win[len(win) // 2])
    per_rank_ms = None
    if world > 1:
        g = [torch.zeros(1, device="cuda") for _ in range(world)]
        dist.all_gather(g, torch.tensor([my_ms], device="cuda"))
        per_rank_ms = [float(x.item()) / K for x in g]
    ms_per_step = ms_total / K
    value = BATCH_PER_GPU * world * K / (ms_total / 1e3)
    host_launches = _capi.lib().mnnb200_launch_count() - lc0
    gpu_launches = sess.launches_per_step * K          # kernels executed (graph replays re-run the captured launches)

    # ---- e2e (C ABI): host buffers -> C ABI -> host buffers, copies inside the timed region, median of >= 0.5 s of windows
    h2d, d2h = sess.make_host_io()

    def windows(run_k, min_s=0.5, max_n=60):
        out, t_end = [], time.time() + min_s
        while True:
            barrier()
            with torch.cuda.stream(sess.stream):
                ev0.record()
            run_k()
            with torch.cuda.stream(sess.stream):
                ev1.record()
            barrier()
            out.append(_max_over_ranks(torch, dist, world, ev0.elapsed_time(ev1)))
            more = 1.0 if (len(out) < 5 or (time.time() < t_end and len(out) < max_n)) else 0.0
            if world > 1:   # every rank must agree on the loop count
                flag = torch.tensor([more], device="cuda")
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                more = float(flag.item())
            if more == 0.0:
                break
        out.sort()
        return out

    def serial_k():
        for _ in range(K):
            sess.run_e2e()
            sess.stream.synchronize()                   # the user reads the result every step
    for _ in range(W):
        sess.run_e2e()
    ws = windows(serial_k)
    e2e_serial = BATCH_PER_GPU * world * K / (ws[len(ws) // 2] / 1e3)
    # same steps with the copies of step k+1 overlapped with the kernels of step k (two pinned-input device buffers)
    sess.run_e2e_pipelined(W)
    wp = windows(lambda: sess.run_e2e_pipelined(K))
    e2e_pipe = BATCH_PER_GPU * world * K / (wp[len(wp) // 2] / 1e3)

    # ---- e2e (the call a user of MNN makes): whole .mnn through Interpreter::runSession on the plugin, host tensors in/out
    plug = None
    if not args.no_extra:
        try:
            plug = plugin_e2e_rate(device=local_rank)
        except Exception as e:
            plug = {"value": None, "note": repr(e)[:200]}
        if rank == 0 and world == 1 and plug.get("value"):
            try:    # the plugin's default: user tensors stay pageable (short run, reported beside the pinned number)
                d = plugin_e2e_rate(device=local_rank, windows=3, pin_user_tensors=False)
                plug["pageable_default"] = {"value": d.get("value"), "ms_per_iter": d.get("ms_per_iter")}
            except Exception as e:
                plug["pageable_default"] = {"error": repr(e)[:120]}
        if world > 1:   # whole job = sum over replicas at the slowest replica's pace
            v = torch.tensor([plug["value"] if plug.get("value") else 0.0], device="cuda")
            dist.all_reduce(v, op=dist.ReduceOp.MIN)
            plug = dict(plug, value=(float(v.item()) * world) if v.item() > 0 else None, per_replica_min=float(v.item()))

    # ---- the WHOLE network through the C ABI (every op on the GPU, no CPU fallback), same model, same batch
    whole = None
    if not args.no_extra:
        try:
            from mnn_b200.session import WholeNetSession
            wsess = WholeNetSession(mnn_file.load(model_bytes), BATCH_PER_GPU, device_id=local_rank)
            if not args.no_graph:
                wsess.capture()
            wh2d, wd2h = wsess.make_host_io()
            for _ in range(W):
                wsess.run()
            barrier()
            with torch.cuda.stream(wsess.stream):
                ev0.record()
            for _ in range(K):
                wsess.run()
            with torch.cuda.stream(wsess.stream):
                ev1.record()
            barrier()
            w_ms = _max_over_ranks(torch, dist, world, ev0.elapsed_time(ev1)) / K
            for _ in range(W):
                wsess.run_e2e()
            barrier()
            with torch.cuda.stream(wsess.stream):
                ev0.record()
            for _ in range(K):
                wsess.run_e2e()
                wsess.stream.synchronize()
            with torch.cuda.stream(wsess.stream):
                ev1.record()
            barrier()
            we_ms = _max_over_ranks(torch, dist, world, ev0.elapsed_time(ev1))
            whole = {"value": BATCH_PER_GPU * world / (w_ms / 1e3), "unit": "img/s", "ms_per_step": w_ms,
                     "kernels_per_step": wsess.launches_per_step,
                     "e2e": {"value": BATCH_PER_GPU * world * K / (we_ms / 1e3), "unit": "img/s",
                             "h2d_bytes_per_step": wh2d, "d2h_bytes_per_step": wd2h},
                     "note": "all 71 ops of the .mnn on the GPU (36 conv, 17 depthwise, 10 add, pool, softmax, casts); "
                             "bit-exact vs the reference CPU backend (tests/test_gpu_wholenet.py)"}
            del wsess
        except Exception as e:  # the headline line must survive
            whole = {"error": repr(e)[:300]}

    # ---- BASELINE configs[2] / configs[3] as driver-timed sub-objects (1 GPU: rank 0 of an N=1 run; Qwen at every N)
    extra = {}
    if not args.no_extra:
        import bench_workloads
        sub = argparse.Namespace(**vars(args))
        sub.steps, sub.warmup, sub.no_cpu_baseline = max(3, min(K, 10)), 3, True
        if world == 1:
            for key, fn in (("resnet_wino", bench_workloads.run_resnet_wino), ("resnet_direct", bench_workloads.run_resnet_direct)):
                try:
                    extra[key] = fn(sub, ClockSampler, rank=rank, world=world, local_rank=local_rank)
                except Exception as e:
                    extra[key] = {"error": repr(e)[:300]}
        try:
            extra["qwen"] = bench_workloads.run_qwen(sub, ClockSampler, rank=rank, world=world, local_rank=local_rank)
        except Exception as e:
            extra["qwen"] = {"error": repr(e)[:300]}
        if world == 1:
            try:
                extra["qwen_decode"] = bench_workloads.run_qwen_decode(sub, ClockSampler, rank=rank, world=world, local_rank=local_rank)
            except Exception as e:
                extra["qwen_decode"] = {"error": repr(e)[:300]}

    if rank == 0:
        peak, peak_src = measured_peaks()
        achieved = sess.bytes / (ms_per_step / 1e3) / 1e9
        traffic = None
        # dram__bytes_read.sum + dram__bytes_write.sum over the kernels of one step, from the committed ncu capture of this
        # command (tools/prof_traffic.sh); written bytes largely stay in the 126 MB L2 under ncu's per-kernel replay
        for name in ("r02_traffic_mbv2_convpath.json", "r01_traffic_mbv2_convpath.json"):
            tp = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tp):
                traffic = json.load(open(tp)).get("traffic_bytes_per_step")
                break
        use_plugin = bool(plug and plug.get("value"))
        e2e = {"value": plug["value"] if use_plugin else e2e_pipe, "unit": "img/s",
               "h2d_bytes_per_step": (plug.get("h2d_bytes_per_step") if use_plugin else h2d),
               "d2h_bytes_per_step": (plug.get("d2h_bytes_per_step") if use_plugin else d2h),
               "mode": ("WHOLE MobileNet-v2 .mnn (a superset of the 36 convs) through the unmodified MNN Interpreter::runSession on "
                        "libmnn_b200_plugin.so: copyFromHostTensor(fp32 NCHW) + runSession + copyToHostTensor every iteration, "
                        "median window" if use_plugin else
                        "C ABI, depth-2 pipeline: H2D of step k+1 overlaps the kernels of step k (plugin harness unavailable)"),
               "plugin": plug,
               "c_abi_conv_path": {"pipelined_value": e2e_pipe, "serial_value": e2e_serial, "unit": "img/s",
                                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "windows": len(wp),
                                   "note": "the 36-conv session through the C ABI with pinned host buffers; every step copies its own "
                                           "fp32 NCHW input in and its own result out; median of K-step windows over >= 0.5 s"}}
        line = {
            "metric": METRIC,
            "value": value, "unit": "img/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "s8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": BATCH_PER_GPU,
                       "implementation": "sm_100a CUDA through the C ABI: conv-group persistent tcgen05 kernel + stem kernel, CUDA-graph replay",
                       "parallelism": f"dp{world} replicas, NCCL model broadcast at build",
                       "l2": "inputs larger than L2 (240 MB distinct bytes per step)",
                       "graph": not args.no_graph, "numa_node": numa_node},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel": "conv_group_tcgen05_kernel" if sess.group is not None else "gemm_i8_tcgen05_kernel",
                         "algorithmic_bytes_per_step": sess.bytes, "macs_per_step": sess.macs},
            "timing": {"ms_per_step_median_window": ms_median / K, "windows": len(win), "per_rank_ms_per_step": per_rank_ms},
            "e2e": e2e,
            "gpu_launches": gpu_launches, "host_launch_calls": int(host_launches), "kernels_per_step": sess.launches_per_step,
            "clocks": sampler.result(),
            "whole_net": whole,
        }
        line.update(extra)
        if world == 1 and not args.no_cpu_baseline:
            # the CPU-baseline leg (the only place this arm executes anything under oracle/): the reference CPU backend on the
            # same 36 layers at the same batch, bounded to 3 timed passes
            try:
                v, cores, kind, sample = cpu_reference_rate(BATCH_PER_GPU, 3, 1)
                line["cpu_baseline"] = {"value": v, "unit": "img/s", "cores": cores, "kind": kind, "sample": sample, "cpu": cpu_info()}
            except Exception as e:  # never lose the GPU line
                line["cpu_baseline"] = {"value": None, "unit": "img/s", "cores": 0, "kind": "unavailable", "sample": repr(e)[:200]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
