#!/usr/bin/env python3
"""Builds libmnn_b200_plugin.so -- the MNN_FORWARD_CUDA plugin (b200_plugin.cpp) -- with g++ against the reference's headers
(MNN_REFERENCE; nothing is copied) into the directory given on the command line.  Links libmnn_b200.so (the C ABI) only: the
MNN core symbols it uses (MNNInsertExtraRuntimeCreator, TensorUtils, ConvolutionCommon, ...) stay undefined and resolve
against whichever libMNN.so the host process has loaded -- that is what makes it a plugin.  It needs the reference headers,
so the project builds it beside the reference core that hosts it, and it travels with that build."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("MNN_REFERENCE", "/root/reference")


def build(out_dir):
    out = os.path.join(os.path.abspath(out_dir), "libmnn_b200_plugin.so")
    if not os.path.isdir(REF):
        print("[build_plugin] reference headers absent; keeping the prebuilt plugin", file=sys.stderr)
        return out if os.path.exists(out) else None
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(HERE, "b200_plugin.cpp")
    inc = ["include", "source", "schema/current", "3rd_party/flatbuffers/include", "3rd_party"]
    cmd = ["g++", "-std=gnu++11", "-O2", "-fPIC", "-shared", "-fno-rtti", "-fno-exceptions", "-fvisibility=hidden", "-w",
           "-DMNN_USE_SSE", "-o", out, src] + ["-I" + os.path.join(REF, i) for i in inc] + \
          ["-L" + PKG, "-lmnn_b200", "-Wl,-rpath,$ORIGIN/" + os.path.relpath(PKG, os.path.dirname(out))]
    subprocess.check_call(cmd)
    print("[build_plugin] wrote", out)
    return out


if __name__ == "__main__":
    build(sys.argv[1])
