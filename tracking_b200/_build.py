"""In-tree build of libbgsb200.so with nvcc for sm_100a (no torch, no JIT cache).

    python -m tracking_b200._build [--force]

The shared library is written next to this file so that it travels to the GPU box with the
repository snapshot.  Model kernels need OpenCV's unfused fp32 arithmetic, so the whole library
is compiled with -fmad=false (the one fused operation of the reference is an explicit fmaf).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJDIR = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libbgsb200.so")
SOURCES = ["capi.cu", "simple_bgs.cu", "mog2.cu", "mog2_t1.cu", "dpz.cu", "dp_simple.cu", "synth.cu", "morph.cu", "ccl.cu", "blobdetect.cu", "pipeline.cu", "pool.cu",
           os.path.join("ingest", "yuv420.cu")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
         "-Xcompiler", "-fPIC,-fvisibility=hidden", "-Xptxas", "-v"]


def _deps():
    d = [os.path.join(base, f) for base, _, names in os.walk(CSRC) for f in names]
    d.append(os.path.join(HERE, "..", "include", "bgsb200.h"))
    return d


def _obj_name(src):
    """ingest/yuv420.cu -> ingest__yuv420.o: one flat object directory for sources in subdirectories"""
    return src.replace(os.sep, "__").replace(".cu", ".o")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _deps())


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJDIR, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    keep = {_obj_name(s) for s in srcs} | {"ptxas.log"}
    for f in os.listdir(OBJDIR):                 # objects of sources that no longer exist must not travel to the GPU box
        if f not in keep:
            os.remove(os.path.join(OBJDIR, f))
    def cc(src):
        obj = os.path.join(OBJDIR, _obj_name(src))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=8) as ex:
        results = list(ex.map(cc, srcs))
    log = "".join(r[1] for r in results)
    with open(os.path.join(OBJDIR, "ptxas.log"), "w") as f:
        f.write(log)
    if verbose:
        sys.stderr.write(log)
    cmd = [NVCC, "-shared", "-o", LIB, *[r[0] for r in results], "-Xcompiler", "-fPIC", "-cudart", "static", "-lpthread", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
