"""Build libbevfusion_b200.so (sm_100a) in-tree with nvcc.  No torch involved: the library is a
plain C-ABI shared object (include/bevfusion_b200.h) that links only the static CUDA runtime."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libbevfusion_b200.so")
SOURCES = ["common.cu", "bevpool.cu", "bevpool_lift.cu", "voxelize.cu", "scatter.cu", "depthmap.cu", "rulebook.cu", "spconv_simt.cu", "spconv_tc.cu", "spconv_v6.cu", "encoder.cu", "spconv_bwd.cu", "spconv_wgrad_tc.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
         "-Xptxas", "-warn-spills"]


def _stale(obj, src):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(HERE, "..", "include", "bevfusion_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIB_DIR, exist_ok=True)
    objdir = os.path.join(LIB_DIR, "obj")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, src):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    failed = False
    for s, p in procs:
        out = p.communicate()[0].decode()
        if p.returncode != 0 or verbose or "warning" in out.lower():
            sys.stderr.write("[nvcc %s]\n%s\n" % (s, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if procs or not os.path.exists(LIB):
        cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
