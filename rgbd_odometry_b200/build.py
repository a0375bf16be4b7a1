"""In-tree build of the sm_100a CUDA library (libdvo_b200.so) and the host-side helpers.

nvcc cross-compiles without a GPU, so this runs in the CPU-only build container as well as on a B200 box.
The .so files are git-ignored but travel to the GPU box with the working tree.
"""
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libdvo_b200.so")
SYNTH_SRC = os.path.join(PKG, "synth", "synth.cpp")
SYNTH_LIB = os.path.join(PKG, "synth", "libdvo_synth.so")
HOST_DIR = os.path.join(PKG, "host")
HOST_LIB = os.path.join(PKG, "libdvo_host.so")


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libdvo_b200.so cannot be built and there is no CPU fallback")


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def cuda_sources():
    srcs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(".cu")]
    deps = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(".cuh")]
    deps.append(os.path.join(ROOT, "include", "dvo_b200.h"))
    return srcs, deps


# per-file extra flags: the photometric path mirrors the oracle's fp64 operation order, so no FMA contraction there
PER_FILE_FLAGS = {"photometric.cu": ["-fmad=false"], "rgbd.cu": ["-fmad=false"], "frontend.cu": ["-fmad=false"]}
COMPILE_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC,-ffp-contract=off"]
OBJ_DIR = os.path.join(PKG, "build")


def build_cuda(force=False, verbose=False):
    srcs, deps = cuda_sources()
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs, relink = [], force or not os.path.exists(LIB)
    for src in srcs:
        name = os.path.basename(src)
        obj = os.path.join(OBJ_DIR, name[:-3] + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + deps):
            extra = os.environ.get("DVO_NVCC_EXTRA", "").split()          # experiments only (e.g. preprocess.cu's -DDVO_NMS_* knobs)
            cmd = [_nvcc()] + COMPILE_FLAGS + PER_FILE_FLAGS.get(name, []) + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
            subprocess.check_call(cmd, cwd=CSRC)
            relink = True
    if relink or _stale(LIB, objs):
        subprocess.check_call([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", LIB] + objs)
    return LIB


def build_synth(force=False):
    if force or _stale(SYNTH_LIB, [SYNTH_SRC]):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", SYNTH_LIB, SYNTH_SRC])
    return SYNTH_LIB


def build_host(force=False):
    """C++ classes mirroring the reference API (SolveDVO, EPoseEstimator, PyramidalStorageStruct, GOP) + their C test shim."""
    if not os.path.isdir(HOST_DIR):
        return None
    srcs = [os.path.join(HOST_DIR, f) for f in sorted(os.listdir(HOST_DIR)) if f.endswith(".cpp")]
    if not srcs:
        return None
    deps = [os.path.join(HOST_DIR, f) for f in sorted(os.listdir(HOST_DIR)) if f.endswith(".h")]
    deps.append(os.path.join(ROOT, "include", "dvo_b200.h"))
    build_cuda()
    if force or _stale(HOST_LIB, srcs + deps + [LIB]):
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-I", HOST_DIR, "-o", HOST_LIB] + srcs + \
              ["-L", PKG, "-ldvo_b200", "-Wl,-rpath,$ORIGIN"]
        subprocess.check_call(cmd)
    return HOST_LIB


def build_all(force=False):
    build_cuda(force)
    build_synth(force)
    build_host(force)


if __name__ == "__main__":
    import sys
    build_all(force="--force" in sys.argv)
    print("built:", LIB)
