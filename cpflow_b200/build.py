"""Build libcpflow_b200.so (sm_100a) in-tree with nvcc.

    python -m cpflow_b200.build [--force]

The shared library is a plain C-ABI CUDA library (static cudart, no torch / python symbols); it
is git-ignored but travels to the GPU box with the repo snapshot.
"""
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libcpflow_b200.so")

# (the Heisenberg kernels are spread over several translation units - tools/gen_heis_inst.py - because one nvcc per
# source runs in parallel and a single file with all of them took four minutes)
SOURCES = ["program.cpp", "inst_f32.cu", "inst_f64.cu", "inst_layer_f32.cu", "inst_layer_f64.cu",
           "inst_heis_f32.cu", "inst_heis_f64.cu",
           "inst_heis_f32_p0.cu", "inst_heis_f32_p1.cu", "inst_heis_f32_p2.cu", "inst_heis_f32_p3.cu",
           "inst_heis_f64_p0.cu", "inst_heis_f64_p1.cu", "inst_heis_f64_p2.cu", "inst_heis_f64_p3.cu",
           "inst_multi_f32.cu", "inst_multi_f64.cu", "inst_iso_f32.cu", "inst_iso_f64.cu", "capi.cu"]
HEADERS = ["program.hpp", "engine.cuh", "engine_impl.cuh", "launch.cuh", "heis_impl.cuh", "iso_impl.cuh",
           os.path.join(ROOT, "include", "cpflow_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-I" + os.path.join(ROOT, "include"), "-I" + CSRC]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(nvcc, src, extra):
    obj = os.path.join(OBJ, os.path.splitext(src)[0] + ".o")
    deps = [os.path.join(CSRC, src)] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    if _newer(obj, deps):
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-x", "cu", "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return obj, r.stderr
    return obj, ""


def build(force=False, verbose=False, extra_flags=()):
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    nvcc = _nvcc()
    extra = list(extra_flags) + (["-Xptxas", "-v"] if verbose else [])
    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(lambda s: _compile(nvcc, s, extra), SOURCES))
    objs = [o for o, _ in results]
    if verbose:
        for _, log in results:
            sys.stderr.write(log)
    if force or _newer(LIB, objs):
        tmp = LIB + f".tmp{os.getpid()}"     # link aside and rename: a reader never sees a half-written library
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
        os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    lib = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(lib)
