"""Builds libaomarl.so in-tree for sm_100a (nvcc cross-compiles without a GPU).

One object per translation unit (compiled in parallel), linked into one shared library."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libaomarl.so")
SOURCES = ["aomarl.cu", "wfs_umma.cu", "extrude_i8.cu", "denoise_tc.cu"]
HEADERS = ["atmos_kernels.cuh", "gemm_kernels.cuh", "gemm_tc.cuh", "gemm_tc_host.h", "rtc_kernels.cuh", "wfs_kernels.cuh", "wfs_params.cuh", "wind_host.h",
           "wfs_mma.cuh", "wfs_tma.cuh", "wfs_umma.cuh", "wfs_umma_ws.cuh", "wfs_umma_host.h", "extrude_i8.cuh", "extrude_i8_host.h", "geo_kernels.cuh",
           "pupil_sweep.cuh", "denoise_kernels.cuh", "denoise_tc.cuh", "denoise_tc_host.h", "fft16.cuh", "twiddles.cuh", "rng.cuh", "dispatch.h", "../../include/aomarl.h"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]


def _newer(path, than):
    return os.path.exists(path) and os.path.getmtime(path) > than


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(_newer(os.path.join(HERE, f), t) for f in SOURCES + HEADERS)


def _obj(src):
    return os.path.join(HERE, "build", os.path.splitext(src)[0] + ".o")


def _compile(args):
    src, nvcc, verbose = args
    cmd = [nvcc] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", _obj(src)]
    r = subprocess.run(cmd, cwd=HERE, capture_output=True, text=True)
    return src, r


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    hdr_time = max(os.path.getmtime(os.path.join(HERE, h)) for h in HEADERS if os.path.exists(os.path.join(HERE, h)))
    todo = []
    for src in SOURCES:
        o = _obj(src)
        stale = force or not os.path.exists(o) or os.path.getmtime(o) < max(hdr_time, os.path.getmtime(os.path.join(HERE, src)))
        if stale:
            todo.append((src, nvcc, verbose))
    with ThreadPoolExecutor(max_workers=max(1, len(todo))) as ex:
        for src, r in ex.map(_compile, todo):
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on %s:\n%s%s" % (src, r.stdout, r.stderr))
            if verbose:
                print(r.stderr)
    r = subprocess.run([nvcc, "-shared", "-o", LIB] + [_obj(s) for s in SOURCES], cwd=HERE, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
