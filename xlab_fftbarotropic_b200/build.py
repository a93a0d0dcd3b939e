"""In-tree build of the CUDA library (sm_100a only) and of the host C++ programs.

  libxfb.so        csrc/xfb_row.cu + xfb_col.cu + xfb_api.cu + xfb_dist.cu + xfb_generic.cu + xfb_spectra.cu  (the C ABI of include/xfb.h)

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with gpurun snapshots.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
BUILD = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libxfb.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
CUDA_SOURCES = ["xfb_row.cu", "xfb_col.cu", "xfb_api.cu", "xfb_dist.cu", "xfb_generic.cu", "xfb_spectra.cu"]
HEADERS = ["xfb_fft.cuh", "xfb_row.cuh", "xfb_rowpair.cuh", "xfb_rowpair2l.cuh", "xfb_col.cuh", "xfb_colt.cuh", "xfb_col2l.cuh", "xfb_internal.h", "xfb_handle.h", os.path.join(ROOT, "include", "xfb.h")]


def _mtime(p):
    return os.path.getmtime(p) if os.path.exists(p) else 0.0


def _compile(src):
    obj = os.path.join(BUILD, os.path.splitext(src)[0] + ".o")
    log = os.path.join(BUILD, os.path.splitext(src)[0] + ".ptxas.log")
    deps = [os.path.join(CSRC, src)] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    if _mtime(obj) >= max(_mtime(d) for d in deps):
        return obj
    r = subprocess.run([NVCC, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj], capture_output=True, text=True)
    with open(log, "w") as fh:
        fh.write(r.stdout + r.stderr)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError(f"nvcc failed on {src}")
    return obj


def build_library(force: bool = False) -> str:
    os.makedirs(BUILD, exist_ok=True)
    if force:
        for s in CUDA_SOURCES:
            o = os.path.join(BUILD, os.path.splitext(s)[0] + ".o")
            if os.path.exists(o):
                os.remove(o)
    with ThreadPoolExecutor(max_workers=len(CUDA_SOURCES)) as ex:
        objs = list(ex.map(_compile, CUDA_SOURCES))
    if _mtime(LIB) < max(_mtime(o) for o in objs):
        r = subprocess.run([NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-ldl"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


HOST = os.path.join(CSRC, "host")
BIN = os.path.join(HERE, "bin")
GENERATORS = {"makefield-elliptic-vortex": 1, "makefield-const-vortex": 2, "makefield-gaussian": 3, "makefield-Kuo2004": 4}


def _gxx(out, sources, extra=()):
    deps = sources + [os.path.join(HOST, f) for f in os.listdir(HOST)] + [os.path.join(ROOT, "include", "xfb.h")]
    if _mtime(out) >= max(_mtime(d) for d in deps) and _mtime(out) >= _mtime(LIB):
        return out
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-o", out, *sources, *extra]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError(f"g++ failed on {out}")
    return out


def build_host() -> dict:
    """Host C++ programs (I/O and control only; all arithmetic goes through libxfb.so):
    bin/main.out, bin/invert_pres.out, bin/makefield-*.out"""
    build_library()
    os.makedirs(BIN, exist_ok=True)
    fio = os.path.join(HOST, "fieldio.cpp")
    link = ["-L", HERE, "-lxfb", "-Wl,-rpath,$ORIGIN/.."]
    out = {}
    out["main"] = _gxx(os.path.join(BIN, "main.out"), [os.path.join(HOST, "main.cpp"), fio], link)
    out["invert_pres"] = _gxx(os.path.join(BIN, "invert_pres.out"), [os.path.join(HOST, "invert_pres.cpp"), fio], link)
    for name, gen in GENERATORS.items():
        out[name] = _gxx(os.path.join(BIN, name + ".out"), [os.path.join(HOST, "makefield.cpp"), fio], [f"-DXFB_GEN={gen}"])
    return out


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv))
    print(build_host())
