"""In-tree build of ``libtaco_b200.so`` (hand-written sm_100a CUDA + C ABI).

``nvcc`` cross-compiles without a GPU; the resulting shared object sits next
to this file so that it travels with the repository snapshot to the GPU box.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtaco_b200.so")
OBJ_DIR = os.path.join(CSRC, "build")

SOURCES = ["gather.cu", "conv_umma.cu", "elementwise.cu", "bigru.cu", "bigru_mma.cu", "decoder.cu", "decoder_cw.cu", "griffin_lim.cu", "spectrogram.cu", "resample.cu", "durations.cu", "taco_abi.cu"]
HEADERS = ["common.cuh", "kernels.cuh", "fft2048.cuh", "decoder_cw.h", "decoder_cw_pack.inc", os.path.join("..", "..", "include", "taco_b200.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile every ``csrc/*.cu`` for sm_100a and link ``libtaco_b200.so``.
    Returns the library path.  Skips up-to-date objects."""
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            jobs.append([nvcc, *NVCC_FLAGS, "-Xptxas", "-v" if verbose else "-warn-spills", "-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for log in ex.map(run, jobs):
                if verbose and log:
                    sys.stderr.write(log)
    if force or jobs or _stale(LIB, objs):
        run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs])
    return LIB


TORCH_OPS_SRC = os.path.join(CSRC, "torch_ops.cpp")
TORCH_OPS_LIB = os.path.join(HERE, "libtaco_b200_torch.so")


def build_torch_ops(force: bool = False) -> str:
    """Compile ``csrc/torch_ops.cpp`` (TORCH_LIBRARY(taco_b200, ...): the C ABI as PyTorch custom operators) with g++ against
    the installed torch headers and link it to ``libtaco_b200.so`` (rpath $ORIGIN).  Load with ``torch.ops.load_library``."""
    build_library()
    if not force and not _stale(TORCH_OPS_LIB, [TORCH_OPS_SRC, LIB, os.path.join(HERE, "..", "include", "taco_b200.h")]):
        return TORCH_OPS_LIB
    import torch
    from torch.utils import cpp_extension as ce
    inc = []
    for d in ce.include_paths("cuda") if hasattr(ce, "include_paths") else []:
        inc += ["-I", d]
    cuda_home = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    inc += ["-I", os.path.join(cuda_home, "include")]
    tlib = os.path.join(os.path.dirname(torch.__file__), "lib")
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI),
           "-DTORCH_API_INCLUDE_EXTENSION_H", *inc, TORCH_OPS_SRC, "-o", TORCH_OPS_LIB,
           "-L", tlib, "-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda", "-ltorch",
           "-L", HERE, "-l:libtaco_b200.so", "-Wl,-rpath,$ORIGIN", "-Wl,-rpath," + tlib]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout, r.stderr))
    return TORCH_OPS_LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
    if "--torch-ops" in sys.argv:
        print(build_torch_ops(force="--force" in sys.argv))
