"""In-tree build of libnttb200.so (nvcc, sm_100a only) and of the C++ host harness.

``python ntt-aie_b200/build.py`` or ``__graft_entry__.build()``.  The shared library
lands in ``ntt-aie_b200/lib/`` (git-ignored, travels to the GPU box with gpurun).
nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libnttb200.so")

NVCC = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-fvisibility=hidden",
              "--use_fast_math", "-Xptxas", "-v"] + ARCH + os.environ.get("NTTB200_NVCC_EXTRA", "").split()

SOURCES = ["api.cu", "kernels_generic.cu", "kernels_fused.cu", "kernels_multi.cu",
           "kernels_small.cu", "tables.cu", "kernels_polymul.cu", "kernels_poly.cu", "kernels_tilecol.cu",
           "kernels_rns_eval.cu", "kernels_rns_conv.cu", "kernels_rns_automorph.cu", "kernels_ckks.cu",
           "kernels_packed.cu", "kernels_rns_keyswitch.cu", "kernels_rns_lintrans.cu"]
HEADERS = ["plan.h", "modarith.cuh", "fused_common.cuh", "tile_common.cuh", os.path.join(ROOT, "include", "nttb200.h")]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    hdrs = [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    objs = []

    def compile_one(src: str) -> str:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            cmd = [NVCC] + NVCC_FLAGS + ["-c", s, "-o", o]
            res = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or res.returncode != 0:
                sys.stderr.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
            if res.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}")
            with open(o + ".ptxas.log", "w") as f:
                f.write(res.stderr)
        return o

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ARCH + ["-lcudart_static", "-lcuda", "-lpthread",
                                                          "-ldl", "-lrt"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
            raise RuntimeError("link failed")
    return LIB


def build_host_harness(force: bool = False) -> str:
    """tests/host/ntt_test.cpp: the C++ successor of the reference's src/test.cpp main."""
    src = os.path.join(ROOT, "tests", "host", "ntt_test.cpp")
    exe = os.path.join(ROOT, "tests", "host", "ntt_test")
    if not os.path.exists(src):
        return ""
    oracle_c = os.path.join(ROOT, "oracle", "ntt_oracle.c")
    if force or _stale(exe, [src, oracle_c, os.path.join(ROOT, "include", "nttb200.h"), LIB]):
        obj = os.path.join(ROOT, "tests", "host", "ntt_oracle.o")
        subprocess.run(["gcc", "-O2", "-std=c99", "-c", oracle_c, "-o", obj], check=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), src, obj,
                        "-o", exe, "-L", LIBDIR, "-lnttb200", f"-Wl,-rpath,{LIBDIR}",
                        "-Wl,-rpath,$ORIGIN/../../ntt-aie_b200/lib", "-lpthread"], check=True)
    return exe


if __name__ == "__main__":
    print(build_library(verbose="-v" in sys.argv, force="-f" in sys.argv))
    print(build_host_harness(force="-f" in sys.argv))
