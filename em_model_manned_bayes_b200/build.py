"""In-tree build of libemb200.so (sm_100a only) with explicit nvcc; no JIT cache, no torch extension.

    python -m em_model_manned_bayes_b200.build [--force] [--verbose]

The shared library lands next to this file so that it travels with a `gpurun` snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libemb200.so")

CU_SOURCES = ["emb_kernels.cu", "emb_terminal.cu"]
CXX_SOURCES = ["emb_model.cpp", "emb_api.cpp", "emb_multi.cpp"]
HEADERS = ["emb_device.cuh", "emb_fast.cuh", "emb_initial.cuh", "emb_terminal.cuh", "emb_integrate.cuh", "emb_loglik.cuh", "emb_loglik_events.cuh", "emb_events_expand.cuh", "emb_exact.cuh", "emb_format.cuh", "emb_parse.cuh", "emb_model.h", "emb_launch.h", os.path.join(ROOT, "include", "emb200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off", "--expt-relaxed-constexpr",
]
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall", "-Wno-unused-function", "-Wno-unknown-pragmas"]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; libemb200.so cannot be built")
    return cand


def _cuda_include() -> str:
    return os.path.join(os.path.dirname(os.path.dirname(_nvcc())), "include")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("build step failed: " + " ".join(cmd))
    if verbose and (r.stdout or r.stderr):
        print(r.stdout + r.stderr)
    return r


def build_variant(name: str, defines) -> str:
    """Scratch builds for kernel tuning: libemb200_<name>.so with extra -D flags (load it with EMB200_LIB=<path>)."""
    out = os.path.join(HERE, "libemb200_%s.so" % name)
    objs = []
    os.makedirs(OBJ, exist_ok=True)
    for src in CU_SOURCES:
        o = os.path.join(OBJ, "%s.%s.o" % (src, name))
        _run([_nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + ["-c", os.path.join(CSRC, src), "-o", o], False)
        objs.append(o)
    for src in CXX_SOURCES:
        objs.append(os.path.join(OBJ, src + ".o"))
    _run([_nvcc(), "-shared", "-o", out] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lpthread", "-ldl"], False)
    return out


def build(force: bool = False, verbose: bool = False, ptxas_info: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    objs = []
    for src in CU_SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            extra = ["-Xptxas", "-v"] if ptxas_info else []
            jobs.append([_nvcc()] + NVCC_FLAGS + extra + ["-c", s, "-o", o])
    for src in CXX_SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            jobs.append(["g++"] + CXX_FLAGS + ["-I", _cuda_include(), "-c", s, "-o", o])
    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            results = list(ex.map(lambda c: _run(c, verbose or ptxas_info), jobs))
        if ptxas_info:
            for r in results:
                sys.stdout.write(r.stderr)
    if jobs or force or _stale(LIB, objs):
        _run([_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lpthread", "-ldl"], verbose)
    return LIB


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--variant":
        build()
        print(build_variant(sys.argv[2], sys.argv[3:]))
        sys.exit(0)
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, ptxas_info="--ptxas" in sys.argv)
    print(path)
