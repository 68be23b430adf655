"""In-tree build of libmgbx.so (nvcc, sm_100a only).  The .so is git-ignored but travels to the GPU box.

One translation unit per responsibility, compiled in parallel and cached as objects under build/; each kernel header is
compiled by one unit only, so that a host-only edit rebuilds one object:
  mgbx.cu          the C ABI, handle life cycle and NCCL communicator (no kernels)
  setup.cu         plans, systems and problem upload             (setup_kernels.cuh)
  evaluate.cu      f0/f1, Hessian assembly, level chain, vectors   (kernels.cuh, dense_kernels.cuh)
  linear_solve.cu  preconditioner setup, direct and PCG solves     (solver_kernels.cuh)
  newton.cu        Newton, mgb_step, matched t (no kernels)
  pcg2.cu          the persistent solve kernel k_pcg2"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libmgbx.so")
HDR = os.path.join("..", "..", "include", "mgbx.h")
# headers every host unit includes (engine.hpp and what it pulls in)
ENGINE = ["engine.hpp", "host_sparse.hpp", "device_common.cuh", "elem_schur.cuh", "node_barrier.cuh", "pcg2.hpp", HDR]
# source -> files whose change forces a recompile of that source
SOURCES = {
    "mgbx.cu": ["mgbx.cu", "host_amg.hpp"] + ENGINE,
    "setup.cu": ["setup.cu", "setup_kernels.cuh"] + ENGINE,
    "evaluate.cu": ["evaluate.cu", "kernels.cuh", "dense_kernels.cuh"] + ENGINE,
    "linear_solve.cu": ["linear_solve.cu", "solver_kernels.cuh"] + ENGINE,
    "newton.cu": ["newton.cu"] + ENGINE,
    "pcg2.cu": ["pcg2.cu", "pcg2.hpp"],
}
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-DNDEBUG", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unused-function"]


def nvcc_path():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _obj(src):
    return os.path.join(OBJ, os.path.splitext(src)[0] + ".o")


def _stale(src):
    o = _obj(src)
    if not os.path.exists(o):
        return True
    t = os.path.getmtime(o)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in SOURCES[src])


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(_stale(s) or os.path.getmtime(_obj(s)) > t for s in SOURCES)


def _compile(src, verbose):
    cmd = [nvcc_path()] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", _obj(src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return src, r


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    todo = [s for s in SOURCES if force or _stale(s)]
    with ThreadPoolExecutor(max_workers=max(1, len(todo))) as ex:
        for src, r in ex.map(lambda s: _compile(s, verbose), todo):
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError("nvcc failed compiling %s" % src)
            if verbose:
                print(r.stdout + r.stderr)
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", LIB] + [_obj(s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed linking libmgbx.so")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
