"""In-tree build of ``libparcels_b200.so`` with nvcc for sm_100a (no other target, no fallback)."""

from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["engine.cu", "afast.cu", "agrid.cu", "aslip.cu", "rk45.cu", "advdiff.cu", "hashbuild.cu", "cgrid.cu", "curva.cu"]  # one translation unit per kernel family: compiled in parallel
# Per-source tuning (measured on B200, profiles/README.md): the A-grid kernel runs best with its corner
# cache in shared memory (float64 copies on float64 grids) and <= 128 registers (4 blocks of 128 threads per SM).
EXTRA_FLAGS = {"afast.cu": ["-DPB_BLOCK=128", "-DPB_MINBLOCKS=3", "-DPB_SMEM_CACHE"], "agrid.cu": ["-DPB_MINBLOCKS=4", "-DPB_SMEM_CACHE"], "aslip.cu": ["-DPB_MINBLOCKS=4", "-DPB_SMEM_CACHE"],
               "rk45.cu": ["-DPB_MINBLOCKS=3", "-DPB_SMEM_CACHE"], "advdiff.cu": ["-DPB_SMEM_CACHE"],
               "cgrid.cu": ["-DPB_MINBLOCKS=3"], "curva.cu": ["-DPB_MINBLOCKS=3"]}  # fmt: skip
DEPS = [os.path.join(CSRC, f) for f in (*SOURCES, "common.cuh", "agrid.cuh", "rk45.cuh", "cgrid.cuh")]
OUT = os.path.join(HERE, "lib", "libparcels_b200.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "parcels_b200.h")

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-fmad=false",  # no FMA contraction: arithmetic must round exactly like the reference's NumPy ops
    "-Xcompiler", "-fPIC",
]  # fmt: skip


def needs_build(out: str = OUT) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(f) > t for f in (*DEPS, HEADER, __file__))


def build(force: bool = False, verbose: bool = False, out: str = OUT) -> str:
    """Compile the library to ``out`` (object files go to ``obj/`` beside it); returns ``out``."""
    if not force and not needs_build(out):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    objdir = os.path.join(os.path.dirname(out), "obj")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *EXTRA_FLAGS.get(src, []), *(["-Xptxas", "-v"] if verbose else []), "-c", "-o", obj,
               os.path.join(CSRC, src)]  # fmt: skip
        procs.append((cmd, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    objs = []
    for cmd, obj, p in procs:
        stdout, err = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed:\n{' '.join(cmd)}\n{stdout}\n{err}")
        if verbose:
            print(err)
        objs.append(obj)
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, *objs, "-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{' '.join(cmd)}\n{res.stdout}\n{res.stderr}")
    return out


if __name__ == "__main__":
    print(build(force=True, verbose=True))
