"""Build ``libvfk.so`` in-tree with nvcc for sm_100a (``python -m vfclik_b200.build``)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libvfk.so")
OBJ_DIR = os.path.join(os.path.dirname(HERE), "build", "obj")
# one translation unit per (precision, joint-count group) of the cycle kernel, one per precision of its vfk_solve variant and
# of the shared-scene step and solve variants, and the ABI: compiled in parallel
UNITS = ["vfk_api", "vfk_cycle_f32_small", "vfk_cycle_f32_large", "vfk_cycle_f64_small", "vfk_cycle_f64_large", "vfk_solve_f32",
         "vfk_solve_f64", "vfk_shared_f32", "vfk_shared_f64", "vfk_shared_solve_f32", "vfk_shared_solve_f64"]
SOURCES = [os.path.join(CSRC, u + ".cu") for u in UNITS]
HEADERS = [os.path.join(CSRC, f) for f in ("vfk_kernels.cuh", "vfk_math.cuh", "vfk_tma.cuh", "vfk_nullspace.cuh", "vfk_split.cuh", "vfk_ctx.cuh", "vfk_launch.cuh", "vfk_ring.cuh")] + [
    os.path.join(os.path.dirname(HERE), "include", "vfk.h")]
DEPS = SOURCES + HEADERS

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]   # cudart linked statically (nvcc default)


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def up_to_date() -> bool:
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(d) <= t for d in DEPS)


def build_library(force: bool = False, verbose: bool = False, extra_flags=(), out: str = OUT) -> str:
    """Compile the translation units in parallel (one nvcc process each) and link them into ``out``."""
    if not force and out == OUT and up_to_date():
        return OUT
    nvcc = find_nvcc()
    tag = "default" if out == OUT else os.path.splitext(os.path.basename(out))[0]
    obj_dir = os.path.join(OBJ_DIR, tag)
    os.makedirs(obj_dir, exist_ok=True)
    flags = NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else [])
    procs = []
    for unit, src in zip(UNITS, SOURCES):
        obj = os.path.join(obj_dir, unit + ".o")
        cmd = [nvcc] + flags + ["-c", "-o", obj, src]
        procs.append((unit, obj, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs, failed = [], []
    for unit, obj, cmd, proc in procs:
        log = proc.communicate()[0]
        if verbose or proc.returncode != 0:
            sys.stderr.write(log)
        if proc.returncode != 0:
            failed.append(" ".join(cmd))
        objs.append(obj)
    if failed:
        raise RuntimeError("nvcc failed: %s" % failed[0])
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out] + objs
    res = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout)
        raise RuntimeError("link failed: %s" % " ".join(link))
    return out


if __name__ == "__main__":
    extra = [a for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[len("--out="):] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build_library(force="--force" in sys.argv or bool(extra) or bool(outs), verbose="-v" in sys.argv, extra_flags=extra,
                        out=outs[0] if outs else OUT))
