"""In-tree build of ``libaft_b200.so`` (sm_100a only) with plain nvcc.

``python -m adafortitran_b200.build`` or :func:`build`.  The shared object lands in
``adafortitran_b200/lib/`` (git-ignored, but it travels to the GPU box with the gpurun snapshot).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(PKG, "build")
LIB_DIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIB_DIR, "libaft_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libaft_b200.so cannot be built (there is no non-CUDA fallback)")


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


VARIANTS = {
    # name -> extra nvcc defines.  "chaos": every mbarrier wait of the tensor-core kernels is preceded by a pseudo-random
    # delay (tc_ptx.cuh), which shakes the relative timing of the kernel's roles; used by the protocol test
    # (tests/test_gpu_bf16.py::test_protocol_under_random_delays) through AFT_B200_LIB.  "tl": the tensor-core kernels
    # record in-kernel timelines (aft_selftest 102 / 103), read by tools/tc_check.py timeline and tools/conv_ab.sh.
    "chaos": ["-DAFT_TC_CHAOS"],
    "tl": ["-DAFT_TC_TIMELINE"],
}


def lib_file(variant: str | None = None) -> str:
    return LIB if not variant else os.path.join(LIB_DIR, f"libaft_b200_{variant}.so")


def build(force: bool = False, verbose: bool = False, variant: str | None = None) -> str:
    """Compile every ``csrc/*.cu`` for sm_100a and link ``libaft_b200.so`` (or a named variant).  Returns its path."""
    obj = os.path.join(PKG, f"build_{variant}") if variant else OBJ   # one object directory per variant
    lib = lib_file(variant)
    defs = VARIANTS[variant] if variant else []
    os.makedirs(obj, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(PKG), "include", "aft.h"))
    nvcc = _nvcc()
    stamp = os.path.join(obj, "defs.stamp")
    if not os.path.exists(stamp) or open(stamp).read() != " ".join(defs):
        force = True     # the compile-time switches changed: rebuild everything
        with open(stamp, "w") as f:
            f.write(" ".join(defs))
    jobs = []
    for src in sources():
        s = os.path.join(CSRC, src)
        o = os.path.join(obj, src[:-3] + ".o")
        if force or _stale(o, [s] + headers):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + defs + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(obj, os.path.basename(s) + ".log")
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return o

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            list(ex.map(compile_one, jobs))
    objs = [os.path.join(obj, s[:-3] + ".o") for s in sources()]
    if force or jobs or _stale(lib, objs):
        cmd = [nvcc, "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib


if __name__ == "__main__":
    var = next((a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")), None)
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, variant=var))
