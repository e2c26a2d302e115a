"""Builds ip_mcmc_b200/libipmcmc.so (hand-written sm_100a CUDA + the C ABI of include/ipmcmc.h).

nvcc cross-compiles without a GPU.  The library is built IN-TREE so it travels to the GPU box
with the repo snapshot; it is git-ignored.
"""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libipmcmc.so")
OBJ = os.path.join(PKG, "_build")
# Translation units: the C ABI + Lorenz + small kernels, and the Burgers kernels once per cells-per-lane value AND
# numerics (0 = the team kernels for 2048 / 4096 cells, one unit).  They compile in parallel, and an edit to one kernel
# family cannot move the code generated for another: with EXACT and FUSED in one unit, an edit to EXACT-only templates
# changed the inlining of the FUSED chain kernel (round 2; the split units reproduce the measured FUSED SASS bit for bit).
UNITS = ([("engine", "engine.cu", [])]
         + [("burgers_cpl%d_%s" % (c, "fused" if num else "exact"), "burgers_inst.cu",
             ["-DIPMCMC_TU_CPL=%d" % c, "-DIPMCMC_TU_NUM=%d" % num]) for c in (32, 16, 8, 7, 4, 2, 1) for num in (1, 0)]
         + [("burgers_cpl0", "burgers_inst.cu", ["-DIPMCMC_TU_CPL=0"])])
# No --split-compile: with it ptxas' output is not reproducible (the schedule of the Burgers time-step loop
# came out in one of two variants, 15 % apart in throughput, from one build of the same source to the next).
CFLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
          "--extended-lambda", "-Xcompiler", "-fPIC"]
NVCC_FLAGS = CFLAGS      # (name kept for tools/)


# headers each kind of unit includes: a unit is recompiled when its object, and the library is relinked when it,
# is older than the unit's source or any of them
_COMMON = ["common.cuh", "philox.cuh", "sampler.cuh", "sched.cuh", "burgers.cuh", "burgers_launch.cuh",
           os.path.join("..", "..", "include", "ipmcmc.h")]
DEPS = {"engine.cu": _COMMON + ["diag.cuh", "lorenz.cuh", "lorenz_kernels.cuh", "tempering.cuh"],
        "burgers_inst.cu": _COMMON + ["burgers_kernels.cuh", "burgers_team.cuh", "burgers_launch_impl.cuh"]}


def _mtime(f):
    return os.path.getmtime(os.path.join(CSRC, f))


def _unit_stale(unit, obj_dir):
    name, src, _ = unit
    obj = os.path.join(obj_dir, name + ".o")
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return any(_mtime(f) > t for f in [src] + DEPS[src])


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(_mtime(f) > t for src, deps in DEPS.items() for f in [src] + deps)


def compile_units(out_lib, extra_flags=(), obj_dir=None, verbose=False, force=True):
    """nvcc -c every (stale) translation unit in parallel, then link them into out_lib."""
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "nvcc")
    obj_dir = obj_dir or OBJ
    os.makedirs(obj_dir, exist_ok=True)

    def one(unit):
        name, src, defs = unit
        obj = os.path.join(obj_dir, name + ".o")
        if not force and not _unit_stale(unit, obj_dir):
            return obj
        cmd = [nvcc] + CFLAGS + list(extra_flags) + defs + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), r.stderr[-4000:]))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max(1, min(len(UNITS), os.cpu_count() or 1))) as ex:
        objs = list(ex.map(one, UNITS))
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out_lib] + objs
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (" ".join(cmd), r.stderr[-4000:]))
    return out_lib


def build(force=False, verbose=False):
    """Compile the library if it is missing or older than its sources. Returns the path."""
    if not force and not _stale():
        return LIB
    return compile_units(LIB, verbose=verbose, force=force)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
