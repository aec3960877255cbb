"""Build libsqpb200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

The active-set kernel is compiled once per team size (qp_solve_inst.cu with -DQP_TEAM/-DQP_CTA), the
object files in parallel.  -fmad=false: FP64 multiply-adds are not contracted, so the solve kernel's
arithmetic is operation-for-operation the CPU oracle's and the L0 kernels' sums are the reference's
(SpHbMat::times evaluates val*x then +=); parity tests can therefore compare bit patterns.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libsqpb200.so")
OBJDIR = os.path.join(HERE, "build")
HEADERS = [os.path.join(CSRC, f) for f in ("qp_kernel.cuh", "l0_kernels.cuh", "tma.cuh")] + [
    os.path.join(os.path.dirname(HERE), "include", "sqpb200.h")]
# (threads per QP, threads per CTA, warps per SM the registers are capped for): one warp per QP, 4/2/1 QPs per CTA
TEAMS = [(32, 128, 16), (32, 64, 16), (32, 32, 16), (32, 128, 32),
         # sub-warp teams: 16 / 8 lanes per QP (2 / 4 QPs per warp) for QPs with nV <= 16 / <= 8
         (16, 128, 16), (8, 128, 16)]
QP_EXTRA_FLAGS = os.environ.get("SQPB200_QP_FLAGS", "").split()
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
              "-Xcompiler", "-fPIC"]


def _nvcc():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return nvcc if os.path.exists(nvcc) else "nvcc"


def _units():
    units = [(os.path.join(CSRC, "capi.cu"), os.path.join(OBJDIR, "capi.o"), []),
             (os.path.join(CSRC, "nlp_eval.cu"), os.path.join(OBJDIR, "nlp_eval.o"), []),
             (os.path.join(CSRC, "sqp_outer.cu"), os.path.join(OBJDIR, "sqp_outer.o"), [])]
    for team, cta, wps in TEAMS:
        # multi-warp teams are compiled fully inlined (see the QP_INLINE_ALL note in qp_kernel.cuh)
        units.append((os.path.join(CSRC, "qp_solve_inst.cu"), os.path.join(OBJDIR, "qp_solve_%d_%d_w%d.o" % (team, cta, wps)),
                      ["-DQP_TEAM=%d" % team, "-DQP_CTA=%d" % cta, "-DQP_WPS=%d" % wps] + QP_EXTRA_FLAGS))
    units.append((os.path.join(CSRC, "qp_solve_large_inst.cu"), os.path.join(OBJDIR, "qp_solve_large.o"), QP_EXTRA_FLAGS))
    return units


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


# the C++ batched host driver (csrc/driver): BatchedAlgorithm + its command-line front end, linked against the library
DRIVER = os.path.join(LIBDIR, "batched_sqp")
DRIVER_SRC = [os.path.join(CSRC, "driver", f) for f in ("BatchedAlgorithm.cpp", "batched_sqp_main.cpp")]
DRIVER_DEPS = DRIVER_SRC + [os.path.join(CSRC, "driver", "BatchedAlgorithm.hpp"), HEADERS[-1]]


def is_stale():
    return _stale(LIB, [u[0] for u in _units()] + HEADERS + [os.path.abspath(__file__)]) or _stale(DRIVER, DRIVER_DEPS + [LIB])


def build_driver(force=False):
    """g++-level C++ (no device code): compiled by nvcc's host compiler, linked with libsqpb200.so and the CUDA runtime."""
    if not force and not _stale(DRIVER, DRIVER_DEPS + [LIB]):
        return DRIVER
    cmd = [_nvcc(), "-O2", "-std=c++17", "-I" + os.path.join(os.path.dirname(HERE), "include"), "-o", DRIVER] + DRIVER_SRC + [
        "-L" + LIBDIR, "-lsqpb200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("driver build failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return DRIVER


def build(force=False, verbose=False):
    """Compile the CUDA extension if it is missing or older than its sources.  Returns the .so path."""
    if not force and not _stale(LIB, [u[0] for u in _units()] + HEADERS + [os.path.abspath(__file__)]):
        build_driver()
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(u):
        src, obj, defs = u
        if not force and not _stale(obj, [src] + HEADERS + [os.path.abspath(__file__)]):
            return ""
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + defs + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    with ThreadPoolExecutor(max_workers=len(_units())) as ex:
        logs = list(ex.map(compile_one, _units()))
    cmd = [nvcc, "-shared", "-o", LIB] + [u[1] for u in _units()] + ["-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print("\n".join(logs))
    build_driver(force=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
