"""Builds svdsolver_b200/libsvdb200.so (the C-ABI library over the sm_100a kernels) in-tree with nvcc.

nvcc cross-compiles without a GPU; the built .so travels to the GPU box with the repo snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsvdb200.so")
SOURCES = ["capi.cu", "stage1_panel.cu", "stage1_panel_reg.cu", "stage1_panel_blk.cu", "stage1_panel_chol.cu", "stage1_tile.cu", "gemm.cu", "gemm_fast.cu", "gemm_tc05.cu", "stage2_chase.cu", "stage2_chase_fast.cu", "bidiag_qr.cu", "bidiag_bisect.cu", "bidiag_sqr.cu", "dist.cu", "rect.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr",
]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(dp, f) for dp, _, fs in os.walk(CSRC) for f in fs]
    deps += [os.path.join(HERE, "..", "include", f) for f in ("svdb200.h", "svdb200_matrix.hpp")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra=(), out=None, only=None):
    """out / only: instrumented side builds (e.g. -DSVDB_PANEL_TIMING=1) into another file, recompiling only the listed sources"""
    if out is not None:
        return _build_variant(out, extra, only or SOURCES)
    if not force and not needs_build():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for s in SOURCES:
        o = os.path.join(HERE, "build", s.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {s} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-ldl"])
    build_cli()
    return LIB


def _build_variant(out, extra, only):
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    objs, procs = [], []
    for s in SOURCES:
        if s in only:
            o = os.path.join(bdir, s.replace(".cu", ".var.o"))
            procs.append(subprocess.Popen([_nvcc(), *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, s), "-o", o]))
        else:
            o = os.path.join(bdir, s.replace(".cu", ".o"))
        objs.append(o)
    if any(p.wait() != 0 for p in procs):
        raise RuntimeError("nvcc failed")
    subprocess.check_call([_nvcc(), "-shared", "-o", out, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-ldl"])
    return out


CLI = os.path.join(HERE, "bin", "svd_b200")


def build_cli():
    """Host-only C++ driver (reference CLI contract) over include/svdb200_matrix.hpp + libsvdb200.so."""
    os.makedirs(os.path.dirname(CLI), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(HERE, "..", "include"),
                           os.path.join(CSRC, "cli", "svd_b200.cpp"), "-o", CLI,
                           "-L", HERE, "-lsvdb200", "-Wl,-rpath,$ORIGIN/.."])
    return CLI


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
