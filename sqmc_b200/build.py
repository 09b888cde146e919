"""Compile libsqmc_b200.so for sm_100a with nvcc (in-tree, no JIT cache).

The element / build translation unit is compiled with --fmad=false: the pattern
test abs(H) > 1e-12 of the reference (chemistry.f90:9901) must see the same
floating-point values as the reference's non-FMA x86-64 build.
"""
import glob
import os
import shutil
import site
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libsqmc_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nccl_paths():
    """Prefer the NCCL that PyTorch loads (pip nvidia-nccl) so one process never holds two NCCLs."""
    for sp in site.getsitepackages():
        inc = os.path.join(sp, "nvidia", "nccl", "include")
        lib = os.path.join(sp, "nvidia", "nccl", "lib")
        if os.path.exists(os.path.join(inc, "nccl.h")) and glob.glob(os.path.join(lib, "libnccl.so*")):
            return inc, lib
    return "/usr/include", "/usr/lib/x86_64-linux-gnu"


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")) +
                  glob.glob(os.path.join(CSRC, "*.h")) + [os.path.join(HERE, "..", "include", "sqmc_b200.h")])


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    inc, lib = _nccl_paths()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    common = [nvcc, "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-I", inc, "--expt-relaxed-constexpr",
              "--expt-extended-lambda"] + ARCH
    if verbose:
        common += ["-Xptxas", "-v"]
    units = [("build.cu", ["--fmad=false"]), ("select.cu", ["--fmad=false"]), ("spmv.cu", []), ("convert.cu", []), ("bundle.cu", []), ("p2p.cu", []), ("growbuf.cu", []), ("local.cu", []), ("davidson.cu", []), ("rdm.cu", []), ("api.cu", [])]
    objs = []
    procs = []
    for name, extra in units:
        obj = os.path.join(objdir, name.replace(".cu", ".o"))
        objs.append(obj)
        procs.append((name, subprocess.Popen(common + extra + ["-c", os.path.join(CSRC, name), "-o", obj],
                                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for name, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("---- nvcc %s ----\n%s\n" % (name, out))
        failed = failed or p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libsqmc_b200.so")
    libnccl = os.path.basename(sorted(glob.glob(os.path.join(lib, "libnccl.so*")))[0])
    cmd = [nvcc, "-shared", "-o", OUT] + objs + ARCH + ["-Xlinker", "-rpath", "-Xlinker", lib, "-L", lib,
                                                        "-l:" + libnccl, "-lcudart"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
