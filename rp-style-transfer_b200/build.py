"""Build librpst.so in-tree with nvcc for sm_100a (no torch headers, plain C ABI)."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "librpst.so")
DEBUG_LIB = os.path.join(PKG, "librpst_debug.so")    # same sources + -DRPST_DEBUG_EXPORTS: white-box test hooks only
DEBUG_SOURCES = ("adain.cu", "nsroot.cu", "seg.cu", "wct.cu")               # translation units that carry a debug export

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build() -> bool:
    if not os.path.exists(LIB) or not os.path.exists(DEBUG_LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(ROOT, "include", "*.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into one shared library; returns its path."""
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(PKG, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    objs, procs = [], []
    dbg_objs = []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        if os.path.basename(src) in DEBUG_SOURCES:
            dobj = obj[:-2] + ".dbg.o"
            dbg_objs.append(dobj)
            procs.append((src, subprocess.Popen([nvcc, *NVCC_FLAGS, "-DRPST_DEBUG_EXPORTS", "-c", src, "-o", dobj],
                                                stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        else:
            dbg_objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    # shared cudart: the static runtime would embed every runtime entry point (batch-memcpy names included) in the
    # shipped binary; torch has libcudart.so.12 loaded already, the rpath covers a bare ctypes load
    shared_rt = ["--cudart", "shared", "-Xlinker", "-rpath=/usr/local/cuda/lib64"]
    link = [nvcc, "-shared", "-o", LIB + ".tmp", *objs, "-gencode", "arch=compute_100a,code=sm_100a", *shared_rt, "-lcuda"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        # libcuda may be absent on a GPU-less build box: the driver API is resolved at run time
        link = link[:-1]
        r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    os.replace(LIB + ".tmp", LIB)
    r = subprocess.run([nvcc, "-shared", "-o", DEBUG_LIB + ".tmp", *dbg_objs, "-gencode", "arch=compute_100a,code=sm_100a", *shared_rt],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link of librpst_debug.so failed")
    os.replace(DEBUG_LIB + ".tmp", DEBUG_LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
