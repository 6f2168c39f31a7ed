"""Build libibt.so (the C-ABI library declared in include/ibt.h) in-tree with nvcc for sm_100a.

    python -m iceberg_tracking_code_b200.build [--force] [--verbose]

The library is self-contained (static cudart) and has no torch / Python types in its ABI.
"""
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libibt.so")
SOURCES = ["core.cu", "gray.cu", "pyramid.cu", "gftt.cu", "lk.cu", "tracks.cu", "utm.cu", "mask.cu", "jpeg.cu", "grid.cu", "scan.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(_HERE, "..", "include", "ibt.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # OpenCV's float arithmetic on this path is unfused; keep ours unfused too (bit-level parity of the
    # 2x2 solves and of the fp64 projection with numpy).
    "-fmad=false",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "-cudart", "static",
]


def nvcc_path():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found; libibt.so cannot be built")
    return p


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ and link libibt.so next to this file.  Returns its path."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = nvcc_path()
    objdir = os.path.join(_HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed on %s:\n%s\n" % (s, out))
        elif verbose or out.strip():
            sys.stderr.write("[%s]\n%s\n" % (s, out))
    if failed:
        raise RuntimeError("building libibt.so failed")
    tmp = LIB_PATH + ".tmp"
    subprocess.check_call([nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
                           "-o", tmp] + objs)
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
