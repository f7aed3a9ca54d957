"""Build libttg_b200.so (the C-ABI library) in-tree with nvcc for sm_100a.

    python falcon-ttdforgnns_b200/build.py [--force] [--verbose]

One object per .cu (compiled in parallel), linked into lib/libttg_b200.so.  No torch headers
are involved: the library is plain CUDA runtime + CUB.  nvcc cross-compiles without a GPU.
"""
import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libttg_b200.so")
SOURCES = ["api.cu", "tt_generic.cu", "tt_sorted.cu", "tt_mma.cu", "tt_tc5.cu", "tt_rmma.cu", "cache.cu", "spmm.cu", "sampler.cu", "gat.cu", "peer.cu", "reorder.cu", "rcm.cu", "kway_host.cu", "kway.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "tc5.cuh"), os.path.join(HERE, "..", "include", "ttg_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: the CUDA extension cannot be built")
    return nvcc


def _digest(paths):
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _compile(src, verbose):
    obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
    stamp = obj + ".sha"
    dig = _digest([os.path.join(CSRC, src)] + HEADERS)
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
        return obj, False, ""
    cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    with open(stamp, "w") as f:
        f.write(dig)
    with open(obj + ".ptxas.log", "w") as f:
        f.write(r.stderr)
    return obj, True, r.stderr if verbose else ""


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    if force:
        for f in os.listdir(OBJDIR):
            os.remove(os.path.join(OBJDIR, f))
    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    objs = [r[0] for r in results]
    changed = any(r[1] for r in results)
    for r in results:
        if r[2]:
            print(r[2])
    if changed or not os.path.exists(LIB):
        cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                        "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    lib = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(lib)
