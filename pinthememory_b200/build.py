"""Build the sm_100a kernel library in-tree: ``pinthememory_b200/_lib/libpinmem_b200.so``.

Plain ``nvcc`` (cross-compiles without a GPU), one object per ``csrc/*.cu`` built in parallel, then a
shared link. The ``.so`` is git-ignored but travels to the GPU box with the tree.

    python -m pinthememory_b200.build [--force] [--verbose]
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libpinmem_b200.so")
SOURCES = ["pm_read.cu", "pm_read_tiled.cu", "pm_score.cu", "pm_readloss.cu", "pm_write.cu", "pm_write_tiled.cu", "pm_bn.cu", "pm_fold.cu", "pm_gemm.cu", "pm_losses.cu", "pm_labels.cu", "pm_readloss8.cu", "pm_readloss10.cu", "pm_segeval.cu", "pm_upcat.cu", "pm_ordered.cu", "pm_exchange.cu", "pm_bn_exchange.cu"]
ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-lineinfo", "-std=c++17", "--use_fast_math=false", "-Xcompiler", "-fPIC"]


def _nvcc():
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; cannot build libpinmem_b200.so")
    return cand


def _deps():
    files = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(CSRC, "pm_common.cuh"), os.path.join(CSRC, "pm_internal.h"), os.path.join(CSRC, "pm_tma.cuh"), os.path.join(CSRC, "pm_umma.cuh"),
                                                         os.path.join(PKG_DIR, "..", "include", "pinmem_b200.h")]
    return files


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > t for f in _deps())


def _compile_one(nvcc, src, obj, verbose):
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    cmd = [nvcc, *ARCH_FLAGS, *flags, "-c", src, "-o", obj]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    return r.stderr


def build(force=False, verbose=False):
    """Compile (if stale) and return the path of the shared library."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(LIB_DIR, exist_ok=True)
    objs = [os.path.join(LIB_DIR, s.replace(".cu", ".o")) for s in SOURCES]
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        futs = [ex.submit(_compile_one, nvcc, os.path.join(CSRC, s), o, verbose) for s, o in zip(SOURCES, objs)]
        logs = [f.result() for f in futs]
    if verbose:
        for lg in logs:
            sys.stderr.write(lg)
    tmp = LIB_PATH + ".tmp"
    r = subprocess.run([nvcc, *ARCH_FLAGS, "-shared", "-o", tmp, *objs], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
