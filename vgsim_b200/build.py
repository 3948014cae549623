"""Builds libvgsim_b200.so in-tree with nvcc for sm_100a (no torch extension machinery needed:
the library has a plain C ABI and is loaded with ctypes)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvgsim_b200.so")
SOURCES = ["capi.cu", "tau_kernel.cu", "prep_kernels.cu", "direct_kernel.cu", "direct_large_kernel.cu", "genealogy_kernel.cu", "curves_kernel.cu", "lineages_kernel.cu", "archive_kernel.cu", "param_grid_kernel.cu", "resample_kernel.cu", "test_taps.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def have_nvcc():
    import shutil
    n = _nvcc()
    return os.path.exists(n) if os.path.isabs(n) else shutil.which(n) is not None


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "vgsim_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"]
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== %s ==\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([nvcc, "-shared", "-o", LIB] + objs + ["-lcudart_static", "-ldl", "-lrt", "-lpthread"])
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
