"""Builds libzstdb200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libzstdb200.so")
SOURCES = ["api.cu", "decode_kernels.cu", "encode_kernels.cu", "dict_train.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-O2,-Wall", "-diag-suppress", "20091", "--cudart", "static",
]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for root, _, files in os.walk(CSRC):
        for f in files:
            if os.path.getmtime(os.path.join(root, f)) > t:
                return True
    return os.path.getmtime(os.path.join(HERE, "..", "include", "zstdb200.h")) > t


def build(force=False, verbose=False, extra=None, out=None):
    """extra / out: development aid — a variant build (e.g. extra=["-DZB_EXEC_DEBUG"]) written next to the product
    library and loaded with ZSTDB200_LIB=<path>."""
    lib = out or LIB
    if not force and not extra and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    bdir = os.path.join(HERE, "_build" if not out else "_build_" + os.path.basename(out))
    os.makedirs(bdir, exist_ok=True)
    for s in SOURCES:
        o = os.path.join(bdir, s.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (extra or []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", o]
        subprocess.run(cmd, check=True)
        objs.append(o)
    cmd = [nvcc, "-shared", "-o", lib] + objs + ["--cudart", "static", "-Xlinker", "--no-undefined", "-lpthread", "-ldl", "-lrt"]
    subprocess.run(cmd, check=True)
    return lib


if __name__ == "__main__":
    if "--variant" in sys.argv:      # e.g. --variant c12 -DEXEC_MIN_CTAS=12
        i = sys.argv.index("--variant")
        print(build(force=True, extra=sys.argv[i + 2:], out=os.path.join(HERE, "libzstdb200_%s.so" % sys.argv[i + 1]), verbose="-v" in sys.argv))
    elif "--debug" in sys.argv:
        print(build(force=True, extra=["-DZB_EXEC_DEBUG"], out=os.path.join(HERE, "libzstdb200_dbg.so")))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
