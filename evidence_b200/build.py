"""
In-tree build of librvlnl.so (hand-written sm_100a CUDA behind the C-ABI of include/rvlnl.h).

nvcc cross-compiles without a GPU; the built library is git-ignored but travels with the
working tree to the GPU box.
"""
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_HERE, "csrc", "rvlnl.cu")
SRC_FIP = os.path.join(_HERE, "csrc", "rvfip.cu")
SRC_ORDER = os.path.join(_HERE, "csrc", "rvorder.cu")
SRC_SLICE = os.path.join(_HERE, "csrc", "rvslice.cu")
DEPS = [SRC, SRC_FIP, SRC_ORDER, SRC_SLICE, os.path.join(_HERE, "csrc", "rvl_math.h"),
        os.path.join(_HERE, "csrc", "rvl_sintab.h"),
        os.path.join(os.path.dirname(_HERE), "include", "rvlnl.h")]
OUT = os.path.join(_HERE, "librvlnl.so")

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    # every fused multiply-add in the kernels is written explicitly; never let the compiler
    # contract a*b+c on its own (SURVEY.md 0.5: an FMA-formed mean anomaly breaks parity)
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared",
]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build librvlnl.so")


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False, defines=(), out=None):
    """Compile evidence_b200/csrc/{rvlnl,rvfip,rvorder,rvslice}.cu -> evidence_b200/librvlnl.so for sm_100a.
    ``defines`` / ``out``: an experimental build beside it (``-DNAME=VALUE`` switches of the kernel
    source, loaded through the RVL_LIB environment variable by the measurement tools)."""
    if out is None and not force and not needs_build():
        return OUT
    out = out or OUT
    cmd = ([nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) +
           [f"-D{d}" for d in defines] + ["-o", out, SRC, SRC_FIP, SRC_ORDER, SRC_SLICE])
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out


if __name__ == "__main__":
    print(build(force=True, verbose=True))
