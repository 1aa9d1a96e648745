"""In-tree build of the CUDA engine: nvcc -> waafle_b200/libwaafle_b200.so (sm_100a only)."""

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = ["wfl_fast.cu", "wfl_pipeline.cu", "wfl_compact.cu", "wfl_parse.cu", "wfl_genecall.cu", "wfl_details.cu", "wfl_inflate.cu",
           "wfl_resident_batch.cu", "wfl_capi.cu"]
HEADERS = [os.path.join(HERE, "csrc", "wfl_device.cuh"), os.path.join(HERE, "csrc", "wfl_warp_common.cuh"),
           os.path.join(HERE, "csrc", "wfl_warp_sort.cuh"),
           os.path.join(HERE, "csrc", "wfl_parser.cuh"), os.path.join(ROOT, "include", "waafle_b200.h")]
LIB = os.path.join(HERE, "libwaafle_b200.so")

NVCC_FLAGS = ["-O3", "-std=c++17", "-diag-suppress=550", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared", "--threads", "4"]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(HERE, "csrc", s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, out=None, defines=()):
    """Compile the engine if the .so is missing or older than its sources; returns its path.
    `out` / `defines`: build a tuning variant (e.g. -DWFL_FAST_CPSM=6) beside the default library."""
    if out is None and not force and not is_stale():
        return LIB
    cmd = [find_nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + ["-I", os.path.join(ROOT, "include"), "-o", out or LIB]
    cmd += [os.path.join(HERE, "csrc", s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True)
    return out or LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
