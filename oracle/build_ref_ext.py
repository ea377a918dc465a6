"""Recipe: build the UNMODIFIED reference CUDA extension `selective_scan_cuda_core` for sm_100a.

    SIGMA_REFERENCE_DIR=<checkout of the original Sigma project> python oracle/build_ref_ext.py [--force]

Compiles the reference's own sources where they lie (<checkout>/models/encoders/selective_scan/
csrc/selective_scan/*.{cpp,cu}) with the reference's own flags (setup.py:80-99) — the only change is
the target architecture (setup.py:56-62 lists sm_70/80/90; a B200 needs compute_100a).  Output:
oracle/_ref/selective_scan_cuda_core.so (git-ignored).  Nothing is copied into the repo.  Without
SIGMA_REFERENCE_DIR the recipe does nothing.

It is the GPU baseline ("the reference kernel on the same box", SURVEY.md §8c(3)); used by
scripts/bench_vs_ref_ext.py, tests/golden/make_ref_ext_golden.py and bench.py's `gpu_baseline` only.
"""
import os
import subprocess
import sys
import sysconfig
from concurrent.futures import ThreadPoolExecutor

import torch
from torch.utils.cpp_extension import include_paths, library_paths

SRC = os.path.join(os.environ.get("SIGMA_REFERENCE_DIR", ""), "models", "encoders", "selective_scan", "csrc", "selective_scan")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
NAME = "selective_scan_cuda_core"


def main():
    if not os.environ.get("SIGMA_REFERENCE_DIR") or not os.path.isdir(SRC):
        print("reference sources not present; keeping whatever is in", OUT)
        return 0
    os.makedirs(os.path.join(OUT, "build"), exist_ok=True)
    so = os.path.join(OUT, NAME + ".so")
    srcs = ["selective_scan.cpp", "selective_scan_core.cu", "selective_scan_core_fwd2.cu",
            "selective_scan_core_fwd3.cu", "selective_scan_core_fwd4.cu"]
    newest = max(os.path.getmtime(os.path.join(SRC, f)) for f in os.listdir(SRC))
    if os.path.exists(so) and os.path.getmtime(so) > newest and "--force" not in sys.argv:
        print("up to date:", so)
        return 0
    inc = [f"-I{p}" for p in include_paths("cuda")] + [f"-I{SRC}", f"-I{sysconfig.get_paths()['include']}"]
    common = ["-O3", "-std=c++17", f"-DTORCH_EXTENSION_NAME={NAME}", "-DTORCH_API_INCLUDE_EXTENSION_H",
              f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}"]
    nvcc_flags = ["-U__CUDA_NO_HALF_OPERATORS__", "-U__CUDA_NO_HALF_CONVERSIONS__",
                  "-U__CUDA_NO_BFLOAT16_OPERATORS__", "-U__CUDA_NO_BFLOAT16_CONVERSIONS__",
                  "-U__CUDA_NO_BFLOAT162_OPERATORS__", "-U__CUDA_NO_BFLOAT162_CONVERSIONS__",
                  "--expt-relaxed-constexpr", "--expt-extended-lambda", "--use_fast_math",
                  "--ptxas-options=-v", "-lineinfo",
                  "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC"]

    def compile_one(f):
        obj = os.path.join(OUT, "build", f + ".o")
        if f.endswith(".cu"):
            cmd = ["nvcc", "-c", os.path.join(SRC, f), "-o", obj] + common + nvcc_flags + inc
        else:
            cmd = ["g++", "-c", os.path.join(SRC, f), "-o", obj, "-fPIC"] + common + inc
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".log", "w") as fh:
            fh.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode:
            raise RuntimeError(f"{f}: {r.stderr[-2000:]}")
        return obj

    with ThreadPoolExecutor(5) as ex:
        objs = list(ex.map(compile_one, srcs))
    libs = [f"-L{p}" for p in library_paths("cuda")]
    cmd = ["g++", "-shared", "-o", so] + objs + libs + ["-lc10", "-ltorch_cpu", "-ltorch", "-ltorch_python",
                                                         "-lc10_cuda", "-ltorch_cuda", "-lcudart"]
    subprocess.run(cmd, check=True)
    print("built", so)
    return 0


if __name__ == "__main__":
    sys.exit(main())
