"""Build shacira_b200/libshacira_b200.so (the C-ABI library) with nvcc for sm_100a.

In-tree, no torch dependency, no JIT cache: the .so is git-ignored but travels to the GPU
box with the gpurun snapshot. `python -m shacira_b200.build [-v] [--force]`.
"""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libshacira_b200.so")
SOURCES = ["capi.cu", "tiled_capi.cu", "grid3d_capi.cu", "session_capi.cu", "peer_capi.cu", "nerf_heads_capi.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3",
]


def _deps():
    d = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".inl", ".h"))]
    d.append(os.path.join(os.path.dirname(PKG), "include", "shacira_b200.h"))
    d.append(os.path.abspath(__file__))
    return d


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _deps())


def build(force=False, verbose=False, extra=(), out=None, tag=""):
    """`out`/`tag`/`extra` build tuning variants beside the product library (see benchmarks/)."""
    global LIB
    if out is None and not force and not is_stale():
        return LIB
    lib_path = out or LIB
    # one object per translation unit, compiled in parallel, then one link
    from concurrent.futures import ThreadPoolExecutor
    objdir = os.path.join(PKG, "build" + tag)
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src + ".o")
        cmd = ["nvcc", "-c"] + NVCC_FLAGS + list(extra) + [os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    link = ["nvcc", "--shared", "-gencode", "arch=compute_100a,code=sm_100a"] + objs + ["-o", lib_path]
    if verbose:
        print(" ".join(link), flush=True)
    subprocess.check_call(link)
    return lib_path


if __name__ == "__main__":
    extra = ["-Xptxas", "-v"] if "--ptxas" in sys.argv else []
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, extra=extra))
