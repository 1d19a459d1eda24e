"""Build libmpb200.so (the sm_100a CUDA library behind include/mpb200.h) in-tree with nvcc.

Run as a script (`python motionplanning.jl_b200/build.py`) or call build_lib() -- this is what
__graft_entry__.build() does.  The .so lands next to the sources so it travels with the tree.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libmpb200.so")
SOURCES = ["api.cu", "grid_rball.cu", "collide.cu", "lq.cu", "mc.cu", "brute_rball.cu", "tc_rball.cu", "order.cu", "xchg.cu", "peaks.cu", "lq_general.cu", "closest.cu", "knn.cu", "cars.cu", "gmt.cu", "gmt_lqg.cu", "shortcut.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    # the reference rounds after every operation; parity kernels additionally use explicit
    # __dmul_rn/__dadd_rn intrinsics, this flag covers everything else
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared",
]


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build_lib(force=False, verbose=False):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(HERE, "..", "include", "mpb200.h"))
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest(deps):
        return LIB
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libmpb200.so cannot be built")
    # one nvcc per translation unit, in parallel (no relocatable device code: device functions are header-inline,
    # only host functions cross translation units), then one link
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])
    with tempfile.TemporaryDirectory(prefix="mpb200_build_") as tmp:
        objs = [os.path.join(tmp, os.path.basename(src)[:-3] + ".o") for src in srcs]

        def compile_one(args):
            src, obj = args
            return subprocess.run([nvcc] + compile_flags + ["-c", src, "-o", obj], capture_output=True, text=True)

        with ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 1)) as pool:
            results = list(pool.map(compile_one, zip(srcs, objs)))
        for src, res in zip(srcs, results):
            if res.returncode != 0:
                raise RuntimeError("nvcc failed on %s:\n%s%s" % (os.path.basename(src), res.stdout, res.stderr))
            if verbose:
                print(res.stderr)
        res = subprocess.run([nvcc, "-shared", "-o", LIB] + objs, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
