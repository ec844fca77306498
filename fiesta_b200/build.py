"""In-tree build of libfiesta_b200.so (sm_100a only) with nvcc.  No CPU fallback is built or exists."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libfiesta_b200.so")
SOURCES = ["fb_map.cu", "fb_esdf.cu", "fb_raycast.cu", "fb_exact.cu", "fb_xrelax.cu", "fb_vis.cu", "fb_depth.cu"]
HEADERS = ["fb_common.cuh", "fb_exact.h", "fb_divmagic.h", "fb_buf.h", os.path.join("..", "..", "include", "fiesta_b200.h")]
# -fmad=false: the ray-casting, query and occupancy code must round every fp64 operation exactly like the reference's
# separate multiply and add (ESDFMap.cpp:122-123, 519-537; raycast.cpp:100-107).
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link fiesta_b200/lib/libfiesta_b200.so.  Returns the library path."""
    os.makedirs(LIBDIR, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            # FIESTA_B200_NVCC_FLAGS: extra flags for experiments (use together with --force)
            extra = os.environ.get("FIESTA_B200_NVCC_FLAGS", "").split()
            cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            subprocess.check_call(cmd)
        objs.append(o)
    if force or _stale(LIB, objs):
        subprocess.check_call([_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
