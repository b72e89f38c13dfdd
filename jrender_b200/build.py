"""In-tree build of libb200raster.so (hand-written sm_100a CUDA, C ABI in include/b200raster.h).

    python -m jrender_b200.build [--force] [--verbose]

Flags: -gencode arch=compute_100a,code=sm_100a (B200 only), -lineinfo (ncu source view),
-fmad=false (no a*b+c contraction: see csrc/common.cuh for the arithmetic contract; IEEE
division / sqrt are nvcc defaults and must not be weakened -- no --use_fast_math).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libb200raster.so")
SOURCES = ["softras_api.cu", "softras_fwd.cu", "softras_bwd.cu",
           "nmr_api.cu", "preraster_api.cu", "mesh_loss_api.cu", "lighting_api.cu", "bake_api.cu", "sss_api.cu", "api_util.cu", "debug_api.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]
OBJDIR = os.path.join(HERE, "lib", "obj")


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _deps():
    out = []
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h")):
                out.append(os.path.join(root, f))
    return out


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(f) > t for f in _deps() + [os.path.abspath(__file__)])


def build_variant(name, defines, verbose=False):
    """Development A/B aid: lib/libb200raster_<name>.so compiled with extra -D flags (selected at
    run time with B200R_LIB=<path>).  The product library is always libb200raster.so."""
    from concurrent.futures import ThreadPoolExecutor
    objdir = os.path.join(OBJDIR, name)
    os.makedirs(objdir, exist_ok=True)
    out = os.path.join(LIBDIR, "libb200raster_%s.so" % name)

    def one(src):
        obj = os.path.join(objdir, src[:-3] + ".o")
        cmd = [_nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", "-o", obj, os.path.join(CSRC, src)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr))
        if verbose:
            print(r.stderr)
        return obj
    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(one, SOURCES))
    subprocess.run([_nvcc(), "-shared", "-o", out] + objs, check=True)
    return out


def build(force=False, verbose=False):
    """Compile every translation unit to an object file (in parallel), then link the .so."""
    if not force and not stale():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJDIR, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    headers = [f for f in _deps() if not f.endswith(".cu")] + [os.path.abspath(__file__)]
    hdr_time = max(os.path.getmtime(h) for h in headers)

    def compile_one(src):
        obj = os.path.join(OBJDIR, os.path.basename(src)[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_time):
            return obj, ""
        cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, r.stderr))
        return obj, r.stderr
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        results = list(ex.map(compile_one, srcs))
    if verbose:
        for _, log in results:
            if log:
                print(log)
    cmd = [_nvcc(), "-shared", "-o", LIB] + [o for o, _ in results]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    if "--variant" in sys.argv:  # python -m jrender_b200.build --variant NAME -DX=1 -DY=2
        k = sys.argv.index("--variant")
        print(build_variant(sys.argv[k + 1], [a[2:] for a in sys.argv if a.startswith("-D")], verbose="--verbose" in sys.argv))
    else:
        print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
