"""Build oracle/_ref/libjrender_ref_sss.so from the reference's OWN subsurface-scattering blur kernel (TEST
INFRASTRUCTURE).

Same recipe as oracle/build_ref.py: the `cuda_header` of _blur_for_SSS (jrender/renderer/utils/gaussian_blur.py:34-165)
is captured where it lies under /root/reference through a stub `jittor` module, a hand-written launcher restates its
`cuda_src`, and both are compiled for sm_100a with nvcc defaults (fmad on, as a stock nvcc/Jittor build would).

    python -m oracle.build_ref_sss

Outputs only into oracle/_ref/ (git-ignored).  Used to generate tests/golden/sss_ref_gpu_blur_*.npz on a B200
(oracle/make_ref_sss_golden.py) and to time the reference's blur on the same GPU (tools/bench_sss.py).
"""
import os
import subprocess
import sys

from oracle.build_ref import OUT, PREAMBLE, REFERENCE, _capture

LIB = os.path.join(OUT, "libjrender_ref_sss.so")

LAUNCH_SSS_BLUR = r'''
// ---- launcher: restates cuda_src of _blur_for_SSS (renderer/utils/gaussian_blur.py:143-165): 32x32 blocks, dim 0 runs
// the y kernel and dim 1 the x kernel.  The output is zero-initialised (jt.zeros_like, :6).  Depth d = 1: every SSS()
// call blurs a 2-D map.  No synchronisation, so that the 36 launches of one SSS() call can be timed back to back.
extern "C" int ref_sss_blur(const float* image, const float* modulate, const float* gauss, float* out, int h, int w,
                            int tap_num, float gauss_width, int dim, cudaStream_t st) {
    cudaMemsetAsync(out, 0, sizeof(float) * (size_t)h * w, st);
    const dim3 block(32, 32);
    const dim3 grid((w - 1) / block.x + 1, (h - 1) / block.y + 1);
    if (dim == 0)
        gaussain_blur_y_Kernel<float32><<<grid, block, 0, st>>>(image, modulate, gauss, out, tap_num, gauss_width, h, w, 1);
    else if (dim == 1)
        gaussain_blur_x_Kernel<float32><<<grid, block, 0, st>>>(image, modulate, gauss, out, tap_num, gauss_width, h, w, 1);
    return (int)cudaGetLastError();
}
'''


def generate():
    os.makedirs(OUT, exist_ok=True)
    hdr = _capture(os.path.join(REFERENCE, "jrender/renderer/utils/gaussian_blur.py"), "_blur_for_SSS", 7)
    text = PREAMBLE + hdr + LAUNCH_SSS_BLUR
    path = os.path.join(OUT, "ref_sss_blur.cu")
    if not os.path.exists(path) or open(path).read() != text:
        open(path, "w").write(text)
    return path


def build(force=False, verbose=False):
    if not os.path.isdir(REFERENCE):
        raise RuntimeError("%s not present: use the prebuilt oracle/_ref" % REFERENCE)
    path = generate()
    if not force and os.path.exists(LIB) and max(os.path.getmtime(path), os.path.getmtime(os.path.abspath(__file__))) <= os.path.getmtime(LIB):
        return LIB
    cmd = ["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-w", "-Xcompiler", "-fPIC", "-shared", "-o", LIB, path]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB


def available():
    return os.path.exists(LIB)


def lib():
    """The reference blur launcher: ref_sss_blur(image, modulate, taps, out, h, w, tap_num, gauss_width, dim, stream)."""
    import ctypes as C
    if not available():
        raise RuntimeError("%s not built (python -m oracle.build_ref_sss where the reference is present)" % LIB)
    L = C.CDLL(LIB)
    L.ref_sss_blur.restype = C.c_int
    L.ref_sss_blur.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]
    return L


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
