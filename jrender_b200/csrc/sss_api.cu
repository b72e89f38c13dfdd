// sss_api.cu -- texture-space subsurface scattering: the stretch map and the stretch-modulated Gaussian blur chain of
// the reference's SSS() (jrender/renderer/lighting/lighting.py:86-156, renderer/utils/ToStretchMap.py,
// renderer/utils/gaussian_blur.py:34-165).
//
//   b200r_sss_blur_chain  <-  computeStretchMap + the 36 _blur_for_SSS launches + the weighted sum of the three basis
//                             images, `* irradiance + specular` and the vertical flip (lighting.py:115-150)
//   b200r_sss_blur        <-  one _blur_for_SSS launch (d = 1), the building block of the chain
//
// The reference recomputes the stretch chain once per colour channel from clones; every redo yields the same maps, so
// the chain is computed once here.  Seven launches in all: the stretch map, then per variance one x pass and one y pass.
// A pass blurs the stretch map (modulated by itself) and, at the same pixel, the three irradiance channels (modulated
// by the stretch value just computed: the reference reads the modulate map only at the centre texel).
//
// Arithmetic: the library builds with -fmad=false; the reference, built by nvcc with defaults, contracts the tap
// interpolation and the tap accumulation into FFMA (cuobjdump -sass of both reference kernels on sm_100a):
//   interpolation = fma(c2 - c, v1, (c - c1) * v2)      v = fma(interpolation, tap[k], v)
// and those two are written with __fmaf_rn here.  The start position `c - nfw * 6 / 2` is an FMUL followed by an FFMA
// with -0.5, which rounds exactly like the unfused expression (the product by 0.5 is exact).  Tap positions advance by
// the same sequential `+= nfw` as the reference: a closed form moves int() across integer boundaries.
#include "../../include/b200raster.h"
#include "api_util.cuh"

namespace {

constexpr int kTaps = 7;

struct SssTaps {
    float tap[kTaps];
    float width;
};

// One output texel of gaussain_blur_{x,y}_Kernel with d = 1: `src` is the map, `centre` = src[pixel], `pos` the pixel's
// coordinate along the blur axis, `stride` the element distance of one step along it, `nfw` the net filter width.
__device__ __forceinline__ float blur_texel(const float* __restrict__ line, float centre, int pos, int stride, int n, float nfw,
                                            const SssTaps& t) {
    if (!(centre > 0.f)) return 0.f;                      // the mask loop: `l` reads the centre texel (d = 1)
    float c = (float)pos - nfw * (float)(kTaps - 1) / 2.f;
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < kTaps; k++) {
        int c1 = (int)c, c2 = (int)c + 1;                 // truncation, then clamp
        c1 = c1 < 0 ? 0 : (c1 > n - 1 ? n - 1 : c1);
        c2 = c2 < 0 ? 0 : (c2 > n - 1 ? n - 1 : c2);
        float v1 = __ldg(line + (size_t)c1 * stride);
        float v2 = __ldg(line + (size_t)c2 * stride);
        v1 = (double)v1 > 1e-6 ? v1 : centre;             // double literal in the reference
        v2 = (double)v2 > 1e-6 ? v2 : centre;
        const float interp = __fmaf_rn((float)c2 - c, v1, __fmul_rn(c - (float)c1, v2));
        v = __fmaf_rn(interp, t.tap[k], v);
        c = c + nfw;
    }
    return v;
}

__device__ __forceinline__ float blur_at(const float* __restrict__ src, const float* __restrict__ modulate, int x, int y, int n,
                                         int dim, const SssTaps& t) {
    const size_t id = (size_t)y * n + x;
    const float nfw = t.width * __ldg(modulate + id);
    if (dim == 1) return blur_texel(src + (size_t)y * n, __ldg(src + id), x, 1, n, nfw, t);
    return blur_texel(src + x, __ldg(src + id), y, n, n, nfw, t);
}

// computeStretchMap(worldcoord * 7): 1 / ||p - right neighbour|| (U) and 1 / ||p - lower neighbour|| (V), replicate
// padding, clamped to [0, 1] (a zero difference gives inf -> 1).  world: planar [>=3, S, S].
__global__ void __launch_bounds__(256) k_sss_stretch(const float* __restrict__ world, float* __restrict__ su, float* __restrict__ sv, int S) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= S) return;
    const size_t plane = (size_t)S * S, id = (size_t)y * S + x;
    const size_t right = (size_t)y * S + min(x + 1, S - 1), below = (size_t)min(y + 1, S - 1) * S + x;
    float du = 0.f, dv = 0.f;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const float p = __ldg(world + c * plane + id) * 7.f;
        const float a = p - __ldg(world + c * plane + right) * 7.f;
        const float b = p - __ldg(world + c * plane + below) * 7.f;
        du = du + a * a;
        dv = dv + b * b;
    }
    su[id] = fminf(fmaxf(1.f / sqrtf(du), 0.f), 1.f);
    sv[id] = fminf(fmaxf(1.f / sqrtf(dv), 0.f), 1.f);
}

// One fused pass of one variance and direction: s_out = blur(s_in, modulate s_in); irr_out[c] = blur(irr_in[c],
// modulate s_out) at the same pixel.  The y pass of variance i also accumulates the basis image into acc with weight
// wgt[c] (step 0 starts from zero); the last one writes out[S-1-y][x][c] = (acc + w * basis) * irradiance + specular.
enum { kAccNone = 0, kAccFirst = 1, kAccAdd = 2, kAccFinal = 3 };

template <int DIM, int ACC>
__global__ void __launch_bounds__(256)
k_sss_blur_pass(const float* __restrict__ s_in, float* __restrict__ s_out, const float* __restrict__ irr_in,
                float* __restrict__ irr_out, float* __restrict__ acc, const float* __restrict__ irradiance,
                const float* __restrict__ specular, float* __restrict__ out, int S, SssTaps t, float3 wgt) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= S) return;
    const size_t plane = (size_t)S * S, id = (size_t)y * S + x;
    const float s = blur_at(s_in, s_in, x, y, S, DIM, t);
    s_out[id] = s;
    const float nfw = t.width * s;
    const float w[3] = {wgt.x, wgt.y, wgt.z};
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const float* src = irr_in + c * plane;
        const float b = DIM == 1 ? blur_texel(src + (size_t)y * S, __ldg(src + id), x, 1, S, nfw, t)
                                 : blur_texel(src + x, __ldg(src + id), y, S, S, nfw, t);
        if (ACC == kAccFinal) {
            const float f = __fadd_rn(__ldg(acc + c * plane + id), __fmul_rn(w[c], b));
            out[((size_t)(S - 1 - y) * S + x) * 3 + c] =
                __fadd_rn(__fmul_rn(f, __ldg(irradiance + c * plane + id)), __ldg(specular + c * plane + id));
        } else {
            irr_out[c * plane + id] = b;
            if (ACC == kAccFirst) acc[c * plane + id] = __fadd_rn(0.f, __fmul_rn(w[c], b));
            if (ACC == kAccAdd) acc[c * plane + id] = __fadd_rn(acc[c * plane + id], __fmul_rn(w[c], b));
        }
    }
}

__global__ void __launch_bounds__(256)
k_sss_blur_one(const float* __restrict__ image, const float* __restrict__ modulate, float* __restrict__ out, int S, int dim, SssTaps t) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= S) return;
    out[(size_t)y * S + x] = blur_at(image, modulate, x, y, S, dim, t);
}

SssTaps make_taps(const float* taps, float width) {
    SssTaps t;
    for (int k = 0; k < kTaps; k++) t.tap[k] = taps[k];
    t.width = width;
    return t;
}

dim3 grid_of(int S) { return dim3((unsigned)((S + 255) / 256), (unsigned)S); }

}  // namespace

extern "C" size_t b200r_sss_workspace_bytes(int image_size) {
    if (image_size <= 0) return 0;
    return (size_t)image_size * image_size * sizeof(float) * 13;
}

extern "C" int b200r_sss_blur(const float* image, const float* modulate, float* out, int image_size, const float* taps,
                              float gauss_width, int dim, void* stream) {
    if (!image || !modulate || !out || !taps) return b200r_fail(B200R_EINVAL, "b200r_sss_blur: NULL pointer argument");
    if (image_size <= 0) return b200r_fail(B200R_EINVAL, "b200r_sss_blur: non-positive image_size");
    if (dim != 0 && dim != 1) return b200r_fail(B200R_EINVAL, "b200r_sss_blur: dim %d is neither 0 (y) nor 1 (x)", dim);
    cudaStream_t st = (cudaStream_t)stream;
    {
        B200rProfScope prof(B200R_K_SSS, st);
        k_sss_blur_one<<<grid_of(image_size), 256, 0, st>>>(image, modulate, out, image_size, dim, make_taps(taps, gauss_width));
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return b200r_cuda_fail(e, "k_sss_blur_one");
    return 0;
}

extern "C" int b200r_sss_blur_chain(const float* worldcoord_map, const float* irradiance_map, const float* specular_map,
                                    float* final_map, void* workspace, size_t workspace_bytes, int image_size,
                                    const float* taps, const float* gauss_widths, const float* weights, void* stream) {
    if (!worldcoord_map || !irradiance_map || !specular_map || !final_map || !workspace || !taps || !gauss_widths || !weights)
        return b200r_fail(B200R_EINVAL, "b200r_sss_blur_chain: NULL pointer argument");
    if (image_size <= 0) return b200r_fail(B200R_EINVAL, "b200r_sss_blur_chain: non-positive image_size");
    if (workspace_bytes < b200r_sss_workspace_bytes(image_size))
        return b200r_fail(B200R_EWORKSPACE, "b200r_sss_blur_chain: workspace %zu < %zu bytes", workspace_bytes,
                          b200r_sss_workspace_bytes(image_size));
    const int S = image_size;
    const size_t plane = (size_t)S * S;
    float* ws = (float*)workspace;           // 13 planes of S x S floats
    float* su[2] = {ws + 0 * plane, ws + 1 * plane};
    float* sv[2] = {ws + 2 * plane, ws + 3 * plane};
    float* irr = ws + 4 * plane;             // 3 planes each: irradiance after a y pass / after an x pass, accumulator
    float* tmp = ws + 7 * plane;
    float* acc = ws + 10 * plane;
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid = grid_of(S);
    {
        B200rProfScope prof(B200R_K_SSS, st);
        k_sss_stretch<<<grid, 256, 0, st>>>(worldcoord_map, su[0], sv[0], S);
    }
    for (int i = 0; i < 3; i++) {
        const SssTaps t = make_taps(taps + i * kTaps, gauss_widths[i]);
        const float3 w = make_float3(weights[0 * 3 + i], weights[1 * 3 + i], weights[2 * 3 + i]);
        const float* xin = i == 0 ? irradiance_map : irr;
        {
            B200rProfScope prof(B200R_K_SSS, st);
            k_sss_blur_pass<1, kAccNone><<<grid, 256, 0, st>>>(su[i & 1], su[(i + 1) & 1], xin, tmp, nullptr, nullptr, nullptr,
                                                              nullptr, S, t, w);
        }
        {
            B200rProfScope prof(B200R_K_SSS, st);
            if (i == 0)
                k_sss_blur_pass<0, kAccFirst><<<grid, 256, 0, st>>>(sv[0], sv[1], tmp, irr, acc, nullptr, nullptr, nullptr, S, t, w);
            else if (i == 1)
                k_sss_blur_pass<0, kAccAdd><<<grid, 256, 0, st>>>(sv[1], sv[0], tmp, irr, acc, nullptr, nullptr, nullptr, S, t, w);
            else
                k_sss_blur_pass<0, kAccFinal><<<grid, 256, 0, st>>>(sv[0], sv[1], tmp, nullptr, acc, irradiance_map, specular_map,
                                                                   final_map, S, t, w);
        }
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return b200r_cuda_fail(e, "k_sss_blur_pass");
    return 0;
}
