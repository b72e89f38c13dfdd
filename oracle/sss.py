"""CPU oracle of the texture-space subsurface scattering chain (TEST INFRASTRUCTURE; product code never imports it).

numpy fp32 restatement of
  renderer/utils/ToStretchMap.py          computeStretchMap (replicate padding), then clamp to [0, 1]
  renderer/utils/gaussian_blur.py:34-165  the 7-tap stretch-modulated blur, d = 1, with the reference's truncation
                                          (int(), not floor), clamping, centre-value masking and the FFMA contraction
                                          nvcc applies to its interpolation and accumulation (fma32 below)
  renderer/lighting/lighting.py:115-150   the three basis steps, weighted sum, `* irradiance + specular`, vertical flip
Pinned against the reference's own blur kernel run on a B200 (tests/golden/sss_ref_gpu_blur_*.npz, generator
oracle/make_ref_sss_golden.py --gpu) and against the reference's own SSS() Python (tests/golden/ref_host_sss_spot.npz,
generator oracle/make_ref_sss_golden.py --host).
"""
import math

import numpy as np

TAP_NUM = 7
GAUSSIAN_BASIS = [0, 25, 100, 400]
WEIGHTS = np.array([[0.7, 0.2, 0.1], [0.1, 0.2, 0.7], [0.1, 0.2, 0.7]], np.float32)   # [channel][basis]


def taps(v, tap_num=TAP_NUM):
    """gaussian_blur.py:4-10 and :28-29 in double, rounded to float32: (taps [tap_num], GaussWidth)."""
    w = math.sqrt(v)
    g = [w * (math.exp(-(-w * ((tap_num - 1) / 2 - i)) ** 2 / (2 * v)) / math.sqrt(2 * math.pi * v)) for i in range(tap_num)]
    return np.array(g, np.float32), np.float32(w)


def fma32(a, b, c):
    """Correctly rounded float32 a*b+c: the product is exact in double; the double sum is rounded to odd (exact two-sum
    error term), which makes the final rounding to float32 correct."""
    a, b, c = (np.asarray(x, np.float32).astype(np.float64) for x in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    even = (s.view(np.int64) & 1) == 0
    fix = (err != 0) & even & np.isfinite(s)
    s = np.where(fix, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def blur(image, modulate, tap, width, dim):
    """gaussain_blur_x_Kernel (dim 1) / gaussain_blur_y_Kernel (dim 0) on one [S, S] float32 map."""
    f32 = np.float32
    img = np.asarray(image, f32)
    a = img if dim == 1 else img.T                  # blur along the last axis
    m = np.asarray(modulate, f32) if dim == 1 else np.asarray(modulate, f32).T
    H, n = a.shape
    pos = np.broadcast_to(np.arange(n, dtype=f32)[None, :], a.shape)
    nfw = f32(width) * m
    c = pos - nfw * f32(TAP_NUM - 1) / f32(2)
    rows = np.arange(H)[:, None]
    v = np.zeros_like(a)
    for k in range(TAP_NUM):
        t = np.trunc(c).astype(np.int64)
        c1, c2 = np.clip(t, 0, n - 1), np.clip(t + 1, 0, n - 1)
        v1, v2 = a[rows, c1], a[rows, c2]
        v1 = np.where(v1.astype(np.float64) > 1e-6, v1, a)
        v2 = np.where(v2.astype(np.float64) > 1e-6, v2, a)
        interp = fma32(c2.astype(f32) - c, v1, (c - c1.astype(f32)) * v2)
        v = fma32(interp, f32(tap[k]), v)
        c = c + nfw
    out = np.where(a > 0, v, f32(0)).astype(f32)
    return out if dim == 1 else np.ascontiguousarray(out.T)


def stretch_maps(world_hwc):
    """computeStretchMap(world * 7), both maps clamped to [0, 1]."""
    w = np.asarray(world_hwc, np.float32) * np.float32(7)
    wx = np.concatenate([w[:, 1:], w[:, -1:]], axis=1)
    wy = np.concatenate([w[1:], w[-1:]], axis=0)
    with np.errstate(divide="ignore"):
        du, dv = w - wx, w - wy
        su = np.float32(1) / np.sqrt(du[..., 0] * du[..., 0] + du[..., 1] * du[..., 1] + du[..., 2] * du[..., 2])
        sv = np.float32(1) / np.sqrt(dv[..., 0] * dv[..., 0] + dv[..., 1] * dv[..., 1] + dv[..., 2] * dv[..., 2])
    return np.clip(su, 0, 1).astype(np.float32), np.clip(sv, 0, 1).astype(np.float32)


def blur_chain(world_hwc, irradiance_hwc, specular_hwc):
    """lighting.py:115-150 from the three rasterized maps ([S, S, 3] each): final_map [S, S, 3], already flipped."""
    su, sv = stretch_maps(world_hwc)
    irr = [np.ascontiguousarray(irradiance_hwc[:, :, c], np.float32) for c in range(3)]
    final = np.zeros(np.asarray(irradiance_hwc).shape, np.float32)
    for i in range(3):
        tap, w = taps(GAUSSIAN_BASIS[i + 1] - GAUSSIAN_BASIS[i])
        su = blur(su, su, tap, w, 1)
        irr = [blur(x, su, tap, w, 1) for x in irr]
        sv = blur(sv, sv, tap, w, 0)
        irr = [blur(x, sv, tap, w, 0) for x in irr]
        for c in range(3):
            final[:, :, c] = final[:, :, c] + WEIGHTS[c, i] * irr[c]
    final = final * np.asarray(irradiance_hwc, np.float32) + np.asarray(specular_hwc, np.float32)
    return np.ascontiguousarray(final[::-1])


def texture_space_params(image_size):
    """The SoftRasterizeFunction configuration of SSS() (lighting.py:90-95), as oracle.softras.Params."""
    from oracle import softras as osr
    return osr.Params(image_size=image_size, near=1, far=100, fill_back=True, eps=1e-5, sigma_val=1e-5,
                      dist_func="barycentric", dist_eps=1e-5, gamma_val=1e-4, aggr_func_rgb="hard",
                      aggr_func_alpha="prod", texture_type="surface")


def texture_space_inputs(face_vertices, face_texcoords, textures, diffuse, specular):
    """(coords [1,nf,3,3], worldcoord textures, irradiance, specular) of lighting.py:88-103, float32 numpy."""
    f32 = np.float32
    irradiance = np.sqrt(np.asarray(textures, f32) * np.asarray(diffuse, f32))
    world = (np.asarray(face_vertices, f32) + f32(1)) / f32(2) * f32(255)
    coords = (np.asarray(face_texcoords, f32) - f32(0.5)) * f32(2)
    coords = np.concatenate([coords, np.full(coords.shape[:3] + (1,), 1.5, f32)], axis=3)
    return coords, world, irradiance, np.asarray(specular, f32)


def sss(face_vertices, face_texcoords, textures, diffuse, specular, texture_res, image_size):
    """SSS() of lighting.py:86-156 for one mesh (batch 1): [1, nf, texture_res**2, 3], before the caller's clamp."""
    from oracle import bake as obake, softras as osr
    P = texture_space_params(image_size)
    coords, world, irradiance, spec = texture_space_inputs(face_vertices, face_texcoords, textures, diffuse, specular)
    maps = [osr.forward(coords, np.ascontiguousarray(t, np.float32), P)["soft_colors"][0, :3].transpose(1, 2, 0)
            for t in (world, irradiance, spec)]
    final = blur_chain(*maps)
    nf = coords.shape[1]
    out = obake.bake_textures_for_softras(final, np.asarray(face_texcoords, np.float32)[0],
                                          np.ones((nf, texture_res ** 2, 3), np.float32), np.ones(nf, np.int32))
    return out[None]
