"""GPU parity tests of the NMR (dr_type='n3mr') kernels against the CPU oracle (oracle/nmr_oracle.c).

Stated tolerances: the forward contains no transcendental function and every +,-,*,/ is evaluated
unfused in the reference's order on both sides, so ALL forward maps are BIT-EXACT (face index,
barycentric weights, depth, sampled colour, sampling indices/weights, face_inv, alpha).
Backward: gradients are sums over pixels accumulated in a different order (warp-parallel scans,
float atomics) than the oracle's sequential double accumulation: max|diff| <= 2e-5 * max|oracle|.
"""
import os

import numpy as np
import pytest

from oracle import nmr as onmr
from tests.util import c4_inputs, input_sums, nmr_scene, nmr_stats, run_nmr_cuda

pytestmark = pytest.mark.gpu
GRAD_RTOL = 2e-5


def check(faces, tex, H, flags=(True, True, True), bg=(0, 0, 0), near=0.1, far=100.0, eps=1e-3, seed=0):
    ref = onmr.forward(faces, tex if flags[0] else None, H, near, far, eps, bg, *flags)
    rng = np.random.default_rng(seed)
    B = faces.shape[0]
    g = (rng.uniform(-1, 1, (B, H, H, 3)).astype(np.float32), rng.uniform(-1, 1, (B, H, H)).astype(np.float32),
         rng.uniform(-1, 1, (B, H, H)).astype(np.float32))
    gf, gt = onmr.backward(faces, tex if flags[0] else None, ref, H, eps, g[0], g[1], g[2], *flags)
    got = run_nmr_cuda(faces, tex, H, near, far, eps, bg, flags, grads=g)
    for k in ("face_index_map", "weight_map", "depth_map"):
        assert np.array_equal(got[k], ref[k]), k
    if flags[0]:
        for k in ("rgb_map", "sampling_index_map", "sampling_weight_map"):
            assert np.array_equal(got[k], ref[k]), k
    if flags[1]:
        assert np.array_equal(got["alpha_map"], ref["alpha_map"])
    if flags[2]:
        assert np.array_equal(got["face_inv_map"].reshape(ref["face_inv_map"].shape), ref["face_inv_map"])
    scale = np.abs(gf).max()
    assert np.abs(got["grad_faces"] - gf).max() <= GRAD_RTOL * max(scale, 1e-30), np.abs(got["grad_faces"] - gf).max() / scale
    if flags[0]:
        assert np.abs(got["grad_textures"] - gt).max() <= GRAD_RTOL * np.abs(gt).max()
    assert (ref["face_index_map"] >= 0).mean() > 0.05   # the case renders something
    return ref, got


def test_rgbad_sphere_fill_back(cuda_device):
    faces, tex = nmr_scene(280, batch=2, ts=2)
    check(faces, tex, 128, bg=(0.2, 0.4, 0.6))


@pytest.mark.parametrize("flags", [(True, False, False), (False, True, False), (False, False, True), (True, True, False)])
def test_output_subsets(cuda_device, flags):
    faces, tex = nmr_scene(280, batch=1, ts=4)
    check(faces, tex, 96, flags=flags)


def test_texture_size_1_and_odd_image(cuda_device):
    faces, tex = nmr_scene(280, batch=1, ts=1)
    check(faces, tex, 75)


def test_texture_size_1_last_faces_visible(cuda_device):
    # texture_size 1 without fill_back: the "+1" trilinear taps of the LAST faces point past the
    # texture tensor (reference UB); product and oracle both read them as 0 and drop their gradient
    faces, tex = nmr_scene(280, batch=2, ts=1, fill_back=False)
    ref, got = check(faces, tex, 48, bg=(0.1, 0.2, 0.3))
    assert (ref["face_index_map"] >= 276).any()


def test_overlapping_random_triangles_and_near_far(cuda_device):
    from jrender_b200 import workloads as wl
    fv, _ = wl.random_triangles(2, 200, seed=5, zmin=0.5, zmax=3.0)
    tex = np.random.default_rng(2).random((2, 200, 2, 2, 2, 3), dtype=np.float32)
    check(fv, tex, 64, near=1.0, far=2.5)


def test_3280_faces_256(cuda_device):
    faces, tex = nmr_scene(3280, batch=1, ts=2)
    check(faces, tex, 256)


def test_39k_faces_forward_and_backward_properties_1024(cuda_device):
    """BASELINE config C4 size: 39 200 (x2 fill_back) faces at 1024^2: forward maps and the edge-scan / texture
    backward against the oracle IN FULL (the oracle needs a few seconds per image), plus properties."""
    faces, tex = nmr_scene(39200, batch=1, ts=2)
    ref = onmr.forward(faces, tex, 1024, 0.1, 100.0, 1e-3, (0, 0, 0), True, True, False)
    g = np.random.default_rng(0).uniform(-1, 1, (1, 1024, 1024, 3)).astype(np.float32)
    ga = np.random.default_rng(1).uniform(-1, 1, (1, 1024, 1024)).astype(np.float32)
    got = run_nmr_cuda(faces, tex, 1024, flags=(True, True, False), grads=(g, ga, None))
    assert np.array_equal(got["face_index_map"], ref["face_index_map"])
    assert np.array_equal(got["rgb_map"], ref["rgb_map"]) and np.array_equal(got["depth_map"], ref["depth_map"])
    gf, gt = onmr.backward(faces, tex, ref, 1024, 1e-3, g, ga, None, True, True, False)
    assert np.abs(gf).max() > 0
    assert np.abs(got["grad_faces"] - gf).max() <= GRAD_RTOL * np.abs(gf).max()
    assert np.abs(got["grad_textures"] - gt).max() <= GRAD_RTOL * np.abs(gt).max()
    got2 = run_nmr_cuda(faces, tex, 1024, flags=(True, True, False), grads=((2 * g).astype(np.float32), (2 * ga).astype(np.float32), None))
    s = np.abs(got["grad_faces"]).max()
    assert np.abs(got2["grad_faces"] - 2 * got["grad_faces"]).max() <= 4 * GRAD_RTOL * s     # linear in the upstream gradient
    assert np.all(got["grad_faces"][..., 2] == 0)                                            # no z gradient without depth output
    back = np.arange(faces.shape[1]) >= 39200                                                # reversed copies of front faces are culled
    culled = (faces[0, :, 2, 1] - faces[0, :, 0, 1]) * (faces[0, :, 1, 0] - faces[0, :, 0, 0]) < \
             (faces[0, :, 1, 1] - faces[0, :, 0, 1]) * (faces[0, :, 2, 0] - faces[0, :, 0, 0])
    assert np.all(got["grad_faces"][0, culled] == 0) and back.any()


def test_c4_against_reference_kernels_on_gpu(cuda_device):
    """Product vs the reference's OWN K7-K11 at BASELINE config C4's size (1024^2, 2 x 39 200 faces, ts=2).  The
    reference's outputs come from tests/golden/refsample_nmr_c4_1024.npz (its kernel strings compiled for sm_100a by
    oracle/build_ref.py and run on a B200 by oracle/make_ref_golden.py --large-only): a stratified sample from which the
    statistics over the whole image and all faces are estimated (tests/util.py).  Tolerances as in
    tests/test_golden.py's NMR fixtures: the reference build contracts a*b+c into FMAs, and its lock-protected z-test
    is race-dependent on exact depth ties, so a handful of pixels on shared edges may go to the neighbouring face."""
    z = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "refsample_nmr_c4_1024.npz")))
    faces, tex, g, ga = c4_inputs()
    assert np.allclose(input_sums(faces, tex, g, ga), z["input_sums"], rtol=1e-6, atol=0)
    got = run_nmr_cuda(faces, tex, 1024, flags=(True, True, False), grads=(g, ga, None))
    s = nmr_stats(z, got, far=100.0)
    assert s["same"] >= 0.999, s
    # sliver faces at the sphere's poles have barycentric weights that cancel almost completely: the reference build's FMA
    # contraction moves their interpolated depth by up to ~1e-3 on a handful of pixels (measured max 1.1e-3), everything
    # else agrees to 1e-4
    assert s["depth_frac"] <= 1e-3 and s["depth_max"] <= 1e-2, s
    assert s["color_frac"] <= 1e-3 and s["color_max"] <= 0.1, s
    assert s["grad_faces"] <= 0.05 and s["grad_textures"] <= 0.01, s


def test_module_api_image_orientation_and_antialiasing(cuda_device):
    """N3mrRasterizer(mesh, mode): fill_back, NCHW + vertical flip, 2x2 mean pooling (n3mr.py:233-256)."""
    import torch
    import jrender_b200 as jr
    from jrender_b200.n3mr import N3mrRasterizer
    from jrender_b200 import workloads as wl
    v, f = wl.sphere_by_faces(280)
    eye = wl.get_points_from_angles(2.732, 30, 0)
    cam = jr.perspective(jr.look_at(torch.from_numpy(v)[None].cuda(), eye), 30.)
    tex = torch.rand(1, 280, 2, 2, 2, 3, device="cuda")
    mesh = jr.Mesh(cam, torch.from_numpy(f).cuda(), textures=tex, dr_type='n3mr')
    r = N3mrRasterizer(image_size=32, anti_aliasing=True, background_color=[0, 0, 0], fill_back=True)
    rgb = r(mesh, 'rgb')
    sil = r(mesh, 'silhouettes')
    assert tuple(rgb.shape) == (1, 3, 32, 32) and tuple(sil.shape) == (1, 1, 32, 32)
    faces2 = np.concatenate([wl.face_vertices(cam.cpu().numpy(), f), wl.face_vertices(cam.cpu().numpy(), f)[:, :, ::-1]], 1)
    tex2 = np.concatenate([tex.cpu().numpy(), tex.cpu().numpy().transpose(0, 1, 4, 3, 2, 5)], 1)
    ref = onmr.forward(faces2, tex2, 64, 0.1, 100.0, 1e-3, (0, 0, 0), True, True, False)
    img = ref["rgb_map"][:, ::-1].transpose(0, 3, 1, 2).reshape(1, 3, 32, 2, 32, 2).mean(axis=(3, 5))
    assert np.abs(rgb.cpu().numpy() - img).max() <= 1e-6
    a = ref["alpha_map"][:, ::-1].reshape(1, 32, 2, 32, 2).mean(axis=(2, 4))
    assert np.abs(sil.cpu().numpy()[:, 0] - a).max() <= 1e-6
    # Renderer(dr_type='n3mr') wires the same rasterizer
    rr = jr.Renderer(image_size=32, dr_type='n3mr')
    assert isinstance(rr.rasterizer, N3mrRasterizer)
