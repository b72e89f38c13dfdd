"""GPU parity tests: the sm_100a kernels (through torch -> ctypes -> C ABI) against the CPU
oracle on identical seeded inputs.

Stated tolerances (fp32; measured margins in profiles/parity_r01.md):
  * integer / index outputs -- faces_id_buffer (slot order), hard-mode aggrs_info
    (depth_min, face_index_min), softmax_max, faces_info (K1) -- BIT-EXACT.  This holds
    because every +,-,*,/ is evaluated unfused in the reference's order on both sides.
  * soft_colors: |diff| <= 2e-6 absolute (values in [0,1]; only expf differs, <= 2 ulp).
  * softmax_sum: relative 2e-6.
  * gradients: max|diff| <= 2e-5 * max|oracle gradient| per tensor (atomic accumulation order
    on the GPU is arbitrary; the oracle accumulates in double).
"""
import itertools
import os

import numpy as np
import pytest

from jrender_b200 import workloads as wl
from oracle import softras as osr
from tests.util import input_sums, large_softras_inputs, run_cuda, run_oracle, softras_stats

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

COLOR_ATOL = 2e-6
SUM_RTOL = 2e-6
GRAD_RTOL = 2e-5


def check(fv, tex, P, seed=2, grads=True):
    H = P["image_size"]
    g = np.random.default_rng(seed).uniform(-1, 1, (fv.shape[0], 4, H, H)).astype(np.float32) if grads else None
    ref = run_oracle(fv, tex, P, grad=g)
    got = run_cuda(fv, tex, P, grad=g)
    assert np.array_equal(got["faces_info"], ref["faces_info"]), "K1 faces_info not bit-exact"
    assert np.array_equal(got["faces_id_buffer"], ref["faces_id_buffer"]), "top-K ids not bit-exact"
    assert not np.isnan(got["soft_colors"]).any()
    d = np.abs(got["soft_colors"] - ref["soft_colors"]).max()
    assert d <= COLOR_ATOL, "soft_colors max abs diff %g" % d
    if P["aggr_func_rgb"] == "softmax":
        assert np.array_equal(got["aggrs_info"][:, 1], ref["aggrs_info"][:, 1]), "softmax_max not bit-exact"
        assert np.allclose(got["aggrs_info"][:, 0], ref["aggrs_info"][:, 0], rtol=SUM_RTOL, atol=0)
    else:
        assert np.array_equal(got["aggrs_info"], ref["aggrs_info"]), "hard-mode aggrs_info not bit-exact"
    if grads:
        for k in ("grad_faces", "grad_textures"):
            a, b = got[k], ref[k]
            # non-finite entries (reference quirk Q6 with fill_back=False) must agree in class;
            # sums of +-inf / NaN contributions are order-independent
            assert np.array_equal(np.isnan(a), np.isnan(b)), "%s NaN pattern differs" % k
            assert np.array_equal(np.isposinf(a), np.isposinf(b)) and np.array_equal(np.isneginf(a), np.isneginf(b))
            m = np.isfinite(b)
            scale = np.abs(b[m]).max() if m.any() else 0.0
            if scale > 0:
                err = np.abs(a[m].astype(np.float64) - b[m]).max() / scale
                assert err <= GRAD_RTOL, "%s rel err %g" % (k, err)
            else:
                assert np.all(a[m] == 0)
    return ref, got


@pytest.fixture(scope="module")
def sphere280(cuda_device):
    return wl.make_scene(280, batch=2)


def test_default_params_256(sphere280):
    check(*sphere280, osr.Params(image_size=256))


def test_non_multiple_of_tile_image_size(sphere280):
    for H in (17, 50, 250):
        check(*sphere280, osr.Params(image_size=H, sigma_val=1e-4))


@pytest.mark.parametrize("dist,rgb,alpha", list(itertools.product(
    ["hard", "barycentric", "euclidean"], ["hard", "softmax", "none"], ["hard", "sum", "prod"])))
def test_all_mode_combinations(sphere280, dist, rgb, alpha):
    check(*sphere280, osr.Params(image_size=96, dist_func=dist, aggr_func_rgb=rgb, aggr_func_alpha=alpha, sigma_val=3e-5))


@pytest.mark.parametrize("rgb", ["hard", "softmax"])
def test_vertex_textures(cuda_device, rgb):
    fv, tex = wl.make_scene(280, batch=1, texture_type="vertex")
    check(fv, tex, osr.Params(image_size=96, texture_type="vertex", aggr_func_rgb=rgb))


@pytest.mark.parametrize("rgb", ["hard", "softmax"])
def test_surface_textures_res5(cuda_device, rgb):
    fv, tex = wl.make_scene(280, batch=1, texture_res=5)
    check(fv, tex, osr.Params(image_size=96, aggr_func_rgb=rgb))


@pytest.mark.parametrize("K", [1, 4, 16, 33, 64])
def test_topk_sizes_on_overlapping_triangles(cuda_device, K):
    fv, tex = wl.random_triangles(2, 300, seed=3)
    check(fv, tex, osr.Params(image_size=80, max_faces_per_pixel_for_grad=K, sigma_val=1e-4))


def test_no_fill_back_reference_nan_pattern(cuda_device):
    """fill_back=False: the reference backward ignores the forward's front-face test (Q6), which
    yields NaN/inf gradients for some back faces; the NaN pattern must match the oracle's."""
    fv, tex = wl.random_triangles(2, 300, seed=3)
    check(fv, tex, osr.Params(image_size=80, fill_back=False))


def test_near_far_rejection(cuda_device):
    fv, tex = wl.random_triangles(1, 200, seed=7, zmin=0.5, zmax=3.0)
    check(fv, tex, osr.Params(image_size=64, near=1.0, far=2.0, sigma_val=1e-4))


def test_single_face_and_degenerate_faces(cuda_device):
    fv = np.array([[[[-0.5, -0.5, 2.0], [0.5, -0.5, 2.0], [0.0, 0.6, 2.5]]]], np.float32)
    tex = np.array([[[[0.2, 0.5, 0.9]]]], np.float32)
    check(fv, tex, osr.Params(image_size=32, sigma_val=1e-3))
    # zero-area and off-screen faces next to a normal one (det clamp +-1e-10, empty rectangles)
    fv2 = np.concatenate([fv, fv * 0 + np.float32([0.1, 0.1, 2.0]), fv + np.float32([5.0, 5.0, 0.0])], axis=1)
    tex2 = np.repeat(tex, 3, axis=1)
    check(fv2, tex2, osr.Params(image_size=32, sigma_val=1e-3))


def test_large_sigma_every_face_touches_every_tile(cuda_device):
    """sqrt(threshold) > 2: check_border never rejects, so every list is the full face list."""
    fv, tex = wl.make_scene(280, batch=1)
    check(fv, tex, osr.Params(image_size=48, sigma_val=0.5, gamma_val=1e-2))


def test_3280_faces_batch_offsets(cuda_device):
    fv, tex = wl.make_scene(3280, batch=3)   # odd batch*nf products exercise unaligned paths
    check(fv[:, :3279], tex[:, :3279], osr.Params(image_size=128))


def test_39k_faces_256(cuda_device):
    fv, tex = wl.make_scene(39200, batch=1)
    check(fv, tex, osr.Params(image_size=256))


def test_full_size_properties_1024_39k(cuda_device):
    """BASELINE full size (1024^2, 39 200 faces), checked through size-independent properties and
    an oracle comparison on a strided row sample (the full oracle run takes minutes)."""
    fv, tex = wl.make_scene(39200, batch=2)
    P = osr.Params(image_size=1024)
    g = np.random.default_rng(2).uniform(-1, 1, (2, 4, 1024, 1024)).astype(np.float32)
    got = run_cuda(fv, tex, P, grad=g, want_faces_info=False)
    sc, ids = got["soft_colors"], got["faces_id_buffer"]
    assert not np.isnan(sc).any() and sc.min() >= 0.0 and sc.max() <= 1.0 + 1e-6
    assert np.all(sc[:, :, :8, :8] == 0) and np.all(ids[:, :, :8, :8] == -1)      # background corner
    cnt = (ids >= 0).sum(1)
    assert cnt.max() == 16 and np.all((ids >= 0) == (np.arange(16)[None, :, None, None] < cnt[:, None]))  # -1 padded tail
    assert ids.max() < 39200
    # rows sampled every 64: oracle vs CUDA, forward outputs
    ref = osr.forward(fv, tex, P, row_stride=64)
    rows = np.arange(0, 1024, 64)
    assert np.array_equal(ids[:, :, rows], ref["faces_id_buffer"][:, :, rows])
    assert np.abs(sc[:, :, rows] - ref["soft_colors"][:, :, rows]).max() <= COLOR_ATOL
    # backward linearity and determinism-to-tolerance at full size
    got2 = run_cuda(fv, tex, P, grad=(2 * g).astype(np.float32), want_faces_info=False)
    scale = np.abs(got["grad_faces"]).max()
    assert np.abs(got2["grad_faces"] - 2 * got["grad_faces"]).max() <= 4 * GRAD_RTOL * scale
    assert np.array_equal(got2["faces_id_buffer"], ids)
    # backward against the oracle AT FULL SIZE: the upstream gradient is zero outside the sampled rows, so the
    # oracle's row-strided top-K backward (same rows) must produce the same face / texture gradients
    gm = np.zeros_like(g)
    gm[:, :, rows] = g[:, :, rows]
    got3 = run_cuda(fv, tex, P, grad=gm, want_faces_info=False)
    rgf, rgt = osr.backward(fv, tex, ref, gm, P, accumulate_double=True, row_stride=64)
    assert np.abs(rgf).max() > 0
    assert np.abs(got3["grad_faces"] - rgf).max() <= GRAD_RTOL * np.abs(rgf).max()
    assert np.abs(got3["grad_textures"] - rgt).max() <= GRAD_RTOL * np.abs(rgt).max()


@pytest.mark.parametrize("H,nfaces", [(2048, 3280), (4096, 280), (1000, 3280)])
def test_large_and_odd_image_sizes(cuda_device, H, nfaces):
    """Coarse bins grow to 128 / 256 px above 1024^2 (common.cuh b200r_geometry) and 4096 is the
    maximum image size of the ABI; 1000 is not a multiple of the 8x4 / 16x16 tiles.  Forward against
    the oracle on a strided row sample, backward through linearity."""
    fv, tex = wl.make_scene(nfaces, batch=1)
    P = osr.Params(image_size=H)
    g = np.random.default_rng(4).uniform(-1, 1, (1, 4, H, H)).astype(np.float32)
    got = run_cuda(fv, tex, P, grad=g, want_faces_info=False)
    stride = H // 16
    ref = osr.forward(fv, tex, P, row_stride=stride)
    rows = np.arange(0, H, stride)
    assert np.array_equal(got["faces_id_buffer"][:, :, rows], ref["faces_id_buffer"][:, :, rows])
    assert np.abs(got["soft_colors"][:, :, rows] - ref["soft_colors"][:, :, rows]).max() <= COLOR_ATOL
    assert (got["faces_id_buffer"][:, 0] >= 0).mean() > 0.1
    got2 = run_cuda(fv, tex, P, grad=(0.5 * g).astype(np.float32), want_faces_info=False)
    scale = np.abs(got["grad_faces"]).max()
    assert scale > 0 and np.abs(got2["grad_faces"] - 0.5 * got["grad_faces"]).max() <= 4 * GRAD_RTOL * scale


def test_image_size_above_abi_maximum_is_refused(cuda_device):
    from jrender_b200._lib import B200RasterError
    fv, tex = wl.make_scene(280, batch=1)
    with pytest.raises(B200RasterError):
        run_cuda(fv, tex, osr.Params(image_size=4104), want_faces_info=False)


def test_public_module_api_and_antialiasing(cuda_device):
    """SoftRasterizer(mesh, mode): AA = render at 2x + 2x2 mean (rasterizer.py:45,54-55), mode slicing."""
    import torch
    from jrender_b200 import SoftRasterizer

    class M:  # minimal stand-in for Mesh: the rasterizer only reads these two
        pass
    fv, tex = wl.make_scene(280, batch=1)
    m = M()
    m.face_vertices = torch.from_numpy(fv).cuda()
    m.face_textures = torch.from_numpy(tex).cuda()
    r = SoftRasterizer(image_size=32, anti_aliasing=True, fill_back=True)
    sil, rgb = r(m)
    assert tuple(sil.shape) == (1, 32, 32) and tuple(rgb.shape) == (1, 3, 32, 32)
    ref = osr.forward(fv, tex, osr.Params(image_size=64))["soft_colors"]
    pooled = ref.reshape(1, 4, 32, 2, 32, 2).mean(axis=(3, 5))
    assert np.abs(rgb.cpu().numpy() - pooled[:, :3]).max() <= 2 * COLOR_ATOL
    assert np.abs(r(m, "silhouettes").cpu().numpy() - pooled[:, 3]).max() <= 2 * COLOR_ATOL


@pytest.mark.parametrize("rgb", ["softmax", "hard"])
def test_silhouette_mode_runs_without_the_colour_path(cuda_device, rgb):
    """mode='silhouettes' compiles the colour aggregation out (B200R_RGB_NONE): alpha must be the same
    bits as channel 3 of the full render and the vertex gradient the same as back-propagating through
    the full render with a zero colour gradient (the oracle run in the reference's own mode)."""
    import torch
    from jrender_b200 import SoftRasterizer

    class M:
        pass
    fv, tex = wl.make_scene(280, batch=2)
    m = M()
    m.face_vertices = torch.from_numpy(fv).cuda().requires_grad_(True)
    m.face_textures = torch.from_numpy(tex).cuda()
    r = SoftRasterizer(image_size=96, fill_back=True, aggr_func_rgb=rgb, sigma_val=1e-4)
    sil = r(m, "silhouettes")
    full_alpha, _ = r(m)
    assert torch.equal(sil, full_alpha)
    g = torch.from_numpy(np.random.default_rng(3).uniform(-1, 1, (2, 96, 96)).astype(np.float32)).cuda()
    sil.backward(g)
    P = osr.Params(image_size=96, aggr_func_rgb=rgb, sigma_val=1e-4)
    ref = osr.forward(fv, tex, P)
    g4 = np.zeros((2, 4, 96, 96), np.float32)
    g4[:, 3] = g.cpu().numpy()
    gf, _ = osr.backward(fv, tex, ref, g4, P)
    assert np.array_equal(sil.detach().cpu().numpy(), ref["soft_colors"][:, 3]) or \
        np.abs(sil.detach().cpu().numpy() - ref["soft_colors"][:, 3]).max() <= COLOR_ATOL
    assert np.abs(m.face_vertices.grad.cpu().numpy() - gf).max() <= GRAD_RTOL * np.abs(gf).max()


@pytest.mark.parametrize("nfaces,H,min_same,grad_l1", [(3280, 512, 0.998, 0.05), (39200, 512, 0.98, 0.15),
                                                        (39200, 1024, 0.99, 0.10)])
def test_against_reference_kernels_on_gpu(cuda_device, nfaces, H, min_same, grad_l1):
    """Product vs the reference's OWN kernels, at a size the CPU oracle would take minutes for.  The reference's
    outputs come from tests/golden/refsample_softras_<faces>_<size>.npz (its kernel strings compiled for sm_100a by
    oracle/build_ref.py and run on a B200 by oracle/make_ref_golden.py --large-only): a stratified sample from which
    the statistics over the whole image and all faces are estimated (tests/util.py).
    Statistical tolerances as in tests/test_golden.py: the reference build contracts a*b+c
    into FMAs, which moves depths by an ulp and flips top-K membership between faces of nearly
    equal depth -- rare for the 3280-face mesh, ~0.7 % of pixels for ~2-pixel triangles (where a
    different face then receives that pixel's gradient: relative L1 of grad_faces ~9 %)."""
    z = dict(np.load(os.path.join(GOLDEN, "refsample_softras_%d_%d.npz" % (nfaces, H))))
    fv, tex, g = large_softras_inputs(nfaces, H)   # 1024 / 39 200 faces is BASELINE config C3's image
    assert np.allclose(input_sums(fv, tex, g), z["input_sums"], rtol=1e-6, atol=0)
    got = run_cuda(fv, tex, osr.Params(image_size=H), grad=g, want_faces_info=False)
    s = softras_stats(z, got)
    assert s["same"] >= min_same, s
    assert s["color_frac"] <= 0.02 and s["color_mean"] <= 2e-3, s
    assert s["grad_faces"] <= grad_l1 and s["grad_textures"] <= grad_l1, s


def test_scheduling_choice_gives_identical_results(cuda_device):
    """The persistent cost-ordered block queue is a pure scheduling choice: one CTA per block (queue off) must give
    bit-identical outputs, also with T > 1 textures and a sigma large enough that every face covers every block."""
    from jrender_b200 import _lib
    fv, tex = wl.make_scene(3280, batch=2)
    P = osr.Params(image_size=200, sigma_val=3e-5)
    fv5, tex5 = wl.make_scene(280, batch=1, texture_res=3)
    P5 = osr.Params(image_size=96, sigma_val=1e-3, gamma_val=1e-3)
    base = run_cuda(fv, tex, P, want_faces_info=False)
    base5 = run_cuda(fv5, tex5, P5, want_faces_info=False)
    try:
        _lib.set_option("softras_fwd_persistent", 0)
        got = run_cuda(fv, tex, P, want_faces_info=False)
        got5 = run_cuda(fv5, tex5, P5, want_faces_info=False)
    finally:
        _lib.set_option("softras_fwd_persistent", 1)
    for k in ("soft_colors", "aggrs_info", "faces_id_buffer"):
        assert np.array_equal(base[k], got[k]) and np.array_equal(base5[k], got5[k]), k
    ref = run_oracle(fv, tex, P)
    assert np.array_equal(ref["faces_id_buffer"], got["faces_id_buffer"])
    ref5 = run_oracle(fv5, tex5, P5)
    assert np.array_equal(ref5["faces_id_buffer"], got5["faces_id_buffer"])
    assert np.abs(ref5["soft_colors"] - got5["soft_colors"]).max() <= COLOR_ATOL


@pytest.mark.parametrize("pool_chunks", [0, 1, 3])
def test_coarse_list_pool_exhaustion_changes_nothing(cuda_device, pool_chunks):
    """The binning lists grow in 512-id chunks out of a shared pool.  With the pool capped (0: every non-empty bin, 1 / 3:
    whichever bins lose the race) the flagged bins' blocks filter the complete face list instead: every output must be
    bit-identical to the uncapped run, which itself is held to the oracle.  3280 faces at sigma 3e-5 put > 512 faces into
    the central bins (multi-chunk lists)."""
    from jrender_b200 import _lib
    fv, tex = wl.make_scene(3280, batch=2)
    P = osr.Params(image_size=200, sigma_val=3e-5)
    g = np.random.default_rng(5).uniform(-1, 1, (2, 4, 200, 200)).astype(np.float32)
    base = run_cuda(fv, tex, P, grad=g, want_faces_info=False)
    try:
        _lib.set_option("softras_list_pool_chunks", pool_chunks)
        got = run_cuda(fv, tex, P, grad=g, want_faces_info=False)
    finally:
        _lib.set_option("softras_list_pool_chunks", -1)
    for k in ("soft_colors", "aggrs_info", "faces_id_buffer"):
        assert np.array_equal(base[k], got[k]), k
    ref = run_oracle(fv, tex, P)
    assert np.array_equal(ref["faces_id_buffer"], got["faces_id_buffer"])
    assert np.abs(ref["soft_colors"] - got["soft_colors"]).max() <= COLOR_ATOL


def test_pool_exhaustion_at_headline_size(cuda_device):
    """One image of the headline configuration (1024^2, 39 200 faces) with the list pool capped at 64 chunks: most of the
    ~100 non-empty bins are flagged and their blocks filter all 39 200 faces; ids, colours and aggregates must not move."""
    from jrender_b200 import _lib
    fv, tex = wl.make_scene(39200, batch=1)
    P = osr.Params(image_size=1024)
    base = run_cuda(fv, tex, P, want_faces_info=False)
    try:
        _lib.set_option("softras_list_pool_chunks", 64)
        got = run_cuda(fv, tex, P, want_faces_info=False)
    finally:
        _lib.set_option("softras_list_pool_chunks", -1)
    for k in ("soft_colors", "aggrs_info", "faces_id_buffer"):
        assert np.array_equal(base[k], got[k]), k


def test_workspace_is_small_and_lists_span_chunks(cuda_device):
    """Workspace of the headline configuration (4 x 1024^2, 39 200 faces) stays below 16 MB (round 1: 162 MB with capacity
    num_faces per bin), and a bin list longer than one chunk (every face of a 3280-face sphere inside one 64-pixel bin)
    is read back correctly across chunk boundaries."""
    from jrender_b200 import _lib
    L = _lib.lib()
    assert L.b200r_softras_workspace_bytes(4, 39200, 1024) < 16 * 2 ** 20
    fv, tex = wl.make_scene(3280, batch=1, distance=40.0)   # the whole sphere projects into ~50 pixels
    P = osr.Params(image_size=512)
    check(fv, tex, P, grads=False)


@pytest.mark.parametrize("mode", [dict(), dict(aggr_func_rgb="hard"), dict(texture_type="vertex"),
                                  dict(dist_func="barycentric", aggr_func_alpha="sum")])
def test_backward_modes_agree_with_oracle(cuda_device, mode):
    """The per-lane backward (16-byte vector atomics + finalize) in the texture / aggregation modes that take different
    accumulation paths (T == 1 colour in the accumulator, texel-indexed and per-vertex texture gradients)."""
    tt = mode.get("texture_type", "surface")
    fv, tex = wl.make_scene(280, batch=2, texture_type=tt, texture_res=1)
    check(fv, tex, osr.Params(image_size=96, sigma_val=3e-5, **mode))
    fv5, tex5 = wl.make_scene(280, batch=1, texture_res=3)
    check(fv5, tex5, osr.Params(image_size=64, aggr_func_rgb=mode.get("aggr_func_rgb", "softmax")))


@pytest.mark.parametrize("mode", [None, "silhouettes", "rgb"])
def test_fused_antialiasing_matches_the_unfused_op_sequence(cuda_device, mode):
    """anti_aliasing=True: the forward's 2x2-mean epilogue and the backward's pooled-gradient prologue
    (b200r_softras_forward_aa / _backward_aa) against render-at-2x + avg_pool2d + autograd (rasterizer.py:45,54-55)."""
    import torch
    from jrender_b200 import SoftRasterizer

    class M:
        pass
    fv, tex = wl.make_scene(280, batch=2)
    res = {}
    for fused in (True, False):
        m = M()
        m.face_vertices = torch.from_numpy(fv).cuda().requires_grad_(True)
        m.face_textures = torch.from_numpy(tex).cuda().requires_grad_(True)
        r = SoftRasterizer(image_size=50, anti_aliasing=True, fill_back=True, sigma_val=3e-5)
        r.fused_antialiasing = fused
        out = r(m, mode)
        outs = list(out) if isinstance(out, tuple) else [out]
        rng = np.random.default_rng(4)
        torch.autograd.backward(outs, [torch.from_numpy(rng.uniform(-1, 1, tuple(o.shape)).astype(np.float32)).cuda() for o in outs])
        res[fused] = ([o.detach().cpu().numpy() for o in outs], m.face_vertices.grad.cpu().numpy(),
                      None if m.face_textures.grad is None else m.face_textures.grad.cpu().numpy())
    for a, b_ in zip(res[True][0], res[False][0]):
        assert a.shape == b_.shape and np.abs(a - b_).max() <= 1e-7
    assert np.abs(res[True][1] - res[False][1]).max() <= GRAD_RTOL * np.abs(res[False][1]).max()
    if res[False][2] is not None and np.abs(res[False][2]).max() > 0:
        assert np.abs(res[True][2] - res[False][2]).max() <= GRAD_RTOL * np.abs(res[False][2]).max()


def test_exact_tail_option(cuda_device):
    """softras_exact_tail=1 evaluates the sigmoid / alpha-product tails in double like the reference;
    the default fp32 tails may move D by <= 1 ulp.  Index / depth outputs must be identical, colours
    agree to a few 1e-7, and both settings satisfy the oracle tolerances."""
    from jrender_b200 import _lib
    fv, tex = wl.make_scene(3280, batch=1)
    P = osr.Params(image_size=192)
    g = np.random.default_rng(2).uniform(-1, 1, (1, 4, 192, 192)).astype(np.float32)
    try:
        _lib.set_option("softras_exact_tail", 1)
        _, exact = check(fv, tex, P)
        _lib.set_option("softras_exact_tail", 0)
        _, fast = check(fv, tex, P)
    finally:
        _lib.set_option("softras_exact_tail", 0)
    assert np.array_equal(exact["faces_id_buffer"], fast["faces_id_buffer"])
    assert np.array_equal(exact["aggrs_info"][:, 1], fast["aggrs_info"][:, 1])
    assert np.abs(exact["soft_colors"] - fast["soft_colors"]).max() <= 5e-7
    assert np.abs(exact["grad_faces"] - fast["grad_faces"]).max() <= GRAD_RTOL * np.abs(exact["grad_faces"]).max()
