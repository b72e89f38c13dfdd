"""GPU tests of the texture-bake kernels (csrc/bake_api.cu <- jrender/io/utils/load_textures.py:3-101 SoftRas, :103-246 NMR) and of BASELINE
config C1 as the reference configures it (demo1-render.py:21-45: spot cow, 5856 faces, texture_res 5, 256^2).

Tolerances: bake vs the numpy oracle 2e-6 absolute (same formulas unfused on both sides; image values in [0, 1]); vs the
reference's own kernel on a B200 (tests/golden/ref_gpu_bake_random40_R5.npz) 1e-5 (its build contracts a*b+c).
C1: top-K ids bit-exact, colours 2e-6, gradients 2e-5 of max -- the SoftRas parity bar (tests/test_softras_gpu.py).
"""
import lzma
import os
import shutil

import numpy as np
import pytest
import torch

import jrender_b200 as jr
from oracle import bake as obake
from oracle import softras as osr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def spot(tmp_path_factory):
    """The reference's spot cow (data/obj/spot: OBJ + MTL + texture PNG), kept xz-compressed under tests/golden/spot and
    unpacked next to its material files; returns the OBJ's path."""
    d = tmp_path_factory.mktemp("spot")
    src = os.path.join(G, "spot")
    with lzma.open(os.path.join(src, "spot_triangulated.obj.xz")) as f, open(d / "spot_triangulated.obj", "wb") as g:
        shutil.copyfileobj(f, g)
    for name in ("spot_triangulated.mtl", "spot_texture.png"):
        shutil.copyfile(os.path.join(src, name), d / name)
    return str(d / "spot_triangulated.obj")


def test_bake_kernel_matches_oracle_and_reference_kernel(cuda_device):
    from jrender_b200.io import bake_textures_for_softras
    rng = np.random.default_rng(3)
    for nf, R, H, W in ((40, 5, 24, 40), (257, 1, 7, 9), (33, 4, 64, 64)):
        image = rng.random((H, W, 3), dtype=np.float32)
        uv = rng.uniform(0.0, 1.0, (nf, 3, 2)).astype(np.float32)      # includes taps on the last row / column
        upd = (rng.random(nf) > 0.3).astype(np.int32)
        tex0 = rng.random((nf, R * R, 3), dtype=np.float32)
        got = bake_textures_for_softras(image, uv, tex0, upd, device=cuda_device).cpu().numpy()
        ref = obake.bake_textures_for_softras(image, uv, tex0, upd)
        assert np.abs(got - ref).max() <= 2e-6
        assert np.array_equal(got[upd == 0], tex0[upd == 0])
    p = os.path.join(G, "ref_gpu_bake_random40_R5.npz")
    if os.path.exists(p):
        g = np.load(p)
        got = bake_textures_for_softras(g["image"], g["faces_uv"], g["textures_in"], g["is_update"], device=cuda_device).cpu().numpy()
        assert np.abs(got - g["textures"]).max() <= 1e-5


@pytest.mark.parametrize("wrap,bilinear", [(w, b) for w in range(4) for b in (True, False)])
def test_n3mr_bake_kernel_matches_oracle(cuda_device, wrap, bilinear):
    """b200r_bake_textures_n3mr (<- load_textures.py:103-246) against oracle/bake.py for every wrapping mode and both
    sampling flavours, UVs far outside [0, 1] (odd and even integer parts, negative), 2e-6 absolute; untouched faces keep
    their texels; texture_size 1 is refused."""
    from jrender_b200 import _lib
    from jrender_b200.io import bake_textures_for_n3mr
    rng = np.random.default_rng(17 + wrap)
    for nf, ts, H, W in ((40, 4, 37, 53), (130, 2, 8, 8), (9, 6, 64, 31)):
        image = rng.random((H, W, 3), dtype=np.float32)
        uv = rng.uniform(-2.3, 3.1, (nf, 3, 2)).astype(np.float32)
        upd = (rng.random(nf) > 0.3).astype(np.int32)
        tex0 = rng.random((nf, ts, ts, ts, 3), dtype=np.float32)
        got = bake_textures_for_n3mr(image, uv, tex0, upd, wrap, bilinear, device=cuda_device).cpu().numpy()
        ref = obake.bake_textures_for_n3mr(image, uv, tex0, upd, wrap, bilinear)
        if bilinear or wrap == 3:
            assert np.abs(got - ref).max() <= 2e-6
        else:   # nearest: a sample point within float rounding of a texel boundary may pick the neighbour
            bad = np.abs(got - ref).max(axis=-1) > 2e-6
            assert bad.mean() <= 2e-3
        assert np.array_equal(got[upd == 0], tex0[upd == 0])
    with pytest.raises(_lib.B200RasterError):
        bake_textures_for_n3mr(np.zeros((4, 4, 3), np.float32), np.zeros((2, 3, 2), np.float32), np.zeros((2, 1, 1, 1, 3), np.float32),
                               np.ones(2, np.int32), 0, True, device=cuda_device)


def test_n3mr_bake_kernel_matches_reference_kernel_golden(cuda_device):
    """... and against the reference's own kernel run on a B200 (tests/golden/ref_gpu_bake_n3mr_*.npz), 1e-5 (its build
    contracts a*b+c)."""
    import glob
    from jrender_b200.io import bake_textures_for_n3mr
    files = sorted(glob.glob(os.path.join(G, "ref_gpu_bake_n3mr_*.npz")))
    assert files, "golden fixtures missing"
    for p in files:
        g = np.load(p)
        got = bake_textures_for_n3mr(g["image"], g["faces_uv"], g["textures_in"], g["is_update"], int(g["texture_wrapping"]),
                                     bool(int(g["use_bilinear"])), device=cuda_device).cpu().numpy()
        d = np.abs(got - g["textures"]).max(axis=-1)
        if int(g["use_bilinear"]):
            assert d.max() <= 1e-5, p
        else:
            assert (d > 1e-5).mean() <= 2e-3, p


def test_n3mr_loader_bakes_the_spot_texture(cuda_device, spot):
    """load_obj(dr_type='n3mr', load_texture=True) as demo4 would call it: [nf, ts, ts, ts, 3] textures whose baked texels
    equal the oracle's bake of the same image / UVs."""
    from jrender_b200 import io as jio
    v, f, t = jio.load_obj(spot, load_texture=True, dr_type='n3mr', texture_res=4)
    assert tuple(t.shape) == (5856, 4, 4, 4, 3) and tuple(f.shape) == (5856, 3)
    faces_uv, names = jio._parse_texture_faces(spot)
    image = jio._imread_rgb01(os.path.join(os.path.dirname(spot), "spot_texture.png"))[::-1]
    ref = obake.bake_textures_for_n3mr(np.ascontiguousarray(image), faces_uv, np.full((5856, 4, 4, 4, 3), 0.5, np.float32),
                                       np.ones(5856, np.int32), 0, True)
    assert np.abs(t.numpy() - ref).max() <= 2e-6
    assert float(t.std()) > 0.05


def test_spot_through_the_nmr_renderer_against_oracle(cuda_device, spot):
    """The textured cow through Renderer(dr_type='n3mr') (demo4's renderer): loader + ts^3 bake + lighting + transform +
    N3mrRasterizer; the rasterizer's inputs are taken from the pipeline and handed to the NMR oracle, whose rgb map the
    returned image must equal bit for bit (after the host side's transpose and vertical flip, n3mr.py:239-247)."""
    from oracle import nmr as onmr
    from jrender_b200.n3mr import vertices_to_faces
    mesh = jr.Mesh.from_obj(spot, load_texture=True, texture_res=4, dr_type='n3mr').to(cuda_device)
    assert tuple(mesh.textures.shape) == (1, 5856, 4, 4, 4, 3)
    renderer = jr.Renderer(dr_type='n3mr', image_size=256, anti_aliasing=False)
    renderer.transform.set_eyes_from_angles(2.732, 30, 40)
    mesh.reset_()
    img = renderer.render_mesh(mesh, mode='rgb')
    assert tuple(img.shape) == (1, 3, 256, 256)
    idx = torch.cat((mesh.faces, mesh.faces.flip(-1)), dim=1)          # fill_back: reversed-winding copies (rasterizer.py:83-88)
    faces = vertices_to_faces(mesh.vertices, idx).detach().cpu().numpy()
    tex = torch.cat((mesh.textures, mesh.textures.permute((0, 1, 4, 3, 2, 5))), dim=1).detach().cpu().numpy()
    ref = onmr.forward(np.ascontiguousarray(faces), np.ascontiguousarray(tex), 256, 0.1, 100.0, 1e-3, (0, 0, 0), True, False, False)
    want = np.ascontiguousarray(ref["rgb_map"].transpose(0, 3, 1, 2)[:, :, ::-1])
    got = img.detach().cpu().numpy()
    d = np.abs(got - want)
    assert np.array_equal(got, want), "max %g, %d of %d values differ" % (d.max(), int((d > 0).sum()), d.size)
    assert 0.05 < float((img.sum(1) > 0).float().mean()) < 0.6 and float(img.std()) > 0.05


def test_c1_spot_render_as_demo1_against_oracle(cuda_device, spot):
    """demo1-render.py: Mesh.from_obj(load_texture=True, texture_res=5) -> Renderer(dr_type='softras') -> render_mesh('rgb').
    The rasterizer's inputs (projected face vertices, lit T=25 textures) are taken from the pipeline and handed to the
    CPU oracle; forward compared in full, backward on every 16th row."""
    mesh = jr.Mesh.from_obj(spot, load_texture=True, texture_res=5, texture_type='surface', dr_type='softras').to(cuda_device)
    assert mesh.faces.shape[1] == 5856 and tuple(mesh.textures.shape) == (1, 5856, 25, 3)
    renderer = jr.Renderer(dr_type='softras')
    renderer.transform.set_eyes_from_angles(2.732, 30, 0)
    mesh.reset_()
    tex_leaf = mesh.textures.detach().clone().requires_grad_(True)
    mesh.textures = tex_leaf
    img = renderer.render_mesh(mesh, mode='rgb')
    assert tuple(img.shape) == (1, 3, 256, 256)      # mode='rgb': images[:, :3] (rasterizer.py:58-59)
    fv = mesh.face_vertices.detach().cpu().numpy()
    lit = mesh.textures.detach().cpu().numpy()
    assert float(lit.std()) > 0.05                                                                # textured
    P = osr.Params(image_size=256)
    ref = osr.forward(fv, lit, P)
    fn = jr.SoftRasterizeFunction(image_size=256)
    fvt = torch.from_numpy(fv).to(cuda_device).requires_grad_(True)
    txt = torch.from_numpy(lit).to(cuda_device).requires_grad_(True)
    sc, ag, ids = fn.raw(fvt, txt)
    from jrender_b200.softras import pad_face_ids
    assert np.array_equal(pad_face_ids(ids).cpu().numpy(), ref["faces_id_buffer"])
    assert np.abs(sc.detach().cpu().numpy() - ref["soft_colors"]).max() <= 2e-6
    assert 0.05 < float((sc[0, 3] > 0.5).float().mean()) < 0.6                                       # the cow is there
    assert np.abs(img.detach().cpu().numpy() - ref["soft_colors"][:, :3]).max() <= 2e-6   # the Renderer returned the same image
    g = np.zeros((1, 4, 256, 256), np.float32)
    g[:, :, ::16] = np.random.default_rng(1).uniform(-1, 1, (1, 4, 16, 256)).astype(np.float32)
    sc.backward(torch.from_numpy(g).to(cuda_device))
    rgf, rgt = osr.backward(fv, lit, ref, g, P, accumulate_double=True, row_stride=16)
    assert np.abs(fvt.grad.cpu().numpy() - rgf).max() <= 2e-5 * np.abs(rgf).max()
    assert np.abs(txt.grad.cpu().numpy() - rgt).max() <= 2e-5 * np.abs(rgt).max()
    # gradient reaches the un-lit texture leaf through the fused lighting kernel
    img.backward(torch.from_numpy(g[:, :3].copy()).to(cuda_device))
    assert tex_leaf.grad is not None and float(tex_leaf.grad.abs().max()) > 0


def test_demo4_texture_optimisation_converges(cuda_device, spot):
    """examples/demo4_optim_textures.py (port of the reference's demo4: NMR renderer, orthogonal camera, ambient light, Adam on
    a [1, nf, 4, 4, 4, 3] texture parameter): 60 iterations against a render of the cow's own baked texture must cut the
    sum-of-squares loss by more than half; and the reference's own loader call (texture_res left at 1) must not fail."""
    import warnings
    from examples import demo4_optim_textures as d4
    model, losses = d4.run(spot, None, iters=60, device=str(cuda_device))
    assert np.isfinite(losses).all() and losses[-1] < 0.5 * losses[0], (losses[0], losses[-1])
    g = model.textures.grad
    assert g is not None and float(g.abs().max()) > 0
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        m = jr.Mesh.from_obj(spot, dr_type='n3mr', load_texture=True)   # demo4-optim_textures.py:24
        assert tuple(m.textures.shape) == (1, 5856, 1, 1, 1, 3) and any("texture_res" in str(x.message) for x in w)
