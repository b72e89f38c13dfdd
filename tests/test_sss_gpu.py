"""Texture-space subsurface scattering on the GPU: the blur kernel against the reference's own kernel, SSS() against the
reference's own SSS() Python, the 2048^2 chain against the CPU oracle, and Renderer.render_mesh with with_SSS."""
import glob
import lzma
import os
import shutil

import numpy as np
import pytest

from tests.conftest import ROOT

pytestmark = pytest.mark.gpu
G = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def spot(tmp_path_factory):
    d = tmp_path_factory.mktemp("spot_sss")
    src = os.path.join(G, "spot")
    with lzma.open(os.path.join(src, "spot_triangulated.obj.xz")) as f, open(d / "spot_triangulated.obj", "wb") as g:
        shutil.copyfileobj(f, g)
    for name in ("spot_triangulated.mtl", "spot_texture.png"):
        shutil.copyfile(os.path.join(src, name), d / name)
    return str(d / "spot_triangulated.obj")


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(G, "sss_ref_gpu_blur_v*_d*.npz"))), ids=os.path.basename)
def test_blur_kernel_matches_reference_kernel(cuda_device, path):
    import torch
    from jrender_b200.lighting import sss_blur
    z = np.load(path)
    img, mod = (torch.from_numpy(z[k]).to(cuda_device) for k in ("image", "modulate"))
    got = sss_blur(img, mod, int(z["variance"]), int(z["dim"])).cpu().numpy()
    ref = z["blurred"]
    assert np.array_equal(got == 0, ref == 0)
    assert np.abs(got.astype(np.float64) - ref).max() <= 1e-6 * np.abs(ref).max()


def _golden_mesh(z, dev):
    import torch
    from jrender_b200 import Mesh
    return Mesh(torch.from_numpy(z["vertices"]).to(dev), torch.from_numpy(z["faces"]).to(dev),
                textures=torch.from_numpy(z["textures"]).to(dev), texture_res=int(z["texture_res"]), with_SSS=True,
                face_texcoords=torch.from_numpy(z["face_texcoords"]).to(dev))


def test_sss_matches_reference_sss(cuda_device):
    import torch
    from jrender_b200 import SSS
    z = np.load(os.path.join(G, "ref_host_sss_spot.npz"))
    mesh = _golden_mesh(z, cuda_device)
    d, s = (torch.from_numpy(z[k]).to(cuda_device) for k in ("diffuse", "specular"))
    got = SSS(d, s, mesh, image_size=int(z["image_size"])).cpu().numpy()
    ref = z["sss_textures"]
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max()


def test_blur_chain_2048_matches_oracle(cuda_device):
    """The three texture-space maps of spot at 2048^2 from the product rasterizer, then the chain on the GPU and in the
    CPU oracle."""
    import torch
    from jrender_b200 import SoftRasterizeFunction
    from jrender_b200.lighting import sss_blur_chain
    from oracle import sss as osss
    z = np.load(os.path.join(G, "ref_host_sss_spot.npz"))
    coords, world, irr, spec = osss.texture_space_inputs(z["vertices"][z["faces"]][None], z["face_texcoords"][None],
                                                         z["textures"], z["diffuse"], z["specular"])
    P = osss.texture_space_params(2048)
    rast = SoftRasterizeFunction(**{k: P[k] for k in ("image_size", "near", "far", "fill_back", "eps", "sigma_val", "dist_func",
                                                      "dist_eps", "gamma_val", "aggr_func_rgb", "aggr_func_alpha", "texture_type")})
    c = torch.from_numpy(coords).to(cuda_device)
    maps = [rast(c, torch.from_numpy(np.ascontiguousarray(t)).to(cuda_device))[0] for t in (world[:, :, :1], irr, spec)]
    got = sss_blur_chain(*maps).cpu().numpy()
    hwc = [m[:3].permute(1, 2, 0).cpu().numpy() for m in maps]
    ref = osss.blur_chain(*hwc)
    assert np.array_equal(got == 0, ref == 0)
    assert np.abs(got.astype(np.float64) - ref).max() <= 1e-5 * np.abs(ref).max()


def _render(spot, dev, with_sss, textures_grad=False):
    import torch
    from jrender_b200 import Mesh, Renderer
    mesh = Mesh.from_obj(spot, load_texture=True, texture_res=3, texture_type='surface', dr_type='softras', normalization=True,
                         with_SSS=with_sss).to(dev)
    if textures_grad:
        mesh.textures = mesh.textures.detach().requires_grad_(True)
    r = Renderer(dr_type='softras', image_size=128, light_intensity_ambient=0.45, light_intensity_directionals=1,
                 light_directions=[0.65, -0.2, -1], dist_func="barycentric", aggr_func_rgb='hard', camera_mode="look_at")
    r.transform.set_eyes_from_angles(2, 20, 40)
    with torch.no_grad() if not textures_grad else torch.enable_grad():
        rgb = r.render_mesh(mesh, mode='rgb')
    return rgb, mesh


def test_render_mesh_with_sss(cuda_device, spot):
    import torch
    rgb, mesh = _render(spot, cuda_device, True, textures_grad=True)
    assert mesh.textures.grad_fn is None and not mesh.textures.requires_grad     # SSS textures carry no gradient
    plain, mesh0 = _render(spot, cuda_device, False, textures_grad=True)
    assert mesh0.textures.grad_fn is not None                                    # the plain path still does
    assert rgb.shape == plain.shape and torch.isfinite(rgb).all()
    assert float(rgb.min()) >= 0 and float(rgb.max()) <= 1
    assert not torch.equal(rgb, plain)


def test_without_sss_is_the_plain_path(cuda_device, spot):
    """with_SSS=False (the loader now also keeps the UVs) renders bit-identically to a mesh built without any UVs."""
    import torch
    from jrender_b200 import Mesh
    rgb, mesh = _render(spot, cuda_device, False)
    assert mesh.face_texcoords is not None
    m2 = Mesh.from_obj(spot, load_texture=True, texture_res=3, texture_type='surface', dr_type='softras', normalization=True)
    bare = Mesh(m2._origin_vertices, m2._origin_faces, m2._origin_textures, texture_res=3).to(cuda_device)
    from jrender_b200 import Renderer
    r = Renderer(dr_type='softras', image_size=128, light_intensity_ambient=0.45, light_intensity_directionals=1,
                 light_directions=[0.65, -0.2, -1], dist_func="barycentric", aggr_func_rgb='hard', camera_mode="look_at")
    r.transform.set_eyes_from_angles(2, 20, 40)
    with torch.no_grad():
        ref = r.render_mesh(bare, mode='rgb')
    assert torch.equal(rgb, ref)


def test_sss_rejects_batch_and_missing_texcoords(cuda_device):
    import torch
    from jrender_b200 import Mesh, SSS
    z = np.load(os.path.join(G, "ref_host_sss_spot.npz"))
    mesh = _golden_mesh(z, cuda_device)
    d, s = (torch.from_numpy(z[k]).to(cuda_device) for k in ("diffuse", "specular"))
    two = Mesh(mesh.vertices.expand(2, -1, -1), mesh.faces.expand(2, -1, -1), textures=mesh.textures.expand(2, -1, -1, -1),
               texture_res=3, with_SSS=True, face_texcoords=mesh.face_texcoords)
    with pytest.raises(ValueError):
        SSS(d, s, two, image_size=64)
    bare = Mesh(mesh.vertices, mesh.faces, textures=mesh.textures, texture_res=3, with_SSS=True)
    with pytest.raises(ValueError):
        SSS(d, s, bare, image_size=64)
