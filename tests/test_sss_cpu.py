"""Texture-space subsurface scattering without a GPU: the numpy oracle (oracle/sss.py) against the reference's own blur
kernel run on a B200 and against the reference's own SSS() Python; Mesh.from_obj's UV triangles."""
import glob
import lzma
import os
import shutil

import numpy as np
import pytest

from tests.conftest import ROOT

G = os.path.join(ROOT, "tests", "golden")
# not named ref_gpu_*: tests/test_golden.py reads every ref_gpu_*.npz outside the NMR / bake families as a SoftRas fixture
BLUR_GOLDENS = sorted(glob.glob(os.path.join(G, "sss_ref_gpu_blur_v*_d*.npz")))


def test_blur_goldens_cover_every_variance_and_direction():
    names = {os.path.basename(p) for p in BLUR_GOLDENS}
    assert names == {"sss_ref_gpu_blur_v%d_d%d.npz" % (v, d) for v in (25, 75, 300) for d in (0, 1)}


@pytest.mark.parametrize("path", BLUR_GOLDENS, ids=os.path.basename)
def test_oracle_blur_matches_reference_kernel(path):
    from oracle import sss as osss
    z = np.load(path)
    tap, w = osss.taps(int(z["variance"]))
    assert np.array_equal(tap, z["taps"]) and w == z["gauss_width"]
    got = osss.blur(z["image"], z["modulate"], tap, w, int(z["dim"]))
    ref = z["blurred"]
    assert np.array_equal(got == 0, ref == 0)                   # masking and zero texels exact
    assert np.abs(got.astype(np.float64) - ref).max() <= 1e-6 * np.abs(ref).max()


def test_oracle_sss_matches_reference_sss():
    from oracle import sss as osss
    z = np.load(os.path.join(G, "ref_host_sss_spot.npz"))
    fv = z["vertices"][z["faces"]][None]
    got = osss.sss(fv, z["face_texcoords"][None], z["textures"], z["diffuse"], z["specular"], int(z["texture_res"]),
                   int(z["image_size"]))
    ref = z["sss_textures"]
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max()


@pytest.fixture()
def spot_obj(tmp_path):
    src = os.path.join(G, "spot")
    with lzma.open(os.path.join(src, "spot_triangulated.obj.xz")) as f, open(tmp_path / "spot_triangulated.obj", "wb") as g:
        shutil.copyfileobj(f, g)
    for name in ("spot_triangulated.mtl", "spot_texture.png"):
        shutil.copyfile(os.path.join(src, name), tmp_path / name)
    return str(tmp_path / "spot_triangulated.obj")


def test_from_obj_fills_face_texcoords(spot_obj, monkeypatch):
    """The bake itself runs on the GPU; here it is replaced by ones so that only the loader's UV plumbing is checked."""
    from jrender_b200 import Mesh, io
    monkeypatch.setattr(io, "load_textures", lambda fn, mtl, res: np.ones((5856, res * res, 3), np.float32))
    uv, _ = io._parse_texture_faces(spot_obj)
    m = Mesh.from_obj(spot_obj, load_texture=True, texture_res=3, dr_type='softras', with_SSS=True)
    assert m.with_SSS and tuple(m.face_texcoords.shape) == (1,) + uv.shape == (1, 5856, 3, 2)
    assert np.array_equal(m.face_texcoords[0].numpy(), uv)
    assert Mesh.from_obj(spot_obj).face_texcoords is None                       # no texture, no UVs
    v, f = io.load_obj(spot_obj)                                                # load_obj's return value is unchanged
    assert tuple(v.shape) == (m.num_vertices, 3) and tuple(f.shape) == (5856, 3)
    assert tuple(Mesh(v, f, face_texcoords=uv).face_texcoords.shape) == (1, 5856, 3, 2)   # [nf,3,2] gains the batch axis


def test_sss_rejects_bad_meshes_before_any_device_work():
    import torch
    from jrender_b200 import Mesh, SSS
    v, f = torch.rand(4, 3), torch.tensor([[0, 1, 2], [0, 2, 3]], dtype=torch.int32)
    light = torch.ones(1, 2, 1, 3)
    with pytest.raises(ValueError, match="face_texcoords"):
        SSS(light, light, Mesh(v, f, texture_res=2, with_SSS=True))
    uv = torch.rand(2, 3, 2)
    two = Mesh(torch.stack([v, v]), torch.stack([f, f]), texture_res=2, with_SSS=True, face_texcoords=uv)
    with pytest.raises(ValueError, match="batch size 1"):
        SSS(light, light, two)
