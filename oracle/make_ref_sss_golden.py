"""Golden vectors of texture-space subsurface scattering (TEST INFRASTRUCTURE).

    python -m oracle.make_ref_sss_golden --host [--out DIR]   needs /root/reference: ref_host_sss_spot.npz
    python -m oracle.make_ref_sss_golden --gpu [--out DIR]    needs a GPU and oracle/_ref/libjrender_ref_sss.so
                                                               (oracle/build_ref_sss.py): sss_ref_gpu_blur_*.npz

--host runs the reference's own SSS() Python (read in place, through oracle/jittor_numpy_stub.py) on the spot cow with
the three CUDA ops replaced by the CPU oracles.  --gpu runs the reference's own blur kernel on seeded 256^2 inputs for
every variance and direction and prints its difference to oracle/sss.py.  DIR defaults to tests/golden.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import build_ref_sss  # noqa: E402
from oracle.make_ref_host_golden import REF, reference_functions  # noqa: E402


def sss_blur_inputs(S=256, seed=21):
    """A stretch-like modulate map in [0, 1] and an image with zero regions, texels below the 1e-6 masking threshold and
    negative values: the cases of the reference blur's masking and clamping."""
    rng = np.random.default_rng(seed)
    img = (rng.integers(1, 64, (S, S)) / 64).astype(np.float32)   # multiples of 1/64: the fixtures compress well
    img[40:70, :] = 0
    img[:, 100:104] = 0
    img[150:170, 150:190] = 5e-7
    img[200:210, 20:60] = -0.5
    mod = np.clip(rng.integers(0, 84, (S, S)) / 64, 0, 1).astype(np.float32)
    mod[0:16, :] = 1
    mod[100:120, :] = 0
    return img, mod


def sss_main(out_dir):
    """The reference's SSS blur kernel (renderer/utils/gaussian_blur.py:34-165 via oracle/build_ref_sss.py) at 256^2 for every
    variance of SSS() and both directions -> sss_ref_gpu_blur_v{25,75,300}_d{0,1}.npz; prints the difference to oracle/sss.py."""
    import ctypes as C
    import torch
    from oracle import sss as osss
    L = build_ref_sss.lib()
    dev = torch.device("cuda:0")
    img, mod = sss_blur_inputs()
    S = img.shape[0]
    for v in (25, 75, 300):
        tap, w = osss.taps(v)
        for dim in (0, 1):
            t = [torch.from_numpy(a).to(dev) for a in (img, mod, tap)]
            out = torch.empty_like(t[0])
            rc = L.ref_sss_blur(*[C.c_void_p(x.data_ptr()) for x in t + [out]], S, S, 7, float(w), dim, None)
            torch.cuda.synchronize()
            assert rc == 0, rc
            ref = out.cpu().numpy()
            cpu = osss.blur(img, mod, tap, w, dim)
            np.savez_compressed(os.path.join(out_dir, "sss_ref_gpu_blur_v%d_d%d.npz" % (v, dim)), image=img, modulate=mod, taps=tap,
                                gauss_width=np.float32(w), variance=v, dim=dim, blurred=ref,
                                provenance=json.dumps(dict(gpu=torch.cuda.get_device_name(0), nvcc="12.9 -O3 -gencode arch=compute_100a,code=sm_100a (fmad default on)",
                                                           source="jrender/renderer/utils/gaussian_blur.py:34-165 via oracle/build_ref_sss.py")))
            d = np.abs(ref.astype(np.float64) - cpu)
            print(json.dumps(dict(name="sss_blur_v%d_d%d" % (v, dim), max_abs_vs_oracle=float(d.max()), max_ref=float(np.abs(ref).max()),
                                  zero_pattern_equal=bool(np.array_equal(ref == 0, cpu == 0)))), flush=True)


def sss_spot(stub, fns, out_dir, image_size=256, texture_res=3):
    """The reference's own SSS() (renderer/lighting/lighting.py:86-156, utils/gaussian_blur.py, utils/ToStretchMap.py),
    called from its own Lighting.execute on its own Mesh of the spot cow with with_SSS=True.  The three jt.code ops come
    from the oracles: the SoftRas forward (oracle/softras.py), the blur kernel (oracle/sss.py) and the texture bake
    (oracle/bake.py); the texture-space size is image_size instead of the literal 2048.  -> ref_host_sss_spot.npz"""
    import lzma
    import re
    import tempfile
    import types
    jt = sys.modules["jittor"]
    jt.nn.ModuleList = list
    # the calls SSS(), gaussian_blur and computeStretchMap make beyond what the stub provides
    jt.concat = stub.concat
    jt.full = lambda shape, val, dtype="float32": np.full((shape,) if isinstance(shape, int) else tuple(shape), val, dtype).view(stub.Var)
    jt.zeros_like = lambda a: np.zeros_like(np.asarray(a)).view(stub.Var)
    jt.int32 = np.int32
    jt.float32 = np.float32
    sys.path.insert(0, ROOT)
    from jrender_b200 import io as jio
    from oracle import bake as obake, softras as osr, sss as osss

    def load(rel, strip, inject, sub=()):
        path = os.path.join(REF, rel)
        src = re.sub(strip, "", open(path).read(), flags=re.M)
        for a, b in sub:
            assert a in src, a
            src = src.replace(a, b)
        mod = types.ModuleType("ref_" + os.path.basename(rel)[:-3])
        mod.__dict__.update(inject)
        exec(compile(src, path, "exec"), mod.__dict__)
        return mod

    def fwd_softras(face_vertices, textures, faces_info, aggrs_info, soft_colors, faces_id_buffer, image_size, near, far, eps,
                    sigma_val, func_dist_type, dist_eps, gamma_val, func_rgb_type, func_alpha_type, texture_type, fill_back):
        P = osr.Params(image_size=int(image_size), near=near, far=far, eps=eps, sigma_val=sigma_val,
                       dist_func={0: "hard", 1: "barycentric", 2: "euclidean"}[int(func_dist_type)],
                       dist_eps=1.0 / (1.0 + np.exp(dist_eps)), gamma_val=gamma_val,
                       aggr_func_rgb={0: "hard", 1: "softmax", 2: "none"}[int(func_rgb_type)],
                       aggr_func_alpha={0: "hard", 1: "sum", 2: "prod"}[int(func_alpha_type)],
                       texture_type={0: "surface", 1: "vertex"}[int(texture_type)], fill_back=bool(fill_back),
                       max_faces_per_pixel_for_grad=int(np.asarray(faces_id_buffer).shape[1]))
        out = osr.forward(np.ascontiguousarray(face_vertices, np.float32), np.ascontiguousarray(textures, np.float32), P)
        return tuple(stub.array(out[k]) for k in ("faces_info", "aggrs_info", "soft_colors", "faces_id_buffer"))

    def blur_op(image_blur, image, modulate_map, Gauss, tap_num, GaussWidth, dim):   # _blur_for_SSS, d = 1, out shaped like image_blur
        img = np.asarray(image, np.float32)[:, :, 0]
        out = osss.blur(img, np.asarray(modulate_map, np.float32), np.asarray(Gauss, np.float32), np.float32(GaussWidth), int(dim))
        return stub.array(out.reshape(np.asarray(image_blur).shape))

    def bake_op(image, faces, textures, is_update):
        return stub.array(obake.bake_textures_for_softras(np.asarray(image, np.float32), np.asarray(faces, np.float32),
                                                          np.asarray(textures, np.float32), np.asarray(is_update, np.int32)))
    s1 = load("renderer/dr/softras/soft_rasterize.py", r"^(from \.cuda.*)$",
              dict(soft_rasterize_cuda=types.SimpleNamespace(forward_soft_rasterize=fwd_softras)))
    gb = load("renderer/utils/gaussian_blur.py", r"^$", {})
    gb._blur_for_SSS = blur_op
    sm = load("renderer/utils/ToStretchMap.py", r"^$", {})
    amb = stub.load_reference_function(os.path.join(REF, "renderer/lighting/ambient_lighting.py"), "ambient_lighting")
    dmod = load("renderer/lighting/directional_lighting.py", r"^$", {})
    lmod = load("renderer/lighting/lighting.py", r"^(from jrender\..*|from skimage.*|from \. import \*)$",
                dict(ambient_lighting=amb, directional_lighting=dmod.directional_lighting, SoftRasterizeFunction=s1.SoftRasterizeFunction,
                     _load_textures_for_softras=bake_op, gaussian_blur=gb.gaussian_blur, computeStretchMap=sm.computeStretchMap),
                sub=[("image_size = 2048", "image_size = %d" % image_size)])
    mmod = load("structures/mesh.py", r"^(from \.\.io import \*|from \.utils import \*)$", dict(face_vertices=fns["face_vertices"]))
    captured = {}
    ref_sss = lmod.SSS

    def sss_capture(diffuseLight, specular, mesh):
        captured["diffuse"], captured["specular"] = np.asarray(diffuseLight, np.float32), np.asarray(specular, np.float32)
        out = ref_sss(diffuseLight, specular, mesh)
        captured["sss"] = np.asarray(out, np.float32)
        return out
    lmod.SSS = sss_capture

    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(ROOT, "tests", "golden", "spot")
        obj = os.path.join(d, "spot.obj")
        with lzma.open(os.path.join(src, "spot_triangulated.obj.xz")) as f, open(obj, "wb") as g:
            g.write(f.read())
        v, f = jio.load_obj(obj, normalization=True)
        uv, _ = jio._parse_texture_faces(obj)
    image = np.ascontiguousarray(jio._imread_rgb01(os.path.join(ROOT, "tests", "golden", "spot", "spot_texture.png"))[::-1])
    nf = uv.shape[0]
    tex = obake.bake_textures_for_softras(image, uv, np.ones((nf, texture_res ** 2, 3), np.float32), np.ones(nf, np.int32))
    mesh = mmod.Mesh(stub.array(v.numpy()), stub.array(f.numpy()), textures=stub.array(tex[None]), texture_res=texture_res,
                     dr_type="softras", with_SSS=True, face_texcoords=stub.array(uv))
    eye = [[1.1, 0.5, -1.5]]
    light = lmod.Lighting(intensity_ambient=0.45, intensity_directionals=1.0, directions=[0.65, -0.2, -1])
    light(mesh, stub.array(eye))   # mesh.textures becomes clamp(SSS(...), 0, 1)
    res = dict(vertices=v.numpy(), faces=f.numpy(), face_texcoords=uv, textures=tex[None], eye=np.asarray(eye, np.float32),
               diffuse=captured["diffuse"], specular=captured["specular"], sss_textures=captured["sss"],
               image_size=image_size, texture_res=texture_res)
    np.savez_compressed(os.path.join(out_dir, "ref_host_sss_spot.npz"), **res)
    print("wrote ref_host_sss_spot.npz", res["sss_textures"].shape, float(res["sss_textures"].mean()))


def main():
    out_dir = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    if "--gpu" in sys.argv:
        sss_main(out_dir)
    if "--host" in sys.argv:
        fns, stub, restore = reference_functions()
        try:
            sss_spot(stub, fns, out_dir)
        finally:
            restore()


if __name__ == "__main__":
    main()
