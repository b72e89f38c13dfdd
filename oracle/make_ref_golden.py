"""Generate golden vectors by running the reference's OWN kernels on a GPU (TEST INFRASTRUCTURE).

    gpurun -- python -m oracle.make_ref_golden        # writes gpurun_out/golden/ref_gpu_*.npz
    cp gpurun_out/golden/*.npz tests/golden/          # commit them

Needs oracle/_ref/libjrender_ref.so (python -m oracle.build_ref, built where /root/reference
exists; it travels to the GPU box).  The reference ships no tests or golden vectors of its own
(SURVEY.md F2), so these files are what pins oracle/softras_oracle.c to the real reference:
tests/test_golden.py compares the CPU oracle to them on every run.

Each .npz holds the inputs (face_vertices, textures, upstream gradient), the parameters, and
the reference kernels' outputs (soft_colors, aggrs_info, faces_id_buffer, faces_info,
grad_faces, grad_textures), plus the nvcc flags and GPU the reference was run with.

--large-only writes refsample_*.npz instead: stratified samples of the reference outputs at C3 / C4 sizes for the
GPU tests that compare the product with the reference there (tests/util.py).  It runs the product too, so the
product library must be built.
"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from jrender_b200 import workloads as wl  # noqa: E402
from oracle import ref_gpu, softras as osr  # noqa: E402


def fixtures():
    fv, tex = wl.make_scene(280, batch=1)
    yield "sphere280_default_64", fv, tex, dict(image_size=64)
    yield "sphere280_demo2_64", fv, tex, dict(image_size=64, sigma_val=1e-4, aggr_func_rgb="hard")
    yield "sphere280_bary_sum_48", fv, tex, dict(image_size=48, dist_func="barycentric", aggr_func_alpha="sum", sigma_val=1e-4)
    yield "sphere280_hard_hard_48", fv, tex, dict(image_size=48, dist_func="hard", aggr_func_rgb="hard", aggr_func_alpha="hard")
    fvv, texv = wl.make_scene(280, batch=1, texture_type="vertex")
    yield "sphere280_vertex_48", fvv, texv, dict(image_size=48, texture_type="vertex")
    fv5, tex5 = wl.make_scene(280, batch=1, texture_res=3)
    yield "sphere280_T9_hardrgb_48", fv5, tex5, dict(image_size=48, aggr_func_rgb="hard")
    fvr, texr = wl.random_triangles(2, 120, seed=11)
    yield "random120_K4_40", fvr, texr, dict(image_size=40, max_faces_per_pixel_for_grad=4, sigma_val=1e-4)
    fv3, tex3 = wl.make_scene(3280, batch=1)
    yield "sphere3280_default_64", fv3, tex3, dict(image_size=64)


def _fill_back(fv, tex):
    """N3mrRasterizer.render_rgb, rasterizer.py:83-88: reversed-winding copies appended, textures permuted."""
    fv = np.concatenate([fv, fv[:, :, ::-1]], axis=1)
    tex = np.concatenate([tex, tex.transpose(0, 1, 4, 3, 2, 5)], axis=1)
    return np.ascontiguousarray(fv), np.ascontiguousarray(tex)


def nmr_fixtures():
    """(name, faces [B,nf,3,3], textures [B,nf,ts,ts,ts,3], kwargs of oracle.nmr.forward)"""
    rng = np.random.default_rng(5)
    fv, _ = wl.make_scene(280, batch=1)
    tex = rng.random((1, fv.shape[1], 2, 2, 2, 3), dtype=np.float32)
    f2, t2 = _fill_back(fv, tex)
    yield "nmr_sphere280_fillback_ts2_64", f2, t2, dict(image_size=64, near=0.1, far=100.0, eps=1e-3, background_color=(0, 0, 0),
                                                        return_rgb=True, return_alpha=True, return_depth=True)
    # (texture_size 1 is left out on purpose: the reference's trilinear taps then leave the face's
    # block and, for the last faces, the tensor -- undefined behaviour; see oracle/nmr_oracle.c K8)
    tex1 = rng.random((1, fv.shape[1], 4, 4, 4, 3), dtype=np.float32)
    yield "nmr_sphere280_ts4_bg_48", fv, tex1, dict(image_size=48, near=0.1, far=100.0, eps=1e-3, background_color=(0.2, 0.4, 0.6),
                                                    return_rgb=True, return_alpha=True, return_depth=False)
    fvr, _ = wl.random_triangles(2, 120, seed=11)
    texr = rng.random((2, 120, 3, 3, 3, 3), dtype=np.float32)
    yield "nmr_random120_ts3_nearfar_32", fvr, texr, dict(image_size=32, near=1.5, far=3.0, eps=1e-3, background_color=(1, 1, 1),
                                                          return_rgb=True, return_alpha=False, return_depth=True)
    fv3, _ = wl.make_scene(3280, batch=1)
    tex3 = rng.random((1, fv3.shape[1], 2, 2, 2, 3), dtype=np.float32)
    f3, t3 = _fill_back(fv3, tex3)
    yield "nmr_sphere3280_alpha_64", f3, t3, dict(image_size=64, near=0.1, far=100.0, eps=1e-3, background_color=(0, 0, 0),
                                                  return_rgb=False, return_alpha=True, return_depth=False)


def nmr_main(out_dir, report):
    import torch
    from oracle import nmr as onmr
    for name, faces, tex, kw in nmr_fixtures():
        H = kw["image_size"]
        B = faces.shape[0]
        flags = (kw["return_rgb"], kw["return_alpha"], kw["return_depth"])
        rng = np.random.default_rng(7)
        grads = (rng.uniform(-1, 1, (B, H, H, 3)).astype(np.float32), rng.uniform(-1, 1, (B, H, H)).astype(np.float32),
                 rng.uniform(-1, 1, (B, H, H)).astype(np.float32))
        ref = ref_gpu.nmr_run(faces, tex, H, kw["near"], kw["far"], kw["eps"], kw["background_color"], flags, grads)
        cpu = onmr.forward(faces, tex if flags[0] else None, **kw)
        gf, gt = onmr.backward(faces, tex if flags[0] else None, cpu, H, kw["eps"], grads[0], grads[1], grads[2], *flags)
        cpu["grad_faces"] = gf
        if gt is not None:
            cpu["grad_textures"] = gt
        save = dict(faces=faces, textures=tex, grad_rgb_map=grads[0], grad_alpha_map=grads[1], grad_depth_map=grads[2],
                    params=json.dumps(kw),
                    provenance=json.dumps(dict(gpu=torch.cuda.get_device_name(0),
                                               nvcc="12.9 -O3 -gencode arch=compute_100a,code=sm_100a (fmad default on)",
                                               source="jrender/renderer/dr/n3mr/cuda/rasterize.py kernels via oracle/build_ref.py")))
        for k, v in ref.items():
            if k in ("alpha_map", "rgb_raw"):
                continue  # alpha = (face_index_map >= 0); rgb_raw = rgb_map before the background mix
            save[k] = v.astype(np.int16) if k == "face_index_map" and faces.shape[1] < 32767 else v
        np.savez_compressed(os.path.join(out_dir, "ref_gpu_%s.npz" % name), **save)
        r = dict(name=name, face_index_equal_frac=float((ref["face_index_map"] == cpu["face_index_map"]).mean()))
        same = ref["face_index_map"] == cpu["face_index_map"]
        for k in ("weight_map", "depth_map", "rgb_map", "sampling_index_map", "sampling_weight_map", "face_inv_map",
                  "grad_faces", "grad_textures"):
            if k not in ref or cpu.get(k) is None:
                continue
            a, b = ref[k].astype(np.float64), np.asarray(cpu[k]).astype(np.float64)
            if a.shape[:3] == same.shape and k not in ("grad_faces", "grad_textures"):
                m = np.broadcast_to(same.reshape(same.shape + (1,) * (a.ndim - 3)), a.shape)   # pixels where both picked the same face
            else:
                m = np.ones(a.shape, bool)
            m = m & ~(np.isnan(a) | np.isnan(b))
            d = np.abs(a - b)[m]
            r[k] = dict(max_abs=float(d.max()) if d.size else 0.0, mean_abs=float(d.mean()) if d.size else 0.0,
                        max_ref=float(np.abs(a[m]).max()) if d.size else 0.0)
        report.append(r)
        print(json.dumps(r), flush=True)


def bake_main(out_dir):
    """Reference texture-bake kernel (io/utils/load_textures.py:3-101 via oracle/build_ref.py) on seeded inputs ->
    ref_gpu_bake_random40_R5.npz; prints the difference to the numpy oracle (oracle/bake.py)."""
    import ctypes as C
    import torch
    from oracle import bake as obake
    rng = np.random.default_rng(7)
    nf, R, H, W = 40, 5, 24, 40
    image = rng.random((H, W, 3), dtype=np.float32)
    uv = rng.uniform(0.02, 0.95, (nf, 3, 2)).astype(np.float32)
    upd = (rng.random(nf) > 0.2).astype(np.int32)
    tex0 = np.full((nf, R * R, 3), 0.5, np.float32)
    L = ref_gpu.lib()
    L.ref_bake_textures_softras.restype = C.c_int
    L.ref_bake_textures_softras.argtypes = [C.c_void_p] * 4 + [C.c_int] * 4
    dev = torch.device("cuda:0")
    t = [torch.from_numpy(a).to(dev) for a in (image, uv, upd, tex0)]
    rc = L.ref_bake_textures_softras(*[C.c_void_p(x.data_ptr()) for x in t], nf, R, H, W)
    assert rc == 0, rc
    ref = t[3].cpu().numpy()
    cpu = obake.bake_textures_for_softras(image, uv, tex0, upd)
    np.savez_compressed(os.path.join(out_dir, "ref_gpu_bake_random40_R5.npz"), image=image, faces_uv=uv, is_update=upd, textures_in=tex0,
                        textures=ref, provenance=json.dumps(dict(gpu=torch.cuda.get_device_name(0), source="jrender/io/utils/load_textures.py:3-101 via oracle/build_ref.py")))
    print(json.dumps(dict(name="bake_random40_R5", max_abs_vs_oracle=float(np.abs(ref - cpu).max()))), flush=True)


def bake_n3mr_main(out_dir):
    """Reference NMR texture-bake kernel (io/utils/load_textures.py:103-246 via oracle/build_ref.py, one build per
    wrapping mode / sampling flavour) on seeded inputs -> ref_gpu_bake_n3mr_w<W>_b<B>.npz.

    The reference wraps the UVs in place from every thread of a face; the fixtures stay away from the values for which
    that race has more than one outcome: no integer UVs (REPEAT maps 0 -> 1 -> 0), and for MIRRORED_REPEAT only UVs with an
    even integer part (the reference re-reads the value between testing mod(x, 2) < 1 and wrapping, so a value another
    thread has already mirrored would be mirrored back)."""
    import ctypes as C
    import torch
    from oracle import bake as obake
    L = ref_gpu.lib()
    dev = torch.device("cuda:0")
    nf, ts, H, W = 40, 4, 37, 53
    for wrap, bil in ((0, 1), (0, 0), (1, 1), (2, 1), (2, 0), (3, 1)):
        rng = np.random.default_rng(11 + 2 * wrap + bil)
        image = rng.random((H, W, 3), dtype=np.float32)
        if wrap == 1:
            uv = (rng.uniform(0.02, 0.98, (nf, 3, 2)) + 2.0 * rng.integers(-1, 2, (nf, 3, 2))).astype(np.float32)
        else:
            uv = rng.uniform(-1.4, 2.4, (nf, 3, 2)).astype(np.float32)
            uv[np.abs(uv - np.round(uv)) < 1e-3] += np.float32(0.01)
        upd = (rng.random(nf) > 0.2).astype(np.int32)
        tex0 = np.full((nf, ts, ts, ts, 3), 0.5, np.float32)
        fn = getattr(L, "ref_bake_textures_n3mr_%d_%d" % (wrap, bil))
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p] * 4 + [C.c_int] * 4
        t = [torch.from_numpy(a.copy()).to(dev) for a in (image, uv, upd, tex0)]
        rc = fn(*[C.c_void_p(x.data_ptr()) for x in t], nf, ts, H, W)
        assert rc == 0, rc
        ref = t[3].cpu().numpy()
        cpu = obake.bake_textures_for_n3mr(image, uv, tex0, upd, wrap, bool(bil))
        name = "ref_gpu_bake_n3mr_w%d_b%d" % (wrap, bil)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), image=image, faces_uv=uv, is_update=upd, textures_in=tex0, textures=ref,
                            texture_wrapping=wrap, use_bilinear=bil,
                            provenance=json.dumps(dict(gpu=torch.cuda.get_device_name(0), source="jrender/io/utils/load_textures.py:103-246 via oracle/build_ref.py")))
        print(json.dumps(dict(name=name, max_abs_vs_oracle=float(np.abs(ref - cpu).max()))), flush=True)


# Fixtures of the GPU tests that compare the product with the reference kernels at sizes the CPU oracle cannot reach
# (test_softras_gpu.py::test_against_reference_kernels_on_gpu, test_nmr_gpu.py::test_c4_against_reference_kernels_on_gpu).
# Whole outputs are tens of MB there, so a stratified sample is kept (tests/util.py:softras_fixture, nmr_fixture); the
# strata follow where the product built from this tree disagrees with the reference, so build it first.
# Sample sizes per fixture: the estimates must sit well inside the tests' tolerances over resampling (measured on a
# B200 over 30 seeds).  39 200 faces at 1024^2 puts grad_faces at 0.097 against a bound of 0.10, so the 2048 faces
# that carry most of that difference are all kept; NMR gradients sit 100x inside their bounds.
LARGE_SOFTRAS = {(3280, 512): dict(n_pixels=1024, n_worst_faces=512, n_faces=512),
                 (39200, 512): dict(n_pixels=1024, n_worst_faces=512, n_faces=512),
                 (39200, 1024): dict(n_pixels=2048, n_worst_faces=2048, n_faces=1024)}
SAMPLE_C4 = dict(n_pixels=2048, n_worst_faces=256, n_faces=256)


def large_main(out_dir):
    import torch
    from tests import util
    prov = lambda src: json.dumps(dict(gpu=torch.cuda.get_device_name(0), source=src + " via oracle/build_ref.py",   # noqa: E731
                                       nvcc="12.9 -O3 -gencode arch=compute_100a,code=sm_100a (fmad default on)"))
    for (nf, H), sample in LARGE_SOFTRAS.items():
        fv, tex, g = util.large_softras_inputs(nf, H)
        P = osr.Params(image_size=H)
        ref, got = ref_gpu.run(fv, tex, P, grad=g), util.run_cuda(fv, tex, P, grad=g, want_faces_info=False)
        np.savez_compressed(os.path.join(out_dir, "refsample_softras_%d_%d.npz" % (nf, H)), input_sums=util.input_sums(fv, tex, g),
                            provenance=prov("jrender/renderer/dr/softras/cuda/soft_rasterize.py kernels"),
                            **util.softras_fixture(ref, got, **sample))
    faces, tex, g, ga = util.c4_inputs()
    args = (faces, tex, 1024, 0.1, 100.0, 1e-3, (0, 0, 0), (True, True, False), (g, ga, None))
    ref, got = ref_gpu.nmr_run(*args), util.run_nmr_cuda(*args)
    np.savez_compressed(os.path.join(out_dir, "refsample_nmr_c4_1024.npz"), input_sums=util.input_sums(faces, tex, g, ga),
                        provenance=prov("jrender/renderer/dr/n3mr/cuda/rasterize.py kernels"),
                        **util.nmr_fixture(ref, got, far=100.0, **SAMPLE_C4))


def main():
    import torch
    out_dir = os.path.join("gpurun_out", "golden")
    os.makedirs(out_dir, exist_ok=True)
    report = []
    if "--large-only" in sys.argv:
        large_main(out_dir)
        return
    if "--bake-only" in sys.argv:
        bake_main(out_dir)
        bake_n3mr_main(out_dir)
        return
    if "--nmr-only" in sys.argv:
        nmr_main(out_dir, report)
        json.dump(report, open(os.path.join(out_dir, "report_nmr.json"), "w"), indent=1)
        return
    for name, fv, tex, kw in fixtures():
        P = osr.Params(**kw)
        H = P["image_size"]
        g = np.random.default_rng(2).uniform(-1, 1, (fv.shape[0], 4, H, H)).astype(np.float32)
        ref = ref_gpu.run(fv, tex, P, grad=g)
        cpu = osr.forward(fv, tex, P)
        cpu["grad_faces"], cpu["grad_textures"] = osr.backward(fv, tex, cpu, g, P)
        ids_ref = ref["faces_id_buffer"]
        assert ids_ref.max() < 32767
        np.savez_compressed(
            os.path.join(out_dir, "ref_gpu_%s.npz" % name),
            face_vertices=fv, textures=tex, grad_soft_colors=g,
            params=json.dumps(dict(P)), soft_colors=ref["soft_colors"], aggrs_info=ref["aggrs_info"],
            faces_id_buffer=ids_ref.astype(np.int16), faces_info=ref["faces_info"],
            grad_faces=ref["grad_faces"], grad_textures=ref["grad_textures"],
            provenance=json.dumps(dict(gpu=torch.cuda.get_device_name(0), nvcc="12.9 -O3 -gencode arch=compute_100a,code=sm_100a (fmad default on)",
                                       source="jrender/renderer/dr/softras/cuda/soft_rasterize.py kernels via oracle/build_ref.py")))
        r = dict(name=name)
        r["ids_equal_px_frac"] = float((np.sort(ids_ref, 1) == np.sort(cpu["faces_id_buffer"], 1)).all(1).mean())
        r["ids_exact"] = bool(np.array_equal(ids_ref, cpu["faces_id_buffer"]))
        for k in ("soft_colors", "aggrs_info", "faces_info", "grad_faces", "grad_textures"):
            a, b = ref[k].astype(np.float64), cpu[k].astype(np.float64)
            m = ~(np.isnan(a) | np.isnan(b))
            d = np.abs(a - b)[m]
            r[k] = dict(max_abs=float(d.max()) if d.size else 0.0, mean_abs=float(d.mean()) if d.size else 0.0,
                        max_ref=float(np.abs(a[m]).max()) if d.size else 0.0, nan_ref=int(np.isnan(a).sum()), nan_cpu=int(np.isnan(b).sum()))
        report.append(r)
        print(json.dumps(r), flush=True)
    nmr_main(out_dir, report)
    json.dump(report, open(os.path.join(out_dir, "report.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
