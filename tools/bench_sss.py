"""Timing of texture-space subsurface scattering on one GPU, with the reference's blur kernels for comparison.

    python tools/bench_sss.py [--iters 20] [--warmup 3]

Prints one JSON line: the GPU name and power limit; ms of the blur chain (b200r_sss_blur_chain, 7 launches) and of a whole
SSS() call (three 2048^2 texture-space rasterizations, the chain and the bake) on the spot cow with texture_res=15; the
reference's blur (36 launches of its own kernel, built by oracle/build_ref_sss.py into oracle/_ref) on the same maps; and
algorithmic bytes over kernel time for both blurs.  Times are CUDA events around `iters` back-to-back calls.
"""
import argparse
import ctypes as C
import json
import lzma
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--image-size", type=int, default=2048)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sss.py measures on a CUDA device; none found")
    import jrender_b200 as jr
    from jrender_b200.lighting import SSS, sss_blur_chain, directional_lighting, ambient_lighting
    from oracle import sss as osss
    dev = torch.device("cuda:0")
    S = args.image_size
    tmp = tempfile.mkdtemp()
    try:
        src = os.path.join(ROOT, "tests", "golden", "spot")
        with lzma.open(os.path.join(src, "spot_triangulated.obj.xz")) as f, open(os.path.join(tmp, "spot.obj"), "wb") as g:
            shutil.copyfileobj(f, g)
        for name in ("spot_triangulated.mtl", "spot_texture.png"):
            shutil.copyfile(os.path.join(src, name), os.path.join(tmp, name))
        mesh = jr.Mesh.from_obj(os.path.join(tmp, "spot.obj"), load_texture=True, texture_res=15, dr_type='softras', normalization=True, with_SSS=True).to(dev)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    nf = mesh.num_faces
    diffuse = ambient_lighting(torch.zeros((1, nf, 3), device=dev), 0.45)
    diffuse, specular = directional_lighting(diffuse, torch.zeros_like(diffuse), mesh.surface_normals, 1.0, (1, 1, 1), (0.65, -0.2, -1))
    diffuse, specular = diffuse[:, :, None], specular[:, :, None]

    # the three texture-space maps, once, for the chain-only timings
    coords, world, irr, spec = osss.texture_space_inputs(mesh.face_vertices.cpu().numpy(), mesh.face_texcoords.cpu().numpy(),
                                                         mesh.textures.cpu().numpy(), diffuse.cpu().numpy(), specular.cpu().numpy())
    P = osss.texture_space_params(S)
    rast = jr.SoftRasterizeFunction(**{k: P[k] for k in ("image_size", "near", "far", "fill_back", "eps", "sigma_val", "dist_func",
                                                         "dist_eps", "gamma_val", "aggr_func_rgb", "aggr_func_alpha", "texture_type")})
    c = torch.from_numpy(coords).to(dev)
    maps = [rast(c, torch.from_numpy(np.ascontiguousarray(t)).to(dev))[0].contiguous() for t in (world[:, :, :1], irr, spec)]

    res = {}
    res["gpu"], res["power_limit"] = gpu_info()
    res["image_size"], res["num_faces"], res["texture_res"] = S, nf, 15
    res["chain_ms"] = timed(lambda: sss_blur_chain(*maps), args.iters, args.warmup)
    res["sss_call_ms"] = timed(lambda: SSS(diffuse, specular, mesh, image_size=S), args.iters, args.warmup)

    # algorithmic bytes of the chain: stretch (read 3 planes, write 2), 6 passes (read 4 planes, write 4; the y passes
    # also read / write the accumulator, the last reads irradiance + specular and writes the [S,S,3] map)
    plane = S * S * 4
    chain_bytes = plane * (3 + 2) + 6 * plane * 8 + plane * (3 + 6 + 3 + 6)
    res["chain_GBps"] = chain_bytes / (res["chain_ms"] * 1e-3) / 1e9

    from oracle import build_ref_sss
    if build_ref_sss.available():
        L = build_ref_sss.lib()
        su, sv = (torch.from_numpy(m).to(dev) for m in osss.stretch_maps(maps[0][:3].permute(1, 2, 0).cpu().numpy()))
        irr_c = [maps[1][k].clone() for k in range(3)]
        tap_t = [torch.from_numpy(osss.taps(v)[0]).to(dev) for v in (25, 75, 300)]
        widths = [float(osss.taps(v)[1]) for v in (25, 75, 300)]
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        p = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731
        bufs = [[torch.empty((S, S), device=dev) for _ in range(2)] for _ in range(4)]   # U, V, irradiance x, irradiance y

        def ref_chain():   # lighting.py:133-143: per channel, 3 variances x (U, irradiance x, V, irradiance y) = 36 launches
            for ch in range(3):
                u, v, x = su, sv, irr_c[ch]
                for i in range(3):
                    nu, nx, nv, ny = bufs[0][i & 1], bufs[2][i & 1], bufs[1][i & 1], bufs[3][i & 1]
                    L.ref_sss_blur(p(u), p(u), p(tap_t[i]), p(nu), S, S, 7, widths[i], 1, st)
                    L.ref_sss_blur(p(x), p(nu), p(tap_t[i]), p(nx), S, S, 7, widths[i], 1, st)
                    L.ref_sss_blur(p(v), p(v), p(tap_t[i]), p(nv), S, S, 7, widths[i], 0, st)
                    L.ref_sss_blur(p(nx), p(nv), p(tap_t[i]), p(ny), S, S, 7, widths[i], 0, st)
                    u, v, x = nu, nv, ny
        res["ref_blur_36_launches_ms"] = timed(ref_chain, args.iters, args.warmup)
        res["ref_blur_GBps"] = 36 * 3 * plane / (res["ref_blur_36_launches_ms"] * 1e-3) / 1e9   # read image + modulate, write out
        res["blur_speedup_vs_ref"] = res["ref_blur_36_launches_ms"] / res["chain_ms"]
    else:
        res["ref_blur_36_launches_ms"] = "not measured (oracle/_ref not built)"
    print(json.dumps(res))


if __name__ == "__main__":
    main()
