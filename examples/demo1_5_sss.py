"""Rendering a mesh with texture-space subsurface scattering from a circle of viewpoints: port of the reference's
demo1.5-SSS.py -- same loader call (with_SSS=True, texture_res=15, normalization), renderer kwargs and camera path.
Frames are written as PNG files.

The reference renders its head model (data/head/head.obj, with a normal map); pass it with -i.  The default input is the
spot cow.  Normal maps are not applied by this package, so the head renders with its geometric normals.

    python examples/demo1_5_sss.py [-i data/head/head.obj] [-o out/] [--step 4]
"""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import jrender_b200 as jr  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_OBJ = os.path.join(ROOT, "baseline", "_ref", "assets", "data", "obj", "spot", "spot_triangulated.obj")


def save_png(path, chw):
    import cv2
    img = (255 * chw.detach().clamp(0, 1).cpu().numpy().transpose(1, 2, 0)).astype(np.uint8)
    cv2.imwrite(path, img[:, :, ::-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('-i', '--filename-input', type=str, default=DEFAULT_OBJ)
    ap.add_argument('-o', '--output-dir', type=str, default='output_render_sss')
    ap.add_argument('--step', type=int, default=4, help="azimuth step in degrees (demo1.5: 4)")
    args = ap.parse_args()
    camera_distance, elevation = 2, 20
    dev = torch.device('cuda:0')
    print("note: normal maps (map_normal) are not applied; shading uses the geometric normals")

    mesh = jr.Mesh.from_obj(args.filename_input, load_texture=True, texture_res=15, texture_type='surface', dr_type='softras',
                            normalization=True, with_SSS=True).to(dev)
    renderer = jr.Renderer(dr_type='softras', image_size=1024, light_intensity_ambient=0.45, light_color_ambient=[1, 1, 1],
                           light_intensity_directionals=1, light_color_directionals=[1.0, 1.0, 1.0],
                           light_directions=[0.65, -0.2, -1], dist_func="barycentric", aggr_func_rgb='hard',
                           camera_mode="look_at", eye=[1.1, 0.5, -1.5], camera_direction=[-0.8, -0.2, 1])
    os.makedirs(args.output_dir, exist_ok=True)
    with torch.no_grad():
        for num, azimuth in enumerate(range(0, 360, args.step)):
            mesh.reset_()
            renderer.transform.set_eyes_from_angles(camera_distance, elevation, azimuth)
            rgb = renderer.render_mesh(mesh, mode='rgb')
            save_png(os.path.join(args.output_dir, 'head_rotation_%03d.png' % num), rgb[0])
    print("wrote %d frames to %s" % (len(os.listdir(args.output_dir)), args.output_dir))


if __name__ == '__main__':
    main()
