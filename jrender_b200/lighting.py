"""Lighting: the surface-mode path (the renderer's default) runs as ONE fused kernel forward and one backward
(csrc/lighting_api.cu, SURVEY.md section 8f rank 1); everything else is the op-by-op PyTorch mirror below.

Mirrors jrender/renderer/lighting/{ambient_lighting,directional_lighting,lighting}.py for the
paths the rasterizer demos use: ambient + directional light in 'surface' and 'vertex' modes,
including the Cook-Torrance specular branch the reference takes by default
(Mesh.with_specular defaults to True, structures/mesh.py:74), and texture-space subsurface scattering
(Mesh.with_SSS, SSS below).  Normal-mapped meshes (surface_ResNormals) and the Gbuffer debug modes are not mirrored.
"""
import ctypes as C
import math

import torch
from torch import nn
import torch.nn.functional as F

from . import _lib


_CONST = {}


def _t(x, like):
    """Python constants (light colours / directions) live on the device once per (value, device):
    building them per call is a pageable H2D copy, which stalls the stream and cannot be captured
    in a CUDA graph."""
    if isinstance(x, torch.Tensor):
        return x.to(device=like.device, dtype=torch.float32)
    key = (repr(x), str(like.device))
    t = _CONST.get(key)
    if t is None:
        t = _CONST[key] = torch.tensor(x, dtype=torch.float32, device=like.device)
    return t


def ambient_lighting(light, light_intensity=0.5, light_color=(1, 1, 1)):
    """ambient_lighting.py:4-9."""
    light_color = _t(light_color, light)
    if light_color.dim() == 1:
        light_color = light_color[None, :]
    return light + light_intensity * light_color[:, None, :]


def GGX(N, H, roughness):
    a = roughness * roughness
    a2 = a * a
    NdotH = F.relu(torch.sum(N * H, dim=2))
    NdotH2 = (NdotH * NdotH)[:, :, None]
    denom = (NdotH2 * (a2 - 1.0) + 1.0)
    denom = 3.1415 * denom * denom
    return a2 / denom


def SchlickGGX(NdotV, roughness):
    r = roughness + 1.0
    k = (r * r) / 8.0
    NdotV = NdotV[:, :, None]
    return NdotV / (NdotV * (1.0 - k) + k)


def GeometrySmith(N, V, L, roughness):
    NdotV = F.relu(torch.sum(N * V, dim=2))
    NdotL = F.relu(torch.sum(N * L, dim=2))
    return SchlickGGX(NdotL, roughness) * SchlickGGX(NdotV, roughness)


def fresnelSchlick(cosTheta, F0):
    return F0 + (1.0 - F0) * torch.pow(1.0 - cosTheta, 5)[:, :, None]


def directional_lighting(diffuseLight, specularLight, normals, light_intensity=0.5, light_color=(1, 1, 1),
                         light_direction=(0, 1, 0), positions=None, eye=None, with_specular=False,
                         metallic_textures=None, roughness_textures=None):
    """directional_lighting.py:54-145 for 3-D normals ([B, n, 3])."""
    light_color = _t(light_color, normals)
    light_direction = F.normalize(_t(light_direction, normals), dim=0, eps=1e-12)
    if light_color.dim() == 1:
        light_color = light_color[None, :]
    if light_direction.dim() == 1:
        light_direction = light_direction[None, :]
    cosine = F.relu(torch.sum(normals * light_direction, dim=2))

    if with_specular and metallic_textures is not None and roughness_textures is not None:
        if metallic_textures.dim() == 4:
            total = metallic_textures.shape[2] * 1.0
            metallic_textures = torch.sum(metallic_textures, dim=2) / total
            roughness_textures = torch.sum(roughness_textures, dim=2) / total
        elif metallic_textures.dim() == 6:
            total = metallic_textures.shape[2] * metallic_textures.shape[3] * metallic_textures.shape[4] * 1.0
            metallic_textures = metallic_textures.sum(dim=(2, 3, 4)) / total
            roughness_textures = roughness_textures.sum(dim=(2, 3, 4)) / total

    if with_specular and eye is not None and positions is not None and metallic_textures is not None \
            and roughness_textures is not None:
        eye = _t(eye, normals)
        if eye.dim() == 1:
            eye = eye[None, :]
        if eye.dim() == 2:
            eye = eye[:, None, :]
        N = normals
        V = F.normalize(eye - positions, dim=2, eps=1e-12)
        L = light_direction
        H = F.normalize(V + L, dim=2, eps=1e-12)
        metallic = metallic_textures
        roughness = roughness_textures
        F0 = _t((0.4, 0.4, 0.4), normals)[None, None, :] * (1 - metallic) + _t((1.0, 1.0, 1.0), normals)[None, None, :] * metallic
        radiance = light_intensity * (light_color[:, None, :] * cosine[:, :, None])
        NDF = GGX(N, H, roughness)
        G = GeometrySmith(N, V, L, roughness)
        Fr = fresnelSchlick(F.relu(torch.sum(H * V, dim=2)), F0)
        KD = (1.0 - Fr) * (1.0 - metallic)
        diffuseLight = diffuseLight + KD * radiance
        numerator = NDF * G * Fr
        denominator = (4.0 * F.relu(torch.sum(N * V, dim=2)) * F.relu(torch.sum(N * L, dim=2)))[:, :, None]
        specular = numerator / torch.clamp(denominator, min=0.01)
        specularLight = specularLight + specular * radiance
    else:
        diffuseLight = diffuseLight + light_intensity * (light_color[:, None, :] * cosine[:, :, None])
    return [diffuseLight, specularLight]


def _f3(x):
    """3 host floats as a ctypes array (light colours / direction are Python constants in the reference's API)."""
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().tolist()
    x = [float(v) for v in x]
    if len(x) != 3:
        raise ValueError("expected 3 components, got %r" % (x,))
    return (C.c_float * 3)(*x)


class _FusedSurfaceLighting(torch.autograd.Function):
    """clamp(textures * diffuse + specular, 0, 1) with diffuse / specular from the face normals: b200r_surface_lighting_*."""

    @staticmethod
    def forward(ctx, vertices, textures, faces, metallic, roughness, eye, params):
        dev = vertices.device
        v = vertices.contiguous()
        tx = textures.contiguous()
        B, nf = tx.shape[0], tx.shape[1]
        T = tx[0, 0].numel() // 3
        Tm = 0 if metallic is None else metallic[0, 0].numel()
        out = torch.empty_like(tx)
        amb_i, amb_c, dir_i, dir_c, direction, with_spec = params
        args = (B, v.shape[0], faces.shape[0], 0 if eye is None else eye.shape[0], v.shape[1], nf, T, Tm,
                float(amb_i), _f3(amb_c), float(dir_i), _f3(dir_c), _f3(direction), int(bool(with_spec)))
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            p = lambda t: C.c_void_p(0 if t is None else t.data_ptr())   # noqa: E731
            _lib.check(_lib.lib().b200r_surface_lighting_forward(p(v), p(faces), p(tx), p(metallic), p(roughness), p(eye), p(out), *args, st),
                       "b200r_surface_lighting_forward")
        ctx.save_for_backward(v, tx, faces, metallic, roughness, eye)
        ctx.args = args
        return out

    @staticmethod
    def backward(ctx, grad_out):
        v, tx, faces, metallic, roughness, eye = ctx.saved_tensors
        dev = v.device
        g = grad_out.contiguous()
        gt = torch.empty_like(tx)
        gv = torch.empty_like(v) if ctx.needs_input_grad[0] else None
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            p = lambda t: C.c_void_p(0 if t is None else t.data_ptr())   # noqa: E731
            _lib.check(_lib.lib().b200r_surface_lighting_backward(p(v), p(faces), p(tx), p(metallic), p(roughness), p(eye), p(g), p(gt), p(gv),
                                                                  *ctx.args, st), "b200r_surface_lighting_backward")
        return gv, (gt if ctx.needs_input_grad[1] else None), None, None, None, None, None


_SSS_BASIS = [0, 25, 100, 400]                                          # lighting.py:115
_SSS_WEIGHTS = [[0.7, 0.2, 0.1], [0.1, 0.2, 0.7], [0.1, 0.2, 0.7]]      # lighting.py:126-129, [channel][basis]
_SSS_TAP_NUM = 7


def _sss_taps(v):
    """gaussian_blur.py:4-10 in double: the 7 taps and GaussWidth = sqrt(v) of one variance.  Both are rounded to float
    on the way to the kernel, as in the reference (float32 tap tensor; jt.float32(GaussWidth) formatted into the launch)."""
    w = math.sqrt(v)
    return [w * (math.exp(-(-w * ((_SSS_TAP_NUM - 1) / 2 - k)) ** 2 / (2 * v)) / math.sqrt(2 * math.pi * v))
            for k in range(_SSS_TAP_NUM)], w


def _sss_host_arrays():
    """Taps (3 x 7), Gauss widths (3) and weights (3 x 3) of the blur chain as host float arrays."""
    taps, widths = [], []
    for i in range(len(_SSS_BASIS) - 1):
        t, w = _sss_taps(_SSS_BASIS[i + 1] - _SSS_BASIS[i])
        taps += t
        widths.append(w)
    return ((C.c_float * len(taps))(*taps), (C.c_float * 3)(*widths),
            (C.c_float * 9)(*[x for row in _SSS_WEIGHTS for x in row]))


def SSS(diffuseLight, specular, mesh, image_size=2048):
    """Texture-space subsurface scattering (lighting.py:86-156) of a softras mesh with 4-D textures and face_texcoords.

    diffuseLight, specular: the per-face surface lighting terms [1, nf, 1, 3].  The mesh's world-space geometry, the
    irradiance sqrt(textures * diffuseLight) and the specular term are rasterized into UV space at image_size^2; the
    stretch-modulated Gaussian blur chain (b200r_sss_blur_chain) turns them into the scattered colour map, which is
    baked back into textures [1, nf, texture_res^2, 3] (not clamped; Lighting clamps).

    The result is DETACHED: the reference's blur and bake ops have no gradient, so neither have these textures.
    Batch 1 only, like the reference (it squeezes the batch axis)."""
    from .io import bake_textures_for_softras
    from .softras import SoftRasterizeFunction
    if mesh.face_texcoords is None:
        raise ValueError("SSS needs mesh.face_texcoords: load the mesh with Mesh.from_obj(..., load_texture=True, dr_type='softras')")
    textures = mesh.textures
    if textures.dim() != 4 or textures.shape[0] != 1:
        raise ValueError("SSS supports batch size 1 with textures [1, nf, R*R, 3], got %s" % (tuple(textures.shape),))
    dev = textures.device
    S = int(image_size)
    with torch.no_grad():
        irradiance = torch.sqrt(textures * diffuseLight)
        rasterize = SoftRasterizeFunction(image_size=S, background_color=[0, 0, 0], near=1, far=100,
                                          fill_back=True, eps=1e-5, sigma_val=1e-5, dist_func='barycentric', dist_eps=1e-5,
                                          gamma_val=1e-4, aggr_func_rgb='hard', aggr_func_alpha='prod', texture_type='surface')
        # (face_vertices + 1) / 2 * 255 has T = 3 texels, so R = int(sqrt(3)) = 1 and every face samples texel 0, its
        # vertex 0: the same map comes from that one texel
        world = ((mesh.face_vertices + 1) / 2 * 255.)[:, :, :1].contiguous()
        coords = (mesh.face_texcoords.to(device=dev, dtype=torch.float32) - 0.5) * 2
        coords = torch.cat([coords, torch.full(coords.shape[:3] + (1,), 1.5, device=dev)], dim=3).contiguous()
        final = sss_blur_chain(*[rasterize(coords, t.contiguous())[0] for t in (world, irradiance, specular)])
        nf, T = textures.shape[1], mesh.texture_res ** 2
        out = bake_textures_for_softras(final, mesh.face_texcoords[0], torch.ones((nf, T, 3), device=dev),
                                        torch.ones((nf,), dtype=torch.int32, device=dev), device=dev)
    return out[None]


def sss_blur_chain(worldcoord_map, irradiance_map, specular_map):
    """The image-space part of SSS (b200r_sss_blur_chain): three texture-space maps [4 (or 3), S, S] float32 on one CUDA
    device -> the scattered colour map [S, S, 3], flipped vertically for the bake."""
    maps = [m.contiguous() for m in (worldcoord_map, irradiance_map, specular_map)]
    dev = maps[0].device
    S = maps[0].shape[-1]
    for m in maps:
        if not m.is_cuda or m.device != dev or m.dtype != torch.float32 or m.dim() != 3 or m.shape[0] < 3 or tuple(m.shape[1:]) != (S, S):
            raise ValueError("sss_blur_chain: three float32 CUDA maps [>=3, S, S] on one device")
    L = _lib.lib()
    final = torch.empty((S, S, 3), dtype=torch.float32, device=dev)
    ws_bytes = L.b200r_sss_workspace_bytes(S)
    workspace = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    taps, widths, weights = _sss_host_arrays()
    p = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731
    with torch.cuda.device(dev):
        _lib.check(L.b200r_sss_blur_chain(p(maps[0]), p(maps[1]), p(maps[2]), p(final), p(workspace), ws_bytes, S,
                                          taps, widths, weights, C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
                   "b200r_sss_blur_chain")
    return final


def sss_blur(image, modulate, variance, dim):
    """One stretch-modulated 7-tap blur of an [S, S] float32 CUDA map (_blur_for_SSS, gaussian_blur.py:34-165): dim 1 along
    x, dim 0 along y, Gauss width sqrt(variance) scaled per pixel by modulate.  The building block of SSS's chain."""
    if not (image.is_cuda and modulate.is_cuda and image.device == modulate.device):
        raise _lib.B200RasterError("sss_blur runs on the GPU (b200r_sss_blur); there is no CPU fallback")
    if image.dtype != torch.float32 or modulate.dtype != torch.float32:
        raise TypeError("sss_blur: image and modulate must be float32")
    if image.dim() != 2 or image.shape[0] != image.shape[1] or modulate.shape != image.shape:
        raise ValueError("sss_blur: image and modulate must be the same square [S, S] map")
    taps, w = _sss_taps(float(variance))
    img, mod = image.contiguous(), modulate.contiguous()
    out = torch.empty_like(img)
    dev = img.device
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().b200r_sss_blur(C.c_void_p(img.data_ptr()), C.c_void_p(mod.data_ptr()), C.c_void_p(out.data_ptr()),
                                             img.shape[0], (C.c_float * _SSS_TAP_NUM)(*taps), w, int(dim),
                                             C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "b200r_sss_blur")
    return out


def _normalized_direction(d):
    """F.normalize(light_direction, dim=0, eps=1e-12) on the host, in float32 like the mirror."""
    t = torch.tensor([float(x) for x in (d.detach().cpu().tolist() if isinstance(d, torch.Tensor) else d)], dtype=torch.float32)
    return F.normalize(t, dim=0, eps=1e-12).tolist()


class AmbientLighting(nn.Module):
    def __init__(self, light_intensity=0.5, light_color=(1, 1, 1)):
        super(AmbientLighting, self).__init__()
        self.light_intensity = light_intensity
        self.light_color = light_color

    def forward(self, light):
        return ambient_lighting(light, self.light_intensity, self.light_color)

    execute = forward


class DirectionalLighting(nn.Module):
    def __init__(self, light_intensity=0.5, light_color=(1, 1, 1), light_direction=(0, 1, 0)):
        super(DirectionalLighting, self).__init__()
        self.light_intensity = light_intensity
        self.light_color = light_color
        self.light_direction = light_direction

    def forward(self, diffuseLight, specularLight, normals, positions=None, eye=None, with_specular=False,
                metallic_textures=None, roughness_textures=None):
        return directional_lighting(diffuseLight, specularLight, normals, self.light_intensity, self.light_color,
                                    self.light_direction, positions, eye, with_specular, metallic_textures,
                                    roughness_textures)

    execute = forward


class Lighting(nn.Module):
    """lighting.py:159-223."""

    def __init__(self, light_mode='surface',
                 intensity_ambient=0.5, color_ambient=[1, 1, 1],
                 intensity_directionals=0.5, color_directionals=[1, 1, 1],
                 directions=[0, 1, 0], Gbuffer='None', transform=None):
        super(Lighting, self).__init__()
        if light_mode not in ['surface', 'vertex']:
            raise ValueError('Lighting mode only support surface and vertex')
        if Gbuffer not in ('None', None, 'albedo'):
            raise NotImplementedError("Gbuffer=%r (render2 debug outputs) is outside this repo's scope" % (Gbuffer,))
        self.Gbuffer = Gbuffer
        self.transform = transform
        self.light_mode = light_mode
        self.ambient = AmbientLighting(intensity_ambient, color_ambient)
        self.directionals = nn.ModuleList([DirectionalLighting(intensity_directionals, color_directionals, directions)])

    fused = True   # CUDA float32 surface-mode inputs take the one-launch kernel (b200r_surface_lighting_forward)

    def _fusable(self, mesh, eyes):
        tx, v = mesh.textures, mesh.vertices
        if not (self.fused and len(self.directionals) == 1 and tx.is_cuda and v.is_cuda and tx.device == v.device):
            return False
        if tx.dtype != torch.float32 or v.dtype != torch.float32 or tx.dim() not in (4, 6) or tx.shape[-1] != 3:
            return False
        if mesh.faces.device != v.device or mesh.faces.dim() != 3 or mesh.faces.shape[1] != tx.shape[1]:
            return False
        d = self.directionals[0]
        for c in (self.ambient.light_color, d.light_color, d.light_direction):
            n = c.numel() if isinstance(c, torch.Tensor) else len(c)
            if n != 3:   # per-batch light colours / directions: op-by-op path
                return False
        for t in (mesh.metallic_textures, mesh.roughness_textures):
            if t is not None and (t.requires_grad or t.device != v.device or t.dtype != torch.float32
                                  or t.shape[:2] != tx.shape[:2] or t.shape[-1] != 1):
                return False
        if isinstance(eyes, torch.Tensor) and eyes.requires_grad:
            return False
        return True

    def _fused_surface(self, mesh, eyes):
        v = mesh.vertices
        d = self.directionals[0]
        eye = None
        spec = bool(mesh.with_specular) and eyes is not None and mesh.metallic_textures is not None and mesh.roughness_textures is not None
        if spec:
            eye = _t(eyes, v).reshape(-1, 3).contiguous()
            if eye.shape[0] not in (1, mesh.textures.shape[0]):
                return None
        faces = mesh.faces if mesh.faces.dtype == torch.int32 else mesh.faces.int()
        params = (self.ambient.light_intensity, self.ambient.light_color, d.light_intensity, d.light_color,
                  _normalized_direction(d.light_direction), spec)
        return _FusedSurfaceLighting.apply(v, mesh.textures, faces.contiguous(),
                                           mesh.metallic_textures.contiguous() if spec else None,
                                           mesh.roughness_textures.contiguous() if spec else None, eye, params)

    def forward(self, mesh, eyes=None):
        if self.Gbuffer == "albedo":
            return mesh
        sss = self.light_mode == 'surface' and mesh.textures.dim() == 4 and mesh.with_SSS
        if self.light_mode == 'surface' and not sss and self._fusable(mesh, eyes):
            lit = self._fused_surface(mesh, eyes)
            if lit is not None:
                mesh.textures = lit
                return mesh
        if self.light_mode == 'surface':
            diffuseLight = torch.zeros(mesh.faces.shape, dtype=torch.float32, device=mesh.vertices.device)
            specularLight = torch.zeros_like(diffuseLight)
            diffuseLight = self.ambient(diffuseLight)
            for directional in self.directionals:
                diffuseLight, specularLight = directional(
                    diffuseLight, specularLight, mesh.surface_normals, torch.sum(mesh.face_vertices, dim=2) / 3.0, eyes,
                    mesh.with_specular, mesh.metallic_textures, mesh.roughness_textures)
            diffuseLight = diffuseLight[:, :, None, :]
            specularLight = specularLight[:, :, None, :]
            if sss:   # the fused kernel returns only diffuse and specular combined: SSS needs them apart
                mesh.textures = torch.clamp(SSS(diffuseLight, specularLight, mesh), 0.0, 1.0)
            elif mesh.textures.dim() == 4:
                mesh.textures = torch.clamp(mesh.textures * diffuseLight + torch.ones_like(mesh.textures) * specularLight, 0.0, 1.0)
            elif mesh.textures.dim() == 6:
                mesh.textures = torch.clamp(mesh.textures * diffuseLight[:, :, :, None, None, :] +
                                            torch.ones_like(mesh.textures) * specularLight[:, :, :, None, None, :], 0.0, 1.0)
        elif self.light_mode == 'vertex':
            diffuseLight = torch.zeros(mesh.vertices.shape, dtype=torch.float32, device=mesh.vertices.device)
            specularLight = torch.zeros_like(diffuseLight)
            diffuseLight = self.ambient(diffuseLight)
            for directional in self.directionals:
                diffuseLight, specularLight = directional(
                    diffuseLight, specularLight, mesh.vertex_normals, mesh.vertices, eyes,
                    mesh.with_specular, mesh.metallic_textures, mesh.roughness_textures)
            # The reference only applies vertex lighting to 4-D / 6-D textures (lighting.py:214-220);
            # the documented vertex texture shape [B, nv, 3] therefore passes through unlit.
            if mesh.textures.dim() == 4:
                mesh.textures = torch.clamp(mesh.textures * diffuseLight[:, :, None, :] +
                                            torch.ones_like(mesh.textures) * specularLight[:, :, None, :], 0.0, 1.0)
            elif mesh.textures.dim() == 6:
                mesh.textures = torch.clamp(mesh.textures * diffuseLight[:, :, None, None, None, :] +
                                            torch.ones_like(mesh.textures) * specularLight[:, :, None, None, None, :], 0.0, 1.0)
        return mesh

    execute = forward
