"""Mesh container (host-side mirror of jrender/structures/mesh.py:8-342 in PyTorch).

Holds vertices [B,nv,3], faces [B,nf,3] and textures; lazily gathers face_vertices
[B,nf,3,3] / face_textures -- the two tensors the rasterizer consumes.  Only the attributes the
rasterizer path (Renderer -> Lighting -> Transform -> rasterizer) reads are mirrored, plus the UV triangles
(face_texcoords) that texture-space subsurface scattering (with_SSS) rasterizes; normal maps / TBN / voxelize are
outside the hot-path scope (SURVEY.md section 8).
"""
import numpy as np
import torch
import torch.nn.functional as F


def face_vertices(vertices, faces):
    """structures/utils/faces_vertices.py:4-19: [B,nv,C] gathered by [B,nf,3] -> [B,nf,3,C]."""
    assert vertices.dim() == 3
    assert faces.dim() == 3
    assert vertices.shape[0] == faces.shape[0]
    assert faces.shape[2] == 3
    bs, nv = vertices.shape[:2]
    faces = faces.long() + (torch.arange(bs, device=vertices.device) * nv)[:, None, None]
    vertices = vertices.reshape((bs * nv, vertices.shape[2]))
    # index_select: its backward is an index_add kernel (the scatter of grad_face_vertices to
    # grad_vertices); `vertices[faces]` would back-propagate through a sort-based index_put that
    # synchronises the host and cannot be captured in a CUDA graph
    return torch.index_select(vertices, 0, faces.reshape(-1)).view(bs, faces.shape[1], 3, vertices.shape[1])


class Mesh(object):
    def __init__(self, vertices, faces, textures=None, texture_res=1, texture_type='surface', dr_type='softras',
                 metallic_textures=None, roughness_textures=None, normal_textures=None, TBN=None, with_SSS=False,
                 face_texcoords=None):
        if isinstance(vertices, np.ndarray):
            vertices = torch.from_numpy(vertices).float()
        if isinstance(faces, np.ndarray):
            faces = torch.from_numpy(faces).int()
        self._vertices = vertices
        self._faces = faces
        self._projector = None
        if self._vertices.dim() == 2:
            self._vertices = self._vertices[None]
        if self._faces.dim() == 2:
            self._faces = self._faces[None]
        if self._faces.device != self._vertices.device:
            self._faces = self._faces.to(self._vertices.device)
        self.texture_type = texture_type
        self.batch_size = self._vertices.shape[0]
        self.num_vertices = self._vertices.shape[1]
        self.num_faces = self._faces.shape[1]
        self._face_vertices = None
        self._face_vertices_update = True
        self._surface_normals = None
        self._surface_normals_update = True
        self._vertex_normals = None
        self._vertex_normals_update = True
        self._with_specular = True   # mesh.py:74: lighting takes the Cook-Torrance branch by default
        self._with_SSS = with_SSS
        if isinstance(face_texcoords, np.ndarray):
            face_texcoords = torch.from_numpy(face_texcoords).float()
        if face_texcoords is not None and face_texcoords.dim() == 3:   # [nf, 3, 2] -> [1, nf, 3, 2] (mesh.py:77-79)
            face_texcoords = face_texcoords[None]
        self._face_texcoords = face_texcoords
        self._fill_back = False
        self.dr_type = dr_type
        self.normal_textures = None
        dev = self._vertices.device

        if textures is None:
            if texture_type == 'surface':
                if self.dr_type == 'softras':
                    self._textures = torch.ones((self.batch_size, self.num_faces, texture_res ** 2, 3), device=dev)
                elif self.dr_type == 'n3mr':
                    self._textures = torch.ones((self.batch_size, self.num_faces, texture_res, texture_res, texture_res, 3), device=dev)
                self.texture_res = texture_res
            elif texture_type == 'vertex':
                self._textures = torch.ones((self.batch_size, self.num_vertices, 3), device=dev)
                self.texture_res = 1
        else:
            if isinstance(textures, np.ndarray):
                textures = torch.from_numpy(textures).float()
            if textures.dim() == 3 and texture_type == 'surface':
                textures = textures[None]
            if textures.dim() == 2 and texture_type == 'vertex':
                textures = textures[None]
            if textures.dim() == 5:
                textures = textures[None]
            self._textures = textures.to(dev)
            if self.dr_type == 'softras':
                if self.texture_type == 'surface':
                    self.texture_res = int(np.sqrt(self._textures.shape[2]))
                elif self.texture_type == 'vertex':
                    self.texture_res = 1
            elif self.dr_type == 'n3mr':
                self.texture_res = self._textures.shape[2]
        # metallic 0 / roughness 1 defaults (mesh.py:83-97)
        if texture_type == 'surface':
            tail = (texture_res ** 2, 1) if self.dr_type == 'softras' else (texture_res, texture_res, texture_res, 1)
            shape = (self.batch_size, self.num_faces) + tail
        else:
            shape = (self.batch_size, self.num_vertices, 1)
        self.metallic_textures = torch.zeros(shape, device=dev) if metallic_textures is None else metallic_textures
        self.roughness_textures = torch.ones(shape, device=dev) if roughness_textures is None else roughness_textures
        self._origin_vertices = self._vertices
        self._origin_faces = self._faces
        self._origin_textures = self._textures

    @property
    def with_specular(self):
        return self._with_specular

    @with_specular.setter
    def with_specular(self, v):
        self._with_specular = v

    @property
    def with_SSS(self):
        return self._with_SSS

    @property
    def faces(self):
        return self._faces

    @faces.setter
    def faces(self, faces):
        self._faces = faces
        self.num_faces = self._faces.shape[1]
        self._face_vertices_update = True
        self._surface_normals_update = True
        self._vertex_normals_update = True

    @property
    def vertices(self):
        if self._vertices is None and self._projector is not None:
            self._vertices = self._projector.vertices()   # lazily, op by op (only if somebody asks)
        return self._vertices

    def attach_projector(self, projector):
        """Transform's fused path: `projector.face_vertices(faces)` yields the camera-space + projected
        face_vertices in one launch from the world-space vertices (jrender_b200/preraster.py);
        `projector.vertices()` is the op-by-op equivalent of `mesh.vertices = transform(mesh.vertices)`."""
        self._projector = projector
        self._vertices = None
        self._face_vertices_update = True
        self._surface_normals_update = True
        self._vertex_normals_update = True

    @vertices.setter
    def vertices(self, vertices):
        self._projector = None
        self._vertices = vertices
        self.num_vertices = self._vertices.shape[1]
        self._face_vertices_update = True
        self._surface_normals_update = True
        self._vertex_normals_update = True

    @property
    def textures(self):
        return self._textures

    @textures.setter
    def textures(self, textures):
        self._textures = textures

    @property
    def face_vertices(self):
        if self._face_vertices_update:
            if self._projector is not None:
                self._face_vertices = self._projector.face_vertices(self.faces)
            else:
                self._face_vertices = face_vertices(self.vertices, self.faces)
            self._face_vertices_update = False
        return self._face_vertices

    @property
    def surface_normals(self):
        """mesh.py:213-229 (float64 cross product, then normalised, back to float32)."""
        if self._surface_normals_update:
            v10 = (self.face_vertices[:, :, 0] - self.face_vertices[:, :, 1]).double()
            v12 = (self.face_vertices[:, :, 2] - self.face_vertices[:, :, 1]).double()
            self._surface_normals = F.normalize(torch.cross(v12, v10, dim=2), p=2, dim=2, eps=1e-12).float()
            self._surface_normals_update = False
        return self._surface_normals

    @property
    def vertex_normals(self):
        """mesh.py:231-248: area-weighted face normals scattered to vertices."""
        if self._vertex_normals_update:
            bs, nv = self.vertices.shape[:2]
            faces = (self.faces.long() + (torch.arange(bs, device=self.vertices.device) * nv)[:, None, None]).view(-1, 3)
            vf = torch.index_select(self.vertices.reshape((bs * nv, 3)), 0, faces.reshape(-1)).view(-1, 3, 3)
            normals = torch.zeros((bs * nv, 3), dtype=self.vertices.dtype, device=self.vertices.device)
            normals.index_add_(0, faces[:, 1], torch.cross(vf[:, 2] - vf[:, 1], vf[:, 0] - vf[:, 1], dim=1))
            normals.index_add_(0, faces[:, 2], torch.cross(vf[:, 0] - vf[:, 2], vf[:, 1] - vf[:, 2], dim=1))
            normals.index_add_(0, faces[:, 0], torch.cross(vf[:, 1] - vf[:, 0], vf[:, 2] - vf[:, 0], dim=1))
            self._vertex_normals = F.normalize(normals, p=2, eps=1e-6, dim=1).reshape((bs, nv, 3))
            self._vertex_normals_update = False
        return self._vertex_normals

    @property
    def face_textures(self):
        if self.texture_type in ['surface']:
            return self.textures
        elif self.texture_type in ['vertex']:
            return face_vertices(self.textures, self.faces)
        else:
            raise ValueError('texture type not applicable')

    def fill_back_(self):
        if not self._fill_back:
            self.faces = torch.cat((self.faces, self.faces[:, :, [2, 1, 0]]), dim=1)
            self.textures = torch.cat((self.textures, self.textures), dim=1)
            self._fill_back = True

    def reset_(self):
        self.vertices = self._origin_vertices
        self.faces = self._origin_faces
        self.textures = self._origin_textures
        self._fill_back = False

    @property
    def face_texcoords(self):
        return self._face_texcoords

    @classmethod
    def from_obj(cls, filename_obj, normalization=False, load_texture=False, dr_type='softras', texture_res=1,
                 texture_type='surface', texture_wrapping='REPEAT', use_bilinear=True, with_SSS=False):
        from .io import load_obj, _parse_texture_faces
        face_texcoords = None
        if load_texture:
            vertices, faces, textures = load_obj(filename_obj, normalization=normalization, texture_res=texture_res,
                                                 load_texture=True, dr_type=dr_type, texture_type=texture_type,
                                                 texture_wrapping=texture_wrapping, use_bilinear=use_bilinear)
            if dr_type == 'softras' and texture_type == 'surface':   # _load_obj_for_softras.py returns the UVs too
                face_texcoords = torch.from_numpy(_parse_texture_faces(filename_obj)[0]).to(vertices.device)
        else:
            vertices, faces = load_obj(filename_obj, normalization=normalization, load_texture=False, dr_type=dr_type)
            textures = None
        return cls(vertices, faces, textures, texture_res, texture_type, dr_type=dr_type, with_SSS=with_SSS,
                   face_texcoords=face_texcoords)

    def save_obj(self, filename_obj, save_texture=False, texture_res_out=16):
        """structures/mesh.py:330-338.  Geometry only: the texture-atlas export (io/save_obj.py:9-29, a separate CUDA
        kernel of the reference) is outside this repo's scope."""
        if self.batch_size != 1:
            raise ValueError('Could not save when batch size >= 1')
        if save_texture:
            raise NotImplementedError("save_obj(save_texture=True): texture-atlas export is not part of the rasterizer hot path")
        from .io import save_obj
        save_obj(filename_obj, self.vertices[0], self.faces[0])

    def to(self, device):
        self._vertices = self.vertices.to(device)
        self._projector = None
        self._faces = self._faces.to(device)
        self._textures = self._textures.to(device)
        self.metallic_textures = self.metallic_textures.to(device)
        self.roughness_textures = self.roughness_textures.to(device)
        if self._face_texcoords is not None:
            self._face_texcoords = self._face_texcoords.to(device)
        self._origin_vertices, self._origin_faces, self._origin_textures = self._vertices, self._faces, self._textures
        self._face_vertices_update = self._surface_normals_update = self._vertex_normals_update = True
        return self

    def cuda(self):
        return self.to(torch.device("cuda"))


def join_meshes_as_scene(meshes, include_texture=True):
    """structures/mesh.py:345-374: one mesh whose vertices / faces (/ textures) are the inputs' concatenated along the
    vertex / face axis, face indices shifted by the running vertex count."""
    verts = [m.vertices for m in meshes]
    faces, shift = [], 0
    for m in meshes:
        faces.append(m.faces + shift)
        shift += m.vertices.shape[1]
    vert, face = torch.cat(verts, dim=1), torch.cat(faces, dim=1)
    if not include_texture:
        return Mesh(vert, face)
    # a Mesh built without textures carries all-ones defaults here (the reference keeps None): treat "every mesh has
    # textures" as the textured case, exactly like the reference when all inputs were given textures
    first = meshes[0]
    if not all(m.dr_type == first.dr_type and m.texture_type == first.texture_type for m in meshes):
        raise ValueError("Inconsistent textures in join_meshes_as_scene (dr_type or texture_type).")
    tex = torch.cat([m.textures for m in meshes], dim=1)
    return Mesh(vertices=vert, faces=face, textures=tex, texture_type=first.texture_type, dr_type=first.dr_type)
