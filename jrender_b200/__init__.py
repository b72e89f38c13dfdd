"""jrender_b200 -- B200-native differentiable mesh rasterizer behind Jittor/jrender's API.

Hot path: hand-written sm_100a CUDA kernels in csrc/, exposed through the C ABI in
include/b200raster.h (libb200raster.so) and bound with ctypes; PyTorch is plumbing only
(device memory, streams, autograd glue) plus the O(nf) host-side mirror of the reference's
camera / lighting / mesh / loss classes so that reference scripts port by changing the import.
"""
from ._lib import B200RasterError  # noqa: F401
from .softras import SoftRasterizeFunction, SoftRasterizer, soft_rasterize  # noqa: F401
from .mesh import Mesh, face_vertices, join_meshes_as_scene  # noqa: F401
from .transform import (Transform, LookAt, Look, Projection, look_at, look, perspective, orthogonal,  # noqa: F401
                        projection, get_points_from_angles)
from .lighting import Lighting, AmbientLighting, DirectionalLighting, SSS  # noqa: F401
from .renderer import Renderer  # noqa: F401
from .preraster import project_faces  # noqa: F401
from .loss import neg_iou_loss, LaplacianLoss, FlattenLoss  # noqa: F401
from .io import load_obj, save_obj  # noqa: F401
