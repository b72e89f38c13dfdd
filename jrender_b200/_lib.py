"""ctypes binding of libb200raster.so (C ABI declared in include/b200raster.h).

The product path has no CPU fallback: if the library is missing or a call fails, an
exception is raised.  The library is never built implicitly at import time on a GPU box --
`__graft_entry__.build()` / `python -m jrender_b200.build` produce it in-tree.
"""
import ctypes as C
import os

from . import build as _build

_lib = None


class B200RasterError(RuntimeError):
    pass


_F = C.c_float
_I = C.c_int
_P = C.c_void_p

_SOFTRAS_SCALARS = [_I, _I, _I, _I, _I, _F, _F, _F, _F, _F, _F, _I, _I, _I, _I, _I, _P]


def lib():
    """Load (once) and return the C ABI library; raises B200RasterError when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("B200R_LIB") or _build.LIB  # B200R_LIB: development A/B builds (build.py --variant)
    if not os.path.exists(path):
        raise B200RasterError(
            "libb200raster.so not built (%s). Run `python -m jrender_b200.build` "
            "(needs nvcc); there is no CPU fallback." % path)
    L = C.CDLL(path)
    L.b200r_version.restype = C.c_char_p
    L.b200r_last_error.restype = C.c_char_p
    L.b200r_launch_count.restype = C.c_ulonglong
    L.b200r_softras_workspace_bytes.restype = C.c_size_t
    L.b200r_softras_workspace_bytes.argtypes = [_I, _I, _I]
    L.b200r_softras_state_bytes.restype = C.c_size_t
    L.b200r_softras_state_bytes.argtypes = [_I, _I]
    L.b200r_softras_forward.restype = _I
    L.b200r_softras_forward.argtypes = [_P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P, C.c_size_t] + _SOFTRAS_SCALARS
    L.b200r_softras_backward.restype = _I
    L.b200r_softras_backward.argtypes = [_P, _P, _P, _P, _P, _P, C.c_size_t, _P, _P, _P] + _SOFTRAS_SCALARS
    L.b200r_softras_forward_aa.restype = _I
    L.b200r_softras_forward_aa.argtypes = [_P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P, C.c_size_t] + _SOFTRAS_SCALARS
    L.b200r_softras_backward_aa.restype = _I
    L.b200r_softras_backward_aa.argtypes = [_P, _P, _P, _P, _P, _P, C.c_size_t, _P, _P, _P] + _SOFTRAS_SCALARS
    L.b200r_profile_enable.restype = None
    L.b200r_profile_enable.argtypes = [_I]
    L.b200r_profile_reset.restype = None
    L.b200r_profile_reset.argtypes = []
    L.b200r_profile_read.restype = _I
    L.b200r_profile_read.argtypes = [_I, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    L.b200r_debug_exact_math.restype = _I
    L.b200r_debug_exact_math.argtypes = [_P, _P, _I, _P, _P]
    L.b200r_nmr_workspace_bytes.restype = C.c_size_t
    L.b200r_nmr_workspace_bytes.argtypes = [_I, _I, _I]
    L.b200r_nmr_forward.restype = _I
    L.b200r_nmr_forward.argtypes = [_P] * 11 + [C.c_size_t, _I, _I, _I, _I, _F, _F, _F, _P, _I, _I, _I, _P]
    L.b200r_nmr_backward.restype = _I
    L.b200r_nmr_backward.argtypes = [_P] * 15 + [C.c_size_t, _I, _I, _I, _I, _F, _I, _I, _I, _P]
    L.b200r_nmr_backward_scratch_bytes.restype = C.c_size_t
    L.b200r_nmr_backward_scratch_bytes.argtypes = [_I, _I]
    L.b200r_project_faces_forward.restype = _I
    L.b200r_project_faces_forward.argtypes = [_P, _P, _P, _P, _P, _P, _F] + [_I] * 8 + [_P]
    L.b200r_project_faces_backward.restype = _I
    L.b200r_project_faces_backward.argtypes = [_P, _P, _P, _P, _P, _P, _P, _F] + [_I] * 8 + [_P]
    L.b200r_flatten_loss.restype = _I
    L.b200r_flatten_loss.argtypes = [_P] * 7 + [_I, _I, _I, _F, _P]
    L.b200r_laplacian_loss.restype = _I
    L.b200r_laplacian_loss.argtypes = [_P] * 6 + [_I, _I, _I, _P]
    L.b200r_surface_lighting_forward.restype = _I
    L.b200r_surface_lighting_forward.argtypes = [_P] * 7 + [_I] * 8 + [_F, _P, _F, _P, _P, _I, _P]
    L.b200r_surface_lighting_backward.restype = _I
    L.b200r_surface_lighting_backward.argtypes = [_P] * 9 + [_I] * 8 + [_F, _P, _F, _P, _P, _I, _P]
    L.b200r_bake_textures_softras.restype = _I
    L.b200r_bake_textures_softras.argtypes = [_P, _P, _P, _P, _I, _I, _I, _I, _P]
    L.b200r_bake_textures_n3mr.restype = _I
    L.b200r_bake_textures_n3mr.argtypes = [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]
    L.b200r_sss_workspace_bytes.restype = C.c_size_t
    L.b200r_sss_workspace_bytes.argtypes = [_I]
    L.b200r_sss_blur_chain.restype = _I
    L.b200r_sss_blur_chain.argtypes = [_P] * 5 + [C.c_size_t, _I, _P, _P, _P, _P]
    L.b200r_sss_blur.restype = _I
    L.b200r_sss_blur.argtypes = [_P, _P, _P, _I, _P, _F, _I, _P]
    L.b200r_set_option.restype = _I
    L.b200r_set_option.argtypes = [C.c_char_p, _I]
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        raise B200RasterError("%s failed (rc=%d): %s" % (what, rc, lib().b200r_last_error().decode()))


def set_option(name, value):
    check(lib().b200r_set_option(name.encode(), int(value)), "b200r_set_option(%s)" % name)
