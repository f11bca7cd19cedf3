"""ctypes description of the C-ABI declared in ``include/deodr_b200.h`` and loader of ``libdeodr_b200.so``.

The shared library holds the hand-written sm_100a kernels; there is no other implementation.  ``load()`` raises if
the library is missing, and every entry point of the library fails with DEODR_B200_ECUDA when no CUDA device is
usable - nothing in this package falls back to a CPU path.
"""

from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DEODR_B200_LIB selects an alternative build of the same library (A/B experiments on one GPU box)
LIB_PATH = os.environ.get("DEODR_B200_LIB") or os.path.join(_HERE, "libdeodr_b200.so")

OK, EINVAL, EUNSUPPORTED, ECUDA, ENOMEM, EREPLAN = 0, 1, 2, 3, 4, 5
ANTIALIASE_ERROR, ERROR_ADJOINT_COMPLETE = 1, 2  # flags of the *_views entry points
FORWARD_GEOMETRY, FORWARD_RESUME = 4, 8        # a forward pass in two calls (render_views only)


class SceneView(C.Structure):
    """``DeodrSceneView`` (include/deodr_b200.h): device-resident scene in the canonical layout."""

    _fields_ = [
        ("faces", C.c_void_p),
        ("faces_uv", C.c_void_p),
        ("ij", C.c_void_p),
        ("depths", C.c_void_p),
        ("uv", C.c_void_p),
        ("colors", C.c_void_p),
        ("shade", C.c_void_p),
        ("edgeflags", C.c_void_p),
        ("textured", C.c_void_p),
        ("shaded", C.c_void_p),
        ("texture", C.c_void_p),
        ("background_image", C.c_void_p),
        ("background_color", C.c_void_p),
        ("nb_triangles", C.c_int32),
        ("nb_vertices", C.c_int32),
        ("nb_uv", C.c_int32),
        ("height", C.c_int32),
        ("width", C.c_int32),
        ("nb_colors", C.c_int32),
        ("texture_height", C.c_int32),
        ("texture_width", C.c_int32),
        ("clockwise", C.c_int32),
        ("backface_culling", C.c_int32),
        ("strict_edge", C.c_int32),
        ("perspective_correct", C.c_int32),
        ("integer_pixel_centers", C.c_int32),
    ]


class Grads(C.Structure):
    """``DeodrGrads``: fp32 device gradient slots, accumulated into."""

    _fields_ = [
        ("ij_b", C.c_void_p),
        ("colors_b", C.c_void_p),
        ("uv_b", C.c_void_p),
        ("shade_b", C.c_void_p),
        ("texture_b", C.c_void_p),
    ]


class ViewIO(C.Structure):
    """``DeodrViewIO``: per-view device framebuffers of the batched entry points."""

    _fields_ = [
        ("image", C.c_void_p),
        ("z_buffer", C.c_void_p),
        ("owner", C.c_void_p),
        ("face_id", C.c_void_p),
        ("barycentric", C.c_void_p),
        ("obs", C.c_void_p),
        ("err_buffer", C.c_void_p),
        ("image_b", C.c_void_p),
        ("err_buffer_b", C.c_void_p),
    ]


class Camera(C.Structure):
    """``DeodrCamera``: extrinsic [3,4], intrinsic [3,3] (row-major), distortion k1 k2 p1 p2 k3."""

    _fields_ = [
        ("extrinsic", C.c_double * 12),
        ("intrinsic", C.c_double * 9),
        ("distortion", C.c_double * 5),
        ("has_distortion", C.c_int32),
        ("pad", C.c_int32),
    ]


class MeshTopology(C.Structure):
    """``DeodrMeshTopology``: static adjacency of a triangulated mesh (device pointers)."""

    _fields_ = [
        ("faces", C.c_void_p),
        ("faces_edges", C.c_void_p),
        ("edge_face_offset", C.c_void_p),
        ("edge_face_index", C.c_void_p),
        ("vertex_face_offset", C.c_void_p),
        ("vertex_face_index", C.c_void_p),
        ("nb_faces", C.c_int32),
        ("nb_edges", C.c_int32),
        ("nb_vertices", C.c_int32),
        ("clockwise", C.c_int32),
    ]


class HostScene(C.Structure):
    """``DeodrHostScene`` == field order of the reference ``struct Scene`` (DifferentiableRenderer.h:56-90)."""

    _fields_ = [
        ("faces", C.c_void_p),
        ("faces_uv", C.c_void_p),
        ("depths", C.c_void_p),
        ("uv", C.c_void_p),
        ("ij", C.c_void_p),
        ("shade", C.c_void_p),
        ("colors", C.c_void_p),
        ("edgeflags", C.c_void_p),
        ("textured", C.c_void_p),
        ("shaded", C.c_void_p),
        ("nb_triangles", C.c_int32),
        ("nb_vertices", C.c_int32),
        ("clockwise", C.c_int32),
        ("backface_culling", C.c_int32),
        ("nb_uv", C.c_int32),
        ("height", C.c_int32),
        ("width", C.c_int32),
        ("nb_colors", C.c_int32),
        ("texture", C.c_void_p),
        ("texture_height", C.c_int32),
        ("texture_width", C.c_int32),
        ("background_image", C.c_void_p),
        ("background_color", C.c_void_p),
        ("uv_b", C.c_void_p),
        ("ij_b", C.c_void_p),
        ("shade_b", C.c_void_p),
        ("colors_b", C.c_void_p),
        ("texture_b", C.c_void_p),
        ("strict_edge", C.c_int32),
        ("perspective_correct", C.c_int32),
        ("integer_pixel_centers", C.c_int32),
    ]


# every symbol include/deodr_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("deodr_b200_workspace_create", C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    ("deodr_b200_workspace_destroy", None, [C.c_void_p]),
    ("deodr_b200_workspace_bytes", C.c_int64, [C.c_void_p]),
    ("deodr_b200_workspace_launches", C.c_int64, [C.c_void_p]),
    ("deodr_b200_render", C.c_int,
     [C.c_void_p, C.POINTER(SceneView), C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("deodr_b200_render_b", C.c_int,
     [C.c_void_p, C.POINTER(SceneView), C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Grads), C.c_void_p]),
    ("deodr_b200_render_views", C.c_int,
     [C.c_void_p, C.c_int, C.POINTER(SceneView), C.POINTER(ViewIO), C.c_double, C.c_int, C.c_void_p]),
    ("deodr_b200_render_b_views", C.c_int,
     [C.c_void_p, C.c_int, C.POINTER(SceneView), C.POINTER(ViewIO), C.POINTER(Grads), C.c_double, C.c_int, C.c_void_p]),
    ("deodr_b200_render_b_views_depths", C.c_int,
     [C.c_void_p, C.c_int, C.POINTER(SceneView), C.POINTER(ViewIO), C.POINTER(Grads), C.POINTER(C.c_void_p), C.c_double,
      C.c_int, C.c_void_p]),
    ("deodr_b200_workspace_set_deferred", C.c_int, [C.c_void_p, C.c_int]),
    ("deodr_b200_workspace_status", C.c_int, [C.c_void_p]),
    ("deodr_b200_view_generation", C.c_int64, [C.c_void_p, C.c_int]),
    ("deodr_b200_workspace_set_colors_ready", C.c_int, [C.c_void_p, C.c_void_p]),
    ("deodr_b200_project_points", C.c_int,
     [C.c_void_p, C.c_int, C.POINTER(Camera), C.c_void_p, C.c_void_p, C.c_void_p]),
    ("deodr_b200_project_points_b", C.c_int,
     [C.c_void_p, C.c_int, C.POINTER(Camera), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    ("deodr_b200_vertex_luminosity", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("deodr_b200_vertex_luminosity_b", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
      C.c_void_p, C.c_void_p]),
    ("deodr_b200_edge_on_silhouette", C.c_int,
     [C.POINTER(MeshTopology), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("deodr_b200_vertex_normals", C.c_int,
     [C.POINTER(MeshTopology), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("deodr_b200_vertex_normals_b", C.c_int,
     [C.POINTER(MeshTopology), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("deodr_b200_render_host", C.c_int,
     [C.c_void_p, C.POINTER(HostScene), C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p]),
    ("deodr_b200_render_b_host", C.c_int,
     [C.c_void_p, C.POINTER(HostScene), C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p,
      C.c_void_p, C.c_void_p]),
    ("deodr_b200_host_zero", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.c_int]),
    ("deodr_b200_check_scene", C.c_int, [C.c_void_p, C.POINTER(SceneView), C.c_void_p]),
    ("deodr_b200_timing_enable", C.c_int, [C.c_void_p, C.c_int]),
    ("deodr_b200_timing_collect", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    ("deodr_b200_phase_name", C.c_char_p, [C.c_int]),
    ("deodr_b200_last_error", C.c_char_p, []),
    ("deodr_b200_version", C.c_char_p, []),
]

_lib = None


def load() -> C.CDLL:
    """Load ``libdeodr_b200.so`` (built by ``__graft_entry__.build()`` / ``make -C deodr_b200/csrc``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build the sm_100a extension first (python -c 'import __graft_entry__ as g; "
                "g.build()').  deodr_b200 has no CPU fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, restype, argtypes in SYMBOLS:
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


class DeodrB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"deodr_b200 error {code}: {message}")
        self.code = code
        self.message = message


def check(code: int) -> None:
    if code != OK:
        raise DeodrB200Error(code, load().deodr_b200_last_error().decode())
