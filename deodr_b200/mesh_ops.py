"""The steps either side of the raster, on the device (SURVEY.md 8f1 / 8f2): thin wrappers over
``deodr_b200_project_points*``, ``deodr_b200_vertex_luminosity*``, ``deodr_b200_edge_on_silhouette`` and
``deodr_b200_vertex_normals*`` (include/deodr_b200.h, kernels in csrc/scene_ops.cu), plus ``DeviceMeshView``: one view
of a mesh rendered and back-propagated without a host round trip - vertices in, image out, ``vertices_b`` back.

Reference code these replace:
  Camera.project_points / project_points_backward        deodr/differentiable_renderer.py:341-438
  Scene3D.compute_vertices_luminosity (+ backward)        deodr/differentiable_renderer.py:814-850
  TriMeshAdjacencies (adjacency, normals, silhouette)     deodr/triangulated_mesh.py:21-166
PyTorch is used for device memory and streams only.
"""

from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _cabi


def _stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _f64(t: torch.Tensor, device) -> torch.Tensor:
    return t.to(device=device, dtype=torch.float64).contiguous()


class CameraParams:
    """Pinhole camera + OpenCV-style distortion, the fields of ``deodr.differentiable_renderer.Camera`` (:248-279)."""

    def __init__(self, extrinsic, intrinsic, distortion=None):
        self.extrinsic = np.ascontiguousarray(extrinsic, dtype=np.float64).reshape(3, 4)
        self.intrinsic = np.ascontiguousarray(intrinsic, dtype=np.float64).reshape(3, 3)
        self.distortion = None if distortion is None else np.ascontiguousarray(distortion, dtype=np.float64).reshape(5)

    @classmethod
    def from_reference(cls, camera) -> "CameraParams":
        """From any object with ``extrinsic`` / ``intrinsic`` / ``distortion`` (e.g. the reference's ``Camera``)."""
        return cls(camera.extrinsic, camera.intrinsic, camera.distortion)

    def c_struct(self) -> _cabi.Camera:
        c = _cabi.Camera()
        c.extrinsic[:] = self.extrinsic.reshape(-1).tolist()
        c.intrinsic[:] = self.intrinsic.reshape(-1).tolist()
        if self.distortion is not None:
            c.distortion[:] = self.distortion.tolist()
            c.has_distortion = 1
        return c


def project_points(points: torch.Tensor, camera: CameraParams) -> Tuple[torch.Tensor, torch.Tensor]:
    """``Camera.project_points``: points [N,3] (CUDA fp64) -> (ij [N,2] fp64 with column 0 = x, depths [N] fp64)."""
    points = _f64(points, points.device)
    n = points.shape[0]
    ij = torch.empty((n, 2), dtype=torch.float64, device=points.device)
    depths = torch.empty((n,), dtype=torch.float64, device=points.device)
    cam = camera.c_struct()
    _cabi.check(_cabi.load().deodr_b200_project_points(points.data_ptr(), n, C.byref(cam), ij.data_ptr(),
                                                       depths.data_ptr(), _stream(points.device)))
    return ij, depths


def project_points_backward(points: torch.Tensor, camera: CameraParams, ij_b: torch.Tensor,
                            depths_b: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                            reference_transpose: bool = False) -> torch.Tensor:
    """``Camera.project_points_backward``: accumulates into ``out`` ([N,3] fp64, created zeroed if None).

    ``reference_transpose=True`` reproduces the reference's final ``p_camera_b.dot(extrinsic[:3,:3].T)`` (:438), which
    is the adjoint only for a symmetric rotation (INTEGRATION.md, defect #3); the default is the true adjoint."""
    points = _f64(points, points.device)
    n = points.shape[0]
    ij_b = ij_b.to(device=points.device, dtype=torch.float32).contiguous()
    if depths_b is not None:
        depths_b = _f64(depths_b, points.device)
    if out is None:
        out = torch.zeros((n, 3), dtype=torch.float64, device=points.device)
    cam = camera.c_struct()
    _cabi.check(_cabi.load().deodr_b200_project_points_b(
        points.data_ptr(), n, C.byref(cam), ij_b.data_ptr(), depths_b.data_ptr() if depths_b is not None else None,
        out.data_ptr(), int(bool(reference_transpose)), _stream(points.device)))
    return out


def _light(light_directional):
    if light_directional is None:
        return None, None
    arr = np.ascontiguousarray(light_directional, dtype=np.float64).reshape(3)
    return arr, arr.ctypes.data


def vertex_luminosity(normals: torch.Tensor, vertex_colors: Optional[torch.Tensor], light_directional,
                      ambient: float) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """-> (luminosity [V] f32, colors [V,C] f32 = vertex_colors * luminosity, or None without vertex_colors)."""
    dev = normals.device
    normals = _f64(normals, dev)
    n = normals.shape[0]
    lum = torch.empty((n,), dtype=torch.float32, device=dev)
    colors = None
    C_ = 0
    if vertex_colors is not None:
        vertex_colors = _f64(vertex_colors, dev)
        C_ = vertex_colors.shape[1]
        colors = torch.empty((n, C_), dtype=torch.float32, device=dev)
    keep, lptr = _light(light_directional)
    _cabi.check(_cabi.load().deodr_b200_vertex_luminosity(
        normals.data_ptr(), vertex_colors.data_ptr() if vertex_colors is not None else None, n, C_, lptr, float(ambient),
        lum.data_ptr(), colors.data_ptr() if colors is not None else None, _stream(dev)))
    del keep
    return lum, colors


def vertex_luminosity_backward(normals: torch.Tensor, vertex_colors: Optional[torch.Tensor], light_directional,
                               ambient: float, colors_b: Optional[torch.Tensor] = None,
                               luminosity_b: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """-> dict(normals_b [V,3] f64, vertex_colors_b [V,C] f64 | None, light_b [4] f64 = (directional_b, ambient_b))."""
    dev = normals.device
    normals = _f64(normals, dev)
    n = normals.shape[0]
    C_ = 0
    vcol_b = None
    if vertex_colors is not None:
        vertex_colors = _f64(vertex_colors, dev)
        C_ = vertex_colors.shape[1]
        vcol_b = torch.zeros((n, C_), dtype=torch.float64, device=dev)
    if colors_b is not None:
        colors_b = colors_b.to(device=dev, dtype=torch.float32).contiguous()
    if luminosity_b is not None:
        luminosity_b = luminosity_b.to(device=dev, dtype=torch.float32).contiguous()
    normals_b = torch.zeros((n, 3), dtype=torch.float64, device=dev)
    light_b = torch.zeros((4,), dtype=torch.float64, device=dev)
    keep, lptr = _light(light_directional)
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    _cabi.check(_cabi.load().deodr_b200_vertex_luminosity_b(
        normals.data_ptr(), ptr(vertex_colors), n, C_, lptr, float(ambient), ptr(colors_b), ptr(luminosity_b),
        normals_b.data_ptr(), ptr(vcol_b), light_b.data_ptr(), _stream(dev)))
    del keep
    return {"normals_b": normals_b, "vertex_colors_b": vcol_b, "light_b": light_b}


def topology_arrays(faces, nb_vertices: Optional[int] = None) -> dict:
    """Host-side adjacency arrays of ``DeodrMeshTopology`` (numpy, int32): unique undirected edges, faces per edge and
    faces per vertex as CSR.  Edge n of a face joins its vertices n and (n + 1) % 3 (TriMeshAdjacencies, :42-44)."""
    faces = np.ascontiguousarray(np.asarray(faces), dtype=np.int64)
    assert faces.ndim == 2 and faces.shape[1] == 3
    T = faces.shape[0]
    V = int(faces.max()) + 1 if nb_vertices is None else int(nb_vertices)
    # unique undirected edges: any injective key works, only equality matters
    a = np.concatenate((faces[:, 0], faces[:, 1], faces[:, 2]))
    b = np.concatenate((faces[:, 1], faces[:, 2], faces[:, 0]))
    key = np.maximum(a, b) + np.minimum(a, b) * V
    _, edge_of = np.unique(key, return_inverse=True)
    edge_of = edge_of.reshape(-1)
    nb_edges = int(edge_of.max()) + 1 if T else 0
    face_of = np.tile(np.arange(T), 3)
    faces_edges = np.empty((T, 3), dtype=np.int32)
    faces_edges[face_of, np.repeat(np.arange(3), T)] = edge_of
    order = np.argsort(edge_of, kind="stable")
    edge_face_offset = np.zeros(nb_edges + 1, dtype=np.int32)
    np.cumsum(np.bincount(edge_of, minlength=nb_edges), out=edge_face_offset[1:])
    flat = faces.reshape(-1)
    vorder = np.argsort(flat, kind="stable")  # faces ascending inside a vertex, with multiplicity
    vertex_face_offset = np.zeros(V + 1, dtype=np.int32)
    np.cumsum(np.bincount(flat, minlength=V), out=vertex_face_offset[1:])
    return {
        "faces": np.ascontiguousarray(faces.astype(np.uint32).view(np.int32)),
        "faces_edges": faces_edges,
        "edge_face_offset": edge_face_offset,
        "edge_face_index": np.ascontiguousarray(face_of[order].astype(np.int32)),
        "vertex_face_offset": vertex_face_offset,
        "vertex_face_index": np.ascontiguousarray((vorder // 3).astype(np.int32)),
        "nb_faces": T, "nb_vertices": V, "nb_edges": nb_edges,
    }


class MeshTopology:
    """Static adjacency of a triangulated mesh on the device (``DeodrMeshTopology``), built once on the host from the
    same arrays as the reference's ``TriMeshAdjacencies`` (deodr/triangulated_mesh.py:21-98): unique undirected edges,
    the faces incident to every edge and to every vertex (CSR).  Edge n of a face joins vertices n and (n + 1) % 3, the
    order of ``faces_edges`` in the reference - which is also the order of the rasteriser's ``edgeflags`` columns."""

    def __init__(self, faces, nb_vertices: Optional[int] = None, clockwise: bool = False, device="cuda"):
        arrays = topology_arrays(faces, nb_vertices)
        self.nb_faces, self.nb_vertices, self.nb_edges = arrays["nb_faces"], arrays["nb_vertices"], arrays["nb_edges"]
        self.clockwise = bool(clockwise)
        dev = torch.device(device)
        self.device = dev
        self.t = {k: torch.from_numpy(v).to(dev) for k, v in arrays.items() if isinstance(v, np.ndarray)}

    def c_struct(self) -> _cabi.MeshTopology:
        m = _cabi.MeshTopology()
        for name, t in self.t.items():
            setattr(m, name, t.data_ptr())
        m.nb_faces, m.nb_edges, m.nb_vertices, m.clockwise = self.nb_faces, self.nb_edges, self.nb_vertices, int(self.clockwise)
        return m

    def edge_on_silhouette(self, ij: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``TriMeshAdjacencies.edge_on_silhouette`` (:153-166): edgeflags [T,3] uint8 for the projection ``ij`` [V,2]."""
        ij = _f64(ij, self.device)
        if out is None:
            out = torch.empty((self.nb_faces, 3), dtype=torch.uint8, device=self.device)
        visible = torch.empty((self.nb_faces,), dtype=torch.uint8, device=self.device)
        m = self.c_struct()
        _cabi.check(_cabi.load().deodr_b200_edge_on_silhouette(C.byref(m), ij.data_ptr(), visible.data_ptr(),
                                                               out.data_ptr(), _stream(self.device)))
        return out

    def vertex_normals(self, vertices: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """-> (face_normals [T,3], vertex_normals [V,3]) fp64 (compute_face_normals + compute_vertex_normals)."""
        vertices = _f64(vertices, self.device)
        fn = torch.empty((self.nb_faces, 3), dtype=torch.float64, device=self.device)
        vn = torch.empty((self.nb_vertices, 3), dtype=torch.float64, device=self.device)
        m = self.c_struct()
        _cabi.check(_cabi.load().deodr_b200_vertex_normals(C.byref(m), vertices.data_ptr(), fn.data_ptr(), vn.data_ptr(),
                                                           _stream(self.device)))
        return fn, vn

    def vertex_normals_backward(self, vertices: torch.Tensor, vertex_normals_b: torch.Tensor,
                                out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Accumulates the adjoint of :meth:`vertex_normals` into ``out`` ([V,3] fp64, created zeroed if None)."""
        vertices = _f64(vertices, self.device)
        vertex_normals_b = _f64(vertex_normals_b, self.device)
        if out is None:
            out = torch.zeros((self.nb_vertices, 3), dtype=torch.float64, device=self.device)
        scratch = torch.empty((self.nb_vertices, 3), dtype=torch.float64, device=self.device)
        m = self.c_struct()
        _cabi.check(_cabi.load().deodr_b200_vertex_normals_b(C.byref(m), vertices.data_ptr(), vertex_normals_b.data_ptr(),
                                                             scratch.data_ptr(), out.data_ptr(), _stream(self.device)))
        return out


class DeviceMeshView:
    """One view of a Gouraud-lit mesh, device-resident end to end: the chain of ``Scene3D.render`` /
    ``render_backward`` (deodr/differentiable_renderer.py:871-1052) with every step on the GPU -

        vertices -> normals -> luminosity -> colours        project_points -> ij, depths -> silhouette flags
        -> rasteriser (deodr_b200_render) -> image          image_b -> rasteriser adjoint -> ij_b, colors_b
        -> luminosity / normals / projection adjoints -> vertices_b (+ vertex_colors_b, light_b)

    No tensor crosses PCIe inside :meth:`render` / :meth:`backward`; the shared gradients of several views are plain
    CUDA tensors that a caller sums over views and all-reduces over ranks (deodr_b200.distributed).

    ``perspective_correct=True`` renders with perspective-correct interpolation; :meth:`backward` then also takes the
    rasteriser's gradient of the vertex depths through the projection adjoint."""

    def __init__(self, faces, nb_vertices: int, camera: CameraParams, height: int, width: int, renderer=None,
                 light_directional=None, ambient: float = 1.0, background_color=(0.0, 0.0, 0.0), sigma: float = 1.0,
                 clockwise: bool = False, device="cuda", slot: int = 0, perspective_correct: bool = False):
        from .renderer import DeviceScene, default_renderer
        from .scenes import SceneArrays

        self.device = torch.device(device)
        self.topology = MeshTopology(faces, nb_vertices, clockwise=clockwise, device=self.device)
        self.camera, self.sigma = camera, float(sigma)
        self.light_directional, self.ambient = light_directional, float(ambient)
        faces_u32 = np.ascontiguousarray(faces, dtype=np.uint32)
        T, V = faces_u32.shape[0], int(nb_vertices)
        nb_colors = len(background_color)
        arrays = SceneArrays(
            faces=faces_u32, faces_uv=np.zeros((T, 3), np.uint32), ij=np.zeros((V, 2)), depths=np.ones(V),
            textured=np.zeros(T, bool), uv=np.zeros((1, 2)), shade=np.zeros(V), colors=np.zeros((V, nb_colors)),
            shaded=np.zeros(T, bool), edgeflags=np.zeros((T, 3), bool), height=height, width=width, nb_colors=nb_colors,
            texture=np.zeros((2, 2, nb_colors)), background_image=None,
            background_color=np.asarray(background_color, dtype=np.float64), clockwise=clockwise, backface_culling=True,
            strict_edge=True, perspective_correct=bool(perspective_correct), integer_pixel_centers=True)
        self.scene = DeviceScene(arrays, self.device)
        self.renderer = renderer if renderer is not None else default_renderer(self.device.index)
        self._saved = None

    def render(self, vertices: torch.Tensor, vertex_colors: torch.Tensor) -> torch.Tensor:
        vertices = _f64(vertices, self.device)
        _, normals = self.topology.vertex_normals(vertices)
        _, colors = vertex_luminosity(normals, vertex_colors, self.light_directional, self.ambient)
        ij, depths = project_points(vertices, self.camera)
        t = self.scene.t
        t["ij"].copy_(ij)
        t["depths"].copy_(depths)
        t["colors"].copy_(colors)
        self.topology.edge_on_silhouette(ij, out=t["edgeflags"])
        fwd = self.renderer.render(self.scene, self.sigma)
        self._saved = (vertices, _f64(vertex_colors, self.device), normals, fwd)
        return fwd["image"]

    def backward(self, image_b: torch.Tensor, reference_transpose: bool = False) -> Dict[str, torch.Tensor]:
        """-> dict(vertices_b [V,3] f64, vertex_colors_b [V,C] f64, light_b [4] f64)."""
        vertices, vertex_colors, normals, fwd = self._saved
        persp = self.scene.perspective_correct
        grads = self.renderer.render_b(self.scene, self.sigma, fwd, image_b, depths_b=persp)
        lum = vertex_luminosity_backward(normals, vertex_colors, self.light_directional, self.ambient,
                                         colors_b=grads["colors_b"])
        vertices_b = self.topology.vertex_normals_backward(vertices, lum["normals_b"])
        project_points_backward(vertices, self.camera, grads["ij_b"],
                                depths_b=grads["depths_b"].to(torch.float64) if persp else None, out=vertices_b,
                                reference_transpose=reference_transpose)
        return {"vertices_b": vertices_b, "vertex_colors_b": lum["vertex_colors_b"], "light_b": lum["light_b"]}
