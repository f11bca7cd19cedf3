"""Device-resident front-end of the sm_100a rasteriser (thin ctypes layer over ``include/deodr_b200.h``).

``DeviceScene`` holds the canonical device copy of a ``Scene2DBase``-shaped object (fp64 ij / depths / uv, fp32
colours / shade / texture, u32 faces, u8 flags) as torch CUDA tensors; ``Renderer`` owns a ``DeodrWorkspace`` and
launches the forward (``renderScene``, DifferentiableRenderer.h:2717) and adjoint (``renderScene_B``,
DifferentiableRenderer.h:2903) passes on torch's current CUDA stream.  PyTorch is used for device memory and streams
only; all arithmetic happens in ``libdeodr_b200.so``.
"""

from __future__ import annotations

import ctypes as C
import threading
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _cabi


def _np(a, dtype):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(np.asarray(a), dtype=dtype)


class DeviceScene:
    """Canonical device copy of a 2.5D scene (fields of ``Scene2DBase``, deodr/differentiable_renderer.py:16-45)."""

    _F64 = ("ij", "depths", "uv")
    _F32 = ("colors", "shade", "texture")
    _U8 = ("edgeflags", "textured", "shaded")

    def __init__(self, scene, device: Optional[torch.device] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("deodr_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.height, self.width, self.nb_colors = int(scene.height), int(scene.width), int(scene.nb_colors)
        self.clockwise = bool(scene.clockwise)
        self.backface_culling = bool(scene.backface_culling)
        self.strict_edge = bool(scene.strict_edge)
        self.perspective_correct = bool(scene.perspective_correct)
        self.integer_pixel_centers = bool(scene.integer_pixel_centers)
        self.t: Dict[str, torch.Tensor] = {}
        # uint32 indices are stored as int32 bit patterns (torch has no general uint32 support)
        self.t["faces"] = self._up(_np(scene.faces, np.uint32).view(np.int32))
        self.t["faces_uv"] = self._up(_np(scene.faces_uv, np.uint32).view(np.int32))
        for name in self._F64:
            self.t[name] = self._up(_np(getattr(scene, name), np.float64))
        for name in self._F32:
            self.t[name] = self._up(_np(getattr(scene, name), np.float32))
        for name in self._U8:
            self.t[name] = self._up(_np(getattr(scene, name), np.uint8))
        bg_image = getattr(scene, "background_image", None)
        bg_color = getattr(scene, "background_color", None)
        assert (bg_image is not None) != (bg_color is not None), "provide background_image xor background_color"
        self.t["background_image"] = self._up(_np(bg_image, np.float32)) if bg_image is not None else None
        self.t["background_color"] = self._up(_np(bg_color, np.float32)) if bg_color is not None else None
        self._check_shapes()

    def _up(self, a: np.ndarray) -> torch.Tensor:
        return torch.from_numpy(a).to(self.device)

    def _check_shapes(self) -> None:
        t = self.t
        T, V, U = t["faces"].shape[0], t["depths"].shape[0], t["uv"].shape[0]
        assert t["faces"].shape == (T, 3) and t["faces_uv"].shape == (T, 3)
        assert t["ij"].shape == (V, 2) and t["uv"].shape == (U, 2)
        assert t["colors"].shape == (V, self.nb_colors) and t["shade"].shape == (V,)
        assert t["edgeflags"].shape == (T, 3) and t["textured"].shape == (T,) and t["shaded"].shape == (T,)
        if t["texture"].numel() > 0:
            assert t["texture"].dim() == 3 and t["texture"].shape[2] == self.nb_colors
        if t["background_image"] is not None:
            assert t["background_image"].shape == (self.height, self.width, self.nb_colors)
        else:
            assert t["background_color"].shape == (self.nb_colors,)

    def update(self, **arrays) -> None:
        """Refresh per-iteration inputs (e.g. ``ij=...``, ``colors=...``) in place; tensors or numpy arrays."""
        for name, value in arrays.items():
            dst = self.t[name]
            if isinstance(value, torch.Tensor):
                dst.copy_(value.to(dst.dtype).reshape(dst.shape), non_blocking=True)
            else:
                np_dtype = {torch.float64: np.float64, torch.float32: np.float32, torch.uint8: np.uint8,
                            torch.int32: np.int32}[dst.dtype]
                dst.copy_(torch.from_numpy(_np(value, np_dtype)).reshape(dst.shape), non_blocking=True)

    def view(self) -> _cabi.SceneView:
        t = self.t
        v = _cabi.SceneView()
        for name in ("faces", "faces_uv", "ij", "depths", "uv", "colors", "shade", "edgeflags", "textured", "shaded",
                     "texture"):
            setattr(v, name, t[name].data_ptr())
        v.background_image = t["background_image"].data_ptr() if t["background_image"] is not None else None
        v.background_color = t["background_color"].data_ptr() if t["background_color"] is not None else None
        v.nb_triangles, v.nb_vertices, v.nb_uv = t["faces"].shape[0], t["depths"].shape[0], t["uv"].shape[0]
        v.height, v.width, v.nb_colors = self.height, self.width, self.nb_colors
        if t["texture"].dim() == 3:
            v.texture_height, v.texture_width = t["texture"].shape[0], t["texture"].shape[1]
        v.clockwise = int(self.clockwise)
        v.backface_culling = int(self.backface_culling)
        v.strict_edge = int(self.strict_edge)
        v.perspective_correct = int(self.perspective_correct)
        v.integer_pixel_centers = int(self.integer_pixel_centers)
        return v

    def zero_grads(self) -> Dict[str, torch.Tensor]:
        t = self.t
        return {
            "ij_b": torch.zeros(t["ij"].shape, dtype=torch.float32, device=self.device),
            "colors_b": torch.zeros(t["colors"].shape, dtype=torch.float32, device=self.device),
            "uv_b": torch.zeros(t["uv"].shape, dtype=torch.float32, device=self.device),
            "shade_b": torch.zeros(t["shade"].shape, dtype=torch.float32, device=self.device),
            "texture_b": torch.zeros(t["texture"].shape, dtype=torch.float32, device=self.device),
        }


class Renderer:
    """Owns one ``DeodrWorkspace`` (one per device / stream).  The workspace is not thread-safe (the reference's Cython
    calls run under the GIL; ctypes releases it), so every call into the library holds this renderer's lock."""

    def __init__(self, device: Optional[int] = None):
        self.lib = _cabi.load()
        if not torch.cuda.is_available():
            raise RuntimeError("deodr_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self._lock = threading.RLock()
        self._ws = C.c_void_p()
        _cabi.check(self.lib.deodr_b200_workspace_create(C.byref(self._ws), self.device_index))

    def __del__(self):
        try:
            if getattr(self, "_ws", None) and self._ws.value:
                self.lib.deodr_b200_workspace_destroy(self._ws)
                self._ws = C.c_void_p()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(self.lib.deodr_b200_workspace_launches(self._ws))

    @property
    def workspace_bytes(self) -> int:
        return int(self.lib.deodr_b200_workspace_bytes(self._ws))

    def timing_enable(self, max_records: int) -> None:
        """Record CUDA-event pairs around the kernel groups of the next render / render_b calls."""
        with self._lock:
            _cabi.check(self.lib.deodr_b200_timing_enable(self._ws, int(max_records)))

    def timing_collect(self, capacity: int = 4096):
        """-> list of (phase name, milliseconds) in launch order; synchronises the recorded events."""
        phase = (C.c_int32 * capacity)()
        ms = (C.c_float * capacity)()
        with self._lock:
            n = self.lib.deodr_b200_timing_collect(self._ws, phase, ms, capacity)
        if n < 0:
            raise RuntimeError("timing_collect failed")
        return [(self.lib.deodr_b200_phase_name(phase[i]).decode(), float(ms[i])) for i in range(n)]

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device_index).cuda_stream

    def check_scene(self, scene: DeviceScene) -> None:
        v = scene.view()
        with self._lock:
            _cabi.check(self.lib.deodr_b200_check_scene(self._ws, C.byref(v), self._stream()))

    # ---- deferred mode / CUDA graphs ------------------------------------------------------------------------------
    def set_deferred(self, on: bool) -> None:
        """Deferred mode: the calls never read the device's verdict (nothing in them waits on the device), which makes
        a forward + adjoint sequence capturable in a CUDA graph; ask :meth:`status` after synchronising."""
        with self._lock:
            _cabi.check(self.lib.deodr_b200_workspace_set_deferred(self._ws, int(bool(on))))

    def status(self) -> None:
        """Raises ``DeodrB200Error`` (code EREPLAN) if a deferred pass overflowed its plan: its outputs are void and the
        pass must be run again (outside a capture) to rebuild the plan."""
        with self._lock:
            _cabi.check(self.lib.deodr_b200_workspace_status(self._ws))

    def set_colors_ready(self, event: Optional["torch.cuda.Event"]) -> None:
        """The next forward call makes only its colour readers (shading, edge records) wait for ``event`` - recorded by
        the caller on the stream where the all-reduce of ``colors_b`` and the optimiser update run - so that they overlap
        the binning and z pass of that forward (deodr_b200_workspace_set_colors_ready).  One-shot."""
        with self._lock:
            _cabi.check(self.lib.deodr_b200_workspace_set_colors_ready(
                self._ws, event.cuda_event if event is not None else None))

    def generation(self, view: int = 0) -> int:
        return int(self.lib.deodr_b200_view_generation(self._ws, int(view)))

    # ---- one view (slot 0) ----------------------------------------------------------------------------------------
    @staticmethod
    def _new_outputs(scene: DeviceScene, face_id: bool, barycentric: bool, err_buffer: bool) -> dict:
        dev, H, W, Cc = scene.device, scene.height, scene.width, scene.nb_colors
        return {
            "image": torch.empty((H, W, Cc), dtype=torch.float32, device=dev),
            "z_buffer": torch.empty((H, W), dtype=torch.float64, device=dev),
            "owner": torch.empty((H, W), dtype=torch.int32, device=dev),
            "face_id": torch.empty((H, W), dtype=torch.int32, device=dev) if face_id else None,
            "barycentric": torch.empty((H, W, 3), dtype=torch.float32, device=dev) if barycentric else None,
            "err_buffer": torch.empty((H, W), dtype=torch.float32, device=dev) if err_buffer else None,
        }

    @staticmethod
    def _io(out: dict, obs=None, image_b=None, err_buffer_b=None) -> _cabi.ViewIO:
        ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        return _cabi.ViewIO(ptr(out.get("image")), ptr(out.get("z_buffer")), ptr(out.get("owner")),
                            ptr(out.get("face_id")), ptr(out.get("barycentric")), ptr(obs), ptr(out.get("err_buffer")),
                            ptr(image_b), ptr(err_buffer_b))

    def render(self, scene: DeviceScene, sigma: float, face_id: bool = False, out: Optional[dict] = None,
               barycentric: bool = False, obs: Optional[torch.Tensor] = None):
        """Forward pass -> dict(image[H,W,C] f32, z_buffer[H,W] f64, owner[H,W] i32, face_id[H,W] i32 | None,
        barycentric[H,W,3] f32 | None, err_buffer[H,W] f32 | None, generation).

        ``obs`` ([H,W,C] f32 CUDA tensor) selects the reference's ``antialiase_error=True`` mode: the silhouette edges
        overdraw the squared residual ``err_buffer`` instead of the image (DR.h:2066-2618)."""
        return self.render_views([scene], sigma, face_id=face_id, out=[out] if out is not None else None,
                                 barycentric=barycentric, obs=[obs] if obs is not None else None)[0]

    def render_b(self, scene: DeviceScene, sigma: float, fwd: dict, image_b: Optional[torch.Tensor] = None,
                 grads: Optional[Dict[str, torch.Tensor]] = None, err_buffer_b: Optional[torch.Tensor] = None,
                 error_adjoint_complete: bool = False, depths_b: bool = False) -> Dict[str, torch.Tensor]:
        """Adjoint pass; accumulates into ``grads`` (created zeroed if None) and returns it.  In antialiase_error mode
        pass ``err_buffer_b`` ([H,W]) instead of ``image_b``.  ``depths_b=True``: see :meth:`render_b_views`."""
        return self.render_b_views([scene], sigma, [fwd], [image_b] if image_b is not None else None,
                                   [grads] if grads is not None else None,
                                   [err_buffer_b] if err_buffer_b is not None else None,
                                   error_adjoint_complete=error_adjoint_complete, depths_b=depths_b)[0]

    # ---- batch of views (slots 0 .. n-1) --------------------------------------------------------------------------
    def render_views(self, scenes: Sequence[DeviceScene], sigma: float, face_id: bool = False,
                     out: Optional[List[dict]] = None, barycentric: bool = False,
                     obs: Optional[Sequence[torch.Tensor]] = None, part: Optional[str] = None) -> List[dict]:
        """Forward passes of ``len(scenes)`` views in ONE library call (deodr_b200_render_views): the views are
        interleaved on a few internal streams and no pass waits for the host.

        ``part="geometry"`` enqueues only the head of the passes (list reset + binning: reads no colour) and
        ``part="resume"``, with the same arguments and ``out``, the rest: a caller whose colours come out of a
        collective puts its stream wait between the two calls (DEODR_B200_FORWARD_GEOMETRY / _RESUME)."""
        n = len(scenes)
        err_mode = obs is not None
        if out is None:
            out = [self._new_outputs(s, face_id, barycentric, err_mode) for s in scenes]
        views = (_cabi.SceneView * n)(*[s.view() for s in scenes])
        if err_mode:
            obs = [o.to(device=s.device, dtype=torch.float32).contiguous() for o, s in zip(obs, scenes)]
            for o, f in zip(out, obs):
                if o.get("err_buffer") is None:
                    o["err_buffer"] = torch.empty(o["z_buffer"].shape, dtype=torch.float32, device=o["z_buffer"].device)
        ios = (_cabi.ViewIO * n)(*[self._io(o, obs[i] if err_mode else None) for i, o in enumerate(out)])
        part_flag = {None: 0, "geometry": _cabi.FORWARD_GEOMETRY, "resume": _cabi.FORWARD_RESUME}[part]
        with self._lock:
            _cabi.check(self.lib.deodr_b200_render_views(self._ws, n, views, ios, float(sigma),
                                                         (_cabi.ANTIALIASE_ERROR if err_mode else 0) | part_flag,
                                                         self._stream()))
            if part == "geometry":
                return out  # no forward state yet: the "resume" call stamps the results
            for i, o in enumerate(out):
                o["generation"] = self.generation(i)
                o["slot"] = i
                o["obs"] = obs[i] if err_mode else None
        return out

    def render_b_views(self, scenes: Sequence[DeviceScene], sigma: float, fwds: Sequence[dict],
                       image_bs: Optional[Sequence[torch.Tensor]] = None,
                       grads: Optional[Sequence[Dict[str, torch.Tensor]]] = None,
                       err_buffer_bs: Optional[Sequence[torch.Tensor]] = None,
                       error_adjoint_complete: bool = False, depths_b: bool = False) -> List[Dict[str, torch.Tensor]]:
        """Adjoint passes of the views rendered by :meth:`render_views` (same order).  Entries of ``grads`` may share
        tensors: gradients of shared parameters accumulate in place (the ``+=`` of deodr/mesh_fitter.py:518-527).

        ``depths_b=True`` goes through deodr_b200_render_b_views_depths: ``perspective_correct`` views are accepted and
        each view's dict gets (or accumulates into its own) ``"depths_b"`` [V] fp32, the gradient of the vertex depths.
        It stays zero for views without ``perspective_correct``, whose image does not depend on the depths."""
        n = len(scenes)
        err_mode = err_buffer_bs is not None
        if grads is None:
            grads = [s.zero_grads() for s in scenes]
        if depths_b:
            for s, g in zip(scenes, grads):
                if g.get("depths_b") is None:
                    g["depths_b"] = torch.zeros(s.t["depths"].shape, dtype=torch.float32, device=s.device)
        for i, f in enumerate(fwds):
            if f.get("generation") is not None and f["generation"] != self.generation(f.get("slot", i)):
                raise RuntimeError(
                    "the forward state of this result has been overwritten by a later forward pass on the same "
                    "renderer slot: render again before render_b (one live forward per slot)")
        keep = []
        ios = []
        for i, (s, f) in enumerate(zip(scenes, fwds)):
            ib = eb = None
            if err_mode:
                eb = err_buffer_bs[i].to(device=s.device, dtype=torch.float32).contiguous()
                assert eb.shape == (s.height, s.width)
            else:
                ib = image_bs[i].to(device=s.device, dtype=torch.float32).contiguous()
                assert ib.shape == (s.height, s.width, s.nb_colors)
            keep.append((ib, eb))
            ios.append(self._io(f, f.get("obs"), ib, eb))
        views = (_cabi.SceneView * n)(*[s.view() for s in scenes])
        gs = (_cabi.Grads * n)(*[
            _cabi.Grads(*(g[k].data_ptr() if g.get(k) is not None and g[k].numel() > 0 else None
                          for k in ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b"))) for g in grads])
        flags = (_cabi.ANTIALIASE_ERROR if err_mode else 0) | (_cabi.ERROR_ADJOINT_COMPLETE if error_adjoint_complete else 0)
        with self._lock:
            if depths_b:
                dbs = (C.c_void_p * n)(*[g["depths_b"].data_ptr() if g["depths_b"].numel() > 0 else None for g in grads])
                _cabi.check(self.lib.deodr_b200_render_b_views_depths(self._ws, n, views, (_cabi.ViewIO * n)(*ios), gs,
                                                                      dbs, float(sigma), flags, self._stream()))
            else:
                _cabi.check(self.lib.deodr_b200_render_b_views(self._ws, n, views, (_cabi.ViewIO * n)(*ios), gs,
                                                               float(sigma), flags, self._stream()))
        del keep
        return list(grads)

    # ---- reference-shaped host entry points (fp64 numpy in / out), used by differentiable_renderer_cython.py ----
    def render_host(self, host_scene: _cabi.HostScene, image: np.ndarray, z_buffer: np.ndarray, sigma: float,
                    antialiase_error: bool = False, obs=None, err_buffer=None) -> None:
        with self._lock:
            _cabi.check(self.lib.deodr_b200_render_host(
                self._ws, C.byref(host_scene), image.ctypes.data, z_buffer.ctypes.data, float(sigma),
                int(bool(antialiase_error)), obs.ctypes.data if obs is not None else None,
                err_buffer.ctypes.data if err_buffer is not None else None))

    def render_b_host(self, host_scene: _cabi.HostScene, image: np.ndarray, z_buffer: np.ndarray,
                      image_b: Optional[np.ndarray], sigma: float, antialiase_error: bool = False, obs=None,
                      err_buffer=None, err_buffer_b=None) -> None:
        ptr = lambda a: a.ctypes.data if a is not None else None  # noqa: E731
        with self._lock:
            _cabi.check(self.lib.deodr_b200_render_b_host(
                self._ws, C.byref(host_scene), image.ctypes.data, z_buffer.ctypes.data, ptr(image_b), float(sigma),
                int(bool(antialiase_error)), ptr(obs), ptr(err_buffer), ptr(err_buffer_b)))

    def zero_host(self, arrays) -> None:
        """Zero-fills C-contiguous numpy arrays in place with the host path's copy threads (deodr_b200_host_zero)."""
        arrays = [a for a in arrays if a.size]
        ptrs = (C.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
        sizes = (C.c_int64 * len(arrays))(*[a.nbytes for a in arrays])
        with self._lock:
            _cabi.check(self.lib.deodr_b200_host_zero(self._ws, ptrs, sizes, len(arrays)))


_default: Dict[int, Renderer] = {}
_default_lock = threading.Lock()


def default_renderer(device: Optional[int] = None) -> Renderer:
    idx = torch.cuda.current_device() if device is None else int(device)
    with _default_lock:
        if idx not in _default:
            _default[idx] = Renderer(idx)
        return _default[idx]
