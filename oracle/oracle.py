"""TEST INFRASTRUCTURE ONLY - ctypes front-end of the CPU oracles.

Two interchangeable back-ends with the same Python API:

* ``kind="reference"``: ``oracle/_ref/libdeodr_ref.so`` = the unmodified reference core
  (C++/DifferentiableRenderer.h ``renderScene`` :2717 / ``renderScene_B`` :2903) compiled by ``oracle/Makefile`` from
  where it lies under /root/reference (never copied into this repository).  ``texfix=True`` selects the variant in
  which the ``=`` of ``bilinear_sample_B`` (DifferentiableRenderer.h:621-624) is patched to ``+=``.
* ``kind="port"``: ``oracle/liboracle.so`` = our own C restatement (``oracle/deodr_oracle.c``).  ``texfix`` is a
  process-wide switch of that library, so every call of a port oracle sets it to the oracle's own ``texfix`` first.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import this module.  The product package ``deodr_b200`` never does.
"""

from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Dict, Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


class SceneC(C.Structure):
    """Mirror of ``struct RefSceneC`` (oracle/ref_shim.cpp) == field order of DifferentiableRenderer.h:56-90."""

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


def build(verbose: bool = False) -> None:
    """Compile liboracle.so (always) and oracle/_ref (only where /root/reference exists)."""
    out = subprocess.run(["make", "-C", _HERE, "all"], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout, out.stderr)
    if out.returncode != 0:
        raise RuntimeError("oracle build failed")


def _lib_path(kind: str, texfix: bool) -> str:
    if kind == "reference":
        return os.path.join(_HERE, "_ref", "libdeodr_ref_texfix.so" if texfix else "libdeodr_ref.so")
    if kind == "port":
        return os.path.join(_HERE, "liboracle.so")
    raise ValueError(kind)


def available(kind: str, texfix: bool = False) -> bool:
    return os.path.exists(_lib_path(kind, texfix))


def _f64(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a), dtype=np.float64)


class Oracle:
    """CPU oracle; ``render``/``render_b`` take any object with the ``Scene2DBase`` attributes."""

    def __init__(self, kind: str = "reference", texfix: bool = False):
        path = _lib_path(kind, texfix)
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run `make -C oracle`")
        self.kind = kind
        self.texfix = texfix
        self.lib = C.CDLL(path)
        prefix = "deodr_ref" if kind == "reference" else "deodr_oracle"
        self._render = getattr(self.lib, prefix + "_render")
        self._render_b = getattr(self.lib, prefix + "_render_b")
        self._err = getattr(self.lib, prefix + "_last_error")
        self._err.restype = C.c_char_p
        self._render.restype = C.c_int
        self._render_b.restype = C.c_int
        self._render.argtypes = [C.POINTER(SceneC), C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p]
        self._render_b.argtypes = [
            C.POINTER(SceneC), C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p,
            C.c_void_p,
        ]

    def _select(self) -> None:
        if self.kind == "port":
            self.lib.deodr_oracle_set_texfix(int(self.texfix))

    # -- marshalling -------------------------------------------------------------------------------------------
    @staticmethod
    def _pack(scene, with_grads: bool) -> Tuple[SceneC, Dict[str, np.ndarray]]:
        keep: Dict[str, np.ndarray] = {}
        keep["faces"] = np.ascontiguousarray(scene.faces, dtype=np.uint32)
        keep["faces_uv"] = np.ascontiguousarray(scene.faces_uv, dtype=np.uint32)
        for name in ("depths", "uv", "ij", "shade", "colors", "texture"):
            keep[name] = _f64(getattr(scene, name))
        for name in ("edgeflags", "textured", "shaded"):
            keep[name] = np.ascontiguousarray(np.asarray(getattr(scene, name)), dtype=np.uint8)
        s = SceneC()
        for name in ("faces", "faces_uv", "depths", "uv", "ij", "shade", "colors", "edgeflags", "textured", "shaded",
                     "texture"):
            setattr(s, name, keep[name].ctypes.data)
        s.nb_triangles = keep["faces"].shape[0]
        s.nb_vertices = keep["depths"].shape[0]
        s.nb_uv = keep["uv"].shape[0]
        s.clockwise = int(bool(scene.clockwise))
        s.backface_culling = int(bool(scene.backface_culling))
        s.height, s.width, s.nb_colors = int(scene.height), int(scene.width), int(scene.nb_colors)
        s.texture_height, s.texture_width = int(keep["texture"].shape[0]), int(keep["texture"].shape[1])
        if getattr(scene, "background_image", None) is not None:
            keep["background_image"] = _f64(scene.background_image)
            s.background_image = keep["background_image"].ctypes.data
            s.background_color = None
        else:
            keep["background_color"] = _f64(scene.background_color)
            s.background_color = keep["background_color"].ctypes.data
            s.background_image = None
        s.strict_edge = int(bool(scene.strict_edge))
        s.perspective_correct = int(bool(scene.perspective_correct))
        s.integer_pixel_centers = int(bool(scene.integer_pixel_centers))
        if with_grads:
            for name, src in (("uv_b", "uv"), ("ij_b", "ij"), ("shade_b", "shade"), ("colors_b", "colors"),
                              ("texture_b", "texture")):
                keep[name] = np.zeros(keep[src].shape, dtype=np.float64)
                setattr(s, name, keep[name].ctypes.data)
        return s, keep

    # -- API ---------------------------------------------------------------------------------------------------
    def render(self, scene, sigma: float, antialiase_error: bool = False, obs: Optional[np.ndarray] = None):
        """Forward pass -> ``(image[H,W,C], z_buffer[H,W])`` (+ ``err_buffer[H,W]`` in antialiase_error mode)."""
        self._select()
        s, keep = self._pack(scene, with_grads=False)
        image = np.zeros((s.height, s.width, s.nb_colors))
        z_buffer = np.zeros((s.height, s.width))
        err_buffer = np.zeros((s.height, s.width)) if antialiase_error else None
        obs_c = _f64(obs) if antialiase_error else None
        rc = self._render(
            C.byref(s), image.ctypes.data, z_buffer.ctypes.data, float(sigma), int(antialiase_error),
            obs_c.ctypes.data if obs_c is not None else None,
            err_buffer.ctypes.data if err_buffer is not None else None,
        )
        if rc != 0:
            raise RuntimeError(self._err().decode())
        del keep
        return (image, z_buffer, err_buffer) if antialiase_error else (image, z_buffer)

    def render_b(self, scene, sigma: float, image: np.ndarray, z_buffer: np.ndarray, image_b: np.ndarray,
                 antialiase_error: bool = False, obs=None, err_buffer=None, err_buffer_b=None) -> Dict[str, np.ndarray]:
        """Adjoint pass on COPIES of ``image`` / ``image_b`` -> dict of zero-initialised-then-accumulated gradients."""
        self._select()
        s, keep = self._pack(scene, with_grads=True)
        image_c = _f64(image).copy()
        z_c = _f64(z_buffer)
        image_b_c = _f64(image_b).copy() if image_b is not None else None
        obs_c = _f64(obs) if obs is not None else None
        err_c = _f64(err_buffer).copy() if err_buffer is not None else None
        err_b_c = _f64(err_buffer_b).copy() if err_buffer_b is not None else None
        ptr = lambda a: a.ctypes.data if a is not None else None  # noqa: E731
        rc = self._render_b(C.byref(s), image_c.ctypes.data, z_c.ctypes.data, ptr(image_b_c), float(sigma),
                            int(antialiase_error), ptr(obs_c), ptr(err_c), ptr(err_b_c))
        if rc != 0:
            raise RuntimeError(self._err().decode())
        grads = {k: keep[k] for k in ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b")}
        grads["image_after"] = image_c
        grads["image_b_after"] = image_b_c
        return grads
