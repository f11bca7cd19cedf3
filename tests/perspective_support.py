"""TEST INFRASTRUCTURE ONLY - checkers of the perspective-correct adjoint (deodr_b200_render_b_views_depths).

* ``PerspOracle``: the port oracle (oracle/deodr_oracle.c) plus our own fp64 perspective-correct adjoint,
  ``render_b_depths`` (tests/perspective/persp_oracle.c).  The reference has no such adjoint.
* ``PerspEmulator``: the CPU emulation of the kernel phases (tests/emul/emul.cpp) plus ``render_b_depths``, the
  emulated form of the new entry point (tests/perspective/persp_emul.cpp).

Both sources include the existing ones unchanged and are compiled here into libraries of their own, next to them.
"""
import ctypes as C
import os
import subprocess
from typing import Dict

import numpy as np
from canon import Emulator

from deodr_b200 import _cabi
from oracle.oracle import Oracle, SceneC, _f64

_HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "perspective")
GRADS = ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b")


def _build(cmd, out, deps, libs=()):
    """Compiles deps[0] into `out` unless it is newer than every dependency."""
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.run(cmd + ["-o", out, deps[0]] + list(libs), check=True, capture_output=True)
    return out


def _oracle_lib() -> str:
    root = os.path.dirname(_HERE)
    src = os.path.join(_HERE, "persp_oracle.c")
    deps = [src, os.path.join(os.path.dirname(root), "oracle", "deodr_oracle.c")]
    cmd = [os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-std=c99", "-ffp-contract=off", "-fno-fast-math", "-Wall",
           "-Wno-unused-function", "-shared"]
    return _build(cmd, os.path.join(_HERE, "libpersp_oracle.so"), deps, ["-lm"])


def _emul_lib(exact_short_wrap: bool = False) -> str:
    src = os.path.join(_HERE, "persp_emul.cpp")
    csrc = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "deodr_b200", "csrc")
    deps = [src, os.path.join(os.path.dirname(_HERE), "emul", "emul.cpp")] + [
        os.path.join(csrc, h) for h in ("phases.h", "shade.h", "rmath.h")]
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall",
           "-Wno-unused-function", "-Wno-maybe-uninitialized", "-shared"]
    if exact_short_wrap:  # the build of tests/emul/Makefile's libemul_wrap.so
        cmd.append("-DDEODR_EXACT_SHORT_WRAP=1")
    name = "libpersp_emul_wrap.so" if exact_short_wrap else "libpersp_emul.so"
    return _build(cmd, os.path.join(_HERE, name), deps)


class PerspOracle(Oracle):
    """The port oracle with ``render_b_depths``: every call goes to the library built from persp_oracle.c."""

    def __init__(self, texfix: bool = True):
        super().__init__("port", texfix=texfix)
        self.lib = C.CDLL(_oracle_lib())
        self._render = self.lib.deodr_oracle_render
        self._render_b = self.lib.deodr_oracle_render_b
        self._err = self.lib.deodr_oracle_last_error
        self._err.restype = C.c_char_p
        self._render.restype = self._render_b.restype = C.c_int
        self._render.argtypes = [C.POINTER(SceneC), C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p]
        self._render_b.argtypes = [C.POINTER(SceneC), C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
        self._render_b_depths = self.lib.deodr_oracle_render_b_depths
        self._render_b_depths.restype = C.c_int
        self._render_b_depths.argtypes = [C.POINTER(SceneC), C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]

    def render_b_depths(self, scene, sigma: float, image: np.ndarray, z_buffer: np.ndarray,
                        image_b: np.ndarray) -> Dict[str, np.ndarray]:
        """Adjoint pass that also accepts ``perspective_correct`` scenes: ``render_b``'s gradients plus ``depths_b`` [V],
        which stays zero without ``perspective_correct``.  Works on copies of ``image`` / ``image_b``."""
        self._select()
        s, keep = self._pack(scene, with_grads=True)
        image_c = _f64(image).copy()
        z_c = _f64(z_buffer)
        image_b_c = _f64(image_b).copy()
        depths_b = np.zeros(keep["depths"].shape, dtype=np.float64)
        rc = self._render_b_depths(C.byref(s), image_c.ctypes.data, z_c.ctypes.data, image_b_c.ctypes.data,
                                   float(sigma), depths_b.ctypes.data)
        if rc != 0:
            raise RuntimeError(self._err().decode())
        grads = {k: keep[k] for k in GRADS}
        grads["depths_b"] = depths_b
        return grads


class PerspEmulator(Emulator):
    """The emulation of the kernel phases with ``render_b_depths`` (emul_render_b_depths)."""

    def __init__(self, exact_short_wrap: bool = False):
        super().__init__(exact_short_wrap=exact_short_wrap)
        base = self.lib
        self.lib = C.CDLL(_emul_lib(exact_short_wrap))
        for name in ("emul_render", "emul_weight_scale", "emul_render_error", "emul_render_error_b", "emul_render_b"):
            getattr(self.lib, name).argtypes = getattr(base, name).argtypes
            getattr(self.lib, name).restype = getattr(base, name).restype
        self.lib.emul_render_b_depths.argtypes = [C.POINTER(_cabi.SceneView), C.c_double, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.POINTER(_cabi.Grads), C.c_void_p]

    def render_b_depths(self, scene, sigma, fwd, image_b):
        a = fwd["_arrays"]
        ib = np.ascontiguousarray(image_b, dtype=np.float32)
        g = {k: np.zeros(a[k[:-2]].shape, np.float32) for k in GRADS + ("depths_b",)}
        gs = _cabi.Grads(*(g[k].ctypes.data for k in GRADS))
        rc = self.lib.emul_render_b_depths(C.byref(fwd["_view"]), float(sigma), fwd["z"].ctypes.data,
                                           fwd["owner"].ctypes.data, ib.ctypes.data, C.byref(gs),
                                           g["depths_b"].ctypes.data)
        assert rc == 0
        return g
