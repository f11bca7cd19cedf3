"""Recorded renderer calls of the reference's own examples and tests, and their results from the reference's extension.

``Recorder`` wraps ``renderSceneCpp`` / ``renderSceneBCpp`` of the reference's extension while the reference's code runs
unchanged (tests/dropin/runner.py).  For every selected call it re-runs the call (an adjoint call on the
results of the re-run forward call before it) on a copy of its arguments in which the image-sized inputs are replaced
by ones that take little room, and keeps what the reference's extension returned for exactly those inputs:

* the scene: every field; geometry, uv, shade and colours rounded to fp32, texture and background image quantized to 8
  bits; the gradients it accumulates into start from zero;
* inputs: obs and err_buffer_b quantized to 8 bits; image_b replaced by a dense uniform [-1, 1) image drawn from a
  seeded generator (``dense_image_b``), so that every pixel's adjoint is exercised;
* forward: the image, z-buffer (and err_buffer) at up to ``SAMPLE`` seeded pixels, plus full per-channel sums;
* adjoint: the accumulated gradients but texture_b (see ``GRADS``), at up to ``SAMPLE`` seeded entries each, plus
  the sums of all their entries and of their absolute values.

Arrays are stored once by content, with a JSON manifest (``save``); ``load`` and ``resolve`` turn such a file back
into calls.
"""
import copy
import hashlib
import io
import json
import zipfile

import numpy as np

SAMPLE = 256
SCENE_ARRAYS = ("faces", "faces_uv", "ij", "depths", "textured", "uv", "shade", "colors", "shaded", "edgeflags",
                "texture", "background_image", "background_color")
SCENE_SCALARS = ("height", "width", "nb_colors", "clockwise", "backface_culling", "strict_edge", "perspective_correct",
                 "integer_pixel_centers")
QUANTIZED = ("texture", "background_image", "obs", "err_buffer_b")
SINGLE = ("ij", "depths", "uv", "shade", "colors")
# texture_b is left out: the reference's bilinear_sample_B stores the texel adjoint with `=` where the sum needs `+=`
# (DifferentiableRenderer.h:621-624), and deodr_b200 returns the sum; texture_b is checked against an oracle with the
# sum (the `checker` fixture, __graft_entry__.smoke)
GRADS = ("ij_b", "colors_b", "uv_b", "shade_b")


def quantize(a):
    """8-bit levels of a non-negative array: ``(q, scale)`` with ``q * scale`` the value that is used and stored."""
    assert a.size == 0 or a.min() >= 0
    scale = float(a.max()) / 255 if a.size and a.max() > 0 else 1.0
    return np.round(a / scale).astype(np.uint8), scale


def dequantize(q, scale):
    return q.astype(np.float64) * scale


def dense_image_b(seed, shape):
    return np.random.default_rng(seed).random(shape) * 2 - 1


def _np(a):
    if a is None:
        return None
    if hasattr(a, "detach"):
        a = a.detach().numpy()
    return np.asarray(a)


class Recorder:
    def __init__(self, render, render_b, keep=None):
        self.fwd, self.bwd, self.keep = render, render_b, keep
        self.n_fwd = 0
        self.recording = False
        self.last = None
        self.arrays, self.calls = {}, []

    def _put(self, a):
        a = np.ascontiguousarray(a)
        key = "a" + hashlib.sha256(a.dtype.str.encode() + str(a.shape).encode() + a.tobytes()).hexdigest()[:16]
        self.arrays[key] = a
        return key

    def _put_q(self, a):
        q, scale = quantize(a)
        return {"q": self._put(q), "scale": scale}

    def _q(self, a):
        return None if a is None else dequantize(*quantize(_np(a)))

    def _scene(self, scene):
        out = {}
        for name in SCENE_ARRAYS:
            a = _np(getattr(scene, name, None))
            out[name] = (None if a is None else self._put_q(a) if name in QUANTIZED else
                         self._put(a.astype(np.float32)) if name in SINGLE else self._put(a))
        out.update({name: int(getattr(scene, name)) for name in SCENE_SCALARS})
        return out

    @staticmethod
    def _reduced_copy(scene):
        s = copy.copy(scene)
        for name in SCENE_ARRAYS:
            a = _np(getattr(s, name, None))
            if a is not None:
                a = (dequantize(*quantize(a)) if name in QUANTIZED else
                     a.astype(np.float32).astype(np.float64) if name in SINGLE else np.array(a))
            setattr(s, name, a)
        for name, like in (("uv_b", "uv"), ("ij_b", "ij"), ("shade_b", "shade"), ("colors_b", "colors"),
                           ("texture_b", "texture")):
            setattr(s, name, np.zeros_like(getattr(s, like)))
        return s

    def _sample(self, shape, seed):
        n = int(np.prod(shape[:2]))
        idx = np.arange(n) if n <= SAMPLE else np.sort(np.random.default_rng(seed).choice(n, SAMPLE, replace=False))
        return idx.astype(np.int32)

    def render(self, scene, sigma, image, z_buffer, antialiase_error=0, obs=None, err_buffer=None, *a, **k):
        self.fwd(scene, sigma, image, z_buffer, antialiase_error, obs, err_buffer, *a, **k)
        self.recording = self.keep is None or self.n_fwd in self.keep
        self.n_fwd += 1
        if not self.recording:
            return
        s = self._reduced_copy(scene)
        obs_r = self._q(obs)
        im = np.zeros_like(image)
        z = np.zeros_like(z_buffer)
        err = None if err_buffer is None else np.zeros_like(err_buffer)
        self.fwd(s, sigma, im, z, antialiase_error, obs_r, err, *a, **k)
        self.last = im, z, err
        idx = self._sample(im.shape, len(self.calls))
        flat = lambda x: x.reshape(x.shape[0] * x.shape[1], -1)[idx]  # noqa: E731
        call = {"kind": "render", "sigma": float(sigma), "antialiase_error": bool(antialiase_error),
                "scene": self._scene(s), "obs": None if obs_r is None else self._put_q(obs_r),
                "image_shape": list(im.shape), "pixels": self._put(idx),
                "image": self._put(flat(im).astype(np.float32)), "z_buffer": self._put(flat(z)[:, 0]),
                "image_sum": [float(v) for v in im.reshape(-1, im.shape[2]).sum(0)],
                "err_buffer": None if err is None else self._put(flat(err)[:, 0].astype(np.float32)),
                "err_sum": None if err is None else float(err.sum())}
        self.calls.append(call)

    def render_b(self, scene, sigma, image, z_buffer, image_b=None, antialiase_error=0, obs=None, err_buffer=None,
                 err_buffer_b=None, *a, **k):
        if self.recording:
            s = self._reduced_copy(scene)
            seed = len(self.calls)
            ib = None if image_b is None else dense_image_b(seed, image_b.shape)
            ob, eb = self._q(obs), self._q(err_buffer_b)
            call = {"kind": "render_b", "sigma": float(sigma), "antialiase_error": bool(antialiase_error),
                    "scene": self._scene(s), "image_b_seed": None if ib is None else seed,
                    "obs": None if ob is None else self._put_q(ob),
                    "err_buffer_b": None if eb is None else self._put_q(eb), "image_shape": list(image.shape)}
            im, z, err = (None if x is None else x.copy() for x in self.last)  # the recorded forward's results
            self.bwd(s, sigma, im, z, None if ib is None else ib.copy(), antialiase_error, ob, err,
                     None if eb is None else eb.copy(), *a, **k)
            for name in GRADS:
                g = _np(getattr(s, name))
                idx = np.arange(g.size) if g.size <= SAMPLE else np.sort(
                    np.random.default_rng(seed).choice(g.size, SAMPLE, replace=False))
                call[name] = {"index": self._put(idx.astype(np.int32)),
                              "values": self._put(g.reshape(-1)[idx].astype(np.float32)), "sum": float(g.sum()),
                              "abs_sum": float(np.abs(g).sum())}
            self.calls.append(call)
        self.bwd(scene, sigma, image, z_buffer, image_b, antialiase_error, obs, err_buffer, err_buffer_b, *a, **k)

    def save(self, path):
        save(path, {"calls": self.calls}, self.arrays)


def save(path, manifest, arrays):
    """An .npz with LZMA-compressed members (np.load reads them): about 15 % smaller than np.savez_compressed."""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for name, a in {"manifest": np.array(json.dumps(manifest)), **arrays}.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(a), allow_pickle=False)
            z.writestr(name + ".npy", buf.getvalue())


def load(path):
    """(manifest, arrays) of a recording: its JSON manifest and the arrays it names."""
    d = np.load(path)
    return json.loads(str(d["manifest"])), {k: d[k] for k in d.files if k != "manifest"}


def resolve(v, arrays):
    """``v`` with every array key replaced by its array and every quantized array by its values."""
    if isinstance(v, dict):
        if set(v) == {"q", "scale"}:
            return dequantize(arrays[v["q"]], v["scale"])
        return {k: resolve(x, arrays) for k, x in v.items()}
    if isinstance(v, str) and v in arrays:
        return arrays[v]
    return v
