"""GPU (-m gpu): drop-in acceptance against the REFERENCE's own extension.

deodr_b200.differentiable_renderer_cython stands in for ``deodr.differentiable_renderer_cython`` - the one-line swap of
INTEGRATION.md.  tests/golden/dropin_calls.npz holds renderer calls made by the reference's own convention tests and
example fitters, recorded while that code ran with the reference's own extension, and what the extension returned for
them (tests/golden/make_dropin_calls.py, tests/dropin/dropin_calls.py).  Each test replays its calls, in order,
through renderSceneCpp / renderSceneBCpp, each adjoint call on the image and z-buffer of the forward call before it,
and compares:

* z-buffer: equal to fp64 round-off (rtol 1e-12) at the stored pixels;
* image and err_buffer: within 4e-6 of the largest value at the stored pixels, per-channel sums within 1e-6 relative;
* gradients: within 5e-5 of the largest stored entry (+1e-6) at the stored entries; sums within 5e-5 of the
  reference's sum of absolute values plus 1e-6 per entry (fp32 accumulation over up to 1e5 entries).

These replace runs of the 50-iteration fits themselves (which need the reference's Python code): each recorded call is
checked on its own, on the scene the reference's fit had reached, and the fits' convergence is no longer checked.
"""
import os

import numpy as np
import pytest
from conftest import GOLDEN
from dropin.dropin_calls import GRADS, dense_image_b, load, resolve

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def recorded():
    return load(os.path.join(GOLDEN, "dropin_calls.npz"))


def _scene(call):
    from deodr_b200.differentiable_renderer import Scene2DBase

    fields = dict(call["scene"])
    for name in ("ij", "depths", "uv", "shade", "colors"):
        fields[name] = fields[name].astype(np.float64)
    for name in ("clockwise", "backface_culling", "strict_edge", "perspective_correct", "integer_pixel_centers"):
        fields[name] = bool(fields[name])
    scene = Scene2DBase(**fields)
    for name, like in (("uv_b", "uv"), ("ij_b", "ij"), ("shade_b", "shade"), ("colors_b", "colors"),
                       ("texture_b", "texture")):
        setattr(scene, name, np.zeros_like(getattr(scene, like)))
    return scene


def _close(got, ref, tol, what):
    err = np.abs(got - ref).max() if ref.size else 0.0
    assert err <= tol, f"{what}: max error {err} > {tol}"


def replay(case, build_native, recorded):
    from deodr_b200 import differentiable_renderer_cython as ffi

    manifest, arrays = recorded
    calls = manifest[case]
    assert calls
    image = z = err = None
    for n, raw in enumerate(calls):
        call = resolve(raw, arrays)
        scene, sigma, aa = _scene(call), call["sigma"], call["antialiase_error"]
        shape = tuple(call["image_shape"])
        what = f"{case} call {n} ({call['kind']})"
        if call["kind"] == "render":
            image, z = np.empty(shape), np.empty(shape[:2])
            err = np.empty(shape[:2]) if aa else None
            ffi.renderSceneCpp(scene, sigma, image, z, aa, call["obs"], err)
            px = call["pixels"]
            np.testing.assert_allclose(z.reshape(-1)[px], call["z_buffer"], rtol=1e-12, atol=0, err_msg=what)
            ref = call["image"].astype(np.float64)
            _close(image.reshape(-1, shape[2])[px], ref, 4e-6 * max(1.0, np.abs(ref).max()), what + " image")
            sums = image.reshape(-1, shape[2]).sum(0)
            np.testing.assert_allclose(sums, call["image_sum"], rtol=1e-6, atol=1e-9, err_msg=what)
            if aa:
                ref = call["err_buffer"].astype(np.float64)
                _close(err.reshape(-1)[px], ref, 4e-6 * max(1.0, np.abs(ref).max()), what + " err_buffer")
                assert abs(err.sum() - call["err_sum"]) <= 1e-6 * abs(call["err_sum"]) + 1e-9, what
        else:
            image_b = None if call["image_b_seed"] is None else dense_image_b(call["image_b_seed"], shape)
            ffi.renderSceneBCpp(scene, sigma, image.copy(), z.copy(), image_b, aa, call["obs"],
                                None if err is None else err.copy(), call["err_buffer_b"])
            for name in GRADS:
                g = np.asarray(getattr(scene, name)).reshape(-1)
                ref = call[name]["values"].astype(np.float64)
                scale = np.abs(ref).max() if ref.size else 0.0
                _close(g[call[name]["index"]], ref, 5e-5 * scale + 1e-6, f"{what} {name}")
                tol = 5e-5 * call[name]["abs_sum"] + 1e-6 * g.size
                assert abs(g.sum() - call[name]["sum"]) <= tol, f"{what} {name} sum"


def test_reference_convention_test_calls(build_native, recorded):
    """Every renderer call of the reference's tests/test_pixel_center_coordinates.py, test_texture_coordinates.py and
    test_render_mesh.py::test_render_mesh_triangle_soup."""
    replay("conventions", build_native, recorded)


@pytest.mark.parametrize("clockwise", [0, 1])
@pytest.mark.parametrize("antialiase_error", [0, 1])
def test_reference_soup_fitting_example(clockwise, antialiase_error, build_native, recorded):
    """deodr/examples/triangle_soup_fitting.py:run - the body of the reference's tests/test_triangle_soup_fitting.py
    (runs 1-4: both windings, with and without antialiase_error): its target render, the first two iterations and the
    last of 50."""
    replay(f"soup_cw{clockwise}_err{antialiase_error}", build_native, recorded)


@pytest.mark.parametrize("library", ["none", "pytorch"])
def test_reference_depth_hand_fitting_example(library, build_native, recorded):
    """deodr/examples/depth_image_hand_fitting.py:run with MeshDepthFitter (numpy) and its PyTorch twin - the body of
    the reference's tests/test_depth_image_hand_fitting.py: the first and the last of 50 iterations."""
    replay(f"hand_depth_{library}", build_native, recorded)


def test_reference_rgb_hand_fitting_example(build_native, recorded):
    """deodr/examples/rgb_image_hand_fitting.py:run: the first and the last of 50 iterations."""
    replay("hand_rgb_none", build_native, recorded)
