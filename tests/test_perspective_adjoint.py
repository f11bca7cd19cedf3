"""CPU: the perspective-correct adjoint (deodr_b200_render_b_views_depths) and its gradient of the vertex depths.

1. The perspective-correct adjoint of the port oracle (tests/perspective/persp_oracle.c) against central finite
   differences of the REFERENCE's forward pass.
2. The emulated kernel phases (emul_render_b_depths) against that oracle, with the gradient criterion of the GPU parity
   tests.
3. Scenes without perspective_correct through the new emulated entry: the gradients of emul_render_b, depths_b zero.

Every scene gets per-vertex depth variation (soups and confetti draw one depth per triangle), or perspective-correct
interpolation would be the affine one.
"""
import numpy as np
import pytest
from perspective_support import PerspEmulator, PerspOracle
from test_gpu_parity import assert_gradient_close

from deodr_b200.scenes import confetti_scene, dense_image_b, soup_scene, torus_scene

GRADS = ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b")


def perspective(scene, seed=0):
    """Per-vertex depth variation (depth * (1 + 0.6 rand)) and perspective_correct on."""
    rng = np.random.default_rng(seed)
    scene.depths = np.asarray(scene.depths, dtype=np.float64) * (1 + 0.6 * rng.random(scene.depths.shape))
    scene.perspective_correct = True
    return scene


@pytest.fixture(scope="module")
def port_texfix(build_native):
    return PerspOracle(texfix=True)


@pytest.fixture(scope="module")
def emulator():
    return PerspEmulator()


# ------------------------------------------------------------------------------------------ 1. finite differences

def finite_difference_check(ref_oracle, port, scene, sigma, samples=10, seed=0):
    image, z = ref_oracle.render(scene, sigma)
    weights = np.random.default_rng(seed).random(image.shape)
    got = port.render_b_depths(scene, sigma, image, z, weights)
    rng = np.random.default_rng(seed + 1)

    def loss():
        return float(np.sum(ref_oracle.render(scene, sigma)[0] * weights))

    for name in ("ij", "depths", "colors", "uv", "shade", "texture"):
        if name in ("uv", "shade", "texture") and not np.any(scene.textured):
            continue
        base = np.asarray(getattr(scene, name), dtype=np.float64).copy()
        grad = got[name + "_b"]
        flat = grad.ravel()
        # the largest gradients and a few random entries
        idx = np.unique(np.concatenate([np.argsort(-np.abs(flat))[:samples], rng.integers(0, flat.size, samples)]))
        worst = 0.0
        for i in idx:
            x0 = base.ravel()[i]
            eps = 1e-6 * abs(x0) if name == "depths" else 1e-6  # relative step on the depths
            hi, lo = base.copy(), base.copy()
            hi.ravel()[i] += eps
            lo.ravel()[i] -= eps
            setattr(scene, name, hi)
            f_hi = loss()
            setattr(scene, name, lo)
            f_lo = loss()
            worst = max(worst, abs((f_hi - f_lo) / (2 * eps) - flat[i]))
        setattr(scene, name, base)
        assert worst <= 2e-3 * np.abs(grad).max() + 1e-4, (name, worst, np.abs(grad).max())
    return got


@pytest.mark.parametrize("sigma", [0.0, 1.0, 2.5])
@pytest.mark.parametrize("textured_ratio", [0.0, 0.5])
@pytest.mark.parametrize("clockwise", [False, True])
def test_oracle_matches_finite_differences_soup(sigma, textured_ratio, clockwise, ref_oracle, port_texfix, texture):
    np.random.seed(7)
    scene = soup_scene(n_tri=10, width=64, height=64, clockwise=clockwise, textured_ratio=textured_ratio,
                       texture=texture[::4, ::4].copy(), min_det=200)
    got = finite_difference_check(ref_oracle, port_texfix, perspective(scene), sigma)
    assert np.abs(got["depths_b"]).max() > 0


def test_oracle_matches_finite_differences_torus(ref_oracle, port_texfix):
    scene = torus_scene(10, 60, 50)
    scene.perspective_correct = True
    got = finite_difference_check(ref_oracle, port_texfix, scene, 1.0)
    assert np.abs(got["depths_b"]).max() > 0


def test_old_oracle_entry_still_refuses_perspective(port_oracle, texture):
    """deodr_oracle_render_b keeps refusing perspective scenes."""
    np.random.seed(7)
    scene = perspective(soup_scene(n_tri=5, width=64, height=64, texture=texture[::4, ::4].copy(), min_det=200))
    image, z = port_oracle.render(scene, 1.0)
    with pytest.raises(RuntimeError, match="perspective_correct"):
        port_oracle.render_b(scene, 1.0, image, z, dense_image_b(image))


# ------------------------------------------------------------------------------- 2. emulated phases vs the oracle

def emulator_check(emulator, port, scene, sigma):
    image, z = port.render(scene, sigma)
    fwd = emulator.render(scene, sigma)
    assert np.array_equal(fwd["z"], z), "z-buffer not bit-exact"
    image_b = dense_image_b(image)
    ref = port.render_b_depths(scene, sigma, image, z, image_b)
    got = emulator.render_b_depths(scene, sigma, fwd, image_b)
    for name in GRADS + ("depths_b",):
        if ref[name].size:
            assert_gradient_close(got[name], ref[name], name)
    assert np.abs(ref["depths_b"]).max() > 0
    return got


@pytest.mark.parametrize("small_records", [False, True])
@pytest.mark.parametrize("strict_edge", [True, False])
@pytest.mark.parametrize("integer_pixel_centers", [True, False])
def test_emulated_phases_match_oracle_soup(small_records, strict_edge, integer_pixel_centers, emulator, port_texfix,
                                           texture):
    emulator.set_small_records(small_records)
    try:
        np.random.seed(3)
        scene = perspective(soup_scene(n_tri=30, width=120, height=100, textured_ratio=0.5, texture=texture,
                                       min_det=300))
        scene.strict_edge, scene.integer_pixel_centers = strict_edge, integer_pixel_centers
        emulator_check(emulator, port_texfix, scene, 1.0)
    finally:
        emulator.set_small_records(False)


@pytest.mark.parametrize("small_records", [False, True])
def test_emulated_phases_match_oracle_confetti(small_records, emulator, port_texfix):
    """micro triangles: the small-triangle adjoint (record-parallel requests take the triangle-parallel form)"""
    emulator.set_small_records(small_records)
    try:
        emulator_check(emulator, port_texfix, perspective(confetti_scene(3000, 64, 48, size=2.5, seed=1)), 1.0)
        emulator_check(emulator, port_texfix,
                       perspective(confetti_scene(1500, 50, 40, size=1.2, seed=2, edge_ratio=0.3), seed=1), 0.7)
    finally:
        emulator.set_small_records(False)


@pytest.mark.parametrize("nb_colors", [1, 3, 4, 16])
def test_emulated_phases_match_oracle_channels(nb_colors, emulator, port_texfix):
    """channel instances 1, 3, 4 and 16; large triangles (interior path) and edge-heavy meshes"""
    scene = torus_scene(16, 90, 70, nb_colors=nb_colors)
    scene.perspective_correct = True
    emulator_check(emulator, port_texfix, scene, 1.0)


def test_emulated_phases_match_oracle_textured_mesh(emulator, port_texfix):
    scene = torus_scene(30, 100, 90, textured=True, texture_size=32)
    scene.perspective_correct = True
    emulator_check(emulator, port_texfix, scene, 1.0)


def test_emulated_phases_match_oracle_many_edges_per_tile(emulator, port_texfix, texture):
    np.random.seed(11)
    scene = perspective(soup_scene(n_tri=120, width=64, height=64, textured_ratio=0.3, texture=texture[::4, ::4].copy(),
                                   min_det=60), seed=2)
    emulator_check(emulator, port_texfix, scene, 2.5)


# ---------------------------------------------------------------------- 3. non-perspective scenes, new entry point

@pytest.mark.parametrize("sigma", [0.0, 1.0])
def test_new_entry_without_perspective_is_render_b(sigma, emulator, texture):
    np.random.seed(3)
    scene = soup_scene(n_tri=30, width=120, height=100, textured_ratio=0.5, texture=texture, min_det=300)
    fwd = emulator.render(scene, sigma)
    image_b = dense_image_b(fwd["image"])
    ref = emulator.render_b(scene, sigma, fwd, image_b)
    got = emulator.render_b_depths(scene, sigma, fwd, image_b)
    for name in GRADS:
        assert np.array_equal(got[name], ref[name]), name
    assert not got["depths_b"].any()
