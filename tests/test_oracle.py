"""CPU: pins the oracle - the C restatement (oracle/deodr_oracle.c) and, where built, the compiled reference
(oracle/_ref) - against the reference's own known-answer vectors and the committed golden fixtures."""
import hashlib
import json
import os

import numpy as np
import pytest
from conftest import GOLDEN, SMALL_TAGS, load_small

from deodr_b200.scenes import dense_image_b, soup_scene, torus_scene
from oracle.oracle import Oracle

sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()  # noqa: E731


def test_soup_generator_reproduces_reference_scene_hashes(texture):
    """SHA-256 of the generated scene arrays, pinned by the reference tests/test_render_mesh.py:34-53."""
    np.random.seed(2)
    s = soup_scene(clockwise=True, texture=texture)
    assert sha(s.ij) == "56a498bf243bd514c9ab4a3bfd90f8105aa2c168023fa288dc39ad82e2d36a20"
    assert sha(s.depths) == "e25eed6310fef37e401aef594c4c95e1b3cccf962a3646976cf546c58ddfac0a"
    assert sha(s.uv) == "f436623445124ecff7139efa57cce21c2768e23727bac974e236ea33651cc7c9"
    assert sha(s.shade) == "4b796b925c4349245e52a3e6311e99d536dc71e8aa8dc43cbd67cbe35d48892f"
    assert sha(s.colors) == "76dbff728be3eb0860bd27adf493e935dbd81cd7232ec732ba30c4f73ea35c94"


@pytest.mark.parametrize("kind", ["port", "reference"])
def test_pinned_image_and_zbuffer_hashes(kind, texture, port_oracle, request):
    """Exact image / z-buffer SHA-256 of the reference tests/test_render_mesh.py:66-74 ("windows" LKG)."""
    oracle = port_oracle if kind == "port" else request.getfixturevalue("ref_oracle")
    np.random.seed(2)
    s = soup_scene(clockwise=True, texture=texture)
    image, z = oracle.render(s, 1.0)
    assert sha(image) == "4de52cc3e902f92ff64324b261ddc45cd6d148ec7e670cf2942532d515af62d8"
    assert sha(z) == "b6f87e03c60bd820efa09d0536495b25d5852f67ecbecd2622f8bf1910d6052a"
    g = np.load(os.path.join(GOLDEN, "soup_pinned.npz"))
    assert str(g["image_sha"]) == sha(image) and str(g["z_sha"]) == sha(z)
    grads = oracle.render_b(s, 1.0, image, z, dense_image_b(image))
    for name in ("ij_b", "colors_b", "uv_b", "shade_b"):
        assert np.array_equal(grads[name], g[name]), name
    assert np.array_equal(grads["texture_b"].astype(np.float32), g["texture_b_last_writer"])


@pytest.mark.parametrize("clockwise,key", [(False, "ccw"), (True, "cw")])
def test_soup_fitting_hashes(clockwise, key, texture, port_oracle):
    """Image hashes at iterations 0 and 1 of the reference tests/test_triangle_soup_fitting.py (lines 29-35, 73-79):
    hash[1] depends on ij_b of iteration 0, so it pins the position gradient bit-exactly."""
    pinned = {"ccw": ("38b6f6954374230aeb1ce5d804308522f6b4c58a6736a040aeef7f2176a20b28",
                      "0434ea722edb9e3364da9b0e8564c3002b9aa3b12791ba8f089689beecd3c4e9"),
              "cw": ("eb9f335a", "6b4cc11e")}[key]
    golden = json.load(open(os.path.join(GOLDEN, "soup_fitting.json")))[key]
    np.random.seed(2)
    gt = soup_scene(clockwise=clockwise, texture=texture)
    target, _ = port_oracle.render(gt, 1.0)
    assert sha(target) == golden["target_sha"]
    n = len(gt.depths)
    gt.ij = gt.ij + np.random.randn(n, 2) * 10
    # examples/triangle_soup_fitting.py:133-135: uv displaced by 0 and clipped to the texture extent
    gt.uv = np.minimum(np.maximum(gt.uv, 0), np.array(gt.texture.shape[:2]) - 1)
    speed = np.zeros((n, 2))
    for it in range(3):
        image, z = port_oracle.render(gt, 1.0)
        diff = image - target
        assert sha(image) == golden["hashes"][it]
        if it < 2:
            assert sha(image).startswith(pinned[it])
        assert float(np.sum(diff**2)) == golden["losses"][it]
        grads = port_oracle.render_b(gt, 1.0, image, z, 2 * diff)
        speed = 0.80 * speed - grads["ij_b"] * 0.01
        gt.ij = gt.ij + speed


@pytest.mark.parametrize("tag", SMALL_TAGS)
def test_port_matches_golden_small(tag, port_oracle):
    scene, d = load_small(tag)
    image, z = port_oracle.render(scene, float(d["sigma"]))
    assert np.array_equal(image, d["image"]) and np.array_equal(z, d["z"])
    if "ij_b" in d:
        g = Oracle("port", texfix=True).render_b(scene, float(d["sigma"]), image, z, dense_image_b(image))
        for name in ("ij_b", "colors_b", "uv_b", "shade_b"):
            assert np.array_equal(g[name], d[name]), name
        assert np.array_equal(g["texture_b"].astype(np.float32), d["texture_b"])


def test_port_bit_identical_to_compiled_reference(texture, port_oracle, ref_oracle):
    """Restatement vs the real thing on seeded scenes with every flag combination (forward and adjoint)."""
    for seed in (3, 11):
        for cw in (False, True):
            np.random.seed(seed)
            s = soup_scene(n_tri=20, width=96, height=80, clockwise=cw, texture=texture, min_det=300)
            for strict in (True, False):
                for halfpix in (True, False):
                    s.strict_edge, s.integer_pixel_centers = strict, not halfpix
                    for sigma in (0.0, 1.0, 2.7):
                        a, za = ref_oracle.render(s, sigma)
                        b, zb = port_oracle.render(s, sigma)
                        assert np.array_equal(a, b) and np.array_equal(za, zb)
                        ib = dense_image_b(a)
                        ga = ref_oracle.render_b(s, sigma, a, za, ib)
                        gb = port_oracle.render_b(s, sigma, b, zb, ib)
                        for name in ga:
                            assert np.array_equal(ga[name], gb[name]), (name, seed, cw, strict, halfpix, sigma)
    s = torus_scene(20, 128, 96, textured=True, texture_size=32)
    a, za = ref_oracle.render(s, 1.0)
    b, zb = port_oracle.render(s, 1.0)
    assert np.array_equal(a, b) and np.array_equal(za, zb)


def test_soup_fitting_hashes_antialiase_error_mode(texture, port_oracle):
    """The reference's pinned run with antialiase_error=True (tests/test_triangle_soup_fitting.py:48-60: image hashes of
    iterations 0 and 1, the second depends on the error-mode ij_b of the first), reproduced by the restatement through
    the loop of examples/triangle_soup_fitting.py:145-175 / Scene2D.render_compare_and_backward (:701-734)."""
    pinned = ("82a7b73fde3615ef7c70008965f4bfda8610b9001c20dd435a880bf45a31d3d6",
              "0de2e8b80730cfc444d0552cd81e5071897a525ec6495e643ca17fb0792496c0")
    np.random.seed(2)
    gt = soup_scene(clockwise=False, texture=texture)
    target, _ = port_oracle.render(gt, 1.0)
    n = len(gt.depths)
    gt.ij = gt.ij + np.random.randn(n, 2) * 10
    gt.uv = np.minimum(np.maximum(gt.uv, 0), np.array(gt.texture.shape[:2]) - 1)
    speed = np.zeros((n, 2))
    mask = np.ones(target.shape[:2])
    for it in range(2):
        image, z, err = port_oracle.render(gt, 1.0, antialiase_error=True, obs=target)
        assert sha(image) == pinned[it]
        grads = port_oracle.render_b(gt, 1.0, image, z, None, antialiase_error=True, obs=target, err_buffer=err * mask,
                                     err_buffer_b=mask.copy())
        speed = 0.80 * speed - grads["ij_b"] * 0.01
        gt.ij = gt.ij + speed


def test_port_bit_identical_to_compiled_reference_antialiase_error_mode(texture, port_oracle, ref_oracle):
    """antialiase_error=True (DR.h:2066-2618, 2824-2837, 3054-3060): the silhouette edges overdraw the squared residual
    against `obs` instead of the colours.  Forward: image, z-buffer and err_buffer bit-identical; adjoint: all five
    gradients bit-identical, including the reference's dropped row adjoint of the interpolated edges (defect #2 of
    SURVEY.md section 0, restated on purpose)."""
    rng = np.random.default_rng(5)
    for seed in (3, 11):
        for cw in (False, True):
            np.random.seed(seed)
            s = soup_scene(n_tri=20, width=96, height=80, clockwise=cw, texture=texture, min_det=300)
            obs = rng.random((s.height, s.width, 3))
            for strict, halfpix in ((True, True), (False, False), (True, False)):
                s.strict_edge, s.integer_pixel_centers = strict, not halfpix
                for sigma in (0.0, 1.0, 2.7):
                    a, za, ea = ref_oracle.render(s, sigma, antialiase_error=True, obs=obs)
                    b, zb, eb = port_oracle.render(s, sigma, antialiase_error=True, obs=obs)
                    assert np.array_equal(a, b) and np.array_equal(za, zb) and np.array_equal(ea, eb)
                    assert ea.min() >= 0 and np.isfinite(ea).all()
                    err_b = rng.random((s.height, s.width)) * 2 - 1
                    ga = ref_oracle.render_b(s, sigma, a, za, None, antialiase_error=True, obs=obs, err_buffer=ea,
                                             err_buffer_b=err_b)
                    gb = port_oracle.render_b(s, sigma, b, zb, None, antialiase_error=True, obs=obs, err_buffer=eb,
                                              err_buffer_b=err_b)
                    for name in ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b"):
                        assert np.array_equal(ga[name], gb[name]), (name, seed, cw, strict, halfpix, sigma)
                    assert np.abs(ga["ij_b"]).max() > 0
    # perspective-correct forward (the adjoint is not defined there)
    s.perspective_correct = True
    a, za, ea = ref_oracle.render(s, 1.0, antialiase_error=True, obs=obs)
    b, zb, eb = port_oracle.render(s, 1.0, antialiase_error=True, obs=obs)
    assert np.array_equal(a, b) and np.array_equal(za, zb) and np.array_equal(ea, eb)


def test_oracle_error_paths(texture, port_oracle):
    np.random.seed(2)
    s = soup_scene(texture=texture)
    image, z = port_oracle.render(s, 1.0)
    s.backface_culling = False
    with pytest.raises(RuntimeError, match="backface_culling"):
        port_oracle.render_b(s, 1.0, image, z, image)
    s.backface_culling, s.perspective_correct = True, True
    with pytest.raises(RuntimeError, match="perspective_correct"):
        port_oracle.render_b(s, 1.0, image, z, image)
    s.perspective_correct = False
    s.faces = s.faces.copy()
    s.faces[0, 0] = 10**6
    with pytest.raises(RuntimeError, match="faces"):
        port_oracle.render(s, 1.0)
