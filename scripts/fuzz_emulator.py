"""Development aid (CPU only): random scenes through the CPU emulation of the kernel phases (tests/emul, the same
__host__ __device__ code the CUDA kernels run) against the reference core compiled from /root/reference (oracle/_ref).

    python scripts/fuzz_emulator.py [seed] [seconds] [scene]     # scene: replay that one scene only and report it

Checks per scene: z-buffer BIT-EXACT; image error <= 6e-5 * max(1, largest |channel| of the pixel, largest |interpolation weight| of its owner) (fp32 colours: the error is relative - at
non-strict boundary pixels of sliver triangles the interpolation extrapolates to values of several hundred - and grows
by half an ulp per stacked silhouette blend); gradients within 2e-4 * max|grad| in generic position.  Two measure-zero
situations are generated on purpose and reported separately instead of failing: texture coordinates exactly on the
texel grid (the bilinear sampler's gradient is discontinuous there, so a 1e-13 difference in u flips the texel) and
vertices snapped to half pixels (pixel centres exactly ON a silhouette edge: T = 0, the un-blend divides by it);
exact z ties between textured triangles are the documented deviation of INTEGRATION.md section 5; scenes with a VISIBLE
SLIVER (barycentric weights above 64 at some pixel, i.e. a triangle thinner than ~1/64 pixel) are also set apart: its
gradient is a sum of fp32 terms hundreds of times larger than the result (observed: up to 1e-3 relative).
Round 1: over 2 million scenes over twenty seeds (1-7 colour channels, background colour / image, triangles from 0.3 to
25 pixels, crowded soups, all flag combinations, one scene in five in antialiase_error mode): no z-buffer mismatch, no
deviation outside these tolerances.  Round 2 adds, per scene, a random choice of who takes the adjoint of the small
triangles (TriBins::small_textured on / off, triangle-parallel / record-parallel kernel).
End of round 2, at the final sources: 15.5 million scenes of the default campaign over ten seeds, 0.9 million on
canvases up to 270 x 270 (DEODR_FUZZ_SCALE=3), 3.7 million with the exact-wrap build and vertices up to 1e9 px away
(DEODR_FUZZ_EXACT_WRAP=1): no z-buffer mismatch, no gradient outside the tolerances; two far-vertex scenes under
perspective_correct at 3-4e-4 relative image error (fp32 attributes of triangles 1e9 px long).  What the campaigns did
find: a pixel owned by a visible sliver judged without its weight scale in error mode (criterion fixed), a first row
of 32768 in the exact-wrap build (fixed), and the reference itself corrupting its heap beyond its `short` range.
Scenes drawn with perspective_correct (one in four) check their adjoint through emul_render_b_depths against the port
oracle's perspective-correct adjoint (tests/perspective_support.py; the compiled reference has none), depths_b included,
under the same
gradient criterion: 417 thousand scenes over five seeds, 83,484 of them perspective-correct adjoints, no failure.
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle.oracle import Oracle  # noqa: E402
from perspective_support import PerspEmulator, PerspOracle  # noqa: E402

from deodr_b200.scenes import confetti_scene, dense_image_b, soup_scene, torus_scene  # noqa: E402

tex = np.load(os.path.join(ROOT, "tests/golden/trefle_texture_u8.npy")).astype(np.float64) / 255
# DEODR_FUZZ_EXACT_WRAP=1: the emulation built with DEODR_EXACT_SHORT_WRAP=1 (rmath.h), and one scene in three gets a few
# vertices pushed 4e4 .. 1e9 pixels away (beyond the reference's `short` range: only that build follows the reference there)
EXACT_WRAP = os.environ.get("DEODR_FUZZ_EXACT_WRAP", "0") == "1"
ora = Oracle("reference", texfix=True)
emu = PerspEmulator(exact_short_wrap=EXACT_WRAP)  # the emulation, with emul_render_b_depths
port = PerspOracle(texfix=True)  # the perspective-correct adjoint (render_b_depths)
rng_far = np.random.default_rng(12345 + (int(sys.argv[1]) if len(sys.argv) > 1 else 0))
rng = np.random.default_rng(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
limit = float(sys.argv[2]) if len(sys.argv) > 2 else 300.0
only = int(sys.argv[3]) if len(sys.argv) > 3 else 0  # replay: generate every scene (same random stream), render one
# DEODR_FUZZ_SCALE=3: canvases up to 270 x 270 (17 x 17 tiles: more tiles per triangle, longer per-tile lists, more
# triangles and edges per scene); the default keeps the scenes of the earlier campaigns (same random streams)
SCALE = float(os.environ.get("DEODR_FUZZ_SCALE", "1"))
t0, n, bad, special, n_persp_b = time.time(), 0, 0, 0, 0
worst = {"image": 0.0, "grad": 0.0}
while time.time() - t0 < limit and (only == 0 or n < only):
    kind = int(rng.integers(0, 4))
    W, H = int(rng.integers(5, int(90 * SCALE))), int(rng.integers(5, int(90 * SCALE)))
    degenerate = False
    if kind == 0:
        np.random.seed(int(rng.integers(0, 1 << 30)))
        W, H = max(W, 24), max(H, 24)
        # one soup in five is crowded: hundreds of silhouette edges per tile (several edge chunks, two-pass adjoint)
        n_soup = int(rng.integers(100, 300)) if rng.random() < 0.2 else int(rng.integers(1, 40))
        scene = soup_scene(n_tri=n_soup, width=W, height=H, clockwise=bool(rng.integers(0, 2)),
                           textured_ratio=float(rng.random()), texture=tex[::4, ::4].copy(),
                           min_det=float(rng.choice([0.005, 0.02, 0.05])) * W * H)
    elif kind == 1:
        scene = confetti_scene(int(rng.integers(1, int(1500 * SCALE * SCALE))), W, H, size=float(rng.choice([0.3, 1.0, 2.5, 6.0, 25.0])),
                               seed=int(rng.integers(0, 1 << 30)), edge_ratio=float(rng.choice([0, 0.05, 0.5, 1.0])),
                               nb_colors=int(rng.choice([1, 2, 3, 4, 7])))
        if rng.random() < 0.3:  # a background image instead of a colour
            scene.background_image = rng.random((H, W, scene.nb_colors))
            scene.background_color = None
    elif kind == 2:
        scene = torus_scene(int(rng.integers(4, int(30 * SCALE))), max(W, 16), max(H, 16), textured=bool(rng.integers(0, 2)),
                            nb_colors=3, texture_size=16)
        if rng.random() < 0.7:
            scene.uv = scene.uv * 0.9973 + 0.0131  # off the texel grid (generic position)
        else:
            degenerate = bool(scene.textured.any())
    else:
        scene = confetti_scene(int(rng.integers(1, 300)), W, H, size=float(rng.choice([1.0, 20.0])),
                               seed=int(rng.integers(0, 1 << 30)), edge_ratio=0.3)
        if rng.random() < 0.5:  # vertices snapped to half pixels, far outside the image
            scene.ij = np.round(scene.ij * 2) / 2 + rng.choice([0, -30, 40], size=(1, 2))
            degenerate = True
    far_scene = False
    if EXACT_WRAP and rng_far.random() < 0.33:
        far_scene = True
        n_far = max(1, scene.ij.shape[0] // 15)
        idx = rng_far.choice(scene.ij.shape[0], size=n_far, replace=False)
        far = float(rng_far.choice([4e4, 7e4, 1e6, 1e9]))
        scene.ij = scene.ij.copy()
        scene.ij[idx] += rng_far.choice([-1, 1], size=(n_far, 2)) * far * rng_far.random((n_far, 2))
        # A vertex whose row wraps to exactly 32767 makes the reference start its `short` row counter at
        # (short)(32767 + 1) = -32768 and WRITE at negative pixel indices (DR.h:925-960: heap corruption that killed a
        # campaign after 40 000 scenes).  The exact-wrap build gives the same picture without the stray writes
        # (replayed: scene 9501/10377); the campaign keeps clear of it so that the reference survives.
        for off in (0.0, 0.5):
            rows = np.floor(scene.ij[:, 1] - off)
            hit = np.isfinite(rows) & (np.abs(rows) < 2.0 ** 31) & ((rows.astype(np.int64) & 0xffff) == 32767)
            scene.ij[hit, 1] += 1.0
        degenerate = True  # gradients of triangles thousands of pixels long: fp32 attribute planes (reported apart)
    scene.strict_edge = bool(rng.integers(0, 2))
    scene.integer_pixel_centers = bool(rng.integers(0, 2))
    scene.backface_culling = bool(rng.random() < 0.8)
    scene.perspective_correct = bool(rng.random() < 0.25)
    sigma = float(rng.choice([0.0, 0.5, 1.0, 2.5]))
    # round 2: who takes the adjoint of a small triangle (both device paths: textured ones triangle- or pixel-parallel;
    # the triangle-parallel kernel or the record-parallel one)
    small_textured, small_records = bool(rng.integers(0, 2)), bool(rng.random() < 0.3)
    n += 1
    error_mode = rng.random() < 0.2 and not scene.perspective_correct and scene.backface_culling
    if error_mode:
        obs = rng.random((scene.height, scene.width, scene.nb_colors)).astype(np.float32).astype(np.float64)
        err_b = rng.random((scene.height, scene.width)) * 2 - 1
    if only and n != only:
        continue
    emu.set_small_textured(small_textured)
    emu.set_small_records(small_records)
    if only:
        print("replaying scene", n, "kind", kind, (W, H), "T", scene.faces.shape[0], "sigma", sigma, "error mode", error_mode,
              "degenerate", degenerate, flush=True)
        np.savez(os.path.join(ROOT, "gpurun_out", f"fuzz_scene_{n}.npz"), **{k: v for k, v in vars(scene).items() if v is not None},
                 sigma=sigma, **({"obs": obs, "err_b": err_b} if error_mode else {}))
    if error_mode:
        # antialiase_error mode (row f3): phases emulated on the CPU, reference defect #2 kept
        image, z, err = ora.render(scene, sigma, antialiase_error=True, obs=obs)
        fwd = emu.render_error(scene, sigma, obs)
        sliver = emu.render(scene, sigma)["weight_scale"]
        if sliver.size and sliver.max() > 64:
            degenerate = True
        fwd = emu.render_error(scene, sigma, obs)  # (the emulator keeps the state of its last forward)
        msg = "" if np.array_equal(fwd["z"], z) else " Z-BUFFER-MISMATCH"
        # (per pixel relative to the interpolation weights of its owner, like the image criterion below: the residual of
        # a pixel owned by a visible sliver - weights in the thousands - carries the fp32 error of that interpolation)
        w_px = np.maximum(1.0, sliver) if sliver.size else 1.0
        e_err = (np.abs(fwd["err"] - err) / w_px).max() / max(1.0, float(np.abs(err).max())) if err.size else 0.0
        if e_err > 6e-5:
            msg += f" err_buffer {e_err:.2e}"
        ref = ora.render_b(scene, sigma, image, z, None, antialiase_error=True, obs=obs, err_buffer=err, err_buffer_b=err_b)
        got = emu.render_error_b(scene, sigma, fwd, err_b, compat=True)
        for name in ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b"):
            if ref[name].size == 0:
                continue
            m, d = np.abs(ref[name]).max(), np.abs(got[name] - ref[name]).max()
            if d > 2e-4 * m + 1e-5:
                if degenerate or (emu.lib.emul_num_ties() > 0 and scene.textured.any()):
                    special += 1
                    break
                msg += f" (error mode) {name} {d:.2e}/{m:.2e}"
        if msg:
            bad += 1
            print("FAIL scene", n, "kind", kind, (W, H), "T", scene.faces.shape[0], "sigma", sigma, "error mode", msg, flush=True)
        continue
    image, z = ora.render(scene, sigma)
    fwd = emu.render(scene, sigma)
    if fwd["ties"] > 0 and scene.textured.any():
        degenerate = True  # exact z ties between textured triangles: documented deviation (INTEGRATION.md section 5)
    if fwd["weight_scale"].size and fwd["weight_scale"].max() > 64:
        degenerate = True  # a visible sliver (barycentric weights > 64): its fp32 gradient terms cancel
    msg = ""
    if not np.array_equal(fwd["z"], z):
        msg += " Z-BUFFER-MISMATCH"
    # scale of a pixel = its largest channel (a small channel next to large ones is a cancellation of the same weights)
    scale = np.maximum(1.0, np.abs(image).max(axis=2, keepdims=True)) if image.size else 1.0
    if image.size:  # ... or of the interpolation weights themselves (edge-on triangles under perspective_correct)
        scale = np.maximum(scale, fwd["weight_scale"][:, :, None])
    err = (np.abs(fwd["image"] - image) / scale).max() if image.size else 0.0
    worst["image"] = max(worst["image"], err)
    # (triangles thousands of pixels long: the fp32 attribute planes are formed from coordinates up to 1e9;
    # observed up to 7.3e-5 over 30 000 such scenes)
    if err > (2.5e-4 if far_scene else 6e-5):
        msg += f" image {err:.2e}"
    if scene.backface_culling:
        image_b = dense_image_b(image)
        names = ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b")
        if scene.perspective_correct:
            n_persp_b += 1
            ref = port.render_b_depths(scene, sigma, image, z, image_b)
            got = emu.render_b_depths(scene, sigma, fwd, image_b)
            names += ("depths_b",)
        else:
            ref = ora.render_b(scene, sigma, image, z, image_b)
            got = emu.render_b(scene, sigma, fwd, image_b)
        for name in names:
            if ref[name].size == 0:
                continue
            m, d = np.abs(ref[name]).max(), np.abs(got[name] - ref[name]).max()
            if m > 1e-3 and not degenerate:
                worst["grad"] = max(worst["grad"], d / m)
            if d > 2e-4 * m + 1e-5:
                if degenerate:
                    special += 1
                    break
                msg += f" {name} {d:.2e}/{m:.2e}"
    if msg:
        bad += 1
        print("FAIL scene", n, "kind", kind, (W, H), "T", scene.faces.shape[0], "sigma", sigma, "strict", scene.strict_edge,
              "half-pixel centres", not scene.integer_pixel_centers, "cull", scene.backface_culling, "persp",
              scene.perspective_correct, msg, flush=True)
print(f"{n} scenes ({n_persp_b} perspective-correct adjoints), {bad} failures, {special} measure-zero cases outside the "
      f"generic tolerance; worst relative image error {worst['image']:.2e}, worst relative gradient error (generic "
      f"position) {worst['grad']:.2e}")
