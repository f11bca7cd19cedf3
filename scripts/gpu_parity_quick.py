"""Quick GPU parity sweep (development aid): device path and host path vs the CPU oracle on a few seeded scenes."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deodr_b200.renderer import DeviceScene, Renderer  # noqa: E402
from deodr_b200.scenes import dense_image_b, soup_scene, torus_scene  # noqa: E402
from oracle.oracle import Oracle, available  # noqa: E402

tex = np.load(os.path.join(ROOT, "tests/golden/trefle_texture_u8.npy")).astype(np.float64) / 255
oracle = Oracle("reference", texfix=True) if available("reference", True) else Oracle("port", texfix=True)
print("oracle:", oracle.kind)
renderer = Renderer(0)


def cmp(scene, sigma, tag):
    t0 = time.time()
    i1, z1 = oracle.render(scene, sigma)
    t_cpu = time.time() - t0
    ds = DeviceScene(scene, "cuda:0")
    fwd = renderer.render(ds, sigma, face_id=True)
    torch.cuda.synchronize()
    z = fwd["z_buffer"].cpu().numpy()
    img = fwd["image"].cpu().numpy()
    zok = np.array_equal(z1, z)
    print(f"{tag}: z exact={zok} img maxdiff={np.abs(i1 - img).max():.2e} cpu_fwd={t_cpu*1e3:.1f}ms", flush=True)
    if not zok:
        bad = np.argwhere(z1 != z)
        print("   bad z px", len(bad), bad[:5])
    if scene.backface_culling and not scene.perspective_correct:
        ib = dense_image_b(i1)
        g1 = oracle.render_b(scene, sigma, i1, z1, ib)
        g2 = renderer.render_b(ds, sigma, fwd, torch.from_numpy(ib).cuda())
        torch.cuda.synchronize()
        msg = "   "
        for k in ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b"):
            a, b = g1[k], g2[k].cpu().numpy()
            d = np.abs(a - b).max() if a.size else 0
            m = np.abs(a).max() if a.size else 0
            msg += f" {k}: {d:.2e}/{m:.2e}"
        print(msg, flush=True)


np.random.seed(2)
sc = soup_scene(clockwise=True, texture=tex)
cmp(sc, 1.0, "soup cw")
cmp(sc, 0.0, "soup cw s0")
sc.strict_edge = False
cmp(sc, 2.5, "nonstrict s2.5")
sc.integer_pixel_centers = False
cmp(sc, 1.0, "halfpix")
sc.perspective_correct = True
cmp(sc, 1.0, "persp")
sc.perspective_correct = False
sc.backface_culling = False
cmp(sc, 1.0, "nocull")
cmp(torus_scene(24, 160, 120), 1.0, "torus24")
cmp(torus_scene(40, 250, 200, textured=True, texture_size=64), 1.0, "torus40 tex")
cmp(torus_scene(158, 1024, 1024, textured=True, texture_size=512), 1.0, "torus158 tex 1024 (c3)")
cmp(torus_scene(100, 512, 512, nb_colors=1), 1.0, "torus100 depth C=1")

# host path (reference-shaped API)
from deodr_b200.differentiable_renderer import Scene2D  # noqa: E402

np.random.seed(2)
s0 = soup_scene(clockwise=True, texture=tex)
s2 = Scene2D(**{k: getattr(s0, k) for k in ("faces", "faces_uv", "ij", "depths", "textured", "uv", "shade", "colors",
                                            "shaded", "edgeflags", "height", "width", "nb_colors", "texture",
                                            "background_image", "background_color", "clockwise")},
             backface_culling=True)
img, z = s2.render(1.0)
i1, z1 = oracle.render(s0, 1.0)
print("host path: z exact", np.array_equal(z, z1), "img", np.abs(img - i1).max())
obs = np.random.default_rng(1).random(img.shape)
img, z, eb, err = s2.render_compare_and_backward(obs, sigma=1.0)
g1 = oracle.render_b(s0, 1.0, i1, z1, 2 * (i1 - obs))
print("host bwd: ij_b", np.abs(s2.ij_b - g1["ij_b"]).max(), "/", np.abs(g1["ij_b"]).max(), " uv_b",
      np.abs(s2.uv_b - g1["uv_b"]).max(), "err", err)
print("launches", renderer.launches)
