"""GPU: the perspective-correct adjoint (deodr_b200_render_b_views_depths) against the port oracle's own
perspective-correct adjoint (tests/perspective_support.py; the reference has none), with the gradient criterion of test_gpu_parity.  The forward is
the existing one: z-buffer bit-exact, image within 1e-6."""
import numpy as np
import pytest
from conftest import GOLDEN
from test_gpu_parity import IMAGE_TOL, assert_gradient_close

from deodr_b200.scenes import SceneArrays, confetti_scene, dense_image_b, soup_scene, torus_scene

pytestmark = pytest.mark.gpu

GRADS = ("ij_b", "depths_b", "colors_b", "uv_b", "shade_b", "texture_b")


def perspective(scene, seed=0):
    rng = np.random.default_rng(seed)
    scene.depths = np.asarray(scene.depths, dtype=np.float64) * (1 + 0.6 * rng.random(scene.depths.shape))
    scene.perspective_correct = True
    return scene


def persp_torus(*args, **kw):
    scene = torus_scene(*args, **kw)
    scene.perspective_correct = True
    return scene


@pytest.fixture(scope="module")
def gpu(build_native):
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from deodr_b200.renderer import Renderer

    return Renderer(0)


@pytest.fixture(scope="module")
def port(build_native):
    from perspective_support import PerspOracle

    return PerspOracle(texfix=True)


def device_check(gpu, port, scene, sigma):
    import torch

    from deodr_b200.renderer import DeviceScene

    image, z = port.render(scene, sigma)
    ds = DeviceScene(scene, "cuda:0")
    fwd = gpu.render(ds, sigma)
    assert np.array_equal(fwd["z_buffer"].cpu().numpy(), z), "z-buffer not bit-exact"
    assert np.abs(fwd["image"].cpu().numpy() - image).max() <= IMAGE_TOL
    image_b = dense_image_b(image)
    got = gpu.render_b(ds, sigma, fwd, torch.from_numpy(image_b.astype(np.float32)).cuda(), depths_b=True)
    ref = port.render_b_depths(scene, sigma, image, z, image_b)
    for name in GRADS:
        if ref[name].size:
            assert_gradient_close(got[name].cpu().numpy(), ref[name], name)
    assert np.abs(ref["depths_b"]).max() > 0
    return got


@pytest.mark.parametrize("sigma", [0.0, 1.0, 2.5])
@pytest.mark.parametrize("textured_ratio", [0.0, 0.5])
@pytest.mark.parametrize("clockwise", [False, True])
def test_soup_against_oracle(sigma, textured_ratio, clockwise, gpu, port, texture):
    np.random.seed(7)
    scene = soup_scene(n_tri=30, width=200, height=200, clockwise=clockwise, textured_ratio=textured_ratio,
                       texture=texture)
    device_check(gpu, port, perspective(scene), sigma)


def test_confetti_against_oracle(gpu, port):
    device_check(gpu, port, perspective(confetti_scene(3000, 64, 48, size=2.5, seed=1)), 1.0)


@pytest.mark.parametrize("nb_colors", [1, 3, 16])
def test_torus_against_oracle(nb_colors, gpu, port):
    device_check(gpu, port, persp_torus(24, 300, 300, nb_colors=nb_colors), 1.0)


def test_large_textured_torus_against_oracle(gpu, port):
    device_check(gpu, port, persp_torus(158, 1024, 1024, textured=True), 1.0)  # ~50k triangles


def test_record_parallel_request_takes_the_triangle_parallel_form(port, monkeypatch, build_native):
    """DEODR_B200_SMALL_ADJOINT=record: perspective views still get their small-triangle adjoint"""
    from deodr_b200.renderer import Renderer

    monkeypatch.setenv("DEODR_B200_SMALL_ADJOINT", "record")
    device_check(Renderer(0), port, perspective(confetti_scene(3000, 64, 48, size=2.5, seed=1)), 1.0)


def test_batch_of_views_with_shared_colors_b(gpu, port):
    import torch

    from deodr_b200.renderer import DeviceScene

    n = 8
    scenes = [persp_torus(316, 512, 512, view=i, n_views=n) for i in range(n)]
    dss = [DeviceScene(s, "cuda:0") for s in scenes]
    fwds = gpu.render_views(dss, 1.0)
    image_bs, grads, refs = [], [], []
    colors_b = torch.zeros(dss[0].t["colors"].shape, dtype=torch.float32, device="cuda:0")
    for s, ds, f in zip(scenes, dss, fwds):
        image, z = port.render(s, 1.0)
        assert np.array_equal(f["z_buffer"].cpu().numpy(), z)
        image_b = dense_image_b(image)
        image_bs.append(torch.from_numpy(image_b.astype(np.float32)).cuda())
        g = ds.zero_grads()
        g["colors_b"] = colors_b  # shared parameter: accumulated over the views
        grads.append(g)
        refs.append(port.render_b_depths(s, 1.0, image, z, image_b))
    gpu.render_b_views(dss, 1.0, fwds, image_bs, grads, depths_b=True)
    for g, r in zip(grads, refs):
        assert_gradient_close(g["ij_b"].cpu().numpy(), r["ij_b"], "ij_b")
        assert_gradient_close(g["depths_b"].cpu().numpy(), r["depths_b"], "depths_b")
    assert_gradient_close(colors_b.cpu().numpy(), sum(r["colors_b"] for r in refs), "colors_b")


def test_cuda_graph_capture(port):
    import torch

    from deodr_b200.renderer import DeviceScene, Renderer

    gpu = Renderer(0)
    scene = persp_torus(23, 320, 240)
    ds = DeviceScene(scene, "cuda:0")
    image, z = port.render(scene, 1.0)
    image_b = torch.from_numpy(dense_image_b(image).astype(np.float32)).cuda()
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        out = gpu.render(ds, 1.0)  # warm-up: builds the plan
        eager = gpu.render_b(ds, 1.0, out, image_b, depths_b=True)
        eager = {k: v.clone() for k, v in eager.items()}
        grads = ds.zero_grads()
        grads["depths_b"] = torch.zeros_like(eager["depths_b"])
        torch.cuda.synchronize()
        gpu.set_deferred(True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for g in grads.values():
                g.zero_()
            gpu.render(ds, 1.0, out=out)
            gpu.render_b(ds, 1.0, out, image_b, grads, depths_b=True)
        for _ in range(2):
            graph.replay()
            torch.cuda.synchronize()
            gpu.status()
            assert np.array_equal(out["z_buffer"].cpu().numpy(), z)
            for name in ("ij_b", "depths_b", "colors_b"):
                assert_gradient_close(grads[name].cpu().numpy(), eager[name].cpu().numpy(), name)
    gpu.set_deferred(False)


def test_non_perspective_scene_through_the_new_entry(gpu, texture):
    import torch

    from deodr_b200.renderer import DeviceScene

    np.random.seed(3)
    scene = soup_scene(n_tri=30, width=200, height=200, texture=texture)
    ds = DeviceScene(scene, "cuda:0")
    fwd = gpu.render(ds, 1.0)
    image_b = torch.from_numpy(dense_image_b(fwd["image"].cpu().numpy()).astype(np.float32)).cuda()
    ref = gpu.render_b(ds, 1.0, fwd, image_b)
    got = gpu.render_b(ds, 1.0, fwd, image_b, depths_b=True)
    for name in ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b"):
        assert_gradient_close(got[name].cpu().numpy(), ref[name].cpu().numpy(), name)
    assert not got["depths_b"].any()


def test_antialiase_error_with_perspective_is_unsupported(gpu, texture):
    import torch

    from deodr_b200 import _cabi
    from deodr_b200.renderer import DeviceScene

    np.random.seed(3)
    scene = perspective(soup_scene(n_tri=10, width=64, height=64, texture=texture[::4, ::4].copy(), min_det=200))
    ds = DeviceScene(scene, "cuda:0")
    obs = torch.rand((64, 64, 3), device="cuda:0")
    fwd = gpu.render(ds, 1.0, obs=obs)
    with pytest.raises(_cabi.DeodrB200Error) as e:
        gpu.render_b(ds, 1.0, fwd, err_buffer_b=torch.ones((64, 64), device="cuda:0"), depths_b=True)
    assert e.value.code == _cabi.EUNSUPPORTED
    assert "antialiase_error" in str(e.value) and "perspective_correct" in str(e.value)


def test_device_mesh_view_with_perspective(port, build_native):
    import os

    import torch

    from deodr_b200.mesh_ops import CameraParams, DeviceMeshView, project_points_backward, vertex_luminosity_backward

    gold = np.load(os.path.join(GOLDEN, "scene_ops.npz"))
    faces, vertices = gold["hand_faces"], gold["hand_vertices"]
    cam = CameraParams(gold["view_extrinsic"], gold["view_intrinsic"])
    light, ambient = gold["lum_light"], float(gold["lum_ambient"])
    view = DeviceMeshView(faces, vertices.shape[0], cam, 480, 640, light_directional=light, ambient=ambient,
                          background_color=(0.3, 0.5, 0.7), perspective_correct=True)
    vcol = gold["lum_vertex_colors"]
    v_t = torch.from_numpy(vertices).cuda()
    image = view.render(v_t, torch.from_numpy(vcol).cuda()).cpu().numpy()
    t = {k: (v.cpu().numpy() if v is not None else None) for k, v in view.scene.t.items()}
    T, V = faces.shape[0], vertices.shape[0]
    scene = SceneArrays(
        faces=faces, faces_uv=np.zeros((T, 3), np.uint32), ij=t["ij"], depths=t["depths"], textured=np.zeros(T, bool),
        uv=np.zeros((1, 2)), shade=np.zeros(V), colors=t["colors"].astype(np.float64), shaded=np.zeros(T, bool),
        edgeflags=t["edgeflags"].astype(bool), height=480, width=640, nb_colors=3, texture=np.zeros((2, 2, 3)),
        background_image=None, background_color=np.array([0.3, 0.5, 0.7]), clockwise=False, backface_culling=True,
        strict_edge=True, perspective_correct=True, integer_pixel_centers=True)
    image_ref, z_ref = port.render(scene, 1.0)
    assert np.isfinite(z_ref).mean() > 0.05
    assert np.abs(image - image_ref).max() < 2e-6
    image_b = dense_image_b(image_ref)
    g_ref = port.render_b_depths(scene, 1.0, image_ref, z_ref, image_b)
    got = view.backward(torch.from_numpy(image_b).cuda())
    # the same composition from the oracle's raster gradients
    _, _, normals, _ = view._saved
    lum = vertex_luminosity_backward(normals, torch.from_numpy(vcol).cuda(), light, ambient,
                                     colors_b=torch.from_numpy(g_ref["colors_b"].astype(np.float32)).cuda())
    base = view.topology.vertex_normals_backward(v_t, lum["normals_b"])
    with_depths = project_points_backward(v_t, cam, torch.from_numpy(g_ref["ij_b"]).cuda(),
                                          depths_b=torch.from_numpy(g_ref["depths_b"]).cuda(), out=base.clone())
    without = project_points_backward(v_t, cam, torch.from_numpy(g_ref["ij_b"]).cuda(), out=base.clone())
    with_depths, without = with_depths.cpu().numpy(), without.cpu().numpy()
    vb = got["vertices_b"].cpu().numpy()
    tol = 1e-4 * np.abs(with_depths).max()
    assert np.abs(vb - with_depths).max() < tol
    assert np.abs(vb - without).max() > tol  # the depth path is wired


def test_autograd_with_depths(gpu, texture):
    import torch

    from deodr_b200.pytorch import CudaDifferentiableRender2D
    from deodr_b200.renderer import DeviceScene, default_renderer

    np.random.seed(3)
    scene = perspective(soup_scene(n_tri=30, width=200, height=200, textured_ratio=0.0, texture=texture))
    ds = DeviceScene(scene, "cuda:0")
    ij = torch.from_numpy(scene.ij).cuda().requires_grad_(True)
    col = torch.from_numpy(scene.colors).cuda().requires_grad_(True)
    depths = torch.from_numpy(scene.depths).cuda().requires_grad_(True)
    image = CudaDifferentiableRender2D(ij, col, ds, 1.0, depths)
    image_b = torch.from_numpy(dense_image_b(image.detach().cpu().numpy()).astype(np.float32)).cuda()
    (image * image_b).sum().backward()
    r = default_renderer(0)
    fwd = r.render(ds, 1.0)
    ref = r.render_b(ds, 1.0, fwd, image_b, depths_b=True)
    for got, name in ((ij.grad, "ij_b"), (col.grad, "colors_b"), (depths.grad, "depths_b")):
        assert_gradient_close(got.cpu().numpy(), ref[name].cpu().numpy().astype(np.float64), name)
    assert depths.grad.abs().max() > 0
