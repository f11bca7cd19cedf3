"""autograd surface of the 2D render, mirroring deodr/pytorch/differentiable_renderer_pytorch.py:41-81.

Two Functions with the reference contract ``(ij, colors, scene) -> image[H,W,C]``, backward ``(ij_b, colors_b, None)``:

* ``TorchDifferentiableRenderer2DFunc`` - signature-compatible with the reference class of the same name: ``scene`` is
  an object with a ``scene_2d`` attribute (``Scene3DPytorch`` in the reference), tensors are CPU float64, sigma is 1;
  data crosses to the GPU through the reference-shaped host entry points.
* ``CudaDifferentiableRenderer2DFunc`` - the zero-copy variant: ``scene`` is a ``deodr_b200.renderer.DeviceScene``,
  ``ij`` / ``colors`` are CUDA tensors, the image stays on the device.
"""

from __future__ import annotations

from typing import Any, Optional

import numpy as np
import torch

from .. import differentiable_renderer_cython
from ..renderer import DeviceScene, default_renderer


class TorchDifferentiableRenderer2DFunc(torch.autograd.Function):
    """CPU-tensor in / CPU-tensor out, same contract as the reference Function."""

    @staticmethod
    def forward(ctx: Any, ij: torch.Tensor, colors: torch.Tensor, scene: Any) -> torch.Tensor:  # type: ignore
        scene_2d = scene.scene_2d
        image = np.empty((scene_2d.height, scene_2d.width, colors.shape[1]))
        z_buffer = np.empty((scene_2d.height, scene_2d.width))
        ctx.scene = scene
        scene_2d.ij = ij.detach().numpy()
        scene.colors = colors.detach().numpy()
        differentiable_renderer_cython.renderSceneCpp(scene_2d, 1, image, z_buffer)
        ctx.save_for_backward(ij, colors)
        ctx.image = image.copy()
        ctx.z_buffer = z_buffer
        return torch.as_tensor(image)

    @staticmethod
    def backward(ctx: Any, *grad_outputs: Any) -> Any:
        assert len(grad_outputs) == 1
        image_b = np.ascontiguousarray(grad_outputs[0].detach().numpy(), dtype=np.float64)
        scene_2d = ctx.scene.scene_2d
        scene_2d.uv_b = np.zeros(scene_2d.uv.shape)
        scene_2d.ij_b = np.zeros(scene_2d.ij.shape)
        scene_2d.shade_b = np.zeros(scene_2d.shade.shape)
        scene_2d.colors_b = np.zeros(scene_2d.colors.shape)
        scene_2d.texture_b = np.zeros(scene_2d.texture.shape)
        differentiable_renderer_cython.renderSceneBCpp(scene_2d, 1, ctx.image, ctx.z_buffer, image_b)
        return torch.as_tensor(scene_2d.ij_b), torch.as_tensor(scene_2d.colors_b), None


TorchDifferentiableRender2D = TorchDifferentiableRenderer2DFunc.apply


class CudaDifferentiableRenderer2DFunc(torch.autograd.Function):
    """Device-resident variant: ``image = f(ij[V,2] f64 cuda, colors[V,C] cuda, DeviceScene, sigma[, depths[V]])``.

    ``depths`` (optional) is written into the scene and receives a gradient: with a ``perspective_correct`` scene the
    image depends on the vertex depths (zero gradient otherwise).

    The renderer keeps ONE live forward state per slot, and the ``DeviceScene`` is shared and mutable, so the node
    snapshots its inputs; if another forward has used the slot by the time ``backward`` runs (two renders before
    ``loss.backward()``), the forward is replayed from the snapshot first."""

    @staticmethod
    def forward(ctx: Any, ij: torch.Tensor, colors: torch.Tensor, scene: DeviceScene, sigma: float = 1.0,  # type: ignore
                depths: Optional[torch.Tensor] = None):
        arrays = {"ij": ij.detach(), "colors": colors.detach()}
        if depths is not None:
            arrays["depths"] = depths.detach()
        scene.update(**arrays)
        fwd = default_renderer(scene.device.index).render(scene, sigma)
        ctx.scene, ctx.sigma, ctx.fwd = scene, float(sigma), fwd
        ctx.in_dtypes = (ij.dtype, colors.dtype, depths.dtype if depths is not None else None)
        ctx.save_for_backward(*[a.clone() for a in arrays.values()])
        # the caller gets its own tensor: the framebuffers of ctx.fwd may be re-rendered into by backward
        return fwd["image"].clone()

    @staticmethod
    def backward(ctx: Any, *grad_outputs: Any) -> Any:
        (image_b,) = grad_outputs
        renderer = default_renderer(ctx.scene.device.index)
        saved = ctx.saved_tensors
        arrays = dict(zip(("ij", "colors", "depths"), saved))
        with_depths = len(saved) == 3
        if ctx.fwd["generation"] != renderer.generation(ctx.fwd["slot"]):
            ctx.scene.update(**arrays)
            ctx.fwd = renderer.render(ctx.scene, ctx.sigma, out=ctx.fwd)
        else:
            ctx.scene.update(**arrays)  # the shared scene may hold another node's inputs by now
        grads = renderer.render_b(ctx.scene, ctx.sigma, ctx.fwd, image_b, depths_b=with_depths)
        depths_b = grads["depths_b"].to(ctx.in_dtypes[2]) if with_depths else None
        return grads["ij_b"].to(ctx.in_dtypes[0]), grads["colors_b"].to(ctx.in_dtypes[1]), None, None, depths_b


CudaDifferentiableRender2D = CudaDifferentiableRenderer2DFunc.apply
