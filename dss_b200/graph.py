"""CUDA-graph replay of a whole render step (forward + backward) for loops with fixed shapes.

A step is ~30 kernel launches and two ctypes calls; at the headline size (1.7 ms of kernels) the launches hide behind the
GPU work, at the smaller BASELINE clouds (100k points: 0.6 ms) they do not.  The C library never synchronises or
allocates in steady state (DESIGN.md "Host side"), so the whole step can be captured once and replayed:

    step = GraphedRenderStep(points, normals, colours, proj, view, h, params, grad_image)
    step.replay()                    # image in step.image, gradients in step.grad_points / step.grad_colours
    step.points.data.add_(...)       # update the step's OWN static leaves in place (optimizer step), replay again

The step owns its differentiated inputs (`step.points`, `step.colours`, `step.normals`: fresh leaf copies of what was passed
in): a leaf that has already been through an eager backward on the default stream carries an AccumulateGrad node bound
to that stream, and synchronising with the legacy default stream is not capturable.

Sizes decided on the host at capture time are frozen into the graph: the forward's tile-list capacity and the staged
window of the occupancy gather.  Both have on-device fallbacks (tiles whose list outgrew the buffer are rasterized from
the records; views whose window does not fit take the direct gather), so a replay is always CORRECT; `stale()` tells when
re-capturing would make it faster again.
"""
import torch
import torch.nn.functional as F

from . import _lib
from .core.rasterizer import vrk_h
from .core.texture import camera_centres
from .ops import Shading, render_points
from .training.image_loss import _dr_terms

__all__ = ["GraphedRenderStep", "GraphedTrainStep"]


class GraphedRenderStep:
    def __init__(self, points, normals, colours, proj, view, h, params, grad_image, shading=None, warmup=3,
                 grad_sync=None):
        dev = _lib.require_cuda(points, normals, colours, proj, view, h, grad_image)
        self.device = dev
        leaf = lambda t: t.detach().clone().requires_grad_(True)
        self.points, self.colours = leaf(points), leaf(colours)
        self.normals = leaf(normals) if shading is not None else normals.detach().clone()
        self._args = (self.points, self.normals, self.colours, proj, view, h, params)
        self._shading = shading
        if grad_sync is not None and grad_sync.world_size > 1:
            # measured on 2 x B200: capturing the two overlapped NCCL all-reduces (issued from two streams inside the
            # backward) deadlocks at replay -- a view-sharded step is launched eagerly
            raise NotImplementedError("GraphedRenderStep does not capture the multi-GPU gradient exchange; "
                                      "call render_points(..., grad_sync=...) eagerly")
        self._sync = grad_sync
        self.grad_image = grad_image
        # warm-up on a side stream (sizes the library's scratch and the caching allocator), then capture
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(max(1, warmup)):
                self._eager()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        self._capacity_at_capture = self._tile_total()
        self._clear_grads()
        self.graph = torch.cuda.CUDAGraph()
        timing = getattr(grad_sync, "timing", False)
        if grad_sync is not None:
            grad_sync.timing = False    # no timing events inside a capture
        try:
            with torch.cuda.graph(self.graph):
                out = self._eager()
        finally:
            if grad_sync is not None:
                grad_sync.timing = timing
        self.image, self.visible = out.image, out.visible
        self.grad_points, self.grad_colours = self.points.grad, self.colours.grad
        self.grad_normals = self.normals.grad if shading is not None else None

    def _clear_grads(self):
        for t in self._args[:3]:
            if t.requires_grad:
                t.grad = None

    def _eager(self):
        self._clear_grads()
        points, normals, colours, proj, view, h, params = self._args
        out = render_points(points, normals, colours, proj, view, h, params, shading=self._shading, grad_sync=self._sync)
        out.image.backward(self.grad_image)
        return out

    def _tile_total(self):
        """the tile-list size the device published last (mapped pinned word; no synchronisation)"""
        return int(_lib.load().dss_debug_tile_total(_lib.ctx(self.device)))

    def replay(self):
        self.graph.replay()
        return self.image

    def stale(self, slack=1.2) -> bool:
        """True when the tile lists have outgrown what they were at capture time by more than `slack` (the replay is
        still correct -- overflowing tiles are rasterized from the records -- but a fresh capture will be faster)."""
        now = self._tile_total()
        return self._capacity_at_capture > 0 and now > slack * 1.25 * self._capacity_at_capture


class GraphedTrainStep:
    """One training iteration of a shared cloud seen from N cameras, captured once and replayed:
    h from the step's own points -> F.normalize(normals) -> render_points -> dr_image_loss -> backward.

        step = GraphedTrainStep(points, normals, colours, proj, view, img, mask, params, h="invariant")
        for batch in loader:
            step.load(batch.proj, batch.view, batch.img, batch.mask)   # copy_ into the step's static inputs
            step.replay()           # step.loss (4,) = {loss, rgb, silhouette, iou}, step.image, step.grad_*
            optimizer.step()        # over step.parameters(); the step's leaves are updated in place

    The leaves (`step.points`, `step.normals`, `step.colours` -- the albedo with ``shading=``) are fresh copies of what
    was passed in; give THEM to the optimizer.  Their gradients are `step.grad_points`, `step.grad_normals` (None
    without shading: the normals then only shape the splats, which the reference does not differentiate) and
    `step.grad_colours`.  The rendered normals are F.normalize of the raw leaf, as Model._get_normals does
    (DSS/models/point_modeling.py:84-86), so the normal gradient reaches the raw leaf.

    h: "invariant" or "isotropic" recomputes the splat variance scale from the current points inside the graph, with the
    rule of SurfaceSplatting._compute_h (Vrk_invariant / Vrk_isotropic, dss_b200.core.rasterizer.vrk_h), as the
    reference does in every forward; a tensor ((N,) or (N*P0,)) is used as given.

    Frozen at capture, so changing one of them needs a NEW step: the SplatParams (e.g. the radii_backward_scaler schedule
    of DSS/training/scheduler.py:36-48), the loss weights, the shapes, the light type and shininess.  The optimizer,
    the projection / repulsion regularisers (their gradient is added to the leaves' before the optimizer step) and
    any multi-GPU gradient exchange stay outside the graph.
    """

    def __init__(self, points, normals, colours, proj, view, img, mask, params, h="invariant", shading=None,
                 lambda_rgb=1.0, lambda_silhouette=1.0, iou_weight=0.01, frnn_radius=0.2, warmup=3, grad_sync=None):
        dev = _lib.require_cuda(points, normals, colours, proj, view, img, mask)
        if grad_sync is not None and grad_sync.world_size > 1:
            raise NotImplementedError("GraphedTrainStep does not capture the multi-GPU gradient exchange; "
                                      "call render_points(..., grad_sync=...) eagerly")
        if isinstance(h, str):
            if h not in ("invariant", "isotropic"):
                raise ValueError('h must be "invariant", "isotropic" or a tensor, got %r' % h)
        else:
            _lib.require_cuda(h)
            h = h.detach().clone()
        self.device = dev
        leaf = lambda t: t.detach().clone().requires_grad_(True)
        self.points, self.normals, self.colours = leaf(points), leaf(normals), leaf(colours)
        static = lambda t: t.detach().clone()
        self.proj, self.view, self.img, self.mask = static(proj), static(view), static(img), static(mask)
        self._shading = None
        if shading is not None:
            self.lights, self.ambient = static(shading.lights), static(shading.ambient)
            self._shading = (int(shading.light_type), float(shading.shininess))
        self._h, self._radius, self.params = h, float(frnn_radius), params
        self._weights = (float(lambda_rgb), float(lambda_silhouette), float(iou_weight))
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(max(1, warmup)):
                self._eager()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        self._capacity_at_capture = self._tile_total()
        self._clear_grads()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.image, self.loss = self._eager()
        self.grad_points, self.grad_normals, self.grad_colours = self.points.grad, self.normals.grad, self.colours.grad

    def parameters(self):
        return [self.points, self.normals, self.colours]

    def _clear_grads(self):
        for t in self.parameters():
            t.grad = None

    def _splat_h(self):
        """the variance scale the step renders with, from the current points (see the class docstring)"""
        N = self.proj.shape[0]
        if not isinstance(self._h, str):
            return self._h
        h0 = vrk_h(self.points, self._h == "invariant", self._radius)
        return h0.expand(N) if self._h == "invariant" else h0.repeat(N)

    def _eager(self):
        self._clear_grads()
        shading = None
        if self._shading is not None:
            shading = Shading(self.lights, self.ambient, camera_centres(self.view), *self._shading)
        out = render_points(self.points, F.normalize(self.normals, dim=-1), self.colours, self.proj, self.view,
                            self._splat_h(), self.params, shading=shading)
        terms = _dr_terms(out.image, self.img, self.mask, *self._weights)
        terms[0].backward()
        return out.image, terms.detach()

    def load(self, proj, view, img, mask, lights=None, ambient=None):
        """copy one batch (cameras, targets and, with shading, the light rows) into the step's static inputs"""
        self.proj.copy_(proj)
        self.view.copy_(view)
        self.img.copy_(img)
        self.mask.copy_(mask)
        if lights is not None or ambient is not None:
            if self._shading is None:
                raise RuntimeError("this step was captured without shading")
            if lights is not None:
                self.lights.copy_(lights)
            if ambient is not None:
                self.ambient.copy_(ambient)

    def replay(self):
        self.graph.replay()
        return self.loss

    _tile_total = GraphedRenderStep._tile_total
    stale = GraphedRenderStep.stale
