"""The fused image objective (dss_b200.training.dr_image_loss, csrc/loss.cu) and the graph-replayed training step
(dss_b200.graph.GraphedTrainStep) on the GPU: values and gradients against the float64 restatement of
Trainer.calc_dr_loss, determinism, CUDA-graph capture, and replay against the eager chain."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from dss_b200.core.camera import camera_matrices
from dss_b200.core.rasterizer import vrk_h
from dss_b200.core.texture import camera_centres
from dss_b200.ops import Shading, SplatParams, make_shading, render_points
from dss_b200.training import dr_image_loss
from tests.test_dr_loss import CASES, golden, restated
from tests.test_shading import _lights
from tests.util import random_cameras, scene

pytestmark = pytest.mark.gpu


def _check(got, got_grad, terms, grad):
    """terms to 1e-6 relative, every gradient channel to 1e-6 x max |grad|"""
    vals = np.array([float(t.detach()) for t in got])
    assert np.all(np.abs(vals - terms) <= 1e-6 * np.abs(terms)), (vals, terms)
    scale = np.abs(grad).max()
    err = np.abs(got_grad.double().cpu().numpy() - grad).max(axis=(0, 1, 2))
    assert np.all(err <= 1e-6 * scale), (err, scale)


def _run(image, img, mask, weights):
    """dr_image_loss and d loss / d image"""
    x = image.detach().clone().requires_grad_(True)
    out = dr_image_loss(x, img, mask, *weights)
    out.loss.backward()
    torch.cuda.synchronize()
    return out, x.grad


@pytest.mark.parametrize("name", CASES)
def test_golden_cases(cuda_device, name):
    case = golden(name)
    d = cuda_device
    image, img, mask = (torch.from_numpy(case[k]).to(d) for k in ("image", "img", "mask"))
    out, grad = _run(image, img, mask, tuple(case["weights"]))
    _check(out, grad, case["terms"], case["grad"])


def _targets(pts, nrm, col, proj, view, h, prm, seed):
    """GT colours (N,3,S,S) and mask (N,1,S,S) rendered from a perturbed cloud"""
    g = torch.Generator().manual_seed(seed)
    d = proj.device
    p = pts + (0.01 * torch.randn(pts.shape, generator=g)).to(d)
    c = (col + 0.2 * torch.rand(col.shape, generator=g).to(d)).clamp(0, 1)
    with torch.no_grad():
        im = render_points(p, nrm, c, proj, view, h, prm).image
    return im[..., :3].permute(0, 3, 1, 2).contiguous(), im[..., 3:].permute(0, 3, 1, 2).contiguous()


def _sphere_images(d, P0=100000, N=8, S=512):
    pts, nrm, col, proj, view, _ = scene(P0, N, seed=11)
    pts, nrm, col, proj, view = (t.to(d) for t in (pts, nrm, col, proj, view))
    prm = SplatParams(image_size=S, znear=0.1)
    h = torch.full((N,), 3e-4, device=d)
    with torch.no_grad():
        image = render_points(pts, nrm, col, proj, view, h, prm).image
    img, mask = _targets(pts, nrm, col, proj, view, h, prm, seed=5)
    return image, img, mask


def test_headline_size_against_the_restatement(cuda_device):
    image, img, mask = _sphere_images(cuda_device)
    assert 0 < float(image[..., 3].mean()) < 1 and 0 < float(mask.mean()) < 1
    out, got_grad = _run(image, img, mask, (1.0, 1.0, 0.01))
    terms, grad = restated({"image": image.cpu().numpy(), "img": img.cpu().numpy(), "mask": mask.cpu().numpy(),
                            "weights": np.array([1.0, 1.0, 0.01])})
    assert terms[1] > 0 and terms[3] > 0
    _check(out, got_grad, terms, grad)


def test_two_calls_are_bit_identical(cuda_device):
    image, img, mask = _sphere_images(cuda_device)
    a, ga = _run(image, img, mask, (1.0, 1.0, 0.01))
    b, gb = _run(image, img, mask, (1.0, 1.0, 0.01))
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert torch.equal(ga, gb)


def test_op_captures_and_replays_on_new_inputs(cuda_device):
    d = cuda_device
    A, B = golden("binary"), golden("exact")
    image = torch.from_numpy(A["image"]).to(d).requires_grad_(True)
    img, mask = torch.from_numpy(A["img"]).to(d), torch.from_numpy(A["mask"]).to(d)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            image.grad = None
            dr_image_loss(image, img, mask).loss.backward()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    image.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = dr_image_loss(image, img, mask)
        out.loss.backward()
    grad = image.grad
    for case in (B, A):
        with torch.no_grad():
            image.copy_(torch.from_numpy(case["image"]))
            img.copy_(torch.from_numpy(case["img"]))
            mask.copy_(torch.from_numpy(case["mask"]))
        graph.replay()
        torch.cuda.synchronize()
        want, want_grad = _run(image.detach(), img.clone(), mask.clone(), (1.0, 1.0, 0.01))
        for x, y in zip(out, want):
            assert torch.equal(x, y)
        assert torch.equal(grad, want_grad)


def _close(a, b):
    assert (a - b).abs().max() <= 1e-6 * b.abs().max(), ((a - b).abs().max(), b.abs().max())


@pytest.mark.parametrize("shaded", [False, True])
def test_graphed_train_step_equals_the_eager_chain(cuda_device, shaded):
    from dss_b200.graph import GraphedTrainStep
    d = cuda_device
    P0, N, S = 30000, 3, 128
    pts, nrm, col, proj, view, _ = scene(P0, N, seed=23)
    pts, nrm, col, proj, view = (t.to(d) for t in (pts, nrm, col, proj, view))
    prm = SplatParams(image_size=S, znear=0.1, clip_pts_grad=0.05)
    h0 = torch.full((N,), 3e-4, device=d)
    projB, viewB = (t.to(d) for t in camera_matrices(random_cameras(N, seed=77)))
    # targets from the unit normals (the renderer's input contract) ...
    batches = [(proj, view) + _targets(pts, nrm, col, proj, view, h0, prm, seed=1),
               (projB, viewB) + _targets(pts, nrm, col, projB, viewB, h0, prm, seed=2)]
    for b in batches:
        assert all(torch.isfinite(t).all() for t in b)
    kind, shin = 1, 64.0
    sh = make_shading(_lights("point", d), view) if shaded else None
    # ... the step's raw normal leaf is not unit length: the step renders F.normalize of it
    step = GraphedTrainStep(pts, 1.5 * nrm, col, *batches[0], prm, h="invariant", shading=sh)

    def eager():
        pe, ne, ce = (t.detach().clone().requires_grad_(True) for t in step.parameters())
        h = vrk_h(pe, True).expand(N)
        s = Shading(step.lights, step.ambient, camera_centres(step.view), kind, shin) if shaded else None
        o = render_points(pe, F.normalize(ne, dim=-1), ce, step.proj, step.view, h, prm, shading=s)
        l = dr_image_loss(o.image, step.img, step.mask)
        l.loss.backward()
        torch.cuda.synchronize()
        return o.image.detach(), torch.stack(list(l)).detach(), pe.grad, ne.grad, ce.grad

    def compare():
        step.replay()
        torch.cuda.synchronize()
        image, terms, gp, gn, gc = eager()
        assert torch.equal(step.image, image)
        assert torch.isfinite(terms).all() and float(terms[0]) > 0
        assert torch.equal(step.loss, terms)
        if shaded:
            _close(step.grad_points, gp)
            _close(step.grad_normals, gn)
        else:
            assert torch.equal(step.grad_points, gp)       # deterministic occupancy gather
            assert step.grad_normals is None and gn is None
        _close(step.grad_colours, gc)                       # colour scatter: float red.add

    compare()
    step.load(*batches[1])
    compare()
    with torch.no_grad():                                  # an optimizer step on the step's leaves
        step.points.add_(0.002 * torch.randn(P0, 3, generator=torch.Generator().manual_seed(3)).to(d))
        step.colours.mul_(0.9)
    compare()
    step.load(*batches[0])
    compare()
