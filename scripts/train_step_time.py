"""Time one training iteration on the bench scene (sphere cloud, 8 views, 512 x 512), three routes:

  torch : eager render + the reference objective in torch (Trainer.calc_dr_loss: boolean-mask L1, `mask_pred.sum() > 0`
          branch, silhouette L1, IouLoss) + backward -- two host waits per step
  fused : eager render + dss_b200.training.dr_image_loss + backward
  graph : dss_b200.graph.GraphedTrainStep.replay()

All three recompute h from the points (Vrk_invariant rule) and render F.normalize(normals).  Also times the objective
alone (forward + backward on a fixed image, CUDA events) for both implementations.

    python scripts/train_step_time.py [--out FILE] [--iters 50]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dss_b200.core.camera import camera_matrices                     # noqa: E402
from dss_b200.core.rasterizer import vrk_h                            # noqa: E402
from dss_b200.graph import GraphedTrainStep                           # noqa: E402
from dss_b200.ops import SplatParams, render_points                   # noqa: E402
from dss_b200.training import IouLoss, L1Loss, dr_image_loss          # noqa: E402
from tests.util import random_cameras, sphere_cloud                   # noqa: E402

l1_loss, iou_loss = L1Loss(reduction="mean"), IouLoss(reduction="mean", channel_dim=None)


def torch_objective(image, img, mask, lambda_rgb=1.0, lambda_sil=1.0):
    """the body of Trainer.calc_dr_loss (trainer.py:332-376) on (N,S,S,4) image, (N,3,S,S) img, (N,1,S,S) mask"""
    gt = img.permute(0, 2, 3, 1)
    m = mask.reshape(mask.shape[0], mask.shape[-2], mask.shape[-1])
    img_pred, mask_img_pred = image[..., :3], image[..., 3]
    loss_rgb = 0.0
    mask_pred = m.bool() & mask_img_pred.bool()
    if mask_pred.sum() > 0:                                  # host wait 1 (and 2: the boolean index below)
        loss_rgb = l1_loss(gt, img_pred, mask=mask_pred, reduction="mean") * lambda_rgb
    loss_mask = (m.float() - mask_img_pred).abs().mean()
    loss_iou = iou_loss(m.float(), mask_img_pred)
    return loss_rgb + (0.01 * loss_iou + loss_mask) * lambda_sil


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or None
    except Exception:
        power = None
    return {"gpu": name, "power_limit": power}


def timed(fn, iters, warmup=5):
    """ms per call: host clock around `iters` calls that end in a device synchronise"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / iters


def event_ms(fn, iters, warmup=5):
    """ms per call from CUDA events around `iters` calls"""
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def run(P0, N, S, iters, dev):
    prm = SplatParams(image_size=S, points_per_pixel=5, cutoff_threshold=1.0, depth_merging_threshold=0.05,
                      antialiasing_sigma=1.0, radii_backward_scaler=5.0, clip_pts_grad=0.05, backface_culling=False,
                      znear=0.1, zfar=100.0)
    pts, nrm, col = (t.to(dev) for t in sphere_cloud(P0, seed=0))
    proj, view = (t.to(dev) for t in camera_matrices(random_cameras(N, seed=0)))
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():   # targets: the cloud perturbed, recoloured
        p_t = pts + (0.005 * torch.randn(pts.shape, generator=g)).to(dev)
        im = render_points(p_t, nrm, (col * 0.8).contiguous(), proj, view, vrk_h(p_t, True).expand(N), prm).image
        img, mask = im[..., :3].permute(0, 3, 1, 2).contiguous(), im[..., 3:].permute(0, 3, 1, 2).contiguous()
    leaves = [t.clone().requires_grad_(True) for t in (pts, nrm, col)]

    def eager(objective):
        def step():
            for t in leaves:
                t.grad = None
            p, n, c = leaves
            out = render_points(p, F.normalize(n, dim=-1), c, proj, view, vrk_h(p, True).expand(N), prm)
            objective(out.image).backward()
        return step

    res = {"points": P0, "views": N, "image_size": S, "iters": iters}
    res["torch_ms"] = timed(eager(lambda im: torch_objective(im, img, mask)), iters)
    res["fused_ms"] = timed(eager(lambda im: dr_image_loss(im, img, mask).loss), iters)
    step = GraphedTrainStep(pts, nrm, col, proj, view, img, mask, prm, h="invariant")
    res["graph_ms"] = timed(step.replay, iters)
    # the objective alone, forward + backward on a fixed rendered image
    with torch.no_grad():
        image = render_points(pts, nrm, col, proj, view, vrk_h(pts, True).expand(N), prm).image
    x = image.clone().requires_grad_(True)

    def obj(f):
        def call():
            x.grad = None
            f(x).backward()
        return call
    res["loss_op_ms"] = event_ms(obj(lambda im: dr_image_loss(im, img, mask).loss), 200)
    res["torch_objective_ms"] = event_ms(obj(lambda im: torch_objective(im, img, mask)), 200)
    # algorithmic bytes of the two kernels' passes: 32 B per pixel forward, 48 B backward
    px = N * S * S
    res["loss_op_algorithmic_bytes"] = 80 * px
    res["loss_op_GBps"] = 80 * px / (res["loss_op_ms"] * 1e-3) / 1e9
    with torch.no_grad():
        want = dr_image_loss(step.image, img, mask).loss
    res["graph_loss_matches_eager_op"] = bool(torch.equal(step.loss[0], want))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("train_step_time.py needs a CUDA device")
    dev = torch.device("cuda:0")
    rows = [run(P0, 8, 512, a.iters, dev) for P0 in (1_000_000, 100_000)]
    result = {"card": card(), "rows": rows}
    print(json.dumps(result, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
