"""Mint tests/golden/reference/dr_loss.npz: the image objective of the reference's training step, evaluated by the
reference's own loss classes (DSS/training/losses.py L1Loss, IouLoss and DSS/utils/mathHelper.py eps_denom) in float64
on seeded inputs, with its autograd gradient with respect to the rendered image.

    python -m tests.golden.make_golden_dr_loss /path/to/DSS-checkout

The body of Trainer.calc_dr_loss (DSS/training/trainer.py:332-376) is run as written, with the rgb and silhouette
terms kept unweighted as well.  tests/test_dr_loss.py and tests/test_gpu_dr_loss.py compare with the file.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference", "dr_loss.npz")
IOU_WEIGHT = 0.01


def cases():
    """name -> (image (N,S,S,4), img (N,3,S,S), mask (N,1,S,S) or (N,S,S), lambda_rgb, lambda_silhouette), float32"""
    rng = np.random.default_rng(2024)
    f = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    out = {}
    N, S = 3, 24
    # 1. random colours, binary masks (the rendered occupancy of the renderer is 0/1)
    image = rng.random((N, S, S, 4))
    image[..., 3] = rng.random((N, S, S)) < 0.6
    out["binary"] = (f(image), f(rng.random((N, 3, S, S))), f(rng.random((N, 1, S, S)) < 0.5), 1.0, 1.0)
    # 2. non-binary masks on both sides (soft GT mattes), other weights, (N,S,S) mask layout
    image = rng.random((N, S, S, 4))
    image[..., 3] *= rng.random((N, S, S)) < 0.7
    mask = rng.random((N, S, S)) * (rng.random((N, S, S)) < 0.8)
    out["soft"] = (f(image), f(rng.random((N, 3, S, S))), f(mask), 2.0, 0.5)
    # 3. view 0: empty GT mask; view 1: empty prediction; view 2: both empty (union 0: eps_denom clamps, no gradient
    #    through U); view 3: union 1e-20 (below the clamp, but the intersection term still has a gradient)
    N4 = 4
    image = rng.random((N4, S, S, 4))
    image[..., 3] = rng.random((N4, S, S)) < 0.5
    mask = (rng.random((N4, 1, S, S)) < 0.5).astype(np.float64)
    mask[0] = 0
    image[1, ..., 3] = 0
    mask[2] = 0
    image[2, ..., 3] = 0
    mask[3] = 0
    image[3, ..., 3] = 0
    mask[3, 0, 5, 7] = 1e-20
    out["empty_views"] = (f(image), f(rng.random((N4, 3, S, S))), f(mask), 1.0, 1.0)
    # 4. M == 0: GT mask and prediction never overlap (no rgb term, no rgb gradient)
    image = rng.random((N, S, S, 4))
    left = np.arange(S)[None, :, None] < S // 2
    image[..., 3] = np.broadcast_to(left, (N, S, S)) * (rng.random((N, S, S)) < 0.7)
    mask = np.broadcast_to(~left, (N, S, S)) * (rng.random((N, S, S)) < 0.7)
    out["no_overlap"] = (f(image), f(rng.random((N, 3, S, S))), f(mask[:, None]), 1.0, 1.0)
    # 5. pred == GT exactly on part of the pixels, in rgb and in alpha (|x|' = 0 at 0)
    image = rng.random((N, S, S, 4))
    image[..., 3] = rng.random((N, S, S)) < 0.6
    img = rng.random((N, 3, S, S))
    mask = (rng.random((N, 1, S, S)) < 0.6).astype(np.float64)
    same = rng.random((N, S, S)) < 0.5
    img = np.where(same[:, None], np.moveaxis(image[..., :3], -1, 1), img)
    mask[:, 0] = np.where(rng.random((N, S, S)) < 0.5, image[..., 3], mask[:, 0])
    out["exact"] = (f(image), f(img), f(mask), 1.0, 1.0)
    return out


def calc_dr_loss(L1Loss, IouLoss, image, img, mask, lambda_rgb, lambda_silhouette):
    """Trainer.calc_dr_loss in float64 on (N,S,S,4) rendered image, (N,3,S,S) GT colours and the GT mask; returns the
    terms (loss, rgb, silhouette, iou) and d loss / d image.  rgb and silhouette are the unweighted terms, loss is the
    reference's loss_dr_rgb + loss_dr_silhouette."""
    N, S = image.shape[0], image.shape[1]
    pred = torch.from_numpy(np.asarray(image, np.float64)).requires_grad_(True)
    gt = torch.from_numpy(np.asarray(img, np.float64)).permute(0, 2, 3, 1)
    mask_img = torch.from_numpy(np.asarray(mask, np.float64)).reshape(N, S, S)
    img_pred, mask_img_pred = pred[..., :3], pred[..., 3]
    l1_loss = L1Loss(reduction="mean")
    iou_loss = IouLoss(reduction="mean", channel_dim=None)
    loss_rgb = torch.zeros((), dtype=torch.float64)
    if lambda_rgb > 0:
        mask_pred = mask_img.bool() & mask_img_pred.bool()
        if mask_pred.sum() > 0:
            loss_rgb = l1_loss(gt, img_pred, mask=mask_pred, reduction="mean")
    # (the reference writes mask_img.float(): the mask holds float32 values already, kept here in float64)
    loss_mask = (mask_img - mask_img_pred).abs().mean()
    loss_iou = iou_loss(mask_img, mask_img_pred)
    loss_sil = IOU_WEIGHT * loss_iou + loss_mask
    loss = loss_rgb * lambda_rgb + loss_sil * lambda_silhouette
    loss.backward()
    terms = np.array([float(t.detach()) for t in (loss, loss_rgb, loss_sil, loss_iou)])
    return terms, pred.grad.numpy()


def main(reference):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, reference)
    from tests import shim
    shim.install()
    from DSS.training.losses import IouLoss, L1Loss   # the reference's classes (eps_denom: DSS/utils/mathHelper.py)
    arrays = {}
    for name, (image, img, mask, lr, ls) in cases().items():
        terms, grad = calc_dr_loss(L1Loss, IouLoss, image, img, mask, lr, ls)
        arrays.update({name + "/image": image, name + "/img": img, name + "/mask": mask,
                       name + "/weights": np.array([lr, ls, IOU_WEIGHT]), name + "/terms": terms,
                       name + "/grad": grad})
    np.savez_compressed(OUT, **arrays)
    print("wrote", OUT, sorted({k.split("/")[0] for k in arrays}))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python -m tests.golden.make_golden_dr_loss /path/to/DSS-checkout")
    main(sys.argv[1])
