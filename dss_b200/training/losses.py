"""Point-cloud regularisers of the training step -- twins of DSS/training/losses.py:24-62 (BaseLoss), :148-277
(SurfaceLoss), :282-397 (ProjectionLoss) and :400-497 (RepulsionLoss), same class names, constructor arguments,
``forward(point_clouds, points_filter=..., rebuild_knn=..., knn_tree=...)`` signature and reductions.

They are rebuilt every iteration by the trainer (trainer.py:134-137, 321-326 with ``knn_k = 12``) and start with a
K-nearest-neighbour search over the cloud: pytorch3d ``knn_points`` in the reference, here
``dss_b200.frnn_grid.knn_points`` (csrc/knn.cu: density-sized grid, ring search -- 1.3 ms per 1 M points).  Everything
behind the search is a handful of elementwise / gather ops on (N, P, K) tensors, kept in torch (autograd gives the
position gradients exactly as in the reference: the neighbour positions and all weights are detached).

CUDA tensors take the CUDA K-NN; a caller on another device passes ``knn_tree=(dists, idx, knn)`` (the reference has
the same keyword) -- there is no CPU search in this package.
"""
from typing import NamedTuple, Optional

import torch
import torch.nn as nn

__all__ = ["BaseLoss", "L1Loss", "L2Loss", "IouLoss", "SurfaceLoss", "ProjectionLoss", "RepulsionLoss", "KNN"]


class KNN(NamedTuple):
    """pytorch3d's ``_KNN``: squared distances (N,P,K), indices (N,P,K) int64, neighbour positions (N,P,K,3)."""
    dists: torch.Tensor
    idx: torch.Tensor
    knn: Optional[torch.Tensor]


def eps_denom(denom, eps=1e-17):
    """DSS/utils/mathHelper.py:10-14: sign-preserving clamp, zero counts as positive."""
    sign = denom.sign().detach()
    sign = torch.where(sign == 0, torch.ones_like(sign), sign)
    return sign * torch.clamp(denom.abs(), min=eps)


def knn_gather(x, idx, lengths=None):
    """pytorch3d.ops.knn_gather: x (N,M,U), idx (N,P,K) -> (N,P,K,U); rows past `lengths` are zero."""
    N, P, K = idx.shape
    U = x.shape[-1]
    out = torch.gather(x[:, None].expand(-1, P, -1, -1), 2, idx[..., None].expand(-1, -1, -1, U))
    if lengths is not None:
        # pytorch3d zeroes neighbours that do not exist (k >= length of the cloud)
        need = torch.arange(K, device=idx.device)[None, None, :] >= lengths[:, None, None]
        out = torch.where(need[..., None], torch.zeros_like(out), out)
    return out


class BaseLoss(nn.Module):
    """losses.py:24-62."""

    def __init__(self, reduction: str = "mean", channel_dim: Optional[int] = -1):
        super().__init__()
        self.reduction = reduction
        self.channel_dim = channel_dim
        self.hooks = []

    def compute(self, *args, **kwargs):
        raise NotImplementedError

    def _reduce(self, loss, reduction=None):
        reduction = reduction or self.reduction
        if reduction == "none":
            return loss
        if reduction == "sum":
            return torch.sum(loss)
        if reduction == "mean":
            return torch.mean(loss)
        raise ValueError("Invalid reduction method ({})".format(self.reduction))

    def forward(self, *args, **kwargs):
        reduction = kwargs.pop("reduction", self.reduction)
        self.channel_dim = kwargs.pop("channel_dim", self.channel_dim)
        loss = self.compute(*args, **kwargs)
        if self.channel_dim is not None:
            loss = torch.sum(loss, dim=self.channel_dim)
        return self._reduce(loss, reduction=reduction)


class L1Loss(BaseLoss):
    def compute(self, x, y, weights=None, mask=None, **kwargs):
        loss = torch.abs(x - y)
        if weights is not None:
            loss = loss * weights
        return loss[mask] if mask is not None else loss


class L2Loss(BaseLoss):
    def compute(self, x, y, weights=None, mask=None, **kwargs):
        loss = (x - y) ** 2
        if weights is not None:
            loss = loss * weights
        return loss[mask] if mask is not None else loss


class IouLoss(BaseLoss):
    """losses.py:498-514: 1 - intersection / union per batch element (dims 1.. summed); the reduction then runs over
    the batch.  The trainer builds it with ``reduction="mean", channel_dim=None`` (trainer.py:138) and calls it as
    ``iou_loss(mask_gt, mask_pred)``; dss_b200.training.image_loss fuses that call into a CUDA op."""

    def compute(self, predict, target, **kwargs):
        dims = tuple(range(predict.ndimension())[1:])
        intersect = (predict * target).sum(dims)
        union = (predict + target - predict * target).sum(dims)
        return 1.0 - intersect / eps_denom(union)


def _padded_to_packed(x, lengths):
    """(N, Pmax, ...) -> (sum lengths, ...)"""
    keep = torch.arange(x.shape[1], device=x.device)[None, :] < lengths[:, None]
    return x[keep]


class SurfaceLoss(BaseLoss):
    """losses.py:148-277: neighbourhood weights shared by the two regularisers."""

    def __init__(self, reduction="mean", knn_k: int = 33, filter_scale: float = 1.0, sharpness_sigma: float = 0.75):
        super().__init__(reduction=reduction, channel_dim=None)
        self.knn_tree = None
        self.knn_mask = None
        self.knn_k = knn_k
        self.filter_scale = filter_scale
        self.sharpness_sigma = sharpness_sigma

    # -- neighbourhood ---------------------------------------------------------------------------
    def _build_knn(self, point_clouds):
        """losses.py:157-180: K nearest neighbours of every point inside its own cloud, the point itself dropped."""
        from ..frnn_grid import knn_points
        points_padded = point_clouds.points_padded()
        lengths = point_clouds.num_points_per_cloud()
        dists, idx, knn = knn_points(points_padded.detach(), points_padded.detach(), lengths, lengths, K=self.knn_k,
                                     return_nn=True)
        self._set_tree(KNN(dists, idx, knn), lengths)

    def _set_tree(self, tree, lengths):
        dists, idx, knn = tree
        K = dists.shape[-1]
        mask = torch.arange(idx.shape[1], device=idx.device)[None, :, None] < lengths[:, None, None]
        mask = mask & (torch.arange(K, device=idx.device)[None, None, :] < lengths.clamp(max=K)[:, None, None])
        self.knn_tree = KNN(dists[:, :, 1:], idx[:, :, 1:], None if knn is None else knn[:, :, 1:, :])
        self.knn_mask = mask[:, :, 1:]

    def _ensure_tree(self, point_clouds, rebuild_knn, kwargs):
        tree = kwargs.get("knn_tree", None)
        points = point_clouds.points_padded()
        lengths = point_clouds.num_points_per_cloud()
        if tree is not None:
            tree = KNN(*tree)
            if tree.dists.shape[-1] == self.knn_k:          # full result incl. the query itself (pytorch3d layout)
                if tree.knn is None:
                    tree = KNN(tree.dists, tree.idx, knn_gather(points.detach(), tree.idx, lengths))
                self._set_tree(tree, lengths)
            else:                                           # already without the query point (losses.py:305)
                self.knn_tree = tree if tree.knn is not None else KNN(tree.dists, tree.idx,
                                                                      knn_gather(points.detach(), tree.idx, lengths))
                self.knn_mask = kwargs.get("knn_mask", self.knn_mask)
        elif rebuild_knn or self.knn_tree is None or self.knn_tree.idx.shape[:2] != points.shape[:2]:
            self._build_knn(point_clouds)

    # -- weights ---------------------------------------------------------------------------------
    def get_phi(self, point_clouds, **kwargs):
        """(1 - |x - xi|^2 / h^2)^4 with h^2 = 4 x the mean squared neighbour distance (losses.py:258-277)."""
        h = self.knn_tree.dists.mean(dim=-1, keepdim=True) * 4
        w = (1 - self.knn_tree.dists / h).clamp(min=0)
        w = w * w
        return w * w

    def _denoise_normals(self, point_clouds, weights, point_clouds_filter=None):
        """robust normal mollification (losses.py:182-222): padded (N,P,3) weighted neighbour average; points that are
        visible AND inside the mask keep their own normal."""
        lengths = point_clouds.num_points_per_cloud()
        normals = point_clouds.normals_padded()
        knn_normals = knn_gather(normals, self.knn_tree.idx, lengths)
        den = torch.sum(knn_normals * weights[..., None], dim=-2) / eps_denom(torch.sum(weights, dim=-1, keepdim=True))
        if point_clouds_filter is not None and getattr(point_clouds_filter, "visibility", None) is not None:
            reliable = point_clouds_filter.visibility
            if getattr(point_clouds_filter, "inmask", None) is not None:
                reliable = reliable & point_clouds_filter.inmask
            if reliable.shape[0] != normals.shape[0] and normals.shape[0] == 1:
                reliable = reliable.any(dim=0, keepdim=True)
            den = torch.where(reliable[..., None], normals, den)
        return den

    def get_normal_w(self, normals, **kwargs):
        """exp(-|n - ni|^2 / sigma^2) over the neighbourhood, both renormalised (losses.py:224-246)."""
        self.sharpness_sigma = kwargs.get("sharpness_sigma", self.sharpness_sigma)
        inv = 1.0 / (self.sharpness_sigma * self.sharpness_sigma)
        knn_normals = torch.nn.functional.normalize(knn_gather(normals, self.knn_tree.idx), dim=-1)
        n = torch.nn.functional.normalize(normals, dim=-1)
        diff = knn_normals - n[:, :, None, :]
        return torch.exp(-torch.sum(diff * diff, dim=-1) * inv)

    def get_spatial_w(self, point_clouds, points=None, **kwargs):
        """exp(-|p - pi|^2 * (P / diag^2) * filter_scale) (losses.py:248-256)."""
        pts = point_clouds.points_padded()
        lengths = point_clouds.num_points_per_cloud()
        valid = torch.arange(pts.shape[1], device=pts.device)[None, :, None] < lengths[:, None, None]
        lo = torch.where(valid, pts, torch.full_like(pts, float("inf"))).min(dim=1)[0]
        hi = torch.where(valid, pts, torch.full_like(pts, float("-inf"))).max(dim=1)[0]
        diag2 = torch.sum((hi - lo) ** 2, dim=-1)
        inv_sigma = lengths.float() / diag2
        self.filter_scale = kwargs.get("filter_scale", self.filter_scale)
        if points is None:
            points = pts
        d = self.knn_tree.knn - points[:, :, None, :]
        return torch.exp(-torch.sum(d * d, dim=-1) * inv_sigma[:, None, None] * self.filter_scale)


class ProjectionLoss(SurfaceLoss):
    """losses.py:282-397: squared distance to the local plane of every neighbour, weighted (Oztireli et al.)."""

    def get_spatial_w(self, point_clouds, **kwargs):
        return torch.ones_like(self.knn_tree.dists)                       # losses.py:293-298

    def compute(self, point_clouds, points_filter=None, rebuild_knn=False, **kwargs):
        self.sharpness_sigma = kwargs.get("sharpness_sigma", self.sharpness_sigma)
        self.filter_scale = kwargs.get("filter_scale", self.filter_scale)
        lengths = point_clouds.num_points_per_cloud()
        points = point_clouds.points_padded()
        with torch.no_grad():
            self._ensure_tree(point_clouds, rebuild_knn, kwargs)
            phi = self.get_phi(point_clouds, **kwargs)
            normals = self._denoise_normals(point_clouds, phi, points_filter)          # Eq. (11)
            normal_w = self.get_normal_w(normals, **kwargs)
            if points_filter is not None and getattr(points_filter, "visibility", None) is not None:
                vis = points_filter.visibility
                if vis.shape[0] != points.shape[0] and points.shape[0] == 1:
                    vis = vis.any(dim=0, keepdim=True)
                vis_nb = knn_gather(vis.unsqueeze(-1), self.knn_tree.idx, lengths).squeeze(-1)
                visibility_w = torch.where(vis_nb, torch.ones_like(phi), torch.full_like(phi, 0.1))   # :335-337
            else:
                visibility_w = torch.ones_like(phi)
            weights = phi * normal_w * visibility_w
            knn_normals = knn_gather(normals, self.knn_tree.idx, lengths)
        sdf = torch.sum((self.knn_tree.knn.detach() - points.unsqueeze(-2)) * knn_normals, dim=-1)   # :373-374
        weights = _padded_to_packed(weights, lengths)
        sdf = _padded_to_packed(sdf, lengths)
        return torch.sum(weights * sdf * sdf, dim=-1) / eps_denom(torch.sum(weights, dim=-1))         # :390-395


class RepulsionLoss(SurfaceLoss):
    """losses.py:400-497: pushes a point away from the weighted centre of its neighbours inside the local plane."""

    def compute(self, point_clouds, points_filter=None, rebuild_knn=True, **kwargs):
        lengths = point_clouds.num_points_per_cloud()
        points = point_clouds.points_padded()
        with torch.no_grad():
            self._ensure_tree(point_clouds, rebuild_knn, kwargs)
            phi = self.get_phi(point_clouds, **kwargs)
            normals = self._denoise_normals(point_clouds, phi, points_filter)
        knn_diff = points.unsqueeze(-2) - self.knn_tree.knn.detach()                                   # :432
        knn_normals = knn_gather(normals, self.knn_tree.idx, lengths)
        proj = knn_diff - (knn_diff * knn_normals).sum(dim=-1, keepdim=True) * knn_normals            # :436-437
        with torch.no_grad():
            spatial_w = self.get_spatial_w(point_clouds, **kwargs)
            normal_w = self.get_normal_w(normals, **kwargs)
            density_w = torch.sum(spatial_w, dim=-1, keepdim=True) + 1.0                               # :470
            weights = spatial_w * normal_w
        weights = _padded_to_packed(weights, lengths)
        proj = _padded_to_packed(proj, lengths)
        density_w = _padded_to_packed(density_w, lengths)
        repel = torch.sum(proj * weights.unsqueeze(-1), dim=1) / eps_denom(torch.sum(weights, dim=1).unsqueeze(-1))
        repel = repel * density_w                                                                      # :482-485
        return torch.exp(-repel.abs())                                                                 # :487
