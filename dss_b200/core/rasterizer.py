"""Surface-splatting rasterizer -- host-side mirror of DSS/core/rasterizer.py (same class and function
names, constructor / forward signatures and attributes), driving libdss_b200.so instead of
DSS._C + frnn + prefix_sum.  Select it from YAML with
``renderer.raster_type: dss_b200.core.rasterizer.SurfaceSplatting`` (config.py:241-262).

Differences from the reference, all documented in DESIGN.md:
  * points rejected by the depth / backface filters keep their packed slot and get view depth z = -1
    (never rasterized, never receive gradients) instead of being compacted into a new cloud
    (rasterizer.py:219-254); ``idx`` therefore always indexes the cloud that was passed in;
  * ``bin_size`` / ``max_points_per_bin`` are accepted and ignored (exact-size tile lists);
  * the backward pass needs no FRNN grid, no per-view host loop and no ``unique()``.
"""
from typing import NamedTuple, Optional

import torch
import torch.autograd as autograd
import torch.nn as nn

from .. import _C
from ..ops import SplatParams, preprocess_points
from .camera import camera_matrices
from .cloud import clouds_share_points
from .knn import knn_sq_dists

__all__ = ["PointFragments", "PointsRasterizationSettings", "SurfaceSplatting", "rasterize_elliptical_points",
           "EllipticalRasterizer", "kMaxPointsPerBin", "vrk_h"]

kMaxPointsPerBin = 22   # pytorch3d constant the reference (mis)uses as a bound on bins per side (rasterizer.py:725-730)


def vrk_h(points: torch.Tensor, invariant: bool, radius: float = 0.2) -> torch.Tensor:
    """Variance scale of ONE cloud's splats from its (P,3) points (rasterizer.py:293-402), on the device without a host
    read-back (the K-NN is csrc/knn.cu), so a CUDA graph can evaluate it on moving points:
    Vrk_invariant: 0-d clamp(mean_p(0.5 max_{6NN} d^2), 5e-5, 1e-3);  Vrk_isotropic: (P,) clamp(0.5 max_{6NN} d^2, 5e-5, 0.01)."""
    if points.shape[0] < 7:   # "knn search is unreliable, set sq_dist manually" (rasterizer.py:320-321)
        h = torch.full((points.shape[0],), 0.5e-3, device=points.device)
    else:
        d2 = knn_sq_dists(points.detach(), K=7, radius=radius)[:, 1:]
        h = 0.5 * d2.max(dim=-1)[0]
    if invariant:
        return (h.mean().clamp(5e-5, 1e-3) if h.numel() else h.new_tensor(1e-3)).float()
    return h.clamp(5e-5, 0.01).float()


class PointFragments(NamedTuple):
    """rasterizer.py:31-36"""
    idx: torch.Tensor
    zbuf: torch.Tensor
    qvalue: torch.Tensor
    scaler: torch.Tensor
    occupancy: torch.Tensor


class PointsRasterizationSettings:
    """Same attributes and defaults as rasterizer.py:39-99."""
    __slots__ = ["cutoff_threshold", "backface_culling", "depth_merging_threshold", "Vrk_invariant",
                 "Vrk_isotropic", "radii_backward_scaler", "image_size", "points_per_pixel", "bin_size",
                 "max_points_per_bin", "clip_pts_grad", "antialiasing_sigma"]

    def __init__(self, backface_culling: bool = True, cutoff_threshold: float = 1,
                 depth_merging_threshold: float = 0.05, Vrk_invariant: bool = False, Vrk_isotropic: bool = True,
                 radii_backward_scaler: float = 10, image_size: int = 256, points_per_pixel: int = 8,
                 bin_size: Optional[int] = 0, max_points_per_bin: Optional[int] = None,
                 clip_pts_grad: Optional[float] = -1, antialiasing_sigma: Optional[float] = 1.0):
        self.cutoff_threshold = cutoff_threshold
        self.backface_culling = backface_culling
        self.depth_merging_threshold = depth_merging_threshold
        self.Vrk_invariant = Vrk_invariant
        self.Vrk_isotropic = Vrk_isotropic
        self.radii_backward_scaler = radii_backward_scaler
        self.image_size = image_size
        self.points_per_pixel = points_per_pixel
        self.bin_size = bin_size
        self.max_points_per_bin = max_points_per_bin
        self.clip_pts_grad = clip_pts_grad
        self.antialiasing_sigma = antialiasing_sigma


def _splat_params(rs: PointsRasterizationSettings, cameras, kwargs=None) -> SplatParams:
    kwargs = kwargs or {}
    znear = getattr(cameras, "znear", kwargs.get("znear", 1.0))
    zfar = getattr(cameras, "zfar", kwargs.get("zfar", 100.0))
    f = lambda v: float(v.reshape(-1)[0]) if torch.is_tensor(v) else float(v)
    return SplatParams(image_size=int(rs.image_size), points_per_pixel=int(rs.points_per_pixel),
                       cutoff_threshold=float(rs.cutoff_threshold),
                       depth_merging_threshold=float(rs.depth_merging_threshold),
                       antialiasing_sigma=float(rs.antialiasing_sigma),
                       radii_backward_scaler=float(rs.radii_backward_scaler),
                       clip_pts_grad=float(rs.clip_pts_grad if rs.clip_pts_grad is not None else -1.0),
                       backface_culling=bool(rs.backface_culling), znear=f(znear), zfar=f(zfar))


class SurfaceSplatting(nn.Module):
    """rasterizer.py:102-664.  Outputs per point the screen-space extent and centre of projection, and per
    pixel the K nearest splats."""

    def __init__(self, cameras=None, raster_settings=None, frnn_radius=0.2):
        super().__init__()
        if raster_settings is None:
            raster_settings = PointsRasterizationSettings()
        self.cameras = cameras
        self.raster_settings = raster_settings
        self.frnn_radius = frnn_radius
        self._Vrk_h = None

    @property
    def device(self):
        cams = self.cameras
        return getattr(cams, "device", torch.device("cpu")) if cams is not None else torch.device("cpu")

    def to(self, device):
        if self.cameras is not None and hasattr(self.cameras, "to"):
            self.cameras = self.cameras.to(device)
        return self

    # ---- geometry ----------------------------------------------------------------------------
    def _cameras(self, kwargs):
        cameras = kwargs.get("cameras", self.cameras)
        if cameras is None:
            raise ValueError("Cameras must be specified either at initialization or in the forward pass")
        self.cameras = cameras
        return cameras

    def transform(self, point_clouds, **kwargs) -> torch.Tensor:
        """World -> (x_ndc, y_ndc, z_view), packed (P,3), differentiable
        (pytorch3d ``PointsRasterizer.transform`` [ext], call site rasterizer.py:614)."""
        cameras = self._cameras(kwargs)
        proj, view = camera_matrices(cameras)
        proj, view = proj.to(point_clouds.device), view.to(point_clouds.device)
        outs = []
        for n, pts in enumerate(point_clouds.points_list()):
            ph = torch.cat([pts, torch.ones_like(pts[:, :1])], dim=1)
            clip = ph @ proj[n]
            zv = ph @ view[n][:, 2]
            outs.append(torch.stack([clip[:, 0] / clip[:, 3], clip[:, 1] / clip[:, 3], zv], dim=1))
        return torch.cat(outs, dim=0) if len(outs) > 1 else outs[0]

    def _compute_h(self, point_clouds, refresh=True, **kwargs):
        """Variance scale of the reconstruction kernel (rasterizer.py:293-402):
        Vrk_invariant: per view h = clamp(mean_p(0.5 max_{6NN} d^2), 5e-5, 1e-3)          -> (N,)
        Vrk_isotropic: per point h_p = clamp(0.5 max_{6NN} d^2, 5e-5, 0.01), cached        -> (P,)"""
        rs = kwargs.get("raster_settings", self.raster_settings)
        num = point_clouds.num_points_per_cloud()
        if not (rs.Vrk_invariant or rs.Vrk_isotropic):
            raise NotImplementedError("anisotropic Vrk (curvature frames + batched SVD, rasterizer.py:256-291) "
                                      "is outside the hot path; use Vrk_invariant or Vrk_isotropic")
        if (not rs.Vrk_invariant and not refresh and self._Vrk_h is not None
                and self._Vrk_h.shape[0] == int(num.sum())):
            return self._Vrk_h
        pts_list = point_clouds.points_list()
        shared = clouds_share_points(point_clouds)
        per_cloud = []
        for n, pts in enumerate(pts_list):
            if shared and n > 0:
                per_cloud.append(per_cloud[0])
                continue
            per_cloud.append(vrk_h(pts, rs.Vrk_invariant, self.frnn_radius))
        if rs.Vrk_invariant:
            return torch.stack(per_cloud)
        self._Vrk_h = torch.cat(per_cloud)
        return self._Vrk_h

    def _get_per_point_info(self, point_clouds, **kwargs):
        """radii (P,2), ellipse_params (P,3), cutoff_threshold (P,), scaler (P,) -- rasterizer.py:525-565,
        fused into one kernel (dss_preprocess).  Also returns ``ndc`` whose z is -1 for filtered points."""
        cameras = self._cameras(kwargs)
        rs = kwargs.get("raster_settings", self.raster_settings)
        proj, view = camera_matrices(cameras)
        dev = point_clouds.device
        h = kwargs.get("Vrk_h", None)
        if h is None:
            h = self._compute_h(point_clouds, **kwargs)
        normals = point_clouds.normals_packed()
        if normals is None:
            raise ValueError("surface splatting needs point normals")
        prm = _splat_params(rs, cameras, kwargs)
        return preprocess_points(point_clouds.points_packed(), normals, proj.to(dev), view.to(dev), h.to(dev), prm,
                                 first_idx=point_clouds.cloud_to_packed_first_idx(),
                                 num_points=point_clouds.num_points_per_cloud(), shared_cloud=False)

    def _empty_fragments(self, batch_size, **kwargs):
        rs = kwargs.get("raster_settings", self.raster_settings)
        S, K = rs.image_size, rs.points_per_pixel
        dev = self.device
        return PointFragments(idx=torch.full((batch_size, S, S, K), -1, dtype=torch.long, device=dev),
                              zbuf=torch.full((batch_size, S, S, K), -1.0, device=dev),
                              qvalue=torch.full((batch_size, S, S, K), -1.0, device=dev),
                              scaler=torch.zeros((batch_size, S, S, K), device=dev),
                              occupancy=torch.zeros((batch_size, S, S), device=dev))

    def _prepare_clouds(self, point_clouds, point_clouds_filter, cameras):
        if point_clouds_filter is not None:   # activation filter (rasterizer.py:231-235)
            max_P = int(point_clouds.num_points_per_cloud().max())
            point_clouds_filter.set_filter(visibility=torch.zeros((len(point_clouds), max_P), dtype=torch.bool,
                                                                  device=point_clouds_filter.device))
            point_clouds = point_clouds_filter.filter_with(point_clouds, ("activation",))
        if cameras.R.shape[0] != len(point_clouds):
            point_clouds = point_clouds.extend(cameras.R.shape[0])
        return point_clouds

    def filter_renderable(self, point_clouds, point_clouds_filter=None, **kwargs):
        """rasterizer.py:219-254 (+ :183-217, :148-181) with the reference's COMPACTION semantics: returns
        ``(filtered_cloud, valid_mask)`` where the cloud holds, per view, only the points with
        ``znear <= z_view <= zfar`` (and, with ``backface_culling``, a view-space normal with z < 0) and ``valid_mask``
        (P,) marks them in the packed input.  The fused path does not need it (filtered points keep their slot with
        depth -1, DESIGN.md hazard 12); ``forward(..., compact_filtered=True)`` renders the compacted cloud so that
        ``idx`` indexes it exactly as in the reference."""
        rs = kwargs.get("raster_settings", self.raster_settings)
        cameras = self._cameras(kwargs)
        if point_clouds.isempty():
            return None, None
        point_clouds = self._prepare_clouds(point_clouds, point_clouds_filter, cameras)
        _, view = camera_matrices(cameras)
        view = view.to(point_clouds.device)
        znear = getattr(cameras, "znear", kwargs.get("znear", 1.0))
        zfar = getattr(cameras, "zfar", kwargs.get("zfar", 100.0))
        znear = float(torch.as_tensor(znear).reshape(-1)[0])
        zfar = float(torch.as_tensor(zfar).reshape(-1)[0])
        pts_l, nrm_l, feat_l, masks = [], [], [], []
        normals, feats = point_clouds.normals_list(), point_clouds.features_list()
        with torch.no_grad():
            for n, pts in enumerate(point_clouds.points_list()):
                zv = pts @ view[n][:3, 2] + view[n][3, 2]
                m = (zv >= znear) & (zv <= zfar)
                if rs.backface_culling and normals is not None:
                    m = m & ((normals[n] @ view[n][:3, 2]) < 0)
                masks.append(m)
        for n, pts in enumerate(point_clouds.points_list()):
            pts_l.append(pts[masks[n]])
            if normals is not None:
                nrm_l.append(normals[n][masks[n]])
            if feats is not None:
                feat_l.append(feats[n][masks[n]])
        out = point_clouds.__class__(pts_l, nrm_l if normals is not None else None, feat_l if feats is not None else None)
        return out, torch.cat(masks)

    def forward(self, point_clouds, point_clouds_filter=None, **kwargs):
        """-> (PointFragments, point_clouds[, per_point_info if verbose])  (rasterizer.py:584-664)."""
        rs = kwargs.get("raster_settings", self.raster_settings)
        cameras = self._cameras(kwargs)
        if point_clouds.isempty():
            return self._empty_fragments(cameras.R.shape[0], **kwargs), point_clouds
        if kwargs.get("compact_filtered", False):
            # the reference's index space: render the compacted clouds (the activation filter has been applied by
            # filter_renderable already; the visibility written back refers to the compacted cloud, as in the reference)
            point_clouds, _ = self.filter_renderable(point_clouds, point_clouds_filter, **kwargs)
            point_clouds_filter_for_prepare = None
        else:
            point_clouds_filter_for_prepare = point_clouds_filter
        point_clouds = self._prepare_clouds(point_clouds, point_clouds_filter_for_prepare, cameras)
        with torch.no_grad():
            info = self._get_per_point_info(point_clouds, **kwargs)
        pts_screen = self.transform(point_clouds, **kwargs)
        # filtered points: view depth -1 (the kernels skip z < 0)
        keep = info["ndc"][:, 2] >= 0
        pts_screen = torch.cat([pts_screen[:, :2], torch.where(keep, pts_screen[:, 2], info["ndc"][:, 2])[:, None]], 1)
        idx, zbuf, qvalue, occ = rasterize_elliptical_points(
            (pts_screen, point_clouds.cloud_to_packed_first_idx(), point_clouds.num_points_per_cloud()),
            info["ellipse_params"], info["cutoff_threshold"], info["radii"],
            depth_merging_threshold=rs.depth_merging_threshold, image_size=rs.image_size,
            points_per_pixel=rs.points_per_pixel, bin_size=rs.bin_size, max_points_per_bin=rs.max_points_per_bin,
            radii_backward_scaler=rs.radii_backward_scaler, clip_pts_grad=rs.clip_pts_grad)
        # scalar * exp(-0.5 Q) uses the per-fragment scaler (rasterizer.py:631-633; 0 where idx < 0)
        frag_scaler = torch.where(idx >= 0, info["scaler"][idx.clamp(min=0).long()], torch.zeros_like(qvalue))
        fragments = PointFragments(idx=idx, zbuf=zbuf, qvalue=qvalue, scaler=frag_scaler, occupancy=occ)
        if point_clouds_filter is not None:
            P = int(point_clouds.num_points_per_cloud().sum())
            vis = _C.visibility_from_idx(idx, P).bool()
            num = point_clouds.num_points_per_cloud()
            max_P = int(num.max())
            padded = torch.zeros((len(point_clouds), max_P), dtype=torch.bool, device=vis.device)
            first = point_clouds.cloud_to_packed_first_idx()
            for n in range(len(point_clouds)):
                padded[n, : int(num[n])] = vis[int(first[n]): int(first[n]) + int(num[n])]
            point_clouds_filter.set_filter(visibility=padded)
        if kwargs.get("verbose", False):
            return fragments, point_clouds, {k: info[k] for k in ("radii", "ellipse_params", "cutoff_threshold", "scaler")}
        return fragments, point_clouds


def _clip_grad(value=0.1):
    """rasterizer.py:667-673"""
    def func(grad):
        scaler = grad.norm(dim=-1, keepdim=True).clamp(0, value)
        return torch.nn.functional.normalize(grad, dim=-1) * scaler
    return func


def rasterize_elliptical_points(pcls_screen, ellipse_params, cutoff_threshold, radii,
                                depth_merging_threshold: float = 0.05, image_size: int = 512,
                                points_per_pixel: int = 5, bin_size: Optional[int] = None,
                                max_points_per_bin: Optional[int] = None, radii_backward_scaler: float = 10.0,
                                clip_pts_grad: float = -1.0):
    """rasterizer.py:681-744.  ``pcls_screen``: an object with ``points_packed() /
    cloud_to_packed_first_idx() / num_points_per_cloud()`` (as in the reference) or the tuple
    ``(points_packed, first_idx, num_points)``.  Returns ``idx, zbuf, qvalue, occupancy``."""
    if isinstance(pcls_screen, (tuple, list)):
        points_packed, first_idx, num_points = pcls_screen
    else:
        points_packed = pcls_screen.points_packed()
        first_idx = pcls_screen.cloud_to_packed_first_idx()
        num_points = pcls_screen.num_points_per_cloud()
    cutoff_threshold = cutoff_threshold.expand(points_packed.shape[0])
    if points_packed.requires_grad and clip_pts_grad is not None and clip_pts_grad > 0:
        points_packed.register_hook(_clip_grad(clip_pts_grad))
    return EllipticalRasterizer.apply(points_packed, ellipse_params, cutoff_threshold, radii, first_idx, num_points,
                                      depth_merging_threshold, image_size, points_per_pixel,
                                      bin_size if bin_size is not None else 0,
                                      max_points_per_bin if max_points_per_bin is not None else 0,
                                      radii_backward_scaler)


class EllipticalRasterizer(autograd.Function):
    """rasterizer.py:747-977.  forward = ``_C.splat_points``; backward = visibility + median search radius +
    occupancy gather + z scatter, all on the device (no FRNN grid, no ``unique()``, no ``.item()``)."""

    @staticmethod
    def forward(ctx, pts_screen, ellipse_param, cutoff_threshold, radii, cloud_to_packed_first_idx,
                num_points_per_cloud, depth_merging_threshold, image_size, points_per_pixel, bin_size: int = 0,
                max_points_per_bin: int = 0, radii_backward_scaler: float = 10.0):
        idx, zbuf, qvalue_map, occ_map = _C.splat_points(
            pts_screen, ellipse_param, cutoff_threshold.contiguous(), radii, cloud_to_packed_first_idx,
            num_points_per_cloud, depth_merging_threshold, image_size, points_per_pixel, bin_size, max_points_per_bin)
        ctx.radii_backward_scaler = radii_backward_scaler
        ctx.save_for_backward(pts_screen.detach(), radii.detach(), idx, cloud_to_packed_first_idx, num_points_per_cloud)
        ctx.mark_non_differentiable(idx)
        return idx, zbuf, qvalue_map, occ_map

    @staticmethod
    def backward(ctx, idx_grad, zbuf_grad, qvalue_grad, occ_grad):
        # qvalue_grad is received and ignored exactly as in the reference (rasterizer.py:788-813)
        pts_screen, radii, idx, first_idx, num_points = ctx.saved_tensors
        P = pts_screen.shape[0]
        dev = pts_screen.device
        grads_xy = torch.zeros((P, 2), dtype=torch.float32, device=dev)
        if occ_grad is not None:
            visible = _C.visibility_from_idx(idx, P)
            rs = _C.search_radius(radii, visible, first_idx, num_points, ctx.radii_backward_scaler)
            grads_xy = _C.occ_backward(pts_screen, radii, visible, rs, occ_grad.contiguous(), first_idx, num_points)
        grads_z = torch.zeros((P, 1), dtype=torch.float32, device=dev)
        if zbuf_grad is not None:
            _C._backward_zbuf(idx, zbuf_grad.contiguous(), grads_z)
        pts_grad = torch.cat([grads_xy, grads_z], dim=-1)
        return (pts_grad,) + (None,) * 11
