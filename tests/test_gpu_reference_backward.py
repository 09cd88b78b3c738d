"""north_star: the backward must match the reference's own CUDA kernel.  The reference's fast occupancy backward
(DSS/csrc/rasterize_points_backward.cu:30-212), driven exactly as EllipticalRasterizer.backward drives it
(DSS/core/rasterizer.py:853-972: visible-point compaction, per-view lower-median search radius, FRNN 2-D grid insert,
prefix sum, counting sort, kernel, un-sort) with the reference's own insert / counting-sort kernels on sm_100a, gave the
gradients stored in tests/golden/reference/occ_backward_fast.npz (a seeded sample of points, with the search radius and
the largest gradient; tests/golden/make_golden_reference.py).  Our gather (one C-ABI call) must give the same
gradients up to the summation order of the reference's float atomics."""
import os

import numpy as np
import pytest
import torch

from tests.util import random_screen_splats

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference", "occ_backward_fast.npz")


@pytest.mark.parametrize("S,P,seed", [(128, 4000, 1), (256, 30000, 2), (512, 100000, 3)])
def test_occ_backward_matches_reference_cuda_fast_kernel(cuda_device, S, P, seed):
    from dss_b200 import _C
    ref = np.load(GOLD)
    K, radii_s = 5, 5.0
    # keep every point inside the image: the reference kernel skips |x|,|y| > 1 (:145) and so do we, but the grid
    # extent then depends on them
    pts, ell, cut, rad, first, num = random_screen_splats(P, 1, S, seed=seed, behind_frac=0.0)
    pts[:, :2] *= 0.9
    d = cuda_device
    tp, te, tc, tr = (torch.from_numpy(x).to(d) for x in (pts, ell, cut, rad))
    tf, tn = torch.from_numpy(first).to(d), torch.from_numpy(num).to(d)
    idx, _, _, _ = _C.splat_points(tp, te, tc, tr, tf, tn, 0.05, S, K, 0, 0)
    vis = _C.visibility_from_idx(idx, P)
    assert int(vis.bool().sum()) == int(ref["S%d_visible" % S])
    g = torch.randn(1, S, S, generator=torch.Generator().manual_seed(seed)).to(d) * 1e-3
    ours_rs = _C.search_radius(tr, vis, tf, tn, radii_s)
    assert np.array_equal(ours_rs.cpu().numpy(), ref["S%d_search_radius" % S])        # exact lower median
    ours = _C.occ_backward(tp, tr, vis, ours_rs, g, tf, tn)
    rows = torch.from_numpy(ref["S%d_rows" % S].astype(np.int64)).to(d)
    want = torch.from_numpy(ref["S%d_grad" % S]).to(d)
    scale = float(ref["S%d_scale" % S])
    assert scale > 0 and torch.isfinite(want).all() and (want != 0).any()
    # the reference accumulates ~1e3 float atomics per point in arbitrary order; ours is a deterministic gather
    err = (ours[rows] - want).abs().max().item()
    assert err <= 1e-4 * scale, (err, scale)
    assert (ours[~vis.bool()] == 0).all()
