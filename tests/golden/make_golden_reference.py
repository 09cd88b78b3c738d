"""Mint the witness vectors under tests/golden/reference/ from the reference's own native code (the modules
oracle/build_ref.py compiles into oracle/_ref) on the seeded inputs of the tests that compare against it:

    python -m tests.golden.make_golden_reference cpu          # reference CPU code, PLY excerpts, settings signature
    python -m tests.golden.make_golden_reference gpu [DIR]    # reference CUDA kernels (needs a B200 and libdss_b200)

The tests then compare with these files and need neither the reference checkout nor oracle/_ref.  Where the
reference's output is larger than a fixture should be, a fixed, seeded sample of pixels or points is stored, together
with the full-size quantities the assertions scale by.
"""
import inspect
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import build_ref                                  # noqa: E402
from tests.util import packed_offsets, random_screen_splats, scene   # noqa: E402

OUT = os.path.join(HERE, "reference")
PIXELS = 512         # sampled pixels per forward witness
ROWS = 512           # sampled points per backward witness
PLY_VERTICES = 1100  # vertices kept of each example cloud


def sample(n, k, seed):
    """fixed, seeded, ascending sample of k of range(n) (all of it when n <= k)"""
    if n <= k:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False)).astype(np.int64)


def sample_rows(nonzero_mask, k, seed):
    """7/8 of the sample from the rows with a non-zero gradient, the rest from all rows"""
    nz = np.nonzero(nonzero_mask)[0]
    a = nz[sample(len(nz), k - k // 8, seed)]
    b = sample(len(nonzero_mask), k // 8, seed + 1)
    return np.union1d(a, b).astype(np.int64)


def fragments_at(pix, idx, zbuf, q, occ):
    """the reference's fragments at the sampled flat pixel indices (of N*S*S)"""
    K = idx.shape[-1]
    c = lambda t, w: t.reshape(-1, w).cpu().numpy()[pix] if w else t.reshape(-1).cpu().numpy()[pix]
    return dict(idx=c(idx, K).astype(np.int32), zbuf=c(zbuf, K), qvalue=c(q, K), occ=c(occ, 0))


# ------------------------------------------------------------------------------------------------------------
# CPU: reference CPU rasterizer and FRNN brute force, example clouds, settings signature
# ------------------------------------------------------------------------------------------------------------
def truncated_ply(path, n):
    """the file's own bytes, cut to its first n vertices (binary PLY with an empty face list)"""
    b = open(path, "rb").read()
    end = b.index(b"end_header\n") + len(b"end_header\n")
    head = b[:end].decode("ascii")
    nvert = [int(h.split()[2]) for h in head.splitlines() if h.startswith("element vertex")][0]
    assert "binary_little_endian" in head and "element face 0" in head
    stride = (len(b) - end) // nvert
    assert stride * nvert == len(b) - end
    head = head.replace("element vertex %d\n" % nvert, "element vertex %d\n" % n)
    return head.encode("ascii") + b[end:end + n * stride]


def reference_settings():
    """keyword defaults of the reference's PointsRasterizationSettings and the leading parameters of
    SurfaceSplatting.forward, read from its DSS/core/rasterizer.py (imported with tests/shim)."""
    import importlib
    from tests import shim
    shim.install()
    sys.path.insert(0, build_ref.REF)
    try:
        rast = importlib.import_module("DSS.core.rasterizer")
        sig = inspect.signature(rast.PointsRasterizationSettings.__init__)
        params = {k: p.default for k, p in sig.parameters.items() if k != "self"}
        forward = list(inspect.signature(rast.SurfaceSplatting.forward).parameters)
    finally:
        sys.path.remove(build_ref.REF)
        shim.uninstall()
    for v in params.values():
        assert v is None or isinstance(v, (bool, int, float, str)), params
    return {"PointsRasterizationSettings": params, "SurfaceSplatting.forward": forward}


def make_cpu():
    ref = build_ref.ref_cpu()
    frnn = build_ref.ref_frnn_cpu()
    assert ref is not None and frnn is not None, "needs the reference's CPU modules (oracle/build_ref.py)"
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    # tests/test_oracle.py::test_oracle_matches_compiled_reference_cpu
    S, K, P, N = 40, 6, 900, 3
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=9)
    idx, zbuf, q, occ = ref.splat_points_naive_cpu(t(pts), t(ell), t(cut), t(rad), t(first), t(num), 0.05, S, K)
    np.savez_compressed(os.path.join(OUT, "oracle_cpu_S40.npz"), idx=idx.numpy().astype(np.int16), zbuf=zbuf.numpy(),
                        qvalue=q.numpy(), occ=occ.numpy())
    # tests/test_knn.py::test_oracle_knn_matches_compiled_reference_witness
    rng = np.random.default_rng(3)
    p1 = rng.uniform(-1, 1, (2, 300, 3)).astype(np.float32)
    p2 = rng.uniform(-1, 1, (2, 400, 3)).astype(np.float32)
    l1, l2 = np.array([300, 180], np.int64), np.array([400, 250], np.int64)
    idxs, dists = frnn.frnn_bf_cpu(t(p1), t(p2), t(l1), t(l2), 5, 0.4)
    np.savez_compressed(os.path.join(OUT, "knn_bruteforce_ragged.npz"),
                        dists=np.concatenate([dists[0, :300].numpy(), dists[1, :180].numpy()]),
                        idxs=np.concatenate([idxs[0, :300].numpy(), idxs[1, :180].numpy()]).astype(np.int32))
    # tests/test_io.py::test_reads_the_reference_example_clouds
    os.makedirs(os.path.join(OUT, "pointclouds"), exist_ok=True)
    for name in ("teapot_normal_dense", "bunny-8000", "sphere_2k"):
        src = os.path.join(build_ref.REF, "example_data", "pointclouds", name + ".ply")
        with open(os.path.join(OUT, "pointclouds", name + ".ply"), "wb") as f:
            f.write(truncated_ply(src, PLY_VERTICES))
    # tests/test_reference_factory.py::test_reference_settings_class_has_the_same_keywords_as_ours
    with open(os.path.join(OUT, "rasterizer_signature.json"), "w") as f:
        json.dump(reference_settings(), f, indent=1, sort_keys=True)
        f.write("\n")


# ------------------------------------------------------------------------------------------------------------
# GPU: reference CUDA kernels
# ------------------------------------------------------------------------------------------------------------
def reference_fast_backward(ref, pts, radii, vis, grad_occ, radii_s):
    """The reference's fast occupancy backward (DSS/csrc/rasterize_points_backward.cu:30-212) driven for one view as
    EllipticalRasterizer.backward drives it (DSS/core/rasterizer.py:853-972: visible-point compaction, lower-median
    search radius, FRNN 2-D grid insert, prefix sum, counting sort, kernel, un-sort).  pts (P,3), radii (P,2),
    vis (P,) bool, grad_occ (1,S,S), all CUDA tensors.  Returns (grad of the visible points (Pv,2), search radius (1,))."""
    dev = pts.device
    pv, rv = pts[vis].contiguous(), radii[vis].contiguous()
    Pv = pv.shape[0]
    num = torch.tensor([Pv], dtype=torch.int64, device=dev)
    first = torch.zeros(1, dtype=torch.int64, device=dev)
    rs = (rv.reshape(-1).median() * radii_s).reshape(1).float()                      # rasterizer.py:888
    p2d = pv[None, :, :2].clone().contiguous()
    gmin, gmax = p2d[0].min(0)[0], p2d[0].max(0)[0]                                   # :894-896
    size = gmax - gmin
    cell = float(rs.item()) / 2                                                       # RADIUS_CELL_RATIO = 2
    if cell < float(size.min()) / 1024:
        cell = float(size.min()) / 1024
    params = torch.zeros((1, 6), dtype=torch.float32, device=dev)
    params[0, :2] = gmin
    params[0, 2] = 1.0 / cell
    params[0, 3:5] = torch.floor(size / cell) + 1
    params[0, 5] = params[0, 3] * params[0, 4]
    G = int(params[0, 5].item())
    cnt = torch.zeros((1, G), dtype=torch.int32, device=dev)
    cellid = torch.full((1, Pv), -1, dtype=torch.int32, device=dev)
    slot = torch.full((1, Pv), -1, dtype=torch.int32, device=dev)
    ref.insert_points_cuda(p2d, num, params, cnt, cellid, slot, G)                    # :909
    off = (torch.cumsum(cnt, 1) - cnt).to(torch.int32).contiguous()                   # exclusive prefix sum (:913-915)
    sorted2d = torch.zeros((1, Pv, 2), dtype=torch.float32, device=dev)
    sorted_idx = torch.full((1, Pv), -1, dtype=torch.int32, device=dev)
    ref.counting_sort_cuda(p2d, num, cellid, slot, off, sorted2d, sorted_idx)         # :921-929
    order = sorted_idx[0].long()
    pts_sorted, radii_sorted = pv[order].contiguous(), rv[order].contiguous()
    g_sorted = ref.splat_points_occ_fast_cuda_backward(pts_sorted, radii_sorted, rs, grad_occ.contiguous(), num, first,
                                                       off, params)                  # :950-951
    g = torch.zeros_like(g_sorted)
    g[order] = g_sorted                                                               # :958
    return g, rs


def _forward_witnesses(ref, ndc, ell, cut, rad, first, num, S, K, coarse_fine, bin_size, max_per_bin, pix):
    """naive (and coarse-to-fine) reference fragments at `pix`; the second set is kept only where it differs"""
    out = fragments_at(pix, *ref.splat_points_naive_cuda(ndc, ell, cut, rad, first, num, 0.05, S, K))
    if coarse_fine:
        bins = ref.rasterize_coarse_cuda(ndc, rad, first, num, S, bin_size, max_per_bin)
        f = fragments_at(pix, *ref.rasterize_fine_cuda(ndc, ell, cut, rad, bins, 0.05, S, bin_size, K))
        del bins
        if all(np.array_equal(out[k], f[k]) for k in out):
            out["coarse_fine_equals_naive"] = np.array(True)
        else:
            out.update({"fine_" + k: v for k, v in f.items()})
            out["coarse_fine_equals_naive"] = np.array(False)
    return out


def gpu_ops(ref, dev, out):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    res = {}
    # test_coarse_bins_match_reference_cuda: per bin, the ascending ids the reference's dense bin list holds
    S, bin_size, P, N = 256, 16, 8000, 2
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=7, ragged=False)
    dense = ref.rasterize_coarse_cuda(*[t(x) for x in (pts, rad, first, num)], S, bin_size, 10000).cpu().numpy()
    valid = dense >= 0
    assert (dense[~valid] == -1).all()
    res["coarse_counts"] = valid.sum(-1).reshape(-1).astype(np.int32)
    res["coarse_ids"] = np.concatenate([np.sort(r[r >= 0]) for r in dense.reshape(-1, dense.shape[-1])]).astype(np.int16)
    # test_splat_points_matches_reference_cuda
    S, P, N, K = 256, 20000, 2, 5
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=3, ragged=False)
    pix = sample(N * S * S, PIXELS, 301)
    w = _forward_witnesses(ref, *[t(x) for x in (pts, ell, cut, rad, first, num)], S, K, True, 16, max(10000, P), pix)
    res.update({"splat_pix": pix.astype(np.int32)}, **{"splat_" + k: v for k, v in w.items()})
    # test_slow_occ_backward_matches_oracle_and_reference_cuda
    for S, P, N, radii_s in ((96, 3000, 2, 2.0), (128, 5000, 3, 3.5)):
        pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=S + N)
        rng = np.random.default_rng(S)
        g = (rng.standard_normal((N, S, S)) * 1e-3).astype(np.float32)
        g[rng.random((N, S, S)) < 0.3] = 0.0
        r = ref.splat_points_occ_backward_cuda(t(pts), t(rad), t(g), t(first), t(num), radii_s, 0.05).cpu().numpy()
        rows = sample_rows((r != 0).any(1), ROWS, S)
        res["slow_S%d_rows" % S] = rows.astype(np.int32)
        res["slow_S%d_grad" % S] = r[rows]
    np.savez_compressed(os.path.join(out, "gpu_ops.npz"), **res)


def occ_backward(ref, dev, out):
    """tests/test_gpu_reference_backward.py"""
    from dss_b200 import _C
    res = {}
    for S, P, seed in ((128, 4000, 1), (256, 30000, 2), (512, 100000, 3)):
        K, radii_s = 5, 5.0
        pts, ell, cut, rad, first, num = random_screen_splats(P, 1, S, seed=seed, behind_frac=0.0)
        pts[:, :2] *= 0.9
        tp, te, tc, tr = (torch.from_numpy(x).to(dev) for x in (pts, ell, cut, rad))
        tf, tn = torch.from_numpy(first).to(dev), torch.from_numpy(num).to(dev)
        idx, _, _, _ = _C.splat_points(tp, te, tc, tr, tf, tn, 0.05, S, K, 0, 0)
        vis = _C.visibility_from_idx(idx, P).bool()
        g = torch.randn(1, S, S, generator=torch.Generator().manual_seed(seed)).to(dev) * 1e-3
        want_vis, rs = reference_fast_backward(ref, tp, tr, vis, g, radii_s)
        want = torch.zeros(P, 2, device=dev)
        want[vis] = want_vis
        want = want.cpu().numpy()
        rows = sample_rows(vis.cpu().numpy(), ROWS, seed)
        res["S%d_visible" % S] = np.array(int(vis.sum()))
        res["S%d_search_radius" % S] = rs.cpu().numpy()
        res["S%d_scale" % S] = np.array(float(want_vis.abs().max()), np.float32)
        res["S%d_rows" % S] = rows.astype(np.int32)
        res["S%d_grad" % S] = want[rows]
    np.savez_compressed(os.path.join(out, "occ_backward_fast.npz"), **res)


def _jacobian_f64(pts, proj):
    """d ndc_xy / d world (N,P0,3,2) in float64 (rasterizer.py:443-496 without the eps clamps)."""
    p = torch.cat([pts.double(), torch.ones_like(pts[:, :1]).double()], 1)
    M = proj.double()
    x, y, t = (p @ M[:, :, 0].T).T, (p @ M[:, :, 1].T).T, (p @ M[:, :, 3].T).T
    J = torch.empty(M.shape[0], p.shape[0], 3, 2, dtype=torch.float64, device=pts.device)
    for k in range(3):
        J[:, :, k, 0] = M[:, k, 0, None] / t - M[:, k, 3, None] * x / (t * t)
        J[:, :, k, 1] = M[:, k, 1, None] / t - M[:, k, 3, None] * y / (t * t)
    return J


def baseline_parity(ref, dev, out):
    """tests/test_gpu_baseline_parity.py: the reference's kernels on the fused renderer's own per-splat records"""
    from dss_b200.ops import SplatParams, render_points
    for tag, P0, N, S, K, seed, coarse_fine in (("c2", 100_000, 8, 512, 5, 2, True), ("headline", 1_000_000, 2, 512, 5, 0, False),
                                                ("k8", 300_000, 2, 512, 8, 3, False)):
        pts, nrm, col, proj, view, _ = scene(P0, N, seed=seed)
        prm = SplatParams(image_size=S, points_per_pixel=K, znear=0.1, clip_pts_grad=-1.0, radii_backward_scaler=5.0)
        h = torch.full((N,), 5e-5 if P0 >= 500_000 else 2e-4, device=dev)
        p = pts.to(dev).requires_grad_(True)
        o = render_points(p, nrm.to(dev), col.to(dev).requires_grad_(True), proj.to(dev), view.to(dev), h, prm, return_fragments=True)
        rec = o.records
        first, num = (x.to(dev) for x in packed_offsets(N, P0))
        ndc, ell, rad = rec[:, :3].contiguous(), rec[:, 5:8].contiguous(), rec[:, 3:5].contiguous()
        cut = torch.ones(N * P0, device=dev)
        pix = sample(N * S * S, PIXELS, seed + 11)
        res = {"pix": pix.astype(np.int32)}
        res.update(_forward_witnesses(ref, ndc, ell, cut, rad, first, num, S, K, coarse_fine, 32, max(10000, P0), pix))
        g = torch.randn(N, S, S, 4, generator=torch.Generator().manual_seed(seed + 5)).to(dev) * 1e-3
        vis = o.visible.view(N, P0).bool()
        J = _jacobian_f64(p.detach(), proj.to(dev))
        want = torch.zeros(P0, 3, dtype=torch.float64, device=dev)
        gnd_all = torch.zeros(N * P0, 2, device=dev)
        for n in range(N):
            sl = slice(n * P0, (n + 1) * P0)
            g_vis, _ = reference_fast_backward(ref, ndc[sl], rad[sl], vis[n], g[n:n + 1, :, :, 3].contiguous(), 5.0)
            gn = torch.zeros(P0, 2, dtype=torch.float64, device=dev)
            gn[vis[n]] = g_vis.double()
            gnd_all[sl] = gn.float()
            want += torch.einsum("pkj,pj->pk", J[n], gn)
        want, gnd_all = want.cpu().numpy(), gnd_all.cpu().numpy()
        rows = sample_rows((want != 0).any(1), ROWS, seed + 21)
        rows_ndc = sample_rows((gnd_all != 0).any(1), ROWS, seed + 31)
        res.update(grad_rows=rows.astype(np.int32), grad_world=want[rows].astype(np.float32),
                   grad_world_scale=np.abs(want).max(), ndc_rows=rows_ndc.astype(np.int32), grad_ndc=gnd_all[rows_ndc],
                   grad_ndc_scale=np.abs(gnd_all).max())
        np.savez_compressed(os.path.join(out, "baseline_parity_%s.npz" % tag), **res)
        del o, rec, ndc, ell, rad, J
        torch.cuda.empty_cache()


def make_gpu(out):
    ref = build_ref.ref_cuda()
    assert ref is not None, "needs the reference's CUDA module (oracle/build_ref.py)"
    dev = torch.device("cuda:0")
    os.makedirs(out, exist_ok=True)
    gpu_ops(ref, dev, out)
    occ_backward(ref, dev, out)
    baseline_parity(ref, dev, out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if sys.argv[1] == "cpu":
        make_cpu()
    else:
        make_gpu(sys.argv[2] if len(sys.argv) > 2 else OUT)
    print("wrote", sorted(os.listdir(sys.argv[2] if len(sys.argv) > 2 else OUT)))
