"""CPU tests: the oracle against the golden fixtures minted from the reference's own CPU code (tests/golden/*.npz and
tests/golden/reference/) and against itself (naive == binned, window == brute force, closed forms == the reference's
literal formulas)."""
import glob
import os

import numpy as np
import pytest
import torch

import oracle
from tests.util import random_screen_splats, scene

GOLDEN = sorted(p for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
                if not os.path.basename(p).startswith("knn_"))


def test_golden_files_exist():
    assert len(GOLDEN) >= 4


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_reproduces_reference_golden_vectors(path):
    """fixtures = outputs of the reference's RasterizePointsNaiveCpu / OccBackwardCpu / ZbufBackwardCpu."""
    d = np.load(path)
    S, K = int(d["S"]), int(d["K"])
    idx, zbuf, q, occ = oracle.splat_points_naive(d["points"], d["ellipse"], d["cutoff"], d["radii"], d["first"],
                                                  d["num"], 0.05, S, K, fma_mode=0, bbox_and=True)
    assert np.array_equal(idx, d["idx"])
    assert np.array_equal(zbuf, d["zbuf"])
    assert np.array_equal(q, d["qvalue"])          # no FMA contraction on either side: bit-exact
    assert np.array_equal(occ, d["occ"])
    # CUDA semantics (`||` bbox test, hazard 1) give the same fragments when radii are the exact ellipse bbox
    idx2, _, _, _ = oracle.splat_points_naive(d["points"], d["ellipse"], d["cutoff"], d["radii"], d["first"],
                                              d["num"], 0.05, S, K, fma_mode=0, bbox_and=False)
    assert (idx2 == d["idx"]).all(-1).mean() > 0.999
    gb = oracle.occ_backward_slow(d["points"], d["radii"], d["grad_occ"], d["first"], d["num"], float(d["radii_s"]),
                                  cpu_twin=True)
    np.testing.assert_allclose(gb, d["occ_backward"], rtol=1e-5, atol=1e-7)
    gz = oracle.zbuf_backward(d["idx"], d["grad_zbuf"], d["points"].shape[0])
    np.testing.assert_allclose(gz, d["zbuf_backward"], rtol=1e-5, atol=1e-6)


def test_oracle_matches_compiled_reference_cpu():
    """against what the reference's RasterizePointsNaiveCpu gave on these inputs (tests/golden/make_golden_reference.py)"""
    d = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference", "oracle_cpu_S40.npz"))
    S, K, P, N = 40, 6, 900, 3
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=9)
    r = (d["idx"].astype(np.int32), d["zbuf"], d["qvalue"], d["occ"])
    o = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K, fma_mode=0, bbox_and=True)
    for a, b in zip(r, o):
        assert a.dtype == b.dtype and np.array_equal(a, b)


@pytest.mark.parametrize("S,bin_size,P,N,K", [(64, 8, 2500, 2, 5), (50, 16, 800, 1, 3), (33, 8, 500, 2, 8)])
def test_oracle_binned_equals_naive(S, bin_size, P, N, K):
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=S)
    a = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K)
    b = oracle.splat_points_binned(pts, ell, cut, rad, first, num, 0.05, S, K, bin_size)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_oracle_edge_cases():
    S, K = 16, 4
    e = np.zeros((0, 3), np.float32)
    first, num = np.zeros(2, np.int64), np.zeros(2, np.int64)
    idx, zbuf, q, occ = oracle.splat_points_naive(e, e, np.zeros(0, np.float32), np.zeros((0, 2), np.float32), first,
                                                  num, 0.05, S, K)
    assert (idx == -1).all() and (zbuf == -1).all() and (occ == 0).all()
    # one splat at the image centre; points behind the camera are never rendered
    pts = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, -1.0]], np.float32)
    ell = np.array([[100.0, 0.0, 100.0]] * 2, np.float32)
    rad = np.full((2, 2), 0.1, np.float32)
    idx, zbuf, q, occ = oracle.splat_points_naive(pts, ell, np.ones(2, np.float32), rad, np.zeros(1, np.int64),
                                                  np.array([2], np.int64), 0.05, S, K)
    assert set(np.unique(idx)) == {-1, 0} and occ.sum() == (idx[..., 0] == 0).sum() > 0
    # depth merging: a second splat farther than the threshold is dropped, within it is kept
    pts = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 1.04], [0.0, 0.0, 1.06]], np.float32)
    ell = np.array([[100.0, 0.0, 100.0]] * 3, np.float32)
    rad = np.full((3, 2), 0.1, np.float32)
    idx, *_ = oracle.splat_points_naive(pts, ell, np.ones(3, np.float32), rad, np.zeros(1, np.int64),
                                        np.array([3], np.int64), 0.05, S, K)
    c = idx[0, S // 2, S // 2]
    assert list(c) == [0, 1, -1, -1]
    # exact z ties are ordered by id (heap of (z, idx, q) tuples: rasterize_points_cpu.cpp:87-121)
    pts[:, 2] = 1.0
    idx, *_ = oracle.splat_points_naive(pts, ell, np.ones(3, np.float32), rad, np.zeros(1, np.int64),
                                        np.array([3], np.int64), 0.05, S, 2)
    assert list(idx[0, S // 2, S // 2]) == [0, 1]


def test_occ_backward_window_equals_bruteforce():
    S, P, N, K = 48, 600, 2, 5
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=4)
    idx, *_ = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K)
    vis = oracle.visibility(idx, P)
    rs = oracle.search_radius(rad, vis, first, num, 4.0)
    g = (np.random.default_rng(0).standard_normal((N, S, S)) * 1e-3).astype(np.float32)
    g[np.random.default_rng(1).random((N, S, S)) < 0.5] = 0
    _, a = oracle.occ_backward_fast(pts, rad, vis, rs, g, first, num)
    _, b = oracle.occ_backward_fast(pts, rad, vis, rs, g, first, num, bruteforce=True)
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-15)
    assert (a[vis == 0] == 0).all() and np.abs(a).sum() > 0


def test_search_radius_is_torch_lower_median():
    rng = np.random.default_rng(3)
    P = 501
    rad = rng.random((P, 2)).astype(np.float32)
    vis = (rng.random(P) < 0.6).astype(np.uint8)
    first, num = np.array([0, 200], np.int64), np.array([200, 301], np.int64)
    rs = oracle.search_radius(rad, vis, first, num, 5.0)
    for n in range(2):
        sel = torch.from_numpy(rad[first[n]:first[n] + num[n]][vis[first[n]:first[n] + num[n]] > 0])
        assert float(sel.median() * 5.0) == float(rs[n])     # rasterizer.py:888


def test_scan_and_grid_primitives():
    a = np.random.default_rng(0).integers(0, 1000, 12345).astype(np.int32)
    out = oracle.exclusive_scan_i32(a)
    assert out[0] == 0 and np.array_equal(out[1:], np.cumsum(a)[:-1].astype(np.int32))
    pts = np.random.default_rng(1).random((1, 2000, 2)).astype(np.float32)
    lengths = np.array([2000], np.int64)
    params = np.array([[0, 0, 10.0, 10, 10, 100]], np.float32)
    cnt, cell, slot = oracle.insert_points_2d(pts, lengths, params, 100)
    assert cnt.sum() == 2000 and cell.max() < 100
    off = oracle.exclusive_scan_i32(cnt.reshape(-1)).reshape(1, 100)
    sp, si = oracle.counting_sort_2d(pts, lengths, cell, slot, off)
    assert np.array_equal(sp[0], pts[0][si[0]]) and (np.diff(cell[0][si[0]]) >= 0).all()


def test_preprocess_closed_forms_equal_the_reference_formulas():
    """The oracle uses Sk^T Sk = I - n n^T and |det(Sk J)| = sqrt(det(J^T (I - n n^T) J)); the reference draws
    Sk from a random tangent frame (rasterizer.py:337-341) and calls det/inverse on 2x2 batches.  Check the
    closed forms against that literal computation in float64, for several random frames."""
    P0, N, S = 400, 2, 128
    pts, nrm, col, proj, view, cams = scene(P0, N, seed=2)
    h = np.array([2e-4, 5e-4], np.float32)
    pre = oracle.preprocess_f64(proj.numpy(), view.numpy(), pts.numpy(), nrm.numpy(), h, 1.0, 1.0, S)
    rng = np.random.default_rng(0)
    M, p, nv = proj.numpy().astype(np.float64), pts.numpy().astype(np.float64), nrm.numpy().astype(np.float64)
    for n in range(N):
        ph = np.concatenate([p, np.ones((P0, 1))], 1)
        t = ph @ M[n][:, 3]
        xy = ph @ M[n][:, :2]
        Jk = np.zeros((P0, 4, 2))
        Jk[:, 0, 0] = Jk[:, 1, 1] = 1 / t
        Jk[:, 3, 0] = -xy[:, 0] / t ** 2
        Jk[:, 3, 1] = -xy[:, 1] / t ** 2
        WJ = np.einsum("ij,pjk->pik", M[n][:3, :], Jk)                       # (P,3,2)  rasterizer.py:494
        u0 = np.cross(nv, nv + rng.random(nv.shape))
        u0 /= np.linalg.norm(u0, axis=1, keepdims=True)
        u1 = np.cross(nv, u0)
        u1 /= np.linalg.norm(u1, axis=1, keepdims=True)
        Sk = np.stack([u0, u1], 1)                                           # (P,2,3)
        Vrk = h[n] * np.einsum("pij,pik->pjk", Sk, Sk)
        Vk = np.einsum("pji,pjk,pkl->pil", WJ, Vrk, WJ)
        GV = Vk + np.eye(2) * (2.0 / S) ** 2
        det = np.linalg.det(GV)
        inv = np.linalg.inv(GV)
        ell = np.stack([inv[:, 0, 0], inv[:, 0, 1] + inv[:, 1, 0], inv[:, 1, 1]], 1)
        detMk = np.abs(np.linalg.det(np.einsum("pij,pjk->pik", Sk, WJ)))
        scaler = detMk / np.sqrt(det * 4 * np.pi ** 2)
        den = 4 * ell[:, 0] * ell[:, 2] - ell[:, 1] ** 2
        radii = np.stack([np.sqrt(4 * ell[:, 2] / den), np.sqrt(4 * ell[:, 0] / den)], 1)
        sl = slice(n * P0, (n + 1) * P0)
        np.testing.assert_allclose(pre["ellipse"][sl], ell, rtol=5e-6, atol=1e-6)   # fp32 normals are unit to ~1e-7
        np.testing.assert_allclose(pre["radii"][sl], radii, rtol=5e-6)
        np.testing.assert_allclose(pre["scaler"][sl], scaler, rtol=5e-6, atol=2e-4 * scaler.max())  # grazing splats: det T cancels
        np.testing.assert_allclose(pre["ndc"][sl][:, :2], xy / t[:, None], rtol=1e-12)
        np.testing.assert_allclose(pre["jac"][sl], WJ, rtol=1e-10, atol=1e-12)
