"""GPU parity tests of the _C-level operators (called through the C ABI) against the CPU oracle and against what the
reference's own CUDA kernels gave on the same inputs (tests/golden/reference/gpu_ops.npz, minted by
tests/golden/make_golden_reference.py; large outputs as a seeded sample of pixels or points)."""
import os

import numpy as np
import pytest
import torch

import oracle
from tests.util import random_screen_splats

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference", "gpu_ops.npz")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _rim_mask(q, cutoff_at_idx):
    """pixels whose fragments sit within a few ulp of the cutoff (FMA contraction can flip them)."""
    return np.abs(q - cutoff_at_idx) <= 8 * np.spacing(np.abs(cutoff_at_idx).astype(np.float32))


@pytest.mark.parametrize("n", [0, 1, 5, 2048, 2049, 10000, 1 << 20])
def test_exclusive_scan_matches_oracle(cuda_device, n):
    from dss_b200.prefix_sum import prefix_sum_cuda
    rng = np.random.default_rng(n)
    a = rng.integers(0, 1000, size=max(n, 1)).astype(np.int32)
    src = _t(a, cuda_device)
    out = torch.full_like(src, -7)
    prefix_sum_cuda(src, n, out)
    want = oracle.exclusive_scan_i32(a[:n]) if n else np.zeros(0, np.int32)
    assert np.array_equal(out.cpu().numpy()[:n], want)
    if n < a.size:
        assert out[n:].eq(-7).all()           # untouched past n
    # in place, reference test (external/prefix_sum/test.py:5-26): values < 1000, random length
    prefix_sum_cuda(src, n, src)
    assert np.array_equal(src.cpu().numpy()[:n], want)


@pytest.mark.parametrize("S,bin_size,P,N", [(64, 8, 3000, 2), (256, 16, 20000, 3), (512, 32, 50000, 2), (100, 16, 2000, 1)])
def test_coarse_bins_bit_exact(cuda_device, S, bin_size, P, N):
    from dss_b200 import _C
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=S)
    off, ids = _C._rasterize_coarse_csr(_t(pts, cuda_device), _t(rad, cuda_device), _t(first, cuda_device),
                                        _t(num, cuda_device), S, bin_size)
    off, ids = off.cpu().numpy().astype(np.int64), ids.cpu().numpy()
    woff, wids = oracle.rasterize_coarse(pts, rad, first, num, S, bin_size)
    assert np.array_equal(off, woff)
    # order inside a bin is unspecified (as in the reference): compare sorted sets
    got = np.concatenate([np.sort(ids[off[b]:off[b + 1]]) for b in range(len(off) - 1)]) if len(ids) else ids
    assert np.array_equal(got, wids)


def test_coarse_bins_match_reference_cuda(cuda_device):
    from dss_b200 import _C
    ref = np.load(GOLD)
    S, bin_size, P, N = 256, 16, 8000, 2
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=7, ragged=False)
    args = [_t(x, cuda_device) for x in (pts, rad, first, num)]
    dense = _C._rasterize_coarse(*args, S, bin_size, 10000).cpu().numpy()
    # the reference's dense bin lists (-1 padded), rebuilt from the stored ascending ids of every bin
    counts, ids = ref["coarse_counts"], ref["coarse_ids"].astype(np.int32)
    dense_ref = np.full((counts.size, dense.shape[-1]), -1, np.int32)
    ends = np.cumsum(counts)
    for b, (n, e) in enumerate(zip(counts, ends)):
        dense_ref[b, dense_ref.shape[1] - n:] = ids[e - n:e]
    dense_ref = dense_ref.reshape(dense.shape)
    assert np.array_equal(np.sort(dense_ref, axis=-1), np.sort(dense, axis=-1))


@pytest.mark.parametrize("S,P,N,K", [(64, 1500, 2, 5), (128, 6000, 3, 8), (96, 800, 1, 1), (64, 3000, 1, 12),
                                     (64, 2000, 1, 20)])
def test_splat_points_matches_oracle(cuda_device, S, P, N, K):
    from dss_b200 import _C
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=K)
    idx, zbuf, q, occ = _C.splat_points(*[_t(x, cuda_device) for x in (pts, ell, cut, rad, first, num)],
                                        0.05, S, K, 0, 0)
    widx, wz, wq, wocc = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K, fma_mode=1)
    idx, zbuf, q, occ = idx.cpu().numpy(), zbuf.cpu().numpy(), q.cpu().numpy(), occ.cpu().numpy()
    same = (idx == widx).all(-1)
    if not same.all():
        # the only admissible differences are rim fragments (|q - cutoff| within a few ulp)
        bad = ~same
        ok = np.zeros_like(bad)
        for (a, b) in ((idx, q), (widx, wq)):
            c = np.where(a >= 0, cut[np.maximum(a, 0)], np.inf)
            ok |= (_rim_mask(b, c) & (a >= 0)).any(-1)
        assert (ok | ~bad).all(), "idx differs at %d non-rim pixels" % int((bad & ~ok).sum())
        assert bad.mean() < 1e-3
    assert np.array_equal(zbuf[same], wz[same])
    np.testing.assert_allclose(q[same], wq[same], rtol=1e-5, atol=1e-6)
    assert np.array_equal(occ[same], wocc[same])


def test_splat_points_matches_reference_cuda(cuda_device):
    """north_star: outputs must match the reference's own DSS/csrc kernels on identical inputs (at the sampled pixels)."""
    from dss_b200 import _C
    ref = np.load(GOLD)
    S, P, N, K = 256, 20000, 2, 5
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=3, ragged=False)
    args = [_t(x, cuda_device) for x in (pts, ell, cut, rad, first, num)]
    pix = _t(ref["splat_pix"].astype(np.int64), cuda_device)
    idx, zbuf, q, occ = _C.splat_points(*args, 0.05, S, K, 16, 0)
    idx, zbuf, q = (x.reshape(-1, K)[pix] for x in (idx, zbuf, q))
    occ = occ.reshape(-1)[pix]
    # the naive kernel and the coarse-to-fine path (bin 16); the latter is stored only where it differs
    witness = lambda pre: tuple(_t(ref[pre + k], cuda_device) for k in ("idx", "zbuf", "qvalue", "occ"))
    witnesses = [witness("splat_")]
    if not bool(ref["splat_coarse_fine_equals_naive"]):
        witnesses.append(witness("splat_fine_"))
    for (a_idx, a_z, a_q, a_occ) in witnesses:
        same = (a_idx == idx).all(-1)
        assert same.float().mean().item() > 0.9999
        assert torch.equal(a_z[same], zbuf[same])
        assert torch.equal(a_q[same], q[same])        # same compiler, same expression tree: bit-exact q
        assert torch.equal(a_occ[same], occ[same])


def test_visibility_and_search_radius(cuda_device):
    from dss_b200 import _C
    S, P, N, K = 128, 5000, 3, 5
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=11)
    widx, _, _, _ = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K, fma_mode=1)
    vis = _C.visibility_from_idx(_t(widx, cuda_device), P)
    wvis = oracle.visibility(widx, P)
    assert np.array_equal(vis.cpu().numpy(), wvis)
    rs = _C.search_radius(_t(rad, cuda_device), vis, _t(first, cuda_device), _t(num, cuda_device), 5.0)
    wrs = oracle.search_radius(rad, wvis, first, num, 5.0)
    assert np.array_equal(rs.cpu().numpy(), wrs)       # exact order statistic
    # torch.median (lower median of the flattened radii) is what the reference calls (rasterizer.py:888)
    for n in range(N):
        sel = torch.from_numpy(rad[first[n]:first[n] + num[n]][wvis[first[n]:first[n] + num[n]] > 0])
        if sel.numel():
            assert float(sel.median() * 5.0) == float(wrs[n])


@pytest.mark.parametrize("dense", [True, False])
def test_occ_backward_matches_oracle(cuda_device, dense):
    from dss_b200 import _C
    S, P, N, K = 128, 4000, 2, 5
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=21)
    pts[:50, 0] = 1.5  # some points outside the renderable area
    widx, _, _, _ = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K, fma_mode=1)
    vis = oracle.visibility(widx, P)
    rs = oracle.search_radius(rad, vis, first, num, 5.0)
    rng = np.random.default_rng(5)
    g = (rng.standard_normal((N, S, S)) * 1e-3).astype(np.float32)
    if not dense:
        g[rng.random((N, S, S)) < 0.7] = 0.0
    out = _C.occ_backward(_t(pts, cuda_device), _t(rad, cuda_device), _t(vis, cuda_device), _t(rs, cuda_device),
                          _t(g, cuda_device), _t(first, cuda_device), _t(num, cuda_device)).cpu().numpy()
    g32, g64 = oracle.occ_backward_fast(pts, rad, vis, rs, g, first, num)
    scale = np.abs(g64).max()
    # fp32 sums of up to ~1e3 signed terms: compare with the fp64 arbiter, tolerance relative to the scale
    assert np.abs(out - g64).max() <= 2e-5 * scale + 1e-9
    assert np.abs(out - g64).max() <= 4 * np.abs(g32 - g64).max() + 1e-6 * scale
    assert (out[vis == 0] == 0).all()
    # drop-in signature: sorted points + grid arguments are accepted and ignored
    sel = np.nonzero(vis)[0]
    num_v = np.array([((sel >= first[n]) & (sel < first[n] + num[n])).sum() for n in range(N)], np.int64)
    first_v = np.concatenate([[0], np.cumsum(num_v)[:-1]]).astype(np.int64)
    out2 = _C._splat_points_occ_fast_cuda_backward(_t(pts[sel], cuda_device), _t(rad[sel], cuda_device),
                                                   _t(rs, cuda_device), _t(g, cuda_device),
                                                   _t(num_v, cuda_device), _t(first_v, cuda_device), None, None)
    # (the two calls may take different kernels -- staged tile windows vs the direct gather, chosen from the previous
    #  call's radii -- so compare to rounding, not bit for bit)
    np.testing.assert_allclose(out2.cpu().numpy(), out[sel], rtol=2e-5, atol=2e-6 * scale)


def test_zbuf_backward(cuda_device):
    from dss_b200 import _C
    S, P, N, K = 64, 1000, 2, 5
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=31)
    widx, _, _, _ = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K, fma_mode=1)
    rng = np.random.default_rng(6)
    gz = rng.standard_normal(widx.shape).astype(np.float32)
    gz[rng.random(widx.shape) < 0.3] = 0
    zg = torch.zeros(P, 1, device=cuda_device)
    assert _C._backward_zbuf(_t(widx, cuda_device), _t(gz, cuda_device), zg) is None
    want = oracle.zbuf_backward(widx, gz, P)
    np.testing.assert_allclose(zg.cpu().numpy()[:, 0], want, rtol=1e-5, atol=1e-6)


def test_grid_insert_and_counting_sort(cuda_device):
    """external/FRNN/tests/frnn_validation_2D_simple.py:22-35: sorted points == gather by sorted idx."""
    from dss_b200 import frnn_grid
    from dss_b200.prefix_sum import prefix_sum_cuda
    N, P = 2, 10000
    rng = np.random.default_rng(8)
    pts = rng.random((N, P, 2)).astype(np.float32)
    lengths = np.array([P, P - 777], np.int64)
    cell = 0.05
    params = np.zeros((N, 6), np.float32)
    for n in range(N):
        mn = pts[n, :lengths[n]].min(0)
        mx = pts[n, :lengths[n]].max(0)
        res = np.floor((mx - mn) / cell) + 1
        params[n] = [mn[0], mn[1], 1 / cell, res[0], res[1], res[0] * res[1]]
    G = int(params[:, 5].max())
    cnt = torch.zeros((N, G), dtype=torch.int32, device=cuda_device)
    gcell = torch.full((N, P), -1, dtype=torch.int32, device=cuda_device)
    gidx = torch.full((N, P), -1, dtype=torch.int32, device=cuda_device)
    frnn_grid.insert_points_cuda(_t(pts, cuda_device), _t(lengths, cuda_device), _t(params, cuda_device), cnt, gcell, gidx, G)
    wcnt, wcell, _ = oracle.insert_points_2d(pts, lengths, params, G)
    assert np.array_equal(cnt.cpu().numpy(), wcnt)
    assert np.array_equal(gcell.cpu().numpy(), wcell)
    off = torch.zeros_like(cnt)
    for n in range(N):
        prefix_sum_cuda(cnt[n], int(params[n, 5]), off[n])
    sp = torch.zeros((N, P, 2), device=cuda_device)
    si = torch.full((N, P), -1, dtype=torch.int32, device=cuda_device)
    frnn_grid.counting_sort_cuda(_t(pts, cuda_device), _t(lengths, cuda_device), gcell, gidx, off, sp, si)
    sp, si = sp.cpu().numpy(), si.cpu().numpy()
    for n in range(N):
        L = lengths[n]
        assert np.array_equal(np.sort(si[n, :L]), np.arange(L))
        assert np.array_equal(sp[n, :L], pts[n][si[n, :L]])
        assert (np.diff(wcell[n][si[n, :L]]) >= 0).all()      # cells ascending


@pytest.mark.parametrize("S,P,rad_px,expect", [
    (96, 3000, (0.8, 4.0), "4 lanes/splat, table-driven rows (S not a power of two)"),
    (256, 6000, (2.0, 5.0), "8 lanes x 3 pairs"),
    (256, 6000, (1.8, 4.2), "around the 4 lanes x 5 pairs mapping (33..40 columns)"),
    (256, 6000, (2.2, 4.4), "around the 4 lanes x 5 pairs mapping (33..40 columns)"),
    (200, 5000, (4.0, 7.0), "8 lanes x 4 pairs, S not a power of two"),
    (256, 5000, (6.0, 9.0), "16 lanes x 3 pairs"),
    (256, 3000, (9.0, 13.0), "window larger than the staged box: direct gather"),
])
def test_occ_backward_window_variants(cuda_device, S, P, rad_px, expect):
    """every lane mapping of the tile kernel (the window width follows the search radius), power-of-two and other image
    sizes, and the direct-gather kernel for windows that do not fit -- each against the float64 oracle.  The staged box
    is sized from the previous call's radii, so the first call of a size may take the direct gather and the second the
    tile kernel: both must be right."""
    from dss_b200 import _C
    N, K = 2, 5
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=S + P, rad_px=rad_px)
    widx, _, _, _ = oracle.splat_points_naive(pts, ell, cut, rad, first, num, 0.05, S, K, fma_mode=1)
    vis = oracle.visibility(widx, P)
    rs = oracle.search_radius(rad, vis, first, num, 5.0)
    g = (np.random.default_rng(S).standard_normal((N, S, S)) * 1e-3).astype(np.float32)
    g32, g64 = oracle.occ_backward_fast(pts, rad, vis, rs, g, first, num)
    scale = np.abs(g64).max()
    args = [_t(x, cuda_device) for x in (pts, rad, vis, rs, g, first, num)]
    for attempt in range(2):
        out = _C.occ_backward(*args).cpu().numpy()
        assert np.abs(out - g64).max() <= 2e-5 * scale + 1e-9, (expect, attempt, np.abs(out - g64).max() / scale)
        assert (out[vis == 0] == 0).all()


@pytest.mark.parametrize("S,P,N,radii_s", [(96, 3000, 2, 2.0), (128, 5000, 3, 3.5)])
def test_slow_occ_backward_matches_oracle_and_reference_cuda(cuda_device, S, P, N, radii_s):
    """A17: the reference's slow occupancy backward (rasterize_points.cu:673-821; rectangular window, every renderable
    point), disabled in the reference but part of its native surface: our gather vs the oracle's restatement and vs the
    reference's own CUDA kernel on a sample of points (float atomics in arbitrary order there)."""
    from dss_b200 import _C
    pts, ell, cut, rad, first, num = random_screen_splats(P, N, S, seed=S + N)
    rng = np.random.default_rng(S)
    g = (rng.standard_normal((N, S, S)) * 1e-3).astype(np.float32)
    g[rng.random((N, S, S)) < 0.3] = 0.0
    d = cuda_device
    out = _C._splat_points_occ_backward(_t(pts, d), _t(rad, d), _t(g, d), _t(first, d), _t(num, d), radii_s, 0.05)
    want = oracle.occ_backward_slow(pts, rad, g, first, num, radii_s, cpu_twin=False)
    scale = np.abs(want).max()
    assert scale > 0
    assert np.abs(out.cpu().numpy() - want).max() <= 1e-4 * scale
    # points behind the camera or outside the image get nothing (rasterize_points.cu:719)
    dead = (pts[:, 2] < 0) | (np.abs(pts[:, 0]) > 1) | (np.abs(pts[:, 1]) > 1)
    assert dead.any() and (out.cpu().numpy()[dead] == 0).all()
    ref = np.load(GOLD)
    rows = ref["slow_S%d_rows" % S].astype(np.int64)
    assert np.abs(out.cpu().numpy()[rows] - ref["slow_S%d_grad" % S]).max() <= 1e-4 * scale
