"""K nearest neighbours within a radius (SURVEY.md section 8(f) row 1).

CPU: the oracle's brute force against golden vectors minted from the reference's own ground truth FRNNBruteForceCPU
(tests/golden/make_golden_knn.py, tests/golden/make_golden_reference.py).
GPU: the grid kernel (through the C ABI) against the oracle, bit for bit -- distances AND indices, ties included --
plus size-independent properties at 1M points."""
import os

import numpy as np
import pytest
import torch

import oracle

GOLD = os.path.join(os.path.dirname(__file__), "golden", "knn_frnn_bruteforce.npz")
CASES = [("k7_r0.2", 7, 0.2), ("k12_r0.05", 12, 0.05)]


def _clouds(d):
    return sorted(k[:-len("__points")] for k in d.files if k.endswith("__points"))


def test_oracle_knn_reproduces_reference_bruteforce_golden_vectors():
    d = np.load(GOLD)
    assert len(_clouds(d)) >= 4
    for name in _clouds(d):
        p = d[name + "__points"]
        f, n = np.zeros(1, np.int64), np.array([len(p)], np.int64)
        for tag, K, r in CASES:
            dist, idx = oracle.knn_brute(p, f, n, p, f, n, K, r)
            assert np.array_equal(dist, d["%s__%s__dists" % (name, tag)]), (name, tag)   # same sums, same order: bit-exact
            assert np.array_equal(idx, d["%s__%s__idxs" % (name, tag)]), (name, tag)     # ties resolved like the reference
    # the small radius leaves some lists short (-1 padding exercised), the self match is always first
    short = d["teapot_normal_dense__k12_r0.05__idxs"]
    assert (short[:, -1] == -1).any() and (short[:, 0] == np.arange(len(short))).all()


def test_oracle_knn_matches_compiled_reference_witness():
    """against what the reference's FRNNBruteForceCPU gave for two ragged clouds (queries and points of different
    lengths), stored as the valid rows of each cloud back to back"""
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference", "knn_bruteforce_ragged.npz"))
    rng = np.random.default_rng(3)
    p1 = rng.uniform(-1, 1, (2, 300, 3)).astype(np.float32)      # queries != points, two clouds of different length
    p2 = rng.uniform(-1, 1, (2, 400, 3)).astype(np.float32)
    l1, l2 = np.array([300, 180], np.int64), np.array([400, 250], np.int64)
    q = np.concatenate([p1[0, :300], p1[1, :180]])
    pts = np.concatenate([p2[0, :400], p2[1, :250]])
    dist, idx = oracle.knn_brute(q, np.array([0, 300]), l1, pts, np.array([0, 400]), l2, 5, 0.4)
    assert np.array_equal(dist, ref["dists"])
    assert np.array_equal(idx, ref["idxs"])


# ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_knn_kernel_matches_golden_and_oracle(cuda_device):
    from dss_b200.frnn_grid import knn_points_packed
    d = np.load(GOLD)
    for name in _clouds(d):
        p = torch.from_numpy(d[name + "__points"]).to(cuda_device)
        f = torch.zeros(1, dtype=torch.int64, device=cuda_device)
        n = torch.tensor([p.shape[0]], dtype=torch.int64, device=cuda_device)
        for tag, K, r in CASES:
            dist, idx = knn_points_packed(p, f, n, K, r)
            assert np.array_equal(dist.cpu().numpy(), d["%s__%s__dists" % (name, tag)]), (name, tag)
            assert np.array_equal(idx.cpu().numpy(), d["%s__%s__idxs" % (name, tag)]), (name, tag)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,P,K,r", [("sphere", 20000, 7, 0.2), ("cube", 15000, 16, 0.1), ("line", 5000, 7, -1.0),
                                        ("tiny", 5, 7, 0.2), ("clustered", 12000, 32, 0.3)])
def test_knn_kernel_matches_oracle_ragged_batches(cuda_device, kind, P, K, r):
    from dss_b200.frnn_grid import knn_points_packed
    rng = np.random.default_rng(len(kind) + P)
    if kind == "sphere":
        x = rng.standard_normal((P, 3)); x = 0.5 * x / np.linalg.norm(x, axis=1, keepdims=True)
    elif kind == "cube":
        x = rng.uniform(-0.5, 0.5, (P, 3))
    elif kind == "line":
        x = np.stack([np.linspace(-1, 1, P), np.zeros(P), np.zeros(P)], 1) + rng.standard_normal((P, 3)) * 1e-4
    elif kind == "tiny":
        x = rng.uniform(-0.1, 0.1, (P, 3))
    else:
        c = rng.uniform(-1, 1, (20, 3))
        x = c[rng.integers(0, 20, P)] + rng.standard_normal((P, 3)) * 0.02
    x = x.astype(np.float32)
    # three clouds of different lengths packed back to back (one of them empty)
    cuts = [0, P // 3, P // 3, P]
    first = np.array(cuts[:-1], np.int64)
    num = np.array([cuts[i + 1] - cuts[i] for i in range(3)], np.int64)
    want_d, want_i = oracle.knn_brute(x, first, num, x, first, num, K, r)
    t = lambda a: torch.from_numpy(a).to(cuda_device)
    got_d, got_i = knn_points_packed(t(x), t(first), t(num), K, r)
    assert np.array_equal(got_d.cpu().numpy(), want_d)
    assert np.array_equal(got_i.cpu().numpy(), want_i)
    # separate query set (general mode), including queries outside the bounding box of the points
    q = (x[::7] * 1.3 + 0.01).astype(np.float32)
    a = min(10, len(q))
    qfirst = np.array([0, a, a], np.int64)
    qnum = np.array([a, 0, len(q) - a], np.int64)
    want_d, want_i = oracle.knn_brute(q, qfirst, qnum, x, first, num, K, r)
    got_d, got_i = knn_points_packed(t(x), t(first), t(num), K, r, t(q), t(qfirst), t(qnum))
    assert np.array_equal(got_d.cpu().numpy(), want_d)
    assert np.array_equal(got_i.cpu().numpy(), want_i)


@pytest.mark.gpu
def test_frnn_grid_points_signature_and_h_rule(cuda_device):
    """the reference-facing twin (padded batches, int64 idxs, -1 padding) and the splat-size rule built on it
    (rasterizer.py:313-326)."""
    from dss_b200.frnn_grid import frnn_grid_points
    rng = np.random.default_rng(1)
    N, P = 2, 3000
    pts = torch.from_numpy(rng.uniform(-0.5, 0.5, (N, P, 3)).astype(np.float32)).to(cuda_device)
    lens = torch.tensor([P, 1800], dtype=torch.int64, device=cuda_device)
    dists, idxs, nn, grid = frnn_grid_points(pts, pts, lens, lens, K=7, r=0.2, return_nn=True)
    assert dists.shape == (N, P, 7) and idxs.dtype == torch.int64 and nn.shape == (N, P, 7, 3) and grid is None
    assert (dists[1, 1800:] == -1).all() and (idxs[1, 1800:] == -1).all()
    x = pts.cpu().numpy()
    for n in range(N):
        L = int(lens[n])
        wd, wi = oracle.knn_brute(x[n, :L], np.zeros(1, np.int64), np.array([L]), x[n, :L], np.zeros(1, np.int64),
                                  np.array([L]), 7, 0.2)
        assert np.array_equal(dists[n, :L].cpu().numpy(), wd) and np.array_equal(idxs[n, :L].cpu().numpy(), wi)
    # pytorch3d-style twin (no radius, zero padding)
    from dss_b200.frnn_grid import knn_points
    kd, ki, _ = knn_points(pts, pts, lens, lens, K=12)
    wd, wi = oracle.knn_brute(x[1, :1800], np.zeros(1, np.int64), np.array([1800]), x[1, :1800], np.zeros(1, np.int64),
                              np.array([1800]), 12, -1.0)
    assert np.array_equal(kd[1, :1800].cpu().numpy(), wd) and np.array_equal(ki[1, :1800].cpu().numpy(), wi)
    assert (kd[1, 1800:] == 0).all() and (ki[1, 1800:] == 0).all()
    ok = idxs[0] >= 0
    g = torch.gather(pts[0][None].expand(P, -1, -1), 1, idxs[0].clamp(min=0)[..., None].expand(-1, -1, 3))
    assert torch.equal(nn[0][ok], g[ok])


@pytest.mark.gpu
def test_knn_fullsize_properties(cuda_device):
    """1M points (BASELINE headline cloud): self match first, ascending, inside the radius, and exact agreement with a
    brute-force torch search for a random sample of queries."""
    from dss_b200.frnn_grid import knn_points_packed
    from tests.util import sphere_cloud
    P, K, r = 1_000_000, 7, 0.2
    pts = sphere_cloud(P)[0].to(cuda_device)
    f = torch.zeros(1, dtype=torch.int64, device=cuda_device)
    n = torch.tensor([P], dtype=torch.int64, device=cuda_device)
    d, i = knn_points_packed(pts, f, n, K, r)
    assert (i[:, 0] == torch.arange(P, device=cuda_device)).all() and (d[:, 0] == 0).all()
    assert (d[:, 1:] >= d[:, :-1]).all() and (d >= 0).all() and (d < r * r).all()
    sel = torch.randperm(P, generator=torch.Generator().manual_seed(0))[:512].to(cuda_device)
    diff = pts[sel][:, None, :] - pts[None, :, :]
    d2 = (diff[..., 0] * diff[..., 0] + diff[..., 1] * diff[..., 1]) + diff[..., 2] * diff[..., 2]
    want = torch.topk(d2, K, dim=1, largest=False)[0]
    assert torch.equal(want, d[sel])
