"""Diagnose occupancy-gradient mismatches vs the reference fast CUDA kernel at the headline size."""
import sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dss_b200 import _C
from dss_b200.ops import SplatParams, render_points
from tests.util import scene, packed_offsets
from tests.golden.make_golden_reference import reference_fast_backward as _reference_fast_backward
from oracle import build_ref
ref = build_ref.ref_cuda()
dev = torch.device("cuda:0")
P0, N, S, K = 1_000_000, 2, 512, 5
pts, nrm, col, proj, view, _ = scene(P0, N, seed=0)
prm = SplatParams(image_size=S, points_per_pixel=K, znear=0.1, clip_pts_grad=-1.0)
h = torch.full((N,), 5e-5, device=dev)
out = render_points(pts.to(dev), nrm.to(dev), col.to(dev), proj.to(dev), view.to(dev), h, prm, return_fragments=True)
rec = out.records
first, num = (t.to(dev) for t in packed_offsets(N, P0))
ndc, rad = rec[:, :3].contiguous(), rec[:, 3:5].contiguous()
g = torch.randn(N, S, S, 4, generator=torch.Generator().manual_seed(5)).to(dev) * 1e-3
vis = out.visible.view(N, P0).bool()
rs_all = _C.search_radius(rad, out.visible, first, num, 5.0)
ours = _C.occ_backward(ndc, rad, out.visible, rs_all, g[..., 3].contiguous(), first, num)
for n in range(N):
    sl = slice(n * P0, (n + 1) * P0)
    g_vis, rs = _reference_fast_backward(ref, ndc[sl], rad[sl], vis[n], g[n:n + 1, :, :, 3].contiguous(), 5.0)
    g_vis2, _ = _reference_fast_backward(ref, ndc[sl], rad[sl], vis[n], g[n:n + 1, :, :, 3].contiguous(), 5.0)
    o = ours[sl][vis[n]]
    print("view", n, "rs", float(rs), float(rs_all[n]), "ref max", float(g_vis.abs().max()), "ref-vs-ref max diff", float((g_vis - g_vis2).abs().max()))
    d = (o - g_vis).abs().max(1)[0]
    top = d.topk(8)
    pv = ndc[sl][vis[n]]
    for e, i in zip(top.values.tolist(), top.indices.tolist()):
        px, py = float(pv[i, 0]), float(pv[i, 1])
        fx, fy = (px + 1) * S / 2 - 0.5, (py + 1) * S / 2 - 0.5      # pixel-index coordinates of the point
        print("   err %.3e  ours (%.6f, %.6f) ref (%.6f, %.6f)  pix (%.4f, %.4f) frac-dist-to-centre %.2e" % (
            e, o[i, 0], o[i, 1], g_vis[i, 0], g_vis[i, 1], fx, fy, ((fx - round(fx)) ** 2 + (fy - round(fy)) ** 2) ** 0.5))
