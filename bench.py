#!/usr/bin/env python
"""bench.py -- forward+backward splat throughput of the surface-splatting hot path.

    python bench.py --gpus 1 --steps 20 --warmup 3            # our arm, one JSON line
    torchrun ... bench.py --gpus N ...                         # view-sharded, one rank per GPU (weak scaling)
    python bench.py --impl reference ...                       # the reference's own CPU rasterizer (oracle/_ref)

Metric (BASELINE.json): Msplats/s forward+backward, 1 splat = one (point, view) pair, on a synthetic
1 M-point cloud rendered at 512x512, V views per GPU.  A "step" is one pass of the whole hot path
[preprocess -> binning -> raster+blend -> injected image gradient -> colour/occupancy backward ->
world-space gradients] over one batch of V views (SURVEY.md section 8d).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BYTES_PER_SPLAT_FMT = "108*P0 + (32+8K)*S^2 per view"


def algorithmic_bytes_per_view(P0, S, K):
    """SURVEY.md section 8(d): compulsory traffic of one view, forward+backward."""
    return 108 * P0 + (32 + 8 * K) * S * S


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--image-size", type=int, default=512)
    ap.add_argument("--views-per-gpu", type=int, default=8)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replays (N = 1)")
    ap.add_argument("--cpu-sample-points", type=int, default=20000)
    ap.add_argument("--colours", default="point", choices=["point", "view", "shaded"],
                    help="point: one RGB per point shared by the views (default, the BASELINE line); view: per-(view,point) "
                         "colours (V*P0,3) as the reference holds them after shading; shaded: per-point albedo + fused "
                         "shading (one directional light), gradients to albedo, normals and positions")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (image and gradients) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES_PER_ARRAY = 15_000_000     # at most four arrays are written: 60 MB in all


def dump_outputs(directory, arrays):
    """Write each array as float32 <directory>/<name>.npy.  One larger than DUMP_BYTES_PER_ARRAY is stored as a fixed,
    seeded sample of its rows (leading dimensions flattened, rows kept in order), so that two builds run with the same
    arguments can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        x = t.detach().float().cpu().numpy()
        if x.nbytes > DUMP_BYTES_PER_ARRAY:
            x = x.reshape(-1, x.shape[-1])
            keep = DUMP_BYTES_PER_ARRAY // (x.itemsize * x.shape[1])
            x = x[np.sort(np.random.default_rng(0).choice(x.shape[0], keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), x)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled from a thread every ~2 ms
    (nvidia-smi -lms cannot deliver a sample inside a region of a few tens of ms); nvidia-smi is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.sm, self.bits, self.mx, self.source = index, [], 0, None, None
        self._stop = threading.Event()
        self.t = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x.strip() for x in vis.split(",") if x.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.source = "nvml"
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
        except Exception:
            self.source = "nvidia-smi"
            self.t = threading.Thread(target=self._poll_smi, daemon=True)
        self.t.start()

    def _poll_nvml(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            time.sleep(0.002)

    def _poll_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        self.smi_reasons = set()
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.sm.append(float(f[0]))
                self.mx = float(f[1])
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        self.smi_reasons.add(nm)
            except Exception:
                time.sleep(0.05)

    def stop(self):
        self._stop.set()
        if self.t is not None:
            self.t.join(timeout=6)
        reasons = set()
        if self.source == "nvml":
            nv = self.nv
            for nm, bit in (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                            ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                            ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                            ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                            ("hw_power_brake", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown)):
                if self.bits & bit:
                    reasons.add(nm)
        else:
            reasons = getattr(self, "smi_reasons", set())
        sm = sorted(self.sm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": ["no clock samples"], "samples": 0,
                    "source": self.source}
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": self.source}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU rasterizer compiled from its sources (oracle/_ref)
# ------------------------------------------------------------------------------------------------
def _cpu_sample_inputs(P_sample, S, K, seed=0):
    """Screen-space inputs of ONE view of the bench workload, subsampled to P_sample points.  The CPU
    preprocess uses the float64 oracle (no GPU needed); only the rasterizer fwd+bwd is timed, which is
    what the reference's native CPU path covers (its Python layer cannot run without pytorch3d)."""
    import numpy as np
    import torch
    import oracle
    from tests.util import scene
    pts, nrm, col, proj, view, _ = scene(P_sample, 1, seed=seed)
    h = np.full((1,), 5e-5, np.float32)
    pre = oracle.preprocess_f64(proj.numpy(), view.numpy(), pts.numpy(), nrm.numpy(), h, 1.0, 1.0, S)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    g = torch.Generator().manual_seed(77)
    return dict(points=t(pre["ndc"]), ellipse=t(pre["ellipse"]), radii=t(pre["radii"]),
                cutoff=torch.ones(P_sample), first=torch.zeros(1, dtype=torch.int64),
                num=torch.full((1,), P_sample, dtype=torch.int64),
                grad_occ=torch.randn(1, S, S, generator=g) * 1e-3)


def _cpu_one_view(args):
    """Time the reference CPU fwd (+ occupancy backward) on one sampled view; returns seconds."""
    P_sample, S, K, seed, radii_s = args
    import torch
    torch.set_num_threads(1)
    from oracle import build_ref
    ref = build_ref.ref_cpu()
    x = _cpu_sample_inputs(P_sample, S, K, seed)
    t0 = time.perf_counter()
    if ref is not None:
        # the reference's production path for this size: coarse + fine with the bin-size heuristic
        # (rasterizer.py:713-722) and M = max(10000, P) (rasterizer.py:732-733)
        bin_size = 8 if S <= 64 else 16 if S <= 256 else 32 if S <= 512 else 64
        bins = ref.rasterize_coarse_cpu(x["points"], x["radii"], x["first"], x["num"], S, bin_size,
                                        max(10000, P_sample))
        ref.rasterize_fine_cpu(x["points"], x["ellipse"], x["cutoff"], x["radii"], bins, 0.05, S, bin_size, K)
        ref.splat_points_occ_backward_cpu(x["points"], x["radii"], x["grad_occ"], x["first"], x["num"],
                                          radii_s, 0.05)
        kind = "reference"
    else:
        import oracle
        idx, _, _, _ = oracle.splat_points_binned(x["points"].numpy(), x["ellipse"].numpy(), x["cutoff"].numpy(),
                                                  x["radii"].numpy(), x["first"].numpy(), x["num"].numpy(), 0.05,
                                                  S, K, 32)
        vis = oracle.visibility(idx, P_sample)
        rs = oracle.search_radius(x["radii"].numpy(), vis, x["first"].numpy(), x["num"].numpy(), radii_s)
        oracle.occ_backward_fast(x["points"].numpy(), x["radii"].numpy(), vis, rs, x["grad_occ"].numpy(),
                                 x["first"].numpy(), x["num"].numpy())
        kind = "port"
    return time.perf_counter() - t0, kind


def cpu_baseline(P_sample, S, K, procs, views, radii_s=5.0):
    """Msplats/s of the reference CPU rasterizer fwd+bwd on `views` sampled views spread over `procs`
    single-threaded processes (the reference CPU code has no threading: SURVEY.md section 8d)."""
    import multiprocessing as mp
    jobs = [(P_sample, S, K, i, radii_s) for i in range(views)]
    t0 = time.perf_counter()
    if procs <= 1:
        res = [_cpu_one_view(j) for j in jobs]
    else:
        with mp.get_context("spawn").Pool(procs) as pool:
            res = pool.map(_cpu_one_view, jobs)
    wall = time.perf_counter() - t0
    kind = res[0][1]
    return {"value": views * P_sample / wall / 1e6, "unit": "Msplats/s", "cores": procs, "kind": kind,
            "sample": "%d view(s) x %d points subsampled from the bench cloud at %dx%d, K=%d: reference "
                      "RasterizePointsCoarseCpu+FineCpu forward + RasterizePointsOccBackwardCpu (radii_s=%g), "
                      "screen-space inputs precomputed; %.1f s wall" % (views, P_sample, S, S, K, radii_s, wall),
            "seconds": wall}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 32))
    P_sample, S, K = a.cpu_sample_points, a.image_size, a.k
    times = []
    for step in range(a.warmup + a.steps):
        if step < a.warmup and step > 0:
            continue                      # one warm-up pass is enough to page the module in
        r = cpu_baseline(P_sample, S, K, procs, procs)
        if step >= a.warmup:
            times.append(r)
        if sum(t["seconds"] for t in times) > 150:   # keep the whole run within a few minutes
            break
    wall = sum(t["seconds"] for t in times)
    value = len(times) * procs * P_sample / wall / 1e6
    line = {
        "impl": "reference", "metric": "Msplats/s fwd+bwd", "value": value, "unit": "Msplats/s",
        "n_gpus": a.gpus, "steps": len(times), "warmup": min(a.warmup, 1), "ms_per_step": 1e3 * wall / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "synthetic sphere %d pts x %d views/GPU, %dx%d, K=%d, fwd+bwd"
                               % (a.points, a.views_per_gpu, S, S, K)},
        "cpu_baseline": {"value": value, "unit": "Msplats/s", "cores": procs, "kind": times[0]["kind"],
                         "sample": times[0]["sample"]},
        "e2e": {"value": value, "unit": "Msplats/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(a):
    import torch
    import torch.distributed as dist
    from dss_b200 import _lib
    from dss_b200.ops import SplatParams, render_points
    from tests.util import sphere_cloud, random_cameras
    from dss_b200.core.camera import camera_matrices

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    P0, S, K, V = a.points, a.image_size, a.k, a.views_per_gpu
    prm = SplatParams(image_size=S, points_per_pixel=K, cutoff_threshold=1.0, depth_merging_threshold=0.05,
                      antialiasing_sigma=1.0, radii_backward_scaler=5.0, clip_pts_grad=0.05,
                      backface_culling=False, znear=0.1, zfar=100.0)            # configs/dss.yml:14-22
    from dss_b200.parallel import GradSync, assign_views, view_costs_from_cameras
    pts, nrm, col = sphere_cloud(P0, seed=0)
    cams = random_cameras(V * world, seed=0)
    proj_all, view_all = camera_matrices(cams)
    # views are dealt to the ranks by estimated cost (close cameras cover more pixels): the slowest rank sets the step
    mine = assign_views(view_costs_from_cameras(view_all).tolist(), world)[rank]
    assert len(mine) == V
    proj_h, view_h = proj_all[mine].contiguous().pin_memory(), view_all[mine].contiguous().pin_memory()
    # the one exchange step of the path (SURVEY.md section 8e): per-point gradients summed over the ranks, issued by
    # the backward itself and overlapped with it (dss_b200/parallel.py)
    sync = GradSync(timing=True) if world > 1 else None
    g = torch.Generator().manual_seed(99 + rank)
    # colours: one RGB per POINT, shared by the views of the step (the quantity an inverse-rendering step optimises
    # and the one exchange step reduces); per-(view,point) colours -- the layout the reference holds on the device after
    # shading -- take the same path with a (V*P0,3) tensor (tests/test_gpu_render.py).
    colours_h = (col.repeat(V, 1) if a.colours == "view" else col).contiguous().pin_memory()
    grad_h = (torch.randn(V, S, S, 4, generator=g) * 1e-3).pin_memory()        # dense, like the IoU term
    pts_h, nrm_h = pts.pin_memory(), nrm.pin_memory()
    h_h = torch.full((V,), 5e-5).pin_memory()   # clamp floor of the 6-NN rule at this density (rasterizer.py:326)

    # resident copies for the device-timed `value`
    pts_d = pts_h.to(dev).requires_grad_(True)
    nrm_d, col_d = nrm_h.to(dev), colours_h.to(dev).requires_grad_(True)
    proj_d, view_d, h_d, grad_d = proj_h.to(dev), view_h.to(dev), h_h.to(dev), grad_h.to(dev)

    shading = None
    if a.colours == "shaded":
        from dss_b200.core.lighting import DirectionalLights
        from dss_b200.ops import make_shading
        shading = make_shading(DirectionalLights(direction=(((0.3, 1.0, 0.4),),), device=dev), view_d, shininess=64.0)
        nrm_d.requires_grad_(True)

    def step_resident():
        pts_d.grad = None
        col_d.grad = None
        nrm_d.grad = None
        out = render_points(pts_d, nrm_d, col_d, proj_d, view_d, h_d, prm, grad_sync=sync, shading=shading)
        out.image.backward(grad_d)            # gradients come back already summed over the ranks
        return out

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-timed region: inputs resident in HBM ----
    for _ in range(max(a.warmup, 3)):
        last = step_resident()
    sync_all()
    n_visible = int(last.visible.sum().item())     # visible (view, point) pairs of this rank's step (for the byte counts)
    if sync is not None:
        sync.timings_ms()
        sync.reset_counters()
    # per-stage device times (the library's own CUDA-event brackets) from an eager pass of a few steps ...
    _lib.profile_reset(dev)
    _lib.profile_enable(True, dev)
    launches0 = _lib.launch_count(dev)
    n_prof = min(a.steps, 20)
    for _ in range(n_prof):
        step_resident()
    sync_all()
    launches_per_step = (_lib.launch_count(dev) - launches0) / n_prof
    stages = {k: (v[0] * a.steps / n_prof, v[1]) for k, v in _lib.profile_read(dev).items()}   # scaled to `steps`
    _lib.profile_enable(False, dev)
    allreduce = None
    if sync is not None:      # device time / bytes of the two overlapped collectives, from the same eager pass
        ar_ms = sync.timings_ms() / n_prof
        ar_bytes = sync.bytes_reduced / n_prof
        allreduce = {"ms_per_step": ar_ms, "bytes_per_step": int(ar_bytes), "collectives_per_step": 2,
                     "busbw_GBs": (2.0 * (world - 1) / world) * ar_bytes / (ar_ms * 1e-3) / 1e9 if ar_ms > 0 else None,
                     "overlap": "d colour reduced on a side stream during the occupancy gather; d position behind the "
                                "chain kernel"}
        sync.timing = False
        sync.reset_counters()
    # ... and the timed region: K steps, replayed from ONE captured CUDA graph of the whole step on a single GPU (the
    # library neither synchronises nor allocates in steady state: dss_b200/graph.py), launched eagerly otherwise
    graphed = None
    if not a.no_graph and world == 1:    # (N > 1 is launched eagerly: the NCCL exchange inside a capture hung on 2 GPUs)
        try:
            from dss_b200.graph import GraphedRenderStep
            graphed = GraphedRenderStep(pts_d, nrm_d, col_d, proj_d, view_d, h_d, prm, grad_d, shading=shading)
            for _ in range(3):
                graphed.replay()
        except Exception as e:   # pragma: no cover
            # a failed capture can leave the process's CUDA state unusable for timing: start over, eagerly
            print("CUDA-graph capture failed (%r): %s" % (e, "re-running with --no-graph" if world == 1 else "eager"),
                  file=sys.stderr)
            sys.stderr.flush()
            if world == 1:
                os.execv(sys.executable, [sys.executable] + sys.argv + ["--no-graph"])
            graphed = None
    sync_all()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        if graphed is not None:
            graphed.replay()
        else:
            last = step_resident()
    e1.record()
    sync_all()
    clocks = sampler.stop()
    if a.dump_outputs and rank == 0:
        if graphed is not None:
            outs = dict(image=graphed.image, grad_points=graphed.grad_points, grad_colours=graphed.grad_colours,
                        grad_normals=graphed.grad_normals)
        else:
            outs = dict(image=last.image, grad_points=pts_d.grad, grad_colours=col_d.grad, grad_normals=nrm_d.grad)
        dump_outputs(a.dump_outputs, {k: v for k, v in outs.items() if v is not None})
    ms = e0.elapsed_time(e1)
    launches = launches_per_step * a.steps      # kernels executed in the timed region (replayed, not re-launched, under a graph)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * V * P0 * a.steps / (ms_max * 1e-3) / 1e6

    # ---- end to end through the public API with HOST buffers ----
    e2e = None
    if not a.no_e2e:
        img_h = torch.empty(V, S, S, 4).pin_memory()
        gpts_h = torch.empty(P0, 3).pin_memory()
        gcol_h = torch.empty_like(colours_h).pin_memory()
        # host-side inputs of a step: the cloud (positions, normals, per-point colours), this rank's cameras and the
        # image gradient.  Colours go up once per POINT (P0,3): the reference only materialises per-(view,point)
        # colours on the device (after shading), it never uploads them.
        host_in = (pts_h, nrm_h, colours_h, proj_h, view_h, h_h, grad_h)
        # double-buffered device staging: the H2D copy of step i+1 and the D2H read of step i run on a copy
        # stream while step i / i+1 computes; every step still moves all of its inputs and results
        dev_in = [[torch.empty_like(x, device=dev) for x in host_in] for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)      # host -> device staging
        back_stream = torch.cuda.Stream(device=dev)      # device -> host read-back (PCIe is full duplex)
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]
        state = {"i": 0}
        keep = [None, None]     # outputs of the step that last used a slot: alive until their read-back has finished

        diag = os.environ.get("BENCH_E2E_SKIP", "")   # diagnosis only: "h2d" / "d2h" drop that half of the traffic
        trace = [] if os.environ.get("BENCH_E2E_TRACE") else None   # diagnosis only: device timeline of the e2e loop

        def mark(name, stream):
            if trace is not None and state["i"] >= 3:
                e = torch.cuda.Event(enable_timing=True)
                e.record(stream)
                trace.append((state["i"], name, e))

        def stage_inputs(slot):
            if "h2d" in diag and state["i"] > 2:
                ev_in[slot].record(copy_stream)
                return
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_done[slot])      # the previous user of this slot has finished
                mark("h2d_begin(for step+1)", copy_stream)
                for d, hsrc in zip(dev_in[slot], host_in):
                    d.copy_(hsrc, non_blocking=True)
                ev_in[slot].record(copy_stream)
                mark("h2d_end(for step+1)", copy_stream)

        def step_e2e():
            i = state["i"]
            slot = i % 2
            if i == 0:
                stage_inputs(0)
            stage_inputs((i + 1) % 2)                      # prefetch the next step's inputs
            main = torch.cuda.current_stream(dev)
            main.wait_event(ev_in[slot])
            main.wait_event(ev_out[slot])                  # result buffers of two steps ago have been read back
            d = dev_in[slot]
            mark("compute_begin", main)
            p = d[0].detach().requires_grad_(True)
            c = d[2].detach().requires_grad_(True)
            nn_ = d[1].detach().requires_grad_(True) if shading is not None else d[1]
            out = render_points(p, nn_, c, d[3], d[4], d[5], prm, grad_sync=sync, shading=shading)
            mark("forward_end", main)
            out.image.backward(d[6])
            gp, gc = p.grad, c.grad        # summed over all ranks' views: the reduced gradients go back to the host
            ev_done[slot].record(main)
            mark("compute_end", main)
            with torch.cuda.stream(back_stream):
                back_stream.wait_event(ev_done[slot])
                if "d2h" in diag:
                    ev_out[slot].record(back_stream)
                    state["i"] = i + 1
                    return
                mark("d2h_begin", back_stream)
                img_h.copy_(out.image.detach(), non_blocking=True)
                gpts_h.copy_(gp, non_blocking=True)
                gcol_h.copy_(gc, non_blocking=True)
                ev_out[slot].record(back_stream)
                mark("d2h_end", back_stream)
            # no record_stream(): the tensors the read-back reads stay referenced until this slot comes round again, and by
            # then the main stream has waited for ev_out[slot] -- the caching allocator sees a plain same-stream free
            # (record_stream defers reuse unpredictably and costs occasional cudaMalloc/cudaFree stalls of ~15 ms)
            keep[slot] = (out, p, c, gp, gc)
            state["i"] = i + 1

        h2d = sum(x.numel() * x.element_size() for x in host_in)
        d2h = sum(x.numel() * x.element_size() for x in (img_h, gpts_h, gcol_h))
        for _ in range(3):
            step_e2e()
        sync_all()
        n_e2e = a.steps
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(n_e2e):
            step_e2e()
        torch.cuda.current_stream(dev).wait_stream(back_stream)   # the last read-back is inside the timed region
        f1.record()
        sync_all()
        if trace:
            base = trace[0][2]
            for i, name, e in trace[:60]:
                print("trace step %d %-22s %8.3f ms" % (i, name, base.elapsed_time(e)), file=sys.stderr)
        t2 = torch.tensor([f0.elapsed_time(f1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        e2e = {"value": world * V * P0 * n_e2e / (float(t2.item()) * 1e-3) / 1e6, "unit": "Msplats/s",
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": n_e2e}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel, from the live per-stage CUDA-event times ----
    peak, peak_src = load_peaks()
    total_stage_ms = sum(v[0] for v in stages.values()) or 1.0
    dom = max(stages, key=lambda k: stages[k][0])
    dom_ms, dom_n = stages[dom]
    per_launch_views = V
    Pv = n_visible                 # visible (view, point) pairs of one step, measured (about 18 % of V*P0)
    alg_all = {
        # algorithmic bytes per step of every stage (its kernels cover the V views of a step); DESIGN.md section 5
        "preprocess": per_launch_views * (24 * P0 + 36 * P0),            # read pos+normal, write record + scaler
        "bin_count": per_launch_views * 20 * P0,                          # read 20 B of every record
        "bin_scatter": per_launch_views * 24 * P0,                        # + 4 B id per entry written (>= 1 per splat)
        "raster_forward": per_launch_views * (36 * P0 + (16 + 4 * K) * S * S),
        # backward binning: visibility byte + record head of every splat, compact record + id of the visible ones
        "occ_bin": 2 * (per_launch_views * P0 * 1 + Pv * 16) + Pv * 20,
        "search_radius": 4 * Pv * 16,                                     # four radix passes over the compact records
        # planes (read the alpha gradient, write g-/g+ once) + gather (read both planes once, compact records, ids,
        # write the gradients of the VISIBLE splats)
        "occ_backward": per_launch_views * ((4 + 8) * S * S + 8 * S * S) + Pv * 28,
        "colour_backward": per_launch_views * ((16 + 8 * K) * S * S) + 12 * P0,
        "chain_world": per_launch_views * 8 * P0 + 24 * P0,
    }
    traffic_all = {}
    try:    # measured DRAM bytes per launch (dram__bytes_read + write, one ncu --set full capture per kernel change)
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        if P0 == 1_000_000 and S == 512 and V == 8 and K == 5:
            traffic_all = {k: v for k, v in tr.items() if isinstance(v, (int, float))}
    except Exception:
        pass
    per_kernel = {}
    for k, (ms_tot, n_br) in stages.items():
        if not n_br or k not in alg_all:
            continue
        ms_k = ms_tot / max(a.steps, 1)
        gbs = alg_all[k] / (ms_k * 1e-3) / 1e9 if ms_k > 0 else 0.0
        per_kernel[k] = {"ms": ms_k, "algorithmic_bytes": int(alg_all[k]), "achieved": gbs, "frac": gbs / peak,
                         "traffic": traffic_all.get(k)}
    alg = alg_all.get(dom, 0)
    dom_avg_ms = dom_ms / max(a.steps, 1)      # per step: a stage's kernels are launched once per step
    achieved = alg / (dom_avg_ms * 1e-3) / 1e9 if dom_avg_ms > 0 else 0.0
    step_bytes = V * algorithmic_bytes_per_view(P0, S, K)
    step_gbs = step_bytes / (ms_max / a.steps * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic_all.get(dom), "peak_source": peak_src,
                "kernel_ms_per_launch": dom_avg_ms, "kernel_share_of_step": dom_ms / total_stage_ms,
                "stage_ms_per_step": {k: v[0] / a.steps for k, v in stages.items() if v[1]},
                # every stage against its own byte roofline (both dominant kernels are always in here: which of the two
                # is `kernel` can flip from run to run)
                "kernels": per_kernel, "visible_pairs_per_step": int(Pv),
                "whole_step": {"algorithmic_bytes": step_bytes, "achieved": step_gbs, "frac": step_gbs / peak,
                               "formula": BYTES_PER_SPLAT_FMT}}

    cpu = None
    if not a.no_cpu_baseline and world == 1:
        try:
            cpu = cpu_baseline(a.cpu_sample_points, S, K, 1, 1)
            cpu.pop("seconds", None)
        except Exception as e:  # pragma: no cover
            cpu = {"value": None, "unit": "Msplats/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}

    work_mb = (pts_d.numel() + nrm_d.numel() + col_d.numel() + grad_d.numel()) * 4 / 1e6
    line = {
        "metric": "Msplats/s fwd+bwd", "value": value, "unit": "Msplats/s", "n_gpus": world, "steps": a.steps,
        "warmup": max(a.warmup, 3), "ms_per_step": ms_max / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "synthetic sphere %d pts x %d views/GPU, %dx%d, K=%d, fwd+bwd" % (P0, V, S, S, K),
                   "views_total": V * world, "parallelism": "views dealt by cost, %d/GPU; NCCL all-reduce of d colour (side stream, "
                   "overlapped with the occupancy gather) and of d position (behind the chain kernel)" % V
                   if world > 1 else "single GPU",
                   "l2": "per-step inputs %.0f MB + %.0f MB of splat records exceed the 126 MB L2" % (work_mb, V * P0 * 32 / 1e6),
                   "colours": {"point": "per point (P0,3), shared by the views",
                               "view": "per (view, point) (V*P0,3), the layout the reference holds after shading",
                               "shaded": "per-point albedo (P0,3) + fused shading (1 directional light): gradients to "
                                         "albedo, normals, positions"}[a.colours],
                   "launch": "one CUDA graph per step (captured fwd+bwd, dss_b200.graph)" if graphed is not None else "eager",
                   "settings": "configs/dss.yml:14-22 (cutoff 1, merge 0.05, K=5, radii_s 5, clip 0.05, sigma 1)"},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "allreduce": allreduce,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
