"""ctypes binding of libdss_b200.so (the C ABI declared in include/dss_b200.h).

There is deliberately NO fallback: if the library is missing, was built for another architecture or
a call fails, a RuntimeError is raised.  PyTorch is used only for device memory and streams.
"""
import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DSS_B200_LIB") or os.path.join(_HERE, "lib", "libdss_b200.so")   # (override: A/B builds)

DSS_OK = 0
DSS_E_CAPACITY = -4
MAX_POINTS_PER_PIXEL = 64
MAX_SHARED_VIEWS = 256
MAX_LIGHTS = 8

_lib = None
_ctx = {}
_lock = threading.Lock()

vp = C.c_void_p


class RenderArgs(C.Structure):
    """Mirror of `struct dss_render_args` (include/dss_b200.h)."""
    _fields_ = [
        ("points_world", vp), ("normals_world", vp), ("colours", vp), ("proj", vp), ("view", vp),
        ("h", vp), ("first_idx", vp), ("num_points", vp),
        ("n_views", C.c_int32), ("shared_cloud", C.c_int32), ("P0", C.c_int64), ("P", C.c_int64),
        ("h_per_splat", C.c_int32), ("image_size", C.c_int32), ("points_per_pixel", C.c_int32),
        ("backface_culling", C.c_int32),
        ("cutoff_threshold", C.c_float), ("depth_merging_threshold", C.c_float),
        ("antialiasing_sigma", C.c_float), ("znear", C.c_float), ("zfar", C.c_float),
        ("radii_backward_scaler", C.c_float), ("clip_pts_grad", C.c_float),
        ("records", vp), ("ndc", vp), ("ellipse", vp), ("radii", vp), ("scaler", vp), ("image", vp),
        ("idx", vp), ("weights", vp), ("zbuf", vp), ("qvalue", vp), ("visible", vp),
        ("grad_image", vp), ("grad_zbuf", vp), ("grad_colours", vp), ("grad_ndc", vp),
        ("grad_points_world", vp), ("search_radius", vp),
        ("shared_colours", C.c_int32),
        ("shade", C.c_int32), ("n_lights", C.c_int32), ("light_type", C.c_int32), ("shininess", C.c_float),
        ("reserved0", C.c_int32),
        ("albedo", vp), ("lights", vp), ("ambient", vp), ("cam_centres", vp), ("shaded", vp),
        ("grad_albedo", vp), ("grad_normals_world", vp), ("grad_points_shading", vp),
        ("cell_counts", vp),
    ]


DR_LOSS_BLOCKS_PER_VIEW = 128
DR_LOSS_NUM_SUMS = 5


class DrLossArgs(C.Structure):
    """Mirror of `struct dss_dr_loss_args` (include/dss_b200.h)."""
    _fields_ = [
        ("image", vp), ("img", vp), ("mask", vp),
        ("n_views", C.c_int32), ("image_size", C.c_int32),
        ("lambda_rgb", C.c_float), ("lambda_silhouette", C.c_float), ("iou_weight", C.c_float),
        ("reserved0", C.c_int32),
        ("partials", vp), ("sums", vp), ("terms", vp), ("grad_loss", vp), ("grad_image", vp),
    ]


_SIGNATURES = {
    "dss_version": (C.c_int, []),
    "dss_last_error": (C.c_char_p, []),
    "dss_create": (C.c_int, [C.POINTER(vp)]),
    "dss_destroy": (None, [vp]),
    "dss_scratch_bytes": (C.c_size_t, [vp]),
    "dss_launch_count": (C.c_int64, [vp]),
    "dss_profile_enable": (C.c_int, [vp, C.c_int]),
    "dss_profile_reset": (C.c_int, [vp]),
    "dss_profile_num_stages": (C.c_int, []),
    "dss_profile_stage_name": (C.c_char_p, [C.c_int]),
    "dss_profile_read": (C.c_int, [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "dss_debug_raster_stats": (C.c_int, [vp, C.c_int, C.POINTER(C.c_uint64)]),
    "dss_debug_limit_tile_capacity": (C.c_int, [vp, C.c_int64]),
    "dss_debug_tile_total": (C.c_int64, [vp]),
    "dss_exclusive_scan_i32": (C.c_int, [vp, vp, vp, C.c_int64, vp]),
    "dss_grid_insert_points_2d": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "dss_grid_counting_sort_2d": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "dss_rasterize_coarse": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int64, C.c_int, C.c_int, vp, vp,
                                       C.c_int64, C.POINTER(C.c_int64), vp]),
    "dss_splat_points": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int64, C.c_float, C.c_int,
                                   C.c_int, C.c_int, vp, vp, vp, vp, vp]),
    "dss_visibility_from_idx": (C.c_int, [vp, vp, C.c_int64, C.c_int, C.c_int64, vp, vp]),
    "dss_search_radius": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int64, C.c_float, vp, vp]),
    "dss_occ_backward": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int64,
                                   C.c_int, vp, vp]),
    "dss_occ_backward_slow": (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int64, C.c_int, C.c_float,
                                        vp, vp]),
    "dss_zbuf_backward": (C.c_int, [vp, vp, vp, C.c_int64, C.c_int, vp, vp]),
    "dss_knn_points": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_float,
                                 vp, vp, vp]),
    "dss_preprocess": (C.c_int, [vp, C.POINTER(RenderArgs), vp]),
    "dss_render_forward": (C.c_int, [vp, C.POINTER(RenderArgs), vp]),
    "dss_render_backward": (C.c_int, [vp, C.POINTER(RenderArgs), vp]),
    "dss_colour_backward": (C.c_int, [vp, C.POINTER(RenderArgs), vp]),
    "dss_dr_loss_forward": (C.c_int, [vp, C.POINTER(DrLossArgs), vp]),
    "dss_dr_loss_backward": (C.c_int, [vp, C.POINTER(DrLossArgs), vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load():
    """dlopen libdss_b200.so and declare every prototype.  Works without a GPU (symbol checks)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libdss_b200.so is missing (%s). Build it with `python -m dss_b200.build` "
                "(nvcc, sm_100a). There is no CPU or PyTorch fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    return load().dss_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != DSS_OK:
        raise RuntimeError("%s failed (status %d): %s" % (what, rc, last_error()))


def ctx(device=None):
    """One dss_ctx per CUDA device of this process."""
    if not torch.cuda.is_available():
        raise RuntimeError("dss_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    if device is None:
        device = torch.cuda.current_device()
    dev = torch.device(device)
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    with _lock:
        if index not in _ctx:
            lib = load()
            h = vp()
            with torch.cuda.device(index):
                check(lib.dss_create(C.byref(h)), "dss_create")
            _ctx[index] = h
        return _ctx[index]


def stream_ptr(device=None):
    return vp(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return vp(0)
    return vp(t.data_ptr())


def launch_count(device=None):
    return int(load().dss_launch_count(ctx(device)))


def profile_enable(on, device=None):
    check(load().dss_profile_enable(ctx(device), int(bool(on))), "dss_profile_enable")


def profile_reset(device=None):
    check(load().dss_profile_reset(ctx(device)), "dss_profile_reset")


def profile_read(device=None):
    """{stage name: (total ms, brackets)} since the last reset; synchronises on the recorded events."""
    lib = load()
    out = {}
    for i in range(lib.dss_profile_num_stages()):
        ms, n = C.c_double(0.0), C.c_int64(0)
        check(lib.dss_profile_read(ctx(device), i, C.byref(ms), C.byref(n)), "dss_profile_read")
        out[lib.dss_profile_stage_name(i).decode()] = (ms.value, n.value)
    return out


def raster_stats(enable, device=None):
    """debug counters of the sliced rasterizer accumulated since they were last enabled (see the header)."""
    out = (C.c_uint64 * 8)()
    check(load().dss_debug_raster_stats(ctx(device), int(bool(enable)), out), "dss_debug_raster_stats")
    names = ["entries_scanned", "survivors", "pixel_tests", "accepted", "slices_skipped", "slices_visited",
             "overflow_tiles"]
    return dict(zip(names, [int(v) for v in out[:7]]))


def limit_tile_capacity(max_entries, device=None):
    """testing: cap the forward's tile-list buffer (0 = no cap) so that the overflow path runs (see the header)."""
    check(load().dss_debug_limit_tile_capacity(ctx(device), int(max_entries)), "dss_debug_limit_tile_capacity")


def scratch_bytes(device=None):
    return int(load().dss_scratch_bytes(ctx(device)))


def as_f32(t, name):
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32, got %s" % (name, t.dtype))
    return t.contiguous()


def require_cuda(*tensors):
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("dss_b200 operators take CUDA tensors only (no CPU fallback); got a %s tensor"
                               % t.device)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("all tensors must be on the same device (%s vs %s)" % (dev, t.device))
    return dev
