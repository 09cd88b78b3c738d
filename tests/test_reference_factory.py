"""The plugin boundary exercised for real: the reference's own, unmodified `config.py` (imported from the reference
checkout where it lies) builds OUR classes from `configs/dss.yml` once the three YAML lines of INTEGRATION.md point at
them (config.py:241-262 `create_renderer`, DSS/utils/__init__.py:68-73 `get_class_from_string`).  That test needs the
reference checkout (oracle.build_ref.REF) and skips without it; the reference's third-party imports that are not
installed are served by tests/shim (stub modules; test infrastructure only).

The settings signature is compared with what the reference's DSS/core/rasterizer.py declares, stored in
tests/golden/reference/rasterizer_signature.json (tests/golden/make_golden_reference.py)."""
import json
import os
import sys

import pytest
import torch

from oracle.build_ref import REF


@pytest.fixture(scope="module")
def ref_config():
    if not os.path.isfile(os.path.join(REF, "config.py")):
        pytest.skip("reference checkout not present")
    from tests import shim
    sys.dont_write_bytecode = True
    shim.install()
    sys.path.insert(0, REF)
    try:
        import config                                  # the reference's file, unmodified
        assert os.path.realpath(config.__file__) == os.path.realpath(os.path.join(REF, "config.py"))
        yield config
    finally:
        sys.path.remove(REF)
        sys.modules.pop("config", None)
        for m in [m for m in sys.modules if m == "DSS" or m.startswith("DSS.")]:
            del sys.modules[m]
        shim.uninstall()
        sys.dont_write_bytecode = False


def _cfg(config):
    cfg = config.load_config(os.path.join(REF, "configs", "dss.yml"), os.path.join(REF, "configs", "default.yaml"))
    # INTEGRATION.md: only these three lines of the YAML change
    cfg.renderer.renderer_type = "dss_b200.core.renderer.SurfaceSplattingRenderer"
    cfg.renderer.raster_type = "dss_b200.core.rasterizer.SurfaceSplatting"
    cfg.renderer.compositor_type = "dss_b200.core.renderer.NormWeightedCompositor"
    return cfg


def test_reference_factory_builds_our_renderer_from_its_yaml(ref_config):
    from dss_b200.core.camera import FoVPerspectiveCameras
    from dss_b200.core.rasterizer import PointsRasterizationSettings, SurfaceSplatting
    from dss_b200.core.renderer import NormWeightedCompositor, SurfaceSplattingRenderer
    cfg = _cfg(ref_config)
    renderer = ref_config.create_renderer(cfg.renderer)                  # config.py:241-262, unmodified
    assert type(renderer) is SurfaceSplattingRenderer
    assert type(renderer.rasterizer) is SurfaceSplatting
    assert type(renderer.compositor) is NormWeightedCompositor
    assert isinstance(renderer.rasterizer.cameras, FoVPerspectiveCameras) and renderer.cameras is renderer.rasterizer.cameras
    rs = renderer.rasterizer.raster_settings
    assert type(rs) is PointsRasterizationSettings
    # configs/dss.yml:14-22 over configs/default.yaml:20-30
    want = dict(cfg.renderer.raster_params)
    for k, v in want.items():
        assert getattr(rs, k) == v, k
    assert rs.cutoff_threshold == 1.0 and rs.points_per_pixel == 5 and rs.Vrk_invariant is True
    assert rs.radii_backward_scaler == 5 and rs.clip_pts_grad == 0.05 and rs.image_size == 512
    # what Trainer / TrainerScheduler touch afterwards (trainer.py:116, scheduler.py:40-45): live, mutable settings
    renderer.rasterizer.raster_settings.radii_backward_scaler = 4.5
    assert renderer.rasterizer.raster_settings.radii_backward_scaler == 4.5
    assert isinstance(renderer, torch.nn.Module) and hasattr(renderer, "to")


def test_reference_settings_class_has_the_same_keywords_as_ours():
    """DSS/core/rasterizer.py:73-99 vs dss_b200.core.rasterizer: same keyword arguments, same defaults."""
    import inspect
    with open(os.path.join(os.path.dirname(__file__), "golden", "reference", "rasterizer_signature.json")) as f:
        ref = json.load(f)
    from dss_b200.core.rasterizer import PointsRasterizationSettings as Ours
    sig_our = inspect.signature(Ours.__init__)
    ref_params = ref["PointsRasterizationSettings"]
    our_params = {k: p.default for k, p in sig_our.parameters.items() if k != "self"}
    assert ref_params == our_params
    # the forward signatures the trainer calls through (rasterizer.py:584, renderer.py:36)
    from dss_b200.core.rasterizer import SurfaceSplatting
    f_our = inspect.signature(SurfaceSplatting.forward)
    assert ref["SurfaceSplatting.forward"][:3] == list(f_our.parameters)[:3]   # self, point_clouds, point_clouds_filter
