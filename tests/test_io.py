"""Host-side data formats (SURVEY.md section 8(f) row 4): PLY read/write and data_dict.npz."""
import os

import numpy as np
import pytest
import torch

from dss_b200.core.camera import FoVPerspectiveCameras, look_at_view_transform
from dss_b200.utils import MVRData, decompose_to_R_and_t, read_ply, save_ply

# the first 1100 vertices of three of the reference's example clouds, byte for byte (header count adjusted)
REF_PLY = os.path.join(os.path.dirname(__file__), "golden", "reference", "pointclouds")


@pytest.mark.parametrize("binary", [True, False])
@pytest.mark.parametrize("with_alpha", [False, True])
def test_ply_round_trip(tmp_path, binary, with_alpha):
    rng = np.random.default_rng(0)
    pts = rng.standard_normal((257, 3)).astype(np.float32)
    nrm = rng.standard_normal((257, 3)).astype(np.float32)
    col = rng.integers(0, 256, (257, 4 if with_alpha else 3)).astype(np.float32) / 255.0
    f = str(tmp_path / "sub" / "cloud.ply")              # the directory is created like the reference does
    save_ply(f, pts, colors=col, normals=nrm, binary=binary)
    got = read_ply(f)
    assert np.array_equal(got["points"], pts) if binary else np.allclose(got["points"], pts, rtol=0, atol=0)
    assert np.array_equal(got["normals"], nrm)
    assert np.allclose(got["colors"], col, atol=1e-6)      # stored as uint8 (x255), read back / 255
    head = open(f, "rb").read(200).decode("ascii", "replace")
    assert "element vertex 257" in head and "property float nx" in head and "property uchar red" in head
    assert ("binary_little_endian" in head) == binary


def test_ply_2d_points_and_no_attributes(tmp_path):
    pts = np.random.default_rng(1).random((10, 2)).astype(np.float32)
    f = str(tmp_path / "p.ply")
    save_ply(f, pts)
    got = read_ply(f)
    assert got["normals"] is None and got["colors"] is None
    assert np.array_equal(got["points"][:, :2], pts) and (got["points"][:, 2] == 0).all()
    with pytest.raises(ValueError):
        save_ply(f, pts, colors=np.zeros((9, 3)))


@pytest.mark.parametrize("name", ["teapot_normal_dense", "bunny-8000", "sphere_2k"])
def test_reads_the_reference_example_clouds(name):
    d = read_ply(os.path.join(REF_PLY, name + ".ply"))
    assert d["points"].shape[1] == 3 and len(d["points"]) > 1000 and np.isfinite(d["points"]).all()
    assert d["normals"] is not None and d["normals"].shape == d["points"].shape
    n = np.linalg.norm(d["normals"], axis=1)
    assert np.isfinite(n).all() and np.median(n) > 0       # (bunny-8000 ships un-normalised normals)


def test_data_dict_cloud_and_cameras(tmp_path):
    rng = np.random.default_rng(2)
    P, V = 500, 6
    pts = rng.standard_normal((P, 3)).astype(np.float32)
    nrm = pts / np.linalg.norm(pts, axis=1, keepdims=True)
    R, T = look_at_view_transform(dist=torch.full((V,), 2.0), elev=torch.linspace(-30, 30, V), azim=torch.linspace(0, 300, V))
    cam = torch.zeros(V, 4, 4)
    cam[:, :3, :3], cam[:, 3, :3], cam[:, 3, 3] = R, T, 1.0      # row-vector world-to-view, as the reference stores it
    np.savez(tmp_path / "data_dict.npz", points=pts, normals=nrm, colors=np.ones_like(pts), camera_mat=cam.tolist())
    data = MVRData(str(tmp_path))
    assert len(data) == V and data[V + 1]["camera_mat"].shape == (4, 4)
    pcl = data.get_pointclouds()
    assert len(pcl) == 1 and torch.equal(pcl.points_packed(), torch.from_numpy(pts))
    cams = data.get_cameras(znear=0.1, zfar=100.0)
    want = FoVPerspectiveCameras(znear=0.1, zfar=100.0, R=R, T=T)
    assert torch.allclose(cams.get_world_to_view_transform().get_matrix(), want.get_world_to_view_transform().get_matrix())
    assert torch.allclose(cams.get_full_projection_transform().get_matrix(), want.get_full_projection_transform().get_matrix())
    Rd, td = decompose_to_R_and_t(cam)
    assert torch.equal(Rd, R) and torch.equal(td, T)
    one = data.get_cameras(camera_mat=data[2]["camera_mat"], znear=0.1)
    assert len(one) == 1
    with pytest.raises(ValueError):
        MVRData(str(tmp_path), images=[0] * (V - 1))


def test_mvr_data_reads_images_and_masks_like_the_reference(tmp_path):
    """DSS/utils/dataset.py:36-101,171-211: files of <dir>/image and <dir>/mask (sorted, by extension), rgb (3,H,W) in
    [0,1], mask (1,H,W) 0/1, one camera_mat per image; unequal counts are an error."""
    import numpy as np
    import torch
    from PIL import Image
    from dss_b200.utils.dataset import MVRData
    rng = np.random.default_rng(0)
    n, H, W = 3, 12, 16
    (tmp_path / "image").mkdir()
    (tmp_path / "mask").mkdir()
    imgs, masks = [], []
    for i in range(n):
        a = rng.integers(0, 256, (H, W, 4), dtype=np.uint8)          # RGBA on disk: alpha is dropped (dataset.py:91)
        m = (rng.random((H, W)) > 0.5).astype(np.uint8) * 255
        Image.fromarray(a, "RGBA").save(tmp_path / "image" / ("%03d.png" % i))
        Image.fromarray(m, "L").save(tmp_path / "mask" / ("%03d.png" % i))
        imgs.append(a[..., :3].astype(np.float32).transpose(2, 0, 1) / 255.0)
        masks.append((m > 0).astype(np.float32)[None])
    (tmp_path / "image" / "notes.txt").write_text("ignored: wrong extension")
    cams = np.tile(np.eye(4, dtype=np.float32), (n, 1, 1))
    cams[:, 3, 2] = [1.5, 2.0, 2.5]
    np.savez(tmp_path / "data_dict.npz", camera_mat=cams, points=rng.random((10, 3)), normals=rng.random((10, 3)))
    data = MVRData(str(tmp_path))
    assert len(data) == n and data.resolution == (H, W)
    for i in range(n):
        item = data[i]
        assert item["img.rgb"].shape == (3, H, W) and item["img.mask"].shape == (1, H, W)
        np.testing.assert_allclose(item["img.rgb"].numpy(), imgs[i], atol=1e-7)
        np.testing.assert_array_equal(item["img.mask"].numpy(), masks[i])
        np.testing.assert_array_equal(item["camera_mat"], cams[i])
    batch = data.pinned_batch([2, 0])
    assert batch["img.rgb"].shape == (2, 3, H, W) and batch["camera_mat"].shape == (2, 4, 4)
    np.testing.assert_allclose(batch["img.rgb"][0].numpy(), imgs[2], atol=1e-7)
    (tmp_path / "mask" / "002.png").unlink()
    with pytest.raises(ValueError, match="unequal number"):
        MVRData(str(tmp_path))
