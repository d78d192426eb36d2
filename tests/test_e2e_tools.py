"""tools/e2e (reference trainer on a synthetic COLMAP scene): the scene writer's binary files are the ones the
reference's own COLMAP reader read back correctly (tests/golden/ref_colmap_reader.npz), and the SSIM stand-in
behaves like an SSIM."""
import importlib.util
import sys
from pathlib import Path

import numpy as np
import torch

from tests import scenes

ROOT = Path(__file__).resolve().parents[1]
E2E = ROOT / "tools" / "e2e"


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, str(path))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_colmap_writers_round_trip_through_the_reference_reader(tmp_path):
    """The writers still write the files the reference's reader was given (bytes equal, float64 fields to 1e-12),
    and what the reader returned from them is the scene that was written."""
    gd = np.load(ROOT / "tests" / "golden" / "ref_colmap_reader.npz")
    mk = _load(E2E / "make_colmap_scene.py", "make_colmap_scene")
    poses, names, xyz, rgb = scenes.colmap_scene(mk)
    mk.write_cameras(tmp_path / "cameras.bin", 640, 416, 560.0, 561.0, 320.0, 208.0)
    mk.write_images(tmp_path / "images.bin", poses, names)
    mk.write_points(tmp_path / "points3D.bin", xyz, rgb)
    for f in ("cameras", "images", "points3D"):
        got, ref = np.frombuffer((tmp_path / f"{f}.bin").read_bytes(), np.uint8), gd[f + "_bytes"]
        assert got.shape == ref.shape, f
        fields = (gd[f + "_f64_at"][:, None] + np.arange(8)).ravel()
        rest = np.ones(ref.size, bool)
        rest[fields] = False
        assert (got[rest] == ref[rest]).all(), f
        assert np.abs(got[fields].view("<f8") - ref[fields].view("<f8")).max() <= 1e-12, f
    assert gd["cam_ids"].tolist() == [1] and gd["cam_model"].tolist() == ["PINHOLE"]
    assert gd["cam_size"][0].tolist() == [640, 416] and np.allclose(gd["cam_params"][0], [560.0, 561.0, 320.0, 208.0])
    assert gd["img_ids"].tolist() == list(range(1, len(poses) + 1))
    for i, T in enumerate(poses):
        assert gd["img_names"][i] == names[i] and gd["img_camera_ids"][i] == 1
        assert np.abs(gd["img_rotmat"][i] - T[:3, :3]).max() < 1e-12
        assert np.abs(gd["img_tvec"][i] - T[:3, 3]).max() < 1e-12
    assert gd["pt_ids"].tolist() == list(range(1, 51))
    assert np.allclose(gd["pt_xyz"][6], xyz[6]) and (gd["pt_rgb"][6] == rgb[6]).all()


def test_ssim_shim_is_an_ssim():
    sys.path.insert(0, str(E2E / "shims"))
    try:
        from torchmetrics.image import StructuralSimilarityIndexMeasure
    finally:
        sys.path.remove(str(E2E / "shims"))
    ssim = StructuralSimilarityIndexMeasure(data_range=1.0)
    g = torch.Generator().manual_seed(0)
    a = torch.rand(1, 3, 48, 64, generator=g)
    b = torch.rand(1, 3, 48, 64, generator=g)
    assert abs(float(ssim(a, a)) - 1.0) < 1e-6
    assert abs(float(ssim(a, b)) - float(ssim(b, a))) < 1e-6 and float(ssim(a, b)) < 0.2
    noisy = (a + 0.05 * torch.randn(a.shape, generator=g)).clamp(0, 1)
    assert float(ssim(a, b)) < float(ssim(a, noisy)) < 1.0
    x = a.clone().requires_grad_(True)
    (1.0 - ssim(x, b)).backward()
    assert torch.isfinite(x.grad).all() and float(x.grad.abs().sum()) > 0
