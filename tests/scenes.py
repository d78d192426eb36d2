"""Shared scene builders for the tests (numpy views of gaussian_splatting_b200.synth scenes and the
reference's 6-gaussian fixture, test/gaussian_test_data.py:7-79, restated), and the two compact forms in which
tests/golden/ keeps reference outputs too large to store whole."""
import hashlib

import numpy as np
import torch

from gaussian_splatting_b200 import synth

SH0 = 0.28209479177387814
SAMPLE_ROWS = 512  # rows of a large gradient a fixture keeps (plus the row holding its largest value)


def bits_digest(a):
    """sha256 of an array's dtype, shape and exact bits: a bit-for-bit comparison with an array not stored."""
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def value_digest(t):
    """bits_digest of a float tensor with -0.0 read as +0.0: equal digests <=> torch.equal."""
    return bits_digest(t.detach() + 0.0)


def sample_rows(ref, candidates, seed):
    """Sorted row indices a fixture keeps of `ref`: SAMPLE_ROWS seeded draws among `candidates` plus the row of
    max |ref|, so that the sample always holds the value that sets the denominator of a relative error."""
    ref = np.asarray(ref)
    rng = np.random.default_rng(seed)
    rows = rng.choice(candidates, size=min(SAMPLE_ROWS, len(candidates)), replace=False) if len(candidates) else []
    top = np.unravel_index(int(np.abs(ref).argmax()), ref.shape)[0] if ref.size else None
    rows = np.union1d(rows, [] if top is None else [top])
    return rows.astype(np.int64)


def keep_rows(d, key, ref, candidates, seed):
    """Store `ref` in fixture dict `d` as key_shape, key_at (rows), key_rows (their values) and key_absmax."""
    ref = np.asarray(ref)
    at = sample_rows(ref, candidates, seed)
    d[key + "_shape"], d[key + "_at"], d[key + "_rows"] = np.array(ref.shape, np.int64), at, ref[at]
    d[key + "_absmax"] = np.float64(np.abs(ref).max() if ref.size else 0.0)


def rel_rows(got, gd, key):
    """max |got - ref| / max |ref| over the rows fixture `gd` kept of `key` (denominator: the whole array's)."""
    got = got.detach().cpu().numpy() if torch.is_tensor(got) else np.asarray(got)
    at, ref = gd[key + "_at"], gd[key + "_rows"]
    assert got.shape == tuple(gd[key + "_shape"]), (key, got.shape, tuple(gd[key + "_shape"]))
    if not at.size:
        return 0.0
    diff = np.abs(got[at].astype(np.float64) - ref.astype(np.float64)).max()
    return float(diff / max(float(gd[key + "_absmax"]), 1e-30))


def np_scene(n, res, sh_degree=3, seed=0, view=0, n_views=3, dtype=np.float32, sigma_px=(1.2, 0.6, 0.3, 12.0)):
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    g = synth.make_gaussians(n, res, sh_degree=sh_degree, seed=seed, dtype=tdt, sigma_px=sigma_px)
    cam = synth.make_camera(res, dtype=tdt)
    T = synth.make_pose(view, n_views, dtype=tdt)
    a = lambda t: None if t is None else t.detach().numpy()  # noqa: E731
    return dict(xyz=a(g.xyz), quaternion=a(g.quaternion), scale=a(g.scale), opacity=a(g.opacity), rgb=a(g.rgb),
                sh=a(g.sh), T=a(T), K=a(cam.K), H=cam.height, W=cam.width)


def general_pose():
    """A pose with roll, pitch and translation (no symmetry of the synthetic scenes' yaw ring)."""
    c, s = np.cos(0.3), np.sin(0.3)
    R = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]], np.float64) @ np.array([[1, 0, 0], [0, 0.995, -0.0998], [0, 0.0998, 0.995]])
    T = np.eye(4)
    T[:3, :3], T[:3, 3] = R, [0.13, -0.21, 0.37]
    return T.astype(np.float32)


def live_720p_scene(pose):
    """100k gaussians, SH 3, 720p; pose "yaw" (the synthetic ring) or "general" (general_pose())."""
    sc = np_scene(100_000, "720p", sh_degree=3, seed=0, view=0, n_views=3)
    if pose == "general":
        sc["T"] = general_pose()
    return sc


EXACT_PATHS_N_EXACT = 300


def exact_paths_scene():
    """Scene built to hit the forward kernel's rare exact paths (DESIGN.md 3.1): splats whose centre falls EXACTLY
    on a pixel centre and splats whose 2-D covariance determinant exceeds 1e18."""
    rng = np.random.default_rng(7)
    sc = np_scene(3000, "tiny", sh_degree=0, seed=3, sigma_px=(2.0, 0.5, 0.5, 8.0))
    sc["K"] = np.array([[64, 0, 32], [0, 64, 32], [0, 0, 1]], np.float32)  # powers of two: u = 64*x/z + 32 is exact
    sc["T"] = np.eye(4, dtype=np.float32)
    n_exact, n_huge = EXACT_PATHS_N_EXACT, 12
    z = np.full(n_exact, 2.0, np.float32)
    px, py = rng.integers(0, 64, n_exact), rng.integers(0, 64, n_exact)
    sc["xyz"][:n_exact] = np.stack([(px - 32) / 64.0 * z, (py - 32) / 64.0 * z, z], 1).astype(np.float32)
    sc["xyz"][n_exact:n_exact + n_huge, 2] = 2.0
    sc["scale"][n_exact:n_exact + n_huge] = 7.5       # exp(7.5) = 1808 world units -> det(Sigma_2D) ~ 1e19
    sc["opacity"][n_exact:n_exact + n_huge] = -3.0
    return sc


def per_pixel_sh_scene():
    """20k gaussians, SH 3, 320x192, fat splats: the fp32 per-pixel SH (use_sh_precompute=False) comparison."""
    return np_scene(20_000, "small", sh_degree=3, seed=5, view=1, n_views=3, sigma_px=(2.5, 0.5, 0.5, 10.0))


def headline_upstream_grad(H):
    """The upstream image gradient of the 3M-gaussian 1920 x H comparison (CPU, float32)."""
    gen = torch.Generator().manual_seed(1)
    return (torch.randn(H, 1920, 3, generator=gen, dtype=torch.float64) / (3.0 * H * 1920)).float()


def colmap_scene(mk):
    """Poses, image names, points and colours the COLMAP writers of tools/e2e/make_colmap_scene.py (`mk`) write."""
    poses = [mk.look_at(np.array([4 * np.cos(a), 4 * np.sin(a), 1.2 + 0.8 * np.sin(3 * a)])) for a in np.linspace(0, 6.2, 17)]
    names = [f"view_{i:03d}.png" for i in range(len(poses))]
    xyz = np.random.default_rng(0).standard_normal((50, 3))
    rgb = np.random.default_rng(1).integers(0, 256, (50, 3)).astype(np.uint8)
    return poses, names, xyz, rgb


def reference_fixture(dtype=np.float32):
    """The reference's own unit-test scene: 6 gaussians, 640x480 camera, tilted pose."""
    xyz = np.array([[1, 2, -4], [4, 5, 6], [7, 8, -9], [1, 2, 15], [2.5, -1, 4], [-1, -2, 10]], dtype)
    rgb = np.full((6, 3), 0.5, dtype)
    rgb[3], rgb[4], rgb[5] = [0.5, 0, 0], [0, 0.5, 0], [0, 0, 0.5]
    rgb = (rgb / dtype(SH0)).astype(dtype)
    opacity = np.ones((6, 1), dtype)
    scale = np.log(np.array([[0.02, 0.03, 0.04], [0.01, 0.05, 0.02], [0.09, 0.03, 0.01], [1, 3, 0.1], [2, 0.2, 0.1],
                             [2, 1, 0.1]], dtype))
    quaternion = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [1, 0, 0, 0], [0.714, -0.002, -0.664, 0.221],
                           [1, 0, 0, 0]], dtype)
    K = np.array([[430, 0, 320], [0, 410, 240], [0, 0, 1]], dtype)
    T = np.array([[0.9999, 0.0089, 0.0073, -0.3283], [-0.0106, 0.9568, 0.2905, -1.9260],
                  [-0.0044, -0.2906, 0.9568, 2.9581], [0, 0, 0, 1]], dtype)
    return dict(xyz=xyz, quaternion=quaternion, scale=scale, opacity=opacity, rgb=rgb, sh=None, T=T, K=K, H=480, W=640)


def inverse_sigmoid(x):
    p = np.clip(x, 1e-4, 1 - 1e-4)
    return np.log(p / (1 - p)).astype(x.dtype)
