"""Parity of the CUDA path (through the C ABI, via the torch binding) — needs a B200.

Three independent checkers, strongest first:
  1. tests/golden/*.npz — outputs of the UNMODIFIED reference run on a B200 (tools/make_golden.py).
     Forward quantities must match BIT FOR BIT (uv, conic, tile lists, image, per-pixel state);
     gradients within max(1e-4, 10 x the reference's own run-to-run noise) of max|ref| (fp32 atomics
     make the reference itself nondeterministic, SURVEY.md Q18).
  2. tests/golden/ref_*.npz — what the compiled reference computed on bigger scenes (100k and 3M gaussians):
     forward quantities as bit digests, gradients as seeded row samples with max|ref| (tests/scenes.py);
     the drop-in test runs the reference's own python on this library when oracle/_ref is built.
  3. the CPU oracle (oracle/cpu_oracle.py), tolerance 1e-4 rel fp32 (north_star), which differs from the
     GPU only in the transcendental functions.
plus size-independent properties at BASELINE.json's full size (1080p, 3M gaussians).
"""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import gaussian_splatting_b200 as gsb
from gaussian_splatting_b200 import synth
from gaussian_splatting_b200.rasterize import rasterize, rasterize_unfused
from gaussian_splatting_b200.structs import Camera, Gaussians
from oracle import cpu_oracle as orc
from oracle import ref_loader
from tests import scenes

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden"
REL_TOL = 1e-4  # BASELINE.json north_star: 1e-4 rel fp32 on rendered RGB and on all returned gradients


def dev():
    return torch.device("cuda:0")


def to_t(a, dtype=None):
    x = torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    return x if dtype is None else x.to(dtype)


def rel(a, b):
    a = a.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = b.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(b) else np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)) if a.size else 0.0


def bits(a):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    return a.view(np.int32) if a.dtype == np.float32 else a


def assert_bits_equal(a, b, what):
    ba, bb = bits(a), bits(b)
    assert ba.shape == bb.shape, (what, ba.shape, bb.shape)
    bad = int((ba != bb).sum())
    assert bad == 0, f"{what}: {bad}/{ba.size} values differ bitwise from the reference"


def assert_digest(a, gd, key, what):
    """Bit-for-bit comparison with a reference array the fixture keeps as a digest (key + "_sha")."""
    assert scenes.bits_digest(a) == str(gd[key + "_sha"]), f"{what}: bits differ from the reference's"


def gaussians_from(sc, requires_grad=True):
    P = {k: to_t(sc[k]).requires_grad_(requires_grad) for k in ("xyz", "rgb", "opacity", "scale", "quaternion")}
    sh = None if sc["sh"] is None else to_t(sc["sh"]).requires_grad_(requires_grad)
    return Gaussians(P["xyz"], P["rgb"], P["opacity"], P["scale"], P["quaternion"], sh)


def run_b200(sc, fn=rasterize, bg=0.5, G=None, near=0.3, far=500.0, pad=100, mh=3.0, sh_precompute=True):
    g = gaussians_from(sc)
    cam = Camera(sc["W"], sc["H"], to_t(sc["K"]))
    image, mask, uv = fn(g, to_t(sc["T"]), cam, near, far, pad, mh, sh_precompute,
                         torch.full((3,), bg, device=dev(), dtype=g.xyz.dtype))
    out = dict(image=image.detach(), culling_mask=mask, uv=uv.detach())
    if G is not None:
        uv.retain_grad()
        image.backward(to_t(G))
        out.update(g_xyz=g.xyz.grad, g_rgb=g.rgb.grad, g_opacity=g.opacity.grad, g_scale=g.scale.grad,
                   g_quaternion=g.quaternion.grad, g_uv=uv.grad)
        if g.sh is not None:
            out["g_sh"] = g.sh.grad
    return out


def load_golden(name):
    p = GOLDEN / name
    if not p.exists():
        pytest.skip(f"{p} missing (generate with tools/make_golden.py on a GPU box)")
    return np.load(p, allow_pickle=False)


# ------------------------------------------------------------------------------------------------
# 1. golden fixtures produced by the reference's own CUDA path
# ------------------------------------------------------------------------------------------------
def test_golden_fixture6_operators_bitwise():
    """The reference's unit-test scene: every operator of the chain, bit for bit."""
    gd = load_golden("fixture6_fp32.npz")
    ext = gsb.native()
    fx = scenes.reference_fixture()
    xyz_cam = to_t(gd["st_xyz_cam"])
    K, T = to_t(fx["K"]), to_t(fx["T"])
    uv = torch.zeros(6, 2, device=dev())
    ext.camera_projection_cuda(xyz_cam, K, uv)
    assert_bits_equal(uv, gd["st_uv_all"], "uv")
    S = torch.zeros(6, 3, 3, device=dev())
    ext.compute_sigma_world_cuda(to_t(fx["quaternion"]), to_t(fx["scale"]), S)
    assert_bits_equal(S, gd["st_sigma_world"], "sigma_world")
    J = torch.zeros(6, 2, 3, device=dev())
    ext.compute_projection_jacobian_cuda(xyz_cam, K, J)
    assert_bits_equal(J, gd["st_jacobian"], "jacobian")
    conic = torch.zeros(6, 3, device=dev())
    ext.compute_conic_cuda(S, J, T, conic)
    assert_bits_equal(conic, gd["st_conic_all"], "conic")
    keep = torch.tensor([False, False, False, True, True, True], device=dev())
    idx, ranges = ext.get_sorted_gaussian_list(1024, uv[keep].contiguous(), xyz_cam[keep].contiguous(),
                                               conic[keep].contiguous(), 40, 30, 3.0)
    assert idx.numel() == 641 and ranges.numel() == 1201  # test/test_tile_culling.py:73-108
    assert_bits_equal(idx, gd["st_sorted_idx"], "sorted_gaussian_idx_by_splat_idx")
    assert_bits_equal(ranges, gd["st_tile_ranges"], "splat_start_end_idx_by_tile_idx")


@pytest.mark.parametrize("mode", ["nosh", "sh_precompute", "sh_perpixel"])
def test_golden_fixture6_rasterize(mode):
    """test/test_rasterize.py: the three end-to-end cases of the reference."""
    gd = load_golden("fixture6_fp32.npz")
    fx = scenes.reference_fixture()
    fx = dict(fx, opacity=scenes.inverse_sigmoid(fx["opacity"]))
    if mode != "nosh":
        fx["sh"] = np.full((6, 3, 15), 0.1, np.float32)
    r = run_b200(fx, bg=0.0, far=100.0, pad=10, sh_precompute=(mode != "sh_perpixel"))
    assert_bits_equal(r["culling_mask"], gd["culling_mask"], "culling_mask")
    assert_bits_equal(r["uv"], gd["uv"], "uv")
    ref_img = gd["image_" + mode]
    if mode == "sh_perpixel":  # generic kernel: same values, no bit contract (SURVEY.md §8(f) row 3)
        assert rel(r["image"], ref_img) < 1e-5
    else:
        assert_bits_equal(r["image"], ref_img, "image")


def test_render_depth_known_answers():
    """test/test_depth.py:33,36 — range to the first surface above alpha 0.2 on the reference fixture."""
    from gaussian_splatting_b200.depth import render_depth

    fx = scenes.reference_fixture()
    fx = dict(fx, opacity=scenes.inverse_sigmoid(fx["opacity"]))
    g = gaussians_from(fx, requires_grad=False)
    depth = render_depth(g, 0.2, to_t(fx["T"]), Camera(640, 480, to_t(fx["K"])), 0.3, 10, 3.0)
    assert depth.shape == (480, 640, 1)
    assert abs(depth[340, 348].item() - 17.29551887512207) < 5e-5
    assert abs(depth[200, 348].item() - 13.205718040466309) < 5e-5
    assert depth[0, 0].item() == -1.0


@pytest.mark.parametrize("name,nG,res,sig,shd", [
    ("synth_tiny", 2000, "tiny", (2.0, 0.5, 0.5, 8.0), 3),
    ("synth_small", 12000, "small", (2.5, 0.5, 0.5, 10.0), 3),
    ("synth_deep_nosh", 60000, "small", (2.5, 0.5, 0.5, 10.0), 0),  # > 960 splats in the busiest tiles (Q9)
])
@pytest.mark.parametrize("path", ["fused", "unfused"])
def test_golden_synthetic(name, nG, res, sig, shd, path):
    gd = load_golden(name + "_fp32.npz")
    sc = scenes.np_scene(nG, res, sh_degree=shd, seed=0, view=0, n_views=3, sigma_px=sig)
    G = synth.make_upstream_grad(res).numpy()
    r = run_b200(sc, fn=rasterize if path == "fused" else rasterize_unfused, G=G)
    assert_bits_equal(r["culling_mask"], gd["culling_mask"], "culling_mask")
    assert_bits_equal(r["uv"], gd["uv"], "uv")
    assert_bits_equal(r["image"], gd["image"], "image")
    noise = dict(zip(gd["ref_noise_keys"].tolist(), gd["ref_noise"].tolist()))
    for k in ("g_xyz", "g_rgb", "g_opacity", "g_scale", "g_quaternion", "g_uv", "g_sh"):
        if k == "g_sh" and not shd:
            continue
        got, ref = r[k], (gd[k] if k in gd.files else None)
        if ref is None:  # large fixtures keep every 8th row
            got, ref = got[::8], gd[k + "_rows8"]
        tol = max(REL_TOL, 10 * noise.get(k, 0.0))
        assert rel(got, ref) < tol, (k, rel(got, ref), tol)


def test_golden_tile_lists_and_pixel_state():
    """Exact tile lists and the renderer's saved per-pixel state on the fat-splat scene
    (> 960 splats in the busiest tile: multi-chunk regime of the reference, SURVEY.md Q9)."""
    gd = load_golden("synth_small_fp32.npz")
    ext = gsb.native()
    assert int(gd["max_splats_per_tile"]) > 128  # more than one TMA batch per tile
    assert int(load_golden("synth_deep_nosh_fp32.npz")["max_splats_per_tile"]) > 960  # multi-chunk regime
    keep = ~gd["culling_mask"]
    uv, conic, xyz_cam = (to_t(gd[k][keep]) for k in ("st_uv_all", "st_conic_all", "st_xyz_cam"))
    idx, ranges = ext.get_sorted_gaussian_list(1024, uv, xyz_cam, conic, 20, 12, 3.0)
    assert_bits_equal(ranges, gd["st_tile_ranges"], "tile ranges")
    assert_bits_equal(idx, gd["st_sorted_idx"], "sorted idx")
    H, W = 192, 320
    img = torch.zeros(H, W, 3, device=dev())
    npp = torch.zeros(H, W, dtype=torch.int32, device=dev())
    wl = torch.zeros(H, W, device=dev())
    ext.render_tiles_cuda(uv, to_t(gd["st_opacity_act"]).reshape(-1, 1).contiguous(), to_t(gd["st_render_rgb"]), conic,
                          torch.zeros(1, 1, 1, device=dev()), ranges, idx, torch.full((3,), 0.5, device=dev()), npp, wl, img)
    assert_bits_equal(npp, gd["num_splats_per_pixel"], "num_splats_per_pixel")
    assert_bits_equal(wl, gd["final_weight_per_pixel"], "final_weight_per_pixel")
    assert_bits_equal(img, gd["image_from_stages"], "image")


@pytest.mark.parametrize("n_sh", [1, 16])
def test_golden_fp64_operator_surface(n_sh):
    """fp64 instantiations (the reference's gradcheck dtype), N_SH = 1 and per-pixel SH-16."""
    gd = load_golden("synth_tiny_fp64.npz")
    from gaussian_splatting_b200 import cuda_autograd_functions as af
    from gaussian_splatting_b200.utils import compute_rays_in_world_frame, transform_points_torch

    sc = scenes.np_scene(128, "tiny", sh_degree=3, seed=3, view=0, n_views=3, dtype=np.float64, sigma_px=(3.0, 0.4, 1.0, 6.0))
    P = {k: to_t(sc[k]).requires_grad_(True) for k in ("xyz", "rgb", "opacity", "scale", "quaternion", "sh")}
    T64, K64 = to_t(sc["T"]), to_t(sc["K"])
    xyz_cam = transform_points_torch(P["xyz"], T64)
    uv = af.CameraPointProjection.apply(xyz_cam, K64)
    conic = af.ComputeConic.apply(af.ComputeSigmaWorld.apply(P["quaternion"], P["scale"]),
                                  af.ComputeProjectionJacobian.apply(xyz_cam, K64), T64)
    sidx, rng = to_t(gd[f"nsh{n_sh}_sorted_idx"]), to_t(gd[f"nsh{n_sh}_ranges"])
    opa = torch.sigmoid(P["opacity"])
    if n_sh == 1:
        rgb_in, rays = P["rgb"], torch.zeros(1, 1, 1, dtype=torch.float64, device=dev())
    else:
        rgb_in = torch.cat((P["rgb"].unsqueeze(2), P["sh"]), dim=2)
        rays = compute_rays_in_world_frame(Camera(64, 64, K64), T64)
    image = af.RenderImage.apply(rgb_in, opa, uv, conic, rays, rng, sidx, (64, 64),
                                 torch.full((3,), 0.5, dtype=torch.float64, device=dev()))
    image.backward(synth.make_upstream_grad("tiny", dtype=torch.float64).to(dev()))
    assert rel(image, gd[f"nsh{n_sh}_image"]) < 1e-12
    for k, v in P.items():
        key = f"nsh{n_sh}_g_{k}"
        if key in gd.files:
            assert rel(v.grad, gd[key]) < 1e-9, (k, rel(v.grad, gd[key]))


# ------------------------------------------------------------------------------------------------
# 2. the compiled reference on bigger scenes (tests/golden/ref_*.npz, tools/make_golden.py --sets comparisons)
# ------------------------------------------------------------------------------------------------
needs_ref = pytest.mark.skipif(not ref_loader.reference_available(), reason="oracle/_ref not present")
GRADS = ("g_xyz", "g_rgb", "g_opacity", "g_scale", "g_quaternion", "g_sh", "g_uv")


@pytest.mark.parametrize("pose", ["yaw", "general"])
def test_live_reference_100k_720p(pose):
    """100k gaussians, SH 3, 720p, the synthetic yaw pose and a general one: forward bit for bit with the compiled
    reference, gradients within 1e-4 of max|ref|."""
    gd = load_golden("ref_live_100k_720p.npz")
    mine = run_b200(scenes.live_720p_scene(pose), G=synth.make_upstream_grad("720p").numpy())
    for k in ("culling_mask", "uv", "image"):
        assert_digest(mine[k], gd, f"{pose}_{k}", k)
    for k in GRADS:
        assert scenes.rel_rows(mine[k], gd, f"{pose}_{k}") < REL_TOL, (k, scenes.rel_rows(mine[k], gd, f"{pose}_{k}"))


def test_live_reference_exact_arithmetic_paths():
    """Scene built to hit the forward kernel's rare exact paths (DESIGN.md 3.1): splats whose centre falls
    EXACTLY on a pixel centre (numerator 0, outside the hoisted-reciprocal division's proven range) and splats
    whose 2-D covariance determinant exceeds 1e18 (record marked unsafe) — the flagged pixels are recomputed by
    render_pixel_exact_warp.  Everything must still match the compiled reference bit for bit."""
    gd = load_golden("ref_exact_paths_tiny.npz")
    mine = run_b200(scenes.exact_paths_scene(), G=synth.make_upstream_grad("tiny").numpy())
    uvn = gd["uv"]
    assert int(((uvn == np.round(uvn)).all(1)).sum()) >= scenes.EXACT_PATHS_N_EXACT // 2  # exact centres survived culling
    assert_bits_equal(mine["culling_mask"], gd["culling_mask"], "culling_mask")
    assert_bits_equal(mine["uv"], gd["uv"], "uv")
    assert_bits_equal(mine["image"], gd["image"], "image")
    for k in ("g_xyz", "g_rgb", "g_opacity", "g_scale", "g_quaternion", "g_uv"):
        assert rel(mine[k], gd[k]) < REL_TOL, (k, rel(mine[k], gd[k]))


@pytest.mark.parametrize("H", [1080, 1088])
def test_live_reference_3M_headline(H):
    """BASELINE.json configs[2]: 3M gaussians, SH 3, 1920 x H against the compiled reference.  H = 1080 is the
    headline; H = 1088 (a multiple of 16) is the strict run, because at H % 16 != 0 the reference's forward has a
    barrier inside `if (valid_pixel)` (src/render.cu:101,164, SURVEY.md Q15) and its bottom tile row is racy for
    tiles with more than one 960-splat chunk.  Forward quantities bit for bit (bottom tile row of H = 1080: only
    where the reference agreed with itself over two runs); gradients within max(1e-4, 10 x the reference's own
    run-to-run noise) of max|ref|."""
    gd = load_golden("ref_headline_3M.npz")
    p = f"h{H}_"
    d = dev()
    names = ("xyz", "quaternion", "scale", "opacity", "rgb", "sh")
    g = synth.make_gaussians(3_000_000, "1080p", sh_degree=3, seed=0, device=d, requires_grad=True)
    cam = Camera(1920, H, synth.make_camera("1080p", device=d).K)
    T = synth.make_pose(2, 8, device=d)
    bg = torch.full((3,), 0.5, device=d)
    G = scenes.headline_upstream_grad(H).to(d)

    image, mask, uv, st = rasterize(g, T, cam, 0.3, 500.0, 100, 3.0, True, bg, return_state=True)
    uv.retain_grad()
    image.backward(G)
    n_mine, w_mine, ranges = st.n_per_pixel, st.w_per_pixel, st.ranges
    del st

    assert_digest(mask, gd, p + "culling_mask", "culling_mask")
    assert_digest(uv, gd, p + "uv", "uv")
    body = (H // 16) * 16
    assert_digest(image[:body], gd, p + "image_body", "image (full tile rows)")
    if body < H:  # ragged bottom tile row: judge only the pixels where the reference reproduced itself
        stable = torch.from_numpy(gd[p + "bottom_stable"]).to(d)
        assert float(stable.float().mean()) > 0.5
        assert_digest(image[body:][stable], gd, p + "bottom_stable", "image (bottom tile row, race-free pixels)")
    cnt = (ranges[1:] - ranges[:-1]).view((H + 15) // 16, 120)
    assert bool((n_mine <= cnt.repeat_interleave(16, 0).repeat_interleave(16, 1)[:H, :1920]).all())
    assert bool(torch.isfinite(w_mine).all())
    for k, got in [(f"g_{k}", getattr(g, k).grad) for k in names] + [("g_uv", uv.grad)]:
        noise = float(gd[p + "noise_" + k])
        tol = max(REL_TOL, 10.0 * noise)
        assert scenes.rel_rows(got, gd, p + k) < tol, (k, scenes.rel_rows(got, gd, p + k), noise)


def test_live_reference_per_pixel_sh_backward_fp32():
    """use_sh_precompute=False (per-pixel view directions, N_SH = 16) in fp32, forward AND backward against the
    compiled reference (src/render.cu:284-333, src/render_backward.cu:402-568): the golden fixtures pin the fp32
    image and the fp64 gradients of this mode, this pins the fp32 gradients."""
    gd = load_golden("ref_per_pixel_sh_small.npz")
    mine = run_b200(scenes.per_pixel_sh_scene(), G=synth.make_upstream_grad("small").numpy(), sh_precompute=False)
    assert_digest(mine["culling_mask"], gd, "culling_mask", "culling_mask")
    assert_digest(mine["uv"], gd, "uv", "uv")
    assert rel(mine["image"], gd["image"]) < 1e-5
    for k in GRADS:
        assert scenes.rel_rows(mine[k], gd, k) < REL_TOL, (k, scenes.rel_rows(mine[k], gd, k))


def test_contribution_masks_do_not_change_the_gradients():
    """The forward records which (8x4 pixel block, splat) pairs contributed and the backward visits only those;
    without the masks (GSR_NO_MASKS=1) the backward walks the forward's conservative candidate lists.  Same
    gradients either way (atomics noise), same image bits."""
    from gaussian_splatting_b200 import rasterize as R

    sc = scenes.np_scene(60_000, "720p", sh_degree=2, seed=4, view=1, n_views=3)
    G = synth.make_upstream_grad("720p").numpy()
    assert R.USE_CONTRIBUTION_MASKS
    with_masks = run_b200(sc, G=G)
    R.USE_CONTRIBUTION_MASKS = False
    try:
        without = run_b200(sc, G=G)
    finally:
        R.USE_CONTRIBUTION_MASKS = True
    assert_bits_equal(with_masks["image"], without["image"], "image")
    for k in ("g_xyz", "g_rgb", "g_opacity", "g_scale", "g_quaternion", "g_sh", "g_uv"):
        assert rel(with_masks[k], without[k]) < 2e-5, (k, rel(with_masks[k], without[k]))  # fp32 atomics noise


@pytest.mark.parametrize("sigma", [(1.2, 0.6, 0.3, 12.0), (14.0, 0.8, 2.0, 60.0)])
def test_tile_hit_masks_and_retested_tiles_give_the_same_lists(sigma):
    """The per-gaussian stage remembers which tiles of a gaussian's window it found hit (64-bit mask) and the pair
    emission only expands that mask; windows of more than 64 tiles (the second scene: footprints up to 180 px) are
    flagged and re-tested.  Either way the tile lists must be the ones GSR_RETEST_TILES=1 (re-test everything, the
    round-1 arrangement) produces, bit for bit."""
    from gaussian_splatting_b200 import rasterize as R

    d = dev()
    n = 60_000 if sigma[0] < 2 else 6_000
    g = synth.make_gaussians(n, "720p", sh_degree=0, seed=12, device=d, sigma_px=sigma)
    cam = synth.make_camera("720p", device=d)
    T = synth.make_pose(1, 3, device=d)
    bg = torch.full((3,), 0.5, device=d)
    out = {}
    for flag in (True, False):
        R.USE_TILE_MASKS = flag
        try:
            with torch.no_grad():
                image, mask, uv, st = rasterize(g, T, cam, 0.3, 500.0, 100, 3.0, True, bg, return_state=True)
            out[flag] = (image, st.ranges.clone(), st.ids_sorted.clone(), st.P)
        finally:
            R.USE_TILE_MASKS = True
    assert out[True][3] == out[False][3] and out[True][3] > 0
    assert torch.equal(out[True][1], out[False][1]), "tile ranges differ"
    assert torch.equal(out[True][2], out[False][2]), "sorted gaussian ids differ"
    assert_bits_equal(out[True][0], out[False][0], "image")


def test_record_gather_and_record_stream_agree():
    """Default: the tile kernels gather their records through the sorted keys with cp.async.  GSR_RECORD_STREAM=1:
    a separate kernel writes the tile-contiguous record stream they read with bulk copies.  Same records either way,
    so the same bits in the forward; gradients to atomics noise.  Also the id-array form of the gather (when the
    gaussian id does not fit the sort key)."""
    from gaussian_splatting_b200 import rasterize as R

    sc = scenes.np_scene(70_000, "720p", sh_degree=1, seed=8, view=0, n_views=3)
    G = synth.make_upstream_grad("720p").numpy()
    assert R.USE_RECORD_GATHER
    gathered = run_b200(sc, G=G)
    R.USE_RECORD_GATHER = False
    try:
        streamed = run_b200(sc, G=G)
    finally:
        R.USE_RECORD_GATHER = True
    assert_bits_equal(gathered["image"], streamed["image"], "image")
    assert_bits_equal(gathered["uv"], streamed["uv"], "uv")
    for k in ("g_xyz", "g_rgb", "g_opacity", "g_scale", "g_quaternion", "g_sh", "g_uv"):
        assert rel(gathered[k], streamed[k]) < 2e-5, (k, rel(gathered[k], streamed[k]))
    # far plane at infinity -> full 32-bit depth keys; 4k -> 15 tile bits: 17 bits are left for the id, so 200 000
    # gaussians do not fit and the sort carries a separate id array (the key/value fallback)
    big = scenes.np_scene(200_000, "4k", sh_degree=0, seed=9, view=0, n_views=1)
    G4 = synth.make_upstream_grad("4k").numpy()
    a = run_b200(big, G=G4, far=float("inf"))
    R.USE_RECORD_GATHER = False
    try:
        b = run_b200(big, G=G4, far=float("inf"))
    finally:
        R.USE_RECORD_GATHER = True
    assert_bits_equal(a["image"], b["image"], "image (full-range depth keys)")
    assert rel(a["g_xyz"], b["g_xyz"]) < 2e-5


def test_speculative_pair_buffers_eager_overflow_and_fit_agree():
    """rasterize() sizes the pair buffers from recent views and reads the real counts only after binning and the
    tile renderer are enqueued.  Three ways through it must give the same bits: the first view of a kind (eager
    read), a view whose pair count overflows the guess (both stages run again) and a view that fits (padding keys
    behind the real pairs)."""
    from gaussian_splatting_b200 import rasterize as R

    sc = scenes.np_scene(80_000, "720p", sh_degree=1, seed=6, view=2, n_views=3)
    G = synth.make_upstream_grad("720p").numpy()
    key = (dev().index if dev().index is not None else torch.cuda.current_device(), 80_000, sc["H"], sc["W"])
    R._PAIR_HISTORY.pop(key, None)
    eager = run_b200(sc, G=G)
    assert len(R._PAIR_HISTORY[key]) == 1
    P = R._PAIR_HISTORY[key][0]
    assert P > 100_000  # well above the 66 Ki-pair capacity of the poisoned guess below
    R._PAIR_HISTORY[key] = [1000]          # a guess far too small: capacity 66 Ki pairs < P
    overflow = run_b200(sc, G=G)
    assert R._PAIR_HISTORY[key][-1] == P
    R._PAIR_HISTORY[key] = [P]             # capacity = 1.04 P + 64 Ki: fits, with padding behind the real pairs
    fit = run_b200(sc, G=G)
    R._PAIR_HISTORY[key] = [2 * P]         # lots of padding
    loose = run_b200(sc, G=G)
    for other, name in ((overflow, "overflow"), (fit, "fit"), (loose, "loose")):
        assert_bits_equal(other["image"], eager["image"], f"image ({name})")
        assert_bits_equal(other["uv"], eager["uv"], f"uv ({name})")
        assert_bits_equal(other["culling_mask"], eager["culling_mask"], f"mask ({name})")
        for k in ("g_xyz", "g_rgb", "g_opacity", "g_scale", "g_quaternion", "g_sh"):
            assert rel(other[k], eager[k]) < 2e-5, (name, k, rel(other[k], eager[k]))
    R._PAIR_HISTORY.pop(key, None)


def test_native_camera_centre_reproduces_torch_inverse():
    """gsr_camera_centre (one kernel) against torch.inverse (the reference's op, splat_py/rasterize.py:91-93) and
    torch.linalg.inv_ex, bit for bit: the bench's pose ring, identity, random rigid poses, general matrices."""
    from gaussian_splatting_b200 import rasterize as R

    ext = gsb.native()
    rng = np.random.default_rng(11)
    mats = [synth.make_pose(v, 8).numpy() for v in range(8)] + [np.eye(4, dtype=np.float32)]
    for k in range(300):
        T = np.eye(4)
        if k % 5 == 4:
            T[:3, :] = rng.standard_normal((3, 4))
        else:
            q = rng.standard_normal(4)
            q /= np.linalg.norm(q)
            w, x, y, z = q
            T[:3, :3] = [[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                         [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                         [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]]
            T[:3, 3] = rng.standard_normal(3) * 4
        mats.append(T.astype(np.float32))
    bad = 0
    for M in mats:
        t = to_t(M)
        mine = ext.camera_centre(t)
        bad += int((bits(mine) != bits(torch.inverse(t)[:3, 3].contiguous())).any())
        bad += int((bits(mine) != bits(torch.linalg.inv_ex(t)[0][:3, 3].contiguous())).any())
    assert bad == 0, f"{bad} of {2 * len(mats)} comparisons differ"
    R._CENTRE_OK.clear()
    assert R.native_centre_ok(dev()) is True


def test_in_kernel_transform_self_check_passes_on_this_device():
    """rasterize() verifies once per device that the in-kernel world->camera transform still reproduces
    torch.matmul bit for bit (and falls back to torch.matmul itself otherwise); on the pinned torch / cuBLAS of
    this image the check must pass, i.e. the fast path is the one the other tests exercise."""
    from gaussian_splatting_b200 import rasterize as R

    R._TRANSFORM_OK.clear()
    assert R.in_kernel_transform_ok(dev()) is True


@needs_ref
def test_reference_python_runs_on_this_library():
    """Drop-in proof: the reference's own splat_py.rasterize on THIS library's `splat_cuda`."""
    ref_loader.load_reference_on_b200()
    ras = sys.modules["splat_py_on_b200.rasterize"]
    structs = sys.modules["splat_py_on_b200.structs"]
    gd = load_golden("synth_tiny_fp32.npz")
    sc = scenes.np_scene(2000, "tiny", sh_degree=3, seed=0, view=0, n_views=3, sigma_px=(2.0, 0.5, 0.5, 8.0))
    g = gaussians_from(sc)
    gr = structs.Gaussians(g.xyz, g.rgb, g.opacity, g.scale, g.quaternion, g.sh)
    image, mask, uv = ras.rasterize(gr, to_t(sc["T"]), structs.Camera(64, 64, to_t(sc["K"])), 0.3, 500.0, 100, 3.0,
                                    True, torch.full((3,), 0.5, device=dev()))
    image.backward(to_t(synth.make_upstream_grad("tiny").numpy()))
    assert_bits_equal(image, gd["image"], "image")
    assert rel(g.xyz.grad, gd["g_xyz"]) < REL_TOL and rel(g.sh.grad, gd["g_sh"]) < REL_TOL


@pytest.mark.parametrize("n", [20000, 65536, 65535 + 100, 100000, 3 * 65535 + 7])
def test_in_kernel_transform_reproduces_torch_matmul(n):
    """The fused kernel forms camera-frame positions itself (saves a 2.3 ms torch.matmul at 3M points).  Their
    bits must equal torch.matmul's — the reference's op (splat_py/utils.py:60-72) — including the short last
    chunk of cuBLAS' 65535-matrix batching, which rasterize() hands to torch."""
    from gaussian_splatting_b200 import rasterize as R
    from gaussian_splatting_b200.utils import transform_points_torch

    g = synth.make_gaussians(n, "1080p", sh_degree=0, seed=n, device=dev())
    cam = synth.make_camera("1080p", device=dev())
    rng = np.random.default_rng(n)
    q = rng.standard_normal(4)
    q /= np.linalg.norm(q)
    w, x, y, z = q
    T = np.eye(4)
    T[:3, :3] = [[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                 [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                 [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]]
    T[:3, 3] = rng.standard_normal(3)
    T = to_t(T.astype(np.float32))
    ref = transform_points_torch(g.xyz, T)
    tail = n % R.CUBLAS_BATCH_CHUNK
    cam_tail = transform_points_torch(g.xyz[n - tail:], T) if 0 < tail < R.SMALL_BATCH else None
    ext = gsb.native()
    rec, zkey, vis, scan = ext.fused_preprocess_forward(g.xyz, cam_tail, g.quaternion, g.scale, g.opacity.reshape(-1),
                                                        g.rgb, None, T, cam.K, None, 1080, 1920, -1e30, 1e30, 1e30, 3.0, 0)
    zref = ref[:, 2].contiguous().view(torch.int32)
    zref = torch.where(zref < 0, ~zref, zref | -2**31)
    assert_bits_equal(zkey, zref, "depth key (camera z)")
    uv = torch.zeros(n, 2, device=dev())
    ext.camera_projection_cuda(ref, cam.K, uv)
    ok = torch.isfinite(uv).all(dim=1) & torch.isfinite(rec[:, :2]).all(dim=1)
    assert_bits_equal(rec[:, 0:2][ok], uv[ok], "uv from in-kernel positions")


# ------------------------------------------------------------------------------------------------
# 3. the CPU oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nG,res,sig,shd", [(2000, "tiny", (2.0, 0.5, 0.5, 8.0), 3), (12000, "small", (2.5, 0.5, 0.5, 10.0), 0),
                                            (128, "tiny", (3.0, 0.4, 1.0, 6.0), 3)])
def test_against_cpu_oracle(nG, res, sig, shd):
    sc = scenes.np_scene(nG, res, sh_degree=shd, seed=1, view=2, n_views=3, sigma_px=sig)
    G = synth.make_upstream_grad(res).numpy()
    r = run_b200(sc, G=G)
    o = orc.rasterize(sc["xyz"], sc["quaternion"], sc["scale"], sc["opacity"], sc["rgb"], sc["sh"], sc["T"], sc["K"],
                      sc["H"], sc["W"], 0.3, 500.0, 100.0, 3.0, background=np.full(3, 0.5, np.float32))
    d = orc.rasterize_backward(o, G)
    assert (r["culling_mask"].cpu().numpy() == o.culling_mask).all()
    assert rel(r["uv"], o.uv) < 1e-6
    # the oracle's libm transcendentals differ from the GPU's by ulps; a pixel whose alpha sits within that
    # of the 1/255 skip threshold may flip — allow a handful, require 1e-4 everywhere else
    diff = np.abs(r["image"].cpu().numpy().astype(np.float64) - o.image)
    bad = int((diff > REL_TOL * np.abs(o.image).max()).sum())
    assert bad <= max(3, diff.size // 100000), f"{bad} image values beyond 1e-4"
    for k, ref in (("g_xyz", d.xyz), ("g_quaternion", d.quaternion), ("g_scale", d.scale), ("g_opacity", d.opacity),
                   ("g_rgb", d.rgb), ("g_uv", d.uv)):
        assert rel(r[k], ref) < 5 * REL_TOL, (k, rel(r[k], ref))
    if shd:
        assert rel(r["g_sh"], d.sh) < 5 * REL_TOL


# ------------------------------------------------------------------------------------------------
# edge cases
# ------------------------------------------------------------------------------------------------
def test_upstream_gradient_on_uv():
    """A loss that also depends on the returned uv: the fused backward must add the upstream uv gradient to the
    render's own — whether or not the render node materialises its compact uv gradient (it does only when uv.grad
    is observable: retain_grad() or a hook) — same result as the operator-by-operator chain, and uv.grad itself
    must be the chain's."""
    sc = scenes.np_scene(4000, "tiny", sh_degree=0, seed=5, sigma_px=(2.0, 0.5, 0.5, 8.0))
    G = to_t(synth.make_upstream_grad("tiny").numpy())
    cam = Camera(sc["W"], sc["H"], to_t(sc["K"]))
    bg = torch.full((3,), 0.5, device=dev())
    grads, uv_grads, hooked = {}, {}, []
    for name, fn, watch in (("fused", rasterize, None), ("fused-retain", rasterize, "retain"),
                            ("fused-hook", rasterize, "hook"), ("unfused", rasterize_unfused, "retain")):
        g = gaussians_from(sc)
        image, _, uv = fn(g, to_t(sc["T"]), cam, 0.3, 500.0, 100, 3.0, True, bg)
        if watch == "retain":
            uv.retain_grad()
        elif watch == "hook":
            uv.register_hook(lambda gr: hooked.append(gr.clone()))
        ((image * G).sum() + 1e-6 * (uv * uv).sum()).backward()
        grads[name] = (g.xyz.grad.clone(), g.scale.grad.clone())
        if watch == "retain":
            uv_grads[name] = uv.grad.clone()
    for name in ("fused", "fused-retain", "fused-hook"):
        for a, b in zip(grads[name], grads["unfused"]):
            assert rel(a, b) < REL_TOL, (name, rel(a, b))
    assert rel(uv_grads["fused-retain"], uv_grads["unfused"]) < REL_TOL
    assert len(hooked) == 1 and rel(hooked[0], uv_grads["unfused"]) < REL_TOL
    # only the render's gradient, observed: uv.grad without any upstream term
    g = gaussians_from(sc)
    image, _, uv = rasterize(g, to_t(sc["T"]), cam, 0.3, 500.0, 100, 3.0, True, bg)
    uv.retain_grad()
    (image * G).sum().backward()
    g2 = gaussians_from(sc)
    image2, _, uv2 = rasterize(g2, to_t(sc["T"]), cam, 0.3, 500.0, 100, 3.0, True, bg)
    (image2 * G).sum().backward()
    assert uv2.grad is None and float(uv.grad.abs().max()) > 0
    assert rel(g2.xyz.grad, g.xyz.grad) < 1e-5 and rel(g2.scale.grad, g.scale.grad) < 1e-5


def test_everything_culled_gives_background():
    sc = scenes.np_scene(64, "tiny", sh_degree=0, seed=0)
    sc["xyz"] = sc["xyz"].copy()
    sc["xyz"][:, 2] = -5.0  # behind the camera
    r = run_b200(sc, G=synth.make_upstream_grad("tiny").numpy())
    assert bool(r["culling_mask"].all()) and r["uv"].shape == (0, 2)
    assert torch.equal(r["image"], torch.full_like(r["image"], 0.5))
    assert float(r["g_xyz"].abs().max()) == 0.0


def test_empty_scene():
    sc = scenes.np_scene(64, "tiny", sh_degree=0, seed=0)
    sc = {k: (v[:0] if isinstance(v, np.ndarray) and v.shape[:1] == (64,) else v) for k, v in sc.items()}
    r = run_b200(sc)
    assert r["uv"].shape == (0, 2) and torch.equal(r["image"], torch.full_like(r["image"], 0.5))


def test_ragged_image_sizes():
    """H, W not multiples of 16 (1080 = 67.5 tiles): edge tiles render and differentiate correctly."""
    sc = scenes.np_scene(3000, "tiny", sh_degree=0, seed=2, sigma_px=(2.0, 0.5, 0.5, 8.0))
    sc["H"], sc["W"] = 50, 37
    sc["K"] = sc["K"].copy()
    sc["K"][0, 2], sc["K"][1, 2] = 18.5, 25.0
    G = np.random.default_rng(0).standard_normal((50, 37, 3)).astype(np.float32) / (3 * 50 * 37)
    r = run_b200(sc, G=G)
    o = orc.rasterize(sc["xyz"], sc["quaternion"], sc["scale"], sc["opacity"], sc["rgb"], None, sc["T"], sc["K"], 50, 37,
                      0.3, 500.0, 100.0, 3.0, background=np.full(3, 0.5, np.float32))
    d = orc.rasterize_backward(o, G)
    assert rel(r["image"], o.image) < REL_TOL and rel(r["g_xyz"], d.xyz) < 5 * REL_TOL


def test_deep_tile_and_saturation():
    """Thousands of opaque splats stacked in one tile: many TMA batches, every pixel saturates, the CTA
    stops early; the backward starts at the saturation depth."""
    n = 6000
    rng = np.random.default_rng(0)
    sc = scenes.np_scene(n, "tiny", sh_degree=0, seed=0)
    sc["xyz"] = np.stack([rng.uniform(-0.05, 0.05, n), rng.uniform(-0.05, 0.05, n), rng.uniform(2, 9, n)], 1).astype(np.float32)
    sc["scale"] = np.log(np.full((n, 3), 0.05, np.float32))
    sc["opacity"] = np.full((n, 1), 3.0, np.float32)
    G = synth.make_upstream_grad("tiny").numpy()
    r = run_b200(sc, G=G)
    o = orc.rasterize(sc["xyz"], sc["quaternion"], sc["scale"], sc["opacity"], sc["rgb"], None, sc["T"], sc["K"], 64, 64,
                      0.3, 500.0, 100.0, 3.0, background=np.full(3, 0.5, np.float32))
    assert o.n.max() < len(o.sorted_idx)  # saturation really cut the walk short
    assert (np.diff(o.ranges).max()) > 2000
    d = orc.rasterize_backward(o, G)
    diff = np.abs(r["image"].cpu().numpy().astype(np.float64) - o.image)
    assert int((diff > REL_TOL).sum()) <= 3
    assert rel(r["g_opacity"], d.opacity) < 5 * REL_TOL and rel(r["g_xyz"], d.xyz) < 5 * REL_TOL


def test_fp64_gradcheck_render_image():
    """The reference's own style of test (test/test_rasterize_autograd.py): fp64 gradcheck of RenderImage."""
    from gaussian_splatting_b200.cuda_autograd_functions import RenderImage

    d = dev()
    uvs = torch.tensor([[15.0, 10.0], [30.0, 20.0], [22.0, 14.0]], dtype=torch.float64, device=d, requires_grad=True)
    conic = torch.tensor([[40.0, 6.0, 30.0], [55.0, -8.0, 25.0], [20.0, 2.0, 45.0]], dtype=torch.float64, device=d,
                         requires_grad=True)
    opacity = torch.tensor([[0.8], [0.6], [0.9]], dtype=torch.float64, device=d, requires_grad=True)
    rgb = torch.rand(3, 3, dtype=torch.float64, device=d, requires_grad=True)
    xyz_cam = torch.tensor([[0, 0, 2.0], [0, 0, 3.0], [0, 0, 4.0]], dtype=torch.float32, device=d)
    idx, ranges = gsb.native().get_sorted_gaussian_list(1024, uvs.detach().float().contiguous(), xyz_cam,
                                                        conic.detach().float().contiguous(), 4, 3, 3.0)
    rays = torch.zeros(1, 1, 1, dtype=torch.float64, device=d)
    bg = torch.full((3,), 0.5, dtype=torch.float64, device=d)
    assert torch.autograd.gradcheck(lambda r, o, u, c: RenderImage.apply(r, o, u, c, rays, ranges, idx, (40, 60), bg),
                                    (rgb, opacity, uvs, conic), atol=1e-6, raise_exception=True)


# ------------------------------------------------------------------------------------------------
# 4. size-independent properties at full size (1080p, 3M gaussians, SH 3)
# ------------------------------------------------------------------------------------------------
def test_full_size_properties():
    d = dev()
    g = synth.make_gaussians(3_000_000, "1080p", sh_degree=3, seed=0, device=d, requires_grad=True)
    cam = synth.make_camera("1080p", device=d)
    T = synth.make_pose(0, 8, device=d)
    bg = torch.full((3,), 0.5, device=d)
    G = synth.make_upstream_grad("1080p", device=d)
    image, mask, uv, st = rasterize(g, T, cam, 0.3, 500.0, 100, 3.0, True, bg, return_state=True)
    image.backward(G)
    grads1 = [p.grad.clone() for p in (g.xyz, g.quaternion, g.scale, g.opacity, g.rgb, g.sh)]
    # tile ranges: monotone, cover exactly P pairs; per-tile lists are depth sorted, ties by gaussian index
    ranges = st.ranges.long()
    assert ranges[0] == 0 and ranges[-1] == st.P and bool((ranges[1:] >= ranges[:-1]).all())
    z = (T[2, :3] @ g.xyz.detach().T + T[2, 3])
    zs = z[st.ids_sorted.long()]
    tile_of = torch.bucketize(torch.arange(st.P, device=d), ranges[1:], right=True)
    same = tile_of[1:] == tile_of[:-1]
    assert bool((zs[1:][same] >= zs[:-1][same] - 1e-4).all())
    # culled gaussians get exactly zero gradient; everything finite
    assert int((~mask).sum()) == st.M == uv.shape[0]
    for gr in grads1:
        assert bool(torch.isfinite(gr).all())
        assert float(gr[mask].abs().max()) == 0.0
    assert bool(torch.isfinite(image).all())  # (colours may be negative: SH terms are unclamped, as in the reference)
    # per-pixel walk length never exceeds the tile's list
    cnt = (ranges[1:] - ranges[:-1]).view(68, 120)
    npp = st.n_per_pixel
    assert bool((npp <= cnt.repeat_interleave(16, 0).repeat_interleave(16, 1)[:1080, :1920]).all())
    # forward is deterministic (bit-identical twice); gradients agree to atomics noise
    for p in (g.xyz, g.quaternion, g.scale, g.opacity, g.rgb, g.sh):
        p.grad = None
    image2, _, _ = rasterize(g, T, cam, 0.3, 500.0, 100, 3.0, True, bg)
    image2.backward(G)
    assert torch.equal(image2, image)
    for a, b in zip(grads1, (g.xyz.grad, g.quaternion.grad, g.scale.grad, g.opacity.grad, g.rgb.grad, g.sh.grad)):
        assert rel(b, a) < 1e-5
    # linearity of the backward in the upstream gradient
    for p in (g.xyz, g.quaternion, g.scale, g.opacity, g.rgb, g.sh):
        p.grad = None
    image3, _, _ = rasterize(g, T, cam, 0.3, 500.0, 100, 3.0, True, bg)
    image3.backward(2.0 * G)
    assert rel(g.rgb.grad, 2.0 * grads1[4]) < 1e-5 and rel(g.xyz.grad, 2.0 * grads1[0]) < 1e-5
