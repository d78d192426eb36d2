"""Generate tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref: its CUDA extension +
its splat_py package, built by oracle/build_ref.py) on a B200:

    python tools/make_golden.py --out <dir> [--sets fixtures comparisons densify colmap]   # then copy into tests/golden/

Scenes are regenerated from seeds by the tests (gaussian_splatting_b200.synth / tests/scenes.py); the
fixtures hold only the reference's OUTPUTS.  Nothing here touches the product code.

  fixtures     fixture6 / synth_* : per-operator outputs, images and gradients of small scenes
  comparisons  ref_*.npz : what the tests comparing with the reference at 100k / 3M gaussians check, in the
               compact forms of tests/scenes.py (bit digests, seeded row samples of the gradients)
  densify      ref_densify_trainer.npz : the reference trainer's densification of a 100k-gaussian case
  colmap       ref_colmap_reader.npz : files of tools/e2e/make_colmap_scene.py and what the reference's
               COLMAP reader read from them (CPU only)
"""
from __future__ import annotations

import argparse
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from gaussian_splatting_b200 import synth  # noqa: E402  (scene generator only)
from oracle import ref_loader  # noqa: E402
from tests import scenes  # noqa: E402

SMALL_SIGMA = (2.5, 0.5, 0.5, 10.0)


def t(a, dev, dtype=None):
    x = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return x if dtype is None else x.to(dtype)


def n(x):
    return x.detach().cpu().numpy()


def run_rasterize(ref, sc, dev, use_sh_precompute=True, bg=0.0, G=None, near=0.3, far=500.0, pad=100, mh=3.0):
    ras = sys.modules["splat_py_ref.rasterize"]
    structs = sys.modules["splat_py_ref.structs"]
    P = {k: t(sc[k], dev).requires_grad_(True) for k in ("xyz", "rgb", "opacity", "scale", "quaternion")}
    sh = None if sc["sh"] is None else t(sc["sh"], dev).requires_grad_(True)
    g = structs.Gaussians(P["xyz"], P["rgb"], P["opacity"], P["scale"], P["quaternion"], sh)
    cam = structs.Camera(sc["W"], sc["H"], t(sc["K"], dev))
    background = torch.full((3,), bg, device=dev, dtype=P["xyz"].dtype)
    image, mask, uv = ras.rasterize(g, t(sc["T"], dev), cam, near, far, pad, mh, use_sh_precompute, background)
    out = dict(image=n(image), culling_mask=n(mask), uv=n(uv))
    if G is not None:
        uv.retain_grad()
        image.backward(t(G, dev))
        out.update(g_xyz=n(P["xyz"].grad), g_rgb=n(P["rgb"].grad), g_opacity=n(P["opacity"].grad),
                   g_scale=n(P["scale"].grad), g_quaternion=n(P["quaternion"].grad), g_uv=n(uv.grad))
        if sh is not None:
            out["g_sh"] = n(sh.grad)
    return out


def stages(ref_ext, sc, dev, near=0.3, far=500.0, pad=100, mh=3.0):
    """Per-operator outputs of the reference on one scene (fp32)."""
    utils = sys.modules["splat_py_ref.utils"]
    N = sc["xyz"].shape[0]
    xyz, q, s, K, T = (t(sc[k], dev) for k in ("xyz", "quaternion", "scale", "K", "T"))
    xyz_cam = utils.transform_points_torch(xyz, T)
    uv = torch.zeros(N, 2, device=dev)
    ref_ext.camera_projection_cuda(xyz_cam, K, uv)
    S = torch.zeros(N, 3, 3, device=dev)
    ref_ext.compute_sigma_world_cuda(q, s, S)
    J = torch.zeros(N, 2, 3, device=dev)
    ref_ext.compute_projection_jacobian_cuda(xyz_cam, K, J)
    conic = torch.zeros(N, 3, device=dev)
    ref_ext.compute_conic_cuda(S, J, T, conic)
    W, H = sc["W"], sc["H"]
    mask = ((xyz_cam[:, 2] < near) | (xyz_cam[:, 2] > far) | (uv[:, 0] < -pad) | (uv[:, 0] > W + pad)
            | (uv[:, 1] < -pad) | (uv[:, 1] > H + pad))
    keep = ~mask
    uvk, xk, ck = uv[keep].contiguous(), xyz_cam[keep].contiguous(), conic[keep].contiguous()
    sorted_idx, ranges = ref_ext.get_sorted_gaussian_list(1024, uvk, xk, ck, (W + 15) // 16, (H + 15) // 16, mh)
    opa = torch.sigmoid(t(sc["opacity"], dev)[keep]).contiguous()
    rgb = t(sc["rgb"], dev)[keep].contiguous()
    if sc["sh"] is not None:
        coeffs = torch.cat((rgb.unsqueeze(2), t(sc["sh"], dev)[keep]), dim=2).contiguous()
        rgb_out = torch.zeros(uvk.shape[0], 3, device=dev)
        ref_ext.precompute_rgb_from_sh_cuda(xyz[keep].contiguous(), coeffs, torch.inverse(T).contiguous(), rgb_out)
        rgb = rgb_out
    return dict(xyz_cam=n(xyz_cam), uv_all=n(uv), sigma_world=n(S), jacobian=n(J), conic_all=n(conic),
                sorted_idx=n(sorted_idx), tile_ranges=n(ranges), opacity_act=n(opa), render_rgb=n(rgb))


def render_state(ref_ext, st, sc, dev, bg):
    """num_splats_per_pixel / final_weight_per_pixel of the reference renderer on stage outputs."""
    keep = ~((st["xyz_cam"][:, 2] < 0.3) | (st["xyz_cam"][:, 2] > 500.0) | (st["uv_all"][:, 0] < -100)
             | (st["uv_all"][:, 0] > sc["W"] + 100) | (st["uv_all"][:, 1] < -100) | (st["uv_all"][:, 1] > sc["H"] + 100))
    H, W = sc["H"], sc["W"]
    img = torch.zeros(H, W, 3, device=dev)
    npp = torch.zeros(H, W, dtype=torch.int32, device=dev)
    wl = torch.zeros(H, W, device=dev)
    ref_ext.render_tiles_cuda(t(st["uv_all"][keep], dev), t(st["opacity_act"], dev).reshape(-1, 1).contiguous(),
                              t(st["render_rgb"], dev), t(st["conic_all"][keep], dev), torch.zeros(1, 1, 1, device=dev),
                              t(st["tile_ranges"], dev), t(st["sorted_idx"], dev),
                              torch.full((3,), bg, device=dev), npp, wl, img)
    return dict(num_splats_per_pixel=n(npp).astype(np.int32), final_weight_per_pixel=n(wl), image_from_stages=n(img))


def fixtures(out, dev, ref_ext, meta):
    # A. the reference's own 6-gaussian unit-test scene (test/gaussian_test_data.py)
    fx = scenes.reference_fixture()
    stA = stages(ref_ext, fx, dev, near=0.3, far=100.0, pad=10, mh=3.0)
    fx_logit = dict(fx, opacity=scenes.inverse_sigmoid(fx["opacity"]))
    rA = run_rasterize(None, fx_logit, dev, True, 0.0, None, 0.3, 100.0, 10, 3.0)
    fx_sh = dict(fx_logit, sh=np.full((6, 3, 15), 0.1, np.float32))
    rA_sh = run_rasterize(None, fx_sh, dev, True, 0.0, None, 0.3, 100.0, 10, 3.0)
    rA_pp = run_rasterize(None, fx_sh, dev, False, 0.0, None, 0.3, 100.0, 10, 3.0)
    np.savez_compressed(out / "fixture6_fp32.npz", **{f"st_{k}": v for k, v in stA.items()},
                        image_nosh=rA["image"], image_sh_precompute=rA_sh["image"], image_sh_perpixel=rA_pp["image"],
                        culling_mask=rA["culling_mask"], uv=rA["uv"])

    # B/C. synthetic scenes: tiny (SH3, 2000 gaussians, 64x64) and small (SH3, 20000 gaussians, 320x192,
    #      fat splats: > 960 splats in some tiles, saturated pixels)
    for name, nG, res, sig, sh_deg in (("synth_tiny", 2000, "tiny", (2.0, 0.5, 0.5, 8.0), 3),
                                       ("synth_small", 12000, "small", SMALL_SIGMA, 3),
                                       ("synth_deep_nosh", 60000, "small", SMALL_SIGMA, 0)):
        sc = scenes.np_scene(nG, res, sh_degree=sh_deg, seed=0, view=0, n_views=3, sigma_px=sig)
        G = synth.make_upstream_grad(res).numpy()
        st = stages(ref_ext, sc, dev)
        rs = render_state(ref_ext, st, sc, dev, 0.5)
        r = run_rasterize(None, sc, dev, True, 0.5, G)
        r2 = run_rasterize(None, sc, dev, True, 0.5, G)  # the reference's own run-to-run noise
        noise = {k: float(np.abs(r2[k] - r[k]).max() / max(np.abs(r[k]).max(), 1e-30)) for k in r if k.startswith("g_")}
        keepers = dict(r)
        if "g_sh" in keepers and nG > 4000:
            keepers["g_sh_rows8"] = keepers.pop("g_sh")[::8].copy()
        if nG > 30000:  # keep the deep fixture small: every 8th gaussian's gradients
            for k in [k for k in keepers if k.startswith("g_") and k != "g_uv"]:
                keepers[k + "_rows8"] = keepers.pop(k)[::8].copy()
            keepers["g_uv_rows8"] = keepers.pop("g_uv")[::8].copy()
        cnt = st["tile_ranges"][1:] - st["tile_ranges"][:-1]
        np.savez_compressed(out / f"{name}_fp32.npz", **keepers, **rs,
                            **({} if nG > 30000 else dict(
                                st_uv_all=st["uv_all"], st_conic_all=st["conic_all"], st_render_rgb=st["render_rgb"],
                                st_opacity_act=st["opacity_act"], st_xyz_cam=st["xyz_cam"])),
                            st_sorted_idx=st["sorted_idx"], st_tile_ranges=st["tile_ranges"],
                            ref_noise=np.array([noise[k] for k in sorted(noise)]), ref_noise_keys=np.array(sorted(noise)),
                            max_splats_per_tile=int(cnt.max()))
        meta[name] = dict(P=int(st["sorted_idx"].size), max_splats_per_tile=int(cnt.max()), M=int((~r["culling_mask"]).sum()),
                          noise=noise, image_self_equal=bool((r2["image"] == r["image"]).all()))

    # D. fp64 operator surface (the reference's gradcheck dtype): RenderImage on 128 gaussians, 64x64,
    #    N_SH = 1 and 16 (per-pixel SH)
    af = sys.modules["splat_py_ref.cuda_autograd_functions"]
    utils = sys.modules["splat_py_ref.utils"]
    structs = sys.modules["splat_py_ref.structs"]
    sc = scenes.np_scene(128, "tiny", sh_degree=3, seed=3, view=0, n_views=3, dtype=np.float64, sigma_px=(3.0, 0.4, 1.0, 6.0))
    d64 = {}
    for n_sh in (1, 16):
        P = {k: t(sc[k], dev).requires_grad_(True) for k in ("xyz", "rgb", "opacity", "scale", "quaternion", "sh")}
        T64, K64 = t(sc["T"], dev), t(sc["K"], dev)
        xyz_cam = utils.transform_points_torch(P["xyz"], T64)
        uv = af.CameraPointProjection.apply(xyz_cam, K64)
        S = af.ComputeSigmaWorld.apply(P["quaternion"], P["scale"])
        J = af.ComputeProjectionJacobian.apply(xyz_cam, K64)
        conic = af.ComputeConic.apply(S, J, T64)
        tiles = structs.Tiles(64, 64, dev)
        sidx, rng = ref_ext.get_sorted_gaussian_list(1024, uv.detach().float().contiguous(), xyz_cam.detach().float().contiguous(),
                                                     conic.detach().float().contiguous(), tiles.x_tiles_count,
                                                     tiles.y_tiles_count, 3.0)
        opa = torch.sigmoid(P["opacity"])
        cam = structs.Camera(64, 64, K64)
        if n_sh == 1:
            rgb_in, rays = P["rgb"], torch.zeros(1, 1, 1, dtype=torch.float64, device=dev)
        else:
            rgb_in = torch.cat((P["rgb"].unsqueeze(2), P["sh"]), dim=2)
            rays = utils.compute_rays_in_world_frame(cam, T64)
        image = af.RenderImage.apply(rgb_in, opa, uv, conic, rays, rng, sidx, torch.tensor([64, 64], device=dev),
                                     torch.full((3,), 0.5, dtype=torch.float64, device=dev))
        G64 = synth.make_upstream_grad("tiny", dtype=torch.float64).to(dev)
        image.backward(G64)
        d64.update({f"nsh{n_sh}_image": n(image), f"nsh{n_sh}_sorted_idx": n(sidx), f"nsh{n_sh}_ranges": n(rng),
                    **{f"nsh{n_sh}_g_{k}": n(v.grad) for k, v in P.items() if v.grad is not None}})
    np.savez_compressed(out / "synth_tiny_fp64.npz", **d64)


GRADS = ("g_xyz", "g_rgb", "g_opacity", "g_scale", "g_quaternion", "g_sh")


def keep_comparison(d, prefix, r, seed):
    """One reference run `r` (run_rasterize with gradients): forward outputs as bit digests, gradients as seeded
    samples of the visible gaussians' rows (g_uv: of all its rows)."""
    for k in ("culling_mask", "uv", "image"):
        d[f"{prefix}{k}_sha"] = np.array(scenes.bits_digest(r[k]))
    visible = np.flatnonzero(~r["culling_mask"])
    for k in GRADS:
        if k in r:
            scenes.keep_rows(d, prefix + k, r[k], visible, seed)
    scenes.keep_rows(d, prefix + "g_uv", r["g_uv"], np.arange(len(r["g_uv"])), seed)


def comparisons(out, dev, meta):
    d = {}
    G = synth.make_upstream_grad("720p").numpy()
    for pose in ("yaw", "general"):
        r = run_rasterize(None, scenes.live_720p_scene(pose), dev, True, 0.5, G)
        keep_comparison(d, pose + "_", r, seed=0)
    np.savez_compressed(out / "ref_live_100k_720p.npz", **d)

    # small enough to keep whole
    r = run_rasterize(None, scenes.exact_paths_scene(), dev, True, 0.5, synth.make_upstream_grad("tiny").numpy())
    np.savez_compressed(out / "ref_exact_paths_tiny.npz", **r)

    r = run_rasterize(None, scenes.per_pixel_sh_scene(), dev, False, 0.5, synth.make_upstream_grad("small").numpy())
    d = dict(image=r["image"])
    for k in ("culling_mask", "uv"):
        d[k + "_sha"] = np.array(scenes.bits_digest(r[k]))
    visible = np.flatnonzero(~r["culling_mask"])
    for k in GRADS:
        scenes.keep_rows(d, k, r[k], visible, seed=0)
    scenes.keep_rows(d, "g_uv", r["g_uv"], np.arange(len(r["g_uv"])), seed=0)
    np.savez_compressed(out / "ref_per_pixel_sh_small.npz", **d)

    # 3M gaussians, SH 3, 1920 x H, pose 2 of 8; the reference twice: its run-to-run noise sets the gradient tolerance
    ras, structs = sys.modules["splat_py_ref.rasterize"], sys.modules["splat_py_ref.structs"]
    names = ("xyz", "quaternion", "scale", "opacity", "rgb", "sh")
    d = {}
    for H in (1080, 1088):
        g = synth.make_gaussians(3_000_000, "1080p", sh_degree=3, seed=0, device=dev, requires_grad=True)
        gr = structs.Gaussians(g.xyz, g.rgb, g.opacity, g.scale, g.quaternion, g.sh)
        camr = structs.Camera(1920, H, synth.make_camera("1080p", device=dev).K)
        T, bg, G = synth.make_pose(2, 8, device=dev), torch.full((3,), 0.5, device=dev), scenes.headline_upstream_grad(H).to(dev)
        runs = []
        for _ in range(2):
            im, mk, uvr = ras.rasterize(gr, T, camr, 0.3, 500.0, 100, 3.0, True, bg)
            uvr.retain_grad()
            im.backward(G)
            grads = {k: getattr(g, k).grad.clone() for k in names}
            for k in names:
                getattr(g, k).grad = None
            runs.append((im.detach(), mk, uvr.detach(), grads, uvr.grad.clone()))
        (im_a, mask, uv, gr_a, guv_a), (im_b, _, _, gr_b, guv_b) = runs
        p = f"h{H}_"
        d[p + "culling_mask_sha"], d[p + "uv_sha"] = np.array(scenes.bits_digest(mask)), np.array(scenes.bits_digest(uv))
        body = (H // 16) * 16
        d[p + "image_body_sha"] = np.array(scenes.bits_digest(im_a[:body]))
        if body < H:  # ragged bottom tile row: only the pixels where the reference reproduces itself
            stable = (im_a[body:] == im_b[body:]).all(dim=2)
            d[p + "bottom_stable"] = n(stable)
            d[p + "bottom_stable_sha"] = np.array(scenes.bits_digest(im_a[body:][stable]))
        visible = np.flatnonzero(~n(mask))
        rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))  # noqa: E731
        for k in names:
            d[p + "noise_g_" + k] = np.float64(rel(gr_b[k], gr_a[k]))
            scenes.keep_rows(d, p + "g_" + k, n(gr_a[k]), visible, seed=H)
        d[p + "noise_g_uv"] = np.float64(rel(guv_b, guv_a))
        scenes.keep_rows(d, p + "g_uv", n(guv_a), np.arange(guv_a.shape[0]), seed=H)
        meta[f"headline_{H}"] = {k: float(v) for k, v in d.items() if k.startswith(p + "noise")}
        del g, gr, runs, im_a, im_b, gr_a, gr_b
        torch.cuda.empty_cache()
    np.savez_compressed(out / "ref_headline_3M.npz", **d)


def densify(out, dev, meta):
    """The reference trainer's adaptive_density_control (trainer.py + optimizer_manager.py on torch.optim.Adam with
    populated state) on tests/test_densify_plan.make_case(100_000, seed=21), two passes; per pass the value digests
    of every parameter and both Adam moments."""
    from tests.test_densify_plan import make_case

    ref_loader.load_reference_trainer()
    RT, RC = sys.modules["splat_py_trainer_ref.trainer"], sys.modules["splat_py_trainer_ref.config"]
    RO, RS = sys.modules["splat_py_trainer_ref.optimizer_manager"], sys.modules["splat_py_trainer_ref.structs"]
    n_g = 100_000
    P, M, V, uv_acc, xyz_acc, cnt = make_case(n_g, seed=21, device=dev, n_rest=15)
    config = RC.SplatConfig()
    gr = RS.Gaussians(*(torch.nn.Parameter(P[k].clone()) for k in ("xyz", "rgb", "opacity", "scale", "quaternion")),
                      sh=torch.nn.Parameter(P["sh"].clone()))
    trainer = object.__new__(RT.SplatTrainer)
    trainer.gaussians, trainer.config = gr, config
    trainer.optimizer_manager = RO.OptimizerManager(gr, config)
    order = ("xyz", "quaternion", "scale", "opacity", "rgb", "sh")  # optimizer_manager.py:13-44 group order
    for k, group in zip(order, trainer.optimizer_manager.optimizer.param_groups):
        trainer.optimizer_manager.optimizer.state[group["params"][0]] = dict(step=torch.tensor(7.0), exp_avg=M[k].clone(),
                                                                             exp_avg_sq=V[k].clone())
    trainer.uv_grad_accum, trainer.xyz_grad_accum, trainer.grad_accum_count = uv_acc, xyz_acc, cnt
    d = {}
    for it in (800, 900):
        torch.manual_seed(100 + it)
        trainer.adaptive_density_control(it)
        state = trainer.optimizer_manager.optimizer.state
        for k, group in zip(order, trainer.optimizer_manager.optimizer.param_groups):
            p = group["params"][0]
            d[f"it{it}_{k}"] = np.array(scenes.value_digest(getattr(gr, k)))
            d[f"it{it}_{k}_exp_avg"] = np.array(scenes.value_digest(state[p]["exp_avg"]))
            d[f"it{it}_{k}_exp_avg_sq"] = np.array(scenes.value_digest(state[p]["exp_avg_sq"]))
        d[f"it{it}_n"] = np.int64(gr.xyz.shape[0])
        d[f"it{it}_count_rows"] = np.int64(trainer.grad_accum_count.shape[0])
        n_now = gr.xyz.shape[0]
        gen = torch.Generator(device=dev).manual_seed(it)
        uv2 = torch.rand(n_now, 2, device=dev, generator=gen) * 1e-3
        xyz2 = torch.rand(n_now, 3, device=dev, generator=gen) * 1e-3
        cnt2 = torch.randint(0, 4, (n_now,), device=dev, generator=gen, dtype=torch.int32)
        uv2[cnt2 == 0] = 0.0
        trainer.uv_grad_accum, trainer.xyz_grad_accum, trainer.grad_accum_count = uv2, xyz2, cnt2
    meta["densify"] = {k: int(v) for k, v in d.items() if k.endswith("_n")}
    np.savez_compressed(out / "ref_densify_trainer.npz", **d)


def colmap(out, meta):
    """tools/e2e/make_colmap_scene.py writes a scene; the reference's read_colmap.py reads it back.  Kept: the
    files' bytes, the byte offsets of their float64 fields and what the reader returned."""
    import importlib.util
    import tempfile

    def load(path, name):
        spec = importlib.util.spec_from_file_location(name, str(path))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    rd = load(ref_loader.REF_DIR / "splat_py" / "read_colmap.py", "ref_read_colmap")
    mk = load(ROOT / "tools" / "e2e" / "make_colmap_scene.py", "make_colmap_scene")
    poses, names, xyz, rgb = scenes.colmap_scene(mk)
    d = {}
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        mk.write_cameras(tmp / "cameras.bin", 640, 416, 560.0, 561.0, 320.0, 208.0)
        mk.write_images(tmp / "images.bin", poses, names)
        mk.write_points(tmp / "points3D.bin", xyz, rgb)
        for f in ("cameras", "images", "points3D"):
            d[f + "_bytes"] = np.frombuffer((tmp / f"{f}.bin").read_bytes(), np.uint8)
        cams = rd.read_cameras_binary(str(tmp / "cameras.bin"))
        imgs = rd.read_images_binary(str(tmp / "images.bin"))
        pts = rd.read_points3D_binary(str(tmp / "points3D.bin"))
    # float64 fields: 8-byte header, then per record (make_colmap_scene.py write_*)
    d["cameras_f64_at"] = np.array([32, 40, 48, 56])
    at, o = [], 8
    for name in names:
        at += [o + 4 + 8 * j for j in range(7)]
        o += 64 + len(name) + 1 + 8
    d["images_f64_at"] = np.array(at)
    d["points3D_f64_at"] = np.array([8 + 51 * i + j for i in range(len(xyz)) for j in (8, 16, 24, 35)])
    d.update(cam_ids=np.array(sorted(cams)), cam_model=np.array([cams[i].model for i in sorted(cams)]),
             cam_size=np.array([[cams[i].width, cams[i].height] for i in sorted(cams)]),
             cam_params=np.array([cams[i].params for i in sorted(cams)]),
             img_ids=np.array(sorted(imgs)), img_names=np.array([imgs[i].name for i in sorted(imgs)]),
             img_camera_ids=np.array([imgs[i].camera_id for i in sorted(imgs)]),
             img_rotmat=np.array([rd.qvec2rotmat(imgs[i].qvec) for i in sorted(imgs)]),
             img_tvec=np.array([imgs[i].tvec for i in sorted(imgs)]),
             pt_ids=np.array(sorted(pts)), pt_xyz=np.array([pts[i].xyz for i in sorted(pts)]),
             pt_rgb=np.array([pts[i].rgb for i in sorted(pts)]))
    np.savez_compressed(out / "ref_colmap_reader.npz", **d)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sets", nargs="+", default=["fixtures", "comparisons", "densify", "colmap"],
                    choices=["fixtures", "comparisons", "densify", "colmap"])
    args = ap.parse_args()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    meta = dict(torch=torch.__version__)
    if "colmap" in args.sets:
        colmap(out, meta)
    if set(args.sets) - {"colmap"}:
        dev = torch.device("cuda")
        ref_ext, _ = ref_loader.load_reference()
        meta["gpu"] = torch.cuda.get_device_name(0)
        if "fixtures" in args.sets:
            fixtures(out, dev, ref_ext, meta)
        if "comparisons" in args.sets:
            comparisons(out, dev, meta)
        if "densify" in args.sets:
            densify(out, dev, meta)

    import json

    (out / "golden_meta.json").write_text(json.dumps(meta, indent=1))
    print(json.dumps(meta, indent=1))


if __name__ == "__main__":
    main()
