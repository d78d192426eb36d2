#!/usr/bin/env python
"""bench.py — fwd+bwd views/s of the rasterizer hot path on synthetic 1080p / 3M-Gaussian / SH-3 scenes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference-cpu] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one view: rasterize() forward + backward of the image
against a fixed upstream gradient.  Views shard across ranks (at step i rank r renders view (i + r) mod 8 of a
ring of 8 poses; Gaussians are replicated; no collective on the raster path) -> weak scaling.  Rank 0 prints
ONE JSON line (contract: see the round prompt / DESIGN.md "Measurement").

  value     views/s, all inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       views/s through the public API with HOST buffers: per step the pose, intrinsics and the
            upstream image gradient are copied from pinned host memory and the rendered image is read
            back to pinned host memory inside the timed region
  roofline  render-backward kernel: algorithmic bytes (76 B per consumed pair + 20 B per pixel,
            SURVEY.md §8(d)) / CUDA-event duration, against the measured HBM peak
  cpu_baseline  the CPU oracle (port of the reference's algorithm) on a bounded sample, rank 0, N=1

--impl reference      the UNMODIFIED reference (its CUDA extension compiled into oracle/_ref, its own
                      splat_py.rasterize) on the same scene/poses on this GPU — the number the ">= 2x the
                      reference's own CUDA rasterizer" target is defined against.  The reference has no CPU
                      implementation of this path; when oracle/_ref is absent this falls back to
--impl reference-cpu  the CPU oracle port on the host cores (bounded sample).

--dump-outputs DIR    (b200) after the timed resident steps, write what the last of them computed to DIR/<name>.npy
                      (see dump_outputs); the inputs depend only on the arguments, so two builds run with the same
                      arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "fwd+bwd views/sec @1080p, 3M Gaussians, SH deg 3"
# the workload both arms run (config.workload of every line)
WORKLOAD = ("synthetic 3M Gaussians, 1080p, SH deg 3 (BASELINE.json configs[2]/[3]); one view per GPU per step, ring "
            "of 8 poses (3 deg yaw steps), fwd + bwd of image against a fixed upstream gradient")
N_GAUSS = 3_000_000
RES = "1080p"
SH_DEGREE = 3
N_POSES = 8
DUMP_ROWS = 65_536  # gaussians whose per-gaussian outputs --dump-outputs writes (fixed seeded sample of N_GAUSS)
MY_KERNELS = ["k_camera_centre", "k_preprocess_fwd", "k_emit_pairs_fused", "k_tile_ranges", "k_render_fwd",
              "k_render_bwd", "k_preprocess_bwd"]  # + k_gather_records_keys with GSR_RECORD_STREAM=1


def log(msg):
    """Stage progress on stderr (a lost box then shows where the arm was)."""
    sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
    sys.stderr.flush()


CPU_LEG_TIMEOUT_S = 90      # hard wall-clock bound of the CPU-baseline child process
CPU_LEG_MAX_THREADS = 32    # host threads the CPU legs may use (stated in cpu_baseline.cores)
TORCH_CPU_SAMPLE = 300_000  # gaussians of the torch-CPU projection/SH leg (1/10 of the workload, scaled x10)


def cpu_threads():
    return max(1, min(CPU_LEG_MAX_THREADS, os.cpu_count() or 1))


def cpu_baseline_sandboxed(args):
    """Run the CPU-baseline leg in a CHILD process: bounded threads, hard timeout, never fatal.  The child
    prints one JSON object; any failure becomes {"error": ...} in the bench line instead of a dead arm."""
    nthreads = cpu_threads()
    env = dict(os.environ, OMP_NUM_THREADS=str(nthreads), MKL_NUM_THREADS=str(nthreads),
               OPENBLAS_NUM_THREADS=str(nthreads), CUDA_VISIBLE_DEVICES="", OMP_WAIT_POLICY="PASSIVE")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    cmd = [sys.executable, str(Path(__file__).resolve()), "--impl", "cpu-baseline-child"]
    t0 = time.time()
    try:
        proc = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=CPU_LEG_TIMEOUT_S)
    except subprocess.TimeoutExpired:
        return {"error": f"cpu-baseline child exceeded {CPU_LEG_TIMEOUT_S}s", "cores": nthreads, "kind": "port"}
    except Exception as e:
        return {"error": repr(e), "cores": nthreads, "kind": "port"}
    if proc.returncode != 0:
        return {"error": f"cpu-baseline child rc={proc.returncode}: {proc.stderr[-300:]}", "cores": nthreads,
                "kind": "port"}
    try:
        out = json.loads(proc.stdout.strip().splitlines()[-1])
    except Exception as e:
        return {"error": f"unparsable child output: {e!r}", "cores": nthreads, "kind": "port"}
    out["child_wall_s"] = time.time() - t0
    return out


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = Path(f"/tmp/gsr_clocks_{os.getpid()}.csv")

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        for line in self.path.read_text().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            busy = [s for s in sm if s > 0.5 * max(sm)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def build_scene(dev):
    import torch

    from gaussian_splatting_b200 import synth

    g = synth.make_gaussians(N_GAUSS, RES, sh_degree=SH_DEGREE, seed=0, device=dev, requires_grad=True)
    cam = synth.make_camera(RES, device=dev)
    poses_host = [synth.make_pose(v, N_POSES).pin_memory() for v in range(N_POSES)]
    poses = [p.to(dev) for p in poses_host]
    G_host = synth.make_upstream_grad(RES).pin_memory()
    G = G_host.to(dev)
    bg = torch.full((3,), 0.5, device=dev)
    return g, cam, poses, poses_host, G, G_host, bg


def zero_grads(g):
    for p in (g.xyz, g.rgb, g.opacity, g.scale, g.quaternion, g.sh):
        if p is not None:
            p.grad = None


def timed_steps(step_fn, steps, warmup, world, dev):
    """W warm-up steps, then K steps bracketed by barrier + synchronize; returns max-over-ranks ms."""
    import torch
    import torch.distributed as dist

    for i in range(warmup):
        step_fn(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step_fn(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    per_rank = [float(ms.item())]
    if world > 1:
        dist.barrier()
        every = [torch.zeros_like(ms) for _ in range(world)]
        dist.all_gather(every, ms)
        per_rank = [float(t.item()) for t in every]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    _LAST_PER_RANK_MS[:] = per_rank
    return float(ms.item())


_LAST_PER_RANK_MS = []  # ms of the last timed_steps() call on every rank (explains max-over-ranks at N > 1)


def dump_outputs(out_dir, image, mask, uv, g):
    """What one step returned to its caller, as float32 / float64 .npy files (about 41 MB): the image in full and, for
    a fixed seeded sample of DUMP_ROWS gaussians (gaussian_rows), the culling mask (1 = culled), uv (0 where
    culled: a culled gaussian has no projection) and the gradient of every parameter.  Every value is finite."""
    import numpy as np
    import torch

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    n = g.xyz.shape[0]
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    at = rows.to(mask.device)
    uv_all = torch.zeros((n, 2), device=uv.device)
    uv_all[~mask] = uv.detach()
    arrays = {"image": image.detach(), "gaussian_rows": rows.double(), "culling_mask": mask[at].float(),
              "uv": uv_all[at]}
    for name in ("xyz", "rgb", "opacity", "scale", "quaternion", "sh"):
        arrays["grad_" + name] = getattr(g, name).grad[at]
    for name, t in arrays.items():
        np.save(out / f"{name}.npy", t.cpu().numpy())
    return sorted(arrays)


def run_b200(args, rank, world, local):
    import torch

    from gaussian_splatting_b200 import synth
    from gaussian_splatting_b200.rasterize import rasterize

    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    log("building the synthetic scene")
    g, cam, poses, poses_host, G, G_host, bg = build_scene(dev)
    cfg = synth.DEFAULTS
    K_host = cam.K.cpu().pin_memory()
    image_host = torch.empty(cam.height, cam.width, 3).pin_memory()

    def view_of(i):
        # step i renders the `world` consecutive views i .. i+world-1 of the pose ring, rank r the r-th of them:
        # every step covers `world` distinct views and every GPU cycles through all 8 poses, so no rank is
        # pinned to the heaviest view (P differs by ~1.5% between poses) when the max over ranks is taken
        return (i + rank) % N_POSES

    last = {}  # the outputs of the latest resident step, kept only for --dump-outputs

    def step_resident(i):
        zero_grads(g)
        image, mask, uv = rasterize(g, poses[view_of(i)], cam, cfg["near_thresh"], cfg["far_thresh"],
                                    cfg["cull_mask_padding"], cfg["mh_dist"], True, bg)
        image.backward(G)
        if args.dump_outputs:
            last.update(image=image, mask=mask, uv=uv)

    h2d_bytes = poses_host[0].numel() * 4 + K_host.numel() * 4 + G_host.numel() * 4
    d2h_bytes = image_host.numel() * 4

    # e2e: host buffers in, host buffer out, every step.  Copies run on a side stream so that the 25 MB
    # upstream-gradient upload overlaps the forward pass and the 25 MB image download overlaps the backward
    # pass; the step ends with a full synchronize (its result is on the host before the next step starts).
    from gaussian_splatting_b200.structs import Camera

    copy_stream = torch.cuda.Stream(device=dev)
    T_buf, K_buf = torch.empty(4, 4, device=dev), torch.empty(3, 3, device=dev)
    G_buf = torch.empty_like(G)
    cam_e2e = Camera(cam.width, cam.height, K_buf)

    def step_e2e(i):
        main = torch.cuda.current_stream()
        zero_grads(g)
        with torch.cuda.stream(copy_stream):  # the forward's inputs first: nothing else delays its first kernel
            T_buf.copy_(poses_host[view_of(i)], non_blocking=True)
            K_buf.copy_(K_host, non_blocking=True)
            ev_small = copy_stream.record_event()
        main.wait_event(ev_small)
        image, _, _ = rasterize(g, T_buf, cam_e2e, cfg["near_thresh"], cfg["far_thresh"],
                                cfg["cull_mask_padding"], cfg["mh_dist"], True, bg)
        ev_img = main.record_event()
        with torch.cuda.stream(copy_stream):
            G_buf.copy_(G_host, non_blocking=True)  # the backward's input: uploaded while the forward runs
            ev_grad = copy_stream.record_event()
            copy_stream.wait_event(ev_img)
            image_host.copy_(image.detach(), non_blocking=True)
        main.wait_event(ev_grad)
        image.backward(G_buf)
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()  # every rank samples its own GPU: the slowest GPU sets the max-over-ranks time
    log("timing: resident")
    ms_res = timed_steps(step_resident, args.steps, args.warmup, world, dev)
    per_rank_res = [m / args.steps for m in _LAST_PER_RANK_MS]
    if args.dump_outputs and rank == 0:  # the gradients of the last resident step are still on the parameters
        names = dump_outputs(args.dump_outputs, last["image"], last["mask"], last["uv"], g)
        log(f"outputs of step {args.warmup + args.steps - 1} (view {view_of(args.warmup + args.steps - 1)}) written "
            f"to {args.dump_outputs}: {', '.join(names)}")
    last.clear()
    log(f"resident {ms_res / args.steps:.3f} ms/step; timing: e2e")
    ms_e2e = timed_steps(step_e2e, args.steps, args.warmup, world, dev)
    per_rank_e2e = [m / args.steps for m in _LAST_PER_RANK_MS]
    log(f"e2e {ms_e2e / args.steps:.3f} ms/step; per-stage profile")
    clocks = sampler.stop()
    per_rank_clocks = None
    if world > 1:
        import torch.distributed as dist

        mine = torch.tensor([clocks.get("sm_mhz") or 0.0], device=dev, dtype=torch.float64)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        per_rank_clocks = [float(t.item()) for t in every]

    # ---- per-stage profile + scene statistics (rank 0; separate from the timed regions) ----
    roofline, stages, stats = None, {}, {}
    if rank == 0:
        prof = []
        n_prof = max(5, min(args.steps, 11))
        last_state = None
        for i in range(n_prof):
            zero_grads(g)
            image, _, _, st = rasterize(g, poses[view_of(i)], cam, cfg["near_thresh"], cfg["far_thresh"],
                                        cfg["cull_mask_padding"], cfg["mh_dist"], True, bg, return_state=True,
                                        profile=prof)
            image.backward(G)
            last_state = st
        torch.cuda.synchronize()
        acc = {}
        for name, e0, e1 in prof:
            acc.setdefault(name, []).append(e0.elapsed_time(e1))
        stages = {k: statistics.median(v) for k, v in acc.items()}  # median: robust to allocator hiccups
        H, W = cam.height, cam.width
        st = last_state
        npp = st.n_per_pixel
        Hp, Wp = (H + 15) // 16 * 16, (W + 15) // 16 * 16
        pad = torch.zeros(Hp, Wp, dtype=npp.dtype, device=dev)
        pad[:H, :W] = npp
        tile_max = pad.view(Hp // 16, 16, Wp // 16, 16).amax(dim=(1, 3))
        P_used = int(tile_max.sum().item())
        stats = dict(N=st.N, M=st.M, P=st.P, P_consumed_by_render_bwd=P_used,
                     splats_per_tile_mean=st.P / ((Hp // 16) * (Wp // 16)),
                     mean_splats_walked_per_pixel=float(npp.float().mean().item()))
        peaks = {}
        pf = ROOT / "MEASURED_PEAKS.json"
        if pf.exists():
            peaks = json.loads(pf.read_text())
        peak = float(peaks.get("hbm_gbs", 6650.0))
        alg_bytes = 76.0 * P_used + 20.0 * H * W
        dur_ms = stages.get("render_bwd", float("nan"))
        achieved = alg_bytes / (dur_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tf = ROOT / "profiles" / "ncu_traffic_latest.json"
        if tf.exists():  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture
            rec = json.loads(tf.read_text()).get("k_render_bwd", {})
            traffic, traffic_src = rec.get("dram_bytes_per_launch"), rec.get("source")
        # the per-gaussian kernels ARE HBM-bound; report them next to the (issue-bound) dominant kernel
        N_, M_ = st.N, st.M
        other = []
        # bytes the kernels actually have to move (their own byte model, larger than SURVEY.md 8(d)'s 236 N + 44 M,
        # which counts neither the 48-byte record + key + flag + scan a kernel writes per gaussian nor the
        # backward's re-read of the geometry parameters): fwd 236 N read + 61 M + 13 N written; bwd 57 N + 36 M read +
        # 236 N written
        for kname, stage, nbytes in (("k_preprocess_fwd", "preprocess_fwd", 236.0 * N_ + 61.0 * M_ + 13.0 * N_),
                                     ("k_preprocess_bwd", "preprocess_bwd", (56.0 + 1.0) * N_ + 36.0 * M_ + 236.0 * N_)):
            if stage in stages:
                ach = nbytes / (stages[stage] * 1e-3) / 1e9
                other.append(dict(kernel=kname, bound="hbm", achieved=ach, peak=peak, unit="GB/s", frac=ach / peak,
                                  algorithmic_bytes=nbytes, duration_ms=stages[stage],
                                  byte_model="kernel's own (see bench.py); SURVEY.md 8(d) counts 236 N + 44 M (fwd), "
                                             "36 M + 472 N (bwd)",
                                  note="stage time includes the kernel's cub scan / output allocation"))
        # instruction-issue roofline of the same kernel: warp instructions per launch from the committed ncu
        # capture / live duration, against 148 SMs x 4 schedulers x max SM clock
        issue = None
        if tf.exists():
            ninst = json.loads(tf.read_text()).get("k_render_bwd", {}).get("warp_instructions_per_launch")
            if ninst:
                peak_issue = 148 * 4 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6
                issue = dict(achieved=ninst / (dur_ms * 1e-3) / 1e9, peak=peak_issue / 1e9, unit="G warp-inst/s",
                             frac=ninst / (dur_ms * 1e-3) / peak_issue,
                             source="smsp__inst_executed.sum of the committed ncu capture / live CUDA-event duration")
        roofline = dict(kernel="k_render_bwd", bound="hbm", achieved=achieved, peak=peak, unit="GB/s",
                        frac=achieved / peak, traffic=traffic,
                        peak_source="MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s",
                        algorithmic_bytes=alg_bytes, duration_ms=dur_ms,
                        note="76 B per (gaussian,tile) pair the kernel has to visit + 20 B per pixel (SURVEY.md 8(d)); "
                             "the kernel is instruction-issue bound, not HBM bound (see issue_roofline and the ncu "
                             "capture named in traffic_source), so frac is small by construction",
                        traffic_source=traffic_src,
                        issue_roofline=issue, other_kernels=other)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log("cpu baseline (child process, bounded)")
        cpu = cpu_baseline_sandboxed(args)
        log("cpu baseline done")

    if rank != 0:
        return
    views = args.steps * world
    value = views / (ms_res * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "views/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "gaussians": N_GAUSS, "image": "1920x1080", "sh_degree": SH_DEGREE, "views_per_step": world,
                   "parallelism": f"views sharded 1 per GPU x{world}, gaussians replicated, no collective",
                   "view_schedule": "step i, rank r -> pose (i + r) mod 8",
                   "l2": "per-step inputs (708 MB of parameters) exceed the 126 MB L2; no flush needed",
                   "scene": stats, "stage_ms": stages},
        "clocks": clocks,
        "e2e": {"value": views / (ms_e2e * 1e-3), "unit": "views/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": ms_e2e / args.steps},
        "per_rank": {"ms_per_step": per_rank_res, "e2e_ms_per_step": per_rank_e2e, "sm_mhz": per_rank_clocks,
                     "note": "value / e2e use the MAX over ranks; ranks differ by their GPU's clocks under load"},
        "gpu_launches": (len(MY_KERNELS) + (1 if os.environ.get("GSR_RECORD_STREAM", "0") == "1" else 0)) * args.steps,
        "kernels": MY_KERNELS,
        "roofline": roofline, "cpu_baseline": cpu, "impl": "b200",
    }
    emit(line)


def cpu_baseline_leg(args, rows=48):
    """The CPU oracle (port of the reference's algorithm) on a bounded sample of the bench workload:
    the whole per-gaussian stage and tile binning for all 3M gaussians, the tile renderer forward +
    backward on a `rows`-pixel band, scaled to the full image height; per-gaussian backward in full."""
    import numpy as np
    import torch

    from gaussian_splatting_b200 import synth
    from oracle import cpu_oracle as orc

    t_all = time.time()
    nthreads = int(os.environ.get("OMP_NUM_THREADS", cpu_threads()))
    g = synth.make_gaussians(N_GAUSS, RES, sh_degree=SH_DEGREE, seed=0)
    cam = synth.make_camera(RES)
    T = synth.make_pose(0, N_POSES)
    a = lambda t: t.detach().numpy()  # noqa: E731
    H, W = cam.height, cam.width
    orc.lib()
    t0 = time.time()
    pg = orc.project(a(g.xyz), a(g.quaternion), a(g.scale), a(g.opacity), a(g.rgb), a(g.sh), a(T), a(cam.K), H, W,
                     0.3, 500.0, 100.0)
    t_proj = time.time() - t0
    keep = pg.visible.astype(bool)
    uv, conic, xyz_cam, opa, rgb = pg.uv[keep], pg.conic[keep], pg.xyz_cam[keep], pg.opacity[keep], pg.rgb[keep]
    t0 = time.time()
    sorted_idx, ranges = orc.tile_lists(uv, xyz_cam, conic, (W + 15) // 16, (H + 15) // 16, 3.0)
    t_bin = time.time() - t0
    band = (512, 512 + rows)
    bgc = np.full(3, 0.5, np.float32)
    t0 = time.time()
    image, n, w = orc.render_forward(uv, opa, rgb, conic, None, ranges, sorted_idx, bgc, H, W, rows=band)
    t_fwd = time.time() - t0
    G = a(synth.make_upstream_grad(RES))
    t0 = time.time()
    gr = orc.render_backward(uv, opa, rgb, conic, None, ranges, sorted_idx, bgc, n, w, G, rows=band)
    t_bwd = time.time() - t0
    scale = H / rows
    est = t_proj * 2.0 + t_bin + (t_fwd + t_bwd) * scale  # per-gaussian backward ~ per-gaussian forward
    del g, pg
    try:
        torch_cpu = torch_cpu_projection_sh_leg(n=TORCH_CPU_SAMPLE, threads=nthreads)
    except Exception as e:  # never let the auxiliary baseline take the bench down
        torch_cpu = {"error": repr(e)}
    return {"value": 1.0 / est, "torch_cpu_projection_sh": torch_cpu, "unit": "views/s", "cores": nthreads,
            "host_cores": os.cpu_count(), "kind": "port",
            "sample": f"CPU oracle (oracle/gsr_oracle.c, OpenMP x{nthreads} of {os.cpu_count()} host cores): "
                      f"per-gaussian stage + tile binning for all {N_GAUSS} gaussians, tile renderer fwd+bwd on a "
                      f"{rows}-row band scaled x{scale:.1f}; torch-CPU projection/SH leg on {TORCH_CPU_SAMPLE} "
                      f"gaussians (scale x{N_GAUSS // TORCH_CPU_SAMPLE} for the full workload)",
            "seconds": {"project": t_proj, "binning": t_bin, "render_fwd_band": t_fwd, "render_bwd_band": t_bwd,
                        "wall": time.time() - t_all}}


def torch_cpu_projection_sh_leg(n=TORCH_CPU_SAMPLE, reps=3, threads=None):
    """The reference's PyTorch-CPU projection / SH path (north_star): splat_py.utils.transform_points_torch,
    the cull expressions of splat_py/rasterize.py:33-49 and batched PyTorch restatements of the per-gaussian
    operators the reference's analytic_diff.ipynb differentiates (pinhole projection, Sigma_world, Sigma_image,
    SH -> RGB), forward + backward on a bounded sample of `n` of the bench's gaussians, `threads` host threads,
    median of `reps`; `seconds_fwd_bwd_scaled` extrapolates linearly to the full N (the ops are elementwise)."""
    import torch

    from gaussian_splatting_b200 import synth
    from gaussian_splatting_b200.utils import quaternion_to_rotation_torch, transform_points_torch

    torch.set_num_threads(threads or cpu_threads())
    g = synth.make_gaussians(n, RES, sh_degree=SH_DEGREE, seed=0, requires_grad=True)
    cam = synth.make_camera(RES)
    T = synth.make_pose(0, N_POSES)
    fx, fy, cx, cy = cam.K[0, 0], cam.K[1, 1], cam.K[0, 2], cam.K[1, 2]
    times = []
    for _ in range(reps):
        for p in (g.xyz, g.rgb, g.opacity, g.scale, g.quaternion, g.sh):
            p.grad = None
        t0 = time.time()
        p_cam = transform_points_torch(g.xyz, T)
        x, y, z = p_cam.unbind(1)
        uv = torch.stack([fx * x / z + cx, fy * y / z + cy], 1)
        mask = ((z < 0.3) | (z > 500.0) | (uv[:, 0] < -100) | (uv[:, 0] > cam.width + 100) | (uv[:, 1] < -100)
                | (uv[:, 1] > cam.height + 100))
        q = g.quaternion / g.quaternion.norm(dim=1, keepdim=True)
        R = quaternion_to_rotation_torch(q)
        RS = R * torch.exp(g.scale).unsqueeze(1)
        sigma = RS @ RS.transpose(1, 2)
        zero = torch.zeros_like(z)
        J = torch.stack([fx / z, zero, -fx * x / (z * z), zero, fy / z, -fy * y / (z * z)], 1).reshape(-1, 2, 3)
        JW = J @ T[:3, :3]
        s2 = JW @ sigma @ JW.transpose(1, 2)
        d = g.xyz - torch.inverse(T)[:3, 3]
        d = d / d.norm(dim=1, keepdim=True)
        dx, dy, dz = d.unbind(1)
        Y = torch.stack([torch.full_like(dx, 0.2820948), -0.4886025 * dy, 0.4886025 * dz, -0.4886025 * dx,
                         1.0925484 * dx * dy, -1.0925484 * dy * dz, 0.3153916 * (3 * dz * dz - 1),
                         -1.0925484 * dx * dz, 0.5462742 * (dx * dx - dy * dy),
                         -0.5900436 * dy * (3 * dx * dx - dy * dy), 2.8906114 * dx * dy * dz,
                         -0.4570458 * dy * (5 * dz * dz - 1), 0.2638755 * dz * (5 * dz * dz - 3),
                         -0.4570458 * dx * (5 * dz * dz - 1), 1.4453057 * dz * (dx * dx - dy * dy),
                         -0.5900436 * dx * (dx * dx - 3 * dy * dy)], 1)
        rgb = (torch.cat([g.rgb.unsqueeze(2), g.sh], 2) * Y.unsqueeze(1)).sum(2) * 3.5449077
        keep = (~mask).float()
        loss = (uv.sum(1) * keep).sum() + (s2.sum((1, 2)) * keep).sum() + (rgb.sum(1) * keep).sum() \
            + torch.sigmoid(g.opacity).sum()
        loss.backward()
        times.append(time.time() - t0)
    times.sort()
    med = times[len(times) // 2]
    return {"seconds_fwd_bwd": med, "seconds_fwd_bwd_scaled": med * (N_GAUSS / n), "threads": torch.get_num_threads(),
            "cores": os.cpu_count(), "gaussians": n, "scaled_to": N_GAUSS}


def run_reference(args, rank, world, local):
    """The unmodified reference on this GPU (oracle/_ref), rank 0 only."""
    if rank != 0:
        return
    from oracle import ref_loader

    if not ref_loader.reference_available():
        return run_reference_cpu(args, rank)
    import torch

    from gaussian_splatting_b200 import synth

    ref_loader.load_reference()
    ref_ras = sys.modules["splat_py_ref.rasterize"]
    ref_structs = sys.modules["splat_py_ref.structs"]
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    g, cam, poses, poses_host, G, G_host, bg = build_scene(dev)
    gaus = ref_structs.Gaussians(g.xyz, g.rgb, g.opacity, g.scale, g.quaternion, g.sh)
    camr = ref_structs.Camera(cam.width, cam.height, cam.K)
    cfg = synth.DEFAULTS

    def step(i):
        zero_grads(g)
        image, _, _ = ref_ras.rasterize(gaus, poses[i % N_POSES], camr, cfg["near_thresh"], cfg["far_thresh"],
                                        cfg["cull_mask_padding"], cfg["mh_dist"], True, bg)
        image.backward(G)

    sampler = ClockSampler(local)
    sampler.start()
    ms = timed_steps(step, args.steps, args.warmup, 1, dev)
    clocks = sampler.stop()
    value = args.steps / (ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "views/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": WORKLOAD, "gaussians": N_GAUSS, "image": "1920x1080", "sh_degree": SH_DEGREE,
                   "views_per_step": 1,
                   "how": "unmodified joeyan/gaussian_splatting: its CUDA extension compiled for sm_100 "
                          "(oracle/_ref) driven by its own splat_py.rasterize.rasterize + backward, on GPU 0",
                   "launched_world_size": world,
                   "note": "the reference has no multi-GPU path: under torchrun only rank 0 runs, so this is a "
                           "1-GPU number whatever --gpus says (n_gpus is 1 in this line)"},
        "clocks": clocks,
        "cpu_baseline": {"value": value, "unit": "views/s", "cores": 0, "kind": "reference",
                         "sample": "full workload on the GPU: the reference implements this path only in CUDA "
                                   "(no CPU implementation exists); see --impl reference-cpu for the CPU port"},
        "e2e": {"value": value, "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def run_reference_cpu(args, rank):
    if rank != 0:
        return
    cpu = cpu_baseline_sandboxed(args)
    if "value" not in cpu:
        return emit({"impl": "reference", "unavailable": f"cpu port failed: {cpu.get('error')}"})
    line = {
        "metric": METRIC, "value": cpu["value"], "unit": "views/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 / cpu["value"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": {"workload": WORKLOAD + " (bounded sample, see cpu_baseline.sample)"},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_REAL_STDOUT = None


def protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL writes its version line to
    stdout at NCCL_DEBUG >= VERSION, ninja / torch extensions chatter): keep the real stdout aside and point
    file descriptor 1 at stderr for everything else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cpu", "cpu-baseline-child"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed resident step computed to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    rank, world, local = dist_env()
    if args.impl == "cpu-baseline-child":  # internal: the sandboxed CPU leg (see cpu_baseline_sandboxed)
        return emit(cpu_baseline_leg(args))
    if args.impl == "reference-cpu":
        return run_reference_cpu(args, rank)
    log(f"impl={args.impl} rank={rank}/{world} importing torch")
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    if world > 1:
        import torch.distributed as dist

        if args.impl == "reference":
            if rank == 0:
                run_reference(args, rank, world, local)
            return
        torch.cuda.set_device(local)
        # NCCL_DEBUG is left as the launcher set it: file descriptor 1 already points at stderr
        # (protect_stdout), so whatever NCCL prints cannot corrupt the one JSON line
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    try:
        if args.impl == "reference":
            run_reference(args, rank, world, local)
        else:
            run_b200(args, rank, world, local)
    finally:
        if world > 1:
            import torch.distributed as dist

            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
