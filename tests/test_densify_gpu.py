"""Clone / split / delete on the flat parameter + Adam buffers (csrc/gsr_densify.cu through the C ABI) — needs a B200.

  1. the native apply pass against a torch-indexing stand-in of the same plan, bit for bit;
  2. AdaptiveDensityControl (plan + native apply on FlatAdam's buffers) against the reference's UNMODIFIED trainer
     code (splat_py/trainer.py `adaptive_density_control` with splat_py/optimizer_manager.py on torch.optim.Adam,
     tests/golden/ref_densify_trainer.npz) on a 100k-gaussian scene: identical surviving / cloned / split rows,
     bit-identical parameters and Adam moments."""
from pathlib import Path

import numpy as np
import pytest
import torch

from gaussian_splatting_b200.densify import (AdaptiveDensityControl, DensificationStats, DensifyConfig, apply_plan,
                                             plan_adaptive_density_control)
from gaussian_splatting_b200.flat_adam import FIELDS, REFERENCE_LR_MULTIPLIERS, FlatAdam
from gaussian_splatting_b200.structs import Gaussians
from tests import scenes
from tests.test_densify_plan import emulate_apply, make_case

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def flat_setup(P, M, V):
    g = Gaussians(P["xyz"].clone(), P["rgb"].clone(), P["opacity"].clone(), P["scale"].clone(), P["quaternion"].clone(),
                  P["sh"].clone())
    for f in FIELDS:
        getattr(g, f).requires_grad_(True)
    opt = FlatAdam.for_gaussians(g)
    start = 0
    for f, end in zip(FIELDS, opt.ends):
        n = P[f].numel()
        opt.m[start:start + n].copy_(M[f].reshape(-1))
        opt.v[start:start + n].copy_(V[f].reshape(-1))
        start = end
    return g, opt


def sections(opt, g, buf):
    out, start = {}, 0
    for f, end in zip(FIELDS, opt.ends):
        t = getattr(g, f)
        out[f] = buf[start:start + t.numel()].view(t.shape)
        start = end
    return out


@pytest.mark.parametrize("n", [100_003, 4096])
def test_native_apply_matches_indexing_bitwise(n):
    cfg = DensifyConfig()
    P, M, V, uv_acc, xyz_acc, cnt = make_case(n, seed=3, device=dev(), n_rest=15)
    g, opt = flat_setup(P, M, V)
    stats = DensificationStats(n, dev())
    stats.uv_grad_accum, stats.xyz_grad_accum, stats.grad_accum_count = uv_acc, xyz_acc, cnt
    torch.manual_seed(9)
    plan = plan_adaptive_density_control(g, stats, cfg, 1500)
    assert plan.info["deleted"] > 0 and plan.info["cloned"] > 0 and plan.info["split"] > 0
    Pe, Me, Ve = emulate_apply(plan, P, M, V)
    apply_plan(plan, g, opt, stats)
    assert g.xyz.shape[0] == plan.n_out == stats.grad_accum_count.shape[0]
    assert float(stats.uv_grad_accum.abs().max()) == 0.0
    m_sec, v_sec = sections(opt, g, opt.m), sections(opt, g, opt.v)
    for f in FIELDS:
        assert torch.equal(getattr(g, f).detach(), Pe[f]), f
        assert torch.equal(m_sec[f], Me[f]) and torch.equal(v_sec[f], Ve[f]), f
        assert getattr(g, f).data_ptr() >= opt.p.data_ptr()  # fields are views of the new flat buffer
    # padding between sections stays zero and the optimizer still steps
    opt.step(torch.zeros_like(opt.p))


def test_adaptive_density_control_matches_the_reference_trainer():
    """Two passes on make_case(100_000, seed=21): after each, every parameter and both Adam moments hold the values
    the reference trainer computed from the same case and seeds (value digests, tools/make_golden.py --sets densify)."""
    gd = np.load(Path(__file__).resolve().parent / "golden" / "ref_densify_trainer.npz")
    n = 100_000
    P, M, V, uv_acc, xyz_acc, cnt = make_case(n, seed=21, device=dev(), n_rest=15)
    g, opt = flat_setup(P, M, V)
    stats = DensificationStats(n, dev())
    stats.uv_grad_accum, stats.xyz_grad_accum, stats.grad_accum_count = uv_acc.clone(), xyz_acc.clone(), cnt.clone()
    adc = AdaptiveDensityControl(g, opt, stats, DensifyConfig())

    for it in (800, 900):  # two consecutive passes: the second one runs on the first one's output
        torch.manual_seed(100 + it)
        info = adc.adaptive_density_control(it)
        assert info["deleted"] > 0 or it != 800
        assert g.xyz.shape[0] == int(gd[f"it{it}_n"]), info
        m_sec, v_sec = sections(opt, g, opt.m), sections(opt, g, opt.v)
        for k in ("xyz", "quaternion", "scale", "opacity", "rgb", "sh"):
            assert scenes.value_digest(getattr(g, k)) == str(gd[f"it{it}_{k}"]), (it, k)
            assert scenes.value_digest(m_sec[k]) == str(gd[f"it{it}_{k}_exp_avg"]), (it, k)
            assert scenes.value_digest(v_sec[k]) == str(gd[f"it{it}_{k}_exp_avg_sq"]), (it, k)
        assert stats.grad_accum_count.shape[0] == int(gd[f"it{it}_count_rows"])
        # new statistics for the next pass (the reference was given the same)
        n_now = g.xyz.shape[0]
        gen = torch.Generator(device=dev()).manual_seed(it)
        uv2 = torch.rand(n_now, 2, device=dev(), generator=gen) * 1e-3
        xyz2 = torch.rand(n_now, 3, device=dev(), generator=gen) * 1e-3
        cnt2 = torch.randint(0, 4, (n_now,), device=dev(), generator=gen, dtype=torch.int32)
        uv2[cnt2 == 0] = 0.0
        stats.uv_grad_accum, stats.xyz_grad_accum, stats.grad_accum_count = uv2.clone(), xyz2.clone(), cnt2.clone()


def test_reset_opacity_and_add_sh_band():
    P, M, V, uv_acc, xyz_acc, cnt = make_case(1001, seed=4, device=dev(), n_rest=3)
    g, opt = flat_setup(P, M, V)
    stats = DensificationStats(1001, dev())
    adc = AdaptiveDensityControl(g, opt, stats, DensifyConfig())
    before = {f: getattr(g, f).detach().clone() for f in FIELDS}
    m_before = sections(opt, g, opt.m)
    m_before = {k: v.clone() for k, v in m_before.items()}
    adc.reset_opacity()
    assert torch.all(g.opacity == torch.tensor(-1.3862943611198906, device=dev()).float())
    m_sec = sections(opt, g, opt.m)
    assert float(m_sec["opacity"].abs().max()) == 0.0 and torch.equal(m_sec["xyz"], m_before["xyz"])
    assert adc.add_sh_band() and g.sh.shape == (1001, 3, 8)
    assert torch.equal(g.sh[:, :, :3].detach(), before["sh"]) and float(g.sh[:, :, 3:].abs().max()) == 0.0
    m_sec = sections(opt, g, opt.m)
    assert float(m_sec["sh"].abs().max()) == 0.0 and torch.equal(m_sec["quaternion"], m_before["quaternion"])
    for f in ("xyz", "quaternion", "scale", "rgb"):
        assert torch.equal(getattr(g, f).detach(), before[f])
    assert adc.add_sh_band() and g.sh.shape == (1001, 3, 15) and not adc.add_sh_band()
    opt.step(torch.zeros_like(opt.p))
