"""The caller contract end to end on CPU (SURVEY §8a row 10, eval/magcache/experiments/Wan2.1_EVAL/wan_magcache.py:289-310): per step the
patched forward for the conditional branch, then for the unconditional one, CFG combine, scheduler step — the product side with the
kernels emulated (tests/emu_ops.py: engine, fused `cfg_step` sampler), the reference side with the oracle forward and the oracle sampler.
Checks: identical hit / miss sequence over the whole video, latents that stay together to bf16-pipeline noise, and the TeaCache
comparator driven through the same loop."""
import copy

import pytest
import torch

import magcache_b200 as mc
from magcache_b200 import patch as patch_mod
from magcache_b200 import sampler as sampler_mod
from magcache_b200 import wan as wan_mod
from oracle import sampler_ref, wan_ref

import emu_ops


@pytest.fixture()
def emulated(monkeypatch):
    for mod in (wan_mod, patch_mod, sampler_mod):
        monkeypatch.setattr(mod, "ops", emu_ops)
    monkeypatch.setattr(torch.Tensor, "is_cuda", property(lambda self: True))


def _models(install_ref, install_ours):
    model = wan_ref.WanModel(dim=256, ffn_dim=512, num_heads=2, num_layers=2, text_dim=128, text_len=32).init_synthetic(4)
    ref = copy.deepcopy(model)
    ref.__class__ = type("Ref", (ref.__class__,), {})
    install_ref(type(ref))
    ours = copy.deepcopy(model)
    ours.__class__ = type("Ours", (ours.__class__,), {})
    install_ours(ours)
    object.__setattr__(ours, "_mc_engine", mc.WanEngine(mc.WanWeights.from_module(ours, torch.device("cpu"))))
    return ref, ours


@pytest.mark.parametrize("solver", ["euler", "unipc"])
def test_magcache_generation_loop(emulated, solver):
    steps, guide = 10, 5.0
    table = mc.tables()["wan2.1_t2v_1.3b"]
    ref, ours = _models(lambda c: wan_ref.install_magcache(c, table, steps, thresh=0.12, K=2, retention_ratio=0.2),
                        lambda m: mc.init_magcache(m, steps, thresh=0.12, K=2, retention_ratio=0.2, mag_ratios=table))
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(16, 2, 8, 8, generator=g)
    ctx, ctx_null = torch.randn(9, 128, generator=g), torch.randn(7, 128, generator=g)
    sig = mc.sampling_sigmas(steps, 5.0)
    sig[0] = 0.9999
    sig_t = torch.tensor(sig, dtype=torch.float64)
    smp = (mc.FlowEulerSampler if solver == "euler" else mc.FlowUniPCSampler)(sig)
    smp_ref = (sampler_ref.EulerRef if solver == "euler" else sampler_ref.UniPCRef)(sig_t)
    x, xr = lat.clone(), lat.clone()
    kinds = []
    with torch.no_grad():
        for i in range(steps):
            t = torch.tensor([smp.timestep], dtype=torch.float32)
            cond = ours([x], t=t, context=[ctx], seq_len=32)[0]
            uncond = ours([x], t=t, context=[ctx_null], seq_len=32)[0]
            x = smp.step(cond, uncond, guide, x)
            c_r = ref([xr], t=t, context=[ctx], seq_len=32)[0]
            kinds.append(int(ref.last_skip))
            u_r = ref([xr], t=t, context=[ctx_null], seq_len=32)[0]
            kinds.append(int(ref.last_skip))
            xr = smp_ref.step(sampler_ref.cfg(c_r, u_r, guide), xr).float()
            assert ours.cnt == ref.cnt and ours.accumulated_err == ref.accumulated_err
            rel = float((x.double() - xr.double()).norm() / xr.double().norm())
            assert rel < 3e-2, (solver, i, rel)
    want = mc.MagCacheConfig("wan2.1", 0.12, 2, 0.2, steps, table="wan2.1_t2v_1.3b").schedule().tolist()
    assert kinds == want and 0 < sum(want) < 2 * steps
    assert bool(torch.isfinite(x).all())


def test_fused_step_equals_two_calls_plus_cfg_step(emulated):
    """`FlowEulerSampler.denoise` (SURVEY §8f-1 as written: CFG combine + scheduler update in the epilogue of the unconditional
    call's head, `mc_head_unpatchify_step`) walks the same hit / miss sequence and produces the same latents, bit for bit, as the
    two patched-forward calls followed by `cfg_step` — over a whole schedule with hits and misses, latent updated in place."""
    steps, guide = 10, 5.0
    table = mc.tables()["wan2.1_t2v_1.3b"]
    inst = lambda m: mc.init_magcache(m, steps, thresh=0.12, K=2, retention_ratio=0.2, mag_ratios=table)  # noqa: E731
    a_model, b_model = _models(lambda c: None, inst)[1], _models(lambda c: None, inst)[1]
    g = torch.Generator().manual_seed(2)
    lat = torch.randn(16, 2, 8, 8, generator=g)
    ctx, ctx_null = torch.randn(9, 128, generator=g), torch.randn(7, 128, generator=g)
    sig = mc.sampling_sigmas(steps, 5.0)
    sa, sb = mc.FlowEulerSampler(sig), mc.FlowEulerSampler(sig)
    xa, xb = lat.clone(), lat.clone()
    with torch.no_grad():
        for i in range(steps):
            t = torch.tensor([sa.timestep], dtype=torch.float32)
            cond = a_model([xa], t=t, context=[ctx], seq_len=32)[0]
            uncond = a_model([xa], t=t, context=[ctx_null], seq_len=32)[0]
            xa = sa.step(cond, uncond, guide, xa)
            out = sb.denoise(b_model, xb, t, ctx, ctx_null, 32, guide)
            assert out.data_ptr() == xb.data_ptr()  # in place
            assert torch.equal(xa, xb), i
            assert a_model.cnt == b_model.cnt and a_model.accumulated_err == b_model.accumulated_err
    assert b_model._mc_engine._step is None


def test_fused_step_under_calibration(emulated):
    """A calibration-installed model (`init_magcache_calibration`, magcache_generate.py:921-928) driven by `FlowEulerSampler.denoise`:
    the armed step is applied once, by the unconditional call's head, and never survives into the next step's conditional call —
    latents bit-equal to the two calls followed by `sampler.step`, same statistics."""
    steps, guide = 4, 5.0
    a_model, b_model = (_models(lambda c: None, lambda m: mc.init_magcache_calibration(m, steps))[1] for _ in range(2))
    for m in (a_model, b_model):
        type(m).calibration_dir = None
    g = torch.Generator().manual_seed(2)
    lat = torch.randn(16, 2, 8, 8, generator=g)
    ctx, ctx_null = torch.randn(9, 128, generator=g), torch.randn(7, 128, generator=g)
    sig = mc.sampling_sigmas(steps, 5.0)
    sa, sb = mc.FlowEulerSampler(sig), mc.FlowEulerSampler(sig)
    xa, xb = lat.clone(), lat.clone()
    with torch.no_grad():
        for i in range(steps):
            t = torch.tensor([sa.timestep], dtype=torch.float32)
            cond = a_model([xa], t=t, context=[ctx], seq_len=32)[0]
            uncond = a_model([xa], t=t, context=[ctx_null], seq_len=32)[0]
            xa = sa.step(cond, uncond, guide, xa)
            sb.denoise(b_model, xb, t, ctx, ctx_null, 32, guide)
            assert b_model._mc_engine._step is None, i
            assert torch.equal(xa, xb), i
    assert len(b_model.norm_ratio) == 2 * steps - 2 and b_model.norm_ratio == a_model.norm_ratio


def test_teacache_generation_loop(emulated):
    steps, coef = 8, [0.02, 0.04, 0.0]
    ref, ours = _models(lambda c: wan_ref.install_teacache(c, steps, 0.08, coef), lambda m: mc.init_teacache(m, steps, teacache_thresh=0.08, coefficients=coef))
    g = torch.Generator().manual_seed(1)
    lat = torch.randn(16, 2, 8, 8, generator=g)
    ctx, ctx_null = torch.randn(9, 128, generator=g), torch.randn(7, 128, generator=g)
    sig = wan_ref.flow_sigmas(steps)
    skips = []
    with torch.no_grad():
        for i in range(steps):
            t = torch.tensor([float(sig[i] * 1000)])
            for c in (ctx, ctx_null):
                a = ref([lat], t=t, context=[c], seq_len=32)[0]
                b = ours([lat], t=t, context=[c], seq_len=32)[0]
                skips.append(int(ref.last_skip))
                assert float((a - b).norm() / a.norm()) < 2e-2
                assert ours.cnt == ref.cnt
                assert abs(ours.accumulated_rel_l1_distance_even - ref.accumulated_rel_l1_distance_even) < 1e-5
    assert 0 < sum(skips) < len(skips) - 4
