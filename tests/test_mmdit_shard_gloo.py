"""Token-sharded FLUX / HunyuanVideo engines (image rows split over the ranks, text rows replicated, image K / V rows all-gathered per
attention, head output gathered) against the single-engine run: world 2 over gloo with the kernels emulated on CPU (tests/emu_ops.py)."""
import copy
import os
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _worker(rank, world, initfile, results, family):
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import emu_ops
    import magcache_b200 as mc
    from magcache_b200 import mmdit
    from magcache_b200 import patch as patch_mod
    dist.init_process_group("gloo", init_method=f"file://{initfile}", rank=rank, world_size=world)
    try:
        mmdit.ops = emu_ops
        patch_mod.ops = emu_ops
        torch.Tensor.is_cuda = property(lambda self: True)
        g = torch.Generator().manual_seed(3)
        outs = {}
        if family == "flux":
            from oracle import flux_ref as fr
            model = fr.FluxTransformer2DModel(in_channels=64, num_layers=2, num_single_layers=2, num_attention_heads=2, joint_attention_dim=96,
                                              pooled_projection_dim=48).init_synthetic(0)
            hs, enc, pooled = torch.randn(1, 48, 64, generator=g).bfloat16(), torch.randn(1, 19, 96, generator=g).bfloat16(), torch.randn(1, 48, generator=g).bfloat16()
            img_ids, txt_ids = fr.make_ids(8, 6, 19)

            def call(m, i):
                return m(hs * (1 - 0.05 * i), enc, pooled, torch.tensor([1.0 - i / 6]), img_ids, txt_ids, torch.tensor([3.5]), return_dict=False)[0]

            def install(m):
                mc.init_magcache_flux(m, 6, thresh=10.0, K=2, retention_ratio=0.34)  # miss miss hit hit miss miss
            eng_attr = "_mc_flux_engine"
        else:
            from oracle import hunyuan_ref as hr
            model = hr.HYVideoDiffusionTransformer(hidden_size=256, heads_num=2, mm_double_blocks_depth=2, mm_single_blocks_depth=2, text_states_dim=96,
                                                   text_states_dim_2=48).init_synthetic(0)
            x = torch.randn(1, 16, 2, 8, 12, generator=g).bfloat16()
            txt, pooled = torch.randn(1, 16, 96, generator=g).bfloat16(), torch.randn(1, 48, generator=g).bfloat16()
            mask = torch.zeros(1, 16, dtype=torch.long)
            mask[0, :11] = 1
            cos, sin = hr.rope_cos_sin((2, 4, 6))

            def call(m, i):
                return m(x * (1 - 0.05 * i), torch.tensor([900.0 - 100 * i]), txt, mask, pooled, cos, sin, torch.tensor([6000.0]), return_dict=False)

            def install(m):
                mc.init_magcache_hunyuan(m, 6, thresh=10.0, K=2, retention_ratio=0.34, mag_ratios=[1.0] * 6)
            eng_attr = "_mc_hunyuan_engine"
        for name in ("single", "sharded"):
            m = copy.deepcopy(model)
            m.__class__ = type("M_" + name, (m.__class__,), {})
            install(m)
            if name == "sharded":
                mc.enable_token_shard(m, rank, world)
            with torch.no_grad():
                outs[name] = ([call(m, i).clone() for i in range(6)], getattr(m, eng_attr))
        eng = outs["sharded"][1]
        errs = [float((a.float() - b.float()).abs().max() / b.float().abs().max()) for a, b in zip(outs["sharded"][0], outs["single"][0])]
        full_res, loc_res = outs["single"][1].res, eng.res
        res_err = float((loc_res.float() - full_res[eng.shard.start:eng.shard.stop].float()).abs().max() / full_res.float().abs().max())
        # calibration twin (magcache_flux.py:21-231 / magcache_sample_video.py:163-290) on the sharded engine: the three statistics are
        # sums over the image tokens, so the ranks' partial sums are added before they are finalised — same lists as one engine
        cal, cal_shard = {}, {}
        for name in ("single", "sharded"):
            m = copy.deepcopy(model)
            m.__class__ = type("C_" + name, (m.__class__,), {})
            (mc.init_magcache_flux_calibration if family == "flux" else mc.init_magcache_hunyuan_calibration)(m, 5)
            type(m).calibration_dir = None
            if name == "sharded":
                mc.enable_token_shard(m, rank, world)
            with torch.no_grad():
                for i in range(4):
                    call(m, i)
            cal[name] = [list(getattr(m, k)) for k in ("norm_ratio", "norm_std", "cos_dis")]
            cal_shard[name] = getattr(m, eng_attr).shard is not None
        results[rank] = (errs, res_err, eng.n_img, eng.n_img_total, eng.S_keys, cal, cal_shard)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("family", ["flux", "hunyuan"])
def test_sharded_mmdit_engine_equals_single_world2(family):
    with tempfile.TemporaryDirectory() as d:
        mgr = mp.get_context("spawn").Manager()
        results = mgr.dict()
        mp.spawn(_worker, args=(2, os.path.join(d, "init"), results, family), nprocs=2, join=True)
        assert set(results.keys()) == {0, 1}
        for r in (0, 1):
            errs, res_err, n_loc, n_tot, s_keys, cal, cal_shard = results[r]
            assert cal_shard == {"single": False, "sharded": True}  # enable_token_shard reaches the calibration engine too
            assert all(len(v) == 3 for v in cal["single"]) and all(len(v) == 3 for v in cal["sharded"]), cal
            for a, b in zip(sum(cal["sharded"], []), sum(cal["single"], [])):
                assert abs(a - b) <= 2e-2 * abs(b) + 2e-3, cal
            assert n_loc * 2 == n_tot == 48 and s_keys == 48 + (19 if family == "flux" else 11)
            assert len(errs) == 6 and max(errs) < 1.2e-2, errs   # bf16 streams: a different GEMM row blocking flips roundings
            assert res_err < 3e-2
