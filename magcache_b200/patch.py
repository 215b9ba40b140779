"""Drop-in replacements for the reference's monkey-patched transformer forwards.

Usage is the reference's own (MagCache4Wan2.1/magcache_generate.py:896-928): assign the function to the model class and set
the class attributes it reads —

    from magcache_b200 import magcache_forward, init_magcache
    init_magcache(wan_t2v.model, sample_steps=50, thresh=0.12, K=4, retention_ratio=0.2, ckpt_dir=args.ckpt_dir)
    # or, literally as the script does:  wan_t2v.model.__class__.forward = magcache_forward ; ...cnt = 0 ; ...

Signatures, attribute names (`cnt, num_steps, magcache_thresh, K, retention_ratio, accumulated_ratio, accumulated_err,
accumulated_steps, residual_cache, mag_ratios`; calibration: `norm_ratio, norm_std, cos_dis`) and error behaviour follow the
reference. Everything between the Python call and the returned tensors runs on the CUDA kernels of libmagcache_b200.so;
there is no eager/PyTorch fallback — a CPU tensor or a missing library raises.
"""
import os

import numpy as np

import torch

from . import ops
from .config import FAMILIES, interp_cfg, nearest_interp, save_json, table_for_ckpt_dir, table_from_calibration, tables
from .controller import AttrController
from .mmdit import FluxEngine, FluxWeights, HunyuanEngine, HunyuanWeights
from .wan import WanEngine, WanWeights


def _cached_engine(self, attr, engine_cls, make_weights):
    """The engine cached on the model under `attr`, built on first use from `make_weights()` (token-sharded when
    `enable_token_shard` was called)."""
    eng = self.__dict__.get(attr)
    if eng is None:
        eng = engine_cls(make_weights(), **self.__dict__.get("_mc_shard_kw", {}))
        object.__setattr__(self, attr, eng)
    return eng


def _wan_weights(self):
    if not hasattr(self, "patch_embedding"):
        raise TypeError("magcache_b200.magcache_forward expects a Wan2.1 WanModel (or an object carrying `_mc_engine`)")
    dev = self.patch_embedding.weight.device
    if dev.type != "cuda":
        raise RuntimeError("magcache_b200: the model must be on a CUDA device (no CPU path)")
    return WanWeights.from_module(self, dev)


def _engine(self):
    return _cached_engine(self, "_mc_engine", WanEngine, lambda: _wan_weights(self))


def _family_controller(self, family):
    """The skip controller of `family` (a key of `config.FAMILIES`) for this model, created on first use."""
    ctrls = self.__dict__.setdefault("_mc_ctrls", {})
    if family not in ctrls:
        ctrls[family] = AttrController(FAMILIES[family])
    return ctrls[family]


def _adopt_residual(cur, buf, valid):
    """The reference keeps the cached residual in a model attribute (`cur`); the engine keeps it in a fixed buffer `buf` that the
    attribute aliases. If a caller replaced the attribute, copy it in; if they cleared it, the buffer is empty. Returns the buffer's
    new validity (`valid`: its current one)."""
    if cur is None:
        return False
    if torch.is_tensor(cur) and cur.data_ptr() != buf.data_ptr():
        buf.copy_(cur.reshape(buf.shape))
        return True
    return valid


def _record_stats(self, stats):
    """Append the calibration statistics of one call, rounded to 5 places, and print the reference's per-call line
    (MagCache4Wan2.1/magcache_generate.py:170-173 ; magcache_flux.py:202-205 ; magcache_sample_video.py:258-261)."""
    norm_ratio, norm_std, cos_dis = stats
    self.norm_ratio.append(round(norm_ratio, 5))
    self.norm_std.append(round(norm_std, 5))
    self.cos_dis.append(round(cos_dis, 5))
    print(f"time: {self.cnt}, norm_ratio: {norm_ratio}, norm_std: {norm_std}, cos_dis: {cos_dis}")


def _print_stats(self):
    print("norm ratio")
    print(self.norm_ratio)
    print("norm std")
    print(self.norm_std)
    print("cos_dis")
    print(self.cos_dis)


def invalidate_engine(model):
    """Drop the engine cached on `model` (and with it the repacked bf16 copy of the weights, the workspaces and any captured CUDA
    graphs). The engine snapshots the module's parameters at the first forward: call this after anything that changes them — a LoRA
    merge, `load_state_dict`, `.to(...)` — and the next forward repacks. The module's own parameters stay resident next to the
    packed copy (about +2.8 GB for the 1.3B model, +28 GB for 14B); free or offload them yourself if that matters."""
    for name in ("_mc_engine", "_mc_flux_engine", "_mc_hunyuan_engine", "_mc_ctrls"):
        model.__dict__.pop(name, None)
    return model


def enable_token_shard(model, rank, world, group=None):
    """Shard the token axis of `model`'s forwards over `world` ranks of one node (call before the first forward; needs an
    initialised torch.distributed NCCL group). Every rank must then make the same calls with the same inputs; outputs are
    replicated, the residual cache stays sharded. Wan engines shard all tokens; the FLUX / HunyuanVideo engines shard the image tokens and
    replicate the text tokens."""
    if any(k in model.__dict__ for k in ("_mc_engine", "_mc_flux_engine", "_mc_hunyuan_engine")):
        raise RuntimeError("enable_token_shard must be called before the first forward")
    object.__setattr__(model, "_mc_shard_kw", dict(shard_world=world, shard_rank=rank, shard_group=group))
    return model


def _stage(self, x, t, context, seq_len, clip_fea, y, calibration=False, vace_context=None, vace_scale=1.0, require_clip=True):
    if getattr(self, "model_type", "t2v") == "i2v" and require_clip:
        assert clip_fea is not None and y is not None  # magcache_generate.py:226-227
    if len(x) != 1 or len(context) != 1 or (y is not None and len(y) != 1):
        raise NotImplementedError("magcache_b200: one sample per call (the reference's caller passes [latents], wan_magcache.py:296-299)")
    eng = _engine(self)
    lat = x[0]
    if not lat.is_cuda:
        raise RuntimeError("magcache_b200: latents must be CUDA tensors (no CPU path)")
    n_tok = lat.shape[1] * (lat.shape[2] // 2) * (lat.shape[3] // 2)
    assert n_tok <= seq_len  # reference: assert seq_lens.max() <= seq_len (:242)
    # seq_len > n_tok (upstream rounds seq_len up to a multiple of the sequence-parallel size): the reference appends zero rows
    # (:243-246) that never reach a real token — keys are masked by k_lens = seq_lens, every other op is per token, unpatchify
    # reads the first n_tok rows — so the forwards simply do not compute them; the only visible difference: residual_cache[i] has
    # n_tok rows instead of seq_len. The calibration statistics DO average over the padded rows upstream: there ONE representative
    # pad row is computed — the padded rows are all identical — and weighted by their count.
    if vace_context is not None and len(vace_context) != 1:
        raise NotImplementedError("magcache_b200: one sample per call")
    eng.stage_inputs(lat, t, context[0], clip_fea=clip_fea, y=None if y is None else y[0],
                     vace_context=None if vace_context is None else vace_context[0], vace_scale=vace_scale,
                     n_pad=seq_len - n_tok if calibration else 0)
    return eng


def _wan_cached_step(self, eng, family, print_skip=False):
    """One cached Wan forward on staged inputs (MagCache4Wan2.1/magcache_generate.py:277-311; VACE :517-559; Wan2.2
    MagCache4Wan2.2/magcache_generate.py:290-334): decide, follow the residual attribute, hit or miss, store the residual, advance."""
    ctrl = _family_controller(self, family)
    slot = int(self.cnt) % 2
    skip_forward = ctrl.decide(self)  # float64 state under the reference's attribute names
    # Wan2.2: the other expert's residual arrives through the class-level list the two experts share
    eng.res_valid[slot] = _adopt_residual(self.residual_cache[slot], eng.res[slot], eng.res_valid[slot])
    if print_skip and skip_forward:
        print("skip: ", self.cnt)  # VACE, :527
    # hit : `x = x + residual_x` (:295) feeds only the head, so the sum is formed inside the head kernel (same fp32 arithmetic)
    # miss: block stack (:297-298), `residual_x = x - ori_x` (:299) written into the slot's buffer
    out = eng.forward("hit" if skip_forward else "miss", slot)
    self.residual_cache[slot] = eng.res[slot].view(1, *eng.res[slot].shape)  # :301
    ctrl.advance(self)  # :306-311
    return [out]


def magcache_forward(self, x, t, context, seq_len, clip_fea=None, y=None):
    r"""MagCache4Wan2.1/magcache_generate.py:198-312 on the B200 kernels.

    Args / returns as the reference: x List[Tensor[C_in, F, H, W]], t Tensor[B], context List[Tensor[L, C]], seq_len int
    -> List[Tensor[C_out, F, H, W]] (float32).
    """
    return _wan_cached_step(self, _stage(self, x, t, context, seq_len, clip_fea, y), "wan2.1")


def magcache_vace_forward(self, x, t, vace_context, context, seq_len, vace_context_scale=1.0, clip_fea=None, y=None):
    r"""MagCache4Wan2.1/magcache_generate.py:439-560 (installed at :1126-1150 with the VACE tables): the T2V forward plus the
    control branch. `vace_context`: List[Tensor[96, F, H, W]]. On a miss the control blocks run first (`forward_vace`, :541) and
    every second main block adds its hint; on a hit nothing of the control branch is computed, as in the reference. `clip_fea` and
    `y` are accepted and ignored (the reference has those lines commented out, :471-476, :505-507)."""
    eng = _stage(self, x, t, context, seq_len, None, None, vace_context=vace_context, vace_scale=vace_context_scale)
    return _wan_cached_step(self, eng, "wan2.1", print_skip=True)  # :517-559


def magcache_vace_calibration(self, x, t, vace_context, context, seq_len, vace_context_scale=1.0, clip_fea=None, y=None):
    r"""MagCache4Wan2.1/magcache_generate.py:314-436: `magcache_calibration` with the control branch."""
    return _calibrate(self, _stage(self, x, t, context, seq_len, None, None, calibration=True, vace_context=vace_context,
                                   vace_scale=vace_context_scale))


def magcache_wan22_forward(self, x, t, context, seq_len, clip_fea=None, y=None):
    r"""MagCache4Wan2.2/magcache_generate.py:209-336 for the A14B experts (T2V and I2V) on the Wan engine: the Wan2.1 forward with the
    two-expert skip windows (`split_step`, `mode`, :294-303) and a counter shared by the high-noise and the low-noise model — two
    instances of one class, one engine (weights) each, one controller state and one residual cache between them (:340-362).
    Wan2.2 gives every token its own timestep (:263-272). A 1-D `t` (the A14B experts) is one value for all tokens; TI2V-5B passes
    [1, seq_len] with t = 0 on the first-frame tokens of an image-conditioned run: the engine reduces it to its distinct values and the
    contiguous token ranges carrying them (`WanEngine._stage_t`), so the arithmetic per token is the reference's. With `split_step` None
    (TI2V, :301-303) the window is the plain `int(num_steps * retention_ratio)`."""
    if getattr(self, "model_type", "t2v") == "i2v":
        assert y is not None  # :239-240
    if t.dim() != 1:
        if t.size(0) != 1:
            raise NotImplementedError("magcache_b200: one sample per call")
        assert t.size(1) == seq_len  # what `.unflatten(0, (bt, seq_len))` (:270) requires
    eng = _stage(self, x, t, context, seq_len, None, y, require_clip=False)
    return _wan_cached_step(self, eng, "wan2.2-i2v" if getattr(self, "mode", "t2v") == "i2v" else "wan2.2-t2v")  # :290-334


def init_magcache_wan22(model, mag_ratios, sample_steps, thresh=0.06, K=2, retention_ratio=0.2, split_steps=None, mode="t2v"):
    """`init_magcache(model, mag_ratios, args, split_steps, mode)` of MagCache4Wan2.2/magcache_generate.py:340-362: patches the CLASS the
    two experts share. `mag_ratios`: the list without its `[1.0]*2` prefix like the script passes it, or a key of `tables()` (which
    already carries the prefix)."""
    cls = model.__class__
    cls.forward = magcache_wan22_forward
    cls.cnt = torch.tensor(0)
    cls.num_steps = sample_steps * 2
    cls.split_step = split_steps * 2 if split_steps else None
    cls.mode = mode
    cls.magcache_thresh, cls.K = thresh, K
    cls.accumulated_err, cls.accumulated_steps, cls.accumulated_ratio = [0.0, 0.0], [0, 0], [1.0, 1.0]
    cls.retention_ratio = retention_ratio
    cls.residual_cache = [None, None]
    mr = tables()[mag_ratios] if isinstance(mag_ratios, str) else np.array([1.0] * 2 + list(mag_ratios))
    cls.mag_ratios = interp_cfg(mr, sample_steps)  # :357-361
    return model


def magcache_calibration(self, x, t, context, seq_len, clip_fea=None, y=None):
    r"""MagCache4Wan2.1/magcache_generate.py:80-194: always runs the block stack and records, per forward, the token-mean
    magnitude ratio, its std and the cosine distance to the previous residual of the same CFG branch (one fused pass)."""
    return _calibrate(self, _stage(self, x, t, context, seq_len, clip_fea, y, calibration=True))


def _calibrate(self, eng):
    slot = self.cnt % 2
    out, residual, stats = eng.calibrate(slot, self.residual_cache[slot] if self.cnt >= 2 else None)  # :163-175
    if stats is not None:
        _record_stats(self, stats)
    self.residual_cache[slot] = residual.view(1, *residual.shape)
    self.cnt += 1
    if self.cnt >= self.num_steps:  # :180-193: the lists are printed and saved at the wrap
        self.cnt = 0
        self.accumulated_ratio = [1.0, 1.0]
        self.accumulated_err = [0.0, 0.0]
        self.accumulated_steps = [0, 0]
        _print_stats(self)
        # :191-193 `save_json("wan2_1_mag_ratio", self.norm_ratio)` ...: same file names, in `calibration_dir` (default: the
        # working directory, like the reference). `config.table_from_calibration` turns the first file into a `mag_ratios` table.
        out_dir = getattr(self, "calibration_dir", ".")
        if out_dir is not None:
            save_json(os.path.join(out_dir, "wan2_1_mag_ratio"), self.norm_ratio)
            save_json(os.path.join(out_dir, "wan2_1_mag_std"), self.norm_std)
            save_json(os.path.join(out_dir, "wan2_1_cos_dis"), self.cos_dis)
    return [out]


def init_magcache(model, sample_steps, thresh=0.12, K=2, retention_ratio=0.2, mag_ratios=None, ckpt_dir=None, table=None):
    """The installation block of magcache_generate.py:896-919 (i2v :989-1010, VACE :1126-1150) as a helper (same form as Wan2.2's
    `init_magcache`, MagCache4Wan2.2/magcache_generate.py:340-362): patches the CLASS, like the reference. VACE models
    (`model_type == "vace"`) get `magcache_vace_forward`."""
    cls = model.__class__
    cls.forward = magcache_vace_forward if getattr(model, "model_type", "t2v") == "vace" else magcache_forward
    cls.cnt = 0
    cls.num_steps = sample_steps * 2
    cls.magcache_thresh = thresh
    cls.K = K
    cls.accumulated_err = [0.0, 0.0]
    cls.accumulated_steps = [0, 0]
    cls.accumulated_ratio = [1.0, 1.0]
    cls.retention_ratio = retention_ratio
    cls.residual_cache = [None, None]
    if isinstance(mag_ratios, (str, os.PathLike)):  # a calibration dump (`wan2_1_mag_ratio.json`) instead of a pasted literal
        mag_ratios = table_from_calibration(mag_ratios)
    if mag_ratios is None:
        mag_ratios = tables()[table] if table is not None else table_for_ckpt_dir(ckpt_dir)
    cls.mag_ratios = interp_cfg(mag_ratios, sample_steps)  # :915-919
    return model


def reset_magcache(model):
    """Start a new video: cnt = 0 and fresh accumulators (what `pipeline.transformer.__class__.cnt = 0` between prompts is
    meant to do, MagCache4FLUX/magcache_flux.py:478). `self.cnt += 1` in the forward creates INSTANCE attributes that shadow
    the class-level ones the scripts install, so both levels are reset here. The residual cache is kept, as in the reference."""
    cls = model.__class__
    for attr in ("cnt", "accumulated_err", "accumulated_steps", "accumulated_ratio"):
        model.__dict__.pop(attr, None)
    cls.cnt = 0
    if isinstance(getattr(cls, "accumulated_err", None), list):
        cls.accumulated_err, cls.accumulated_steps, cls.accumulated_ratio = [0.0, 0.0], [0, 0], [1.0, 1.0]
    else:
        cls.accumulated_err, cls.accumulated_steps, cls.accumulated_ratio = 0, 0, 1.0
    return model


def init_magcache_calibration(model, sample_steps):
    """magcache_generate.py:921-928."""
    cls = model.__class__
    cls.forward = magcache_vace_calibration if getattr(model, "model_type", "t2v") == "vace" else magcache_calibration
    cls.cnt = 0
    cls.num_steps = sample_steps * 2
    cls.norm_ratio, cls.norm_std, cls.cos_dis = [], [], []
    cls.residual_cache = [None, None]
    return model


# ------------------------------------------------------------------------------------------------------------------
# Other adapters: controller + cache kernels around a caller-supplied block stack
# ------------------------------------------------------------------------------------------------------------------
def magcache_branch(self, hidden, run_blocks, family, cache_attr):
    """The hit/miss branch of the other adapters' forwards — FLUX / Kontext (magcache_flux.py:326-427), HunyuanVideo
    (magcache_sample_video.py:88-141), FramePack (magcache_demo_gradio.py:252-300), Wan2.2 / Qwen-Image
    (MagCache4Wan2.2/magcache_generate.py:290-334): decides with the family's controller (`config.FAMILIES`), then either adds
    the cached residual (K1 kernel) or calls `run_blocks(hidden)` (the model's own transformer stack) and stores `out - hidden`
    (K2 kernel) under `cache_attr` — a tensor for scalar-state families, a 2-list indexed by `cnt % 2` for per-branch ones.
    Advances the counter. Wan2.2's expert boundary is read from `self.split_step` like upstream (:344)."""
    ctrl = _family_controller(self, family)
    per_branch = FAMILIES[family]["branches"] == 2
    slot = int(self.cnt) % 2 if per_branch else None
    if ctrl.decide(self):
        cur = getattr(self, cache_attr)[slot] if per_branch else getattr(self, cache_attr)
        if cur is None:
            raise TypeError("magcache_b200: cache hit with an empty residual cache (reference: Tensor + NoneType)")
        out = ops.cache_hit_add(hidden.contiguous(), cur)
    else:
        out = run_blocks(hidden)
        cur = ops.residual_sub(out.contiguous(), hidden.contiguous())
    if per_branch:
        getattr(self, cache_attr)[slot] = cur
    else:
        setattr(self, cache_attr, cur)
    ctrl.advance(self)
    return out


# ------------------------------------------------------------------------------------------------------------------
# FLUX and HunyuanVideo: the whole patched forward on the MMDiT engines (magcache_b200/mmdit.py)
# ------------------------------------------------------------------------------------------------------------------
class _Sample:
    """Stand-in for diffusers' Transformer2DModelOutput (`.sample`), which is not importable here."""

    def __init__(self, sample):
        self.sample = sample


def _mmdit_cached_step(self, eng, family, res_attr):
    """One cached MMDiT forward on staged inputs (magcache_flux.py:326-436 ; magcache_sample_video.py:88-154): decide, follow the
    residual attribute `res_attr`, hit or miss, store the residual, advance. Returns the engine's output."""
    ctrl = _family_controller(self, family)
    skip_forward = ctrl.decide(self)
    eng.res_valid = _adopt_residual(getattr(self, res_attr), eng.res, eng.res_valid)
    out = eng.forward("hit" if skip_forward else "miss")
    setattr(self, res_attr, eng.res.view(1, *eng.res.shape))  # :427 ; :141
    ctrl.advance(self)
    return out


def _mmdit_calibration_step(self, eng, res_attr):
    """One MMDiT calibration call on staged inputs: block stack, statistics from the second call of a generation on, residual
    stored under `res_attr`. Returns the engine's output."""
    if self.cnt == 0:
        eng.res_valid = False  # `if self.cnt>=1` (magcache_flux.py:198 ; magcache_sample_video.py:254): nothing to compare with
    out, stats = eng.calibrate()
    if stats is not None:
        _record_stats(self, stats)
    setattr(self, res_attr, eng.res.view(1, *eng.res.shape))
    return out


def _flux_stage(self, hidden_states, encoder_hidden_states, pooled_projections, timestep, img_ids, txt_ids, guidance,
                joint_attention_kwargs, controlnet_block_samples, controlnet_single_block_samples):
    if joint_attention_kwargs or controlnet_block_samples is not None or controlnet_single_block_samples is not None:
        raise NotImplementedError("magcache_b200: joint_attention_kwargs / ControlNet residuals are not built for the FLUX engine")
    if not hidden_states.is_cuda:
        raise RuntimeError("magcache_b200: hidden_states must be CUDA tensors (no CPU path)")
    eng = _cached_engine(self, "_mc_flux_engine", FluxEngine, lambda: FluxWeights.from_module(self, hidden_states.device))
    eng.stage_inputs(hidden_states, encoder_hidden_states, pooled_projections, timestep, guidance,
                     img_ids[0] if img_ids.ndim == 3 else img_ids, txt_ids[0] if txt_ids.ndim == 3 else txt_ids)  # :305-316 (3-D ids)
    return eng


def magcache_flux_forward(self, hidden_states, encoder_hidden_states=None, pooled_projections=None, timestep=None, img_ids=None,
                          txt_ids=None, guidance=None, joint_attention_kwargs=None, controlnet_block_samples=None,
                          controlnet_single_block_samples=None, return_dict=True, controlnet_blocks_repeat=False):
    r"""MagCache4FLUX/magcache_flux.py:234-440 on the B200 kernels: same signature, same state attributes (`cnt, num_steps,
    magcache_thresh, K, retention_ratio, accumulated_ratio / _err / _steps, previous_residual, mag_ratios`), `(output,)` or an object
    with `.sample`. LoRA scaling, ip-adapter and ControlNet residuals (:275-288, :321-324, :371-381, :410-420) are not built and raise."""
    eng = _flux_stage(self, hidden_states, encoder_hidden_states, pooled_projections, timestep, img_ids, txt_ids, guidance,
                      joint_attention_kwargs, controlnet_block_samples, controlnet_single_block_samples)
    out = _mmdit_cached_step(self, eng, "flux", "previous_residual")
    output = out.view(1, *out.shape)
    if not return_dict:
        return (output,)
    return _Sample(output)


def magcache_flux_calibration(self, hidden_states, encoder_hidden_states=None, pooled_projections=None, timestep=None, img_ids=None,
                              txt_ids=None, guidance=None, joint_attention_kwargs=None, controlnet_block_samples=None,
                              controlnet_single_block_samples=None, return_dict=True, controlnet_blocks_repeat=False):
    r"""MagCache4FLUX/magcache_flux.py:21-231: every call runs the block stack and, from the second call on, records the token-mean
    magnitude ratio, its std and the cosine distance to the previous residual (`norm_ratio / norm_std / cos_dis`, rounded to 5 places);
    the lists are printed on the last call of a generation and cleared at the wrap (:207-221)."""
    eng = _flux_stage(self, hidden_states, encoder_hidden_states, pooled_projections, timestep, img_ids, txt_ids, guidance,
                      joint_attention_kwargs, controlnet_block_samples, controlnet_single_block_samples)
    out = _mmdit_calibration_step(self, eng, "previous_residual")
    if self.cnt >= self.num_steps - 1:  # :207-213
        _print_stats(self)
    self.cnt += 1
    if self.cnt >= self.num_steps:  # :219-222
        self.cnt = 0
        self.norm_ratio, self.norm_std, self.cos_dis = [], [], []
    output = out.view(1, *out.shape)
    return _Sample(output) if return_dict else (output,)


def init_magcache_flux_calibration(transformer, num_inference_steps=28):
    """magcache_flux.py:446-458 with `FluxTransformer2DModel.forward = magcache_calibration`."""
    cls = transformer.__class__
    cls.forward = magcache_flux_calibration
    cls.cnt, cls.num_steps = 0, num_inference_steps
    cls.norm_ratio, cls.norm_std, cls.cos_dis = [], [], []
    cls.previous_residual = None
    return transformer


def init_magcache_flux(transformer, num_inference_steps=28, thresh=0.24, K=5, retention_ratio=0.1, mag_ratios=None, table="flux_dev"):
    """The installation statements of magcache_flux.py:446-471 (Kontext: magcache_flux_kontext.py:445-470 with table "flux_kontext",
    thresh 0.05, K 4, retention 0.2): patches the CLASS."""
    cls = transformer.__class__
    cls.forward = magcache_flux_forward
    cls.cnt, cls.num_steps = 0, num_inference_steps
    mr = np.asarray(tables()[table] if mag_ratios is None else mag_ratios, dtype=np.float64)
    if len(mr) != num_inference_steps:  # :461-463
        mr = nearest_interp(mr, num_inference_steps)
    cls.mag_ratios = mr
    cls.K, cls.magcache_thresh, cls.retention_ratio = K, thresh, retention_ratio
    cls.accumulated_ratio, cls.accumulated_err, cls.accumulated_steps = 1, 0, 0
    cls.previous_residual = None
    return transformer


def _hunyuan_stage(self, x, t, text_states, text_mask, text_states_2, freqs_cos, freqs_sin, guidance):
    if not x.is_cuda:
        raise RuntimeError("magcache_b200: x must be a CUDA tensor (no CPU path)")
    eng = _cached_engine(self, "_mc_hunyuan_engine", HunyuanEngine, lambda: HunyuanWeights.from_module(self, x.device))
    eng.stage_inputs(x, t, text_states, text_mask, text_states_2, freqs_cos, freqs_sin, guidance)
    return eng


def magcache_hunyuan_forward(self, x, t, text_states=None, text_mask=None, text_states_2=None, freqs_cos=None, freqs_sin=None,
                             guidance=None, return_dict=True):
    r"""MagCache4HunyuanVideo/magcache_sample_video.py:29-160 on the B200 kernels (MMDiT engine, magcache_b200/mmdit.py): same
    signature and state attributes (`cnt, num_steps, magcache_thresh, K, retention_ratio, accumulated_ratio / _err / _steps,
    residual_cache, mag_ratios`), returns `{"x": img}` or the tensor. x [1, 16, T, H, W]; text_mask marks the valid (right-padded)
    text tokens."""
    eng = _hunyuan_stage(self, x, t, text_states, text_mask, text_states_2, freqs_cos, freqs_sin, guidance)
    img = _mmdit_cached_step(self, eng, "hunyuan", "residual_cache")
    if return_dict:
        return {"x": img}
    return img


def magcache_hunyuan_calibration(self, x, t, text_states=None, text_mask=None, text_states_2=None, freqs_cos=None, freqs_sin=None,
                                 guidance=None, return_dict=True):
    r"""MagCache4HunyuanVideo/magcache_sample_video.py:163-290: the calibration twin (statistics from the second call on, lists printed
    from call 49 on — hard-coded upstream, :264 — and a counter that is never wrapped, :277)."""
    eng = _hunyuan_stage(self, x, t, text_states, text_mask, text_states_2, freqs_cos, freqs_sin, guidance)
    img = _mmdit_calibration_step(self, eng, "residual_cache")
    if self.cnt >= 49:  # :264-270
        _print_stats(self)
    self.cnt += 1
    return {"x": img} if return_dict else img


def init_magcache_hunyuan_calibration(transformer, infer_steps=50):
    """magcache_sample_video.py:307-314 with `forward = magcache_calibration` (:324)."""
    cls = transformer.__class__
    cls.forward = magcache_hunyuan_calibration
    cls.cnt, cls.num_steps = 0, infer_steps
    cls.norm_ratio, cls.norm_std, cls.cos_dis = [], [], []
    cls.residual_cache = None
    return transformer


def init_magcache_hunyuan(transformer, infer_steps=50, thresh=0.24, K=6, retention_ratio=0.2, video_height=720, mag_ratios=None):
    """The installation statements of magcache_sample_video.py:303-328 (table chosen by `args.video_size[0]` in {720, 544}, :315-318)."""
    cls = transformer.__class__
    cls.cnt, cls.num_steps, cls.magcache_thresh, cls.K = 0, infer_steps, thresh, K
    cls.residual_cache = None
    if mag_ratios is None:
        if video_height not in (720, 544):
            raise KeyError(f"no calibrated table for video height {video_height} (the reference would hit AttributeError later)")
        mag_ratios = tables()["hunyuan_720p" if video_height == 720 else "hunyuan_544p"]
    mr = np.asarray(mag_ratios, dtype=np.float64)
    if len(mr) != infer_steps:
        mr = nearest_interp(mr, infer_steps)
    cls.mag_ratios, cls.retention_ratio = mr, retention_ratio
    cls.forward = magcache_hunyuan_forward
    cls.accumulated_ratio, cls.accumulated_err, cls.accumulated_steps = 1, 0, 0
    return transformer


# ------------------------------------------------------------------------------------------------------------------
# The paper-evaluation variant of the Wan forward (the code behind the published Wan2.1 numbers)
# ------------------------------------------------------------------------------------------------------------------
def magcache_eval_forward(self, x, t, context, seq_len, clip_fea=None, y=None):
    r"""eval/magcache/experiments/Wan2.1_EVAL/wan_magcache.py:682-817 on the B200 kernels, state under THAT script's attribute
    names (`t, num_steps, magcache_thresh, magcache_K, ratio, accumulated_sim, accumulated_err, accumulated_steps, residual_cache,
    skip_steps, pre_con`). Differences from `magcache_forward`, all reproduced: `<=` threshold compare, table indexed `ratio[t-10]`,
    retention fixed at `int(num_steps*0.2)`, residuals kept from call 10 on (`cache_time`) in a `[2, B, N, D, 1]` tensor — the
    depth-1 `push_tensor_roll` FIFO (:67-85, :796-799) is the engine's two residual slots viewed in place, no roll, no copy —
    and the conditional output of each step remembered in `pre_con` (:804-805)."""
    import ctypes

    from . import _lib
    from .controller import make_ctrl_config
    eng = _stage(self, x, t, context, seq_len, clip_fea, y)
    cache_time = 10                                  # :771
    ratio = self.ratio
    cc = self.__dict__.get("_mc_eval_cfg")
    key = (hash(np.ascontiguousarray(np.asarray(ratio, dtype=np.float64)).tobytes()), len(ratio), self.num_steps, float(self.magcache_thresh),
           int(self.magcache_K))
    if cc is None or cc[0] != key:
        cc = (key, make_ctrl_config(self.num_steps, self.magcache_thresh, self.magcache_K, 0.2, ratio, **FAMILIES["wan2.1-eval"]))
        object.__setattr__(self, "_mc_eval_cfg", cc)
    cfg = cc[1]
    st = _lib.CtrlState()
    st.cnt = int(self.t)
    for i in range(2):
        st.accumulated_ratio[i], st.accumulated_err[i], st.accumulated_steps[i] = float(self.accumulated_sim[i]), float(self.accumulated_err[i]), int(self.accumulated_steps[i])
    skip = ctypes.c_int32()
    _lib.check(_lib.lib.mc_ctrl_decide(ctypes.byref(cfg), ctypes.byref(st), ctypes.byref(skip)))  # :774-786
    for i in range(2):  # the reference mutates the lists in place
        self.accumulated_sim[i], self.accumulated_err[i], self.accumulated_steps[i] = st.accumulated_ratio[i], st.accumulated_err[i], st.accumulated_steps[i]
    slot = self.t % 2
    if skip.value:
        self.skip_steps += 1
        print(f"skip time {self.t}, cur_scale: {ratio[self.t - 10]}, acc_sim: {self.accumulated_sim[slot]}, total_steps: {self.skip_steps}")  # :790
    out = eng.forward("hit" if skip.value else "miss", slot)
    if self.t >= cache_time:                         # :796-799
        self.residual_cache = eng.res_buf.view(2, 1, *eng.res_buf.shape[1:], 1)
    if self.t % 2 == 0:
        self.pre_con = [out]                         # :804-805
    self.t += 1                                      # :807-815
    if self.t >= self.num_steps:
        self.t = 0
        self.skip_steps = 0
        self.accumulated_sim = [1.0, 1.0]
        self.accumulated_steps = [0, 0]
        self.accumulated_err = [0, 0]
    return [out]


def init_magcache_eval(model, sample_steps, thresh=0.12, K=2, ratio=None):
    """The installation block of wan_magcache.py:1129-1150 as a helper ("slow" = 0.12/K2, "fast" = 0.12/K4, wan_eval.sh:30-31,66-67)."""
    cls = model.__class__
    cls.forward = magcache_eval_forward
    cls.magcache_thresh, cls.magcache_K = thresh, K
    cls.t, cls.accumulated_err, cls.skip_steps, cls.pre_con = 0, [0, 0], 0, None
    cls.num_steps = sample_steps * 2
    cls.ratio = np.asarray(tables()["wan2.1_eval"] if ratio is None else ratio, dtype=np.float64)
    cls.residual_cache = None
    cls.accumulated_sim, cls.accumulated_steps = [1, 1], [0, 0]
    return model


# ------------------------------------------------------------------------------------------------------------------
# TeaCache comparator (the baseline of every published MagCache table) on the same engine
# ------------------------------------------------------------------------------------------------------------------
# coefficients of eval/magcache/experiments/Wan2.1_EVAL/wan_teacache.py:913-926 (t2v) — keyed by (use_ret_steps, model size)
TEACACHE_COEFFICIENTS = {
    (True, "1.3B"): [-5.21862437e+04, 9.23041404e+03, -5.28275948e+02, 1.36987616e+01, -4.99875664e-02],
    (True, "14B"): [-3.03318725e+05, 4.90537029e+04, -2.65530556e+03, 5.87365115e+01, -3.15583525e-01],
    (False, "1.3B"): [2.39676752e+03, -1.31110545e+03, 2.01331979e+02, -8.29855975e+00, 1.37887774e-01],
    (False, "14B"): [-5784.54975374, 5449.50911966, -1811.16591783, 256.27178429, -13.02252404],
}


def _tea_structs(self):
    import ctypes

    from . import _lib
    coef = [float(c) for c in self.coefficients]
    cfg = _lib.TeaConfig()
    cfg.num_steps, cfg.ret_steps, cfg.cutoff_steps, cfg.n_coef, cfg.thresh = int(self.num_steps), int(self.ret_steps), int(self.cutoff_steps), len(coef), float(self.teacache_thresh)
    for i, c in enumerate(coef):
        cfg.coef[i] = c
    st = _lib.TeaState()
    st.cnt = int(self.cnt)
    st.accumulated[0], st.accumulated[1] = float(self.accumulated_rel_l1_distance_even), float(self.accumulated_rel_l1_distance_odd)
    return ctypes, _lib, cfg, st


def teacache_forward(self, x, t, context, seq_len, clip_fea=None, y=None):
    r"""eval/magcache/experiments/Wan2.1_EVAL/wan_teacache.py:457-590 on the B200 kernels, state under the reference's attribute
    names (`cnt, num_steps, teacache_thresh, accumulated_rel_l1_distance_even/odd, previous_e0_even/odd,
    previous_residual_even/odd, use_ref_steps, ret_steps, cutoff_steps, coefficients, enable_teacache`). The decision reads the
    relative L1 change of the modulated time embedding (one tiny reduction + the `.item()` sync the reference has), the hit /
    miss branches are the MagCache ones (`x += previous_residual` | block stack, residual = x - ori_x)."""
    eng = _stage(self, x, t, context, seq_len, clip_fea, y)
    if not self.enable_teacache:  # :584-586: plain forward (the counter still advances, :587-589)
        out = eng.forward("miss", self.cnt % 2)
        self.cnt = 0 if self.cnt + 1 >= self.num_steps else self.cnt + 1
        return [out]
    ctypes, _lib, cfg, st = _tea_structs(self)
    slot = self.cnt % 2
    suffix = "even" if slot == 0 else "odd"
    e, e0 = eng.time_embedding()
    modulated = (e0 if self.use_ref_steps else e).reshape(-1)  # :534
    needs = ctypes.c_int32()
    _lib.check(_lib.lib.mc_tea_needs_distance(ctypes.byref(cfg), ctypes.byref(st), ctypes.byref(needs)))
    dist = ops.rel_l1(modulated, getattr(self, "previous_e0_" + suffix).reshape(-1)) if needs.value else 0.0
    calc = ctypes.c_int32()
    _lib.check(_lib.lib.mc_tea_decide(ctypes.byref(cfg), ctypes.byref(st), dist, ctypes.byref(calc)))
    self.accumulated_rel_l1_distance_even, self.accumulated_rel_l1_distance_odd = st.accumulated[0], st.accumulated[1]
    setattr(self, "previous_e0_" + suffix, modulated.clone().view((e0 if self.use_ref_steps else e).shape))  # :549 / :564
    eng.res_valid[slot] = _adopt_residual(getattr(self, "previous_residual_" + suffix), eng.res[slot], eng.res_valid[slot])
    eng.hit_sum_bf16 = True  # `x += self.previous_residual_*` in place on the bf16 patch embedding (:569 / :577): the sum is rounded to bf16
    try:
        out = eng.forward("miss" if calc.value else "hit", slot)
    finally:
        eng.hit_sum_bf16 = False
    setattr(self, "previous_residual_" + suffix, eng.res[slot].view(1, *eng.res[slot].shape))
    _lib.check(_lib.lib.mc_tea_advance(ctypes.byref(cfg), ctypes.byref(st)))
    self.cnt = st.cnt  # :587-589
    return [out]


def init_teacache(model, sample_steps, teacache_thresh=0.2, use_ret_steps=False, ckpt_dir=None, coefficients=None):
    """The installation block of wan_teacache.py:899-928 as a helper: patches the CLASS. Coefficients are chosen by the '1.3B' /
    '14B' substring of `ckpt_dir` like the reference, or passed explicitly."""
    cls = model.__class__
    cls.enable_teacache = True
    cls.forward = teacache_forward
    cls.cnt = 0
    cls.num_steps = sample_steps * 2
    cls.teacache_thresh = teacache_thresh
    cls.accumulated_rel_l1_distance_even = 0
    cls.accumulated_rel_l1_distance_odd = 0
    cls.previous_e0_even = cls.previous_e0_odd = None
    cls.previous_residual_even = cls.previous_residual_odd = None
    cls.use_ref_steps = use_ret_steps
    if coefficients is None:
        size = "1.3B" if "1.3B" in (ckpt_dir or "") else ("14B" if "14B" in (ckpt_dir or "") else None)
        if size is None:
            raise KeyError(f"no TeaCache coefficients match ckpt_dir={ckpt_dir!r} (the reference would hit AttributeError later)")
        coefficients = TEACACHE_COEFFICIENTS[(bool(use_ret_steps), size)]
    cls.coefficients = list(coefficients)
    if use_ret_steps:
        cls.ret_steps, cls.cutoff_steps = 10 * 2, sample_steps * 2
    else:
        cls.ret_steps, cls.cutoff_steps = 1 * 2, sample_steps * 2 - 2
    return model
