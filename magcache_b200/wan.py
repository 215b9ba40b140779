"""Wan2.1 DiT engine: device-resident weights in the layout the sm_100a kernels want, plus the kernel sequence of one forward.

This is the cache-miss branch of the reference (`for block in self.blocks: x = block(x, **kwargs)`,
MagCache4Wan2.1/magcache_generate.py:297-298) and the prologue / epilogue around it (:229-275, :304-305), rebuilt on the
C-ABI kernels. Block arithmetic follows upstream Wan2.1 `wan/modules/model.py` [EXT] as restated in SURVEY.md Appendix B.1.

HBM layout per forward (N tokens, D model dim, F ffn dim; Wan2.1-1.3B at 832x480x81: N=32760, D=1536, F=8960):
  x0   bf16 [N, D]     patch-embedding output (`ori_x`)            h    bf16 [N, D]    LN+modulate output (GEMM A operand)
  xs   fp32 [N, D]     residual stream, updated in place           qkv  bf16 [N, 3D]   fused q|k|v projection (one GEMM; RMSNorm+RoPE in
  att  bf16 [N, D]     attention output                                                place on the q and k column blocks)
  ffn  bf16 [N, F]     GELU(ffn[0]) output                         ctx  bf16 [512, D]  text embedding; ckv bf16 [512, 2D] its per-layer k|v
The attention kernel reads q, k and v as column slices of `qkv` (row pitch 3D): V stays row-major, nothing is transposed.
All buffers are allocated once per engine and reused by every forward (no allocator traffic in the loop).
"""
import math
import os
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, ops

E = _lib


@dataclass
class WanDims:
    dim: int = 1536
    ffn_dim: int = 8960
    num_heads: int = 12
    num_layers: int = 30
    in_dim: int = 16
    out_dim: int = 16
    freq_dim: int = 256
    text_dim: int = 4096
    text_len: int = 512
    eps: float = 1e-6
    model_type: str = "t2v"   # "i2v": in_dim 36 (noise | mask + first-frame latents), CLIP image tokens through `img_emb`
    clip_dim: int = 1280
    clip_len: int = 257
    vace_layers: tuple = ()   # "vace": main-block indices that receive a hint (upstream default: every second block)
    vace_in_dim: int = 96

    @property
    def head_dim(self):
        return self.dim // self.num_heads


WAN_CONFIGS = {
    "t2v-1.3B": WanDims(1536, 8960, 12, 30),
    "t2v-14B": WanDims(5120, 13824, 40, 40),
    "i2v-14B": WanDims(5120, 13824, 40, 40, in_dim=36, model_type="i2v"),
    "vace-1.3B": WanDims(1536, 8960, 12, 30, model_type="vace", vace_layers=tuple(range(0, 30, 2))),
    "vace-14B": WanDims(5120, 13824, 40, 40, model_type="vace", vace_layers=tuple(range(0, 40, 5))),
    # Wan2.2 TI2V-5B (MagCache4Wan2.2, table `wan2.2_ti2v_5b_*`): 48 latent channels in and out, per-token timesteps
    "ti2v-5B": WanDims(3072, 14336, 24, 30, in_dim=48, out_dim=48),
}

MAX_T_VALUES = 8    # distinct timesteps in one call (the time MLP kernel takes <= 8 rows)
MAX_T_RUNS = 64     # contiguous token ranges of equal timestep in one call


def _bf16(t, device):
    return t.detach().to(device=device, dtype=torch.bfloat16).contiguous()


def _f32(t, device):
    return t.detach().to(device=device, dtype=torch.float32).contiguous()


def _bias_autocast(t, device):
    """Under bf16 autocast nn.Linear casts its bias to bf16 too; the epilogue adds it in fp32, so keep the rounded value as fp32.
    The MMDiT engines keep their (bf16) biases and norm weights this way as well."""
    return t.detach().to(device=device, dtype=torch.bfloat16).float().contiguous()


class WanWeights:
    """Weights of one WanModel, repacked for the kernels. Build with `from_module` (any module exposing upstream Wan attribute
    names: patch_embedding, text_embedding, time_embedding, time_projection, blocks[i].{norm3,self_attn,cross_attn,ffn,modulation},
    head.{head,modulation}) or `random` (seeded synthetic weights created directly on the device)."""

    def __init__(self, dims: WanDims, device):
        self.dims, self.device = dims, device
        self.blocks = []

    @classmethod
    def from_module(cls, m, device):
        D = m.dim
        dims = WanDims(dim=D, ffn_dim=m.ffn_dim, num_heads=m.num_heads, num_layers=len(m.blocks), in_dim=m.patch_embedding.in_channels,
                       out_dim=m.out_dim, freq_dim=m.freq_dim, text_dim=m.text_embedding[0].in_features, text_len=m.text_len,
                       eps=getattr(m, "eps", 1e-6), model_type=getattr(m, "model_type", "t2v"))
        if dims.model_type == "i2v" and not hasattr(m, "img_emb"):
            dims.model_type = "t2v"  # Wan2.2 I2V-A14B: `y` under the latent channels (in_dim 36) but no CLIP tokens, plain text cross-attention
        if dims.model_type not in ("t2v", "i2v", "vace"):
            raise NotImplementedError(f"model_type {dims.model_type!r}: t2v, i2v and vace forwards are built")
        if dims.head_dim != 128:
            raise NotImplementedError(f"head_dim {dims.head_dim}: the attention kernel is built for head_dim 128 (Wan2.1 1.3B and 14B)")
        assert tuple(m.patch_embedding.kernel_size) == (1, 2, 2), "patch size (1,2,2) only"
        w = cls(dims, device)
        pe = m.patch_embedding
        w.patch_w = _bf16(pe.weight.flatten(1), device)            # [D, C*4] in (c, kt, kh, kw) order
        w.patch_b = _bias_autocast(pe.bias, device)
        te = m.text_embedding
        w.text_w1, w.text_b1 = _bf16(te[0].weight, device), _bias_autocast(te[0].bias, device)
        w.text_w2, w.text_b2 = _bf16(te[2].weight, device), _bias_autocast(te[2].bias, device)
        tm = m.time_embedding
        w.time_w1, w.time_b1 = _f32(tm[0].weight, device), _f32(tm[0].bias, device)
        w.time_w2, w.time_b2 = _f32(tm[2].weight, device), _f32(tm[2].bias, device)
        tp = m.time_projection[1]
        w.tproj_w, w.tproj_b = _f32(tp.weight, device), _f32(tp.bias, device)
        w.blocks = [cls._pack_block(blk, dims, device) for blk in m.blocks]
        if dims.model_type == "vace":  # VaceWanModel: control-stream blocks with before/after projections, own patch embedding
            dims.vace_layers, dims.vace_in_dim = tuple(m.vace_layers), m.vace_patch_embedding.in_channels
            w.vace_patch_w = _bf16(m.vace_patch_embedding.weight.flatten(1), device)
            w.vace_patch_b = _bias_autocast(m.vace_patch_embedding.bias, device)
            w.vace_blocks = []
            for j, vb in enumerate(m.vace_blocks):
                b = cls._pack_block(vb, dims, device)
                if j == 0:
                    b["w_before"], b["b_before"] = _bf16(vb.before_proj.weight, device), _bias_autocast(vb.before_proj.bias, device)
                b["w_after"], b["b_after"] = _bf16(vb.after_proj.weight, device), _bias_autocast(vb.after_proj.bias, device)
                w.vace_blocks.append(b)
        if dims.model_type == "i2v":
            pj = m.img_emb.proj  # MLPProj: LayerNorm, Linear, GELU(erf), Linear, LayerNorm
            dims.clip_dim = pj[1].in_features
            w.img_ln1_w, w.img_ln1_b, w.img_ln1_eps = _f32(pj[0].weight, device), _f32(pj[0].bias, device), pj[0].eps
            w.img_w1, w.img_b1 = _bf16(pj[1].weight, device), _bias_autocast(pj[1].bias, device)
            w.img_w2, w.img_b2 = _bf16(pj[3].weight, device), _bias_autocast(pj[3].bias, device)
            w.img_ln2_w, w.img_ln2_b, w.img_ln2_eps = _f32(pj[4].weight, device), _f32(pj[4].bias, device), pj[4].eps
        w.head_mod = _f32(m.head.modulation.reshape(2, D), device)
        w.head_wt = _f32(m.head.head.weight.t(), device)           # [D, 64]: transposed for the head kernel's K-chunk staging
        w.head_b = _f32(m.head.head.bias, device)
        return w

    @staticmethod
    def _pack_block(blk, dims, device):
        D = dims.dim
        sa, ca = blk.self_attn, blk.cross_attn
        b = {
            "mod": _f32(blk.modulation.reshape(6, D), device),
            "w_qkv": _bf16(torch.cat([sa.q.weight, sa.k.weight, sa.v.weight], 0), device),   # one [3D, D] projection
            "b_qkv": _bias_autocast(torch.cat([sa.q.bias, sa.k.bias, sa.v.bias], 0), device),
            "w_o": _bf16(sa.o.weight, device), "b_o": _bias_autocast(sa.o.bias, device),
            "nqk": _f32(torch.stack([sa.norm_q.weight, sa.norm_k.weight]), device),   # [2, D]: q | k normalised in one launch
            "n3_w": _f32(blk.norm3.weight, device), "n3_b": _f32(blk.norm3.bias, device),
            "c_wq": _bf16(ca.q.weight, device), "c_bq": _bias_autocast(ca.q.bias, device),
            "c_wkv": _bf16(torch.cat([ca.k.weight, ca.v.weight], 0), device),                # text k|v: one [2D, D] projection
            "c_bkv": _bias_autocast(torch.cat([ca.k.bias, ca.v.bias], 0), device),
            "c_wo": _bf16(ca.o.weight, device), "c_bo": _bias_autocast(ca.o.bias, device),
            "c_nq": _f32(ca.norm_q.weight, device), "c_nk": _f32(ca.norm_k.weight, device),
            "w_f1": _bf16(blk.ffn[0].weight, device), "b_f1": _bias_autocast(blk.ffn[0].bias, device),
            "w_f2": _bf16(blk.ffn[2].weight, device), "b_f2": _bias_autocast(blk.ffn[2].bias, device),
        }
        if dims.model_type == "i2v":  # WanI2VCrossAttention: own k / v projections and key norm for the CLIP tokens
            b.update({"c_wkv_img": _bf16(torch.cat([ca.k_img.weight, ca.v_img.weight], 0), device),
                      "c_bkv_img": _bias_autocast(torch.cat([ca.k_img.bias, ca.v_img.bias], 0), device),
                      "c_nk_img": _f32(ca.norm_k_img.weight, device)})
        return b

    @classmethod
    def random(cls, dims: WanDims, device, seed=0):
        """Seeded synthetic weights with upstream's init scales (xavier-uniform Linears, N(0, 0.02) embeddings) but non-zero
        biases / head so every term is exercised. Created on the device: a 1.3B model is 2.8 GB in bf16."""
        g = torch.Generator(device=device).manual_seed(seed)
        D, F = dims.dim, dims.ffn_dim
        w = cls(dims, device)

        def xav(o, i):
            a = math.sqrt(6.0 / (i + o))
            return ((torch.rand(o, i, device=device, generator=g) * 2 - 1) * a)

        def small(*shape):
            return 0.02 * torch.randn(*shape, device=device, generator=g)

        def bias(n):
            return small(n).bfloat16().float()

        w.patch_w, w.patch_b = xav(D, dims.in_dim * 4).bfloat16(), bias(D)
        w.text_w1, w.text_b1 = small(D, dims.text_dim).bfloat16(), bias(D)
        w.text_w2, w.text_b2 = small(D, D).bfloat16(), bias(D)
        w.time_w1, w.time_b1 = small(D, dims.freq_dim), small(D)
        w.time_w2, w.time_b2 = small(D, D), small(D)
        w.tproj_w, w.tproj_b = small(6 * D, D), small(6 * D)
        def rand_block():
            blk = {
                "mod": torch.randn(6, D, device=device, generator=g) / math.sqrt(D),
                "w_qkv": torch.cat([xav(D, D), xav(D, D), xav(D, D)], 0).bfloat16(), "b_qkv": bias(3 * D),
                "w_o": xav(D, D).bfloat16(), "b_o": bias(D),
                "nqk": 1 + 0.1 * torch.randn(2, D, device=device, generator=g),
                "n3_w": 1 + 0.1 * torch.randn(D, device=device, generator=g), "n3_b": small(D),
                "c_wq": xav(D, D).bfloat16(), "c_bq": bias(D), "c_wkv": torch.cat([xav(D, D), xav(D, D)], 0).bfloat16(), "c_bkv": bias(2 * D),
                "c_wo": xav(D, D).bfloat16(), "c_bo": bias(D),
                "c_nq": 1 + 0.1 * torch.randn(D, device=device, generator=g), "c_nk": 1 + 0.1 * torch.randn(D, device=device, generator=g),
                "w_f1": xav(F, D).bfloat16(), "b_f1": bias(F), "w_f2": xav(D, F).bfloat16(), "b_f2": bias(D),
            }
            if dims.model_type == "i2v":
                blk.update({"c_wkv_img": torch.cat([xav(D, D), xav(D, D)], 0).bfloat16(), "c_bkv_img": bias(2 * D),
                            "c_nk_img": 1 + 0.1 * torch.randn(D, device=device, generator=g)})
            return blk

        for _ in range(dims.num_layers):
            w.blocks.append(rand_block())
        if dims.model_type == "vace":
            assert dims.vace_layers and dims.vace_layers[0] == 0
            w.vace_patch_w, w.vace_patch_b = xav(D, dims.vace_in_dim * 4).bfloat16(), bias(D)
            w.vace_blocks = []
            for j in range(len(dims.vace_layers)):
                blk = rand_block()
                if j == 0:
                    blk["w_before"], blk["b_before"] = (0.3 * xav(D, D)).bfloat16(), bias(D)
                blk["w_after"], blk["b_after"] = (0.3 * xav(D, D)).bfloat16(), bias(D)
                w.vace_blocks.append(blk)
        if dims.model_type == "i2v":
            Cd = dims.clip_dim
            w.img_ln1_w, w.img_ln1_b, w.img_ln1_eps = 1 + 0.1 * torch.randn(Cd, device=device, generator=g), small(Cd), 1e-5
            w.img_w1, w.img_b1 = small(Cd, Cd).bfloat16(), bias(Cd)
            w.img_w2, w.img_b2 = small(D, Cd).bfloat16(), bias(D)
            w.img_ln2_w, w.img_ln2_b, w.img_ln2_eps = 1 + 0.1 * torch.randn(D, device=device, generator=g), small(D), 1e-5
        w.head_mod = torch.randn(2, D, device=device, generator=g) / math.sqrt(D)
        w.head_wt = small(D, 4 * dims.out_dim).contiguous()
        w.head_b = small(4 * dims.out_dim)
        return w


def rope_table(grid, head_dim, device):
    """cos/sin of the 3-axis rotary embedding for every token of an (f, h, w) grid, computed in float64 exactly as upstream
    `rope_params` + `rope_apply` build them (theta 10000, split c-2(c//3) | c//3 | c//3 with c = head_dim/2), stored fp32
    [f*h*w, head_dim] as interleaved (cos, sin) pairs."""
    f, h, w = grid
    c = head_dim // 2
    split = [c - 2 * (c // 3), c // 3, c // 3]
    dims = [head_dim - 4 * (head_dim // 6), 2 * (head_dim // 6), 2 * (head_dim // 6)]
    angs = []
    for n, d, s in zip((f, h, w), dims, split):
        inv = 1.0 / np.power(10000.0, np.arange(0, d, 2, dtype=np.float64) / d)
        assert len(inv) == s
        angs.append(np.outer(np.arange(n, dtype=np.float64), inv))
    ang = np.concatenate([np.broadcast_to(angs[0][:, None, None, :], (f, h, w, split[0])),
                          np.broadcast_to(angs[1][None, :, None, :], (f, h, w, split[1])),
                          np.broadcast_to(angs[2][None, None, :, :], (f, h, w, split[2]))], axis=-1).reshape(f * h * w, c)
    cs = np.stack([np.cos(ang), np.sin(ang)], axis=-1).reshape(f * h * w, head_dim)
    return torch.from_numpy(cs.astype(np.float32)).clone().to(device)  # clone: torch-allocated (64-byte aligned) storage on CPU too


class WanEngine:
    """Runs prologue / block stack / head of one Wan forward on the kernels. One engine per (weights, token count)."""

    def __init__(self, weights: WanWeights, shard_world=1, shard_rank=0, shard_group=None, native=None):
        self.w = weights
        self.dims = weights.dims
        self.device = weights.device
        self._n = None
        self._rope = {}
        # token-axis sharding (magcache_b200/shard.py): world 1 = single GPU
        self.world, self.rank, self.group = shard_world, shard_rank, shard_group
        self.shard = None
        # CUDA-graph replay of the whole forward (one graph per {miss, hit} x CFG slot). On by default for sharded runs, where
        # ~650 launches per ~40 ms forward would otherwise leave the GPU waiting for the host; MC_GRAPHS=0/1 overrides.
        env = os.environ.get("MC_GRAPHS")
        self.use_graphs = (shard_world > 1) if env is None else (env == "1")
        self._graphs = {}
        self.xch = None  # K|V exchange of a token-sharded engine (shard.py)
        # native=True / MC_NATIVE=1: plain forwards (one timestep, one GPU, t2v, 16 output channels) are ONE call into the library —
        # `mc_dit_forward` (csrc/dit_forward.cu) issues the launch sequence below from native code, bit-identically. Off by default:
        # per-kernel timing tags (`ops.PROFILE`, what bench.py's attribution reads) exist only on the Python-sequenced path.
        env_n = os.environ.get("MC_NATIVE")
        self.native = (env_n == "1") if native is None else bool(native)
        self._nat, self._nat_grid = None, None
        self._slot = 0   # CFG slot of the forward in flight (selects the output window of a sharded engine)
        self.hit_sum_bf16 = False  # TeaCache comparator: the hit sum is rounded to bf16 before the head (wan_teacache.py:569/577)
        self._step = None          # (cond, x_latent, guide_scale, coef_x, coef_v, out) armed by `arm_step` for the next forward
        # per-token timesteps (Wan2.2, MagCache4Wan2.2/magcache_generate.py:263-272): the distinct values of this call and the
        # contiguous LOCAL row ranges that carry them, [(row0, row1, value index)]; None = one timestep for every token
        self.t_values, self.runs, self._runs_key = 1, None, None
        # the head kernel produces 64 output features (16 channels x the 2x2 patch) per launch: a model with more output channels
        # (TI2V-5B: 48) runs it once per group of 16 channels, on the matching columns of head.weight (feature index = p * C + c)
        C = self.dims.out_dim
        if C % 16:
            raise NotImplementedError(f"out_dim {C}: the head kernel writes 16 channels per launch")
        if C == 16:
            self.head_groups = [(weights.head_wt, weights.head_b)]
        else:
            wt, hb = weights.head_wt.view(self.dims.dim, 4, C), weights.head_b.view(4, C)
            self.head_groups = [(wt[:, :, g:g + 16].reshape(self.dims.dim, 64).contiguous(), hb[:, g:g + 16].reshape(64).contiguous())
                                for g in range(0, C, 16)]

    # ------------------------------------------------------------------------------------------ workspace
    def _workspace(self, n_total, pad_row=0):
        """`pad_row` = 1 (calibration with seq_len > token count): one extra row after the tokens stands for ALL the zero rows the
        reference pads the sequence with (magcache_generate.py:243-246) — they are identical (zero input, no RoPE, same keys), so one
        is computed and the caller weights it. It is a query only: keys / values stay the `n_total` tokens (`k_lens` upstream)."""
        if self._n == (n_total, pad_row):
            return
        d, dev = self.dims, self.device
        D, F = d.dim, d.ffn_dim
        self.n_keys, self.pad_row = n_total, pad_row
        bf = dict(dtype=torch.bfloat16, device=dev)
        if self.world > 1:
            if pad_row:
                raise NotImplementedError("magcache_b200: calibration with seq_len > token count on a token-sharded engine")
            from .shard import TokenShard, make_exchange
            self.shard = TokenShard(self.rank, self.world, n_total, self.group)
            n = self.shard.n_local
            # local q projection; the k | v rows are written straight into this rank's segment of the gathered buffers, which the
            # exchange (magcache_b200/shard.py) fills with every other rank's rows while the attention kernel already runs
            self.q_loc = torch.empty(n, D, **bf)
            if self.xch is not None:
                self.xch.close()
            self.xch = make_exchange(self.shard, 2 * D, (d.out_dim, self.grid[0], 2 * self.grid[1], 2 * self.grid[2]), dev)
            self._xi = 0
        else:
            n = n_total + pad_row
            self.qkv = torch.empty(n, 3 * D, **bf)
        self.x0 = torch.empty(n, D, **bf)
        self.xs = torch.empty(n, D, dtype=torch.float32, device=dev)
        self.h = torch.empty(n, D, **bf)
        self.att = torch.empty(n, D, **bf)
        self.ffn = torch.empty(n, F, **bf)
        self.cq = torch.empty(n, D, **bf)
        self.ckv = torch.empty(d.text_len, 2 * D, **bf)
        self.ctx_in = torch.zeros(d.text_len, d.text_dim, **bf)
        self.ctx_h = torch.empty(d.text_len, D, **bf)
        self.ctx = torch.empty(d.text_len, D, **bf)
        self.em = torch.empty(MAX_T_VALUES, 6, D, dtype=torch.float32, device=dev)  # modulation + e0, one [6, D] per timestep value
        if d.model_type == "vace":
            self.cs = torch.empty(n, D, dtype=torch.float32, device=dev)             # control stream (fp32 like the main one)
            self.cbf = torch.empty(len(d.vace_layers), n, D, **bf)                   # bf16 copies = A operands of the after_proj GEMMs
            self.vgate = torch.ones(D, dtype=torch.float32, device=dev)              # vace_context_scale, broadcast over features
            self.s_vace = None
        if d.model_type == "i2v":
            cl = d.clip_len
            self.clip_in = torch.zeros(cl, d.clip_dim, dtype=torch.float32, device=dev)
            self.clip_h1 = torch.empty(cl, d.clip_dim, **bf)
            self.clip_h2 = torch.empty(cl, d.clip_dim, **bf)
            self.clip_h3 = torch.empty(cl, D, **bf)
            self.ctx_img = torch.empty(cl, D, **bf)
            self.ckv_img = torch.empty(cl, 2 * D, **bf)
            self.att_img = torch.empty(n, D, **bf)
        # engine-owned residual cache storage (one slot per CFG branch) and staged inputs: fixed addresses for graph replay
        self.res_buf = torch.empty(2, n, D, dtype=torch.float32, device=dev)  # one buffer: the paper-eval forward exposes it whole
        self.res = [self.res_buf[0], self.res_buf[1]]
        self.res_valid = [False, False]
        self.s_t = torch.zeros(MAX_T_VALUES, dtype=torch.float64, device=dev)
        self.s_lat = None
        self._graphs = {}
        self._n = (n_total, pad_row)

    def _rope_for(self, grid):
        key = (grid, self.pad_row)
        if key not in self._rope:
            tab = rope_table(grid, self.dims.head_dim, self.device)
            if self.pad_row:  # the padded rows are not rotated (`rope_apply` leaves the tail untouched): cos 1, sin 0
                ident = torch.tensor([1.0, 0.0], device=self.device).repeat(self.dims.head_dim // 2)[None]
                tab = torch.cat([tab, ident]).contiguous()
            self._rope[key] = tab
        return self._rope[key]

    # ------------------------------------------------------------------------------------------ prologue (:229-275)
    def stage_inputs(self, latent, t, context, clip_fea=None, y=None, vace_context=None, vace_scale=1.0, n_pad=0):
        """Copy one call's inputs into the engine's fixed buffers (outside any captured graph): latent fp32 [C, F, H, W],
        t tensor [1], context [L <= text_len, text_dim] (zero-padded to text_len, cast to bf16 as autocast would); i2v also
        y [C_y, F, H, W] (concatenated under the latent channels, magcache_generate.py:233-234) and clip_fea [1, 257, clip_dim].
        `n_pad` (calibration only): the zero rows the reference appends after the tokens (seq_len - token count); `calibrate` weights
        one representative pad row by that count."""
        d = self.dims
        C, Fr, H, W = latent.shape
        if d.model_type == "i2v":
            assert clip_fea is not None and y is not None  # :226-227
        c_y = 0 if y is None else y.shape[0]
        if C + c_y != d.in_dim:
            raise ValueError(f"magcache_b200: {C}+{c_y} input channels, the patch embedding takes {d.in_dim}")
        self.grid = (Fr, H // 2, W // 2)
        self.n_pad = n_pad
        self._workspace(self.grid[0] * self.grid[1] * self.grid[2], 1 if n_pad else 0)
        shape = (C + c_y, Fr, H, W)
        if self.s_lat is None or tuple(self.s_lat.shape) != shape:
            self.s_lat = torch.empty(shape, dtype=torch.float32, device=self.device)
            self._graphs = {}
        self.s_lat[:C].copy_(latent)
        if y is not None:
            assert tuple(y.shape[1:]) == (Fr, H, W)
            self.s_lat[C:].copy_(y)
        if d.model_type == "vace":
            if vace_context is None:
                raise TypeError("magcache_b200: a VACE model needs vace_context (magcache_generate.py:439-449)")
            assert tuple(vace_context.shape) == (d.vace_in_dim, Fr, H, W), tuple(vace_context.shape)
            if self.s_vace is None or self.s_vace.shape != vace_context.shape:
                self.s_vace = torch.empty(vace_context.shape, dtype=torch.float32, device=self.device)
                self._graphs = {}
            self.s_vace.copy_(vace_context)
            self.vgate.fill_(float(vace_scale))
        if clip_fea is not None:
            assert tuple(clip_fea.shape[-2:]) == (d.clip_len, d.clip_dim) and clip_fea.numel() == d.clip_len * d.clip_dim, "one sample per call"
            self.clip_in.copy_(clip_fea.reshape(d.clip_len, d.clip_dim))
        self._stage_t(t)
        L = context.shape[0]
        assert L <= d.text_len and context.shape[1] == d.text_dim
        self.ctx_in.zero_()
        self.ctx_in[:L].copy_(context)

    def _stage_t(self, t):
        """One timestep (`t` with one element: Wan2.1, the Wan2.2 A14B experts) is copied device to device. A per-token `t`
        ([1, seq_len], MagCache4Wan2.2/magcache_generate.py:263-264 — TI2V-5B gives its first-frame tokens t = 0) is read back once
        (the only host synchronisation of a forward) and reduced to its distinct values and the contiguous row ranges that carry
        them: the time MLP then runs once per VALUE, and every op that consumes the modulation runs once per RANGE with that value's
        vectors — the same arithmetic per token as the reference's per-token embedding. Rows past the tokens (`seq_len` padding) are
        not computed, except the one representative pad row of a calibration call, which takes the first padded position's t."""
        if t.numel() == 1:
            self.s_t[:1].copy_(t.reshape(-1))
            self.t_values, self.runs, key = 1, None, None
        else:
            n_rows = self.n_keys + self.pad_row
            tv = t.detach().reshape(-1).to(torch.float64).cpu().numpy()
            if tv.shape[0] < n_rows:
                raise ValueError(f"magcache_b200: {tv.shape[0]} timesteps for {n_rows} token rows")
            if self.pad_row and np.any(tv[self.n_keys:] != tv[self.n_keys]):
                raise NotImplementedError("magcache_b200: the padded positions of a calibration call must share one timestep")
            tv = tv[:n_rows]
            cuts = np.flatnonzero(tv[1:] != tv[:-1]) + 1
            bounds = np.concatenate([[0], cuts, [n_rows]])
            values, runs = [], []
            for r0, r1 in zip(bounds[:-1].tolist(), bounds[1:].tolist()):
                v = float(tv[r0])
                if v not in values:
                    values.append(v)
                runs.append((r0, r1, values.index(v)))
            if len(values) == 1:
                self.s_t[:1].copy_(t.reshape(-1)[:1])
                self.t_values, self.runs, key = 1, None, None
            else:
                if len(values) > MAX_T_VALUES or len(runs) > MAX_T_RUNS:
                    raise NotImplementedError(f"magcache_b200: {len(values)} distinct timesteps in {len(runs)} token ranges "
                                              f"(built for <= {MAX_T_VALUES} values, <= {MAX_T_RUNS} ranges; TI2V-5B has 2 and 2)")
                self.s_t[:len(values)].copy_(torch.tensor(values, dtype=torch.float64))
                if self.shard is not None:  # this rank's rows of every range, in local coordinates
                    a, b = self.shard.start, self.shard.start + self.shard.n_local
                    runs = [(max(r0, a) - a, min(r1, b) - a, u) for r0, r1, u in runs if min(r1, b) > max(r0, a)]
                self.t_values, self.runs, key = len(values), runs, tuple(runs)
        if key != self._runs_key:
            self._runs_key, self._graphs = key, {}  # a captured forward bakes the ranges in

    def time_embedding(self):
        """`e = time_embedding(sinusoid(t))`, `e0 = time_projection(e)` (fp32 region, magcache_generate.py:249-254) from the staged t:
        e fp32 [1, D], e0 fp32 [6, D] ([U, D] and [U, 6, D] for U > 1 distinct per-token timesteps). Also what the TeaCache comparator
        measures between steps (wan_teacache.py:534)."""
        d, w, U = self.dims, self.w, self.t_values
        sin = ops.time_sinusoid(self.s_t[:U], d.freq_dim)
        e = ops.linear_f32_small(ops.linear_f32_small(sin, w.time_w1, w.time_b1, act=2), w.time_w2, w.time_b2, act=0)
        e0 = ops.linear_f32_small(e, w.tproj_w, w.tproj_b, act=1)
        return e, (e0.view(6, d.dim) if U == 1 else e0.view(U, 6, d.dim))

    def prologue(self, need_ctx=True):
        """Embeddings from the staged inputs. Returns (x0 bf16 [N_local, D], e fp32 [1, D], e0 fp32 [6, D], ctx bf16 [text_len, D]).
        `need_ctx=False` (cache hit): the text / image-token embeddings feed only the blocks, which a hit skips — the reference
        computes them anyway (:255-266); leaving them out changes no output."""
        d, w = self.dims, self.w
        tok = ops.patchify(self.s_lat)
        if self.shard is not None:
            tok = self.shard.rows(tok)  # this rank embeds only its own tokens
        ops.gemm(tok, w.patch_w, w.patch_b, E.MC_EPI_BIAS_BF16, out=self.x0[:tok.shape[0]])
        if self.pad_row:
            self.x0[tok.shape[0]:].zero_()  # `u.new_zeros(1, seq_len - u.size(1), u.size(2))` (:244-245)
        e, e0 = self.time_embedding()
        # the head's modulated weight depends on the time embedding only: prepared here, off the tail of the forward
        self._head_prep = {(u, g): ops.head_prepare(w.head_mod, e[u], wt, hb, slot=u * len(self.head_groups) + g)
                           for u in range(self.t_values) for g, (wt, hb) in enumerate(self.head_groups)}
        if not need_ctx:
            return self.x0, e, e0, None
        ops.gemm(self.ctx_in, w.text_w1, w.text_b1, E.MC_EPI_BIAS_GELU_BF16, out=self.ctx_h)
        ops.gemm(self.ctx_h, w.text_w2, w.text_b2, E.MC_EPI_BIAS_BF16, out=self.ctx)
        if d.model_type == "i2v":
            # context_clip = self.img_emb(clip_fea) (:264-266): LN(fp32) - Linear - GELU(erf) - Linear - LN(fp32). The block's k_img /
            # v_img Linears cast their input to bf16, so the last LN writes bf16 directly (same value as fp32 -> autocast cast).
            ops.ln_affine(self.clip_in, w.img_ln1_w, w.img_ln1_b, eps=w.img_ln1_eps, out=self.clip_h1)
            ops.gemm(self.clip_h1, w.img_w1, w.img_b1, E.MC_EPI_BIAS_GELU_ERF_BF16, out=self.clip_h2)
            ops.gemm(self.clip_h2, w.img_w2, w.img_b2, E.MC_EPI_BIAS_BF16, out=self.clip_h3)
            ops.ln_affine(self.clip_h3, w.img_ln2_w, w.img_ln2_b, eps=w.img_ln2_eps, out=self.ctx_img)
        return self.x0, e, e0, self.ctx

    # ------------------------------------------------------------------------------------------ one patched forward
    def _body(self, kind, slot, step=None):
        """prologue -> {hit: head(x0 + residual) | miss: block stack, residual = x - x0, head(x)} on the staged inputs."""
        self._slot = slot
        if self._native_ok(step):
            return self._native_body(kind, slot)
        x0, e, e0, ctx = self.prologue(need_ctx=(kind != "hit"))
        if kind == "hit":
            # `x + residual_x` (:295) is formed inside the head kernel; TeaCache's in-place bf16 `x += residual` rounds the sum first
            return self.head(x0, e, self.grid, residual=self.res[slot], round_sum_to_bf16=self.hit_sum_bf16, step=step)
        xs = self.run_blocks(x0, e0, ctx, self.grid)
        ops.residual_sub(xs, x0, out=self.res[slot])  # magcache_generate.py:299, written into the slot's fixed buffer
        return self.head(xs, e, self.grid, step=step)

    def _native_ok(self, step):
        if not self.native or self.shard is not None or self.runs is not None or self.pad_row or step is not None or self.hit_sum_bf16:
            return False
        from . import native
        return native.supported(self.dims) and getattr(ops, "PROFILE", None) is None

    def _native_body(self, kind, slot):
        """The same forward through `mc_dit_forward`: staged latent / timestep / text in, the slot's residual read (hit) or written (miss)."""
        from . import native
        if self._nat is None:
            self._nat = native.NativeWanForward(self.w)
        if self._nat_grid != self.grid:
            self._nat.bind(self.grid, self._rope_for(self.grid))
            self._nat_grid = self.grid
        skip = kind == "hit"
        out = self._nat.forward(self.s_lat, self.s_t, self.ctx_in, skip, self.res[slot])
        ops._count(self._nat.launches(skip))
        return out

    def arm_step(self, cond, x_latent, guide_scale, coef_x, coef_v, out=None):
        """Fold the caller loop's CFG combine + scheduler update (eval/.../wan_magcache.py:301-310) into the head pass of the NEXT
        forward, which must be the unconditional call of the step whose conditional prediction is `cond`: that forward then returns
        `coef_x * x_latent + coef_v * (uncond + guide_scale * (cond - uncond))` (written into `out`, which may be `x_latent` itself)
        instead of the unconditional prediction. One-shot: the next `forward` or `calibrate` takes it off the engine, whether it
        succeeds or not. Bit-equal to the plain forward followed by `ops.cfg_step`."""
        if self.shard is not None:
            raise NotImplementedError("magcache_b200: the fused step is built for the unsharded engine (sharded runs use ops.cfg_step)")
        if len(self.head_groups) != 1:
            raise NotImplementedError("magcache_b200: the fused step is built for 16 output channels (use ops.cfg_step)")
        self._step = (cond, x_latent, float(guide_scale), float(coef_x), float(coef_v), out)

    def forward(self, kind, slot):
        """Run (or replay) one forward of the given kind for CFG slot `slot`; returns a fresh fp32 [C, F, H, W] tensor."""
        step, self._step = self._step, None
        if kind == "hit" and not self.res_valid[slot]:
            raise TypeError("magcache_b200: cache hit with an empty residual_cache slot (reference: Tensor + NoneType)")
        if not self.use_graphs or step is not None:  # an armed step carries per-step scalars: never captured
            out = self._body(kind, slot, step)
        else:
            key = (kind, slot, self.hit_sum_bf16)
            st = self._graphs.get(key)
            if st is None:  # first use: eager (sets kernel attributes, sizes the allocator pools)
                out = self._body(kind, slot)
                self._graphs[key] = "warm"
            else:
                if st == "warm":
                    prof, ops.PROFILE = ops.PROFILE, None  # event records are not capturable
                    n0 = ops.LAUNCHES
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        gout = self._body(kind, slot)
                    ops.PROFILE = prof
                    st = self._graphs[key] = (g, gout, ops.LAUNCHES - n0)
                    ops.LAUNCHES = n0
                g, gout, n_launch = st
                g.replay()
                ops._count(n_launch)
                out = gout.clone()  # callers keep outputs across calls (cond is alive while uncond runs)
        if kind == "miss":
            self.res_valid[slot] = True
        return out

    def calibrate(self, slot, prev):
        """The calibration twin of `forward("miss", slot)` (MagCache4Wan2.1/magcache_generate.py:80-194): always runs the block stack.
        `prev`: the previous fp32 residual of this CFG branch (N x D elements, any shape) or None. Returns (head output, residual,
        (norm_ratio, norm_std, cos_dis) against `prev` or None). The residual is a new fp32 [N, D] tensor on every call: `prev` may
        alias an earlier one, so nothing is written into the engine's residual slots."""
        step, self._step = self._step, None
        self._slot = slot
        x0, e, e0, ctx = self.prologue()
        xs = self.run_blocks(x0, e0, ctx, self.grid)
        if prev is None:
            residual, stats = ops.residual_sub(xs, x0), None
        elif self.pad_row:
            # seq_len > token count: rows [n_tok, seq_len) of the reference's tensors are identical copies of the one pad row computed
            # here; its three per-row terms enter the means n_pad times (:167-169 average over dim 1 of [1, seq_len, D])
            prev, n, wgt, keep = prev.view(x0.shape), self.n_keys, float(self.n_pad), {}
            ops.residual_sub_stats(xs[n:], x0[n:], prev[n:].contiguous(), reduce=lambda st: keep.setdefault("pad", st.clone()))
            residual_tok, stats = ops.residual_sub_stats(
                xs[:n], x0[:n], prev[:n].contiguous(), reduce=lambda st: st + keep["pad"] * st.new_tensor([wgt, wgt, wgt, wgt]))
            residual = torch.cat([residual_tok, xs[n:] - x0[n:].float()])
        else:
            reduce = None
            if self.shard is not None:  # the statistics are sums over tokens: add the partial sums of every token shard
                from .shard import allreduce_stats
                reduce = lambda st: allreduce_stats(st, self.shard.group)  # noqa: E731
            residual, stats = ops.residual_sub_stats(xs, x0, prev.view(x0.shape), reduce=reduce)
        return self.head(xs, e, self.grid, step=step), residual, stats

    # ------------------------------------------------------------------------------------------ block stack (:297-298)
    def run_blocks(self, x0, e0, ctx, grid):
        """30 (1.3B) / 40 (14B) WanAttentionBlocks (VACE models: the control-stream pass first, then the main blocks with their
        hints). Returns the fp32 residual stream [N, D] (engine-owned buffer)."""
        d = self.dims
        rope = self._rope_for(grid)
        if self.shard is not None:
            rope = self.shard.rows(rope)  # RoPE uses the GLOBAL token index -> (f, h, w)
        if d.model_type == "vace":
            self._vace_pass(x0, e0, ctx, rope)
        xs = self.xs
        ops.cast_into(x0, xs)  # block 0 sees the bf16 patch embedding; every later op works on the fp32 stream
        for li, b in enumerate(self.w.blocks):
            self._block(b, xs, e0, ctx, rope, first=(li == 0))
            if li in d.vace_layers:
                # BaseWanAttentionBlock: x = x + hints[j] * context_scale, hints[j] = after_proj(c_j). The projection runs HERE, its
                # epilogue adding bf16(acc + bias) * scale straight into the fp32 stream (no hint tensors, no separate add pass).
                j = d.vace_layers.index(li)
                vb = self.w.vace_blocks[j]
                ops.gemm(self.cbf[j], vb["w_after"], vb["b_after"], E.MC_EPI_BIAS_GATE_RESID, out=xs, gate=self.vgate, tag="gemm_vace_after")
        return xs

    def _vace_pass(self, x0, e0, ctx, rope):
        """`forward_vace` (upstream VaceWanModel, called at magcache_generate.py:541): patch-embed the control video, mix it with the
        main stream's input in the first control block (`c = before_proj(c) + x`), run the control blocks and keep a bf16 copy of the
        stream after each one (what `after_proj` — a Linear under autocast — reads)."""
        w = self.w
        tok = ops.patchify(self.s_vace)
        if self.shard is not None:
            tok = self.shard.rows(tok)
        ops.gemm(tok, w.vace_patch_w, w.vace_patch_b, E.MC_EPI_BIAS_BF16, out=self.att)
        vb0 = w.vace_blocks[0]
        ops.gemm(self.att, vb0["w_before"], vb0["b_before"], E.MC_EPI_BIAS_BF16, out=self.cq)
        ops.cache_hit_add(self.cq, x0, out=self.h)  # bf16 + bf16 -> bf16
        ops.cast_into(self.h, self.cs)
        for j, vb in enumerate(w.vace_blocks):
            self._block(vb, self.cs, e0, ctx, rope, first=(j == 0))
            ops.cast_into(self.cs, self.cbf[j])

    def _block(self, b, xs, e0, ctx, rope, first):
        """One WanAttentionBlock on the fp32 stream `xs` (updated in place). `first`: the stream still holds bf16 values (block 0
        input), so the LayerNorm output is rounded to bf16 before the modulation like upstream's `.type_as(x)`."""
        d, H = self.dims, self.dims.num_heads
        D = d.dim
        n = xs.shape[0]
        sh = self.shard
        self._modulation(b["mod"], e0)  # e = modulation + e0 (fp32)
        # --- self attention
        self._ln_modulate(xs, 1, 0, first)
        if sh is None:
            q, k, v = self.qkv[:, :D], self.qkv[:, D:2 * D], self.qkv[:, 2 * D:]
            ops.gemm(self.h, b["w_qkv"], b["b_qkv"], E.MC_EPI_BIAS_BF16, out=self.qkv, tag="gemm_qkv")
            ops.rmsnorm_rope_segs_(self.qkv, b["nqk"], 2, rope, d.head_dim, eps=d.eps)  # q and k column blocks, one launch
            ops.attention(q, k[:self.n_keys], v[:self.n_keys], H, out=self.att, tag="attn_self")  # keys = the tokens (`k_lens`), never the pad row
        else:
            # k | v first: their rows start travelling to the other ranks (copy engines, side stream) while this rank projects q;
            # the attention kernel then begins on the local keys and picks the peers' segments up as they land
            xi = self._xi
            self._xi ^= 1
            kv_own = self.xch.own_rows(xi)
            ops.gemm(self.h, b["w_qkv"][D:], b["b_qkv"][D:], E.MC_EPI_BIAS_BF16, out=kv_own, tag="gemm_qkv")
            ops.rmsnorm_rope_(kv_own[:, :D], b["nqk"][1], rope, d.head_dim, eps=d.eps)
            self.xch.begin(xi)
            ops.gemm(self.h, b["w_qkv"][:D], b["b_qkv"][:D], E.MC_EPI_BIAS_BF16, out=self.q_loc, tag="gemm_qkv")
            ops.rmsnorm_rope_(self.q_loc, b["nqk"][0], rope, d.head_dim, eps=d.eps)
            kv_all, kw = self.xch.keys_values(xi)
            ops.attention(self.q_loc, kv_all[:, :D], kv_all[:, D:], H, out=self.att, tag="attn_self", **kw)
        self._gemm_gated(self.att, b["w_o"], b["b_o"], xs, 2, "gemm_o")
        # --- cross attention (text)
        ops.ln_affine(xs, b["n3_w"], b["n3_b"], eps=d.eps, out=self.h)
        ops.gemm(self.h, b["c_wq"], b["c_bq"], E.MC_EPI_BIAS_BF16, out=self.cq, tag="gemm_cq")
        ops.rmsnorm_rope_(self.cq, b["c_nq"], None, d.head_dim, eps=d.eps)
        ops.gemm(ctx, b["c_wkv"], b["c_bkv"], E.MC_EPI_BIAS_BF16, out=self.ckv, tag="gemm_ckv")
        ops.rmsnorm_rope_(self.ckv[:, :D], b["c_nk"], None, d.head_dim, eps=d.eps)
        ops.attention(self.cq, self.ckv[:, :D], self.ckv[:, D:], H, out=self.att, tag="attn_cross")
        att = self.att
        if d.model_type == "i2v":  # WanI2VCrossAttention: x = attn(q, k, v) + attn(q, k_img, v_img), summed in bf16
            ops.gemm(self.ctx_img, b["c_wkv_img"], b["c_bkv_img"], E.MC_EPI_BIAS_BF16, out=self.ckv_img)
            ops.rmsnorm_rope_(self.ckv_img[:, :D], b["c_nk_img"], None, d.head_dim, eps=d.eps)
            ops.attention(self.cq, self.ckv_img[:, :D], self.ckv_img[:, D:], H, out=self.att_img, tag="attn_cross_img")
            att = ops.cache_hit_add(self.att, self.att_img, out=self.h)  # h (norm3 output) is dead once cq is projected
        ops.gemm(att, b["c_wo"], b["c_bo"], E.MC_EPI_BIAS_GATE_RESID, out=xs, gate=None, tag="gemm_co")
        # --- FFN
        self._ln_modulate(xs, 4, 3, False)
        ops.gemm(self.h, b["w_f1"], b["b_f1"], E.MC_EPI_BIAS_GELU_BF16, out=self.ffn, tag="gemm_ffn1")
        self._gemm_gated(self.ffn, b["w_f2"], b["b_f2"], xs, 5, "gemm_ffn2")

    # The three places a block consumes the time modulation. With one timestep they are single launches over all rows; with per-token
    # timesteps (`self.runs`) each runs once per contiguous row range, on row slices of the same buffers, with that range's vectors.
    def _modulation(self, mod, e0):
        if self.runs is None:
            return ops.cache_hit_add(mod, e0, out=self.em[0])
        for u in range(self.t_values):
            ops.cache_hit_add(mod, e0[u], out=self.em[u])
        return self.em

    def _ln_modulate(self, xs, scale_idx, shift_idx, first):
        eps = self.dims.eps
        if self.runs is None:
            ops.ln_modulate(xs, self.em[0], scale_idx, shift_idx, eps=eps, round_ln_to_bf16=first, out=self.h)
            return
        for r0, r1, u in self.runs:
            ops.ln_modulate(xs[r0:r1], self.em[u], scale_idx, shift_idx, eps=eps, round_ln_to_bf16=first, out=self.h[r0:r1])

    def _gemm_gated(self, a, w, bias, xs, gate_idx, tag):
        """xs += (a @ w.T + bias) * gate (the gated residual adds of the block), gate = row `gate_idx` of modulation + e0."""
        if self.runs is None:
            ops.gemm(a, w, bias, E.MC_EPI_BIAS_GATE_RESID, out=xs, gate=self.em[0][gate_idx], tag=tag)
            return
        for r0, r1, u in self.runs:
            ops.gemm(a[r0:r1], w, bias, E.MC_EPI_BIAS_GATE_RESID, out=xs[r0:r1], gate=self.em[u][gate_idx], tag=tag)

    # ------------------------------------------------------------------------------------------ epilogue (:304-305)
    def head(self, x, e, grid, residual=None, round_sum_to_bf16=False, step=None):
        """head + unpatchify of the stream `x` (or of x0 + `residual` on a hit). `step`: the `arm_step` tuple of the forward in flight,
        applied in the epilogue."""
        w, G = self.w, len(self.head_groups)
        tag = "head_hit_fused" if residual is not None else "head"
        kw = dict(c_out=16, eps=self.dims.eps, tag=tag, round_sum_to_bf16=round_sum_to_bf16)
        row_offset, out, peer_outs = 0, None, None
        if self.shard is None:
            if self.pad_row:  # unpatchify reads the token rows only (`u[:math.prod(v)]`)
                x = x[:self.n_keys]
                if residual is not None:
                    residual = residual[:self.n_keys]
        else:
            self.xch.join()  # every push of this forward is ordered before its end (and inside a captured graph)
            out, peer_outs = self.xch.head_output(self._slot)
            row_offset = self.shard.start
        if self.runs is None and G == 1:  # one timestep, 16 output channels: a single launch
            (wt, hb), = self.head_groups
            if self.shard is None and step is not None:
                kw["step"], out = step[:5], step[5]
            out = ops.head_unpatchify(x, w.head_mod, e, wt, hb, grid, residual=residual, row_offset=row_offset, out=out, peer_outs=peer_outs,
                                      prep=self._head_prep[(0, 0)], **kw)
        else:
            # per-token timesteps and / or more than 16 output channels: one launch per (row range, channel group), each writing
            # its own rows x channels of the same output tensor
            if step is not None:
                raise NotImplementedError("magcache_b200: the fused step is built for one timestep and 16 output channels (use ops.cfg_step)")
            n_rows = x.shape[0]
            if out is None:
                out = torch.empty(self.dims.out_dim, grid[0], 2 * grid[1], 2 * grid[2], dtype=torch.float32, device=x.device)
            group_bytes = 16 * out[0].numel() * 4
            for r0, r1, u in (self.runs if self.runs is not None else [(0, n_rows, 0)]):
                r1 = min(r1, n_rows)  # a calibration call's pad row is not unpatchified
                if r1 <= r0:
                    continue
                for g, (wt, hb) in enumerate(self.head_groups):
                    ops.head_unpatchify(x[r0:r1], w.head_mod, e[u], wt, hb, grid, residual=None if residual is None else residual[r0:r1],
                                        row_offset=row_offset + r0, out=out[16 * g:16 * g + 16],
                                        peer_outs=None if peer_outs is None else [int(p) + g * group_bytes for p in peer_outs],
                                        prep=self._head_prep[(u, g)], **kw)
        if self.shard is None:
            return out
        return self.xch.finish_head(out, self._slot)  # every rank ends up with the full noise prediction


class WanModelHandle:
    """Minimal stand-in for `wan.modules.model.WanModel` when the weights do not come from an nn.Module (bench.py, tests):
    carries the engine and receives the reference's class attributes (`cnt`, `mag_ratios`, ...) through `init_magcache`.
    Each handle is its own class so two pipelines in one process do not share controller state (SURVEY §5, race note)."""

    model_type = "t2v"

    def __new__(cls, weights: WanWeights, **engine_kw):
        sub = type("WanModelHandle", (cls,), {})
        self = object.__new__(sub)
        return self

    def __init__(self, weights: WanWeights, **engine_kw):
        self.dim, self.num_heads = weights.dims.dim, weights.dims.num_heads
        self._mc_engine = WanEngine(weights, **engine_kw)

    def __call__(self, *args, **kwargs):
        return self.forward(*args, **kwargs)
