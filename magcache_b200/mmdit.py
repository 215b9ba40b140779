"""MMDiT engines (SURVEY §8f rank 4): the transformers behind `magcache_forward` of MagCache4FLUX/magcache_flux.py:234-440 (FLUX.1,
FLUX.1-Kontext) and of MagCache4HunyuanVideo/magcache_sample_video.py:29-160 (HunyuanVideo) on the same sm_100a kernels as the Wan path — tcgen05 GEMMs (fused bias / GELU / SiLU / bf16 gated-residual epilogues), the tcgen05 flash
attention over the joint text+image sequence, LN+modulate, per-head RMSNorm + RoPE, the K1/K2 cache kernels.

Block arithmetic follows diffusers' `FluxTransformerBlock` / `FluxSingleTransformerBlock` and hyvideo's `MMDoubleStreamBlock` /
`MMSingleStreamBlock` / `SingleTokenRefiner` [EXT, not in the reference tree] as restated in oracle/flux_ref.py and oracle/hunyuan_ref.py;
the forwards' own statements (embedders, controller, hit / miss, residual, final layer, counter) are the reference's (file:line cited in
`magcache_flux_forward` / `magcache_hunyuan_forward`, magcache_b200/patch.py). The two families share one block-stack implementation
(`MMDiTCore`): same modulation chunk order, same per-head q/k RMSNorm, same `cat(attn, act(mlp))` single block; they differ in the
token order of the joint sequence, in which rows get RoPE, and in their embedders.

STATUS: parity-green on a B200 against the oracles at reduced depth / token counts (tests/test_flux_forward_gpu.py,
tests/test_hunyuan_forward_gpu.py) and pinned on CPU through the kernel emulation (tests/test_*_engine_emulated_cpu.py); run and timed at
full size with synthetic weights by `bench.py --workload flux|hunyuan720p` (profiles/r02_bench_flux_1024.json,
profiles/r02_bench_hunyuan_720p.json, and token-sharded over 2 GPUs profiles/r02_bench_hunyuan_720p_2gpu.json). Nothing on the Wan path
depends on this module.

HBM layout (S = n_txt + n_img tokens; FLUX puts the text rows FIRST — `torch.cat([encoder_hidden_states, hidden_states], dim=1)`,
magcache_flux.py:384 — HunyuanVideo the image rows — `torch.cat((img, txt), 1)`, magcache_sample_video.py:123; D = heads*128;
everything bf16 like the reference pipelines, which run without autocast):
  hs   [S, D]    both residual streams; the double-stream blocks work on the two row ranges, the single-stream blocks on all rows
  x0   [n_img, D] x_embedder output (`ori_hidden_states`)         res [n_img, D]  cached residual (`previous_residual`)
  h    [S, D]    LN+modulate output (GEMM A operand)              qk  [S, 2D]     q | k projections, per-head RMSNorm + RoPE in place
  v    [S, D]    row-major V (attention reads it as is)          cat [S, 5D]     single blocks: attention output | GELU(proj_mlp);
                                                                                  double blocks borrow cat[:, D:] as the FF hidden
  ada  [R]       ALL AdaLayerNorm projections of the forward from ONE GEMM over silu(temb) (they depend on temb only)
"""
import numpy as np
import torch

from . import _lib, ops
from .wan import _bf16, _bias_autocast

E = _lib


def _mlp2(lin1, lin2, dev):
    """(w1, b1, w2, b2) of a two-Linear embedder MLP."""
    return _bf16(lin1.weight, dev), _bias_autocast(lin1.bias, dev), _bf16(lin2.weight, dev), _bias_autocast(lin2.bias, dev)


class _AdaStack:
    """The Linear projections of a forward's AdaLayerNorm / ModulateDiT layers stacked into one matrix (they all read the same
    conditioning vector: one GEMM computes them). `add` returns a projection's first row in the stack."""

    def __init__(self):
        self.ws, self.bs, self.rows = [], [], 0

    def add(self, lin):
        self.ws.append(lin.weight.detach())
        self.bs.append(lin.bias.detach())
        start, self.rows = self.rows, self.rows + lin.weight.shape[0]
        return start

    def pack(self, dev):
        """(weight bf16, bias fp32, rows) of the stack."""
        return _bf16(torch.cat(self.ws, 0), dev), _bias_autocast(torch.cat(self.bs, 0), dev), self.rows


class FluxWeights:
    """Weights of one FluxTransformer2DModel (diffusers attribute names), repacked: q|k weights concatenated, every AdaLayerNorm
    projection stacked into one matrix, biases / norm weights as fp32 copies of their bf16 values."""

    def __init__(self):
        self.double, self.single = [], []

    @classmethod
    def from_module(cls, m, dev):
        cfg = m.config
        w = cls()
        w.heads, w.head_dim = cfg.num_attention_heads, cfg.attention_head_dim
        if w.head_dim != 128 or tuple(cfg.axes_dims_rope) != (16, 56, 56):
            raise NotImplementedError("FLUX engine: head_dim 128 with RoPE axes (16, 56, 56)")
        w.dim = D = w.heads * w.head_dim
        w.in_channels, w.joint_dim, w.pooled_dim = cfg.in_channels, cfg.joint_attention_dim, cfg.pooled_projection_dim
        w.guidance = bool(cfg.guidance_embeds)
        w.x_w, w.x_b = _bf16(m.x_embedder.weight, dev), _bias_autocast(m.x_embedder.bias, dev)
        w.ctx_w, w.ctx_b = _bf16(m.context_embedder.weight, dev), _bias_autocast(m.context_embedder.bias, dev)
        tte = m.time_text_embed
        w.t_mlp = _mlp2(tte.timestep_embedder.linear_1, tte.timestep_embedder.linear_2, dev)
        w.p_mlp = _mlp2(tte.text_embedder.linear_1, tte.text_embedder.linear_2, dev)
        w.g_mlp = _mlp2(tte.guidance_embedder.linear_1, tte.guidance_embedder.linear_2, dev) if w.guidance else None
        ada = _AdaStack()
        for blk in m.transformer_blocks:
            a = blk.attn
            w.double.append({
                "ada": ada.add(blk.norm1.linear), "ada_c": ada.add(blk.norm1_context.linear),
                "qk_w": _bf16(torch.cat([a.to_q.weight, a.to_k.weight], 0), dev),
                "qk_b": _bias_autocast(torch.cat([a.to_q.bias, a.to_k.bias], 0), dev),
                "v_w": _bf16(a.to_v.weight, dev), "v_b": _bias_autocast(a.to_v.bias, dev),
                "o_w": _bf16(a.to_out[0].weight, dev), "o_b": _bias_autocast(a.to_out[0].bias, dev),
                "nq": _bias_autocast(a.norm_q.weight, dev), "nk": _bias_autocast(a.norm_k.weight, dev),
                "cqk_w": _bf16(torch.cat([a.add_q_proj.weight, a.add_k_proj.weight], 0), dev),
                "cqk_b": _bias_autocast(torch.cat([a.add_q_proj.bias, a.add_k_proj.bias], 0), dev),
                "cv_w": _bf16(a.add_v_proj.weight, dev), "cv_b": _bias_autocast(a.add_v_proj.bias, dev),
                "co_w": _bf16(a.to_add_out.weight, dev), "co_b": _bias_autocast(a.to_add_out.bias, dev),
                "cnq": _bias_autocast(a.norm_added_q.weight, dev), "cnk": _bias_autocast(a.norm_added_k.weight, dev),
                "ff1_w": _bf16(blk.ff.net[0].proj.weight, dev), "ff1_b": _bias_autocast(blk.ff.net[0].proj.bias, dev),
                "ff2_w": _bf16(blk.ff.net[2].weight, dev), "ff2_b": _bias_autocast(blk.ff.net[2].bias, dev),
                "cff1_w": _bf16(blk.ff_context.net[0].proj.weight, dev), "cff1_b": _bias_autocast(blk.ff_context.net[0].proj.bias, dev),
                "cff2_w": _bf16(blk.ff_context.net[2].weight, dev), "cff2_b": _bias_autocast(blk.ff_context.net[2].bias, dev),
            })
        for blk in m.single_transformer_blocks:
            a = blk.attn
            w.single.append({
                "ada": ada.add(blk.norm.linear),
                "qk_w": _bf16(torch.cat([a.to_q.weight, a.to_k.weight], 0), dev),
                "qk_b": _bias_autocast(torch.cat([a.to_q.bias, a.to_k.bias], 0), dev),
                "v_w": _bf16(a.to_v.weight, dev), "v_b": _bias_autocast(a.to_v.bias, dev),
                "nq": _bias_autocast(a.norm_q.weight, dev), "nk": _bias_autocast(a.norm_k.weight, dev),
                "mlp_w": _bf16(blk.proj_mlp.weight, dev), "mlp_b": _bias_autocast(blk.proj_mlp.bias, dev),
                "out_w": _bf16(blk.proj_out.weight, dev), "out_b": _bias_autocast(blk.proj_out.bias, dev),
            })
        w.ada_out = ada.add(m.norm_out.linear)
        w.ada_w, w.ada_b, w.ada_rows = ada.pack(dev)
        w.out_w, w.out_b = _bf16(m.proj_out.weight, dev), _bias_autocast(m.proj_out.bias, dev)
        w.device = dev
        return w


def rope_table(ids, device, axes_dim=(16, 56, 56), theta=10000.0):
    """cos / sin of `FluxPosEmbed` (float64 angles, fp32 values) for ids [S, 3], stored [S, 128] as interleaved (cos, sin) pairs."""
    pos = ids.detach().double().cpu().numpy()
    ang = [np.outer(pos[:, i], 1.0 / theta ** (np.arange(0, d, 2, dtype=np.float64) / d)) for i, d in enumerate(axes_dim)]
    ang = np.concatenate(ang, axis=1)  # [S, 64]
    cs = np.stack([np.cos(ang), np.sin(ang)], axis=-1).reshape(len(pos), 2 * ang.shape[1])
    return torch.tensor(cs.astype(np.float32)).to(device)  # torch-allocated (aligned) storage on every device


class MMDiTCore:
    """Workspace + block stack shared by the FLUX and HunyuanVideo engines, on the family's packed weights (dim, heads, double,
    single, ada_w / ada_b / ada_rows). A subclass provides the token order (`txt_first`), the RoPE table of the rows that get RoPE,
    and its own prologue / head."""

    txt_first = True

    def __init__(self, weights, shard_world=1, shard_rank=0, shard_group=None):
        self.w, self.device = weights, weights.device
        self.world, self.rank, self.group = shard_world, shard_rank, shard_group
        self._shape = None
        self._rope_key, self._rope = None, None
        self.res_valid = False

    def _alloc_core(self, n_img, n_txt):
        """Buffers for one (image tokens, text tokens) shape. Token-sharded (`self.world > 1`, SURVEY §8e): the IMAGE rows are split over
        the ranks, the (few) text rows are replicated — every rank carries all of them and computes the identical text stream. Per
        attention the K|V rows of a rank's image tokens travel through the same exchange as the Wan engine's (`shard.make_exchange`:
        copy-engine pushes into every peer's gathered buffer, consumed segment by segment inside the attention kernel; or the
        all-gather formulation), and the text K|V rows are written locally behind the image rows of the gathered buffer — the key
        order [image | text] differs from the unsharded engine's, which a softmax over keys cannot see."""
        D, dev = self.w.dim, self.device
        bf = dict(dtype=torch.bfloat16, device=dev)
        self.n_img_total, self.n_txt = n_img, n_txt
        self.shard = None
        if self.world > 1:
            from .shard import TokenShard
            self.shard = TokenShard(self.rank, self.world, n_img, self.group)
            if self.shard.pad:
                raise NotImplementedError(f"magcache_b200: {n_img} image tokens over {self.world} ranks needs the pad rule, built for the Wan engines only")
            n_img = self.shard.n_local
        S = n_img + n_txt                      # rows this rank carries
        Sg = self.n_img_total + n_txt          # keys every query attends to
        self.n_img, self.S, self.S_keys = n_img, S, Sg
        if self.txt_first:
            self.txt, self.img = slice(0, n_txt), slice(n_txt, S)
            self.txt_g, self.img_g = slice(0, n_txt), slice(n_txt, Sg)
        else:
            self.img, self.txt = slice(0, n_img), slice(n_img, S)
            self.img_g, self.txt_g = slice(0, self.n_img_total), slice(self.n_img_total, Sg)
        self.hs, self.h, self.att = torch.empty(S, D, **bf), torch.empty(S, D, **bf), torch.empty(S, D, **bf)
        self.x0, self.res, self.hit = torch.empty(n_img, D, **bf), torch.empty(n_img, D, **bf), torch.empty(n_img, D, **bf)
        if self.shard is None:
            self.qk = torch.empty(S, 2 * D, **bf)
            self.v = torch.empty(S, D, **bf)   # row-major V: the attention kernel consumes it as is (MN-major B operand)
        else:
            from .shard import make_exchange
            self.q_loc, self.k_loc = torch.empty(S, D, **bf), torch.empty(S, D, **bf)  # k_loc: the text refiner's own (local) keys
            self.xch = make_exchange(self.shard, 2 * D, (1,), dev, extra_rows=n_txt)
            self._xi, self._kv_cur = 0, None
        self.cat = torch.empty(S, 5 * D, **bf)
        self.ada = torch.empty(1, self.w.ada_rows, **bf)
        self.adaf = torch.empty(self.w.ada_rows, dtype=torch.float32, device=dev)
        self.res_valid = False

    def _em(self, start, k):
        D = self.w.dim
        return self.adaf[start:start + k * D].view(k, D)

    def _modulation_table(self, vec):
        """Every `Linear(silu(vec))` of the block stack (AdaLayerNormZero / ModulateDiT / final layer) from ONE GEMM: they depend on the
        conditioning vector only. bf16 like the reference, then an exact fp32 copy for the kernels that read modulation / gates."""
        w = self.w
        ops.gemm(ops.silu(vec), w.ada_w, w.ada_b, E.MC_EPI_BIAS_BF16, out=self.ada)
        ops.cast_into(self.ada.view(-1), self.adaf)

    def _rope_for(self, rows):
        """RoPE table rows for a token range, or None when that range gets no RoPE (HunyuanVideo text tokens)."""
        raise NotImplementedError

    # ------------------------------------------------------------------------------------------ attention over the joint sequence
    def _project(self, rows, h_rows, qk_w, qk_b, v_w, v_b):
        """q | k and V projections of the token range `rows` from its LN+modulate output."""
        D = self.w.dim
        if self.shard is not None:
            # K | V straight into the exchange's gathered buffer: image rows into this rank's segment (pushed to the peers by
            # `_joint_attention`), text rows into the local tail; q stays local
            own, tail = self._kv_views()
            ops.gemm(h_rows, qk_w[:D], qk_b[:D], E.MC_EPI_BIAS_BF16, out=self.q_loc[rows])
            if rows == self.img:
                parts = ((h_rows, own),)
            elif rows == self.txt:
                parts = ((h_rows, tail),)
            else:  # the whole local sequence (single-stream blocks)
                parts = ((h_rows[self.img], own), (h_rows[self.txt], tail))
            for hp, dst in parts:
                ops.gemm(hp, qk_w[D:], qk_b[D:], E.MC_EPI_BIAS_BF16, out=dst[:, :D])
                ops.gemm(hp, v_w, v_b, E.MC_EPI_BIAS_BF16, out=dst[:, D:])
            return
        ops.gemm(h_rows, qk_w, qk_b, E.MC_EPI_BIAS_BF16, out=self.qk[rows])
        ops.gemm(h_rows, v_w, v_b, E.MC_EPI_BIAS_BF16, out=self.v[rows])

    def _qk_norm(self, rows, nq, nk):
        """Per-head RMSNorm of q and k (+ RoPE where the family applies it), in place."""
        D, H = self.w.dim, self.w.heads
        rope = self._rope_for(rows)
        if self.shard is not None:
            own, tail = self._kv_views()
            q, k = self.q_loc[rows], (own if rows == self.img else tail)[:, :D]
        else:
            q, k = self.qk[rows][:, :D], self.qk[rows][:, D:]
        ops.rmsnorm_head_rope_(q, nq, H, rope)
        ops.rmsnorm_head_rope_(k, nk, H, rope)

    def _kv_views(self):
        """(this rank's image segment, the local text tail) of the gathered K|V buffer the NEXT joint attention reads, [rows, 2 D]."""
        if self._kv_cur is None:
            self._kv_cur = (self.xch.own_rows(self._xi), self.xch.tail_rows(self._xi))
        return self._kv_cur

    def _joint_attention(self, out):
        D, H = self.w.dim, self.w.heads
        if self.shard is not None:
            xi = self._xi
            self.xch.begin(xi)  # this rank's normalised image K|V rows start travelling to the peers
            kv_all, kw = self.xch.keys_values(xi)
            ops.attention(self.q_loc, kv_all[:, :D], kv_all[:, D:], H, out=out, tag="mmdit_attn", **kw)
            self._xi, self._kv_cur = xi ^ 1, None
            return
        ops.attention(self.qk[:, :D], self.qk[:, D:], self.v, H, out=out, tag="mmdit_attn")

    def _gather_output(self, o_local):
        """Per-token head output of this rank's image rows -> all image rows, replicated (tiny: 64 features per token)."""
        if self.shard is None:
            return o_local
        from .shard import gather_rows
        full = torch.empty(self.n_img_total, o_local.shape[1], dtype=o_local.dtype, device=o_local.device)
        gather_rows(o_local.contiguous(), full, self.shard.group)
        return full

    def run_blocks(self):
        """Double-stream then single-stream blocks (magcache_flux.py:343-424; magcache_sample_video.py:108-139) on `hs`; the image rows of
        `hs` must hold the embedded image tokens and the text rows the embedded text. Returns the image rows."""
        w, D, S = self.w, self.w.dim, self.S
        txt, img = self.txt, self.img
        hs, h = self.hs, self.h
        for b in w.double:
            em, emc = self._em(b["ada"], 6), self._em(b["ada_c"], 6)  # (shift1, scale1, gate1, shift2, scale2, gate2)
            ops.ln_modulate(hs[img], em, 1, 0, round_ln_to_bf16=True, out=h[img])
            ops.ln_modulate(hs[txt], emc, 1, 0, round_ln_to_bf16=True, out=h[txt])
            self._project(img, h[img], b["qk_w"], b["qk_b"], b["v_w"], b["v_b"])
            self._project(txt, h[txt], b["cqk_w"], b["cqk_b"], b["cv_w"], b["cv_b"])
            self._qk_norm(img, b["nq"], b["nk"])
            self._qk_norm(txt, b["cnq"], b["cnk"])
            self._joint_attention(self.att)
            ops.gemm(self.att[img], b["o_w"], b["o_b"], E.MC_EPI_BIAS_GATE_RESID_BF16, out=hs[img], gate=em[2])
            ops.gemm(self.att[txt], b["co_w"], b["co_b"], E.MC_EPI_BIAS_GATE_RESID_BF16, out=hs[txt], gate=emc[2])
            for rows, e, f1w, f1b, f2w, f2b in ((img, em, b["ff1_w"], b["ff1_b"], b["ff2_w"], b["ff2_b"]),
                                                (txt, emc, b["cff1_w"], b["cff1_b"], b["cff2_w"], b["cff2_b"])):
                ops.ln_modulate(hs[rows], e, 4, 3, round_ln_to_bf16=True, out=h[rows])
                ffh = self.cat[rows][:, D:]
                ops.gemm(h[rows], f1w, f1b, E.MC_EPI_BIAS_GELU_BF16, out=ffh)
                ops.gemm(ffh, f2w, f2b, E.MC_EPI_BIAS_GATE_RESID_BF16, out=hs[rows], gate=e[5])
        allr = slice(0, S)
        for b in w.single:
            em = self._em(b["ada"], 3)  # (shift, scale, gate)
            ops.ln_modulate(hs, em, 1, 0, round_ln_to_bf16=True, out=h)
            ops.gemm(h, b["mlp_w"], b["mlp_b"], E.MC_EPI_BIAS_GELU_BF16, out=self.cat[:, D:])
            self._project(allr, h, b["qk_w"], b["qk_b"], b["v_w"], b["v_b"])
            self._qk_norm(img, b["nq"], b["nk"])
            self._qk_norm(txt, b["nq"], b["nk"])
            self._joint_attention(self.cat[:, :D])
            ops.gemm(self.cat, b["out_w"], b["out_b"], E.MC_EPI_BIAS_GATE_RESID_BF16, out=hs, gate=em[2])
        return hs[img]

    def _time_mlp(self, x_bf16, mlp):
        w1, b1, w2, b2 = mlp
        return ops.gemm(ops.gemm(x_bf16, w1, b1, E.MC_EPI_BIAS_SILU_BF16), w2, b2, E.MC_EPI_BIAS_BF16)

    def _sinusoid(self, t64):
        """256-channel [cos | sin] timestep embedding of a float64 device scalar, rounded to bf16 (`.to(dtype=...)` in both families)."""
        f = ops.time_sinusoid(t64, 256)
        return ops.cast_into(f, torch.empty(1, 256, dtype=torch.bfloat16, device=self.device))

    def forward(self, kind):
        """prologue -> {hit: x0 + cached residual | miss: block stack, residual = x - x0} -> family head."""
        x0 = self.prologue()
        if kind == "hit":
            if not self.res_valid:
                raise TypeError("magcache_b200: cache hit with an empty residual cache (reference: Tensor + NoneType)")
            x = ops.cache_hit_add(x0, self.res, out=self.hit)                     # magcache_flux.py:340 ; magcache_sample_video.py:104
        else:
            self.hs[self.img].copy_(x0)                                           # `ori_hidden_states` / `ori_img` stays in x0
            x = self.run_blocks()
            if self.shard is not None:
                self.xch.join()  # every push of this forward is ordered before its end
            ops.residual_sub(x.contiguous(), x0, out=self.res)                    # :426 ; :140 (x is a contiguous row range of hs)
            self.res_valid = True
        return self.head(x)


    def calibrate(self):
        """The calibration twin of `forward("miss")` (magcache_flux.py:21-231; magcache_sample_video.py:163-290): always runs the block
        stack; returns (head output, (norm_ratio, norm_std, cos_dis) against the previous residual or None on the first call). The
        statistics come from the fused fp32/fp64 reduction kernel — finer than the reference's bf16 tensor ops, which quantise them to
        multiples of 2^-8 (the shipped FLUX table is visibly bf16-quantised, SURVEY §8a row 9)."""
        x0 = self.prologue()
        self.hs[self.img].copy_(x0)
        x = self.run_blocks()
        reduce = None
        if self.shard is not None:  # the statistics are sums over the image tokens: add the partial sums of every token shard
            from .shard import allreduce_stats
            self.xch.join()
            reduce = lambda st: allreduce_stats(st, self.shard.group)  # noqa: E731
        new = self.hit
        ops.residual_sub(x.contiguous(), x0, out=new)
        stats = ops.residual_stats(new, self.res, reduce=reduce) if self.res_valid else None
        self.res, self.hit = new, self.res
        self.res_valid = True
        return self.head(x), stats


class FluxEngine(MMDiTCore):
    txt_first = True

    def _workspace(self, n_img, n_txt):
        if self._shape == (n_img, n_txt):
            return
        bf = dict(dtype=torch.bfloat16, device=self.device)
        self._alloc_core(n_img, n_txt)
        self.s_hidden = torch.empty(self.n_img, self.w.in_channels, **bf)  # this rank's image tokens
        self.s_enc = torch.empty(n_txt, self.w.joint_dim, **bf)
        self.s_pooled = torch.empty(1, self.w.pooled_dim, **bf)
        self.s_t = torch.zeros(2, dtype=torch.float64, device=self.device)  # timestep*1000, guidance*1000 (already rounded like the reference)
        self._shape = (n_img, n_txt)

    def _rope_for(self, rows):
        if self.shard is None:
            return self._rope[rows]
        if rows == self.txt:
            return self._rope[self.txt_g]
        if rows == self.img:  # this rank's image rows sit at their GLOBAL positions in the table (text rows first)
            return self._rope[self.n_txt + self.shard.start:self.n_txt + self.shard.stop]
        return torch.cat([self._rope[self.txt_g], self._rope[self.n_txt + self.shard.start:self.n_txt + self.shard.stop]])

    # ------------------------------------------------------------------------------------------ inputs (:290-319)
    def stage_inputs(self, hidden_states, encoder_hidden_states, pooled, timestep, guidance, img_ids, txt_ids):
        w = self.w
        assert hidden_states.shape[0] == 1 and encoder_hidden_states.shape[0] == 1, "one sample per call"
        n_img, n_txt = hidden_states.shape[1], encoder_hidden_states.shape[1]
        self._workspace(n_img, n_txt)
        self.s_hidden.copy_(hidden_states[0] if self.shard is None else self.shard.rows(hidden_states[0]))
        self.s_enc.copy_(encoder_hidden_states[0])
        self.s_pooled.copy_(pooled.reshape(1, -1))
        if (w.guidance and guidance is None) or (not w.guidance and guidance is not None):
            raise ValueError("guidance must be given exactly when the model has guidance_embeds")
        # `timestep.to(hidden_states.dtype) * 1000` (:292-294): both the cast and the product round to bf16
        tv = (timestep.reshape(-1)[:1].to(torch.bfloat16) * 1000).double()
        gv = (guidance.reshape(-1)[:1].to(torch.bfloat16) * 1000).double() if guidance is not None else torch.zeros(1, dtype=torch.float64, device=tv.device)
        self.s_t.copy_(torch.cat([tv, gv.to(tv.device)]))
        key = (img_ids.data_ptr(), txt_ids.data_ptr(), n_img, n_txt)
        if self._rope_key != key:  # ids are constant over a generation
            self._rope = rope_table(torch.cat((txt_ids.reshape(-1, 3), img_ids.reshape(-1, 3)), dim=0), self.device)  # :318
            self._rope_key = key
            assert self._rope.shape == (self.S_keys, 128)

    def prologue(self):
        """x_embedder, time_text_embed, context_embedder (:290-303) and every AdaLayerNorm projection of the forward."""
        w = self.w
        ops.gemm(self.s_hidden, w.x_w, w.x_b, E.MC_EPI_BIAS_BF16, out=self.x0)
        temb = self._time_mlp(self._sinusoid(self.s_t[0:1]), w.t_mlp)
        if w.guidance:
            temb = ops.cache_hit_add(temb, self._time_mlp(self._sinusoid(self.s_t[1:2]), w.g_mlp))
        temb = ops.cache_hit_add(temb, self._time_mlp(self.s_pooled, w.p_mlp))
        self._modulation_table(temb)
        ops.gemm(self.s_enc, w.ctx_w, w.ctx_b, E.MC_EPI_BIAS_BF16, out=self.hs[self.txt])
        return self.x0

    def head(self, x_img):
        """`norm_out(hidden_states, temb)`, `proj_out` (:429-430): AdaLayerNormContinuous chunks (scale, shift) in that order."""
        w = self.w
        em = self._em(w.ada_out, 2)
        ops.ln_modulate(x_img, em, 0, 1, round_ln_to_bf16=True, out=self.h[self.img])
        return self._gather_output(ops.gemm(self.h[self.img], w.out_w, w.out_b, E.MC_EPI_BIAS_BF16))


# ======================================================================================================================
# HunyuanVideo
# ======================================================================================================================
class HunyuanWeights:
    """Weights of one HYVideoDiffusionTransformer (hyvideo attribute names), repacked like FluxWeights: fused qkv / linear1 matrices
    split into q|k, v (and mlp) row blocks, every ModulateDiT / final adaLN projection stacked into one matrix."""

    def __init__(self):
        self.double, self.single, self.refiner = [], [], []

    @classmethod
    def from_module(cls, m, dev):
        w = cls()
        w.dim = D = m.hidden_size
        w.heads = m.heads_num
        if D // w.heads != 128:
            raise NotImplementedError("HunyuanVideo engine: head_dim 128")
        if list(m.patch_size) != [1, 2, 2] or m.text_projection != "single_refiner":
            raise NotImplementedError("HunyuanVideo engine: patch (1, 2, 2) and the single_refiner text projection")
        w.in_channels, w.out_channels, w.guidance = m.in_channels, m.out_channels, bool(m.guidance_embed)
        w.patch_w, w.patch_b = _bf16(m.img_in.proj.weight.flatten(1), dev), _bias_autocast(m.img_in.proj.bias, dev)
        w.t_mlp = _mlp2(m.time_in.mlp[0], m.time_in.mlp[2], dev)
        w.p_mlp = _mlp2(m.vector_in.in_layer, m.vector_in.out_layer, dev)
        w.g_mlp = _mlp2(m.guidance_in.mlp[0], m.guidance_in.mlp[2], dev) if w.guidance else None
        w.pooled_dim = m.vector_in.in_layer.in_features
        r = m.txt_in
        w.text_dim = r.input_embedder.in_features
        w.r_in_w, w.r_in_b = _bf16(r.input_embedder.weight, dev), _bias_autocast(r.input_embedder.bias, dev)
        w.r_t_mlp = _mlp2(r.t_embedder.mlp[0], r.t_embedder.mlp[2], dev)
        w.r_c_mlp = _mlp2(r.c_embedder.linear_1, r.c_embedder.linear_2, dev)
        r_ada = _AdaStack()
        for blk in r.individual_token_refiner.blocks:
            W = blk.self_attn_qkv.weight
            Bq = blk.self_attn_qkv.bias
            r_ada.add(blk.adaLN_modulation[1])
            w.refiner.append({
                "n1_w": _bias_autocast(blk.norm1.weight, dev), "n1_b": _bias_autocast(blk.norm1.bias, dev),
                "n2_w": _bias_autocast(blk.norm2.weight, dev), "n2_b": _bias_autocast(blk.norm2.bias, dev),
                "qk_w": _bf16(W[:2 * D], dev), "qk_b": _bias_autocast(Bq[:2 * D], dev),
                "v_w": _bf16(W[2 * D:], dev), "v_b": _bias_autocast(Bq[2 * D:], dev),
                "nq": _bias_autocast(blk.self_attn_q_norm.weight, dev), "nk": _bias_autocast(blk.self_attn_k_norm.weight, dev),
                "o_w": _bf16(blk.self_attn_proj.weight, dev), "o_b": _bias_autocast(blk.self_attn_proj.bias, dev),
                "f1_w": _bf16(blk.mlp.fc1.weight, dev), "f1_b": _bias_autocast(blk.mlp.fc1.bias, dev),
                "f2_w": _bf16(blk.mlp.fc2.weight, dev), "f2_b": _bias_autocast(blk.mlp.fc2.bias, dev),
            })
        w.r_ada_w, w.r_ada_b, _ = r_ada.pack(dev)
        ada = _AdaStack()
        for blk in m.double_blocks:
            d = {"ada": ada.add(blk.img_mod.linear), "ada_c": ada.add(blk.txt_mod.linear)}
            for pre, key in (("img", ""), ("txt", "c")):
                W, Bq = getattr(blk, f"{pre}_attn_qkv").weight, getattr(blk, f"{pre}_attn_qkv").bias
                proj, mlp = getattr(blk, f"{pre}_attn_proj"), getattr(blk, f"{pre}_mlp")
                d.update({f"{key}qk_w": _bf16(W[:2 * D], dev), f"{key}qk_b": _bias_autocast(Bq[:2 * D], dev),
                          f"{key}v_w": _bf16(W[2 * D:], dev), f"{key}v_b": _bias_autocast(Bq[2 * D:], dev),
                          f"{key}nq": _bias_autocast(getattr(blk, f"{pre}_attn_q_norm").weight, dev),
                          f"{key}nk": _bias_autocast(getattr(blk, f"{pre}_attn_k_norm").weight, dev),
                          f"{key}o_w": _bf16(proj.weight, dev), f"{key}o_b": _bias_autocast(proj.bias, dev),
                          f"{key}ff1_w": _bf16(mlp.fc1.weight, dev), f"{key}ff1_b": _bias_autocast(mlp.fc1.bias, dev),
                          f"{key}ff2_w": _bf16(mlp.fc2.weight, dev), f"{key}ff2_b": _bias_autocast(mlp.fc2.bias, dev)})
            w.double.append(d)
        for blk in m.single_blocks:
            W, Bq = blk.linear1.weight, blk.linear1.bias
            w.single.append({
                "ada": ada.add(blk.modulation.linear),
                "qk_w": _bf16(W[:2 * D], dev), "qk_b": _bias_autocast(Bq[:2 * D], dev),
                "v_w": _bf16(W[2 * D:3 * D], dev), "v_b": _bias_autocast(Bq[2 * D:3 * D], dev),
                "mlp_w": _bf16(W[3 * D:], dev), "mlp_b": _bias_autocast(Bq[3 * D:], dev),
                "nq": _bias_autocast(blk.q_norm.weight, dev), "nk": _bias_autocast(blk.k_norm.weight, dev),
                "out_w": _bf16(blk.linear2.weight, dev), "out_b": _bias_autocast(blk.linear2.bias, dev),
            })
        w.ada_out = ada.add(m.final_layer.adaLN_modulation[1])
        w.ada_w, w.ada_b, w.ada_rows = ada.pack(dev)
        w.out_w, w.out_b = _bf16(m.final_layer.linear.weight, dev), _bias_autocast(m.final_layer.linear.bias, dev)
        w.device = dev
        return w


class HunyuanEngine(MMDiTCore):
    """Image tokens first, RoPE on the image tokens only, text tokens through the two-block token refiner. The padded text tokens form
    their own attention segment in the reference (`get_cu_seqlens`, magcache_sample_video.py:82) and never reach an image token, so only
    the valid ones are embedded and carried."""

    txt_first = False

    def __init__(self, weights: HunyuanWeights, **shard_kw):
        super().__init__(weights, **shard_kw)
        self._mask_key, self._valid = None, None

    def _workspace(self, grid, n_txt):
        n_img = grid[0] * grid[1] * grid[2]
        if self._shape == (grid, n_txt):
            return
        w, dev = self.w, self.device
        bf = dict(dtype=torch.bfloat16, device=dev)
        self._alloc_core(n_img, n_txt)
        self.grid = grid
        self.s_lat = torch.empty(w.in_channels, grid[0], 2 * grid[1], 2 * grid[2], dtype=torch.float32, device=dev)
        self.s_txt = torch.empty(n_txt, w.text_dim, **bf)
        self.s_pooled = torch.empty(1, w.pooled_dim, **bf)
        self.s_t = torch.zeros(2, dtype=torch.float64, device=dev)
        self.rv = torch.empty(n_txt, w.dim, **bf)  # V of the token refiner's self-attention
        self.rada = torch.empty(1, w.r_ada_w.shape[0], **bf)
        self.radaf = torch.empty(w.r_ada_w.shape[0], dtype=torch.float32, device=dev)
        self._shape = (grid, n_txt)

    def _rope_for(self, rows):
        if rows != self.img or self._rope is None:
            return None  # the text tokens get no RoPE (magcache_sample_video.py:108-120 -> hyvideo blocks)
        return self._rope if self.shard is None else self._rope[self.shard.start:self.shard.stop]

    # ------------------------------------------------------------------------------------------ inputs (:42-86)
    def stage_inputs(self, x, t, text_states, text_mask, text_states_2, freqs_cos, freqs_sin, guidance):
        w = self.w
        assert x.shape[0] == 1 and text_states.shape[0] == 1, "one sample per call"
        _, c, ot, oh, ow = x.shape
        grid = (ot, oh // 2, ow // 2)
        mkey = (text_mask.data_ptr(), tuple(text_mask.shape))
        if self._mask_key != mkey:  # the mask is constant over a generation: one host read
            m = text_mask.reshape(-1).to(torch.int64).cpu()
            valid = int(m.sum())
            if valid < 1 or not bool((m[:valid] == 1).all()):
                raise NotImplementedError("magcache_b200: the valid text tokens must be a non-empty prefix of text_states (right padding)")
            self._mask_key, self._valid = mkey, valid
        n_txt = self._valid
        self._workspace(grid, n_txt)
        self.s_lat.copy_(x[0])
        self.s_txt.copy_(text_states[0, :n_txt])
        self.s_pooled.copy_(text_states_2.reshape(1, -1))
        if w.guidance and guidance is None:
            raise ValueError("Didn't get guidance strength for guidance distilled model.")  # :58-61
        gv = guidance.reshape(-1)[:1].double() if guidance is not None else torch.zeros(1, dtype=torch.float64, device=t.device)
        self.s_t.copy_(torch.cat([t.reshape(-1)[:1].double(), gv.to(t.device)]))
        if freqs_cos is not None:
            key = (freqs_cos.data_ptr(), freqs_sin.data_ptr(), self.n_img_total)
            if self._rope_key != key:
                n = self.n_img_total
                assert tuple(freqs_cos.shape) == (n, 128) and tuple(freqs_sin.shape) == (n, 128)
                cs = torch.stack([freqs_cos.float()[:, 0::2], freqs_sin.float()[:, 0::2]], dim=-1).reshape(n, 128)
                self._rope, self._rope_key = cs.contiguous().to(self.device), key
        else:
            self._rope = None

    # ------------------------------------------------------------------------------------------ token refiner (`self.txt_in`, :69)
    def _refine_text(self):
        """SingleTokenRefiner over the valid text tokens: c = t_embedder(t) + c_embedder(mean of the raw states); two blocks of
        LN(affine) -> qkv -> per-head RMSNorm -> self-attention -> gated proj, LN(affine) -> SiLU MLP -> gated; in place on hs[txt]."""
        w, D, H = self.w, self.w.dim, self.w.heads
        txt, n = self.txt, self.n_txt
        c = ops.cache_hit_add(self._time_mlp(self._sinusoid(self.s_t[0:1]), w.r_t_mlp), self._time_mlp(ops.colmean(self.s_txt), w.r_c_mlp))
        ops.gemm(ops.silu(c), w.r_ada_w, w.r_ada_b, E.MC_EPI_BIAS_BF16, out=self.rada)
        ops.cast_into(self.rada.view(-1), self.radaf)
        x, h = self.hs[txt], self.h[txt]
        ops.gemm(self.s_txt, w.r_in_w, w.r_in_b, E.MC_EPI_BIAS_BF16, out=x)
        sharded = self.shard is not None
        q, k = (self.q_loc[txt], self.k_loc[txt]) if sharded else (self.qk[txt][:, :D], self.qk[txt][:, D:])
        rv = self.rv[:n]
        for i, b in enumerate(w.refiner):
            g = self.radaf[i * 2 * D:(i + 1) * 2 * D].view(2, D)  # gate_msa, gate_mlp
            ops.ln_affine(x, b["n1_w"], b["n1_b"], eps=1e-6, out=h)
            if sharded:
                ops.gemm(h, b["qk_w"][:D], b["qk_b"][:D], E.MC_EPI_BIAS_BF16, out=q)
                ops.gemm(h, b["qk_w"][D:], b["qk_b"][D:], E.MC_EPI_BIAS_BF16, out=k)
            else:
                ops.gemm(h, b["qk_w"], b["qk_b"], E.MC_EPI_BIAS_BF16, out=self.qk[txt])
            ops.gemm(h, b["v_w"], b["v_b"], E.MC_EPI_BIAS_BF16, out=rv)
            ops.rmsnorm_head_rope_(q, b["nq"], H, None)
            ops.rmsnorm_head_rope_(k, b["nk"], H, None)
            ops.attention(q, k, rv, H, out=self.att[txt], tag="refiner_attn")
            ops.gemm(self.att[txt], b["o_w"], b["o_b"], E.MC_EPI_BIAS_GATE_RESID_BF16, out=x, gate=g[0])
            ops.ln_affine(x, b["n2_w"], b["n2_b"], eps=1e-6, out=h)
            ffh = self.cat[txt][:, D:]
            ops.gemm(h, b["f1_w"], b["f1_b"], E.MC_EPI_BIAS_SILU_BF16, out=ffh)
            ops.gemm(ffh, b["f2_w"], b["f2_b"], E.MC_EPI_BIAS_GATE_RESID_BF16, out=x, gate=g[1])

    def prologue(self):
        """time_in + vector_in (+ guidance_in), img_in, txt_in (:52-69) and the modulation table of the whole block stack."""
        w = self.w
        vec = ops.cache_hit_add(self._time_mlp(self._sinusoid(self.s_t[0:1]), w.t_mlp), self._time_mlp(self.s_pooled, w.p_mlp))
        if w.guidance:
            vec = ops.cache_hit_add(vec, self._time_mlp(self._sinusoid(self.s_t[1:2]), w.g_mlp))
        tok = ops.patchify(self.s_lat)
        ops.gemm(tok if self.shard is None else self.shard.rows(tok), w.patch_w, w.patch_b, E.MC_EPI_BIAS_BF16, out=self.x0)
        self._refine_text()
        self._modulation_table(vec)
        return self.x0

    def head(self, x_img):
        """`final_layer(img, vec)` (shift, scale in that order) and `unpatchify` (:144-146): [1, C, T, H, W] bf16."""
        w = self.w
        em = self._em(w.ada_out, 2)
        ops.ln_modulate(x_img, em, 1, 0, round_ln_to_bf16=True, out=self.h[self.img])
        o = self._gather_output(ops.gemm(self.h[self.img], w.out_w, w.out_b, E.MC_EPI_BIAS_BF16))  # [n_img, C*1*2*2], (c, pt, ph, pw)
        t, hh, ww = self.grid
        c = w.out_channels
        o = o.view(1, t, hh, ww, c, 1, 2, 2)
        return torch.einsum("nthwcopq->nctohpwq", o).reshape(1, c, t, 2 * hh, 2 * ww)  # pure data movement


# ======================================================================================================================
# Synthetic weights created directly on the device (benchmarks: a FLUX.1-dev / HunyuanVideo-sized nn.Module does not fit a CPU box)
# ======================================================================================================================
def _rand_block_weights(D, dev, g, keys_prefix=("", "c")):
    import math

    def xav(o, i, s=1.0):
        return ((torch.rand(o, i, device=dev, generator=g) * 2 - 1) * (s * math.sqrt(6.0 / (i + o)))).bfloat16()

    def bias(n):
        return (0.02 * torch.randn(n, device=dev, generator=g)).bfloat16().float()

    def nw():
        return (1 + 0.1 * torch.randn(128, device=dev, generator=g)).bfloat16().float()

    d = {}
    for k in keys_prefix:
        d.update({f"{k}qk_w": xav(2 * D, D), f"{k}qk_b": bias(2 * D), f"{k}v_w": xav(D, D), f"{k}v_b": bias(D), f"{k}o_w": xav(D, D), f"{k}o_b": bias(D),
                  f"{k}nq": nw(), f"{k}nk": nw(), f"{k}ff1_w": xav(4 * D, D), f"{k}ff1_b": bias(4 * D), f"{k}ff2_w": xav(D, 4 * D), f"{k}ff2_b": bias(D)})
    return d, xav, bias, nw


def _random_stack(w, D, n_double, n_single, dev, g):
    """Double / single block weights + the stacked modulation matrix (rows: 12D per double block, 3D per single block, 2D final)."""
    off = 0
    for _ in range(n_double):
        d, xav, bias, nw = _rand_block_weights(D, dev, g)
        d["ada"], d["ada_c"] = off, off + 6 * D
        off += 12 * D
        w.double.append(d)
    for _ in range(n_single):
        _, xav, bias, nw = _rand_block_weights(D, dev, g, keys_prefix=())
        w.single.append({"ada": off, "qk_w": xav(2 * D, D), "qk_b": bias(2 * D), "v_w": xav(D, D), "v_b": bias(D), "nq": nw(), "nk": nw(),
                         "mlp_w": xav(4 * D, D), "mlp_b": bias(4 * D), "out_w": xav(D, 5 * D), "out_b": bias(D)})
        off += 3 * D
    w.ada_out = off
    off += 2 * D
    _, xav, bias, nw = _rand_block_weights(D, dev, g, keys_prefix=())
    w.ada_w, w.ada_b, w.ada_rows = xav(off, D, 0.3), bias(off), off
    return xav, bias, nw


def random_flux_weights(dev, heads=24, num_layers=19, num_single_layers=38, in_channels=64, joint_dim=4096, pooled_dim=768, guidance=True, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    w = FluxWeights()
    w.heads, w.head_dim, w.dim = heads, 128, heads * 128
    D = w.dim
    w.in_channels, w.joint_dim, w.pooled_dim, w.guidance, w.device = in_channels, joint_dim, pooled_dim, guidance, dev
    xav, bias, _ = _random_stack(w, D, num_layers, num_single_layers, dev, g)
    w.x_w, w.x_b, w.ctx_w, w.ctx_b = xav(D, in_channels), bias(D), xav(D, joint_dim), bias(D)
    w.t_mlp = (xav(D, 256), bias(D), xav(D, D), bias(D))
    w.p_mlp = (xav(D, pooled_dim), bias(D), xav(D, D), bias(D))
    w.g_mlp = (xav(D, 256), bias(D), xav(D, D), bias(D)) if guidance else None
    w.out_w, w.out_b = xav(in_channels, D), bias(in_channels)
    return w


def random_hunyuan_weights(dev, heads=24, double_depth=20, single_depth=40, in_channels=16, text_dim=4096, pooled_dim=768, guidance=True, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    w = HunyuanWeights()
    w.heads, w.dim = heads, heads * 128
    D = w.dim
    w.in_channels, w.out_channels, w.guidance, w.text_dim, w.pooled_dim, w.device = in_channels, in_channels, guidance, text_dim, pooled_dim, dev
    xav, bias, nw = _random_stack(w, D, double_depth, single_depth, dev, g)
    w.patch_w, w.patch_b = xav(D, in_channels * 4), bias(D)
    w.t_mlp = (xav(D, 256), bias(D), xav(D, D), bias(D))
    w.p_mlp = (xav(D, pooled_dim), bias(D), xav(D, D), bias(D))
    w.g_mlp = (xav(D, 256), bias(D), xav(D, D), bias(D)) if guidance else None
    w.r_in_w, w.r_in_b = xav(D, text_dim), bias(D)
    w.r_t_mlp = (xav(D, 256), bias(D), xav(D, D), bias(D))
    w.r_c_mlp = (xav(D, text_dim), bias(D), xav(D, D), bias(D))
    for _ in range(2):
        w.refiner.append({"n1_w": nw().new_ones(D) + 0.1 * torch.randn(D, device=dev, generator=g), "n1_b": bias(D),
                          "n2_w": nw().new_ones(D) + 0.1 * torch.randn(D, device=dev, generator=g), "n2_b": bias(D),
                          "qk_w": xav(2 * D, D), "qk_b": bias(2 * D), "v_w": xav(D, D), "v_b": bias(D), "nq": nw(), "nk": nw(),
                          "o_w": xav(D, D), "o_b": bias(D), "f1_w": xav(4 * D, D), "f1_b": bias(4 * D), "f2_w": xav(D, 4 * D), "f2_b": bias(D)})
    w.r_ada_w, w.r_ada_b = xav(4 * D, D, 0.3), bias(4 * D)
    w.out_w, w.out_b = xav(in_channels * 4, D), bias(in_channels * 4)
    return w


class MMDiTHandle:
    """Stand-in for the pipeline's transformer object when the weights do not come from an nn.Module (benchmarks): carries the engine
    and receives the reference's class attributes through `init_magcache_flux` / `init_magcache_hunyuan`."""

    def __new__(cls, engine):
        sub = type("MMDiTHandle", (cls,), {})
        return object.__new__(sub)

    def __init__(self, engine):
        key = "_mc_flux_engine" if isinstance(engine, FluxEngine) else "_mc_hunyuan_engine"
        object.__setattr__(self, key, engine)

    def __call__(self, *a, **k):
        return self.forward(*a, **k)
