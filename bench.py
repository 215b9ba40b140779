#!/usr/bin/env python
"""bench.py — denoising steps/sec of the MagCache hot path on Wan2.1-T2V-1.3B, 832x480x81 frames (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-cache] [--dump-outputs DIR]

One "step" = one denoising step = the cond + uncond pair of patched-forward calls the reference's caller makes
(eval/magcache/experiments/Wan2.1_EVAL/wan_magcache.py:296-299) under the E012K4R02 schedule
(thresh 0.12, K 4, retention 0.2: MagCache4Wan2.1/README.md:13), 50-step video => 42 block-stack forwards + 58 cache hits.
The K timed steps walk that schedule from cnt = 0 (warm-up steps are extra, then the controller is reset), so the default
K = 50 times exactly one video. Synthetic latents / text embeddings / seeded random weights of the named architecture
(no checkpoints offline). Prints ONE JSON line (see the task contract): value = steps/sec with inputs resident in HBM,
e2e = the same through the public `model(x, t, context, seq_len)` call with host tensors (H2D + D2H inside the timed region),
roofline = the dominant kernel (self-attention) from CUDA events recorded live around each of its launches,
cpu_baseline = the CPU oracle timed on this box's host cores on a bounded sample.

`--impl reference` times the reference's own path on the host CPU: the reference is pure Python/torch whose model code
(`wan`) is not installable offline, so the arm runs the oracle restatement (oracle/wan_ref.py, "port") with all host threads.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GRID = (21, 30, 52)          # latent 16 x 21 x 60 x 104  -> 32760 tokens
LATENT = (16, 21, 60, 104)
SAMPLE_STEPS = 50
PRESET = dict(thresh=0.12, K=4, retention_ratio=0.2)
N_TOK = GRID[0] * GRID[1] * GRID[2]
D, FFN, HEADS, LAYERS, TEXT_LEN, TEXT_DIM = 1536, 8960, 12, 30, 512, 4096
ATTN_SELF_FLOPS = 4.0 * N_TOK * N_TOK * D  # QK^T + PV, 2 flop per MAC (SURVEY §8d: 6.594 TF per layer)
LAYER_FLOPS = 9.433e12                     # SURVEY §8d
FWD_FLOPS = 283.0e12
WORKLOAD = "Wan2.1-T2V-1.3B 832x480x81f"
MODEL_KEY, TABLE = "t2v-1.3B", "wan2.1_t2v_1.3b"


def select_workload(name):
    """Default = BASELINE configs[1]. `wan14b` = configs[4]'s model and resolution (Wan2.1-T2V-14B, 1280x720x81f, E024K6R02):
    not what the driver times, kept to show the 14B shapes run at full size (one GPU holds it: 28 GB of bf16 weights)."""
    global GRID, LATENT, PRESET, N_TOK, D, FFN, HEADS, LAYERS, ATTN_SELF_FLOPS, FWD_FLOPS, WORKLOAD, MODEL_KEY, TABLE
    if name == "wan14b":
        GRID, LATENT = (21, 45, 80), (16, 21, 90, 160)
        PRESET = dict(thresh=0.24, K=6, retention_ratio=0.2)
        N_TOK = GRID[0] * GRID[1] * GRID[2]
        D, FFN, HEADS, LAYERS = 5120, 13824, 40, 40
        ATTN_SELF_FLOPS = 4.0 * N_TOK * N_TOK * D
        FWD_FLOPS = 6523.0e12  # SURVEY §8d
        WORKLOAD, MODEL_KEY, TABLE = "Wan2.1-T2V-14B 1280x720x81f", "t2v-14B", "wan2.1_t2v_14b"


DUMP_BYTES_MAX = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the arrays the timed path returned in its last step, as <out_dir>/<name>.npy in float32. The inputs and
    weights are seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    host = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_BYTES_MAX, f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES_MAX}-byte budget"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        busy = [v for v in sm if mx and v > 0.3 * mx] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle "port" of the reference path) — bounded sample, extrapolated; states exactly what was timed
# ---------------------------------------------------------------------------------------------------------------------
def host_cores():
    """CPU threads this process may really use: affinity mask, clipped by the cgroup CPU quota when one is set."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(math.ceil(int(quota) / int(period)))))
    except Exception:  # noqa: BLE001
        pass
    return n


CPU_LAYERS = 2  # layers of the full-shape oracle model the CPU arm really runs (of LAYERS); the block stack is scaled by LAYERS / CPU_LAYERS


def cpu_model():
    """The oracle restatement of the reference path (oracle/wan_ref.py) at the FULL benchmarked shape — 32760 tokens x 1536,
    12 heads, ffn 8960, text 512 x 4096 — but CPU_LAYERS of the 30 blocks, with the reference's patched forward installed so a
    call is literally `model([latent], t=t, context=[ctx], seq_len=N)` (MagCache4Wan2.1/magcache_generate.py:198-312)."""
    import torch
    from oracle import wan_ref
    torch.manual_seed(0)
    m = wan_ref.WanModel(dim=D, ffn_dim=FFN, num_heads=HEADS, num_layers=CPU_LAYERS, text_dim=TEXT_DIM, text_len=TEXT_LEN).init_synthetic(0)
    cls = type("CpuRefWan", (m.__class__,), {})
    m.__class__ = cls
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(*LATENT, generator=g)
    ctx = torch.randn(TEXT_LEN, TEXT_DIM, generator=g)
    return m, lat, ctx, torch.tensor([500.0])


def cpu_cycle(state):
    """One bounded sample = the 4-call cycle (miss, miss, hit, hit) of the CPU_LAYERS-layer full-shape model. Returns seconds per
    (miss forward, hit forward), each the mean of the two calls of that kind."""
    import torch
    from oracle import wan_ref
    m, lat, ctx, t = state
    m.__dict__.pop("cnt", None)
    # calls 0, 1 miss (fill both CFG slots), calls 2, 3 hit: the window opens at cnt 2 and thresh 10 makes every eligible call a hit
    wan_ref.install_magcache(type(m), [1.0] * 2 + [0.97] * 6, 4, thresh=10.0, K=3, retention_ratio=0.25)
    ts, kinds = [], []
    with torch.no_grad():
        for _ in range(4):
            t0 = time.perf_counter()
            m([lat], t=t, context=[ctx], seq_len=N_TOK)
            ts.append(time.perf_counter() - t0)
            kinds.append(bool(m.last_skip))
    assert kinds == [False, False, True, True], kinds
    return 0.5 * (ts[0] + ts[1]), 0.5 * (ts[2] + ts[3])


def cpu_extrapolate(t_miss_small, t_hit):
    """Full-model times from the sample: a miss forward = prologue + head (what a hit forward costs, minus its add) + LAYERS blocks;
    the CPU_LAYERS measured blocks are scaled by LAYERS / CPU_LAYERS. Nothing else is scaled: token count, widths, text length,
    attention (full 32760 x 32760 per head) are the benchmarked ones."""
    t_blocks = max(t_miss_small - t_hit, 0.0) * (LAYERS / CPU_LAYERS)
    t_miss = t_hit + t_blocks
    sec_video = 42 * t_miss + 58 * t_hit
    return SAMPLE_STEPS / sec_video, sec_video, t_miss


def cpu_threads():
    import torch
    n = host_cores()
    torch.set_num_threads(n)
    return n


def cpu_sample_text(n_cycles, cores, t_miss_small, t_hit, t_miss, sec_video):
    return (f"{n_cycles} x [2 miss + 2 hit forwards] of the oracle port at the FULL shape ({N_TOK} tokens x {D}, {HEADS} heads, ffn {FFN}, "
            f"text {TEXT_LEN}x{TEXT_DIM}) with {CPU_LAYERS} of {LAYERS} blocks, torch-CPU bf16-autocast emulation, {cores} threads: "
            f"miss({CPU_LAYERS} blocks) {t_miss_small:.2f}s, hit {t_hit:.2f}s; only the block stack is scaled (x{LAYERS // CPU_LAYERS}): "
            f"miss forward {t_miss:.1f}s; video = 42 miss + 58 hit forwards (E012K4R02) = {sec_video:.0f}s")


def run_reference_arm(args, rank):
    if rank != 0:
        return
    state = cpu_model()
    cores = cpu_threads()
    if args.warmup > 0:
        cpu_cycle(state)
    tm, th = [], []
    for _ in range(args.steps):
        a, b = cpu_cycle(state)
        tm.append(a)
        th.append(b)
    t_miss_small, t_hit = statistics.median(tm), statistics.median(th)
    value, sec_video, t_miss = cpu_extrapolate(t_miss_small, t_hit)
    sample = cpu_sample_text(len(tm), cores, t_miss_small, t_hit, t_miss, sec_video)
    line = {"metric": "denoising_steps_per_sec", "value": value, "unit": "steps/s", "n_gpus": args.gpus, "gpus_used": 0, "steps": len(tm), "warmup": min(args.warmup, 1),
            "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "impl": "reference", "sec_per_video": sec_video,
            "config": {"workload": "Wan2.1-T2V-1.3B 832x480x81f, 50 steps, MagCache E012K4R02 (BASELINE configs[1])", "tokens": N_TOK,
                       "note": "reference = pure-Python/torch path; upstream `wan` not installable offline -> oracle restatement on host CPU; "
                               "one timed step here = one 4-forward sample cycle, value = 50 / (42 t_miss + 58 t_hit)"},
            "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
WARM_START_STEP = 8  # warm-up walks the schedule from this step: steps 8, 9 miss on both CFG slots, steps 10.. hit (E012K4R02)


def run_ours(args, rank, world):
    import torch
    import torch.distributed as dist

    import magcache_b200 as mc
    from magcache_b200 import ops

    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    weights = mc.WanWeights.random(mc.WAN_CONFIGS[MODEL_KEY], dev, seed=0)  # same seed on every rank: replicated weights
    # N > 1: ONE video, token axis sharded over the ranks (K/V exchange per layer), see magcache_b200/shard.py
    model = mc.WanModelHandle(weights, shard_world=world, shard_rank=rank) if world > 1 else mc.WanModelHandle(weights)
    thresh = 1e-9 if args.no_cache else PRESET["thresh"]  # --no-cache: the controller never skips (same code path, same shapes)
    mc.init_magcache(model, SAMPLE_STEPS, thresh=thresh, K=PRESET["K"], retention_ratio=PRESET["retention_ratio"], table=TABLE)

    g = torch.Generator().manual_seed(0)
    lat_h = torch.randn(*LATENT, generator=g).pin_memory()
    ctx_h = torch.randn(TEXT_LEN, TEXT_DIM, generator=torch.Generator().manual_seed(1)).bfloat16().pin_memory()
    ctxn_h = torch.randn(TEXT_LEN, TEXT_DIM, generator=torch.Generator().manual_seed(2)).bfloat16().pin_memory()
    out_h = torch.empty(2, *LATENT).pin_memory()
    lat_d, ctx_d, ctxn_d = lat_h.to(dev), ctx_h.to(dev), ctxn_h.to(dev)
    shift = 5.0
    s = torch.linspace(1.0, 1.0 / SAMPLE_STEPS, SAMPLE_STEPS)
    sig = torch.cat([shift * s / (1 + (shift - 1) * s), torch.zeros(1)])
    t_dev = [(sig[i:i + 1] * 1000.0).to(dev) for i in range(SAMPLE_STEPS)]
    guide = 5.0
    fwd_events = []  # (start, end) CUDA events around every patched-forward call of the current pass

    def fwd(x, t, c):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = model([x], t=t, context=[c], seq_len=N_TOK)[0]
        e1.record()
        fwd_events.append((e0, e1))
        return out

    def step_resident(i, x):
        t = t_dev[i % SAMPLE_STEPS]
        # caller-side code (wan_magcache.py:296-310): cond call, uncond call, CFG combine + an Euler flow step standing in for
        # FlowUniPC. One GPU: the combine and the update ride in the epilogue of the unconditional call's head kernel
        # (mc_head_unpatchify_step); token-sharded: one mc_cfg_step launch after the two calls.
        return mc.cfg_denoise_step(model, x, t, ctx_d, ctxn_d, N_TOK, guide, float(sig[(i % SAMPLE_STEPS) + 1] - sig[i % SAMPLE_STEPS]), forward=fwd)

    def step_e2e(i, x_unused):
        t = t_dev[i % SAMPLE_STEPS]
        x = lat_h.to(dev, non_blocking=True)
        c = ctx_h.to(dev, non_blocking=True)
        cond = fwd(x, t, c)
        out_h[0].copy_(cond, non_blocking=True)
        x2 = lat_h.to(dev, non_blocking=True)
        cn = ctxn_h.to(dev, non_blocking=True)
        uncond = fwd(x2, t, cn)
        out_h[1].copy_(uncond, non_blocking=True)
        return None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def set_step(i):
        """Restart the controller at denoising step i of a video (cnt = 2 i, accumulators cleared): for i inside the retention
        window (i < 10) this is exactly the state a video walked from step 0 has there."""
        mc.reset_magcache(model)
        model.cnt = 2 * i

    def timed(run_step, steps, profile_tags, warmup, start_step=0):
        # warm-up OUTSIDE the timed region: walks steps 8, 9, 10, ... so that with W >= 3 every (miss | hit) x CFG-slot forward has
        # run eagerly, and — when the engine replays CUDA graphs — has been captured and replayed once, before the clock starts
        x = lat_d.clone()
        if warmup > 0:
            set_step(WARM_START_STEP)
            for i in range(WARM_START_STEP, WARM_START_STEP + warmup):
                r = run_step(i, x)
                x = r if r is not None else x
        set_step(start_step)
        x = lat_d.clone()
        fwd_events.clear()
        ops.PROFILE = {} if profile_tags is not False else None
        ops.PROFILE_TAGS = profile_tags if profile_tags else None
        launches0 = ops.LAUNCHES
        sampler = ClockSampler(local)
        barrier()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(start_step, start_step + steps):
            r = run_step(i, x)
            x = r if r is not None else x
        e1.record()
        barrier()
        clocks = sampler.stop()
        ms = e0.elapsed_time(e1)
        prof, ops.PROFILE, ops.PROFILE_TAGS = ops.PROFILE, None, None
        per_fwd = [a.elapsed_time(b) for a, b in fwd_events]
        if world > 1:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        return ms, ops.LAUNCHES - launches0, clocks, prof, x, per_fwd

    eng = model._mc_engine
    graphs = eng.use_graphs
    live_tags = {"attn_self", "head", "head_hit_fused"}  # recorded live inside the timed region; the full attribution runs separately
    ms, launches, clocks, prof, x_final, per_fwd = timed(step_resident, args.steps, False if graphs else live_tags, args.warmup)
    assert torch.isfinite(x_final).all(), "non-finite latents after the timed steps"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"latent": x_final})
    ms_e2e, _, _, _, _, _ = timed(step_e2e, args.steps, False, args.warmup)
    roofline_source = "CUDA events around every launch inside the timed region"

    # skip schedule actually walked in the timed region
    from magcache_b200.controller import make_ctrl_config, schedule_mask
    cfgm = mc.MagCacheConfig("wan2.1", thresh, PRESET["K"], PRESET["retention_ratio"], SAMPLE_STEPS, table=TABLE)
    mask = schedule_mask(make_ctrl_config(cfgm.num_steps, cfgm.thresh, cfgm.K, cfgm.retention_ratio, cfgm.resolved_ratios(), **cfgm.ctrl_kwargs()), 2 * SAMPLE_STEPS)
    walked = [int(mask[c % (2 * SAMPLE_STEPS)]) for c in range(2 * args.steps)]
    n_hit, n_miss = sum(walked), len(walked) - sum(walked)
    n_hit_video, n_miss_video = int(sum(mask)), 2 * SAMPLE_STEPS - int(sum(mask))
    t_miss = statistics.mean([t for t, h in zip(per_fwd, walked) if not h]) if n_miss else None
    t_hit = statistics.mean([t for t, h in zip(per_fwd, walked) if h]) if n_hit else None
    t_glue = max(ms - sum(per_fwd), 0.0) / args.steps  # per step: the CFG + sampler kernel and host gaps between the two forwards

    # ---- attribution pass (eager, every launch recorded under its tag): 2 steps of the window where the schedule has both kinds
    use_graphs_saved = eng.use_graphs
    eng.use_graphs = False
    attr_steps = 2 if not args.no_cache else 1
    ms_attr, _, _, prof_all, _, per_fwd_attr = timed(step_resident, attr_steps, None, 1 if graphs else 0, start_step=9 if not args.no_cache else 0)
    eng.use_graphs = use_graphs_saved
    if graphs:
        prof = prof_all
        roofline_source = "eager pass of 2 steps with CUDA events around every launch (the timed region replays CUDA graphs)"

    pk = peaks()
    kern = {}
    for tag, evs in (prof or {}).items():
        ts = [a.elapsed_time(b) for a, b in evs]
        kern[tag] = {"launches": len(ts), "ms_avg": sum(ts) / len(ts), "ms_total": sum(ts)}
    attribution = None
    if prof_all:
        tot = {tag: sum(a.elapsed_time(b) for a, b in evs) for tag, evs in prof_all.items()}
        fwd_total = sum(per_fwd_attr)
        attribution = {"steps": attr_steps, "forward_ms_total": fwd_total, "tagged_ms_total": sum(v for k2, v in tot.items() if k2 != "cfg_step"),
                       "share_of_forward_time": {k2: v / fwd_total for k2, v in sorted(tot.items(), key=lambda kv: -kv[1]) if k2 != "cfg_step"}}
        attribution["attributed_frac"] = attribution["tagged_ms_total"] / fwd_total
    roof = None
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_attn_traffic.json")
    if world == 1 and MODEL_KEY == "t2v-1.3B" and os.path.exists(tp):  # dram__bytes_read + write of one full-shape launch, from the committed ncu capture
        with open(tp) as f:
            traffic = json.load(f)["traffic_bytes_per_launch"]
    if "attn_self" in kern:
        ach = (ATTN_SELF_FLOPS / world) / (kern["attn_self"]["ms_avg"] * 1e-3) / 1e12  # per GPU: N/world query rows x N keys
        roof = {"kernel": f"attn_long_kernel (self-attention, {N_TOK}x{N_TOK}x{HEADS} heads)", "bound": "tensor", "achieved": ach, "peak": pk["tf_sustained"],
                "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"], "traffic": traffic, "peak_source": pk["src"] + " (sustained bf16)",
                "share_of_step": (kern["attn_self"]["ms_total"] / ms) if not graphs else None, "flops_per_launch": ATTN_SELF_FLOPS / world,
                "measured": roofline_source}
    # the cache-hit branch as the path runs it: `x + residual_x` formed inside the head kernel (bf16 x0 + fp32 residual in, fp32 latent out)
    hit_path = None
    if "head_hit_fused" in kern:
        n_loc = N_TOK // world
        hb = n_loc * D * 6 + n_loc * 64 * 4
        if world == 1:
            # one GPU: every second hit launch (the unconditional call) also carries the caller step in its epilogue and reads the
            # conditional prediction and the latent at its output positions (2 x n x 256 B): the mean over the launches
            hb += n_loc * 64 * 4
        gbs = hb / (kern["head_hit_fused"]["ms_avg"] * 1e-3) / 1e9
        hit_path = {"kernel": "head_tc_kernel<hit> (cache-hit add + LN + modulate + Linear + unpatchify, one pass; one GPU: + CFG combine and "
                              "scheduler update in the epilogue of the unconditional call)", "bound": "hbm",
                    "algorithmic_bytes": hb, "ms": kern["head_hit_fused"]["ms_avg"], "achieved": gbs, "unit": "GB/s", "peak": pk["hbm_gbs"],
                    "frac": gbs / pk["hbm_gbs"], "frac_of_8TBps": gbs / 8000.0, "peak_source": pk["src"], "measured": roofline_source}
        if world == 1:
            # a hit forward is host-bound (8 small launches, the GPU idles between them), so the events around its head launch also see
            # the host's launch latency; the same launch on the engine's own buffers, queued back to back, gives the kernel's own rate
            try:
                hit_path["queued"] = bench_hit_head(eng, n_loc * D * 6 + n_loc * 64 * 4, pk)
            except Exception as exc:  # noqa: BLE001 — supplementary figure: never takes the line down
                hit_path["queued"] = {"error": repr(exc)[:200]}
    # the stand-alone `x + residual_x` kernel (FLUX / HunyuanVideo hit branch, VACE): a micro-benchmark, NOT on the Wan hit path above
    k1 = bench_k1(dev, pk) if MODEL_KEY == "t2v-1.3B" else None

    # ---- non-cached leg at identical shapes: the same two steps with the controller never skipping
    speedup = None
    nocache = None
    if not args.no_cache and t_miss is not None and t_hit is not None:
        model.magcache_thresh = 1e-9
        ms_nc, _, _, _, _, per_fwd_nc = timed(step_resident, 2, False, 1 if graphs else 0, start_step=10)
        model.magcache_thresh = thresh
        t_step_nc = ms_nc / 2
        sec_video_nc = t_step_nc * SAMPLE_STEPS * 1e-3
        sec_video = (n_miss_video * t_miss + n_hit_video * t_hit + SAMPLE_STEPS * t_glue) * 1e-3
        nocache = {"steps": 2, "ms_per_step": t_step_nc, "sec_per_video": sec_video_nc, "forwards": {"miss": len(per_fwd_nc), "hit": 0}}
        speedup = sec_video_nc / sec_video
    elif t_miss is not None:
        sec_video = (2 * SAMPLE_STEPS * t_miss + SAMPLE_STEPS * t_glue) * 1e-3 if args.no_cache else (ms * 1e-3) * SAMPLE_STEPS / args.steps
    else:
        sec_video = (ms * 1e-3) * SAMPLE_STEPS / args.steps

    # ---- token-sharded runs: the sharded forward against a single-GPU forward of the same engine code on rank 0 (miss and hit)
    shard_parity = None
    if world > 1:
        shard_parity = check_shard_parity(mc, model, weights, lat_d, ctx_d, t_dev[0], rank, dev)

    steps_per_s = args.steps / (ms * 1e-3)  # whole job: all ranks work on the same video
    e2e_v = args.steps / (ms_e2e * 1e-3)
    h2d = 2 * (lat_h.numel() * 4 + ctx_h.numel() * 2)
    d2h = 2 * lat_h.numel() * 4
    line = {"metric": "denoising_steps_per_sec", "value": steps_per_s, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD + ", 50 steps, MagCache " + ("disabled (non-cached loop)" if args.no_cache else
                                    f"E{int(PRESET['thresh'] * 100):03d}K{PRESET['K']}R{int(PRESET['retention_ratio'] * 10):02d}") +
                                    (" (BASELINE configs[1])" if MODEL_KEY == "t2v-1.3B" else " (BASELINE configs[4] model and shape)"),
                       "tokens": N_TOK, "dim": D, "layers": LAYERS, "forwards_timed": {"miss": n_miss, "hit": n_hit},
                       "parallelism": "single GPU" if world == 1 else f"token-axis shard over {world} GPUs ({N_TOK // world} tokens each), K|V rows exchanged per layer, replicated weights",
                       "cuda_graphs": bool(graphs),
                       "warmup_walks": f"steps {WARM_START_STEP}..{WARM_START_STEP + args.warmup - 1} of the schedule (misses and hits on both CFG slots), outside the timed region",
                       "l2_policy": "per-forward working set (>= 1.3 GB of activations + 2.8 GB weights) exceeds the 126 MB L2; no explicit flush"},
            "sec_per_video": sec_video,
            "sec_per_video_how": f"{n_miss_video} x t_miss + {n_hit_video} x t_hit + 50 x t_glue from the per-forward CUDA events of the timed region "
                                 f"(t_miss {t_miss and round(t_miss, 3)} ms, t_hit {t_hit and round(t_hit, 3)} ms, t_glue {round(t_glue, 3)} ms)",
            "forward_ms": {"miss": t_miss, "hit": t_hit, "glue_per_step": t_glue},
            "noncached": nocache, "speedup_vs_noncached": speedup,
            "e2e": {"value": e2e_v, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "hit_path": hit_path, "kernels": kern, "attribution": attribution,
            "k1_cache_hit_add_microbench": k1, "shard_parity": shard_parity,
            "model_flops_per_miss_forward": FWD_FLOPS,
            "achieved_tflops_miss_only_whole_job": (n_miss * FWD_FLOPS / 1e12) / (ms * 1e-3) if n_miss else None}
    if rank == 0:
        if world == 1 and not args.skip_cpu and MODEL_KEY == "t2v-1.3B":
            line["cpu_baseline"] = cpu_baseline_leg()
        print(json.dumps(line), flush=True)
    if world > 1:
        shutdown_distributed(model)


def check_shard_parity(mc, model, weights, lat_d, ctx_d, t, rank, dev):
    """All ranks run a miss and a hit of the sharded engine; rank 0 also runs them on a single-GPU engine over the same weights.
    The two differ only by the attention's work split (partial softmaxes merged in a different order): rel-L2 must stay at that level."""
    import torch
    import torch.distributed as dist
    outs = []
    mc.reset_magcache(model)
    model.cnt = 0
    saved = (model.magcache_thresh, model.retention_ratio)
    model.magcache_thresh, model.retention_ratio = 10.0, 0.02  # window opens at cnt 2: miss, miss, hit, hit
    for _ in range(4):
        outs.append(model([lat_d], t=t, context=[ctx_d], seq_len=N_TOK)[0].clone())
    model.magcache_thresh, model.retention_ratio = saved
    mc.reset_magcache(model)
    res = None
    if rank == 0:
        single = mc.WanModelHandle(weights)
        mc.init_magcache(single, SAMPLE_STEPS, thresh=10.0, K=PRESET["K"], retention_ratio=0.02, table=TABLE)
        ref = [single([lat_d], t=t, context=[ctx_d], seq_len=N_TOK)[0] for _ in range(4)]
        rel = [float((a.double() - b.double()).norm() / b.double().norm()) for a, b in zip(outs, ref)]
        res = {"rel_l2_vs_single_gpu": {"miss": max(rel[0], rel[1]), "hit": max(rel[2], rel[3])}, "bound": 5e-3}
        del single
        torch.cuda.empty_cache()
        assert max(rel) < 5e-3, f"sharded forward differs from the single-GPU forward: {rel}"
    dist.barrier()
    return res


def run_mmdit(args, rank, world):
    """BASELINE configs[0] / configs[3] on the MMDiT engines (magcache_b200/mmdit.py): FLUX.1-dev 1024x1024 (4096 image + 512 text
    tokens, 19 + 38 blocks, E024K5R01, 28 steps) and HunyuanVideo 720p x 129 frames (118 800 image + 256 text tokens, 20 + 40 blocks,
    E024K6R02, 50 steps), synthetic device-side weights. One step = one patched-forward call (these pipelines use distilled guidance:
    no CFG pair). Same JSON contract as the Wan workload; the roofline object is the joint-attention kernel."""
    import torch

    import magcache_b200 as mc
    from magcache_b200 import mmdit, ops

    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", rank))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(local)
    if world > 1:  # ONE sample, image tokens sharded over the ranks, text tokens replicated, K|V rows exchanged peer to peer per attention
        dist.init_process_group("nccl", device_id=dev)
    skw = dict(shard_world=world, shard_rank=rank) if world > 1 else {}
    g = torch.Generator(device=dev).manual_seed(0)
    flux = args.workload == "flux"
    if flux:
        total_steps, preset = 28, dict(thresh=0.24, K=5, retention_ratio=0.1)
        model = mmdit.MMDiTHandle(mmdit.FluxEngine(mmdit.random_flux_weights(dev), **skw))
        mc.init_magcache_flux(model, total_steps, **preset)
        n_img, n_txt, heads, layers = 4096, 512, 24, 19 + 38
        hs_h = torch.randn(1, n_img, 64, generator=torch.Generator().manual_seed(0)).bfloat16().pin_memory()
        enc_h = torch.randn(1, n_txt, 4096, generator=torch.Generator().manual_seed(1)).bfloat16().pin_memory()
        hs, enc = hs_h.to(dev), enc_h.to(dev)
        pooled = torch.randn(1, 768, device=dev, generator=g).bfloat16()
        img_ids = torch.zeros(n_img, 3, device=dev)
        img_ids[:, 1], img_ids[:, 2] = torch.arange(n_img, device=dev) // 64, torch.arange(n_img, device=dev) % 64
        txt_ids = torch.zeros(n_txt, 3, device=dev)
        gd = torch.tensor([3.5], device=dev)
        ts = [torch.tensor([1.0 - i / total_steps], device=dev) for i in range(total_steps)]

        def call(i, x, c):
            return model(x, c, pooled, ts[i % total_steps], img_ids, txt_ids, gd, return_dict=False)[0]
        workload = "FLUX.1-dev 1024x1024, 28 steps, MagCache E024K5R01 (BASELINE configs[0])"
    else:
        total_steps, preset = 50, dict(thresh=0.24, K=6, retention_ratio=0.2)
        model = mmdit.MMDiTHandle(mmdit.HunyuanEngine(mmdit.random_hunyuan_weights(dev), **skw))
        mc.init_magcache_hunyuan(model, total_steps, **preset)
        grid = (33, 45, 80)  # 129 frames -> 33 latent frames; 720 x 1280 -> 90 x 160 latent -> 45 x 80 patches
        n_img, n_txt, heads, layers = grid[0] * grid[1] * grid[2], 256, 24, 20 + 40
        hs_h = torch.randn(1, 16, grid[0], 2 * grid[1], 2 * grid[2], generator=torch.Generator().manual_seed(0)).bfloat16().pin_memory()
        enc_h = torch.randn(1, n_txt, 4096, generator=torch.Generator().manual_seed(1)).bfloat16().pin_memory()
        hs, enc = hs_h.to(dev), enc_h.to(dev)
        mask = torch.zeros(1, n_txt, dtype=torch.long, device=dev)
        mask[0, :48] = 1
        pooled = torch.randn(1, 768, device=dev, generator=g).bfloat16()
        ang = torch.rand(n_img, 64, device=dev, generator=g) * 6.28
        cos, sin = ang.cos().repeat_interleave(2, dim=1), ang.sin().repeat_interleave(2, dim=1)
        gd = torch.tensor([6000.0], device=dev)
        ts = [torch.tensor([1000.0 * (1 - i / total_steps)], device=dev) for i in range(total_steps)]

        def call(i, x, c):
            return model(x, ts[i % total_steps], c, mask, pooled, cos, sin, gd, return_dict=False)
        workload = "HunyuanVideo 720p x 129 frames, 50 steps, MagCache E024K6R02 (BASELINE configs[3])"
    out_h = torch.empty_like(hs_h).pin_memory()
    steps = args.steps

    def timed(e2e, tags):
        mc.reset_magcache(model)
        for i in range(args.warmup):
            call(i, hs, enc)
        # warm the hit path too (first eligible call of the schedule) before the clock starts
        model.cnt = total_steps // 2
        call(total_steps // 2, hs, enc)
        mc.reset_magcache(model)
        ops.PROFILE = {} if tags else None
        ops.PROFILE_TAGS = tags
        n0 = ops.LAUNCHES
        sampler = ClockSampler(local)

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
        barrier()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            if e2e:
                x, c = hs_h.to(dev, non_blocking=True), enc_h.to(dev, non_blocking=True)
                o = call(i, x, c)
                out_h.view(-1)[:o.numel()].copy_(o.reshape(-1), non_blocking=True)
            else:
                o = call(i, hs, enc)
        e1.record()
        barrier()
        clocks = sampler.stop()
        prof, ops.PROFILE, ops.PROFILE_TAGS = ops.PROFILE, None, None
        t_ms = e0.elapsed_time(e1)
        if world > 1:  # the job's time is the slowest rank's
            tms = torch.tensor([t_ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            t_ms = float(tms.item())
        return t_ms, ops.LAUNCHES - n0, clocks, prof, o

    ms, launches, clocks, prof, out = timed(False, {"mmdit_attn"})
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"prediction": out})
    ms_e2e, _, _, _, _ = timed(True, None)
    pk = peaks()
    S = n_img + n_txt
    attn_flops = 4.0 * (n_img // world + n_txt) * S * heads * 128  # per GPU: its image rows + the replicated text rows x all keys
    kern = {t: {"launches": len(ev), "ms_avg": sum(a.elapsed_time(b) for a, b in ev) / len(ev), "ms_total": sum(a.elapsed_time(b) for a, b in ev)} for t, ev in (prof or {}).items()}
    roof = None
    if "mmdit_attn" in kern:
        ach = attn_flops / (kern["mmdit_attn"]["ms_avg"] * 1e-3) / 1e12
        roof = {"kernel": f"attn_long_kernel (joint attention, {n_img // world + n_txt}x{S}x{heads} heads per GPU)", "bound": "tensor", "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_sustained"], "traffic": None, "peak_source": pk["src"] + " (sustained bf16)", "share_of_step": kern["mmdit_attn"]["ms_total"] / ms,
                "flops_per_launch": attn_flops, "measured": "CUDA events around every launch inside the timed region"}
    line = {"metric": "denoising_steps_per_sec", "value": steps / (ms * 1e-3), "unit": "steps/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload, "image_tokens": n_img, "text_tokens": n_txt, "layers": layers,
                       "parallelism": "single GPU" if world == 1 else f"image tokens sharded over {world} GPUs ({n_img // world} each), text tokens replicated, "
                                      f"K|V rows pushed peer to peer per attention ({type(getattr(model, '_mc_flux_engine', None) or model._mc_hunyuan_engine).__name__})",
                       "schedule": f"the first {steps} calls of the {total_steps}-step schedule from cnt = 0"},
            "sec_per_sample_if_linear": (ms * 1e-3) * total_steps / steps,
            "e2e": {"value": steps / (ms_e2e * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": hs_h.numel() * 2 + enc_h.numel() * 2,
                    "d2h_bytes_per_step": hs_h.numel() * 2, "ms_per_step": ms_e2e / steps},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "kernels": kern}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        shutdown_distributed(model)


def shutdown_distributed(model):
    """Leave cleanly and in bounded time: captured CUDA graphs hold NCCL work, and tearing the process group down under them
    can block forever — drop the graphs first, and never wait more than a few seconds for the communicator to go away."""
    import gc

    import torch
    import torch.distributed as dist
    eng = getattr(model, "_mc_engine", None)
    if eng is not None:
        eng._graphs.clear()
    gc.collect()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    done = threading.Event()

    def _destroy():
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass
        done.set()

    th = threading.Thread(target=_destroy, daemon=True)
    th.start()
    done.wait(timeout=15)
    os._exit(0)


def bench_k1(dev, pk):
    import torch
    from magcache_b200 import ops
    n = N_TOK * D
    sets = [(torch.randn(n, device=dev).bfloat16(), torch.randn(n, device=dev), torch.empty(n, device=dev)) for _ in range(3)]
    for i in range(6):
        ops.cache_hit_add(sets[i % 3][0], sets[i % 3][1], out=sets[i % 3][2])
    torch.cuda.synchronize()
    iters = 30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        ops.cache_hit_add(sets[i % 3][0], sets[i % 3][1], out=sets[i % 3][2])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    gbs = n * 10 / (ms * 1e-3) / 1e9
    return {"kernel": "axpb_kernel<bf16,f32,f32> (x + residual as a stand-alone pass, 503.2 MB algorithmic; micro-benchmark)", "bound": "hbm", "ms": ms, "achieved": gbs, "unit": "GB/s",
            "peak": pk["hbm_gbs"], "frac": gbs / pk["hbm_gbs"], "frac_of_8TBps": gbs / 8000.0, "peak_source": pk["src"],
            "method": "30 back-to-back launches rotating over 3 buffer sets (1.5 GB), CUDA events"}


def bench_hit_head(eng, algorithmic_bytes, pk):
    """The hit branch's kernel exactly as the path launches it (bf16 patch embedding + the slot's fp32 residual -> fp32 prediction,
    no step epilogue), 30 launches queued back to back on the engine's buffers of the last forward; every launch streams 302 MB
    (> the 126 MB L2)."""
    import torch
    e, _ = eng.time_embedding()
    for _ in range(3):
        eng.head(eng.x0, e, eng.grid, residual=eng.res[0])
    torch.cuda.synchronize()
    iters = 30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        eng.head(eng.x0, e, eng.grid, residual=eng.res[0])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    gbs = algorithmic_bytes / (ms * 1e-3) / 1e9
    return {"ms": ms, "achieved": gbs, "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "frac_of_8TBps": gbs / 8000.0, "algorithmic_bytes": algorithmic_bytes,
            "method": "30 launches of head_tc_kernel<hit> on the engine's own x0 / residual buffers queued back to back, CUDA events around the batch"}


def cpu_baseline_leg():
    state = cpu_model()
    cores = cpu_threads()
    t_miss_small, t_hit = cpu_cycle(state)  # one cycle: ~10-30 s of CPU work
    value, sec_video, t_miss = cpu_extrapolate(t_miss_small, t_hit)
    return {"value": value, "unit": "steps/s", "cores": cores, "kind": "port", "sample": cpu_sample_text(1, cores, t_miss_small, t_hit, t_miss, sec_video)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=SAMPLE_STEPS)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cache", action="store_true", help="time the non-cached DiT loop at identical shapes")
    ap.add_argument("--skip-cpu", action="store_true", help="omit the cpu_baseline leg (debugging)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32)")
    ap.add_argument("--workload", default="wan1.3b", choices=["wan1.3b", "wan14b", "flux", "hunyuan720p"],
                    help="wan14b: BASELINE configs[4] model/shape; flux: configs[0] (FLUX.1-dev 1024x1024, 28 steps); hunyuan720p: configs[3] "
                         "(720p x 129 frames, 50 steps) — none of these is the driver's metric")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm's timed cycle keeps no outputs")
    select_workload(args.workload)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.workload in ("flux", "hunyuan720p"):
        run_mmdit(args, rank, world)
        return
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if world != args.gpus and args.gpus > 1:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    run_ours(args, rank, world)


if __name__ == "__main__":
    main()
