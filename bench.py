#!/usr/bin/env python
"""bench.py — DiT-step latent tokens/s of the B200-native miniFLUX sampler step (BASELINE.json metric).

A "step" is ONE DiT forward (the pipeline's `self.dit(...)` call, P:760-766) at the headline single-step shape of the
768p / 10 s configuration (BASELINE.md §2): unit 30, stage 2 — CFG batch B=2, S = 128 text + 28x240 + 960 + 3840 history
+ 3840 current = 15488 tokens, full 8+16-block miniFLUX (D=1920, 30 heads), synthetic latents / text embeddings and
random-init weights (no checkpoints offline).  tokens/s = B * S / t_step; with --gpus N the SAME step is sharded over
the N GPUs (CFG pair first, then Ulysses sequence parallel with the exchange fused into the kernels over NVLink peer
memory; strong scaling, `parity_vs_n1` = max |sharded - single-GPU| of the step's output on the same inputs).
The line also carries the second half of BASELINE's metric: `vae_decode` (768p causal-VAE decode, frames/s + conv roofline)
and `video_e2e` (the whole 768p / 10 s pyramidal sampler + decode, frames/s), and two baselines timed in the same run: the
reference algorithm on the host cores (`cpu_baseline`) and the UNMODIFIED reference modules in eager PyTorch bf16 on the
same B200 (`gpu_eager_baseline`, when oracle/pin/stage_reference.py has staged the reference in oracle/_ref).

  python bench.py [--gpus N] [--steps K] [--warmup W]           our arm (CUDA kernels through the C-ABI)
  python bench.py --impl reference ...                           the reference algorithm's CPU path (oracle port), host cores
  python bench.py ... --dump-outputs DIR                         also write the last timed step's output to DIR/<name>.npy

Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for the definitions of value / e2e / roofline / cpu_baseline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

ATTN_TRAFFIC_BYTES = 460.71e6   # profiles/r02_attn2_final_ncu.txt: dram__bytes_read 358.04 MB + dram__bytes_write 102.67 MB per launch
METRIC = "dit_step_latent_tokens_per_sec"
UNIT = "tokens/s"
WORKLOAD = ("miniFLUX 768p/10s (BASELINE configs[2]) — one DiT forward at unit 30 / stage 2: CFG batch 2, "
            "S=15488 (128 text + 28x240 + 960 + 3840 history + 3840 current), 8 double + 16 single blocks, D=1920, 30 heads")


def step_clip_shapes(batch=2):
    """Latent clips the pipeline feeds at unit 30, stage 2 of 768p (P:1159-1182): low-res history first, current last."""
    return [(batch, 16, 28, 24, 40), (batch, 16, 1, 48, 80), (batch, 16, 1, 96, 160), (batch, 16, 1, 96, 160)]


def cpu_sample_clip_shapes(batch=2):
    """Bounded CPU sample: same model width/sequence structure at unit 30, stage 0 (S = 128 + 31*240 = 7568)."""
    return [(batch, 16, 30, 24, 40), (batch, 16, 1, 24, 40)]


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"tflops_sustained": d.get("bf16_tflops_sustained"), "tflops_burst": d.get("bf16_tflops"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the arrays the timed path returned in its last timed step, as DIR/<name>.npy in float32 (a few MB),
    so that two builds can be compared output for output: inputs and weights come from fixed seeds, identical from run to
    run with the same arguments."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(d / f"{name}.npy", t.detach().float().cpu().numpy())


# ----------------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(n_double=1, n_single=2, threads=None, repeats=1):
    """Time the reference algorithm's CPU path (oracle port, fp32) on a bounded sample; returns tokens/s extrapolated to
    the full 8+16-block forward, and a description of the sample."""
    import torch
    from oracle import flux_oracle as FO
    # every host core, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1: round 1's N>1 CPU arm ran on one thread)
    torch.set_num_threads(threads or os.cpu_count() or 1)
    threads = torch.get_num_threads()
    cfg = FO.FluxConfig(num_layers=n_double, num_single_layers=n_single)
    params = FO.synthetic_flux_params(cfg, seed=0)
    g = torch.Generator().manual_seed(1)
    clips = [torch.randn(s, generator=g) for s in cpu_sample_clip_shapes()]
    b = clips[0].shape[0]
    enc = torch.randn(b, 128, 4096, generator=g) * 0.2
    mask = torch.ones(b, 128, dtype=torch.long)
    pooled = torch.randn(b, 768, generator=g)
    t = torch.full((b,), 386.0)
    s = 128 + sum(c.shape[2] * (c.shape[3] // 2) * (c.shape[4] // 2) for c in clips)
    times = []
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            out = FO.flux_forward(params, cfg, clips, t, enc, mask, pooled)
            times.append(time.perf_counter() - t0)
    dt = sorted(times)[len(times) // 2]
    full = dt * (8 + 16) / (n_double + n_single)   # block cost dominates; embedders/head are <1 %
    return {"tokens_per_s": b * s / full, "sample_s": dt, "threads": threads, "tokens": b * s, "out": out,
            "sample": (f"oracle port (PyTorch fp32, {threads} threads): {n_double} double + {n_single} single miniFLUX blocks at "
                       f"B={b}, S={s} (768p unit 30 / stage 0 sequence), time x{(8 + 16) / (n_double + n_single):.0f} to the "
                       f"24-block forward")}


def run_reference(args):
    """--impl reference: the reference's own CPU path (oracle port) on this box's host cores.  A step = one bounded sample
    (1 double + 2 single blocks at the 768p unit-30 / stage-0 sequence, scaled x8 to the 24-block forward): `warmup` untimed
    samples, then exactly `steps` timed ones; `value` is the mean over the timed samples."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    for _ in range(max(1, args.warmup)):
        cpu_reference_sample(repeats=1)             # untimed: page-in, thread pool
    t0 = time.perf_counter()
    vals = [cpu_reference_sample(repeats=1) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"reference_sample_out": vals[-1]["out"]})
    tok = vals[0]["tokens"]
    mean_full_s = sum(v["tokens"] / v["tokens_per_s"] for v in vals) / len(vals)     # extrapolated 24-block seconds per step
    value = tok / mean_full_s
    line = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
            "steps": len(vals), "warmup": max(1, args.warmup), "ms_per_step": 1e3 * mean_full_s,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "same_config": False,
            "config": {"workload": WORKLOAD,
                       "note": ("CPU arm: every step is a bounded SAMPLE of the workload, not the S=15488 step itself (see "
                                "cpu_baseline.sample); ms_per_step is the sample time x8; the timed samples took "
                                f"{wall:.1f} s of wall clock")},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": vals[0]["threads"], "kind": "port",
                             "sample": vals[0]["sample"] + f"; mean of {len(vals)} timed samples after {max(1, args.warmup)} warm-up"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def gpu_eager_reference(dev, host, steps=2):
    """The UNMODIFIED reference `PyramidFluxTransformer` (oracle/_ref copy through oracle/pin/ref_shim.py) in eager PyTorch
    under bf16 autocast on this GPU: the full 8+16-block forward at the bench shape, dense [B,1,S,S] bool mask + SDPA as the
    reference builds them (F:318-350, B:363-365).  A reported baseline (SURVEY.md §8d), never on the product path."""
    import torch
    try:
        from oracle.pin import ref_shim
        if not ref_shim.reference_available():
            return {"unavailable": "reference packages not staged in oracle/_ref (oracle/pin/stage_reference.py)"}
        ref_shim.install()
        from pyramid_dit.flux_modules import PyramidFluxTransformer
        with torch.device(dev):
            m = PyramidFluxTransformer(num_layers=8, num_single_layers=16, num_attention_heads=30, attention_head_dim=64,
                                       in_channels=64, joint_attention_dim=4096, pooled_projection_dim=768).eval()
        g = torch.Generator(device=dev).manual_seed(0)
        with torch.no_grad():
            for prm in m.parameters():                      # the reference zero-inits AdaLN/proj_out (F:168-183)
                prm.copy_(torch.randn(prm.shape, device=dev, generator=g) * 0.02)
        m = m.to(torch.bfloat16)
        clips = [x.to(dev) for x in host["clips"]]
        kw = dict(sample=[clips], timestep_ratio=host["t"].to(dev), encoder_hidden_states=host["enc"].to(dev),
                  encoder_attention_mask=host["mask"].to(dev), pooled_projections=host["pooled"].to(dev))
        times = []
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            for i in range(1 + steps):
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                out = m(**kw)[0]
                e.record()
                torch.cuda.synchronize()
                if i > 0:
                    times.append(s.elapsed_time(e))
        ms = sum(times) / len(times)
        b, seq = clips[-1].shape[0], 128 + sum(c.shape[2] * (c.shape[3] // 2) * (c.shape[4] // 2) for c in clips)
        res = {"value": b * seq / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "warmup": 1,
               "kind": "reference (unmodified modules, eager PyTorch, bf16 autocast, SDPA with the dense bool mask)",
               "same_config": True, "output_finite": bool(torch.isfinite(out.float()).all())}
        del m, out
        torch.cuda.empty_cache()
        return res
    except Exception as ex:  # noqa: BLE001  (a baseline leg must never take the bench line down)
        return {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}


# ----------------------------------------------------------------------------------------------------------------------
def random_flux_state_dict(cfg_kw, device, seed=0):
    """Random-init weights of the named architecture, generated on the device (2 B parameters; no checkpoint offline).
    Same distribution as oracle.flux_oracle.synthetic_flux_params; shapes from the reference key layout."""
    import math
    import torch
    from pyramid_flow_b200.dit import FluxConfigB200
    c = FluxConfigB200(**cfg_kw)
    d, hd = c.inner_dim, c.attention_head_dim
    g = torch.Generator(device=device).manual_seed(seed)
    sd = {}

    def lin(name, o, i, mod=False):
        std = (0.5 if mod else 1.0) / math.sqrt(i)
        sd[name + ".weight"] = (torch.randn(o, i, device=device, generator=g) * std).bfloat16()
        sd[name + ".bias"] = torch.randn(o, device=device, generator=g) * 0.02

    def nw(name):
        sd[name] = 1.0 + 0.1 * torch.randn(hd, device=device, generator=g)

    lin("time_text_embed.timestep_embedder.linear_1", d, 256); lin("time_text_embed.timestep_embedder.linear_2", d, d)
    lin("time_text_embed.text_embedder.linear_1", d, c.pooled_projection_dim); lin("time_text_embed.text_embedder.linear_2", d, d)
    lin("context_embedder", d, c.joint_attention_dim); lin("x_embedder", d, c.in_channels)
    for i in range(c.num_layers):
        p = f"transformer_blocks.{i}"
        lin(p + ".norm1.linear", 6 * d, d, True); lin(p + ".norm1_context.linear", 6 * d, d, True)
        for n in ("to_q", "to_k", "to_v", "add_q_proj", "add_k_proj", "add_v_proj", "to_out.0", "to_add_out"):
            lin(f"{p}.attn.{n}", d, d)
        for n in ("norm_q", "norm_k", "norm_added_q", "norm_added_k"):
            nw(f"{p}.attn.{n}.weight")
        lin(p + ".ff.net.0.proj", 4 * d, d); lin(p + ".ff.net.2", d, 4 * d)
        lin(p + ".ff_context.net.0.proj", 4 * d, d); lin(p + ".ff_context.net.2", d, 4 * d)
    for i in range(c.num_single_layers):
        p = f"single_transformer_blocks.{i}"
        lin(p + ".norm.linear", 3 * d, d, True); lin(p + ".proj_mlp", 4 * d, d); lin(p + ".proj_out", d, 5 * d)
        for n in ("to_q", "to_k", "to_v"):
            lin(f"{p}.attn.{n}", d, d)
        nw(p + ".attn.norm_q.weight"); nw(p + ".attn.norm_k.weight")
    lin("norm_out.linear", 2 * d, d, True); lin("proj_out", c.in_channels, d)
    return c, sd


def random_vae_state_dict(device, seed=0, block_out_channels=(128, 256, 512, 512), layers_per_block=(3, 3, 3, 3),
                          spatial_up=(True, True, True, False), temporal_up=(True, True, True, False), latent=16):
    """Random-init causal-VAE decoder weights in the reference key layout (`decoder.*`, `post_quant_conv.*`)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    sd = {}
    rev = list(reversed(block_out_channels))

    def conv(name, co, ci, k):
        sd[name + ".conv.weight"] = (torch.randn(co, ci, k, k, k, device=device, generator=g) * (ci * k ** 3) ** -0.5).cpu()
        sd[name + ".conv.bias"] = (torch.randn(co, device=device, generator=g) * 0.02).cpu()

    def norm(name, c):
        sd[name + ".weight"] = (1 + 0.1 * torch.randn(c, device=device, generator=g)).cpu()
        sd[name + ".bias"] = (0.05 * torch.randn(c, device=device, generator=g)).cpu()

    def res(name, ci, co):
        norm(name + ".norm1", ci); conv(name + ".conv1", co, ci, 3); norm(name + ".norm2", co); conv(name + ".conv2", co, co, 3)
        if ci != co:
            conv(name + ".conv_shortcut", co, ci, 1)

    top = rev[0]
    conv("post_quant_conv", latent, latent, 1); conv("decoder.conv_in", top, latent, 3)
    res("decoder.mid_block.resnets.0", top, top); res("decoder.mid_block.resnets.1", top, top)
    norm("decoder.mid_block.attentions.0.group_norm", top)
    for n in ("to_q", "to_k", "to_v", "to_out.0"):
        sd[f"decoder.mid_block.attentions.0.{n}.weight"] = (torch.randn(top, top, device=device, generator=g) * top ** -0.5).cpu()
        sd[f"decoder.mid_block.attentions.0.{n}.bias"] = (torch.randn(top, device=device, generator=g) * 0.02).cpu()
    prev = top
    for i, co in enumerate(rev):
        for j in range(layers_per_block[i]):
            res(f"decoder.up_blocks.{i}.resnets.{j}", prev if j == 0 else co, co)
        if spatial_up[i]:
            conv(f"decoder.up_blocks.{i}.upsamplers.0.conv", 4 * co, co, 3)
        if temporal_up[i]:
            conv(f"decoder.up_blocks.{i}.temporal_upsamplers.0.conv", 2 * co, co, 3)
        prev = co
    norm("decoder.conv_norm_out", block_out_channels[0]); conv("decoder.conv_out", 3, block_out_channels[0], 3)
    return sd


def random_mmdit_state_dict(cfg, device, seed=0):
    """Random-init SD3-MMDiT weights in the reference key layout (mmdit_modules/modeling_pyramid_mmdit.py:420-497 consumers)."""
    import math
    import torch
    d, hd = cfg.inner_dim, cfg.attention_head_dim
    g = torch.Generator(device=device).manual_seed(seed)
    sd = {}

    def lin(name, o, i, mod=False):
        sd[name + ".weight"] = (torch.randn(o, i, device=device, generator=g) * ((0.5 if mod else 1.0) / math.sqrt(i))).bfloat16()
        sd[name + ".bias"] = torch.randn(o, device=device, generator=g) * 0.02

    sd["pos_embed.pos_embed"] = torch.randn(1, cfg.pos_embed_max_size ** 2, d, device=device, generator=g) * 0.1
    sd["pos_embed.proj.weight"] = (torch.randn(d, cfg.in_channels, 2, 2, device=device, generator=g) * (4 * cfg.in_channels) ** -0.5).bfloat16()
    sd["pos_embed.proj.bias"] = torch.randn(d, device=device, generator=g) * 0.02
    lin("time_text_embed.timestep_embedder.linear_1", d, 256); lin("time_text_embed.timestep_embedder.linear_2", d, d)
    lin("time_text_embed.text_embedder.linear_1", d, cfg.pooled_projection_dim); lin("time_text_embed.text_embedder.linear_2", d, d)
    lin("context_embedder", d, cfg.joint_attention_dim)
    for i in range(cfg.num_layers):
        pre, last = f"transformer_blocks.{i}", i == cfg.num_layers - 1
        lin(pre + ".norm1.linear", 6 * d, d, True); lin(pre + ".norm1_context.linear", (2 if last else 6) * d, d, True)
        for n in ("to_q", "to_k", "to_v", "add_k_proj", "add_v_proj", "add_q_proj", "to_out.0"):
            lin(f"{pre}.attn.{n}", d, d)
        for n in ("norm_q", "norm_k", "norm_add_q", "norm_add_k"):
            sd[f"{pre}.attn.{n}.weight"] = 1.0 + 0.1 * torch.randn(hd, device=device, generator=g)
        lin(pre + ".ff.net.0.proj", 4 * d, d); lin(pre + ".ff.net.2", d, 4 * d)
        if not last:
            lin(pre + ".attn.to_add_out", d, d); lin(pre + ".ff_context.net.0.proj", 4 * d, d); lin(pre + ".ff_context.net.2", d, 4 * d)
    lin("norm_out.linear", 2 * d, d, True); lin("proj_out", 4 * cfg.in_channels, d)
    return sd


def run_mmdit(args):
    """--model mmdit: BASELINE configs[4] — one SD3-MMDiT forward (24 joint blocks, D=1536, 24 heads) at the headline step of
    768p / 5 s (temp 16): unit 15 / stage 2, CFG batch 2, S = 128 + 13x240 + 960 + 2x3840 = 11888.  One GPU, host-launched."""
    import torch
    from pyramid_flow_b200 import _lib
    from pyramid_flow_b200.mmdit import B200MMDiT, MMDiTConfigB200
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    _lib.require_device()
    cfg = MMDiTConfigB200()
    model = B200MMDiT(cfg, random_mmdit_state_dict(cfg, dev), device=dev)
    torch.cuda.empty_cache()
    b = 2
    g = torch.Generator().manual_seed(100)
    shapes = [(b, 16, 13, 24, 40), (b, 16, 1, 48, 80), (b, 16, 1, 96, 160), (b, 16, 1, 96, 160)]
    host = {"clips": [torch.randn(sh, generator=g).bfloat16().pin_memory() for sh in shapes],
            "enc": (torch.randn(b, 128, 4096, generator=g) * 0.2).bfloat16().pin_memory(),
            "mask": torch.ones(b, 128, dtype=torch.int64).pin_memory(),
            "pooled": torch.randn(b, 2048, generator=g).bfloat16().pin_memory(),
            "t": torch.tensor([3.0] * b).bfloat16().pin_memory()}
    dev_in = {k: ([x.to(dev) for x in v] if isinstance(v, list) else v.to(dev)) for k, v in host.items()}
    out_host = torch.empty(b, 16, 1, 96, 160, dtype=torch.bfloat16).pin_memory()

    def step_resident():
        return model(sample=[dev_in["clips"]], timestep_ratio=dev_in["t"], encoder_hidden_states=dev_in["enc"],
                     encoder_attention_mask=dev_in["mask"], pooled_projections=dev_in["pooled"])[0]

    def step_e2e():
        o = model(sample=[[x.to(dev, non_blocking=True) for x in host["clips"]]], timestep_ratio=host["t"].to(dev, non_blocking=True),
                  encoder_hidden_states=host["enc"].to(dev, non_blocking=True), encoder_attention_mask=host["mask"].to(dev, non_blocking=True),
                  pooled_projections=host["pooled"].to(dev, non_blocking=True))[0]
        out_host.copy_(o, non_blocking=True)

    def timed(fn, steps):
        torch.cuda.synchronize()
        s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _lib.launch_count()
        s_.record()
        for _ in range(steps):
            out = fn()
        e_.record()
        torch.cuda.synchronize()
        return s_.elapsed_time(e_) / steps, _lib.launch_count() - n0, out

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(dev.index)
    sampler.start()
    time.sleep(0.25)
    t0 = time.time()
    ms, launches, step_out = timed(step_resident, args.steps)
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"mmdit_step_out": step_out})
    step_e2e()
    ms_e2e, _, _ = timed(step_e2e, args.steps)
    plan = model.last_plan
    d = cfg.inner_dim
    tokens = b * plan.seq
    # per token per joint block 24 D^2 (qkv 6, out 2, ff 16); the last block's text stream stops after attention (MB:659-660)
    gemm = 24.0 * d * d * (b * plan.seq * cfg.num_layers - b * plan.text_len * (18.0 / 24.0))
    attn = 4.0 * 64 * cfg.num_attention_heads * plan.allowed_pairs * cfg.num_layers
    peaks = measured_peaks()
    ach = (gemm + attn) / (ms * 1e-3) / 1e12
    h2d = sum(x.numel() * x.element_size() for x in host["clips"]) + sum(host[k].numel() * host[k].element_size() for k in ("enc", "mask", "pooled", "t"))
    line = {"metric": METRIC, "value": tokens / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": ("SD3 MMDiT 768p/5s (BASELINE configs[4]) — one DiT forward at unit 15 / stage 2: CFG batch 2, "
                                    "S=11888 (128 text + 13x240 + 960 + 3840 history + 3840 current), 24 joint blocks, D=1536, 24 heads"),
                       "global_batch": b, "seq_len": plan.seq, "parallelism": "single GPU", "launch_mode": "host-launched",
                       "l2": "per-step working set exceeds the 126 MB L2; no explicit flush",
                       "step_tflop": {"gemm": gemm / 1e12, "attention_masked": attn / 1e12}},
            "clocks": clocks,
            "e2e": {"value": tokens / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": out_host.numel() * out_host.element_size(),
                    "api": "B200MMDiT.__call__ with pinned host inputs, result copied back to host"},
            "gpu_launches": launches,
            "roofline": {"kernel": "whole step (GEMM + attention flops of every pf:: kernel launched)", "bound": "tensor",
                         "achieved": ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": ach / peaks["tflops_sustained"],
                         "peak_source": peaks["source"] + ", sustained cuBLAS bf16", "traffic": None},
            "cpu_baseline": None}
    print(json.dumps(line), flush=True)


def vae_decode_leg(dev, world, rank):
    """Causal-VAE decode at 768p (BASELINE configs[2], second half of the metric): un-tiled, temporally chunked (window 4),
    5 latent -> 33 video frames on one GPU; with N GPUs 1 + 4 N latent frames, context-parallel (temporal split + 2-frame
    halo exchange per causal conv).  Conv roofline: 1.10e7 MAC per output pixel-frame (SURVEY.md §8a) against the measured
    sustained bf16 peak."""
    import torch
    from pyramid_flow_b200.vae import B200CausalVAE, VaeConfigB200
    vae = B200CausalVAE(VaeConfigB200(), random_vae_state_dict(dev), device=dev)
    t_lat = 5 if world == 1 else 1 + 4 * world
    g = torch.Generator().manual_seed(7)
    z = torch.randn(1, 16, t_lat, 96, 160, generator=g).bfloat16().to(dev)
    if world > 1:
        vae.set_context_parallel(None)

    def run():
        return vae.decode(z, temporal_chunk=True, window_size=4).sample

    run()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    s.record()
    for _ in range(reps):
        out = run()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / reps
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    frames = 1 + 8 * (t_lat - 1)
    flops = 2.0 * 1.10e7 * frames * 768 * 1280
    peaks = measured_peaks()
    res = {"ms": ms, "frames": frames, "frames_per_s": frames / (ms * 1e-3), "latent": [1, 16, t_lat, 96, 160],
           "out_shape": list(out.shape), "mode": "un-tiled, temporal chunks of 4 latent frames" + (", context-parallel over %d GPUs" % world if world > 1 else ""),
           "tflops": flops / (ms * 1e-3) / 1e12, "frac_of_sustained_bf16": flops / (ms * 1e-3) / 1e12 / (peaks["tflops_sustained"] * world),
           "algorithmic_flops": flops, "peak_mem_gib": torch.cuda.max_memory_allocated() / 2 ** 30,
           "output_finite": bool(torch.isfinite(out.float()).all())}
    del vae, out
    torch.cuda.empty_cache()
    return res


def video_e2e_leg(dit, dev, world, rank):
    """frames/s end to end at 768p / 10 s (temp 31 -> 241 frames): the 3-stage pyramidal sampler loop (960 DiT calls, steps
    20/10, CFG) + causal-VAE decode, text embeddings synthetic (text encoding excluded as SURVEY.md §8d defines).  Every rank
    runs the same loop; the DiT step is CFG x SP sharded, the decode context-parallel."""
    import torch
    from pyramid_flow_b200.sampler import B200PyramidSampler
    from pyramid_flow_b200.scheduler import B200FlowMatchScheduler
    from pyramid_flow_b200.vae import B200CausalVAE, VaeConfigB200
    vae = B200CausalVAE(VaeConfigB200(), random_vae_state_dict(dev), device=dev)
    if world > 1:
        vae.set_context_parallel(None)
    torch.manual_seed(1234)                              # block noise comes from the global CPU RNG: identical on every rank
    g = torch.Generator().manual_seed(0)
    enc = (torch.randn(2, 128, 4096, generator=g) * 0.2).bfloat16().to(dev)
    mask = torch.ones(2, 128, dtype=torch.long, device=dev)
    pooled = torch.randn(2, 768, generator=g).bfloat16().to(dev)
    tokens = [0]
    orig = dit.forward

    def counting(*a, **k):
        out = orig(*a, **k)
        tokens[0] += 2 * dit.last_plan.seq
        return out

    dit.forward = counting
    try:
        sampler = B200PyramidSampler(dit, B200FlowMatchScheduler(), vae=vae)
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        t0 = time.time()
        lat = sampler.generate(enc, mask, pooled, height=768, width=1280, temp=31, num_inference_steps=[20, 20, 20],
                               video_num_inference_steps=[10, 10, 10], guidance_scale=7.0, video_guidance_scale=5.0,
                               generator=torch.Generator().manual_seed(1), output_type="latent")
        torch.cuda.synchronize()
        t1 = time.time()
        lat = torch.nan_to_num(lat.float()).clamp(-4, 4).to(lat.dtype)    # random weights: keep the decoder input sane
        lat_n = lat.clone()
        lat_n[:, :, :1] = lat_n[:, :, :1] / sampler.vae_scale_factor + sampler.vae_shift_factor
        lat_n[:, :, 1:] = lat_n[:, :, 1:] / sampler.vae_video_scale_factor + sampler.vae_video_shift_factor
        img = vae.decode(lat_n, temporal_chunk=True, window_size=4).sample
        u8 = img.float().mul(127.5).add(127.5).clamp(0, 255).byte().permute(0, 2, 3, 4, 1).contiguous().cpu()
        torch.cuda.synchronize()
        t2 = time.time()
    finally:
        dit.forward = orig
    frames = 241
    res = {"config": "miniFLUX 768x1280, temp=31 (241 frames), steps 20/10, guidance 7/5, un-tiled decode (window 4)",
           "frames_per_s_end_to_end": frames / (t2 - t0), "seconds": t2 - t0, "dit_seconds": t1 - t0,
           "decode_seconds": t2 - t1, "dit_calls": sampler.dit_calls, "dit_token_passes_per_s": tokens[0] / (t1 - t0),
           "video_shape": list(u8.shape), "latent_finite": bool(torch.isfinite(lat.float()).all())}
    del vae, img, u8
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    import torch
    import torch.distributed as dist
    from pyramid_flow_b200 import _lib
    from pyramid_flow_b200.dit import B200FluxTransformer

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.require_device()

    cfg_kw = dict(num_layers=args.layers[0], num_single_layers=args.layers[1])
    # N > 1: ONE step sharded over the GPUs (CFG pair first, then the token sequence: pyramid_flow_b200/sp.py) — the same
    # weights and inputs on every rank, strong scaling of the single step
    cfg, sd = random_flux_state_dict(cfg_kw, dev, seed=0)
    model = B200FluxTransformer(cfg, sd, device=dev)
    del sd
    torch.cuda.empty_cache()
    if args.attn_variant is not None:
        model.attn_variant = args.attn_variant
    if args.attn_phase is not None:
        _lib.set_option(_lib.PF_OPT_ATTN_TILE_PHASE, args.attn_phase)
    lay = None
    b = 2
    g = torch.Generator().manual_seed(100)
    shapes = step_clip_shapes(b)
    host = {
        "clips": [torch.randn(s, generator=g).bfloat16().pin_memory() for s in shapes],
        "enc": (torch.randn(b, 128, 4096, generator=g) * 0.2).bfloat16().pin_memory(),
        "mask": torch.ones(b, 128, dtype=torch.int64).pin_memory(),
        "pooled": torch.randn(b, 768, generator=g).bfloat16().pin_memory(),
        "t": torch.tensor([3.0] * b).bfloat16().pin_memory(),
    }
    dev_in = {k: ([x.to(dev) for x in v] if isinstance(v, list) else v.to(dev)) for k, v in host.items()}
    out_host = torch.empty(b, 16, 1, 96, 160, dtype=torch.bfloat16).pin_memory()

    def step_resident():
        return model(sample=[dev_in["clips"]], timestep_ratio=dev_in["t"], encoder_hidden_states=dev_in["enc"],
                     encoder_attention_mask=dev_in["mask"], pooled_projections=dev_in["pooled"])[0]

    def step_e2e():
        clips = [x.to(dev, non_blocking=True) for x in host["clips"]]
        enc = host["enc"].to(dev, non_blocking=True)
        pooled = host["pooled"].to(dev, non_blocking=True)
        t = host["t"].to(dev, non_blocking=True)
        mask = host["mask"].to(dev, non_blocking=True)
        o = model(sample=[clips], timestep_ratio=t, encoder_hidden_states=enc, encoder_attention_mask=mask,
                  pooled_projections=pooled)[0]
        out_host.copy_(o, non_blocking=True)
        return o

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.exchange is None:
        from pyramid_flow_b200.dit import DEFAULT_EXCHANGE
        args.exchange = DEFAULT_EXCHANGE
    parity_ref = None
    if world > 1:
        # the SAME step on one GPU (every rank computes it, host-launched) before the layout is attached: the reference the
        # sharded step's output is compared with (`parity_vs_n1`)
        parity_ref = step_resident().float().clone()
        torch.cuda.synchronize()
        from pyramid_flow_b200 import sp as SP
        lay = SP.make_layout()
        model.peer_max_seq, model.peer_max_last = 15488, 3840          # one peer arena for every shape of the 768p run
        model.peer_max_vel_bytes = 16 * 96 * 160 * 4
        model.set_parallel_layout(lay, exchange=args.exchange)
    # CUDA-graph replay at every N: the peer-memory exchange is plain kernels (no NCCL call inside the step)
    use_graph = not args.no_graph and not (world > 1 and args.exchange == "nccl")
    model.use_cuda_graph = use_graph

    host_ms = {}

    def timed(fn, steps, events=False):
        barrier()
        if events:
            model.attn_events = []      # events around each attention launch: forces the host-launched (eager) path
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _lib.launch_count() + model.graph_launches_replayed
        s.record()
        h0 = time.perf_counter()
        for _ in range(steps):
            out = fn()
        host_ms["last"] = (time.perf_counter() - h0) * 1e3 / steps     # host time to ENQUEUE a step (no sync inside)
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        launches = _lib.launch_count() + model.graph_launches_replayed - n0
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        return ms / steps, launches, out

    for _ in range(max(args.warmup, 3)):
        step_resident()
    plan = model.last_plan
    tokens = b * plan.seq

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.25)
    t0 = time.time()
    ms_step, launches, step_out = timed(step_resident, args.steps, events=False)
    host_enqueue_ms = host_ms["last"]
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"dit_step_out": step_out})
    del step_out
    # the timed region above carries no per-launch instrumentation (graph replay, or plain host launches with --no-graph);
    # the dominant kernel's launch durations come from the same number of host-launched steps run right after it, with CUDA
    # events around each attention launch
    ms_eager, _, _ = timed(step_resident, args.steps, events=True)
    # dominant kernel: the masked attention; per-launch duration from CUDA events recorded around each launch
    ev = model.attn_events or []
    model.attn_events = None
    attn_ms = [a.elapsed_time(bq) for a, bq in ev]
    n_attn_step = cfg.num_layers + cfg.num_single_layers
    if world == 1 and model.trim_last_block and len(attn_ms) % n_attn_step == 0:
        # the last block's launch computes the current clip's query rows only: not a full-size launch, keep it out of
        # the per-launch average that the roofline figure is built on
        attn_ms = [x for i, x in enumerate(attn_ms) if i % n_attn_step != n_attn_step - 1]
    attn_avg = sum(attn_ms) / max(1, len(attn_ms))
    step_e2e()
    step_e2e()
    ms_e2e, _, _ = timed(step_e2e, args.steps)
    # per-kernel-family breakdown of ONE extra (untimed-for-the-metric) step, CUDA events around every launch
    model.timer.enabled = True
    model.attn_events = []
    step_resident()
    torch.cuda.synchronize()
    breakdown = model.timer.totals_ms()
    breakdown["attention"] = sum(a.elapsed_time(bq) for a, bq in model.attn_events)
    model.timer.enabled = False
    model.attn_events = None

    parity_vs_n1 = None
    if parity_ref is not None:
        parity_vs_n1 = (step_resident().float() - parity_ref).abs().max().item()       # graph-replayed sharded step
        tt = torch.tensor([parity_vs_n1], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        parity_vs_n1 = float(tt.item())
        del parity_ref

    vae_leg = None if args.no_vae else vae_decode_leg(dev, world, rank)
    video_leg = None if args.no_video else video_e2e_leg(model, dev, world, rank)
    eager_leg = None
    if world == 1 and not args.no_eager:
        model._graphs.clear()
        model._ws.clear()
        torch.cuda.empty_cache()
        eager_leg = gpu_eager_reference(dev, host)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    fl = model.step_flops(b, plan)
    n_attn = cfg.num_layers + cfg.num_single_layers
    attn_flops_launch = fl["attention"] / n_attn
    if lay is not None:   # per rank: one CFG branch, Hp/sp (padded) heads of the 30
        attn_flops_launch = 4.0 * 64 * (model._hp // lay.sp) * (plan.allowed_pairs / b)
    achieved = attn_flops_launch / (attn_avg * 1e-3) / 1e12 if attn_avg > 0 else None
    peak = peaks["tflops_sustained"]
    h2d = sum(x.numel() * x.element_size() for x in host["clips"]) + sum(
        host[k].numel() * host[k].element_size() for k in ("enc", "mask", "pooled", "t"))
    d2h = out_host.numel() * out_host.element_size()
    # which attention kernel the step launched: the three-q-tile kernel unless the launches carry peer stores (SP > 1)
    triple = bool(_lib.get_option(_lib.PF_OPT_ATTN_TRIPLE_KERNEL)) and (lay is None or lay.sp == 1) and args.attn_variant in (None, 0, 0x20)
    attn_kernel_name = ("pf::attn3q_fwd_kernel (masked joint attention, three q tiles per CTA, 64-column kv steps, tcgen05)" if triple
                        else "pf::attn2_fwd_kernel (masked joint attention, two q tiles per CTA, tcgen05)")
    line = {
        "metric": METRIC, "value": tokens / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": b, "seq_len": plan.seq,
                   "parallelism": ("single GPU" if world == 1 else
                                   f"cfg{lay.cfg_ways} x sp{lay.sp}: CFG pair split first, then Ulysses sequence parallel "
                                   f"(heads 30 -> {model._hp}); exchange = " +
                                   ("remote stores fused into the QKV-GEMM / attention epilogues over NVLink peer memory + "
                                    "flag barriers, no NCCL call in the step" if args.exchange == "peer" else
                                    "NCCL all_to_all_single each side of attention")),
                   "layers": list(args.layers), "l2": "per-step working set (>1.5 GB of activations + 3.9 GB weights) exceeds the 126 MB L2; no explicit flush",
                   "step_tflop": {"gemm": fl["gemm"] / 1e12, "attention_masked": fl["attention"] / 1e12},
                   "step_tflops_achieved": (fl["gemm"] + fl["attention"]) / (ms_step * 1e-3) / 1e12,
                   "launch_mode": ("CUDA graph replay of the step's launch sequence (captured once in warm-up), no per-launch "
                                   "instrumentation in the timed region; roofline launch durations from the host-launched "
                                   "steps timed right after"
                                   if use_graph else "host-launched (one C-ABI call per kernel), no per-launch instrumentation"),
                   "ms_per_step_host_launched": ms_eager,
                   # host wall time to enqueue one step of the timed region (rank 0): close to ms_per_step = launch-bound
                   "host_enqueue_ms_per_step": host_enqueue_ms,
                   "breakdown_ms_one_step": {k_: round(v_, 3) for k_, v_ in sorted(breakdown.items())}},
        "clocks": clocks,
        "e2e": {"value": tokens / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "B200FluxTransformer.__call__(sample=[clips], timestep_ratio, encoder_hidden_states, encoder_attention_mask, pooled_projections) with pinned host inputs, result copied back to host"},
        "gpu_launches": launches,
        "parity_vs_n1": parity_vs_n1,
        "vae_decode": vae_leg, "video_e2e": video_leg, "gpu_eager_baseline": eager_leg,
        "roofline": {"kernel": attn_kernel_name, "bound": "tensor",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None,
                     "peak_source": peaks["source"] + ", sustained cuBLAS bf16 (kernel timed inside a long step)",
                     "launches_timed": len(attn_ms), "avg_launch_ms": attn_avg,
                     "share_of_step": (attn_avg * n_attn / ms_eager) if ms_eager else None,
                     "algorithmic_flops_per_launch": attn_flops_launch,
                     # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel at this
                     # shape (profiles/r02_attn2_final_ncu.txt) -- the algorithmic bytes are Q+K+V+O
                     "traffic": ATTN_TRAFFIC_BYTES if (lay is None and not triple) else None, "traffic_unit": "B/launch",
                     "traffic_note": ("no ncu capture of the three-q-tile kernel (GPU budget of the round spent); the two-q-tile "
                                      "kernel at this shape: 460.7 MB = Q+K+V+O once (profiles/r02_attn2_final_ncu.txt)") if triple else None,
                     "algorithmic_bytes_per_launch": 4.0 * b * plan.seq * cfg.inner_dim * 2},
    }
    if args.no_cpu:
        line["cpu_baseline"] = None
    else:
        cb = cpu_reference_sample()
        line["cpu_baseline"] = {"value": cb["tokens_per_s"], "unit": UNIT, "cores": cb["threads"], "kind": "port",
                                "sample": cb["sample"] + f" ({cb['sample_s']:.1f} s measured)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, nargs=2, default=[8, 16], help="(debug) double/single block counts")
    ap.add_argument("--no-cpu", action="store_true", help="(debug) skip the CPU baseline leg")
    ap.add_argument("--no-graph", action="store_true", help="(debug) launch every kernel from the host instead of replaying the captured CUDA graph")
    ap.add_argument("--model", default="flux", choices=["flux", "mmdit"], help="flux = miniFLUX (the headline, configs[2]); mmdit = SD3 MMDiT 768p/5s (configs[4])")
    ap.add_argument("--exchange", default=None, choices=["peer", "nccl"], help="N>1: peer-memory fused exchange (default) or NCCL all-to-all (A/B)")
    ap.add_argument("--attn-variant", type=lambda x: int(x, 0), default=None, help="(debug) pf_attn_desc.variant of the DiT's attention launches")
    ap.add_argument("--attn-phase", type=int, default=None, help="(debug) pf_set_option(PF_OPT_ATTN_TILE_PHASE, clocks)")
    ap.add_argument("--no-vae", action="store_true", help="skip the VAE decode leg")
    ap.add_argument("--no-video", action="store_true", help="skip the 768p/10s end-to-end sampler + decode leg (~1 min at N=1)")
    ap.add_argument("--no-eager", action="store_true", help="skip the reference-eager-on-GPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    elif args.model == "mmdit":
        run_mmdit(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
