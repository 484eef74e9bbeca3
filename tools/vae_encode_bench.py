"""Video encode on one GPU with the default-width encoder (128, 256, 512, 512) x (2, 2, 2, 2), synthetic weights:

  video_chunked   121 uint8 frames of 768x1280 on the host, encode_frames_u8 with windows of 16 (the reference's
                  chunk_encode, its VAE demo's way of encoding a clip)
  i2v_tiled       one 768x1280 image, encode() with enable_tiling() and 256 px tiles: 28 tiles (the app's i2v encode)
  whole_33 / chunked_33   33 frames of 768x1280 as one chunk and in windows of 16: memory of the whole clip vs chunked

One JSON line per case: device name and power limit (read in the same run), ms per clip (CUDA events, after a warm-up
of the same shapes; median of --reps), frames/s, peak allocated GiB, and algorithmic TFLOP/s from the FLOPs of the
encoder's convs and mid-block attention counted here from the config (3 real input channels; the padding of conv_in to
64 channels is not counted).

    python tools/vae_encode_bench.py [--reps 3] [--out FILE.jsonl] [--cases video_chunked,i2v_tiled,whole_33,chunked_33]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def encoder_flops(cfg, t: int, h: int, w: int) -> int:
    """Multiply-adds x 2 of every conv of CausalVaeEncoder + quant_conv (D:149-198, V:301) and the mid-block attention
    (projections, QK^T, PV) for a clip of t frames of h x w encoded whole (= chunked with a window multiple of 8)."""
    def conv(ci, co, k, vox):
        return 2 * co * ci * k ** 3 * vox

    c0 = cfg.enc_block_out_channels[0]
    f = conv(cfg.enc_in_channels, c0, 3, t * h * w)
    prev = c0
    for i, co in enumerate(cfg.enc_block_out_channels):
        for j in range(cfg.enc_layers_per_block[i]):
            ci = prev if j == 0 else co
            f += conv(ci, co, 3, t * h * w) + conv(co, co, 3, t * h * w) + (conv(ci, co, 1, t * h * w) if ci != co else 0)
        if cfg.enc_spatial_down_sample[i]:
            h, w = h // 2, w // 2
            f += conv(co, co, 3, t * h * w)
        if cfg.enc_temporal_down_sample[i]:
            t = (t - 1) // 2 + 1
            f += conv(co, co, 3, t * h * w)
        prev = co
    c, n = prev, h * w
    f += 2 * 2 * conv(c, c, 3, t * n)                                   # two mid-block resnets
    f += t * (4 * 2 * n * c * c + 2 * 2 * n * n * c)                   # q, k, v, out projections; QK^T and PV per frame
    lat2 = 2 * cfg.latent_channels
    f += conv(c, lat2, 3, t * n) + conv(lat2, lat2, 1, t * n)           # conv_out, quant_conv
    return f


def tiled_flops(cfg, t: int, height: int, width: int, tile: int, vae_cls) -> int:
    rows, cols, _, _ = vae_cls.encode_tile_grid(height, width, tile)
    return sum(encoder_flops(cfg, t, min(tile, height - r), min(tile, width - c)) for r in rows for c in cols)


def device_info() -> dict:
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(q[0]), float(q[1])
    except Exception as e:                                              # noqa: BLE001  reported, not fatal
        info["power_limit_w"] = f"unavailable: {e}"
    return info


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--cases", default="video_chunked,i2v_tiled,whole_33,chunked_33")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vae_encode_bench measures on a CUDA GPU; none is visible")
    from oracle import vae_oracle as VO
    from pyramid_flow_b200 import _lib
    from pyramid_flow_b200.vae import B200CausalVAE, VaeConfigB200

    _lib.require_device()
    dev = torch.device("cuda:0")
    cfg = VaeConfigB200()
    ocfg = VO.VaeEncoderConfig(block_out_channels=cfg.enc_block_out_channels, layers_per_block=cfg.enc_layers_per_block)
    vae = B200CausalVAE(cfg, VO.synthetic_vae_params(ocfg, seed=0), device=dev)
    info = device_info()
    gen = torch.Generator().manual_seed(0)
    H, W = 768, 1280

    def clip(n):                                                        # bf16 [1, 3, n, H, W] on the host
        return (torch.rand(1, 3, n, H, W, generator=gen) * 2 - 1).bfloat16()

    cases = {
        "video_chunked": dict(frames=121, window=16, tile=None,
                              run=lambda x: vae.encode_frames_u8(x, window_size=16),
                              make=lambda: torch.randint(0, 256, (121, H, W, 3), generator=gen, dtype=torch.uint8)),
        "i2v_tiled": dict(frames=1, window=None, tile=256, run=lambda x: vae.encode(x, tile_sample_min_size=256),
                          make=lambda: clip(1).to(dev)),
        "whole_33": dict(frames=33, window=None, tile=None, run=lambda x: vae.encode(x), make=lambda: clip(33)),
        "chunked_33": dict(frames=33, window=16, tile=None, run=lambda x: vae.encode(x, temporal_chunk=True, window_size=16),
                           make=lambda: clip(33)),
    }
    lines = []
    for name in args.cases.split(","):
        c = cases[name]
        x = c["make"]()
        vae.enable_tiling(c["tile"] is not None)
        c["run"](x)                                                     # warm-up: same shapes
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        times = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = c["run"](x).latent_dist.parameters
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        ms = sorted(times)[len(times) // 2]
        flops = (tiled_flops(cfg, c["frames"], H, W, c["tile"], B200CausalVAE) if c["tile"]
                 else encoder_flops(cfg, c["frames"], H, W))
        rec = {"case": name, **info, "frames": c["frames"], "height": H, "width": W, "window_size": c["window"],
               "tile_sample_min_size": c["tile"], "input": "uint8 host" if x.dtype == torch.uint8 else
               f"bf16 {'device' if x.is_cuda else 'host'}", "latent_shape": list(out.shape), "reps": args.reps,
               "ms_per_clip": round(ms, 2), "ms_all": [round(t, 2) for t in times],
               "frames_per_s": round(c["frames"] / (ms / 1e3), 2),
               "peak_alloc_gib": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2),
               "gflop": round(flops / 1e9, 1), "mflop_per_pixel_frame": round(flops / (c["frames"] * H * W) / 1e6, 3),
               "tflops": round(flops / (ms / 1e3) / 1e12, 1)}
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
        del x, out
        torch.cuda.empty_cache()
    vae.disable_tiling()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
