"""ORACLE (test infrastructure, not product code): plain-PyTorch restatement of the reference causal-VAE VIDEO encode.

Extends oracle/vae_oracle.py (the un-chunked encoder `encode_moments`) with the two paths CausalVideoVAE.encode
(video_vae/modeling_causal_vae.py:274-308) takes for videos and large frames:
  * `chunk_encode_moments` = chunk_encode (V:311-341): the encoder runs chunk by chunk and every causal conv carries a front
    cache (C:126-143).  Unlike the decoder, this is NOT always equal to the whole-clip encode: in a later chunk the stride-2
    temporal down-samplers read only the last cached frame (C:140-141), so only windows that are multiples of
    2^(temporal down-samplers) reproduce the whole clip, and other windows can return fewer latent frames.
  * `tiled_encode` = tiled_encode (V:409-466) with blend_v / blend_h (V:397-407).
Pinned to the unmodified reference by oracle/pin/make_golden_video.py -> tests/golden/vae_encode_video.pt.

Only tests/ and tools/ may import this module.
"""
from __future__ import annotations

from typing import Dict

import torch
import torch.nn.functional as F

from oracle.vae_oracle import (Params, VaeEncoderConfig, _blend_h, _blend_v, causal_group_norm, encode_moments,
                               mid_attention)


def chunk_bounds(n_frames: int, window_size: int):
    """Temporal chunks [a, b) of CausalVideoVAE.chunk_encode (V:314-327): window_size + 1 frames, full windows, remainder."""
    init = window_size + 1
    bounds = [(0, min(init, n_frames))]
    fid = init
    for _ in range((n_frames - init) // window_size):
        bounds.append((fid, fid + window_size))
        fid += window_size
    if fid < n_frames:
        bounds.append((fid, n_frames))
    return bounds


def _cached_conv3d(p: Params, pre: str, x: torch.Tensor, cache: Dict[str, torch.Tensor], first: bool,
                   stride=(1, 1, 1)) -> torch.Tensor:
    """CausalConv3d.forward with temporal_chunk=True (C:126-145): the first chunk is zero-padded in front; a later chunk is
    prefixed with the 2 cached frames (stride 1) or the last cached frame only (temporal stride 2); the cache becomes the
    last 2 frames of the conv's (padded / prefixed) input.  1x1x1 convs use no cache."""
    w, b = p[pre + ".conv.weight"], p.get(pre + ".conv.bias")
    kt, kh, kw = w.shape[2:]
    x = F.pad(x, (kw // 2, kw // 2, kh // 2, kh // 2, 0, 0))
    if kt == 3:
        if first:
            x = F.pad(x, (0, 0, 0, 0, 2, 0))
        else:
            x = torch.cat([cache[pre] if stride[0] == 1 else cache[pre][:, :, -1:], x], dim=2)
        cache[pre] = x[:, :, -2:]
    return F.conv3d(x, w, b, stride=stride)


def _cached_resnet_block(p: Params, pre: str, x: torch.Tensor, groups: int, cache, first: bool) -> torch.Tensor:
    h = _cached_conv3d(p, pre + ".conv1", F.silu(causal_group_norm(p, pre + ".norm1", x, groups)), cache, first)
    h = _cached_conv3d(p, pre + ".conv2", F.silu(causal_group_norm(p, pre + ".norm2", h, groups)), cache, first)
    if (pre + ".conv_shortcut.conv.weight") in p:
        x = _cached_conv3d(p, pre + ".conv_shortcut", x, cache, first)
    return x + h


def chunk_encode_moments(p: Params, cfg: VaeEncoderConfig, x: torch.Tensor, window_size: int) -> torch.Tensor:
    """CausalVideoVAE.chunk_encode (V:311-341): the encoder + quant_conv run chunk by chunk with every causal conv's front
    cache.  Equal to encode_moments when window_size is a multiple of 2^(temporal down-samplers); otherwise the stride-2
    cache rule changes the result and may drop latent frames."""
    g = cfg.norm_num_groups
    cache: Dict[str, torch.Tensor] = {}
    outs = []
    for k, (a, b) in enumerate(chunk_bounds(x.shape[2], window_size)):
        first = k == 0
        h = _cached_conv3d(p, "encoder.conv_in", x[:, :, a:b], cache, first)
        for i in range(len(cfg.block_out_channels)):
            for j in range(cfg.layers_per_block[i]):
                h = _cached_resnet_block(p, f"encoder.down_blocks.{i}.resnets.{j}", h, g, cache, first)
            if cfg.spatial_down_sample[i]:
                h = _cached_conv3d(p, f"encoder.down_blocks.{i}.downsamplers.0.conv", h, cache, first, stride=(1, 2, 2))
            if cfg.temporal_down_sample[i]:
                h = _cached_conv3d(p, f"encoder.down_blocks.{i}.temporal_downsamplers.0.conv", h, cache, first,
                                   stride=(2, 1, 1))
        h = _cached_resnet_block(p, "encoder.mid_block.resnets.0", h, g, cache, first)
        h = mid_attention(p, "encoder.mid_block.attentions.0", h, g)
        h = _cached_resnet_block(p, "encoder.mid_block.resnets.1", h, g, cache, first)
        h = _cached_conv3d(p, "encoder.conv_out", F.silu(causal_group_norm(p, "encoder.conv_norm_out", h, g)), cache, first)
        outs.append(_cached_conv3d(p, "quant_conv", h, cache, first))
    return torch.cat(outs, dim=2)


def tiled_encode(p: Params, cfg: VaeEncoderConfig, x: torch.Tensor, tile_sample_min_size: int = 256,
                 overlap_factor: float = 0.25, downsample: int = 8, window_size=None) -> torch.Tensor:
    """CausalVideoVAE.tiled_encode (V:409-466) with blend_v/blend_h (V:397-407) -> moments [B, 2*latent, T', h, w]; each
    tile is encoded whole, or by chunk_encode_moments when window_size is given (temporal_chunk=True)."""
    tile_latent = int(tile_sample_min_size / downsample)
    overlap = int(tile_sample_min_size * (1 - overlap_factor))
    extent = int(tile_latent * overlap_factor)
    limit = tile_latent - extent
    rows = []
    for i in range(0, x.shape[3], overlap):
        row = []
        for j in range(0, x.shape[4], overlap):
            tile = x[:, :, :, i:i + tile_sample_min_size, j:j + tile_sample_min_size]
            row.append(encode_moments(p, cfg, tile) if window_size is None else chunk_encode_moments(p, cfg, tile, window_size))
        rows.append(row)
    out_rows = []
    for i, row in enumerate(rows):
        res = []
        for j, tile in enumerate(row):
            if i > 0:
                tile = _blend_v(rows[i - 1][j], tile, extent)
            if j > 0:
                tile = _blend_h(row[j - 1], tile, extent)
            res.append(tile[:, :, :, :limit, :limit])
        out_rows.append(torch.cat(res, dim=4))
    return torch.cat(out_rows, dim=3)


def seeded_clips(specs, seed: int) -> Dict[str, torch.Tensor]:
    """Video inputs in [-1, 1] rounded to bf16 (the dtype the pipeline feeds the VAE), drawn in `specs` order
    [(name, shape), ...] from one CPU generator."""
    g = torch.Generator().manual_seed(seed)
    return {name: (torch.rand(tuple(shape), generator=g) * 2 - 1).bfloat16() for name, shape in specs}
