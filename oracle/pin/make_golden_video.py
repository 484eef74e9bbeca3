"""Generate tests/golden/vae_encode_video.pt by running the UNMODIFIED reference's video encode (imported through ref_shim).

    PF_REFERENCE_ROOT=/path/to/Pyramid-Flow python oracle/pin/make_golden_video.py [vae_encode_video]

(or with the reference staged by oracle/pin/stage_reference.py).  Same model and conventions as make_golden.py's
`vae_encoder` target: the small encoder config with synthetic parameters (seed 1), CPU, fp32.
"""
from __future__ import annotations

import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[2]))
from oracle.pin.make_golden import GOLD, VAE_ENC_SMALL  # noqa: E402  (installs the reference shim)

VAE_ENCODE_VIDEO_INPUTS = [("clip33", (1, 3, 33, 32, 48)), ("clip25", (1, 3, 25, 32, 48)), ("image", (1, 3, 1, 96, 160)),
                           ("clip17", (1, 3, 17, 96, 160))]


def make_vae_encode_video():
    """Video encode of the vae_encoder model: chunk_encode (V:311-341) at window 8 with a partial last chunk (33 = 9+8+8+8
    frames) and at window 12 (25 = 13+12 frames; not a multiple of the 8x temporal down-sampling, so the stride-2 cache
    rule C:140-141 shows), and tiled_encode (V:409-466) with 64 px tiles on 96x160 frames (2x4 tiles, ragged last row and
    column), for one image and for a 17-frame clip with and without temporal_chunk.  Inputs are regenerated from
    seeded_clips(VAE_ENCODE_VIDEO_INPUTS, input_seed); their float64 sums are stored to detect drift."""
    from video_vae import CausalVideoVAE
    from oracle import vae_oracle as VO
    from oracle import vae_video_oracle as VVO
    cfg = VO.VaeEncoderConfig(**VAE_ENC_SMALL)
    params = VO.synthetic_vae_params(cfg, seed=1)
    vae = CausalVideoVAE(encoder_out_channels=16, decoder_in_channels=16, encoder_block_out_channels=cfg.block_out_channels,
                         encoder_layers_per_block=cfg.layers_per_block, decoder_block_out_channels=(32, 32, 32, 32),
                         decoder_layers_per_block=(1, 1, 1, 1)).eval()
    sd = vae.state_dict()
    sd.update(params)
    vae.load_state_dict(sd, strict=True)
    seed = 6
    x = VVO.seeded_clips(VAE_ENCODE_VIDEO_INPUTS, seed)
    lens = []
    enc_forward = vae.encoder.forward

    def recording_forward(sample, *a, **k):       # records the frames of every encoder call = the chunk lengths
        lens.append(sample.shape[2])
        return enc_forward(sample, *a, **k)

    vae.encoder.forward = recording_forward
    out = {"cfg": VAE_ENC_SMALL, "param_seed": 1, "input_seed": seed, "inputs": VAE_ENCODE_VIDEO_INPUTS,
           "input_sums": {k: float(v.double().sum()) for k, v in x.items()}}
    with torch.no_grad():
        f = lambda t: t.float()                   # noqa: E731  the reference runs in fp32 on the bf16-rounded input
        whole33 = vae.encode(f(x["clip33"])).latent_dist.parameters
        lens.clear()
        out["chunk8"] = vae.encode(f(x["clip33"]), temporal_chunk=True, window_size=8).latent_dist.parameters
        out["chunk8_lens"] = list(lens)
        out["chunk8_maxdiff"] = float((out["chunk8"] - whole33).abs().max())
        lens.clear()
        out["chunk12"] = vae.encode(f(x["clip25"]), temporal_chunk=True, window_size=12).latent_dist.parameters
        out["chunk12_lens"] = list(lens)
        out["whole25_shape"] = tuple(vae.encode(f(x["clip25"])).latent_dist.parameters.shape)
        vae.enable_tiling()
        out["tiled64_image"] = vae.encode(f(x["image"]), tile_sample_min_size=64).latent_dist.parameters
        out["tiled64_clip"] = vae.encode(f(x["clip17"]), tile_sample_min_size=64).latent_dist.parameters
        out["tiled64_clip_chunk8"] = vae.encode(f(x["clip17"]), temporal_chunk=True, window_size=8,
                                                tile_sample_min_size=64).latent_dist.parameters
    print("vae_encode_video: chunk8", tuple(out["chunk8"].shape), out["chunk8_lens"], "max|chunked - whole|",
          out["chunk8_maxdiff"], "| chunk12", tuple(out["chunk12"].shape), out["chunk12_lens"], "whole",
          out["whole25_shape"], "| tiled", tuple(out["tiled64_image"].shape), tuple(out["tiled64_clip_chunk8"].shape))
    torch.save(out, GOLD / "vae_encode_video.pt")


if __name__ == "__main__":
    for w in sys.argv[1:] or ["vae_encode_video"]:
        globals()["make_" + w]()
