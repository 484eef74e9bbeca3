"""Video encode on the B200: chunked encode (chunk_encode V:311-341 with the causal convs' front cache C:126-143), tiled
encode (tiled_encode V:409-466) and the uint8 frame path, against the whole-clip encode, the unmodified reference's
outputs (tests/golden/vae_encode_video.pt) and the oracle."""
import pytest
import torch

from oracle import vae_oracle as VO
from oracle import vae_video_oracle as VVO

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _vae(cfg, params):
    from pyramid_flow_b200.vae import B200CausalVAE, VaeConfigB200
    return B200CausalVAE(VaeConfigB200(enc_block_out_channels=cfg.block_out_channels,
                                       enc_layers_per_block=cfg.layers_per_block), params, device=DEV)


@pytest.fixture(scope="module")
def small(golden_dir):
    g = torch.load(golden_dir / "vae_encode_video.pt", weights_only=False)
    cfg = VO.VaeEncoderConfig(**g["cfg"])
    params = VO.synthetic_vae_params(cfg, seed=g["param_seed"])
    return g, cfg, params, _vae(cfg, params)


def _moments(vae, x, **kw):
    out = vae.encode(x, **kw).latent_dist.parameters
    torch.cuda.synchronize()
    return out


def test_chunked_encode_equals_whole_clip_bit_for_bit(small):
    """Windows that are multiples of the 8x temporal down-sampling put every chunk boundary on a stride-2 output boundary
    at every level; GroupNorm statistics are per frame and every conv accumulates in the same K order, so the chunked
    moments are the whole-clip moments exactly.  41 frames: window 8 = 9+8+8+8+8, window 16 = 17+16+8 (partial)."""
    _, _, _, vae = small
    x = VVO.seeded_clips([("x", (2, 3, 41, 32, 48))], seed=21)["x"]          # on the host
    whole = _moments(vae, x)
    assert whole.shape == (2, 32, 6, 4, 6)
    for w in (8, 16):
        chunked = _moments(vae, x, temporal_chunk=True, window_size=w)
        assert torch.equal(chunked, whole), (w, (chunked.float() - whole.float()).abs().max().item())
    assert torch.equal(_moments(vae, x.to(DEV), temporal_chunk=True, window_size=16), whole)
    assert whole.float().abs().mean().item() > 0.1


def test_encode_video_matches_reference(small):
    """chunk_encode at windows 8 and 12 (not a multiple of 8: the stride-2 cache rule, one latent frame fewer than the whole
    clip) and tiled_encode with 64 px tiles with and without chunking, vs the reference golden (< 6e-2) and the fp32
    oracle (no worse than 1.5x the reference's own bf16 policy), the bounds of the single-image encoder test."""
    g, cfg, params, vae = small
    x = VVO.seeded_clips(g["inputs"], g["input_seed"])
    pd = {k: v.to(DEV) for k, v in params.items()}
    cases = [
        ("chunk8", "clip33", dict(temporal_chunk=True, window_size=8), dict(window_size=8)),
        ("chunk12", "clip25", dict(temporal_chunk=True, window_size=12), dict(window_size=12)),
        ("tiled64_image", "image", dict(tile_sample_min_size=64), dict(tile_sample_min_size=64)),
        ("tiled64_clip", "clip17", dict(tile_sample_min_size=64), dict(tile_sample_min_size=64)),
        ("tiled64_clip_chunk8", "clip17", dict(temporal_chunk=True, window_size=8, tile_sample_min_size=64),
         dict(tile_sample_min_size=64, window_size=8)),
    ]

    def oracle(p, inp, okw):
        if "tile_sample_min_size" in okw:
            return VVO.tiled_encode(p, cfg, inp, **okw)
        return VVO.chunk_encode_moments(p, cfg, inp, okw["window_size"])

    vae.enable_tiling()
    try:
        for name, inp, kw, okw in cases:
            ours = _moments(vae, x[inp], **kw).float().cpu()
            with torch.no_grad():
                ref = oracle(params, x[inp].float(), okw)
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    ref_bf16 = oracle(pd, x[inp].to(DEV), okw).float().cpu()
            err = (ours - ref).abs().max().item()
            err_gold = (ours - g[name]).abs().max().item()
            err_pol = (ref_bf16 - ref).abs().max().item()
            print(f"vae encode video {name}: shape {tuple(ours.shape)} max_abs vs oracle {err:.3e}, vs reference golden "
                  f"{err_gold:.3e}, reference bf16 policy {err_pol:.3e}, |ref| mean {ref.abs().mean():.3f}")
            assert ours.shape == ref.shape == g[name].shape
            assert err_gold < 6e-2 and err <= max(1.5 * err_pol, 1e-2)
    finally:
        vae.disable_tiling()


def test_default_width_chunked_encode_matches_oracle():
    """The default encoder width (128, 256, 512, 512) x (2, 2, 2, 2): 33 frames at 128x192 in windows of 16 vs the fp32
    oracle on the same GPU (TF32 off), at least as close as the oracle under bf16 autocast."""
    cfg = VO.VaeEncoderConfig()
    params = VO.synthetic_vae_params(cfg, seed=2)
    x = VVO.seeded_clips([("x", (1, 3, 33, 128, 192))], seed=22)["x"]
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    pd = {k: v.to(DEV) for k, v in params.items()}
    with torch.no_grad():
        ref = VO.encode_moments(pd, cfg, x.to(DEV).float()).float().cpu()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ref_bf16 = VO.encode_moments(pd, cfg, x.to(DEV)).float().cpu()
    del pd
    vae = _vae(cfg, params)
    ours = _moments(vae, x, temporal_chunk=True, window_size=16).float().cpu()
    err, mse = (ours - ref).abs().max().item(), ((ours - ref) ** 2).mean().item()
    e2, m2 = (ref_bf16 - ref).abs().max().item(), ((ref_bf16 - ref) ** 2).mean().item()
    print(f"vae encode default width: ours vs fp32 oracle max_abs {err:.3e} mse {mse:.3e} | bf16-autocast oracle vs fp32 "
          f"{e2:.3e} mse {m2:.3e} | |ref| mean {ref.abs().mean():.3f}")
    assert ours.shape == ref.shape == (1, 32, 5, 16, 24)
    # measured on a B200: max-abs 3.22e-2, mse 3.20e-5 (bf16-autocast oracle: 4.83e-2 / 5.28e-5); thresholds x 1.3
    assert err < 4.2e-2 and mse < 4.2e-5
    assert err <= e2 and mse <= m2
    assert ref.abs().mean().item() > 0.05


def test_encode_frames_u8_equals_encode_of_normalised_frames(small):
    """pf_pack_frames_u8 == ToTensor + Normalize(0.5, 0.5) in torch, cast to bf16, through encode(): bit for bit, chunked
    and tiled, from host or device frames, batched or not."""
    _, _, _, vae = small
    gen = torch.Generator().manual_seed(23)
    frames = torch.randint(0, 256, (2, 17, 64, 96, 3), generator=gen, dtype=torch.uint8)
    x = ((frames.float() / 255 - 0.5) / 0.5).permute(0, 4, 1, 2, 3).bfloat16()      # [B, 3, T, H, W]
    for tiled in (False, True):
        vae.enable_tiling(tiled)
        ref = _moments(vae, x, temporal_chunk=True, window_size=8, tile_sample_min_size=64)
        u8 = vae.encode_frames_u8(frames, window_size=8, tile_sample_min_size=64).latent_dist.parameters
        assert torch.equal(u8, ref), (tiled, (u8.float() - ref.float()).abs().max().item())
        one = vae.encode_frames_u8(frames[1].to(DEV), window_size=8, tile_sample_min_size=64).latent_dist.parameters
        assert torch.equal(one, ref[1:])
    vae.disable_tiling()
    assert u8.shape == (2, 32, 3, 8, 12)


def test_chunked_encode_memory_is_bounded_by_the_window(small):
    """With the clip on the host, the peak device memory of a chunked encode depends on the window, not the clip length."""
    _, _, _, vae = small
    peaks = {}
    for n in (17, 65):
        x = VVO.seeded_clips([("x", (1, 3, n, 256, 384))], seed=24)["x"]
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(DEV)
        m = _moments(vae, x, temporal_chunk=True, window_size=16)
        peaks[n] = torch.cuda.max_memory_allocated(DEV)
        assert m.shape[2] == (n - 1) // 8 + 1
        del m
    print(f"vae encode peak allocated: 17 frames {peaks[17] / 2**20:.1f} MiB, 65 frames {peaks[65] / 2**20:.1f} MiB")
    assert peaks[65] <= 1.15 * peaks[17], peaks


def test_unchanged_paths_are_the_whole_clip_encode(small):
    """Tiling off, or a frame no larger than the tile, and a window covering the clip: the whole-clip encode, bit for bit."""
    _, _, _, vae = small
    x = VVO.seeded_clips([("x", (2, 3, 9, 64, 96))], seed=25)["x"].to(DEV)
    whole = _moments(vae, x)
    assert torch.equal(_moments(vae, x, tile_sample_min_size=32), whole)                     # tiling off
    assert torch.equal(_moments(vae, x, is_init_image=False), whole)                         # no effect, as in the reference
    assert torch.equal(_moments(vae, x, temporal_chunk=True, window_size=8), whole)          # one chunk
    assert torch.equal(vae.encode(x, return_dict=False)[0].parameters, whole)
    vae.enable_tiling()
    try:
        assert torch.equal(_moments(vae, x, tile_sample_min_size=96), whole)                 # frame == tile
        tiled = _moments(vae, x, tile_sample_min_size=64)                                     # frame > tile: tiles
        assert tiled.shape == whole.shape and not torch.equal(tiled, whole)
    finally:
        vae.disable_tiling()
