"""Video encode without a GPU: the oracle's chunk_encode / tiled_encode restatements against the unmodified reference's
outputs (tests/golden/vae_encode_video.pt), and the chunk / tile geometry B200CausalVAE uses against the reference's
formulas (V:311-327, V:429-438)."""
import pytest
import torch

from oracle import vae_oracle as VO
from oracle import vae_video_oracle as VVO
from pyramid_flow_b200.vae import B200CausalVAE

# fp32 CPU restatement vs the fp32 CPU reference: only summation order differs (the reference's own chunked-vs-whole
# difference is 3.3e-6 on these moments, |moments| ~ 1)
TOL = 1e-4


@pytest.fixture(scope="module")
def gold(golden_dir):
    g = torch.load(golden_dir / "vae_encode_video.pt", weights_only=False)
    cfg = VO.VaeEncoderConfig(**g["cfg"])
    params = VO.synthetic_vae_params(cfg, seed=g["param_seed"])
    x = VVO.seeded_clips(g["inputs"], g["input_seed"])
    for k, v in x.items():
        assert abs(float(v.double().sum()) - g["input_sums"][k]) < 1e-6, f"regenerated input {k} drifted"
    return g, cfg, params, {k: v.float() for k, v in x.items()}


def test_chunk_bounds_match_reference(golden_dir):
    g = torch.load(golden_dir / "vae_encode_video.pt", weights_only=False)
    for n, w, lens in ((33, 8, g["chunk8_lens"]), (25, 12, g["chunk12_lens"])):
        assert [b - a for a, b in VVO.chunk_bounds(n, w)] == lens
    for n in (1, 9, 17, 25, 33, 121, 241):
        for w in (1, 2, 5, 8, 12, 16, 64, 300):
            ours = B200CausalVAE.chunk_bounds(n, w)
            assert ours == VVO.chunk_bounds(n, w), (n, w)
            assert ours[0][0] == 0 and ours[-1][1] == n and all(a[1] == b[0] for a, b in zip(ours, ours[1:]))


def test_chunk_encode_matches_reference(gold):
    g, cfg, params, x = gold
    with torch.no_grad():
        c8 = VVO.chunk_encode_moments(params, cfg, x["clip33"], 8)
        whole = VO.encode_moments(params, cfg, x["clip33"])
        c12 = VVO.chunk_encode_moments(params, cfg, x["clip25"], 12)
    assert c8.shape == g["chunk8"].shape == (1, 32, 5, 4, 6)
    assert (c8 - g["chunk8"]).abs().max().item() < TOL
    # a window that is a multiple of the 8x temporal down-sampling reproduces the whole clip
    assert (c8 - whole).abs().max().item() < TOL and g["chunk8_maxdiff"] < TOL
    # window 12: the stride-2 convs read only the last cached frame, so the result differs and has fewer latent frames
    assert c12.shape == g["chunk12"].shape == (1, 32, 3, 4, 6) and g["whole25_shape"] == (1, 32, 4, 4, 6)
    assert (c12 - g["chunk12"]).abs().max().item() < TOL
    assert c12.abs().mean().item() > 0.1


def test_tiled_encode_matches_reference(gold):
    g, cfg, params, x = gold
    with torch.no_grad():
        img = VVO.tiled_encode(params, cfg, x["image"], tile_sample_min_size=64)
        clip = VVO.tiled_encode(params, cfg, x["clip17"], tile_sample_min_size=64)
        clip8 = VVO.tiled_encode(params, cfg, x["clip17"], tile_sample_min_size=64, window_size=8)
        untiled = VO.encode_moments(params, cfg, x["image"])
    for ours, ref in ((img, g["tiled64_image"]), (clip, g["tiled64_clip"]), (clip8, g["tiled64_clip_chunk8"])):
        assert ours.shape == ref.shape and (ours - ref).abs().max().item() < TOL
    assert img.shape == untiled.shape == (1, 32, 1, 12, 20)
    # tiles see less context than the whole frame: the tiled latent is a different one (the reason encode() must tile)
    assert (img - untiled).abs().max().item() > 1e-2


@pytest.mark.parametrize("tile", [256, 512])
def test_encode_tile_grid_768x1280(tile):
    rows, cols, extent, limit = B200CausalVAE.encode_tile_grid(768, 1280, tile)
    stride = int(tile * (1 - 0.25))                       # V:429-431
    assert rows == list(range(0, 768, stride)) and cols == list(range(0, 1280, stride))
    assert extent == int(tile // 8 * 0.25) and limit == tile // 8 - extent
    if tile == 256:
        assert (len(rows), len(cols)) == (4, 7)          # 28 tiles; the last row is 192 px, the last column 128 px
        assert (768 - rows[-1], 1280 - cols[-1]) == (192, 128) and (extent, limit) == (8, 24)
    else:
        assert (len(rows), len(cols)) == (2, 4) and (768 - rows[-1], 1280 - cols[-1]) == (384, 128)
    # the cropped tiles tile the latent frame exactly
    crop = lambda starts, size: sum(min(limit, min(tile, size - s) // 8) for s in starts)   # noqa: E731
    assert (crop(rows, 768), crop(cols, 1280)) == (96, 160)
