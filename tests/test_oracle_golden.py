"""The oracle restatement (oracle/flux_oracle.py) against fixtures produced by the UNMODIFIED reference
(oracle/pin/make_golden.py, run where /root/reference exists).  CPU only."""
import torch

from oracle import flux_oracle as FO


def _load(golden_dir, name):
    return torch.load(golden_dir / name, weights_only=False)


def test_flux_small_forward_matches_reference(golden_dir):
    g = _load(golden_dir, "flux_small.pt")
    cfg = FO.FluxConfig(**g["cfg"])
    p = FO.synthetic_flux_params(cfg, seed=g["param_seed"])
    with torch.no_grad():
        out = FO.flux_forward(p, cfg, g["clips"], g["timestep"], g["enc"], g["mask"], g["pooled"])
        out_full = FO.flux_forward(p, cfg, g["clips"], g["timestep"], g["enc"], torch.ones_like(g["mask"]), g["pooled"])
        out_first = FO.flux_forward(p, cfg, [g["clips"][-1]], g["timestep"] * 0.5, g["enc"], g["mask"], g["pooled"])
    # fp32 vs fp32 on the same machine class: only summation-order noise is allowed
    assert (out - g["out"]).abs().max().item() < 2e-5
    assert (out_full - g["out_full_mask"]).abs().max().item() < 2e-5
    assert (out_first - g["out_first"]).abs().max().item() < 2e-5
    # the ragged mask must matter for the sample that has padded text (otherwise the mask test is vacuous)
    assert (g["out"][0] - g["out_full_mask"][0]).abs().max().item() > 1e-3
    assert g["out"].abs().mean().item() > 0.1  # non-degenerate (the reference's own init would give exactly 0)


def test_config1_blocks_match_reference(golden_dir):
    """BASELINE.json configs[0]: one double + one single miniFLUX block, D=1920/H=30, 256 video + 77 text tokens, fp32."""
    g = _load(golden_dir, "flux_block_cfg1.pt")
    cfg = FO.FluxConfig(num_layers=1, num_single_layers=1)
    p = FO.synthetic_flux_params(cfg, seed=0)
    d, heads = cfg.inner_dim, cfg.num_attention_heads
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(1, 256, d, generator=gen)
    ctx = torch.randn(1, 77, d, generator=gen)
    temb = torch.randn(1, d, generator=gen)
    ids = torch.cat([torch.zeros(77, 3), FO.clip_ids(1, 16, 16, 16, 16, 0)], 0)
    cs = FO.rope_table(ids, cfg.axes_dims_rope)
    mask = torch.ones(1, 1, 333, 333, dtype=torch.bool)
    with torch.no_grad():
        c_out, x_out = FO.double_block(p, "transformer_blocks.0", x, ctx, temb, cs, mask, heads)
        s_out = FO.single_block(p, "single_transformer_blocks.0", torch.cat([ctx, x], 1), temb, cs, mask, heads)
    assert (x_out[:, ::16] - g["x_out_rows"]).abs().max().item() < 5e-5
    assert (c_out[:, ::16] - g["c_out_rows"]).abs().max().item() < 5e-5
    assert (s_out[:, ::16] - g["s_out_rows"]).abs().max().item() < 5e-5
    assert (x_out.mean(-1) - g["x_out_mean"]).abs().max().item() < 5e-5
    assert (s_out.mean(-1) - g["s_out_mean"]).abs().max().item() < 5e-5


def test_mask_restatement_matches_dense_definition():
    seg = torch.tensor([[0, 1, 1, 1, 1, 1]])
    t = torch.tensor([0.0, 0.0, 0.0, 1.0, 1.0, 2.0])
    m = FO.attention_mask(seg, t)[0, 0]
    assert m[1].tolist() == [False, True, True, False, False, False]
    assert m[5].tolist() == [False, True, True, True, True, True]
    assert m[0].tolist() == [True, False, False, False, False, False]


def test_vae_decode_oracle_matches_reference(golden_dir):
    from oracle import vae_oracle as VO
    g = _load(golden_dir, "vae_small.pt")
    cfg = VO.VaeDecoderConfig(**g["cfg"])
    p = VO.synthetic_vae_params(cfg, seed=g["param_seed"])
    with torch.no_grad():
        out = VO.decode(p, cfg, g["z"])
        tiled = VO.tiled_decode(p, cfg, g["z"], tile_sample_min_size=32)
    assert out.shape == g["full"].shape == (1, 3, 17, 48, 80)
    assert (out - g["full"]).abs().max().item() < 5e-5
    # the reference's own temporal chunking (window 1 and 2) reproduces its un-chunked decode => one oracle serves both
    assert g["chunk1_maxdiff"] < 1e-4 and g["chunk2_maxdiff"] < 1e-4
    assert tuple(tiled.shape) == g["tiled32_shape"]
    assert (tiled.flatten()[::g["tiled32_stride"]] - g["tiled32_sample"]).abs().max().item() < 5e-5
    assert g["full"].abs().mean().item() > 0.05


def test_vae_encode_oracle_matches_reference(golden_dir):
    """Encoder + quant_conv (stride-2 spatial / temporal causal convs) against the unmodified reference's moments."""
    from oracle import vae_oracle as VO
    g = _load(golden_dir, "vae_encoder_small.pt")
    cfg = VO.VaeEncoderConfig(**g["cfg"])
    p = VO.synthetic_vae_params(cfg, seed=g["param_seed"])
    with torch.no_grad():
        m_image = VO.encode_moments(p, cfg, g["image"])
        m_clip = VO.encode_moments(p, cfg, g["clip"])
    assert m_image.shape == g["moments_image"].shape == (1, 32, 1, 8, 12)
    assert m_clip.shape == g["moments_clip"].shape == (1, 32, 2, 4, 6)
    assert (m_image - g["moments_image"]).abs().max().item() < 5e-5
    assert (m_clip - g["moments_clip"]).abs().max().item() < 5e-5
    mean, logvar = m_image.chunk(2, dim=1)
    assert (mean - g["mean_image"]).abs().max().item() < 5e-5
    assert (logvar.clamp(-30.0, 20.0) - g["logvar_image"]).abs().max().item() < 5e-5
    assert g["moments_image"].abs().mean().item() > 0.05


def test_mmdit_small_forward_matches_reference(golden_dir):
    from oracle import mmdit_oracle as MO
    g = _load(golden_dir, "mmdit_small.pt")
    cfg = MO.MMDiTConfig(**g["cfg"])
    p = MO.synthetic_mmdit_params(cfg, seed=g["param_seed"])
    with torch.no_grad():
        out = MO.mmdit_forward(p, cfg, g["clips"], g["timestep"], g["enc"], g["mask"], g["pooled"])
    assert (out - g["out"]).abs().max().item() < 2e-5
    assert g["out"].abs().mean().item() > 0.1
