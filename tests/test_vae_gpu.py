"""Parity of the CUDA causal-VAE decode (through the C-ABI) against the oracle / the reference's golden output. B200."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# bf16 activations through ~60 convs + 30 GroupNorms; decoded samples are O(0.5) (|ref| mean ~0.43, range ~[-2, 2]).
# Stated tolerance on the decoded sample vs the fp32 oracle: max-abs 0.1 (the max over ~2.6e5 values), MSE 1e-4
# (RMS error 1e-2), and no worse than 1.5x the error of the reference's own dtype policy (oracle under bf16 autocast).
# Measured (round 2): max-abs 5.5e-2 .. 6.1e-2, mse 5.5e-5 .. 5.9e-5 (reference bf16 policy: 6.7e-2 / 9.5e-5); thresholds x 1.3.
TOL_MAX_ABS = 8e-2
TOL_MSE = 7.7e-5


def _conv_ref(x_cl, w, b, kt):
    """x_cl [T, H, W, C] (no halo) -> causal conv, channels-last out."""
    x = x_cl.permute(3, 0, 1, 2)[None].float()
    k = w.shape[-1]
    x = F.pad(x, (k // 2, k // 2, k // 2, k // 2, kt - 1, 0))
    y = F.conv3d(x, w.float(), b.float())
    return y[0].permute(1, 2, 3, 0)


def test_conv3d_kernel_modes():
    from pyramid_flow_b200.vae import B200CausalVAE, _Conv
    torch.manual_seed(0)
    dev = torch.device("cuda:0")
    holder = B200CausalVAE.__new__(B200CausalVAE)   # only the _conv wrapper is needed
    for (ci, co, k, t, h, w) in [(64, 128, 3, 3, 6, 10), (128, 256, 3, 2, 17, 33), (256, 64, 1, 4, 9, 20), (64, 512, 3, 2, 12, 150)]:
        wt = (torch.randn(co, ci, k, k, k) * (ci * k ** 3) ** -0.5).bfloat16().float()
        bias = torch.randn(co) * 0.1
        cv = _Conv({"c.conv.weight": wt, "c.conv.bias": bias}, "c", dev)
        x = torch.randn(t, h, w, ci, device=dev).bfloat16()
        xin = torch.zeros(t + k - 1, h, w, ci, device=dev, dtype=torch.bfloat16)
        xin[k - 1:] = x
        ref = _conv_ref(x, wt.to(dev), bias.to(dev), k)
        out = torch.zeros(t, h, w, co, device=dev, dtype=torch.bfloat16)
        B200CausalVAE._conv(holder, cv, xin, t, h, w, out=out)
        torch.cuda.synchronize()
        err = (out.float() - ref).abs().max().item()
        assert err < 3e-2, (ci, co, k, err)
        # residual + halo'd output
        res = torch.randn(t, h, w, co, device=dev).bfloat16()
        out2 = torch.zeros(t + 2, h, w, co, device=dev, dtype=torch.bfloat16)
        B200CausalVAE._conv(holder, cv, xin, t, h, w, out=out2, out_t_offset=2, residual=res)
        torch.cuda.synchronize()
        assert (out2[2:].float() - (ref + res.float())).abs().max().item() < 4e-2
        assert bool((out2[:2] == 0).all())
        if co % 256 == 0 or co == 128:
            # spatial depth-to-space: 'b (c p1 p2) t h w -> b c t (h p1) (w p2)'
            o3 = torch.zeros(t, 2 * h, 2 * w, co // 4, device=dev, dtype=torch.bfloat16)
            B200CausalVAE._conv(holder, cv, xin, t, h, w, out=o3, store_mode=1)
            r3 = ref.reshape(t, h, w, co // 4, 2, 2).permute(0, 1, 4, 2, 5, 3).reshape(t, 2 * h, 2 * w, co // 4)
            torch.cuda.synchronize()
            assert (o3.float() - r3).abs().max().item() < 3e-2
            # temporal depth-to-space with the first frame dropped
            o4 = torch.zeros(2 * t - 1, h, w, co // 2, device=dev, dtype=torch.bfloat16)
            B200CausalVAE._conv(holder, cv, xin, t, h, w, out=o4, out_t_offset=-1, store_mode=2)
            r4 = ref.reshape(t, h, w, co // 2, 2).permute(0, 4, 1, 2, 3).reshape(2 * t, h, w, co // 2)[1:]
            torch.cuda.synchronize()
            assert (o4.float() - r4).abs().max().item() < 3e-2


def _ours(cfg_kw, params, z, **dec_kw):
    from pyramid_flow_b200.vae import B200CausalVAE, VaeConfigB200
    dev = torch.device("cuda:0")
    vae = B200CausalVAE(VaeConfigB200(**cfg_kw), params, device=dev)
    out = vae.decode(z.to(dev), **dec_kw).sample
    torch.cuda.synchronize()
    return out.float().cpu(), vae


def test_small_vae_matches_reference_golden(golden_dir):
    from oracle import vae_oracle as VO
    g = torch.load(golden_dir / "vae_small.pt", weights_only=False)
    cfg = VO.VaeDecoderConfig(**g["cfg"])
    params = VO.synthetic_vae_params(cfg, seed=g["param_seed"])
    z = g["z"].bfloat16().float()
    with torch.no_grad():
        ref = VO.decode(params, cfg, z)
    out, vae = _ours(g["cfg"], params, z, temporal_chunk=False)
    err, mse = (out - ref).abs().max().item(), ((out - ref) ** 2).mean().item()
    err_gold = (out - g["full"]).abs().max().item()
    print(f"vae small: max_abs vs oracle {err:.3e} mse {mse:.3e}; vs reference golden {err_gold:.3e}; |ref| mean {ref.abs().mean():.3f}")
    assert out.shape == ref.shape
    assert err < TOL_MAX_ABS and mse < TOL_MSE and err_gold < TOL_MAX_ABS
    # temporal chunking with the 2-frame cache reproduces the un-chunked result BIT FOR BIT (all kernels deterministic,
    # per-frame statistics independent of the chunking) — the reference's own property is 4.9e-6 in fp32
    for wsz in (1, 2):
        out_c = vae.decode(z.to("cuda:0"), temporal_chunk=True, window_size=wsz).sample.float().cpu()
        assert torch.equal(out_c, out), (wsz, (out_c - out).abs().max().item())
    # tiled decode vs the reference's tiled golden
    vae.enable_tiling()
    out_t = vae.decode(z.to("cuda:0"), temporal_chunk=True, window_size=1, tile_sample_min_size=32).sample.float().cpu()
    assert tuple(out_t.shape) == g["tiled32_shape"]
    assert (out_t.flatten()[::g["tiled32_stride"]] - g["tiled32_sample"]).abs().max().item() < TOL_MAX_ABS


def test_default_width_vae_matches_oracle():
    from oracle import vae_oracle as VO
    cfg = VO.VaeDecoderConfig()
    params = VO.synthetic_vae_params(cfg, seed=1)
    g = torch.Generator().manual_seed(5)
    z = torch.randn(1, 16, 3, 8, 12, generator=g).bfloat16().float()
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    pd = {k: v.to(dev) for k, v in params.items()}
    with torch.no_grad():
        ref = VO.decode(pd, cfg, z.to(dev)).float().cpu()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ref_bf16 = VO.decode(pd, cfg, z.to(dev).bfloat16()).float().cpu()
    out, _ = _ours({}, params, z, temporal_chunk=True, window_size=1)
    err, mse = (out - ref).abs().max().item(), ((out - ref) ** 2).mean().item()
    e2, m2 = (ref_bf16 - ref).abs().max().item(), ((ref_bf16 - ref) ** 2).mean().item()
    print(f"vae default width: ours vs fp32 oracle max_abs {err:.3e} mse {mse:.3e} | bf16-autocast oracle vs fp32 {e2:.3e} mse {m2:.3e} | |ref| mean {ref.abs().mean():.3f}")
    assert out.shape == ref.shape == (1, 3, 17, 64, 96)
    assert err < TOL_MAX_ABS and mse < TOL_MSE
    assert err <= 1.5 * e2 + 1e-2 and mse <= 2.0 * m2 + 1e-5, "must be comparable to the reference's own bf16 error"
    assert ref.abs().mean().item() > 0.05


def test_conv3d_strided_kernel():
    """The encoder's down-samplers: 3x3x3 causal conv with stride (1,2,2) / (2,1,1) (strided TMA box) vs F.conv3d."""
    from pyramid_flow_b200.vae import B200CausalVAE, _Conv
    torch.manual_seed(1)
    dev = torch.device("cuda:0")
    holder = B200CausalVAE.__new__(B200CausalVAE)
    cases = [((1, 2, 2), 64, 128, 3, 6, 10), ((1, 2, 2), 128, 128, 2, 17, 33), ((1, 2, 2), 64, 128, 2, 96, 160),
             ((2, 1, 1), 64, 64, 3, 9, 20), ((2, 1, 1), 128, 256, 1, 12, 150), ((2, 1, 1), 64, 128, 5, 48, 80)]
    for (stride, ci, co, t_out, h_out, w_out) in cases:
        st, sh, sw = stride
        wt = (torch.randn(co, ci, 3, 3, 3) * (ci * 27) ** -0.5).bfloat16().float()
        bias = torch.randn(co) * 0.1
        cv = _Conv({"c.conv.weight": wt, "c.conv.bias": bias}, "c", dev)
        cv.stride = stride
        t_in = (t_out - 1) * st + 1                       # real frames; 2 causal zero frames go in front
        x = torch.randn(t_in, h_out * sh, w_out * sw, ci, device=dev).bfloat16()
        xin = torch.zeros(t_in + 2, h_out * sh, w_out * sw, ci, device=dev, dtype=torch.bfloat16)
        xin[2:] = x
        xr = F.pad(x.permute(3, 0, 1, 2)[None].float(), (1, 1, 1, 1, 2, 0))
        ref = F.conv3d(xr, wt.to(dev), bias.to(dev), stride=stride)[0].permute(1, 2, 3, 0)
        assert tuple(ref.shape) == (t_out, h_out, w_out, co), (ref.shape, stride)
        out = torch.zeros(t_out, h_out, w_out, co, device=dev, dtype=torch.bfloat16)
        B200CausalVAE._conv(holder, cv, xin, t_out, h_out, w_out, out=out)
        torch.cuda.synchronize()
        err = (out.float() - ref).abs().max().item()
        assert err < 3e-2, (stride, ci, co, t_out, h_out, w_out, err)


def test_vae_encoder_matches_reference_golden(golden_dir):
    """encode() (encoder + quant_conv moments, P:911's image latent) vs the unmodified reference's moments and the oracle."""
    from oracle import vae_oracle as VO
    from pyramid_flow_b200.vae import B200CausalVAE, VaeConfigB200
    g = torch.load(golden_dir / "vae_encoder_small.pt", weights_only=False)
    ecfg = VO.VaeEncoderConfig(**g["cfg"])
    params = VO.synthetic_vae_params(ecfg, seed=g["param_seed"])
    dev = torch.device("cuda:0")
    vae = B200CausalVAE(VaeConfigB200(enc_block_out_channels=ecfg.block_out_channels,
                                      enc_layers_per_block=ecfg.layers_per_block), params, device=dev)
    assert vae.has_encoder and not vae.has_decoder
    pd = {k: v.to(dev) for k, v in params.items()}
    for name in ("image", "clip"):
        x = g[name].bfloat16()                             # the pipeline feeds the image in the VAE dtype (bf16), P:911
        dist = vae.encode(x.to(dev)).latent_dist
        torch.cuda.synchronize()
        ours = dist.parameters.float().cpu()
        with torch.no_grad():
            ref = VO.encode_moments(params, ecfg, x.float())
            with torch.autocast("cuda", dtype=torch.bfloat16):
                ref_bf16 = VO.encode_moments(pd, ecfg, x.to(dev)).float().cpu()
        err = (ours - ref).abs().max().item()
        err_gold = (ours - g["moments_" + name]).abs().max().item()    # reference ran on the un-rounded fp32 input
        err_pol = (ref_bf16 - ref).abs().max().item()
        print(f"vae encode {name}: max_abs vs oracle {err:.3e}, vs reference golden {err_gold:.3e}, reference bf16 policy {err_pol:.3e}, |ref| mean {ref.abs().mean():.3f}")
        assert ours.shape == ref.shape
        assert err < 5e-2 and err_gold < 6e-2 and err <= max(1.5 * err_pol, 1e-2)
        assert torch.equal(dist.mean.float().cpu(), ours[:, :16]) and dist.std.shape == dist.mean.shape
    gen = torch.Generator().manual_seed(0)
    z = dist.sample(gen)
    assert z.shape == dist.mean.shape and z.device.type == "cuda" and z.dtype == torch.bfloat16


def test_decode_latent_u8_fused_matches_two_step(golden_dir):
    """decode_latent_u8: un-normalisation fused into the latent pack + uint8 store in conv_out's epilogue == the reference's
    order of operations (un-normalise in torch, decode, mul(127.5).add(127.5).clamp(0,255).byte(), P:1226-1238) to within one
    grey level (the two-step path rounds the un-normalised latent to bf16 first)."""
    from oracle import vae_oracle as VO
    from pyramid_flow_b200.vae import B200CausalVAE, VaeConfigB200
    g = torch.load(golden_dir / "vae_small.pt", weights_only=False)
    cfg = VO.VaeDecoderConfig(**g["cfg"])
    params = VO.synthetic_vae_params(cfg, seed=g["param_seed"])
    dev = torch.device("cuda:0")
    vae = B200CausalVAE(VaeConfigB200(**g["cfg"]), params, device=dev)
    z = g["z"].to(dev).bfloat16()
    sc, sh, vsc, vsh = 1 / 1.8726, -0.04, 1 / 3.0986, -0.2343
    u8 = vae.decode_latent_u8(z, sc, sh, vsc, vsh, window_size=1)
    zz = z.float().clone()
    zz[:, :, :1] = zz[:, :, :1] / sc + sh
    zz[:, :, 1:] = zz[:, :, 1:] / vsc + vsh
    img = vae.decode(zz, temporal_chunk=True, window_size=1).sample
    ref = img.float().mul(127.5).add(127.5).clamp(0, 255).byte().permute(0, 2, 3, 4, 1).reshape(-1, img.shape[3], img.shape[4], 3)
    torch.cuda.synchronize()
    assert u8.dtype == torch.uint8 and u8.shape == ref.shape
    d = (u8.int() - ref.int()).abs()
    assert d.max().item() <= 1 and d.float().mean().item() < 0.05, (d.max().item(), d.float().mean().item())
    assert ref.float().std().item() > 5
