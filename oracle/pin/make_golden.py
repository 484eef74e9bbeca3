"""Generate tests/golden/* by running the UNMODIFIED reference (imported through ref_shim).

    PF_REFERENCE_ROOT=/path/to/Pyramid-Flow python oracle/pin/make_golden.py [flux] [block] [sched] [vae] [vae_encoder] [sampler] [sampler_i2v] [mmdit]
    python oracle/pin/make_golden.py dropin         (needs a CUDA GPU; the reference staged by oracle/pin/stage_reference.py)

The tests never import the reference; they only see the small fixtures this script writes under tests/golden/.
Inputs and parameters are regenerated from seeds by the tests (torch CPU generators are deterministic), so the fixtures
hold the reference OUTPUTS plus the exact inputs for safety.  Files stay under 1 MB: a large output is stored as the
fixed strided sample `t.flatten()[::SAMPLE_STRIDE]` (the stride is coprime with every axis length, so each row, column and
channel is sampled).
"""
from __future__ import annotations

import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle.pin import ref_shim  # noqa: E402

ref_shim.install()
from oracle import flux_oracle as FO  # noqa: E402

GOLD = ROOT / "tests" / "golden"
GOLD.mkdir(parents=True, exist_ok=True)

SAMPLE_STRIDE = 13
SMALL_CFG = dict(num_layers=2, num_single_layers=2, num_attention_heads=4, attention_head_dim=64, in_channels=64,
                 joint_attention_dim=128, pooled_projection_dim=64)


def small_inputs(seed: int = 1, batch: int = 2, text_len: int = 24):
    g = torch.Generator().manual_seed(seed)
    clips = [torch.randn(batch, 16, 2, 4, 8, generator=g), torch.randn(batch, 16, 1, 8, 16, generator=g),
             torch.randn(batch, 16, 1, 16, 32, generator=g)]
    enc = torch.randn(batch, text_len, SMALL_CFG["joint_attention_dim"], generator=g) * 0.5
    mask = torch.ones(batch, text_len, dtype=torch.long)
    mask[0, 9:] = 0
    pooled = torch.randn(batch, SMALL_CFG["pooled_projection_dim"], generator=g)
    timestep = torch.tensor([972.0] * batch)
    return clips, enc, mask, pooled, timestep


def make_flux():
    from pyramid_dit.flux_modules import PyramidFluxTransformer
    cfg = FO.FluxConfig(**SMALL_CFG)
    params = FO.synthetic_flux_params(cfg, seed=0)
    model = PyramidFluxTransformer(**SMALL_CFG).eval()
    missing = model.load_state_dict(params, strict=True)   # pins the key layout and shapes of flux_param_shapes()
    print("load_state_dict:", missing)
    clips, enc, mask, pooled, timestep = small_inputs()
    with torch.no_grad():
        out = model(sample=[clips], timestep_ratio=timestep, encoder_hidden_states=enc, encoder_attention_mask=mask,
                    pooled_projections=pooled)[0]
        # all-ones mask case too
        out_full = model(sample=[clips], timestep_ratio=timestep, encoder_hidden_states=enc,
                         encoder_attention_mask=torch.ones_like(mask), pooled_projections=pooled)[0]
        # single-clip (first unit) case
        out_first = model(sample=[[clips[-1]]], timestep_ratio=timestep * 0.5, encoder_hidden_states=enc,
                          encoder_attention_mask=mask, pooled_projections=pooled)[0]
    torch.save({"cfg": SMALL_CFG, "param_seed": 0, "input_seed": 1, "clips": clips, "enc": enc, "mask": mask,
                "pooled": pooled, "timestep": timestep, "out": out, "out_full_mask": out_full, "out_first": out_first},
               GOLD / "flux_small.pt")
    print("flux_small:", out.shape, float(out.abs().mean()), float(out_first.abs().mean()))


def make_block():
    """BASELINE.json configs[0]: one miniFLUX double block + one single block, D=1920/H=30, 256 video + 77 text tokens."""
    from pyramid_dit.flux_modules import FluxSingleTransformerBlock, FluxTransformerBlock
    cfg = FO.FluxConfig(num_layers=1, num_single_layers=1)
    params = FO.synthetic_flux_params(cfg, seed=0)
    d, heads = cfg.inner_dim, cfg.num_attention_heads
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 256, d, generator=g)
    ctx = torch.randn(1, 77, d, generator=g)
    temb = torch.randn(1, d, generator=g)
    ids = torch.cat([torch.zeros(77, 3), FO.clip_ids(1, 16, 16, 16, 16, 0)], 0)
    cs = FO.rope_table(ids, cfg.axes_dims_rope)
    rot = torch.stack([cs[..., 0], -cs[..., 1], cs[..., 1], cs[..., 0]], dim=-1).view(1, 333, 1, 32, 2, 2)
    mask = torch.ones(1, 1, 333, 333, dtype=torch.bool)
    blk = FluxTransformerBlock(dim=d, num_attention_heads=heads, attention_head_dim=64).eval()
    blk.load_state_dict({k[len("transformer_blocks.0."):]: v for k, v in params.items() if k.startswith("transformer_blocks.0.")}, strict=True)
    sblk = FluxSingleTransformerBlock(dim=d, num_attention_heads=heads, attention_head_dim=64).eval()
    sblk.load_state_dict({k[len("single_transformer_blocks.0."):]: v for k, v in params.items() if k.startswith("single_transformer_blocks.0.")}, strict=True)
    with torch.no_grad():
        c_out, x_out = blk(hidden_states=x, encoder_hidden_states=ctx, encoder_attention_mask=None, temb=temb,
                           attention_mask=[mask], hidden_length=[256], image_rotary_emb=[rot])
        h = torch.cat([ctx, x], 1)
        s_out = sblk(hidden_states=h, temb=temb, encoder_attention_mask=None, attention_mask=[mask],
                     hidden_length=[333], image_rotary_emb=[rot])
    torch.save({"x_out_rows": x_out[:, ::16].clone(), "c_out_rows": c_out[:, ::16].clone(),
                "s_out_rows": s_out[:, ::16].clone(), "x_out_mean": x_out.mean(-1), "s_out_mean": s_out.mean(-1)},
               GOLD / "flux_block_cfg1.pt")
    print("block:", float(x_out.abs().mean()), float(c_out.abs().mean()), float(s_out.abs().mean()))


def make_sched():
    from diffusion_schedulers import PyramidFlowMatchEulerDiscreteScheduler
    s = PyramidFlowMatchEulerDiscreteScheduler(shift=1.0, stages=3, stage_range=[0, 1 / 3, 2 / 3, 1], gamma=1 / 3)
    out = {"start_sigmas": dict(s.start_sigmas), "end_sigmas": dict(s.end_sigmas), "ori_start_sigmas": dict(s.ori_start_sigmas),
           "timestep_ratios": {k: list(v) for k, v in s.timestep_ratios.items()},
           "timesteps_per_stage": {k: v.clone() for k, v in s.timesteps_per_stage.items()},
           "sigmas_per_stage": {k: v.clone() for k, v in s.sigmas_per_stage.items()}}
    for n in (10, 20):
        for st in range(3):
            s.set_timesteps(n, st)
            out[f"timesteps_{n}_{st}"] = s.timesteps.clone()
            out[f"sigmas_{n}_{st}"] = s.sigmas.clone()
    # one Euler step in fp32
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 16, 1, 8, 8, generator=g)
    v = torch.randn(1, 16, 1, 8, 8, generator=g)
    s.set_timesteps(10, 1)
    out["step_x"] = x
    out["step_v"] = v
    out["step_out"] = s.step(model_output=v, timestep=s.timesteps[0], sample=x).prev_sample.clone()
    torch.save(out, GOLD / "scheduler.pt")
    print("sched:", out["start_sigmas"], out["end_sigmas"])


VAE_SMALL = dict(block_out_channels=(64, 128, 128, 128), layers_per_block=(2, 2, 2, 2))
VAE_ENC_SMALL = dict(block_out_channels=(64, 128, 128, 128), layers_per_block=(1, 2, 1, 1))


def make_vae():
    """Tiny-width VAE decoder (all structural features: shortcut conv, spatial+temporal upsamplers, mid attention)."""
    from video_vae import CausalVideoVAE
    from oracle import vae_oracle as VO
    cfg = VO.VaeDecoderConfig(**VAE_SMALL)
    params = VO.synthetic_vae_params(cfg, seed=0)
    vae = CausalVideoVAE(encoder_out_channels=16, decoder_in_channels=16, decoder_block_out_channels=cfg.block_out_channels,
                         decoder_layers_per_block=cfg.layers_per_block).eval()
    sd = vae.state_dict()
    dec_keys = {k for k in sd if k.startswith("decoder.") or k.startswith("post_quant_conv.")}
    assert dec_keys == set(params.keys()), (dec_keys ^ set(params.keys()))
    for k, v in params.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    sd.update(params)
    vae.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(2)
    z = torch.randn(1, 16, 3, 6, 10, generator=g)
    with torch.no_grad():
        full = vae.decode(z, temporal_chunk=False).sample
        chunk1 = vae.decode(z, temporal_chunk=True, window_size=1).sample
        chunk2 = vae.decode(z, temporal_chunk=True, window_size=2).sample
        vae.enable_tiling()
        tiled = vae.decode(z, temporal_chunk=True, window_size=1, tile_sample_min_size=32).sample
    print("vae:", full.shape, float(full.abs().mean()), "chunk1 diff", float((full - chunk1).abs().max()),
          "chunk2 diff", float((full - chunk2).abs().max()), "tiled diff", float((full - tiled).abs().max()))
    torch.save({"cfg": VAE_SMALL, "param_seed": 0, "z": z, "full": full, "chunk1_maxdiff": float((full - chunk1).abs().max()),
                "chunk2_maxdiff": float((full - chunk2).abs().max()), "tiled32_shape": tuple(tiled.shape),
                "tiled32_stride": SAMPLE_STRIDE, "tiled32_sample": tiled.flatten()[::SAMPLE_STRIDE].clone()},
               GOLD / "vae_small.pt")


def make_vae_encoder():
    """Tiny-width VAE encoder (stride-2 spatial / temporal causal convs, shortcut conv, mid attention) + quant_conv: the
    moments the i2v path samples its image latent from (P:911), for a 1-frame image and for a 9-frame clip."""
    from video_vae import CausalVideoVAE
    from oracle import vae_oracle as VO
    cfg = VO.VaeEncoderConfig(**VAE_ENC_SMALL)
    params = VO.synthetic_vae_params(cfg, seed=1)
    vae = CausalVideoVAE(encoder_out_channels=16, decoder_in_channels=16, encoder_block_out_channels=cfg.block_out_channels,
                         encoder_layers_per_block=cfg.layers_per_block, decoder_block_out_channels=(32, 32, 32, 32),
                         decoder_layers_per_block=(1, 1, 1, 1)).eval()
    sd = vae.state_dict()
    enc_keys = {k for k in sd if k.startswith("encoder.") or k.startswith("quant_conv.")}
    assert enc_keys == set(params.keys()), (enc_keys ^ set(params.keys()))
    for k, v in params.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    sd.update(params)
    vae.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(3)
    image = torch.randn(1, 3, 1, 64, 96, generator=g)
    clip = torch.randn(1, 3, 9, 32, 48, generator=g)
    with torch.no_grad():
        m_image = vae.encode(image).latent_dist.parameters
        m_clip = vae.encode(clip).latent_dist.parameters
        d = vae.encode(image).latent_dist
    print("vae encoder:", m_image.shape, float(m_image.abs().mean()), m_clip.shape, float(m_clip.abs().mean()))
    torch.save({"cfg": VAE_ENC_SMALL, "param_seed": 1, "image": image, "clip": clip, "moments_image": m_image,
                "moments_clip": m_clip, "mean_image": d.mean, "logvar_image": d.logvar, "std_image": d.std},
               GOLD / "vae_encoder_small.pt")


def make_sampler():
    """The UNMODIFIED reference generate() loop (P:1006-1219) on CPU fp32 with a tiny reference DiT, a fake text encoder and
    injected block noise (the reference draws it from the global CPU RNG in a python loop, P:697-703)."""
    from pyramid_dit import PyramidDiTForVideoGeneration
    from pyramid_dit.flux_modules import PyramidFluxTransformer
    from diffusion_schedulers import PyramidFlowMatchEulerDiscreteScheduler
    cfg = FO.FluxConfig(**SMALL_CFG)
    params = FO.synthetic_flux_params(cfg, seed=0)
    dit = PyramidFluxTransformer(**SMALL_CFG).eval()
    dit.load_state_dict(params, strict=True)
    g = torch.Generator().manual_seed(7)
    enc = torch.randn(2, 24, SMALL_CFG["joint_attention_dim"], generator=g) * 0.5      # [negative ; positive]
    mask = torch.ones(2, 24, dtype=torch.long)
    mask[0, 11:] = 0
    pooled = torch.randn(2, SMALL_CFG["pooled_projection_dim"], generator=g)

    class FakeText:
        def __init__(self):
            self.calls = 0

        def __call__(self, prompt, device):   # generate() calls it for the prompt, then for the negative prompt
            i = 1 if self.calls == 0 else 0
            self.calls += 1
            return enc[i:i + 1], mask[i:i + 1], pooled[i:i + 1]

    pipe = object.__new__(PyramidDiTForVideoGeneration)
    pipe.dit = dit
    pipe.text_encoder = FakeText()
    pipe.vae = None
    pipe.scheduler = PyramidFlowMatchEulerDiscreteScheduler(shift=1.0, stages=3, stage_range=[0, 1 / 3, 2 / 3, 1], gamma=1 / 3)
    pipe.stages = [1, 2, 4]
    pipe.frame_per_unit = 1
    pipe.model_name = "pyramid_flux"
    pipe.sequential_offload_enabled = False
    pipe.downsample = 8
    pipe.vae_scale_factor = 1 / 1.8726
    ng = torch.Generator().manual_seed(11)
    noises = []

    def fake_block_noise(bs, ch, temp, height, width):
        n = torch.randn(bs, ch, temp, height, width, generator=ng)
        noises.append(n)
        return n

    pipe.sample_block_noise = fake_block_noise
    gen = torch.Generator().manual_seed(3)
    with torch.no_grad():
        lat = pipe.generate(prompt="x", height=128, width=128, temp=4, num_inference_steps=[2, 2, 2],
                            video_num_inference_steps=[2, 1, 2], guidance_scale=7.0, video_guidance_scale=5.0,
                            generator=gen, output_type="latent", save_memory=True)
    print("sampler:", lat.shape, float(lat.abs().mean()), "block-noise draws", len(noises))
    torch.save({"cfg": SMALL_CFG, "param_seed": 0, "enc": enc, "mask": mask, "pooled": pooled, "noises": noises,
                "latent_seed": 3, "latents": lat, "args": dict(height=128, width=128, temp=4, num_inference_steps=[2, 2, 2],
                                                                video_num_inference_steps=[2, 1, 2], guidance_scale=7.0,
                                                                video_guidance_scale=5.0)}, GOLD / "sampler_small.pt")


def make_sampler_i2v():
    """The UNMODIFIED reference generate_i2v() loop (P:791-1003) on CPU fp32: tiny reference DiT, fake text encoder, a fake
    VAE whose encode() returns a fixed image latent, injected block noise."""
    from PIL import Image
    from pyramid_dit import PyramidDiTForVideoGeneration
    from pyramid_dit.flux_modules import PyramidFluxTransformer
    from diffusion_schedulers import PyramidFlowMatchEulerDiscreteScheduler
    cfg = FO.FluxConfig(**SMALL_CFG)
    params = FO.synthetic_flux_params(cfg, seed=0)
    dit = PyramidFluxTransformer(**SMALL_CFG).eval()
    dit.load_state_dict(params, strict=True)
    g = torch.Generator().manual_seed(17)
    enc = torch.randn(2, 24, SMALL_CFG["joint_attention_dim"], generator=g) * 0.5      # [negative ; positive]
    mask = torch.ones(2, 24, dtype=torch.long)
    mask[0, 13:] = 0
    pooled = torch.randn(2, SMALL_CFG["pooled_projection_dim"], generator=g)
    image_latent_raw = torch.randn(1, 16, 1, 16, 16, generator=g)     # what vae.encode(...).latent_dist.sample() returns

    class FakeText:
        def __init__(self):
            self.calls = 0

        def __call__(self, prompt, device):
            i = 1 if self.calls == 0 else 0
            self.calls += 1
            return enc[i:i + 1], mask[i:i + 1], pooled[i:i + 1]

    class FakeDist:
        def sample(self):
            return image_latent_raw

    class FakeVae:
        device, dtype = torch.device("cpu"), torch.float32
        seen = []

        def encode(self, x):
            FakeVae.seen.append(x)
            return type("O", (), {"latent_dist": FakeDist()})()

    pipe = object.__new__(PyramidDiTForVideoGeneration)
    pipe.dit = dit
    pipe.text_encoder = FakeText()
    pipe.vae = FakeVae()
    pipe.scheduler = PyramidFlowMatchEulerDiscreteScheduler(shift=1.0, stages=3, stage_range=[0, 1 / 3, 2 / 3, 1], gamma=1 / 3)
    pipe.stages = [1, 2, 4]
    pipe.frame_per_unit = 1
    pipe.model_name = "pyramid_flux"
    pipe.sequential_offload_enabled = False
    pipe.downsample = 8
    pipe.vae_shift_factor, pipe.vae_scale_factor = -0.04, 1 / 1.8726
    ng = torch.Generator().manual_seed(12)
    noises = []

    def fake_block_noise(bs, ch, temp, height, width):
        n = torch.randn(bs, ch, temp, height, width, generator=ng)
        noises.append(n)
        return n

    pipe.sample_block_noise = fake_block_noise
    img = Image.fromarray((torch.rand(128, 128, 3, generator=g) * 255).byte().numpy())
    gen = torch.Generator().manual_seed(5)
    args = dict(temp=4, num_inference_steps=[2, 1, 2], guidance_scale=7.0, video_guidance_scale=4.0)
    with torch.no_grad():
        lat = pipe.generate_i2v(prompt="x", input_image=img, generator=gen, output_type="latent", save_memory=True, **args)
    print("sampler_i2v:", lat.shape, float(lat.abs().mean()), "block-noise draws", len(noises), "image tensor", FakeVae.seen[0].shape)
    torch.save({"cfg": SMALL_CFG, "param_seed": 0, "enc": enc, "mask": mask, "pooled": pooled, "noises": noises,
                "latent_seed": 5, "latents": lat, "image_tensor": FakeVae.seen[0], "image_latent_raw": image_latent_raw,
                "args": dict(height=128, width=128, **args)}, GOLD / "sampler_i2v_small.pt")


DROPIN_VAE_DEC = dict(block_out_channels=(64, 64, 128, 128), layers_per_block=(1, 1, 1, 1))
DROPIN_VAE_ENC = dict(block_out_channels=(64, 64, 128, 128), layers_per_block=(1, 1, 1, 1))


def make_dropin():
    """The UNMODIFIED reference pipeline `PyramidDiTForVideoGeneration` with the reference's own modules on a CUDA GPU, bf16
    weights under torch.autocast (the README's way of running it): generate() final latents on the inputs of
    sampler_small.pt, and generate_i2v() -> decode_latent() uint8 frames on those of sampler_i2v_small.pt (tiny reference
    DiT, small reference VAE with synthetic weights).  tests/test_dropin_gpu.py drives the B200 modules, built through
    from_reference() from the module configs stored here, on the same inputs and compares with these outputs."""
    import numpy as np
    from PIL import Image
    from diffusion_schedulers import PyramidFlowMatchEulerDiscreteScheduler
    from oracle import vae_oracle as VO
    from pyramid_dit import PyramidDiTForVideoGeneration
    from pyramid_dit.flux_modules import PyramidFluxTransformer
    from video_vae import CausalVideoVAE
    dev = torch.device("cuda:0")

    def ref_dit(g):
        dit = PyramidFluxTransformer(**g["cfg"]).eval()
        dit.load_state_dict(FO.synthetic_flux_params(FO.FluxConfig(**g["cfg"]), seed=g["param_seed"]), strict=True)
        return dit.to(dev, torch.bfloat16)

    def make_pipe(g, dit, vae):
        class FakeText:   # generate() asks for the prompt first, then for the negative prompt (P:1066-1067)
            calls = 0

            def __call__(self, prompt, device):
                i = 1 if self.calls % 2 == 0 else 0
                self.calls += 1
                return (g["enc"][i:i + 1].to(dev).bfloat16(), g["mask"][i:i + 1].to(dev),
                        g["pooled"][i:i + 1].to(dev).bfloat16())

        pipe = object.__new__(PyramidDiTForVideoGeneration)
        pipe.dit, pipe.vae, pipe.text_encoder = dit, vae, FakeText()
        pipe.scheduler = PyramidFlowMatchEulerDiscreteScheduler(shift=1.0, stages=3, stage_range=[0, 1 / 3, 2 / 3, 1], gamma=1 / 3)
        pipe.stages = [1, 2, 4]
        pipe.frame_per_unit = 1
        pipe.model_name = "pyramid_flux"
        pipe.sequential_offload_enabled = False
        pipe.downsample = 8
        pipe.vae_shift_factor, pipe.vae_scale_factor = -0.04, 1 / 1.8726
        pipe.vae_video_shift_factor, pipe.vae_video_scale_factor = -0.2343, 1 / 3.0986
        noises = [n.clone() for n in g["noises"]]
        pipe.sample_block_noise = lambda bs, ch, temp, height, width: noises.pop(0)
        return pipe

    g = torch.load(GOLD / "sampler_small.pt", weights_only=False)
    dit = ref_dit(g)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        lat = make_pipe(g, dit, None).generate(prompt="x", generator=torch.Generator().manual_seed(g["latent_seed"]),
                                               output_type="latent", save_memory=True, **g["args"])

    gi = torch.load(GOLD / "sampler_i2v_small.pt", weights_only=False)
    dcfg, ecfg = VO.VaeDecoderConfig(**DROPIN_VAE_DEC), VO.VaeEncoderConfig(**DROPIN_VAE_ENC)
    vae = CausalVideoVAE(encoder_out_channels=16, decoder_in_channels=16, encoder_block_out_channels=ecfg.block_out_channels,
                         encoder_layers_per_block=ecfg.layers_per_block, decoder_block_out_channels=dcfg.block_out_channels,
                         decoder_layers_per_block=dcfg.layers_per_block).eval()
    sd = vae.state_dict()
    new = {**VO.synthetic_vae_params(dcfg, seed=4), **VO.synthetic_vae_params(ecfg, seed=5)}
    assert set(new) == set(sd), set(new) ^ set(sd)
    # latent_dist.sample() draws from the global RNG (D:381-389): pin log-variance at -30 so the image latent is its mean
    new["quant_conv.conv.weight"][16:] = 0
    new["quant_conv.conv.bias"][16:] = -30.0
    vae.load_state_dict(new, strict=True)
    vae = vae.to(dev, torch.bfloat16)
    vae.enable_tiling()
    img = Image.fromarray((gi["image_tensor"][0, :, 0].permute(1, 2, 0) * 127.5 + 127.5).round().clamp(0, 255).byte().numpy())
    args = {k: v for k, v in gi["args"].items() if k not in ("height", "width")}
    torch.manual_seed(123)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        out = make_pipe(gi, ref_dit(gi), vae).generate_i2v(prompt="x", input_image=img, output_type="pil", save_memory=True,
                                                           generator=torch.Generator().manual_seed(gi["latent_seed"]), **args)
    frames = torch.from_numpy(np.stack([np.asarray(f) for f in out]))
    print("dropin:", lat.shape, float(lat.float().abs().mean()), "frames", tuple(frames.shape), float(frames.float().std()))
    torch.save({"dit_config": dict(dit.config), "vae_config": dict(vae.config), "latents": lat.cpu(),
                "frames_shape": tuple(frames.shape), "frames_stride": SAMPLE_STRIDE,
                "frames_sample": frames.flatten()[::SAMPLE_STRIDE].clone(),
                "device": torch.cuda.get_device_name(dev), "torch": torch.__version__}, GOLD / "dropin_gpu.pt")


MMDIT_SMALL = dict(num_layers=3, num_attention_heads=4, attention_head_dim=64, in_channels=16, patch_size=2,
                   joint_attention_dim=128, pooled_projection_dim=64, pos_embed_max_size=24, sample_size=32)


def make_mmdit():
    from pyramid_dit.mmdit_modules import PyramidDiffusionMMDiT
    from oracle import mmdit_oracle as MO
    cfg = MO.MMDiTConfig(**MMDIT_SMALL)
    params = MO.synthetic_mmdit_params(cfg, seed=0)
    model = PyramidDiffusionMMDiT(sample_size=cfg.sample_size, patch_size=2, in_channels=16, num_layers=cfg.num_layers,
                                  attention_head_dim=64, num_attention_heads=cfg.num_attention_heads,
                                  caption_projection_dim=cfg.inner_dim, pooled_projection_dim=cfg.pooled_projection_dim,
                                  pos_embed_max_size=cfg.pos_embed_max_size, joint_attention_dim=cfg.joint_attention_dim,
                                  pos_embed_type="sincos", temp_pos_embed_type="rope", add_temp_pos_embed=True,
                                  use_flash_attn=False, use_temporal_causal=True, use_t5_mask=True,
                                  interp_condition_pos=True).eval()
    sd = model.state_dict()
    assert set(sd.keys()) == set(params.keys()), set(sd.keys()) ^ set(params.keys())
    # the oracle's sincos table must equal the buffer the reference computed for itself
    assert torch.allclose(sd["pos_embed.pos_embed"], params["pos_embed.pos_embed"], atol=1e-6)
    model.load_state_dict(params, strict=True)
    g = torch.Generator().manual_seed(1)
    clips = [torch.randn(2, 16, 2, 4, 8, generator=g), torch.randn(2, 16, 1, 8, 16, generator=g),
             torch.randn(2, 16, 1, 16, 32, generator=g)]
    enc = torch.randn(2, 24, cfg.joint_attention_dim, generator=g) * 0.5
    mask = torch.ones(2, 24, dtype=torch.long)
    mask[0, 9:] = 0
    pooled = torch.randn(2, cfg.pooled_projection_dim, generator=g)
    t = torch.tensor([972.0, 972.0])
    with torch.no_grad():
        out = model(sample=[clips], timestep_ratio=t, encoder_hidden_states=enc, encoder_attention_mask=mask,
                    pooled_projections=pooled)[0]
    torch.save({"cfg": MMDIT_SMALL, "param_seed": 0, "clips": clips, "enc": enc, "mask": mask, "pooled": pooled,
                "timestep": t, "out": out}, GOLD / "mmdit_small.pt")
    print("mmdit_small:", out.shape, float(out.abs().mean()))


if __name__ == "__main__":
    which = sys.argv[1:] or ["flux", "block", "sched"]
    for w in which:
        globals()["make_" + w]()
