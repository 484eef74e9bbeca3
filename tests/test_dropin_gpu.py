"""THE DROP-IN (SURVEY.md §7 step 6, INTEGRATION.md): the B200 modules, built with `from_reference()` from what a loaded
reference module exposes (its registered `.config`, its bf16 `.state_dict()`), run the pyramidal sampler loop on a B200
and are compared with what the UNMODIFIED reference pipeline `PyramidDiTForVideoGeneration` computed on a GPU with the
reference's own modules (bf16 weights under torch.autocast, the README's way of running it) on identical seeds, text
embeddings and injected block noise: `generate()` final latents, and `generate_i2v()` -> `decode_latent()` uint8 frames.

The reference side is tests/golden/dropin_gpu.pt (oracle/pin/make_golden.py dropin: module configs, latents, a fixed
strided sample of the frames); the loop on this side is pyramid_flow_b200/sampler.py, pinned to the reference loop by
tests/test_sampler_cpu.py.  Both are also compared with the CPU fp32 goldens (tests/golden/sampler_small.pt,
sampler_i2v_small.pt)."""
from types import SimpleNamespace

import pytest
import torch

pytestmark = pytest.mark.gpu

# the small reference VAE of the i2v case (oracle/pin/make_golden.py DROPIN_VAE_DEC / DROPIN_VAE_ENC)
VAE_DEC = dict(block_out_channels=(64, 64, 128, 128), layers_per_block=(1, 1, 1, 1))
VAE_ENC = dict(block_out_channels=(64, 64, 128, 128), layers_per_block=(1, 1, 1, 1))


@pytest.fixture(scope="module")
def ref_gpu(golden_dir):
    return torch.load(golden_dir / "dropin_gpu.pt", weights_only=False)


class _LoadedReferenceModule:
    """What from_reference() reads from a loaded reference module: `.config` and `.state_dict()`."""

    def __init__(self, config, state_dict):
        self.config = SimpleNamespace(**config)
        self._sd = state_dict

    def state_dict(self):
        return self._sd


def _ours_dit(ref_gpu, g, dev):
    from oracle import flux_oracle as FO
    from pyramid_flow_b200.dit import B200FluxTransformer
    params = FO.synthetic_flux_params(FO.FluxConfig(**g["cfg"]), seed=g["param_seed"])
    ref = _LoadedReferenceModule(ref_gpu["dit_config"], {k: v.to(dev, torch.bfloat16) for k, v in params.items()})
    ours = B200FluxTransformer.from_reference(ref, device=dev)
    assert ours.config.in_channels == ref.config.in_channels and next(ours.parameters()).device == dev
    return ours


def _sampler(dit, vae, g):
    from pyramid_flow_b200.sampler import B200PyramidSampler
    from pyramid_flow_b200.scheduler import B200FlowMatchScheduler
    noises = [n.clone() for n in g["noises"]]
    return B200PyramidSampler(dit, B200FlowMatchScheduler(), vae=vae, block_noise_fn=lambda *a: noises.pop(0))


def _text(g, dev):
    """The CFG batch [negative ; positive] the pipeline builds from its text encoder (P:1066-1072), bf16 like the encoder."""
    return g["enc"].to(dev).bfloat16(), g["mask"].to(dev), g["pooled"].to(dev).bfloat16()


def _rel_mse(a, b):
    return (((a - b) ** 2).mean() / (b ** 2).mean()).item()


def test_unmodified_generate_with_swapped_dit(ref_gpu, golden_dir):
    dev = torch.device("cuda:0")
    g = torch.load(golden_dir / "sampler_small.pt", weights_only=False)
    s = _sampler(_ours_dit(ref_gpu, g, dev), None, g)
    gen = torch.Generator().manual_seed(g["latent_seed"])
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        lat = s.generate(*_text(g, dev), generator=gen, output_type="latent", save_memory=True, **g["args"])
    torch.cuda.synchronize()
    ref = ref_gpu["latents"].float()
    assert lat.shape == ref.shape == g["latents"].shape
    ours, gold = lat.float().cpu(), g["latents"]
    r_pair = _rel_mse(ours, ref)
    r_ref, r_ours = _rel_mse(ref, gold), _rel_mse(ours, gold)
    print(f"generate() final latents: drop-in vs the reference's own modules on a GPU (both bf16): relative MSE {r_pair:.3e}; "
          f"|latent| mean {ref.abs().mean():.3f}.  (vs the CPU fp32 golden: reference {r_ref:.3e}, drop-in {r_ours:.3e} -- "
          f"not comparable: on the GPU the pipeline draws its start noise in bf16, a different random stream than the fp32 CPU run)")
    # measured 2.95e-4 on a B200 at a 1000 W power limit: 6 Euler steps of bf16 latents through two different bf16
    # implementations of the DiT (frames below: mean |diff| 0.98 / 255)
    assert r_pair < 1e-3 and ref.abs().mean().item() > 1.0
    assert abs(r_ours - r_ref) < 0.05 * r_ref + 1e-3, "both runs must sit at the same distance from the fp32 CPU run"


def test_unmodified_generate_i2v_and_decode_latent_with_swapped_vae(ref_gpu, golden_dir):
    """generate_i2v() needs vae.encode (image latent, P:911) and, with pixel output, decode_latent (P:1221-1243): the whole
    call runs on the B200 objects; frames are compared as uint8 images with the reference modules' frames."""
    from oracle import vae_oracle as VO
    from pyramid_flow_b200.vae import B200CausalVAE
    dev = torch.device("cuda:0")
    g = torch.load(golden_dir / "sampler_i2v_small.pt", weights_only=False)
    dcfg, ecfg = VO.VaeDecoderConfig(**VAE_DEC), VO.VaeEncoderConfig(**VAE_ENC)
    params = {**VO.synthetic_vae_params(dcfg, seed=4), **VO.synthetic_vae_params(ecfg, seed=5)}
    # the reference run pinned log-variance at -30 so that latent_dist.sample() is the mean (D:381-389)
    params["quant_conv.conv.weight"][16:] = 0
    params["quant_conv.conv.bias"][16:] = -30.0
    vae = B200CausalVAE.from_reference(
        _LoadedReferenceModule(ref_gpu["vae_config"], {k: v.to(dev, torch.bfloat16) for k, v in params.items()}), device=dev)
    vae.enable_tiling()
    s = _sampler(_ours_dit(ref_gpu, g, dev), vae, g)
    gen = torch.Generator().manual_seed(g["latent_seed"])
    args = {k: v for k, v in g["args"].items() if k not in ("height", "width")}
    torch.manual_seed(123)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        # image_tensor: the input image as the pipeline's ToTensor + Normalize(0.5, 0.5) left it (P:906-910)
        out = s.generate_i2v(g["image_tensor"], *_text(g, dev), height=g["args"]["height"], width=g["args"]["width"],
                             generator=gen, output_type="uint8", save_memory=True, **args)
    torch.cuda.synchronize()
    out = out.cpu()
    assert tuple(out.shape) == ref_gpu["frames_shape"] and out.shape[0] == 1 + 8 * (g["args"]["temp"] - 1)
    a, b = out.flatten()[::ref_gpu["frames_stride"]].float(), ref_gpu["frames_sample"].float()
    diff = (a - b).abs()
    print(f"generate_i2v -> decode_latent, uint8 frames {tuple(out.shape)} (every {ref_gpu['frames_stride']}th value): mean |diff| "
          f"{diff.mean():.3f} / 255, 99.9th pct {diff.kthvalue(int(0.999 * diff.numel())).values.item():.0f}, max {diff.max():.0f}; "
          f"frame std {b.std():.1f}")
    assert diff.mean().item() < 2.0 and b.std().item() > 5.0
