"""B200CausalVAE — drop-in for the reference `CausalVideoVAE` (video_vae/modeling_causal_vae.py) as the sampler uses it.

Call surface used by the pipeline (pyramid_dit_for_video_gen_pipeline.py:1221-1243, :911):

    self.vae.decode(latents, temporal_chunk=True, window_size=w, tile_sample_min_size=s).sample    # [B, 3, T', H', W']
    self.vae.encode(image[:, :, None]).latent_dist.sample()                                        # i2v image latent

plus `.device`, `.dtype`, `.to()`, `.enable_tiling()`.  encode() also takes the reference's video arguments
(`temporal_chunk`, `window_size`, `tile_sample_min_size`) with their meaning, and `encode_frames_u8` encodes uint8 video
frames straight from a decoder.  Weights come from a state-dict in the reference key layout
(`decoder.*`, `post_quant_conv.*`, and — when present — `encoder.*`, `quant_conv.*`; SURVEY.md §8b).  The encoder reuses the
decoder's kernels; its down-samplers are the same implicit-GEMM conv with a strided TMA box (`stride_*` in pf_conv3d_desc).

Execution model (all math in libpf_b200 kernels, channels-last bf16 activations `[T, H, W, C]`, batch handled one sample
at a time as the pipeline does):
  * every CausalConv3d  -> `pf_causal_conv3d` (tcgen05 implicit GEMM, TMA im2col-free, bias/residual/depth-to-space fused)
  * every CausalGroupNorm(+SiLU) -> `pf_groupnorm_stats` + `pf_groupnorm_apply`, the apply writing straight into the next
    conv's input buffer behind its 2-frame causal halo
  * mid-block attention -> 1x1x1 convs for q/k/out, `pf_gemm_bf16` for V^T, QK^T and PV, `pf_softmax_rows`
  * temporal chunking = the reference's feature cache (C:126-143): each 3x3x3 conv keeps the last two frames of its padded
    input and they become the halo of the next chunk; chunking is exact, so the chunk length is a memory knob only.
    The encoder's stride-2 temporal down-samplers read only the last cached frame in a later chunk (C:140-141), so an
    encode is exact only when the window is a multiple of 2^(temporal down-samplers); other windows follow the reference's
    rule and may return fewer latent frames.
Spatial tiling (V:409-466, V:468-519) is reproduced by encoding / decoding tiles independently and cross-fading them
(`tile_sample_min_size`), but on 180 GB the un-tiled path is the default unless `enable_tiling()` was called, as in the
reference.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch

from . import _lib, ops
from ._lib import ConvDesc, PF_EPI_STORE_BF16


@dataclass
class VaeConfigB200:
    latent_channels: int = 16
    out_channels: int = 3
    block_out_channels: Tuple[int, ...] = (128, 256, 512, 512)
    layers_per_block: Tuple[int, ...] = (3, 3, 3, 3)
    spatial_up_sample: Tuple[bool, ...] = (True, True, True, False)
    temporal_up_sample: Tuple[bool, ...] = (True, True, True, False)
    norm_num_groups: int = 32
    downsample_scale: int = 8
    # encoder side (V:76-93); used only when the state-dict carries `encoder.*`
    enc_in_channels: int = 3
    enc_block_out_channels: Tuple[int, ...] = (128, 256, 512, 512)
    enc_layers_per_block: Tuple[int, ...] = (2, 2, 2, 2)
    enc_spatial_down_sample: Tuple[bool, ...] = (True, True, True, False)
    enc_temporal_down_sample: Tuple[bool, ...] = (True, True, True, False)


class DecoderOutput:
    def __init__(self, sample):
        self.sample = sample


class DiagonalGaussian:
    """DiagonalGaussianDistribution (D:369-391) over moments [B, 2C, T, h, w]: mean | logvar (clamped to [-30, 20])."""

    def __init__(self, parameters: torch.Tensor):
        self.parameters = parameters
        self.mean, logvar = torch.chunk(parameters, 2, dim=1)
        self.logvar = torch.clamp(logvar, -30.0, 20.0)
        self.std = torch.exp(0.5 * self.logvar)
        self.var = torch.exp(self.logvar)

    def sample(self, generator: Optional[torch.Generator] = None) -> torch.Tensor:
        # randn_tensor semantics (P:676-695): a CPU generator draws on the CPU, then the noise moves to the device
        gdev = generator.device if generator is not None else self.mean.device
        noise = torch.randn(self.mean.shape, generator=generator, device=gdev, dtype=self.mean.dtype).to(self.mean.device)
        return self.mean + self.std * noise

    def mode(self) -> torch.Tensor:
        return self.mean


class EncoderOutput:
    def __init__(self, latent_dist):
        self.latent_dist = latent_dist


def _pad64(n: int) -> int:
    return (n + 63) // 64 * 64


class _Conv:
    """One CausalConv3d: weights re-laid out to [Cout_pad, taps*Cin_pad] bf16 (tap-major), fp32 bias, halo cache."""

    def __init__(self, sd, name: str, device):
        w = sd[name + ".conv.weight"].float()
        co, ci, kt, kh, kw = w.shape
        self.cin, self.cout, self.kt, self.kh, self.kw = ci, co, kt, kh, kw
        self.cin_p, self.cout_p = _pad64(ci), _pad64(co)
        wp = torch.zeros(self.cout_p, kt, kh, kw, self.cin_p)
        wp[:co, :, :, :, :ci] = w.permute(0, 2, 3, 4, 1)
        self.w = wp.reshape(self.cout_p, kt * kh * kw * self.cin_p).to(device=device, dtype=torch.bfloat16).contiguous()
        b = torch.zeros(self.cout_p)
        if (name + ".conv.bias") in sd:
            b[:co] = sd[name + ".conv.bias"].float()
        self.bias = b.to(device)
        self.cache: Optional[torch.Tensor] = None   # last (kt-1) frames of the previous chunk's padded input
        # conv stride (t, h, w): the encoder's CausalDownsample2x (R:322) / CausalTemporalDownsample2x (R:486)
        self.stride = (2, 1, 1) if ".temporal_downsamplers." in name else (1, 2, 2) if ".downsamplers." in name else (1, 1, 1)


class B200CausalVAE(torch.nn.Module):
    def __init__(self, config: VaeConfigB200, state_dict: Dict[str, torch.Tensor], device="cuda"):
        super().__init__()
        self.cfg = config
        self.use_tiling = False
        self._cp = None                     # (group, rank, world) when context-parallel decode is on
        self._cp_ctx = None
        self.cp_frames_per_round = 4        # latent frames per rank per round (memory knob: ~6 GiB per frame at 768p)
        self.encode_tile_overlap_factor = 0.25
        self.decode_tile_overlap_factor = 0.25
        dev = torch.device(device)
        self._dev = dev
        sd = state_dict
        self.convs: Dict[str, _Conv] = {}
        self.norms: Dict[str, Tuple[torch.Tensor, torch.Tensor]] = {}
        sides = ("decoder.", "post_quant_conv.", "encoder.", "quant_conv.")
        for k in sd:
            if k.endswith(".conv.weight") and k.startswith(sides):
                name = k[: -len(".conv.weight")]
                self.convs[name] = _Conv(sd, name, dev)
        for k in sd:
            if k.startswith(("decoder.", "encoder.")) and k.endswith(".weight") and sd[k].ndim == 1:
                name = k[: -len(".weight")]
                self.norms[name] = (sd[k].float().to(dev).contiguous(), sd[name + ".bias"].float().to(dev).contiguous())
        self.has_decoder = "decoder.conv_in" in self.convs
        self.has_encoder = "encoder.conv_in" in self.convs
        # mid-block attention (diffusers Attention): q/k/out as 1x1x1 convs, v as a transposed GEMM
        self.attn: Dict[str, dict] = {}
        for side in ("decoder", "encoder"):
            a = side + ".mid_block.attentions.0"
            if (a + ".to_q.weight") not in sd:
                continue
            c = sd[a + ".to_q.weight"].shape[0]

            def lin_as_conv(prefix, bias_override=None, c=c):
                fake = {"x.conv.weight": sd[prefix + ".weight"].float().reshape(c, c, 1, 1, 1),
                        "x.conv.bias": sd[prefix + ".bias"].float() if bias_override is None else bias_override}
                return _Conv(fake, "x", dev)

            wo, bo = sd[a + ".to_out.0.weight"].float(), sd[a + ".to_out.0.bias"].float()
            bv = sd[a + ".to_v.bias"].float()
            self.attn[side] = dict(
                q=lin_as_conv(a + ".to_q"), k=lin_as_conv(a + ".to_k"),
                # softmax rows sum to 1 => P(V + 1 b_v^T) = PV + b_v^T: fold W_o b_v into the output bias
                o=lin_as_conv(a + ".to_out.0", bias_override=bo + wo @ bv),
                wv=sd[a + ".to_v.weight"].float().to(device=dev, dtype=torch.bfloat16).contiguous())
        self.register_buffer("_anchor", torch.zeros(1, device=dev, dtype=torch.bfloat16))

    @classmethod
    def from_reference(cls, ref_vae, device="cuda") -> "B200CausalVAE":
        rc = ref_vae.config
        cfg = VaeConfigB200(latent_channels=rc.decoder_in_channels, out_channels=rc.decoder_out_channels,
                            block_out_channels=tuple(rc.decoder_block_out_channels),
                            layers_per_block=tuple(rc.decoder_layers_per_block),
                            spatial_up_sample=tuple(rc.decoder_spatial_up_sample),
                            temporal_up_sample=tuple(rc.decoder_temporal_up_sample),
                            norm_num_groups=rc.decoder_norm_num_groups, downsample_scale=rc.downsample_scale,
                            enc_in_channels=rc.encoder_in_channels,
                            enc_block_out_channels=tuple(rc.encoder_block_out_channels),
                            enc_layers_per_block=tuple(rc.encoder_layers_per_block),
                            enc_spatial_down_sample=tuple(rc.encoder_spatial_down_sample),
                            enc_temporal_down_sample=tuple(rc.encoder_temporal_down_sample))
        return cls(cfg, ref_vae.state_dict(), device=device)

    @property
    def device(self):
        return self._anchor.device

    @property
    def dtype(self):
        return torch.bfloat16

    # ---- context parallel decode (temporal split + 2-frame halo exchange per causal conv) ------------------------------
    def set_context_parallel(self, group=None) -> None:
        """Split the latent frames over the ranks of `group` following the reference's VAE context-parallel layout
        (video_vae/context_parallel_ops.py:14-38 split, :76-114 halo pass; the reference uses it in training only):
        rank 0 takes the image frame plus its share, every 3x3x3 causal conv receives the last two input frames of the
        previous rank (NCCL p2p over NVLink) instead of the zero / cached halo, and only rank 0 drops the first
        up-sampled frame.  `group=None` = the default process group; world size 1 disables it."""
        import torch.distributed as dist
        self._cp = None
        if not (dist.is_available() and dist.is_initialized()):
            return
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        if world > 1:
            self._cp = (group, rank, world)

    @staticmethod
    def cp_frame_split(n_frames: int, world: int, frames_per_round: int = 4):
        """Context-parallel schedule: a list of rounds, each a list of per-rank latent-frame ranges [a, b).  Round 0 gives rank 0
        the image frame plus `frames_per_round` frames and every other rank `frames_per_round` (the reference's split,
        X:24-33, applied to the first world*c frames); later rounds continue in time order, so a rank never holds more than
        c (+1) latent frames of activations at once — one round covering the whole clip is the reference's layout, but at
        768p it needs ~6 GiB per latent frame (15 frames per rank = 147 GiB measured).  Only the last round may be partial."""
        rounds, f, k = [], 0, 0
        while f < n_frames:
            ranges = []
            for r in range(world):
                ln = frames_per_round + (1 if (k == 0 and r == 0) else 0)
                a, b = min(f, n_frames), min(f + ln, n_frames)
                ranges.append((a, b))
                f = b
            rounds.append(ranges)
            k += 1
        return rounds

    def enable_tiling(self, use_tiling: bool = True):
        self.use_tiling = use_tiling

    def disable_tiling(self):
        self.use_tiling = False

    # ---- kernel wrappers (single sample: tensors are [T, H, W, C]) ---------------------------------------------------
    def _conv(self, cv: _Conv, x: torch.Tensor, t: int, h: int, w: int, *, out: torch.Tensor, out_t_offset: int = 0,
              store_mode: int = 0, residual: Optional[torch.Tensor] = None, res_t_offset: int = 0,
              store_channels: Optional[int] = None, out_f32: int = 0, kernel_variant: int = 0) -> None:
        """t, h, w = OUTPUT dims.  x: [(t-1)*st + kt, h*sh, w*sw, cin_p] (halo frames first); out: [out_t_total, H', W', out_c]."""
        st, sh, sw = cv.stride
        assert x.is_contiguous() and out.is_contiguous() and x.shape[-1] == cv.cin_p
        assert tuple(x.shape[:3]) == ((t - 1) * st + cv.kt, h * sh, w * sw), (tuple(x.shape), t, h, w, cv.stride)
        d = ConvDesc()
        d.stride_t, d.stride_h, d.stride_w = st, sh, sw
        d.x = x.data_ptr()
        d.b, d.t, d.h, d.w, d.cin = 1, t, h, w, cv.cin_p
        d.wgt, d.bias = cv.w.data_ptr(), cv.bias.data_ptr()
        d.cout, d.kt, d.kh, d.kw = cv.cout_p, cv.kt, cv.kh, cv.kw
        d.store_mode = store_mode
        d.out, d.out_f32 = out.data_ptr(), int(out_f32)
        d.out_t_total, d.out_t_offset, d.out_c = out.shape[0], out_t_offset, out.shape[-1]
        d.store_channels = store_channels if store_channels is not None else cv.cout_p
        d.kernel_variant = kernel_variant
        if residual is not None:
            d.residual, d.res_t_total, d.res_t_offset = residual.data_ptr(), residual.shape[0], res_t_offset
        _lib.check(_lib.load().pf_causal_conv3d(C.byref(d), _lib.stream_ptr()), "pf_causal_conv3d")

    def _halo(self, cv: _Conv, buf: torch.Tensor, first: bool) -> None:
        """Fill the 2 leading frames of a 3x3x3 conv's input buffer from its cache (zeros for the first chunk) and
        remember the last 2 frames of the padded input for the next chunk (reference C:126-143).  A stride-2 temporal conv
        reads a later chunk's buffer from frame 1 (see _encode_chunk)."""
        if cv.kt == 1:
            return
        if self._cp is not None:
            # ring of rounds: my halo = the last two (padded) input frames of the rank before me in this round; rank 0 takes
            # the zero pad in round 0 and afterwards what the LAST rank sent it during the previous round (kept in cv.cache)
            import torch.distributed as dist
            group, rank, world = self._cp
            ctx = self._cp_ctx
            peer = (lambda r: dist.get_global_rank(group, r)) if group is not None else (lambda r: r)
            p2p, nxt = [], None
            if ctx["send_next"]:
                p2p.append(dist.P2POp(dist.isend, buf[-2:], peer(rank + 1), group))
            if ctx["ring_send"]:
                p2p.append(dist.P2POp(dist.isend, buf[-2:], peer(0), group))
            if rank > 0:
                p2p.append(dist.P2POp(dist.irecv, buf[:2], peer(rank - 1), group))
            else:
                if ctx["round"] == 0:
                    buf[:2].zero_()
                else:
                    buf[:2].copy_(cv.cache)
                if ctx["ring_recv"]:
                    nxt = torch.empty_like(buf[:2])
                    p2p.append(dist.P2POp(dist.irecv, nxt, peer(world - 1), group))
            for work in (dist.batch_isend_irecv(p2p) if p2p else []):
                work.wait()
            if nxt is not None:
                cv.cache = nxt
            return
        if first or cv.cache is None:
            buf[:2].zero_()
        else:
            buf[:2].copy_(cv.cache)
        cv.cache = buf[-2:].clone()

    def _gn(self, name: str, x: torch.Tensor, y: torch.Tensor, y_t_offset: int, silu: bool) -> None:
        """x [T, H, W, C] -> y [Ty, H, W, C] frames [y_t_offset, y_t_offset + T)."""
        t, h, w, c = x.shape
        groups = self.cfg.norm_num_groups
        stats = torch.empty(t, groups, 2, device=x.device, dtype=torch.float32)
        nsplit = min(64, max(1, (h * w + 4095) // 4096))
        ws = torch.empty(t * nsplit * c * 2, device=x.device, dtype=torch.float32)
        lib = _lib.load()
        _lib.check(lib.pf_groupnorm_stats(x.data_ptr(), t, h * w, c, groups, 1e-6, stats.data_ptr(), ws.data_ptr(),
                                          ws.numel(), _lib.stream_ptr()), "pf_groupnorm_stats")
        g, b = self.norms[name]
        _lib.check(lib.pf_groupnorm_apply(x.data_ptr(), y.data_ptr(), 1, t, h * w, c, groups, stats.data_ptr(),
                                          g.data_ptr(), b.data_ptr(), int(silu), y.shape[0], y_t_offset,
                                          _lib.stream_ptr()), "pf_groupnorm_apply")

    def _resnet(self, pre: str, x: torch.Tensor, first: bool, halo_out: bool = False) -> torch.Tensor:
        """CausalResnetBlock3D (R:115-150). x: [T, H, W, Cin] view; returns [T(+2 if halo_out), H, W, Cout]."""
        t, h, w, cin = x.shape
        c1, c2 = self.convs[pre + ".conv1"], self.convs[pre + ".conv2"]
        dev = x.device
        a = torch.empty(t + 2, h, w, cin, device=dev, dtype=torch.bfloat16)
        self._gn(pre + ".norm1", x, a, 2, True)
        self._halo(c1, a, first)
        h1 = torch.empty(t, h, w, c1.cout_p, device=dev, dtype=torch.bfloat16)
        self._conv(c1, a, t, h, w, out=h1)
        del a
        bbuf = torch.empty(t + 2, h, w, c1.cout_p, device=dev, dtype=torch.bfloat16)
        self._gn(pre + ".norm2", h1, bbuf, 2, True)
        del h1
        self._halo(c2, bbuf, first)
        if (pre + ".conv_shortcut") in self.convs:
            sc_cv = self.convs[pre + ".conv_shortcut"]
            sc = torch.empty(t, h, w, sc_cv.cout_p, device=dev, dtype=torch.bfloat16)
            self._conv(sc_cv, x.contiguous(), t, h, w, out=sc)
        else:
            sc = x
        off = 2 if halo_out else 0
        out = torch.empty(t + off, h, w, c2.cout_p, device=dev, dtype=torch.bfloat16)
        # `sc` may be a contiguous view into a halo'd buffer: its data_ptr already points at the first data frame
        self._conv(c2, bbuf, t, h, w, out=out, out_t_offset=off, residual=sc, res_t_offset=0)
        return out

    def _mid_attention(self, x: torch.Tensor, side: str = "decoder") -> torch.Tensor:
        """Per-frame single-head attention over the h*w tokens (K:454-460 + diffusers Attention). x [T, H, W, C]."""
        at = self.attn[side]
        t, h, w, c = x.shape
        dev = x.device
        n = h * w
        npad = _pad64(n)
        slack = 128
        xn = torch.zeros(t * n + slack, c, device=dev, dtype=torch.bfloat16)
        self._gn(side + ".mid_block.attentions.0.group_norm", x, xn[: t * n].view(t, h, w, c), 0, False)
        q = torch.empty(t, h, w, c, device=dev, dtype=torch.bfloat16)
        k = torch.zeros(t * n + slack, c, device=dev, dtype=torch.bfloat16)
        self._conv(at["q"], xn[: t * n].view(t, h, w, c), t, h, w, out=q)
        self._conv(at["k"], xn[: t * n].view(t, h, w, c), t, h, w, out=k[: t * n].view(t, h, w, c))
        o = torch.empty(t, h, w, c, device=dev, dtype=torch.bfloat16)
        vt = torch.empty(c, npad, device=dev, dtype=torch.bfloat16)
        s = torch.empty(n, npad, device=dev, dtype=torch.bfloat16)
        qf, of = q.view(t, n, c), o.view(t, n, c)
        for f in range(t):
            xf = xn[f * n: f * n + npad]          # rows beyond n are the next frame / zero slack: finite, masked below
            kf = k[f * n: f * n + npad]
            ops.gemm(at["wv"], xf, None, PF_EPI_STORE_BF16, rows_per_batch=c, out=vt)           # V^T [C, npad]
            ops.gemm(qf[f], kf, None, PF_EPI_STORE_BF16, rows_per_batch=n, out=s)               # S = Q K^T
            _lib.check(_lib.load().pf_softmax_rows(s.data_ptr(), n, n, npad, float(c) ** -0.5, _lib.stream_ptr()),
                       "pf_softmax_rows")
            ops.gemm(s, vt, None, PF_EPI_STORE_BF16, rows_per_batch=n, out=of[f])               # O = P V
        out = torch.empty(t, h, w, c, device=dev, dtype=torch.bfloat16)
        self._conv(at["o"], o, t, h, w, out=out, residual=x, res_t_offset=0)
        return out

    def _reset_caches(self):
        for cv in self.convs.values():
            cv.cache = None

    def _decode_chunk(self, z: torch.Tensor, first: bool, affine=None, u8: bool = False) -> torch.Tensor:
        """z: latent frames [1, C, T, h, w] of ONE chunk -> fp32 [T', 8h, 8w, 3] (uint8 frames with u8).
        affine = (scale[T], shift[T]) fp32 device vectors: z*scale[t] + shift[t] fused into the latent pack (the
        un-normalisation of decode_latent, P:1226-1230)."""
        cfg = self.cfg
        dev = self.device
        _, cl, t, h, w = z.shape
        pq, cin = self.convs["post_quant_conv"], self.convs["decoder.conv_in"]
        zin = torch.empty(t, h, w, pq.cin_p, device=dev, dtype=torch.bfloat16)
        zz = z if z.dtype in (torch.float32, torch.bfloat16) else z.float()
        fs, fh = (None, None) if affine is None else (affine[0].data_ptr(), affine[1].data_ptr())
        _lib.check(_lib.load().pf_pack_latent(zz.contiguous().data_ptr(), int(zz.dtype == torch.float32), 1, cl, t, h, w,
                                              zin.data_ptr(), pq.cin_p, t, 0, fs, fh, _lib.stream_ptr()), "pf_pack_latent")
        a = torch.empty(t + 2, h, w, cin.cin_p, device=dev, dtype=torch.bfloat16)
        self._conv(pq, zin, t, h, w, out=a, out_t_offset=2)                      # post_quant_conv (1x1x1), V:365/368
        self._halo(cin, a, first)
        x = torch.empty(t, h, w, cin.cout_p, device=dev, dtype=torch.bfloat16)
        self._conv(cin, a, t, h, w, out=x)                                       # conv_in, D:310
        x = self._resnet("decoder.mid_block.resnets.0", x, first)
        x = self._mid_attention(x, "decoder")
        x = self._resnet("decoder.mid_block.resnets.1", x, first)
        n_blocks = len(cfg.block_out_channels)
        for i in range(n_blocks):
            xb = None
            has_up = cfg.spatial_up_sample[i] or cfg.temporal_up_sample[i]
            for j in range(cfg.layers_per_block[i]):
                last = j == cfg.layers_per_block[i] - 1
                x = self._resnet(f"decoder.up_blocks.{i}.resnets.{j}", x, first, halo_out=last and has_up)
                if last and has_up:
                    xb = x               # [t+2, h, w, c]: data in frames [2:]
            if cfg.spatial_up_sample[i]:
                cv = self.convs[f"decoder.up_blocks.{i}.upsamplers.0.conv"]
                self._halo(cv, xb, first)
                off = 2 if cfg.temporal_up_sample[i] else 0
                y = torch.empty(t + off, 2 * h, 2 * w, cv.cout_p // 4, device=dev, dtype=torch.bfloat16)
                self._conv(cv, xb, t, h, w, out=y, out_t_offset=off, store_mode=1)
                h, w = 2 * h, 2 * w
                xb = y
                x = y[off:]
            if cfg.temporal_up_sample[i]:
                cv = self.convs[f"decoder.up_blocks.{i}.temporal_upsamplers.0.conv"]
                self._halo(cv, xb, first)
                t_out = 2 * t - 1 if first else 2 * t
                y = torch.empty(t_out, h, w, cv.cout_p // 2, device=dev, dtype=torch.bfloat16)
                self._conv(cv, xb, t, h, w, out=y, out_t_offset=-1 if first else 0, store_mode=2)
                t = t_out
                x = y
        co = self.convs["decoder.conv_out"]
        a = torch.empty(t + 2, h, w, x.shape[-1], device=dev, dtype=torch.bfloat16)
        self._gn("decoder.conv_norm_out", x, a, 2, True)
        self._halo(co, a, first)
        out = torch.empty(t, h, w, cfg.out_channels, device=dev, dtype=torch.uint8 if u8 else torch.float32)
        self._conv(co, a, t, h, w, out=out, store_channels=cfg.out_channels, out_f32=2 if u8 else 1)
        return out

    # ---- encoder (i2v image latent P:911, video latents V:274-341) ---------------------------------------------------
    def _encode_chunk(self, x: torch.Tensor, first: bool) -> torch.Tensor:
        """One temporal chunk of one sample -> moments fp32 [T', h, w, 2*latent] (CausalVaeEncoder.forward D:149-198, then
        quant_conv V:301).  x (on the device): [1, C, T, H, W] fp32 / bf16, or uint8 frames [T, H, W, C] normalised by
        pf_pack_frames_u8.  `first` = the clip's first chunk: zero causal pad; later chunks continue from every 3x3x3 conv's
        cache (C:126-143), so the whole clip as one chunk is the un-chunked encode."""
        cfg, dev = self.cfg, self.device
        if x.dtype == torch.uint8:
            t, h, w, cx = x.shape
        else:
            _, cx, t, h, w = x.shape
        n_blocks = len(cfg.enc_block_out_channels)
        n_sp = sum(cfg.enc_spatial_down_sample)
        assert h % (1 << n_sp) == 0 and w % (1 << n_sp) == 0, "height / width must be divisible by the spatial down-sampling"
        cin = self.convs["encoder.conv_in"]
        a = torch.empty(t + 2, h, w, cin.cin_p, device=dev, dtype=torch.bfloat16)
        if x.dtype == torch.uint8:
            _lib.check(_lib.load().pf_pack_frames_u8(x.contiguous().data_ptr(), 1, t, h, w, cx, a.data_ptr(), cin.cin_p, t + 2,
                                                     2, _lib.stream_ptr()), "pf_pack_frames_u8")
        else:
            xx = x if x.dtype in (torch.float32, torch.bfloat16) else x.float()
            _lib.check(_lib.load().pf_pack_latent(xx.contiguous().data_ptr(), int(xx.dtype == torch.float32), 1, cx, t, h, w,
                                                  a.data_ptr(), cin.cin_p, t + 2, 2, None, None, _lib.stream_ptr()),
                       "pf_pack_latent")
        self._halo(cin, a, first)
        y = torch.empty(t, h, w, cin.cout_p, device=dev, dtype=torch.bfloat16)
        self._conv(cin, a, t, h, w, out=y)                                        # conv_in, D:152
        del a
        for i in range(n_blocks):
            sp, tp = cfg.enc_spatial_down_sample[i], cfg.enc_temporal_down_sample[i]
            xb = None
            for j in range(cfg.enc_layers_per_block[i]):
                last = j == cfg.enc_layers_per_block[i] - 1
                y = self._resnet(f"encoder.down_blocks.{i}.resnets.{j}", y, first, halo_out=last and (sp or tp))
                if last and (sp or tp):
                    xb = y                                  # [t+2, h, w, c]: data in frames [2:]
            if sp:                                          # CausalDownsample2x: 3x3x3, stride (1,2,2), K:532-534
                cv = self.convs[f"encoder.down_blocks.{i}.downsamplers.0.conv"]
                self._halo(cv, xb, first)
                off = 2 if tp else 0
                h, w = h // 2, w // 2
                y = torch.empty(t + off, h, w, cv.cout_p, device=dev, dtype=torch.bfloat16)
                self._conv(cv, xb, t, h, w, out=y, out_t_offset=off)
                xb = y
                y = y[off:]
            if tp:                                          # CausalTemporalDownsample2x: 3x3x3, stride (2,1,1), K:536-538
                cv = self.convs[f"encoder.down_blocks.{i}.temporal_downsamplers.0.conv"]
                self._halo(cv, xb, first)
                # a later chunk's input is [cache[-1:] ; chunk] (C:140-141): the older cached frame is skipped.  The cache
                # _halo kept is still the last two frames of that input, whether or not the strided conv reads the last one.
                src = xb if first else xb[1:]
                assert src.shape[0] >= 3, "a later temporal chunk is too short for the stride-2 conv (window_size >= 2)"
                t_out = (src.shape[0] - 3) // 2 + 1
                y = torch.empty(t_out, h, w, cv.cout_p, device=dev, dtype=torch.bfloat16)
                self._conv(cv, src[: 2 * (t_out - 1) + 3], t_out, h, w, out=y)
                t = t_out
        y = self._resnet("encoder.mid_block.resnets.0", y, first)
        y = self._mid_attention(y, "encoder")
        y = self._resnet("encoder.mid_block.resnets.1", y, first)
        co, qc = self.convs["encoder.conv_out"], self.convs["quant_conv"]
        a = torch.empty(t + 2, h, w, y.shape[-1], device=dev, dtype=torch.bfloat16)
        self._gn("encoder.conv_norm_out", y, a, 2, True)
        self._halo(co, a, first)
        m = torch.zeros(t, h, w, qc.cin_p, device=dev, dtype=torch.bfloat16)      # padded channels must read as zero
        self._conv(co, a, t, h, w, out=m, store_channels=co.cout)                 # conv_out -> 2*latent channels
        out = torch.empty(t, h, w, qc.cout, device=dev, dtype=torch.float32)
        self._conv(qc, m, t, h, w, out=out, store_channels=qc.cout, out_f32=True)  # quant_conv (1x1x1), V:301
        return out

    @staticmethod
    def chunk_bounds(n_frames: int, window_size: int):
        """Temporal chunks [a, b) of chunk_encode / chunk_decode (V:311-327, V:347-360): the first window_size + 1 frames,
        then full windows of window_size, then the remainder."""
        init = min(n_frames, window_size + 1)
        bounds, f = [(0, init)], init
        while f < n_frames:
            bounds.append((f, min(n_frames, f + window_size)))
            f += window_size
        return bounds

    @staticmethod
    def encode_tile_grid(height: int, width: int, tile_sample_min_size: int, overlap_factor: float = 0.25,
                         downsample: int = 8):
        """Tile geometry of tiled_encode (V:429-438): tile origins (rows, columns) in pixels, every tile_sample_min_size
        wide (edge tiles are cut by the frame), the latent blend extent and the latent rows / columns kept per tile."""
        tile_latent = int(tile_sample_min_size / downsample)
        stride = int(tile_sample_min_size * (1 - overlap_factor))
        extent = int(tile_latent * overlap_factor)
        return list(range(0, height, stride)), list(range(0, width, stride)), extent, tile_latent - extent

    @staticmethod
    def _window(x: torch.Tensor, b: int, ts=slice(None), hs=slice(None), ws=slice(None)) -> torch.Tensor:
        """Sample b, frames ts, rows hs, columns ws of a clip [B, C, T, H, W] (-> [1, C, t, h, w]) or of uint8 frames
        [B, T, H, W, C] (-> [t, h, w, C])."""
        return x[b, ts, hs, ws] if x.dtype == torch.uint8 else x[b:b + 1, :, ts, hs, ws]

    def _encode_moments(self, x: torch.Tensor, window: int, hs=slice(None), ws=slice(None)) -> torch.Tensor:
        """chunk_encode (V:311-341) of rows hs / columns ws of every sample, with `window` frames per chunk (the whole clip
        when window >= T - 1): moments fp32 [B, T', h, w, 2*latent].  Chunks move to the device one at a time, so a clip on
        the host never has to be resident on the device."""
        n = x.shape[1] if x.dtype == torch.uint8 else x.shape[2]
        n_tp = sum(self.cfg.enc_temporal_down_sample)
        assert (n - 1) % (1 << n_tp) == 0, "frames must be 1 + k * temporal down-sampling (V:315)"
        outs = []
        for b in range(x.shape[0]):
            self._reset_caches()
            parts = [self._encode_chunk(self._window(x, b, slice(f0, f1), hs, ws).to(self.device), k == 0)
                     for k, (f0, f1) in enumerate(self.chunk_bounds(n, window))]
            self._reset_caches()
            outs.append(torch.cat(parts, 0) if len(parts) > 1 else parts[0])
        return torch.stack(outs, 0)

    def _tiled_encode(self, x: torch.Tensor, window: int, tile_sample_min_size: int) -> torch.Tensor:
        """tiled_encode (V:409-466): tiles encoded independently (chunked with `window`), fp32 moments cross-faded with the
        tile above and to the left, then cropped -> [B, 2*latent, T', h, w]."""
        hh, ww = (x.shape[2], x.shape[3]) if x.dtype == torch.uint8 else (x.shape[3], x.shape[4])
        row0, col0, extent, limit = self.encode_tile_grid(hh, ww, tile_sample_min_size, self.encode_tile_overlap_factor,
                                                          self.cfg.downsample_scale)
        s = tile_sample_min_size
        rows = [[self._encode_moments(x, window, slice(i, i + s), slice(j, j + s)).permute(0, 4, 1, 2, 3).contiguous()
                 for j in col0] for i in row0]
        result_rows = []
        for i, row in enumerate(rows):
            res = []
            for j, tile in enumerate(row):
                if i > 0:
                    tile = _blend(rows[i - 1][j], tile, extent, 3)
                if j > 0:
                    tile = _blend(row[j - 1], tile, extent, 4)
                res.append(tile[:, :, :, :limit, :limit])
            result_rows.append(torch.cat(res, dim=4))
        return torch.cat(result_rows, dim=3)

    def _encode(self, x: torch.Tensor, temporal_chunk: bool, window_size: int, tile_sample_min_size: int):
        """The control flow of CausalVideoVAE.encode (V:290-303): tiled when tiling is on and the frame is larger than the
        tile, else chunked with temporal_chunk, else the whole clip as one chunk.  x: [B, C, T, H, W] or uint8 frames
        [B, T, H, W, C], on the host or the device."""
        _lib.require_device()
        assert self.has_encoder, "this B200CausalVAE was built from a state-dict without encoder.* weights"
        t, hh, ww = x.shape[1:4] if x.dtype == torch.uint8 else x.shape[2:5]
        assert window_size >= 1 or not temporal_chunk, "window_size must be positive"
        window = window_size if temporal_chunk else t
        saved_cp, self._cp = self._cp, None
        try:
            if self.use_tiling and (ww > tile_sample_min_size or hh > tile_sample_min_size):
                moments = self._tiled_encode(x, window, tile_sample_min_size)
            else:
                moments = self._encode_moments(x, window).permute(0, 4, 1, 2, 3)       # [B, T', h, w, 2C] -> [B, 2C, ...]
        finally:
            self._cp = saved_cp
        return EncoderOutput(DiagonalGaussian(moments.to(self.dtype)))

    @torch.no_grad()
    def encode(self, x: torch.Tensor, return_dict: bool = True, is_init_image: bool = True, temporal_chunk: bool = False,
               window_size: int = 16, tile_sample_min_size: int = 256):
        """CausalVideoVAE.encode (V:274-308): x [B, 3, T, H, W] (T = 1 + 8k) on the host or the device.  With
        enable_tiling() and a frame larger than tile_sample_min_size the frame is encoded in tiles (tiled_encode,
        V:409-466), otherwise in chunks of window_size frames with temporal_chunk (chunk_encode, V:311-341), otherwise whole.
        is_init_image has no effect on the result, as in the reference.  Returns `.latent_dist` with mean / logvar / std /
        sample()."""
        out = self._encode(x, temporal_chunk, window_size, tile_sample_min_size)
        return out if return_dict else (out.latent_dist,)

    @torch.no_grad()
    def encode_frames_u8(self, frames: torch.Tensor, temporal_chunk: bool = True, window_size: int = 16,
                         tile_sample_min_size: int = 256) -> EncoderOutput:
        """encode() of video frames as they are decoded from a file: uint8 [T, H, W, 3] or [B, T, H, W, 3], on the host or
        the device.  ToTensor + Normalize(0.5, 0.5) (P:906-910) runs in pf_pack_frames_u8 on the device, and only uint8
        tiles / chunks cross from the host.  Same tiling and chunking rules and result as encode() of the normalised
        frames in bf16."""
        assert frames.dtype == torch.uint8 and frames.dim() in (4, 5), "frames must be uint8 [(B,) T, H, W, C]"
        return self._encode(frames if frames.dim() == 5 else frames[None], temporal_chunk, window_size, tile_sample_min_size)

    def _decode_sample_cp(self, z: torch.Tensor) -> torch.Tensor:
        """Context-parallel decode of one sample (schedule: cp_frame_split): per round every rank decodes its frame range as
        ONE chunk with the halo of every causal conv passed along the ring; the decoded frames of each round are
        all-gathered in time order (every rank returns the full clip)."""
        import torch.distributed as dist
        group, rank, world = self._cp
        n = z.shape[2]
        c = max(2, min(self.cp_frames_per_round, -(-(n - 1) // world)))     # short clips: spread the frames over all ranks
        rounds = self.cp_frame_split(n, world, c)
        self._reset_caches()
        outs = []
        up = 2 ** sum(bool(x) for x in self.cfg.spatial_up_sample)
        tail_shape = (z.shape[3] * up, z.shape[4] * up, self.cfg.out_channels)
        for k, ranges in enumerate(rounds):
            a, b = ranges[rank]
            more = k + 1 < len(rounds)
            self._cp_ctx = dict(round=k,
                                send_next=rank + 1 < world and ranges[rank + 1][1] > ranges[rank + 1][0] and b > a,
                                ring_send=more and rank == world - 1, ring_recv=more and rank == 0)
            mine = self._decode_chunk(z[:, :, a:b].contiguous(), k == 0 and rank == 0) if b > a else None
            tf = 2 ** sum(1 for u in self.cfg.temporal_up_sample if u)      # temporal up-sampling factor of this decoder (8 by default)
            counts = [tf * (e - s0) - ((tf - 1) if (k == 0 and r == 0) else 0) if e > s0 else 0 for r, (s0, e) in enumerate(ranges)]
            if mine is not None:
                assert mine.shape[0] == counts[rank] and tuple(mine.shape[1:]) == tail_shape, (mine.shape, counts, rank)
            pad = torch.zeros(max(counts), *tail_shape, device=self.device, dtype=torch.float32)
            if mine is not None:
                pad[: mine.shape[0]] = mine
            parts = [torch.empty_like(pad) for _ in range(world)]
            dist.all_gather(parts, pad, group=group)
            outs.extend(p_[:c] for p_, c in zip(parts, counts) if c > 0)
        self._cp_ctx = None
        self._reset_caches()
        return torch.cat(outs, 0)

    def _decode_sample(self, z: torch.Tensor, window_size: int, affine=None, u8: bool = False) -> torch.Tensor:
        """chunk_decode (V:346-374) for one sample: first chunk window+1 latent frames, then `window` each."""
        if self._cp is not None:
            assert affine is None and not u8, "the fused un-normalise / uint8 path is single-GPU (decode_latent_u8 falls back)"
            if z.shape[2] - 1 >= 2 * self._cp[2] and self.cp_frames_per_round >= 2:   # full shares own their halo source
                return self._decode_sample_cp(z)
            saved, self._cp = self._cp, None              # short clip: every rank decodes all of it (replicas)
            try:
                return self._decode_sample(z, window_size)
            finally:
                self._cp = saved
        self._reset_caches()
        bounds = self.chunk_bounds(z.shape[2], window_size)
        if affine is None and not u8:
            outs = [self._decode_chunk(z[:, :, a:b], i == 0) for i, (a, b) in enumerate(bounds)]
        else:
            outs = [self._decode_chunk(z[:, :, a:b], i == 0, None if affine is None else (affine[0][a:b], affine[1][a:b]), u8)
                    for i, (a, b) in enumerate(bounds)]
        self._reset_caches()
        return torch.cat(outs, 0) if len(outs) > 1 else outs[0]

    @torch.no_grad()
    def decode(self, z: torch.Tensor, is_init_image: bool = True, temporal_chunk: bool = False, return_dict: bool = True,
               window_size: int = 2, tile_sample_min_size: int = 256):
        _lib.require_device()
        assert is_init_image, "the sampler always decodes clips that start with the image frame"
        z = z.to(self.device)
        tile_latent = int(tile_sample_min_size / self.cfg.downsample_scale)
        if self.use_tiling and (z.shape[-1] > tile_latent or z.shape[-2] > tile_latent):
            dec = self._tiled_decode(z, window_size if temporal_chunk else z.shape[2], tile_sample_min_size)
        else:
            w = window_size if temporal_chunk else z.shape[2]
            outs = [self._decode_sample(z[i:i + 1], w) for i in range(z.shape[0])]
            dec = torch.stack(outs, 0).permute(0, 4, 1, 2, 3)      # [B, T, H, W, 3] -> view as [B, 3, T, H, W]
        if not return_dict:
            return (dec,)
        return DecoderOutput(dec)

    @torch.no_grad()
    def decode_latent_u8(self, latents: torch.Tensor, scale: float, shift: float, video_scale: float, video_shift: float,
                         window_size: int = 1, tile_sample_min_size: int = 256) -> torch.Tensor:
        """decode_latent (P:1221-1243) in one pass: the per-frame un-normalisation  z / scale + shift  (first frame: image
        constants, the rest: video constants, P:1226-1230) is fused into the latent pack kernel and the
        `mul(127.5).add(127.5).clamp(0, 255).byte()` of P:1238 into conv_out's epilogue: the decoder writes uint8 frames
        [(B T), H, W, 3] directly (1 B/value instead of a 4 B fp32 image + 3 torch passes).  Tiled or context-parallel
        decodes blend / gather fp32 tiles, so they take the two-step path."""
        _lib.require_device()
        z = latents.to(self.device)
        b, _, t = z.shape[:3]
        tile_latent = int(tile_sample_min_size / self.cfg.downsample_scale)
        if (self.use_tiling and (z.shape[-1] > tile_latent or z.shape[-2] > tile_latent)) or self._cp is not None:
            zz = z.clone().float()
            zz[:, :, :1] = zz[:, :, :1] / scale + shift
            if t > 1:
                zz[:, :, 1:] = zz[:, :, 1:] / video_scale + video_shift
            img = self.decode(zz.to(z.dtype), temporal_chunk=True, window_size=window_size,
                              tile_sample_min_size=tile_sample_min_size).sample
            img = img.float().mul(127.5).add(127.5).clamp(0, 255).byte()
            return img.permute(0, 2, 3, 4, 1).reshape(-1, img.shape[3], img.shape[4], img.shape[1])
        fs = torch.full((t,), 1.0 / video_scale, device=self.device, dtype=torch.float32)
        fh = torch.full((t,), float(video_shift), device=self.device, dtype=torch.float32)
        fs[0], fh[0] = 1.0 / scale, float(shift)
        outs = [self._decode_sample(z[i:i + 1], window_size, affine=(fs, fh), u8=True) for i in range(b)]
        return torch.cat(outs, 0)                      # [(B T'), H, W, 3] uint8

    def _tiled_decode(self, z: torch.Tensor, window: int, tile_sample_min_size: int) -> torch.Tensor:
        """tiled_decode (V:468-519): independent tiles, linear cross-fade with the tile above and to the left."""
        tile_latent = int(tile_sample_min_size / self.cfg.downsample_scale)
        overlap = int(tile_latent * (1 - self.decode_tile_overlap_factor))
        extent = int(tile_sample_min_size * self.decode_tile_overlap_factor)
        limit = tile_sample_min_size - extent
        rows = []
        for i in range(0, z.shape[3], overlap):
            row = []
            for j in range(0, z.shape[4], overlap):
                tile = z[:, :, :, i:i + tile_latent, j:j + tile_latent]
                outs = [self._decode_sample(tile[b:b + 1].contiguous(), window) for b in range(z.shape[0])]
                row.append(torch.stack(outs, 0).permute(0, 4, 1, 2, 3).contiguous())
            rows.append(row)
        result_rows = []
        for i, row in enumerate(rows):
            res = []
            for j, tile in enumerate(row):
                if i > 0:
                    tile = _blend(rows[i - 1][j], tile, extent, 3)
                if j > 0:
                    tile = _blend(row[j - 1], tile, extent, 4)
                res.append(tile[:, :, :, :limit, :limit])
            result_rows.append(torch.cat(res, dim=4))
        return torch.cat(result_rows, dim=3)


def _blend(a: torch.Tensor, b: torch.Tensor, extent: int, dim: int) -> torch.Tensor:
    """blend_v / blend_h (V:397-407): b[..., y, ...] = a[..., -extent+y, ...]*(1-y/extent) + b*(y/extent), one kernel
    (pf_blend_tiles) on the contiguous fp32 tiles, in place on b."""
    extent = min(a.shape[dim], b.shape[dim], extent)
    if extent <= 0:
        return b
    assert a.is_contiguous() and b.is_contiguous() and a.dtype == torch.float32 and b.dtype == torch.float32
    assert a.shape[:dim] == b.shape[:dim] and a.shape[dim + 1:] == b.shape[dim + 1:], "tiles must agree off the blended axis"
    outer = 1
    for n in b.shape[:dim]:
        outer *= int(n)
    inner = 1
    for n in b.shape[dim + 1:]:
        inner *= int(n)
    _lib.check(_lib.load().pf_blend_tiles(a.data_ptr(), b.data_ptr(), outer, a.shape[dim], b.shape[dim], inner, extent,
                                          _lib.stream_ptr()), "pf_blend_tiles")
    return b
