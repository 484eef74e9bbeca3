"""Dependency shim so the UNMODIFIED reference (a jy0205/Pyramid-Flow checkout) imports without its pip dependencies.

TEST INFRASTRUCTURE, used by oracle/pin/make_golden.py to pin the oracle restatement and to generate tests/golden/*, and by
bench.py's optional `gpu_eager_baseline` leg.  No test and no product module imports this.

The image lacks diffusers / accelerate / timm / tensorboardX / IPython (SURVEY.md §8c).  The pieces of those packages
the reference touches at import time are stubbed; the four that carry arithmetic are restated from the diffusers 0.30
semantics (requirements.txt:6 pins diffusers>=0.30.1):
  * diffusers.models.activations.GELU            -> F.gelu(Linear(x), approximate=...)         (call sites B:73-75, MB:57-59)
  * diffusers.models.attention_processor.Attention with _from_deprecated_attn_block=True        (VAE mid block K:413-427, K:458)
  * diffusers.models.activations.get_activation  -> nn.SiLU for "silu"/"swish"
  * diffusers.utils.torch_utils.randn_tensor     -> CPU-generator-then-move semantics           (P:694)
"""
from __future__ import annotations

import functools
import inspect
import sys
import types
from dataclasses import dataclass

import torch
import torch.nn as nn
import torch.nn.functional as F

import os as _os

# the checkout named by $PF_REFERENCE_ROOT, else the byte-for-byte copy oracle/pin/stage_reference.py staged in oracle/_ref
_STAGED = _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__)))), "oracle", "_ref")
REFERENCE_ROOT = _os.environ.get("PF_REFERENCE_ROOT") or _STAGED


def reference_available() -> bool:
    return _os.path.isdir(_os.path.join(REFERENCE_ROOT, "pyramid_dit"))



def _mod(name: str) -> types.ModuleType:
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__path__ = []  # behave like a package
    sys.modules[name] = m
    if "." in name:
        parent, child = name.rsplit(".", 1)
        setattr(_mod(parent), child, m)
    return m


class _Config(dict):
    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e


class ConfigMixin:
    config_name = "config.json"

    def register_to_config(self, **kw):
        if not hasattr(self, "_internal_dict"):
            object.__setattr__(self, "_internal_dict", _Config())
        self._internal_dict.update(kw)

    @property
    def config(self):
        return self._internal_dict


def register_to_config(init):
    @functools.wraps(init)
    def inner(self, *args, **kwargs):
        sig = inspect.signature(init)
        params = [p for n, p in sig.parameters.items() if n != "self"]
        cfg = {p.name: p.default for p in params if p.default is not inspect.Parameter.empty}
        for p, a in zip(params, args):
            cfg[p.name] = a
        cfg.update(kwargs)
        ConfigMixin.register_to_config(self, **cfg)  # BEFORE the body runs (S:65 reads self.config in __init__)
        init(self, *args, **kwargs)
    return inner


class ModelMixin(nn.Module):
    @property
    def device(self):
        return next(self.parameters()).device

    @property
    def dtype(self):
        return next(self.parameters()).dtype


class SchedulerMixin:
    pass


class BaseOutput:
    """Attribute-style outputs; the reference only reads named fields (.prev_sample, .sample, .latent_dist)."""

    def __getitem__(self, i):
        return tuple(self.__dict__.values())[i]


@dataclass
class AutoencoderKLOutput(BaseOutput):
    latent_dist: object = None


class _Logger:
    def __getattr__(self, name):
        return lambda *a, **k: None


class _Logging:
    @staticmethod
    def get_logger(name=None):
        return _Logger()


def is_torch_version(op: str, ver: str) -> bool:
    from packaging import version
    import operator
    ops = {">": operator.gt, ">=": operator.ge, "==": operator.eq, "<": operator.lt, "<=": operator.le}
    return ops[op](version.parse(torch.__version__.split("+")[0]), version.parse(ver))


def deprecate(*a, **k):
    return None


def randn_tensor(shape, generator=None, device=None, dtype=None, layout=None):
    """diffusers.utils.torch_utils.randn_tensor: sample on the generator's device (CPU), then move."""
    rand_device = device
    if generator is not None:
        gen_device = generator.device.type if not isinstance(generator, list) else generator[0].device.type
        if gen_device != (device.type if isinstance(device, torch.device) else str(device)) and gen_device == "cpu":
            rand_device = "cpu"
    return torch.randn(shape, generator=generator, device=rand_device, dtype=dtype).to(device)


# ---- diffusers.models.activations ---------------------------------------------------------------------------------
class GELU(nn.Module):
    def __init__(self, dim_in: int, dim_out: int, approximate: str = "none", bias: bool = True):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out, bias=bias)
        self.approximate = approximate

    def forward(self, hidden_states):
        return F.gelu(self.proj(hidden_states), approximate=self.approximate)


class _Unused(nn.Module):
    def __init__(self, *a, **k):
        raise NotImplementedError("not on the hot path")


class FP32SiLU(nn.Module):
    def forward(self, x):
        return F.silu(x.float(), inplace=False).to(x.dtype)


def get_activation(name: str):
    name = name.lower()
    if name in ("silu", "swish"):
        return nn.SiLU()
    if name == "mish":
        return nn.Mish()
    if name == "gelu":
        return nn.GELU()
    if name == "relu":
        return nn.ReLU()
    raise ValueError(name)


# ---- diffusers.models.attention_processor.Attention (deprecated-attn-block form used by the VAE mid block) --------
class Attention(nn.Module):
    def __init__(self, query_dim, heads=8, dim_head=64, rescale_output_factor=1.0, eps=1e-5, norm_num_groups=None,
                 spatial_norm_dim=None, residual_connection=False, bias=False, upcast_softmax=False,
                 _from_deprecated_attn_block=False, **unused):
        super().__init__()
        assert spatial_norm_dim is None
        self.inner_dim = dim_head * heads
        self.heads = heads
        self.rescale_output_factor = rescale_output_factor
        self.residual_connection = residual_connection
        self.group_norm = nn.GroupNorm(num_channels=query_dim, num_groups=norm_num_groups, eps=eps, affine=True) \
            if norm_num_groups is not None else None
        self.to_q = nn.Linear(query_dim, self.inner_dim, bias=bias)
        self.to_k = nn.Linear(query_dim, self.inner_dim, bias=bias)
        self.to_v = nn.Linear(query_dim, self.inner_dim, bias=bias)
        self.to_out = nn.ModuleList([nn.Linear(self.inner_dim, query_dim, bias=True), nn.Dropout(0.0)])

    def forward(self, hidden_states, temb=None, **kw):
        residual = hidden_states
        b, c, h, w = hidden_states.shape
        x = hidden_states.view(b, c, h * w).transpose(1, 2)
        if self.group_norm is not None:
            x = self.group_norm(x.transpose(1, 2)).transpose(1, 2)
        q, k, v = self.to_q(x), self.to_k(x), self.to_v(x)
        hd = self.inner_dim // self.heads
        q = q.view(b, -1, self.heads, hd).transpose(1, 2)
        k = k.view(b, -1, self.heads, hd).transpose(1, 2)
        v = v.view(b, -1, self.heads, hd).transpose(1, 2)
        x = F.scaled_dot_product_attention(q, k, v, dropout_p=0.0, is_causal=False)
        x = x.transpose(1, 2).reshape(b, -1, self.heads * hd).to(q.dtype)
        x = self.to_out[1](self.to_out[0](x))
        x = x.transpose(-1, -2).reshape(b, c, h, w)
        if self.residual_connection:
            x = x + residual
        return x / self.rescale_output_factor


def install() -> None:
    """Register the stubs and put REFERENCE_ROOT on sys.path."""
    import transformers  # noqa: F401  (must be imported before a version-less `accelerate` stub exists)

    d = _mod("diffusers")
    d.__version__ = "0.30.1"
    du = _mod("diffusers.utils")
    du.is_torch_version = is_torch_version
    du.deprecate = deprecate
    du.BaseOutput = BaseOutput
    du.logging = _Logging
    du.is_wandb_available = lambda: False
    dut = _mod("diffusers.utils.torch_utils")
    dut.randn_tensor = randn_tensor
    dc = _mod("diffusers.configuration_utils")
    dc.ConfigMixin = ConfigMixin
    dc.register_to_config = register_to_config
    _mod("diffusers.models")
    dmm = _mod("diffusers.models.modeling_utils")
    dmm.ModelMixin = ModelMixin
    da = _mod("diffusers.models.activations")
    da.GELU = GELU
    da.GEGLU = _Unused
    da.ApproximateGELU = _Unused
    da.SwiGLU = _Unused
    da.FP32SiLU = FP32SiLU
    da.get_activation = get_activation
    dap = _mod("diffusers.models.attention_processor")
    dap.Attention = Attention
    for n in ("SpatialNorm", "AttentionProcessor", "AttnProcessor", "AttnAddedKVProcessor"):
        setattr(dap, n, _Unused)
    dap.ADDED_KV_ATTENTION_PROCESSORS = ()
    dap.CROSS_ATTENTION_PROCESSORS = ()
    dl = _mod("diffusers.models.lora")
    dl.LoRACompatibleConv = nn.Conv2d
    dl.LoRACompatibleLinear = nn.Linear
    dn = _mod("diffusers.models.normalization")
    dn.AdaGroupNorm = _Unused
    dmo = _mod("diffusers.models.modeling_outputs")
    dmo.AutoencoderKLOutput = AutoencoderKLOutput
    _mod("diffusers.schedulers")
    dsu = _mod("diffusers.schedulers.scheduling_utils")
    dsu.SchedulerMixin = SchedulerMixin

    acc = _mod("accelerate")
    acc.Accelerator = object
    acc.cpu_offload = lambda *a, **k: None
    acc.FullyShardedDataParallelPlugin = object
    acc.__version__ = "1.0.0"
    _mod("accelerate.utils")

    _mod("timm")
    _mod("timm.models")
    tl = _mod("timm.models.layers")
    tl.trunc_normal_ = nn.init.trunc_normal_
    tl.drop_path = lambda x, *a, **k: x
    tl.to_2tuple = lambda x: x if isinstance(x, tuple) else (x, x)
    _mod("timm.models.hub")

    tb = _mod("tensorboardX")
    tb.SummaryWriter = object
    ip = _mod("IPython")
    ip.embed = lambda *a, **k: None

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def reinit_all_parameters(module: nn.Module, seed: int, std: float = 0.02) -> None:
    """The reference zero-inits AdaLN / output layers (F:168-183) => a fresh model outputs exactly 0.  Parity needs
    every parameter non-trivial: weights N(0, std^2), biases N(0, std^2), norm weights 1 + N(0, 0.1^2)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            if p.ndim >= 2:
                p.copy_(torch.randn(p.shape, generator=g) * std)
            elif name.endswith("weight"):  # norm weights (RMSNorm / GroupNorm)
                p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=g))
            else:
                p.copy_(torch.randn(p.shape, generator=g) * std)
