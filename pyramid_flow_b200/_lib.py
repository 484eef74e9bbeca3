"""ctypes binding of libpf_b200.so (the C-ABI declared in include/pf_b200.h).

PyTorch is used only for device memory and streams: every call passes raw `data_ptr()`s and the current CUDA stream.
There is no fallback: if the library is missing or the device is not sm_100, calls raise RuntimeError.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libpf_b200.so"

# every symbol include/pf_b200.h declares (tests check the .so exports exactly these)
SYMBOLS = [
    "pf_last_error", "pf_version", "pf_device_check", "pf_warmup", "pf_set_option", "pf_get_option", "pf_launch_count",
    "pf_gemm_bf16",
    "pf_attn_build_schedule", "pf_attn_build_pair_schedule", "pf_attn_build_pair_masks", "pf_attn_build_group_schedule",
    "pf_attn_build_group_masks", "pf_attn_fwd_masked",
    "pf_ln_modulate", "pf_small_linear", "pf_timestep_embedding",
    "pf_patchify", "pf_unpatchify", "pf_cfg_euler_step", "pf_stage_hop",
    "pf_causal_conv3d", "pf_groupnorm_stats", "pf_groupnorm_apply", "pf_softmax_rows", "pf_pack_latent", "pf_pack_frames_u8",
    "pf_blend_tiles", "pf_ctx_create", "pf_ctx_destroy", "pf_ctx_record_begin", "pf_ctx_record_end", "pf_ctx_replay", "pf_dit_step_flux",
    "pf_dit_step_mmdit", "pf_vae_decode_chunk",
    "pf_peer_alloc", "pf_peer_free", "pf_peer_export", "pf_peer_open", "pf_peer_close", "pf_peer_barrier", "pf_peer_bcast",
    "pf_debug_umma",
    "pf_debug_attn_trace",
    "pf_debug_attn_cta_trace",
]

PF_OPT_GEMM_STAGED_RESID, PF_OPT_GEMM_WAVE_TILING, PF_OPT_ATTN_PAIR_KERNEL, PF_OPT_ATTN_TILE_PHASE, PF_OPT_ATTN_TRIPLE_KERNEL = range(5)
PF_EPI_STORE_BF16, PF_EPI_GELU_BF16, PF_EPI_STORE_F32, PF_EPI_GATE_RESID, PF_EPI_QKV_ROPE, PF_EPI_QKV_GELU = range(6)


class GemmDesc(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("lda", C.c_int64),
        ("batches", C.c_int32), ("rows_per_batch", C.c_int32), ("row_begin", C.c_int32), ("row_count", C.c_int32),
        ("w", C.c_void_p), ("n", C.c_int32), ("k", C.c_int32),
        ("bias", C.c_void_p), ("epilogue", C.c_int32),
        ("out", C.c_void_p), ("ldo", C.c_int64),
        ("out_batch_rows", C.c_int32), ("out_row_begin", C.c_int32), ("out_col_begin", C.c_int32),
        ("gate", C.c_void_p), ("gate_batch_stride", C.c_int64),
        ("q_out", C.c_void_p), ("k_out", C.c_void_p), ("v_out", C.c_void_p),
        ("rope", C.c_void_p), ("q_norm_w", C.c_void_p), ("k_norm_w", C.c_void_p),
        ("norm_eps", C.c_float),
        ("heads", C.c_int32), ("head_dim", C.c_int32), ("seq_len", C.c_int32),
        ("n_split", C.c_int32), ("kernel_variant", C.c_int32),
        ("peer_qkv", C.c_void_p * 8),
        ("peer_count", C.c_int32), ("peer_heads", C.c_int32), ("peer_seq", C.c_int32), ("peer_row0", C.c_int32),
    ]


class AttnDesc(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p), ("ldo", C.c_int64),
        ("batch", C.c_int32), ("heads", C.c_int32), ("seq", C.c_int32), ("head_dim", C.c_int32),
        ("scale", C.c_float),
        ("seg", C.c_void_p), ("time", C.c_void_p), ("tile_sched", C.c_void_p),
        ("sched_stride", C.c_int32), ("variant", C.c_int32), ("q_row_begin", C.c_int32),
        ("pair_sched", C.c_void_p),
        ("pair_mask_index", C.c_void_p), ("pair_mask_bits", C.c_void_p),
        ("peer_out", C.c_void_p * 8),
        ("peer_count", C.c_int32), ("peer_chunk_rows", C.c_int32), ("peer_col_begin", C.c_int32),
        ("group_sched", C.c_void_p), ("group_mask_index", C.c_void_p), ("group_mask_bits", C.c_void_p),
    ]


class PeerGroup(C.Structure):
    _fields_ = [("ptr", C.c_void_p * 8), ("n", C.c_int32), ("my_index", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("x", C.c_void_p),
        ("b", C.c_int32), ("t", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("cin", C.c_int32),
        ("wgt", C.c_void_p), ("bias", C.c_void_p),
        ("cout", C.c_int32), ("kt", C.c_int32), ("kh", C.c_int32), ("kw", C.c_int32),
        ("store_mode", C.c_int32),
        ("out", C.c_void_p), ("out_f32", C.c_int32),
        ("out_t_total", C.c_int32), ("out_t_offset", C.c_int32), ("out_c", C.c_int32),
        ("store_channels", C.c_int32),
        ("residual", C.c_void_p), ("res_t_total", C.c_int32), ("res_t_offset", C.c_int32),
        ("stride_t", C.c_int32), ("stride_h", C.c_int32), ("stride_w", C.c_int32), ("kernel_variant", C.c_int32),
    ]


class UmmaProbe(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("b", C.c_void_p), ("d", C.c_void_p),
        ("n", C.c_int32), ("k", C.c_int32),
        ("b_rows", C.c_int32), ("b_cols", C.c_int32), ("b_box_rows", C.c_int32), ("b_mn_major", C.c_int32),
        ("b_lbo", C.c_uint32), ("b_sbo", C.c_uint32), ("b_k_step_bytes", C.c_uint32), ("b_kblock_bytes", C.c_uint32),
        ("a_from_tmem", C.c_int32), ("a_rows", C.c_int32), ("a_row_offset", C.c_int32), ("a_base_offset", C.c_int32),
    ]


_lib = None
_warm_devices = set()


def load() -> C.CDLL:
    """dlopen the library and declare signatures. Works without a GPU (no CUDA call is made)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first. "
            "pyramid_flow_b200 has no fallback path.")
    lib = C.CDLL(str(LIB_PATH))
    missing = [s for s in SYMBOLS if not hasattr(lib, s)]
    if missing:
        raise RuntimeError(f"libpf_b200.so does not export: {missing}")
    lib.pf_last_error.restype = C.c_char_p
    lib.pf_launch_count.restype = C.c_int64
    if int(os.environ.get("WORLD_SIZE", "1")) > 2:
        # world = CFG(2) x SP(world / 2): with SP > 1 the attention launches carry peer stores and run the two-q-tile kernel (the
        # three-q-tile kernel has only been validated on one GPU).  Keep the WHOLE process on that kernel, so the single-GPU
        # reference a sharded step is compared with (bench.py `parity_vs_n1`, tools/sp_check.py) stays bit-identical to it.
        lib.pf_set_option(PF_OPT_ATTN_TRIPLE_KERNEL, 0)
    lib.pf_gemm_bf16.argtypes = [C.POINTER(GemmDesc), C.c_void_p]
    lib.pf_attn_fwd_masked.argtypes = [C.POINTER(AttnDesc), C.c_void_p]
    lib.pf_attn_build_schedule.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.pf_attn_build_pair_schedule.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.pf_attn_build_pair_masks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_int64]
    lib.pf_attn_build_pair_masks.restype = C.c_int64
    lib.pf_attn_build_group_schedule.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.pf_attn_build_group_masks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                              C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.pf_attn_build_group_masks.restype = C.c_int64
    lib.pf_ctx_create.argtypes = [C.POINTER(C.c_void_p)]
    for name in ("pf_ctx_destroy", "pf_ctx_record_end"):
        getattr(lib, name).argtypes = [C.c_void_p]
    for name in ("pf_ctx_record_begin", "pf_ctx_replay", "pf_dit_step_flux", "pf_dit_step_mmdit", "pf_vae_decode_chunk"):
        getattr(lib, name).argtypes = [C.c_void_p, C.c_void_p]
    lib.pf_peer_alloc.argtypes = [C.c_int64, C.POINTER(C.c_void_p)]
    lib.pf_peer_free.argtypes = [C.c_void_p]
    lib.pf_peer_export.argtypes = [C.c_void_p, C.c_void_p]
    lib.pf_peer_open.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    lib.pf_peer_close.argtypes = [C.c_void_p]
    lib.pf_peer_barrier.argtypes = [C.POINTER(PeerGroup), C.c_void_p, C.c_void_p]
    lib.pf_peer_bcast.argtypes = [C.POINTER(PeerGroup), C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
    lib.pf_ln_modulate.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p]
    lib.pf_small_linear.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.pf_timestep_embedding.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
    lib.pf_patchify.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    lib.pf_unpatchify.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
    lib.pf_cfg_euler_step.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.pf_stage_hop.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_float,
                                 C.c_float, C.POINTER(C.c_float), C.c_void_p]
    lib.pf_blend_tiles.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_void_p]
    lib.pf_debug_umma.argtypes = [C.POINTER(UmmaProbe), C.c_void_p]
    lib.pf_debug_attn_trace.argtypes = [C.c_void_p]
    lib.pf_debug_attn_cta_trace.argtypes = [C.c_void_p, C.c_int64]
    lib.pf_causal_conv3d.argtypes = [C.POINTER(ConvDesc), C.c_void_p]
    lib.pf_groupnorm_stats.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                       C.c_void_p, C.c_int64, C.c_void_p]
    lib.pf_groupnorm_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.pf_softmax_rows.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_float, C.c_void_p]
    lib.pf_pack_latent.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.pf_pack_frames_u8.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RuntimeError(f"libpf_b200 {what} failed ({rc}): {load().pf_last_error().decode()}")


def require_device() -> None:
    """Fail loudly unless the CUDA extension is usable on this machine (no CPU fallback exists)."""
    lib = load()
    check(lib.pf_device_check(), "pf_device_check")
    import torch
    dev = torch.cuda.current_device()
    if dev not in _warm_devices:
        check(lib.pf_warmup(), "pf_warmup")
        _warm_devices.add(dev)


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def set_option(key: int, value: int) -> None:
    check(load().pf_set_option(int(key), int(value)), "pf_set_option")


def get_option(key: int) -> int:
    return int(load().pf_get_option(int(key)))


def launch_count() -> int:
    return int(load().pf_launch_count())
