/* pf_b200.h — C-ABI of libpf_b200.so: the sm_100a kernels behind the Pyramid-Flow sampler hot path.
 *
 * Boundary contract (SURVEY.md §8b):
 *   - plain C, raw device pointers + sizes + a cudaStream_t (passed as void*); no torch types;
 *   - every function returns 0 on success, <0 on error; pf_last_error() gives the message;
 *   - the caller owns every buffer; kernels are stream-ordered and hold no global mutable state;
 *   - there is NO CPU fallback: on a machine without an sm_100 GPU every compute entry fails.
 *
 * Each entry cites the reference op site (file:line under jy0205/Pyramid-Flow @3040d71) it replaces.
 * Abbreviations: F = pyramid_dit/flux_modules/modeling_pyramid_flux.py, B = .../modeling_flux_block.py,
 * N = .../modeling_normalization.py, E = .../modeling_embedding.py, P = pyramid_dit/pyramid_dit_for_video_gen_pipeline.py,
 * S = diffusion_schedulers/scheduling_flow_matching.py, C = video_vae/modeling_causal_conv.py,
 * R = video_vae/modeling_resnet.py, K = video_vae/modeling_block.py, D = video_vae/modeling_enc_dec.py,
 * V = video_vae/modeling_causal_vae.py.
 */
#ifndef PF_B200_H_
#define PF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PF_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------ misc */
PF_API const char* pf_last_error(void);
PF_API int pf_version(void);
/* 0 if the current CUDA device is sm_100 (B200) and the driver exposes cuTensorMapEncodeTiled; <0 otherwise. */
PF_API int pf_device_check(void);
/* Loads every kernel instantiation of the library on the CURRENT device and sets its dynamic shared-memory attribute, so
 * that no later launch initialises anything host-side (required before capturing launches into a CUDA graph; also what makes
 * a second GPU driven from the same process work).  Idempotent, thread-safe. */
PF_API int pf_warmup(void);
/* Library options: data-path choices that do not change results (same arithmetic, same bits) but are A/B-measured. */
enum {
  PF_OPT_GEMM_STAGED_RESID = 0, /* GATE_RESID epilogue: residual read-modify-write transposed through shared memory */
  PF_OPT_GEMM_WAVE_TILING = 1,  /* wave-quantisation-aware tile width for GEMMs with few rows */
  PF_OPT_ATTN_PAIR_KERNEL = 2,  /* variant 0 of pf_attn_fwd_masked = the two-q-tile kernel (needs pair_sched) */
  PF_OPT_ATTN_TILE_PHASE = 3,   /* two-q-tile attention kernel: SM clocks the second q tile's softmax warps are held back once per
                                 * CTA so the two tiles run out of phase (0 = start together) */
  PF_OPT_ATTN_TRIPLE_KERNEL = 4, /* variant 0 of pf_attn_fwd_masked = the three-q-tile kernel when group_sched is given and the
                                  * launch has no peer stores (the sequence-parallel path keeps the two-q-tile kernel: the
                                  * three-q-tile kernel was validated on one GPU only) */
  PF_OPT_COUNT = 5
};
#define PF_OPT_DEFAULT_GEMM_STAGED_RESID 1
#define PF_OPT_DEFAULT_GEMM_WAVE_TILING 1
#define PF_OPT_DEFAULT_ATTN_PAIR_KERNEL 1
#define PF_OPT_DEFAULT_ATTN_TRIPLE_KERNEL 1   /* measured on B200: 2.80 -> 2.60 ms per launch at the bench shape, whole GPU suite green with it */
#define PF_OPT_DEFAULT_ATTN_TILE_PHASE 800   /* measured on B200: 2.84 -> 2.78 ms per launch at the bench shape (tools/gpu_check.py attn_phase_sweep) */
PF_API int pf_set_option(int key, int value);
PF_API int pf_get_option(int key);
/* number of kernels launched by this library since load (bench.py's gpu_launches claim). */
PF_API int64_t pf_launch_count(void);

/* ------------------------------------------------------------------ step contexts (SURVEY.md §8b: pf_ctx_*, pf_dit_step_*)
 * A pf_ctx owns ONE recorded launch sequence: between pf_ctx_record_begin and pf_ctx_record_end every pf_* launch issued on
 * `stream` by the calling thread is recorded instead of executed (descriptor validation, tensor-map encoding and kernel
 * selection happen once, at record time); pf_dit_step_flux / pf_dit_step_mmdit / pf_vae_decode_chunk then re-issue the whole
 * sequence with one call, on any stream.  What the sequence is -- the ~280 launches of PyramidFluxTransformer.forward
 * (F:392-542) at one (plan, shapes), of PyramidDiffusionMMDiT.forward (M:420-497), or one temporal chunk of
 * CausalVaeDecoder.forward (D:302-366) -- is whatever the host recorded; the three entry points are the same replay under the
 * names of the reference functions they stand for.  The caller owns every buffer the recorded launches point to and must
 * keep them alive and at the same addresses; peer-memory barriers (pf_peer_barrier) may be part of the sequence.
 * pf_ctx_record_end returns the number of recorded launches (>= 0) or < 0 on error. */
typedef struct pf_ctx pf_ctx;
PF_API int pf_ctx_create(pf_ctx** out);
PF_API int pf_ctx_destroy(pf_ctx* ctx);
PF_API int pf_ctx_record_begin(pf_ctx* ctx, void* stream);
PF_API int pf_ctx_record_end(pf_ctx* ctx);
PF_API int pf_ctx_replay(pf_ctx* ctx, void* stream);
PF_API int pf_dit_step_flux(pf_ctx* ctx, void* stream);
PF_API int pf_dit_step_mmdit(pf_ctx* ctx, void* stream);
PF_API int pf_vae_decode_chunk(pf_ctx* ctx, void* stream);

/* ------------------------------------------------------------------ peer memory (sequence parallel over NVLink / NVSwitch)
 * Replaces the reference's all-to-all at the attention boundary (trainer_misc/communicate.py:7-24, called at
 * modeling_flux_block.py:285-295, 314-321, 535-560) and its contiguous()/cat copies: producers store straight into the owning
 * rank's buffer through mapped peer pointers (pf_gemm_desc.peer_qkv, pf_attn_desc.peer_out); pf_peer_barrier orders those
 * stores against their consumers.  One process per GPU on one node; buffers come from pf_peer_alloc (cudaMalloc + CUDA IPC). */
#define PF_MAX_PEERS 8
typedef struct PfPeerGroup {
  void* ptr[PF_MAX_PEERS]; /* one mapped pointer per group member (ptr[my_index] = the local buffer) */
  int32_t n;               /* members */
  int32_t my_index;
} PfPeerGroup;
PF_API int pf_peer_alloc(int64_t bytes, void** ptr);   /* zero-filled device memory that peers can map */
PF_API int pf_peer_free(void* ptr);
PF_API int pf_peer_export(void* ptr, void* handle64);  /* 64-byte CUDA IPC handle of a pf_peer_alloc buffer */
PF_API int pf_peer_open(const void* handle64, void** peer_ptr);
PF_API int pf_peer_close(void* peer_ptr);
/* Barrier over the group: grp->ptr[i] = member i's flag array (PF_MAX_PEERS uint32, zero-initialised, peer memory);
 * epoch_counter = one uint32 in local device memory, advanced by the kernel (graph-replay safe).  Everything this rank's
 * earlier kernels stored to peers is visible to a peer's kernels launched after ITS matching barrier. */
PF_API int pf_peer_barrier(const PfPeerGroup* grp, uint32_t* epoch_counter, void* stream);
/* dst->ptr[i][dst_offset_bytes ...] = src[0 .. bytes) for every member (16-byte granularity). */
PF_API int pf_peer_bcast(const PfPeerGroup* dst, const void* src, int64_t bytes, int64_t dst_offset_bytes, void* stream);

/* ------------------------------------------------------------------ GEMM (tcgen05 + TMA)
 * out = epilogue(A[rows, K] . W[N, K]^T + bias).  bf16 operands, fp32 accumulation in TMEM.
 * Replaces every nn.Linear on the DiT path: x_embedder/context_embedder F:290,F:401; to_q/k/v, add_*_proj B:816-835;
 * to_out/to_add_out B:868-872; FeedForward B:73-100; proj_mlp/proj_out B:923-938; norm_out+proj_out F:538-539;
 * with the elementwise ops around them fused into the epilogue (bias, GELU-tanh, per-head RMSNorm N:66-79,
 * RoPE B:34-39, gate*x + residual B:1019-1039).
 *
 * A is addressed as [batches][rows_per_batch][K] (row stride lda); only rows [row_begin, row_begin+row_count) of each
 * batch are computed (the text / video ranges of the joint sequence).  Output row of (b, m) is
 * b*out_batch_rows + out_row_begin + m.
 */
enum {
  PF_EPI_STORE_BF16 = 0, /* out_bf16 = acc + bias                                         */
  PF_EPI_GELU_BF16 = 1,  /* out_bf16 = gelu_tanh(acc + bias)          (diffusers GELU, B:73-75) */
  PF_EPI_STORE_F32 = 2,  /* out_f32  = acc + bias                     (embedders into the fp32 residual stream) */
  PF_EPI_GATE_RESID = 3, /* out_f32 += gate[b, n] * (acc + bias)      (B:1019-1020, 1027-1028, 1032-1039, 937-938) */
  PF_EPI_QKV_ROPE = 4,   /* N = 3*H*hd: bias, RMSNorm(q,k) per head, RoPE(q,k); head-major Q/K/V stores */
  PF_EPI_QKV_GELU = 5    /* N = 3*H*hd + n_mlp: columns < n_split as QKV_ROPE, the rest as GELU_BF16 (single block, B:923-936) */
};

typedef struct pf_gemm_desc {
  const void* a; /* bf16 */
  int64_t lda;   /* elements between rows of A */
  int32_t batches, rows_per_batch, row_begin, row_count;
  const void* w; /* bf16 [n, k] row-major (nn.Linear.weight) */
  int32_t n, k;
  const float* bias; /* fp32 [n] or NULL */
  int32_t epilogue;
  /* generic output (STORE_*, GELU, GATE_RESID, and the GELU half of QKV_GELU) */
  void* out;
  int64_t ldo;
  int32_t out_batch_rows, out_row_begin, out_col_begin;
  /* GATE_RESID: fp32 gate[b*gate_batch_stride + n] */
  const float* gate;
  int64_t gate_batch_stride;
  /* QKV_*: outputs bf16 [batches, heads, seq_len, head_dim]; position of (b, m) is out_row_begin + m */
  void* q_out;
  void* k_out;
  void* v_out;
  const float* rope;     /* fp32 [seq_len, head_dim/2, 2] = (cos, sin) per rotation pair, or NULL (no rotation) */
  const float* q_norm_w; /* fp32 [head_dim] */
  const float* k_norm_w; /* fp32 [head_dim] */
  float norm_eps;
  int32_t heads, head_dim, seq_len;
  int32_t n_split; /* QKV_GELU: first n_split (=3*H*hd) columns are q|k|v */
  int32_t kernel_variant; /* 0 = auto (measured policy); 1 = force 1-CTA tiles; 2 = force 2-CTA (cta_group::2) tiles.
                           * Same bits either way (same K order); exists so tests can pin each kernel. */
  /* QKV_ROPE under sequence parallelism (peer_count > 1): head h of this rank's token chunk is stored into rank
   * (h / peer_heads)'s buffer peer_qkv[h / peer_heads], laid out [3 (q,k,v)][peer_heads][peer_seq][head_dim], at sequence
   * position peer_row0 + (out_row_begin + m).  q_out/k_out/v_out are ignored.  batches must be 1. */
  void* peer_qkv[PF_MAX_PEERS];
  int32_t peer_count, peer_heads, peer_seq, peer_row0;
} pf_gemm_desc;

PF_API int pf_gemm_bf16(const pf_gemm_desc* desc, void* stream);

/* ------------------------------------------------------------------ masked joint attention (tcgen05 + TMA)
 * softmax(Q K^T * scale + mask) V with mask(q, kv) = (seg[q] == seg[kv]) && (time[q] >= time[kv])  (F:318-350),
 * replacing F.scaled_dot_product_attention with the dense bool mask at B:363-365 and B:596-598.
 * q,k,v: bf16 [batch, heads, seq, 64]; out: bf16 [batch, seq, heads*64] with row stride ldo (elements).
 * seg/time: int32 [batch, seq].  tile_sched: int32, built by pf_attn_build_schedule (host) from seg/time.
 */
typedef struct pf_attn_desc {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  int64_t ldo;
  int32_t batch, heads, seq, head_dim;
  float scale;
  const int32_t* seg;        /* device [batch, seq] */
  const int32_t* time;       /* device [batch, seq] */
  const int32_t* tile_sched; /* device; layout documented at pf_attn_build_schedule */
  int32_t sched_stride;      /* int32 entries per (batch, q_tile) row */
  int32_t variant;           /* 0 = default; 0x20 = the three-q-tile kernel; 0x10 = the two-q-tile kernel; 1 / 2 / 3 = the one-tile
                              * kernel (A/B, see pf_attn.cu) */
  int32_t q_row_begin;       /* only q rows >= q_row_begin are computed (multiple of 128; 0 = all).  The last single block
                              * needs the current clip's rows only (history outputs are discarded, reference F:380). */
  const int32_t* pair_sched; /* device; built by pf_attn_build_pair_schedule from tile_sched, same sched_stride.  When set (and
                              * variant does not ask for the one-tile kernel) the launch uses the two-q-tiles-per-CTA kernel. */
  const int32_t* pair_mask_index; /* device; from pf_attn_build_pair_masks (required with pair_sched) */
  const void* pair_mask_bits;     /* device; [blocks, 128, 4] uint32 */
  /* sequence parallelism (peer_count > 1, batch 1, two-q-tile kernel): row q of this rank's head group is stored into rank
   * (q / peer_chunk_rows)'s buffer peer_out[...] at row q % peer_chunk_rows, columns peer_col_begin + h*64 (row stride ldo);
   * `out` is ignored. */
  void* peer_out[PF_MAX_PEERS];
  int32_t peer_count, peer_chunk_rows, peer_col_begin;
  /* three-q-tile kernel (variant 0x20, or variant 0 under PF_OPT_ATTN_TRIPLE_KERNEL, the default): schedule and row masks of groups of three
   * q tiles from pf_attn_build_group_schedule / pf_attn_build_group_masks (group = 3), same sched_stride */
  const int32_t* group_sched;
  const int32_t* group_mask_index;
  const void* group_mask_bits;
} pf_attn_desc;

/* Host helper: from host copies of seg/time ids builds, for each (batch, 128-row q tile), the list of 128-wide kv
 * tiles that contain at least one allowed pair, flagged full (no element mask needed) or partial.
 * Row layout: [count, (kv_tile << 1) | needs_mask, ...].  Returns the number of int32 written per row
 * (sched_stride) or <0 on error.  `out` may be NULL to query the size: stride = 1 + ceil(seq/128). */
PF_API int pf_attn_build_schedule(const int32_t* seg_host, const int32_t* time_host, int32_t batch, int32_t seq,
                                  int32_t* out, int64_t* allowed_pairs /* [batch] or NULL */);
/* Host helper: pairs the q tiles from the end of the sequence (pair p = tiles q_tiles-2-2p and q_tiles-1-2p; the first tile is
 * alone when q_tiles is odd) and merges their kv lists.  Row layout per (batch, pair): [count, entry...], entry =
 * (kv_tile << 4) | flags_lo | (flags_hi << 2), flags = bit0: the tile has an allowed pair in this kv tile, bit1: it needs the
 * element mask (a tile without bit0 is computed fully masked).  `out` holds batch * ceil(q_tiles/2) rows of sched_stride. */
PF_API int pf_attn_build_pair_schedule(const int32_t* tile_sched_host, int32_t batch, int32_t seq, int32_t sched_stride,
                                       int32_t* out);
/* Host helper: the element masks of the two-q-tile kernel.  For every (pair entry, tile X) whose flags say "partial" it
 * assigns a block index (mask_index[batch, n_pairs, 2 * sched_stride], entry e / tile X at [2 e + X], -1 otherwise) and, when
 * mask_bits != NULL, fills block = 128 rows x 4 uint32: bit i of word w of row r = q row r of the tile may attend kv column
 * 32 w + i of the kv tile.  Returns the number of blocks needed (call once with mask_bits = NULL to size the buffer). */
PF_API int64_t pf_attn_build_pair_masks(const int32_t* seg_host, const int32_t* time_host, const int32_t* pair_sched_host,
                                        int32_t batch, int32_t seq, int32_t sched_stride, int32_t* mask_index,
                                        uint32_t* mask_bits, int64_t capacity_blocks);
/* Host helpers of the three-q-tile kernel, the pair forms generalised to groups of `group` (2..4) q tiles counted from the end
 * of the sequence.  Entry = (kv_tile << 8) | flags, 2 flag bits per tile X at bit 2 X (X = 0 the lowest tile of the group);
 * mask_index[batch, n_groups, group * sched_stride], entry e / tile X at [group e + X]; blocks as in the pair form.  With
 * pair_sched_host / pair_mask_index_host (the pair schedule of the same tile_sched) no bits are built: the indices point into
 * the PAIR schedule's block pool (a block depends on (q tile, kv tile) only), mask_bits is ignored, and the return value is
 * the number of pool blocks referenced. */
PF_API int pf_attn_build_group_schedule(const int32_t* tile_sched_host, int32_t batch, int32_t seq, int32_t sched_stride,
                                        int32_t group, int32_t* out);
PF_API int64_t pf_attn_build_group_masks(const int32_t* seg_host, const int32_t* time_host, const int32_t* group_sched_host,
                                         int32_t batch, int32_t seq, int32_t sched_stride, int32_t group,
                                         int32_t* mask_index, uint32_t* mask_bits, int64_t capacity_blocks,
                                         const int32_t* pair_sched_host /* or NULL */,
                                         const int32_t* pair_mask_index_host /* or NULL */);
PF_API int pf_attn_fwd_masked(const pf_attn_desc* desc, void* stream);

/* ------------------------------------------------------------------ LayerNorm + AdaLN modulate pre-pass (HBM-bound)
 * y_bf16[r, :] = LN(x_f32[r, :], eps) * (1 + scale[b, :]) + shift[b, :]   (N:174, N:234, N:120, B:1022-1023, B:1035-1036)
 * rows [row_begin, row_begin+row_count) of each batch of the joint [batches, rows_per_batch, dim] stream.
 */
PF_API int pf_ln_modulate(const float* x, void* y_bf16, int32_t batches, int32_t rows_per_batch, int32_t row_begin,
                          int32_t row_count, int32_t dim, const float* shift, const float* scale,
                          int64_t mod_batch_stride, float eps, void* stream);

/* ------------------------------------------------------------------ small-M linear (HBM-bound GEMV)
 * y[m, n] (+)= act_out( sum_k act_in(x[m, k]) * W[n, k] + bias[n] ), m <= 8; W bf16, x/y fp32.
 * Used for the per-step AdaLN modulation of ALL layers in one launch (N:147,164,209,223,99,110) and the
 * timestep/text conditioning MLPs (E:84-158, E:185-201).  act: 0 none, 1 SiLU.
 */
PF_API int pf_small_linear(const float* x, int32_t m, int32_t k, const void* w_bf16, const float* bias, int32_t n,
                           float* y, int32_t act_in, int32_t act_out, int32_t accumulate, int32_t round_in_bf16,
                           void* stream);

/* sinusoidal timestep embedding, flip_sin_to_cos=True, downscale_freq_shift=0 (E:11-62): out fp32 [m, dim],
 * out[:, :dim/2] = cos(t * f_i), out[:, dim/2:] = sin(t * f_i), f_i = exp(-ln(1e4) * i / (dim/2)); rounded to bf16
 * values when round_bf16 != 0 (E:195).  t is fp32 [m] (already rounded to bf16 by the caller, P:750). */
PF_API int pf_timestep_embedding(const float* t, int32_t m, int32_t dim, float* out, int32_t round_bf16,
                                 void* stream);

/* patchify one clip: latent bf16/fp32 [B, C, T, H, W] -> tokens bf16 [B, tok_begin + (t h w), (p1 p2 c)], p=2 (F:285-286).
 * tokens row stride = 4*C; rows_per_batch = total tokens of all clips of the unit. */
PF_API int pf_patchify(const void* latent, int32_t latent_is_f32, int32_t b, int32_t c, int32_t t, int32_t h, int32_t w,
                       void* tokens_bf16, int32_t rows_per_batch, int32_t tok_begin, void* stream);
/* unpatchify: x fp32 [B, rows_per_batch, 4*C] rows [row_begin, +t*h/2*w/2) -> out [B, C, T, H, W] (F:383-387). */
PF_API int pf_unpatchify(const float* x, int32_t rows_per_batch, int32_t row_begin, int32_t b, int32_t c, int32_t t,
                         int32_t h, int32_t w, void* out, int32_t out_is_f32, void* stream);

/* fused CFG combine + Euler step (P:771-776, S:278-286):
 * v = vu + g*(vc - vu); x_out = x + dsigma * v.  v: fp32 [2, n] (uncond, cond); x fp32 [n]. */
PF_API int pf_cfg_euler_step(const float* v2, float guidance, float dsigma, const float* x, float* x_out, int64_t n,
                             void* stream);
/* Stage hop of generate_one_unit (P:729-743) in one kernel: nearest x2 up-sampling of the latent planes x [planes, h, w]
 * (bf16 or fp32), block noise of sample_block_noise (P:697-703: each 2x2 block ~ N(0, (1+gamma) I - gamma 11^T)) formed as L z
 * from iid normals z [planes, 2h, 2w] (fp32, drawn on the device) with L = chol16 (host, row-major lower-triangular 4x4), and
 * the renoise  out = alpha * up(x) + beta * noise.  Opt-in on the host side: same distribution as the reference's python loop
 * of MultivariateNormal.sample() calls, different RNG consumption. */
PF_API int pf_stage_hop(const void* x, int32_t x_is_f32, const float* z, void* out, int64_t planes, int32_t h, int32_t w,
                        float alpha, float beta, const float* chol16, void* stream);

/* ------------------------------------------------------------------ causal 3-D convolution (VAE decode, tcgen05 + TMA)
 * Replaces CausalConv3d -> nn.Conv3d (C:46-146), kernel 3x3x3 or 1x1x1, stride 1, on channels-last bf16 activations.
 * x: [B, T + kt - 1, H, W, Cin]: the (kt-1) causal-padding frames are physically present in front (zeros for the first
 * chunk, the previous chunk's last input frames afterwards = the reference's feature cache C:126-143); spatial zero
 * padding is implicit (TMA out-of-bounds fill).  wgt: bf16 [Cout, kt*kh*kw*Cin], K index = tap*Cin + ci with
 * tap = (dt*kh + dh)*kw + dw (re-laid out once at weight import).  Cin and Cout must be multiples of 64 (pad).
 * store_mode: 0 plain [B, out_t_total, H, W, out_c] at frame t + out_t_offset (+ optional bf16 residual, R:148);
 *             1 spatial depth-to-space 'b (c p1 p2) t h w -> b c t (h p1) (w p2)' (CausalUpsample2x R:616);
 *             2 temporal depth-to-space 'b (c p) t h w -> b c (t p) h w' at frame 2t + p + out_t_offset, frames < 0
 *               dropped (CausalTemporalUpsample2x R:724-727 with is_init_image => out_t_offset = -1).
 */
typedef struct pf_conv3d_desc {
  const void* x;
  int32_t b, t, h, w, cin; /* OUTPUT frames / height / width (= input dims at unit stride) */
  const void* wgt;
  const float* bias; /* fp32 [cout] or NULL */
  int32_t cout, kt, kh, kw;
  int32_t store_mode;
  void* out;
  int32_t out_f32; /* plain mode output type: 0 = bf16, 1 = fp32, 2 = uint8 image clamp(v*127.5+127.5, 0, 255) (decode_latent, P:1238) */
  int32_t out_t_total, out_t_offset, out_c;
  int32_t store_channels; /* first store_channels conv outputs are stored (the rest is filter padding) */
  const void* residual;   /* bf16 [B, res_t_total, H, W, out_c] read at frame t + res_t_offset, plain mode only */
  int32_t res_t_total, res_t_offset;
  int32_t stride_t, stride_h, stride_w; /* 0/1 = unit stride; 2 = the encoder's down-samplers (C:66-67: CausalDownsample2x
                                         * stride (1,2,2) R:322, CausalTemporalDownsample2x stride (2,1,1) R:486).  b,t,h,w
                                         * stay OUTPUT dims; x is [B, (t-1)*stride_t + kt, h*stride_h, w*stride_w, cin]. */
  int32_t kernel_variant; /* 0 = auto; 1 = 1-CTA tiles (conv3d); 2 = 2-CTA pairs, one TMA box per tap (conv3d2);
                           * 3 = 2-CTA pairs with kw-tap reuse (conv3d2w: needs 128-voxel rows, 3x3x3, unit stride).
                           * Every kernel accumulates in the same K order: the choice never changes the bits. */
} pf_conv3d_desc;
PF_API int pf_causal_conv3d(const pf_conv3d_desc* desc, void* stream);

/* per-frame GroupNorm (CausalGroupNorm C:36-43) on channels-last bf16 [frames, voxels, channels]:
 * stats[frame, group] = (mean, rstd); workspace: >= frames * 64 * channels * 2 floats.  Deterministic, and independent of
 * how many frames are passed per call (chunk-invariant). */
PF_API int pf_groupnorm_stats(const void* x_bf16, int32_t frames, int64_t voxels, int32_t channels, int32_t groups,
                              float eps, float* stats, float* workspace, int64_t workspace_floats, void* stream);
/* y[b, t + y_t_offset, vox, c] = act((x[b, t, vox, c] - mean) * rstd * gamma[c] + beta[c]), act = SiLU if silu
 * (R:127-129, R:139-141, D:362-363); y has y_t_total frames per batch (room for the next conv's causal halo). */
PF_API int pf_groupnorm_apply(const void* x_bf16, void* y_bf16, int32_t b, int32_t t, int64_t voxels, int32_t channels,
                              int32_t groups, const float* stats, const float* gamma, const float* beta, int32_t silu,
                              int32_t y_t_total, int32_t y_t_offset, void* stream);
/* in-place row softmax of bf16 scores [rows, ld]: softmax over the first `cols` columns of scale*s, zeros in the padding
 * (mid-block attention, diffusers Attention used at K:454-460). */
PF_API int pf_softmax_rows(void* s_bf16, int64_t rows, int32_t cols, int64_t ld, float scale, void* stream);
/* latent [B, C, T, H, W] -> channels-last bf16 [B, y_t_total, H, W, cpad] at frame t + y_t_offset, channels >= C zero,
 * optional per-frame affine z*scale[t] + shift[t] (decode_latent's un-normalisation, P:1226-1230). */
PF_API int pf_pack_latent(const void* z, int32_t z_is_f32, int32_t b, int32_t c, int32_t t, int32_t h, int32_t w,
                          void* y_bf16, int32_t cpad, int32_t y_t_total, int32_t y_t_offset, const float* frame_scale,
                          const float* frame_shift, void* stream);
/* uint8 video frames [B, T, H, W, C] (channels last) -> the encoder's conv_in input, channels-last bf16
 * [B, y_t_total, H, W, cpad] at frame t + y_t_offset (behind the causal halo), channels >= C zero (cpad % 8 == 0).
 * Each value is ((v / 255) - 0.5) / 0.5 in fp32, rounded once to bf16: ToTensor + Normalize(0.5, 0.5) in the reference's
 * order (P:906-910, causal_video_vae_demo.ipynb), replacing the host-side float conversion and the device repack. */
PF_API int pf_pack_frames_u8(const void* frames_u8, int32_t b, int32_t t, int32_t h, int32_t w, int32_t c, void* y_bf16,
                             int32_t cpad, int32_t y_t_total, int32_t y_t_offset, void* stream);
/* Cross-fade of neighbouring decoded tiles (blend_v / blend_h, V:397-407), tensors viewed as fp32 [outer, L, inner] with L the
 * blended axis: b[o, y, i] = a[o, la - extent + y, i] * (1 - y/extent) + b[o, y, i] * (y/extent) for y < extent (in place). */
PF_API int pf_blend_tiles(const float* a, float* b, int64_t outer, int32_t la, int32_t lb, int64_t inner, int32_t extent,
                          void* stream);

/* ------------------------------------------------------------------ debug probe (used only by tests/tools)
 * One CTA, one 128 x N x K tcgen05.mma chain with host-chosen descriptor bits, so descriptor encodings can be
 * pinned on hardware without recompiling.  a: bf16 [128, K] (K-major) or staged to TMEM when a_from_tmem;
 * b: bf16, loaded by TMA as [rows_b, cols_b] boxes of 64 columns.  d: fp32 [128, N]. */
typedef struct pf_umma_probe {
  const void* a;
  const void* b;
  float* d;
  int32_t n, k;
  int32_t b_rows, b_cols;  /* global shape of b (row-major) */
  int32_t b_box_rows;      /* TMA box rows for b (box cols fixed at 64 = 128 B) */
  int32_t b_mn_major;      /* instruction-descriptor bit 16 */
  uint32_t b_lbo, b_sbo;   /* bytes */
  uint32_t b_k_step_bytes; /* descriptor start-address advance per UMMA_K=16 inside a 64-wide k block */
  uint32_t b_kblock_bytes; /* descriptor start-address advance per 4 UMMA_K steps (one 64-wide k block) */
  int32_t a_from_tmem;     /* 1: A is converted to packed bf16 pairs in TMEM (lane = row, 32-bit column = 2 k) */
  int32_t a_rows;          /* rows of a staged in shared memory (0 = 128); the MMA reads rows [a_row_offset, +128) */
  int32_t a_row_offset;    /* start-address advance of the A descriptor in 128-byte rows (inside the swizzle atom) */
  int32_t a_base_offset;   /* value of the descriptor's base-offset field, bits [49,52) */
} pf_umma_probe;
PF_API int pf_debug_umma(const pf_umma_probe* p, void* stream);

/* Debug timeline of the attention kernel: `device_buf` = 3 * 48 * 8 uint64 (clock64 stamps of one CTA: two softmax warps
 * and the MMA issuer, first 48 kv tiles), filled by pf_attn_fwd_masked launches with variant bit 1 (value 2) set.  While a
 * buffer is set, launches of the two-q-tile kernel use its timeline instantiation and fill 4 x 64 x 12 uint64 instead
 * (softmax thread 0 of q tile A / B and the two MMA issuers of CTA (0, 0, 0), first 64 kv tiles).
 * NULL disables.  Test/profiling aid only (tools/gpu_check.py attn_trace). */
PF_API int pf_debug_attn_trace(void* device_buf);
/* Per-CTA records of the same trace variant: `device_buf` = capacity x 8 uint64 (clock64 at CTA entry, at exit, number of
 * kv tiles, SM id), indexed by the linear block index.  NULL disables. */
PF_API int pf_debug_attn_cta_trace(void* device_buf, int64_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* PF_B200_H_ */
