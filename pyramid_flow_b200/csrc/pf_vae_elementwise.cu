// pf_vae_elementwise.cu — HBM-bound kernels of the causal-VAE decode on channels-last bf16 activations:
//   per-frame GroupNorm statistics + apply(+SiLU) (CausalGroupNorm C:36-43, R:127-141, D:362-363),
//   row softmax for the mid-block attention (diffusers Attention, K:454-460), latent layout packing.
#include "../../include/pf_b200.h"
#include "pf_common.cuh"

namespace pf {

// ---------------------------------------------------------------------------------------------------------------
// GroupNorm statistics, pass 1: per (frame, split) partial sum / sum-of-squares per CHANNEL.
// Each thread owns one 8-channel vector position and strides over voxels; 128-bit loads, fp32 partials.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gn_partial_kernel(const __nv_bfloat16* __restrict__ x, long long voxels, int channels, int nsplit,
                  float* __restrict__ partial /* [frames, nsplit, channels, 2] */) {
  // deterministic: per-thread partials are parked in shared memory [vstep][channels][2] and summed in a fixed order
  extern __shared__ float sh[];
  const int frame = blockIdx.x / nsplit;
  const int split = blockIdx.x - frame * nsplit;
  const int cvecs = channels >> 3;
  const long long v0 = voxels * split / nsplit, v1 = voxels * (split + 1) / nsplit;
  const int cv = threadIdx.x % cvecs;
  const int vlane = threadIdx.x / cvecs;
  const int vstep = blockDim.x / cvecs;
  float s[8], ss[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = ss[i] = 0.f;
  if (vlane < vstep) {
    const __nv_bfloat16* base = x + static_cast<size_t>(frame) * voxels * channels;
    for (long long v = v0 + vlane; v < v1; v += vstep) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(base + v * channels) + cv);
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        s[2 * i] += f.x; ss[2 * i] += f.x * f.x;
        s[2 * i + 1] += f.y; ss[2 * i + 1] += f.y * f.y;
      }
    }
    float* dst = sh + (static_cast<size_t>(vlane) * channels + cv * 8) * 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      dst[2 * i] = s[i];
      dst[2 * i + 1] = ss[i];
    }
  }
  __syncthreads();
  float* out = partial + (static_cast<size_t>(frame) * nsplit + split) * channels * 2;
  for (int i = threadIdx.x; i < 2 * channels; i += blockDim.x) {
    float acc = 0.f;
    for (int l = 0; l < vstep; ++l) acc += sh[static_cast<size_t>(l) * channels * 2 + i];
    out[i] = acc;
  }
}

// pass 2: (mean, rstd) per (frame, group), combined in double
__global__ void gn_finalize_kernel(const float* __restrict__ partial, int frames, int nsplit, int channels, int groups,
                                   long long voxels, float eps, float* __restrict__ stats /* [frames, groups, 2] */) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= frames * groups) return;
  const int frame = idx / groups, g = idx - frame * groups;
  const int cpg = channels / groups;
  double s = 0.0, ss = 0.0;
  for (int sp = 0; sp < nsplit; ++sp) {
    const float* p = partial + ((static_cast<size_t>(frame) * nsplit + sp) * channels + g * cpg) * 2;
    for (int c = 0; c < cpg; ++c) {
      s += p[2 * c];
      ss += p[2 * c + 1];
    }
  }
  const double n = static_cast<double>(voxels) * cpg;
  const double mean = s / n;
  double var = ss / n - mean * mean;
  if (var < 0.0) var = 0.0;
  stats[2 * idx] = static_cast<float>(mean);
  stats[2 * idx + 1] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
}

// apply: y[b, t + t_off, vox, c] = act((x[b, t, vox, c] - mean) * rstd * gamma[c] + beta[c]); 8 channels per thread
__global__ void __launch_bounds__(256)
gn_apply_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int b, int t, long long voxels,
                int channels, int groups, const float* __restrict__ stats, const float* __restrict__ gamma,
                const float* __restrict__ beta, int silu, int y_t_total, int y_t_offset) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int cvecs = channels >> 3;
  const long long total = static_cast<long long>(b) * t * voxels * cvecs;
  if (idx >= total) return;
  const int cv = static_cast<int>(idx % cvecs);
  long long r = idx / cvecs;
  const long long vox = r % voxels;
  r /= voxels;
  const int tt = static_cast<int>(r % t);
  const int bb = static_cast<int>(r / t);
  const int frame = bb * t + tt;
  const int cpg = channels / groups;
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + (static_cast<size_t>(frame) * voxels + vox) * channels) + cv);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
  float o[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(h[i]);
    o[2 * i] = f.x;
    o[2 * i + 1] = f.y;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = cv * 8 + i;
    const int g = c / cpg;
    const float mean = __ldg(stats + 2 * (frame * groups + g));
    const float rstd = __ldg(stats + 2 * (frame * groups + g) + 1);
    float v = (o[i] - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
    if (silu) v = silu_f(v);
    o[i] = v;
  }
  uint4 w;
  w.x = pack_bf16x2(o[0], o[1]);
  w.y = pack_bf16x2(o[2], o[3]);
  w.z = pack_bf16x2(o[4], o[5]);
  w.w = pack_bf16x2(o[6], o[7]);
  const size_t yrow = (static_cast<size_t>(bb) * y_t_total + tt + y_t_offset) * voxels + vox;
  reinterpret_cast<uint4*>(y + yrow * channels)[cv] = w;
}

// row softmax: p[r, c] = softmax_c(scale * s[r, c]) over c < cols, zeros in [cols, ld); one warp per row, in place
__global__ void __launch_bounds__(256)
softmax_rows_kernel(__nv_bfloat16* __restrict__ s, long long rows, int cols, long long ld, float scale) {
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  __nv_bfloat16* p = s + row * ld;
  float m = -INFINITY;
  for (int c = lane; c < cols; c += 32) m = fmaxf(m, __bfloat162float(p[c]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float l = 0.f;
  for (int c = lane; c < cols; c += 32) l += __expf((__bfloat162float(p[c]) - m) * scale);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
  const float inv = 1.f / l;
  for (int c = lane; c < ld; c += 32) {
    const float v = c < cols ? __expf((__bfloat162float(p[c]) - m) * scale) * inv : 0.f;
    p[c] = __float2bfloat16(v);
  }
}

// latent [B, C, T, H, W] (fp32/bf16) -> channels-last bf16 [B, T + t_off.., H, W, Cpad] with per-frame affine
// x*scale[t] + shift[t] (decode_latent's un-normalisation P:1226-1230 folded in); channels >= C are zero.
template <typename T>
__global__ void pack_latent_kernel(const T* __restrict__ z, int b, int c, int t, int h, int w, __nv_bfloat16* __restrict__ y,
                                   int cpad, int y_t_total, int y_t_offset, const float* __restrict__ fscale,
                                   const float* __restrict__ fshift) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(b) * t * h * w * cpad;
  if (idx >= total) return;
  const int cc = static_cast<int>(idx % cpad);
  long long r = idx / cpad;
  const int ww = static_cast<int>(r % w); r /= w;
  const int hh = static_cast<int>(r % h); r /= h;
  const int tt = static_cast<int>(r % t);
  const int bb = static_cast<int>(r / t);
  float v = 0.f;
  if (cc < c) {
    v = static_cast<float>(z[(((static_cast<size_t>(bb) * c + cc) * t + tt) * h + hh) * w + ww]);
    if (fscale) v = v * fscale[tt] + fshift[tt];
  }
  y[((((static_cast<size_t>(bb) * y_t_total + tt + y_t_offset) * h + hh) * w + ww)) * cpad + cc] = __float2bfloat16(v);
}

// uint8 frames [B, T, H, W, C] -> channels-last bf16 [B, y_t_total, H, W, cpad] at frame t + y_t_offset, in the order of
// ToTensor + Normalize(0.5, 0.5) (P:906-910): ((v / 255) - 0.5) / 0.5 in fp32, channels >= C zero.  One thread per
// 8-channel output vector (one 16-byte store).
__global__ void __launch_bounds__(256)
pack_frames_u8_kernel(const uint8_t* __restrict__ frames, int b, int t, int h, int w, int c, __nv_bfloat16* __restrict__ y,
                      int cpad, int y_t_total, int y_t_offset) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int cvecs = cpad >> 3;
  const long long total = static_cast<long long>(b) * t * h * w * cvecs;
  if (idx >= total) return;
  const int cv = static_cast<int>(idx % cvecs);
  const long long pix = idx / cvecs;                    // ((bb * t + tt) * h + hh) * w + ww
  const long long hw = static_cast<long long>(h) * w;
  const long long frame = pix / hw;
  const int bb = static_cast<int>(frame / t), tt = static_cast<int>(frame % t);
  const uint8_t* src = frames + pix * c;
  float o[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ch = cv * 8 + i;
    o[i] = ch < c ? __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(src[ch]), 255.f), 0.5f), 0.5f) : 0.f;
  }
  uint4 u;
  u.x = pack_bf16x2(o[0], o[1]);
  u.y = pack_bf16x2(o[2], o[3]);
  u.z = pack_bf16x2(o[4], o[5]);
  u.w = pack_bf16x2(o[6], o[7]);
  const size_t yrow = (static_cast<size_t>(bb) * y_t_total + tt + y_t_offset) * hw + (pix - frame * hw);
  reinterpret_cast<uint4*>(y + yrow * cpad)[cv] = u;
}

// Cross-fade of two neighbouring decoded tiles (blend_v / blend_h, V:397-407): tensors viewed as [outer, L, inner] with L the
// blended axis; b[o, y, i] = a[o, La - extent + y, i] * (1 - y / extent) + b[o, y, i] * (y / extent) for y < extent.
__global__ void blend_tiles_kernel(const float* __restrict__ a, float* __restrict__ b, long long outer, int la, int lb,
                                   long long inner, int extent) {
  const long long total = outer * extent * inner;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const long long i = idx % inner;
  const int y = static_cast<int>((idx / inner) % extent);
  const long long o = idx / (inner * extent);
  const float w = static_cast<float>(y) / static_cast<float>(extent);
  const float av = a[(o * la + (la - extent + y)) * inner + i];
  float* bp = b + (o * lb + y) * inner + i;
  *bp = av * (1.f - w) + *bp * w;
}

}  // namespace pf

extern "C" {

int pf_groupnorm_stats(const void* x, int32_t frames, int64_t voxels, int32_t channels, int32_t groups, float eps,
                       float* stats, float* workspace, int64_t workspace_floats, void* stream_) {
  using namespace pf;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  PF_REQUIRE(x && stats && workspace, "pf_groupnorm_stats: null pointer");
  PF_REQUIRE(channels % 8 == 0 && channels % groups == 0 && channels <= 2048, "pf_groupnorm_stats: channels=%d unsupported", channels);
  // the split count depends on the frame SIZE only, never on how many frames are in the call: per-frame statistics are
  // bitwise identical whatever the temporal chunking
  long long nsplit = (voxels + 4095) / 4096;
  if (nsplit < 1) nsplit = 1;
  if (nsplit > 64) nsplit = 64;
  PF_REQUIRE(static_cast<long long>(frames) * nsplit * channels * 2 <= workspace_floats, "pf_groupnorm_stats: workspace too small (need %lld floats)",
             static_cast<long long>(frames) * nsplit * channels * 2);
  const int vstep = 256 / (channels / 8);
  PF_REQUIRE(vstep >= 1, "pf_groupnorm_stats: too many channels for one block");
  gn_partial_kernel<<<static_cast<int>(frames * nsplit), 256, static_cast<size_t>(vstep) * channels * 2 * sizeof(float), stream>>>(
      static_cast<const __nv_bfloat16*>(x), voxels, channels, static_cast<int>(nsplit), workspace);
  int rc = check_launch("pf_groupnorm_stats(partial)");
  if (rc) return rc;
  const int n = frames * groups;
  gn_finalize_kernel<<<(n + 127) / 128, 128, 0, stream>>>(workspace, frames, static_cast<int>(nsplit), channels, groups,
                                                          voxels, eps, stats);
  return check_launch("pf_groupnorm_stats(finalize)");
}

int pf_groupnorm_apply(const void* x, void* y, int32_t b, int32_t t, int64_t voxels, int32_t channels, int32_t groups,
                       const float* stats, const float* gamma, const float* beta, int32_t silu, int32_t y_t_total,
                       int32_t y_t_offset, void* stream) {
  using namespace pf;
  PF_REQUIRE(x && y && stats && gamma && beta, "pf_groupnorm_apply: null pointer");
  PF_REQUIRE(channels % 8 == 0 && channels % groups == 0, "pf_groupnorm_apply: channels=%d unsupported", channels);
  PF_REQUIRE(y_t_offset >= 0 && y_t_offset + t <= y_t_total, "pf_groupnorm_apply: frame window out of range");
  const long long total = static_cast<long long>(b) * t * voxels * (channels / 8);
  gn_apply_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(y), b, t, voxels, channels, groups, stats, gamma,
      beta, silu, y_t_total, y_t_offset);
  return check_launch("pf_groupnorm_apply");
}

int pf_softmax_rows(void* s, int64_t rows, int32_t cols, int64_t ld, float scale, void* stream) {
  using namespace pf;
  PF_REQUIRE(s && rows > 0 && cols > 0 && ld >= cols, "pf_softmax_rows: bad arguments");
  const long long threads = rows * 32;
  softmax_rows_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<__nv_bfloat16*>(s), rows, cols, ld, scale);
  return check_launch("pf_softmax_rows");
}

int pf_pack_latent(const void* z, int32_t z_is_f32, int32_t b, int32_t c, int32_t t, int32_t h, int32_t w, void* y,
                   int32_t cpad, int32_t y_t_total, int32_t y_t_offset, const float* frame_scale,
                   const float* frame_shift, void* stream_) {
  using namespace pf;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  PF_REQUIRE(z && y && cpad >= c && y_t_offset >= 0 && y_t_offset + t <= y_t_total, "pf_pack_latent: bad arguments");
  const long long total = static_cast<long long>(b) * t * h * w * cpad;
  const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
  if (z_is_f32)
    pack_latent_kernel<float><<<blocks, 256, 0, stream>>>(static_cast<const float*>(z), b, c, t, h, w,
                                                          static_cast<__nv_bfloat16*>(y), cpad, y_t_total, y_t_offset,
                                                          frame_scale, frame_shift);
  else
    pack_latent_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(z), b, c, t, h, w,
                                                                  static_cast<__nv_bfloat16*>(y), cpad, y_t_total,
                                                                  y_t_offset, frame_scale, frame_shift);
  return check_launch("pf_pack_latent");
}

int pf_pack_frames_u8(const void* frames, int32_t b, int32_t t, int32_t h, int32_t w, int32_t c, void* y, int32_t cpad,
                      int32_t y_t_total, int32_t y_t_offset, void* stream) {
  using namespace pf;
  PF_REQUIRE(frames && y && b > 0 && t > 0 && h > 0 && w > 0 && c > 0 && cpad >= c && cpad % 8 == 0 && y_t_offset >= 0 &&
                 y_t_offset + t <= y_t_total,
             "pf_pack_frames_u8: bad arguments");
  const long long total = static_cast<long long>(b) * t * h * w * (cpad / 8);
  pack_frames_u8_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint8_t*>(frames), b, t, h, w, c, static_cast<__nv_bfloat16*>(y), cpad, y_t_total, y_t_offset);
  return check_launch("pf_pack_frames_u8");
}


int pf_blend_tiles(const float* a, float* b, int64_t outer, int32_t la, int32_t lb, int64_t inner, int32_t extent, void* stream) {
  using namespace pf;
  PF_REQUIRE(a && b && outer > 0 && inner > 0 && extent > 0 && extent <= la && extent <= lb, "pf_blend_tiles: bad arguments");
  const long long total = outer * extent * inner;
  blend_tiles_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a, b, outer, la, lb,
                                                                                                              inner, extent);
  return check_launch("pf_blend_tiles");
}

}  // extern "C"
