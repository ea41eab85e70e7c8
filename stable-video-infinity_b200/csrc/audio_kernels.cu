// Kernels of the wav2vec2 audio encoder of SVI-Talk (chinese-wav2vec2-base, group-norm / post-LN variant) that are not
// GEMMs: the first convolution with its whole-sequence GroupNorm and GELU, the 50 Hz -> 25 Hz linear interpolation with
// the feature-projection LayerNorm, the grouped positional convolution and a LayerNorm with an fp32 + bf16 output pair.
// Convolutions 2-7, the projections and the feed-forward layers run on svi_gemm_bf16 (tcgen05), the attention on
// svi_attn_small.  Nothing here uses atomics: every reduction has a fixed order, so an embedding is bit-identical from
// run to run and on every rank.
//
// Replaces (transformers models/wav2vec2/modeling_wav2vec2.py, driven by the reference's
// utils/src/audio_analysis/wav2vec2.py:30-32 and torch_utils.py:16-19):
//   Wav2Vec2GroupNormConvLayer (conv 1->512, k 10, s 5, no bias; GroupNorm(512, 512); GELU),
//   linear_interpolation + Wav2Vec2FeatureProjection.layer_norm,
//   Wav2Vec2PositionalConvEmbedding (grouped conv, weight norm folded on the host, SamePad, GELU) + the residual add,
//   the LayerNorms of Wav2Vec2Encoder / Wav2Vec2EncoderLayer.
#include "common.cuh"
#include "../../include/svi_b200.h"

namespace svi {
namespace audio {

constexpr int C0_TB = 1024;      // conv-0 output rows per block
constexpr int C0_MAX_K = 16;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// sum over a block of `nthreads` (multiple of 32, <= 1024) threads; red: 32 floats
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  const int nw = blockDim.x >> 5;
  float t = threadIdx.x < nw ? red[threadIdx.x] : 0.f;
  if (threadIdx.x < 32) {
    t = warp_sum(t);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  return red[0];
}

// Samples [t0*stride, t0*stride + rows*stride + k) of the waveform into shared memory (zero past the end).
__device__ __forceinline__ void load_wave(const float* __restrict__ wav, long long n, long long base, int count, float* s) {
  for (int i = threadIdx.x; i < count; i += blockDim.x) s[i] = base + i < n ? wav[base + i] : 0.f;
}

// Pass 1: thread c = channel; per block the fp64 sum and sum of squares of the conv output over its C0_TB rows.
// partials [nblk][2][C].
__global__ void conv0_partials_kernel(const float* __restrict__ wav, long long n, const float* __restrict__ w, int C, int k,
                                      int stride, long long T0, double* __restrict__ partials) {
  extern __shared__ float s_wav[];
  const long long t0 = (long long)blockIdx.x * C0_TB;
  const int rows = (int)min((long long)C0_TB, T0 - t0);
  load_wave(wav, n, t0 * stride, rows * stride + k, s_wav);
  __syncthreads();
  const int c = threadIdx.x;
  float wr[C0_MAX_K];
#pragma unroll
  for (int j = 0; j < C0_MAX_K; ++j) wr[j] = j < k ? w[c * k + j] : 0.f;
  double s = 0.0, q = 0.0;
  for (int r = 0; r < rows; ++r) {
    const float* x = s_wav + r * stride;
    float v = 0.f;
#pragma unroll
    for (int j = 0; j < C0_MAX_K; ++j)
      if (j < k) v = fmaf(wr[j], x[j], v);
    s += v;
    q += (double)v * v;
  }
  partials[((long long)blockIdx.x * 2 + 0) * C + c] = s;
  partials[((long long)blockIdx.x * 2 + 1) * C + c] = q;
}

// Merge of the block partials in block order (fp64), then the per-channel mean and 1/sqrt(var + eps) (biased variance,
// as nn.GroupNorm).
__global__ void conv0_stats_kernel(const double* __restrict__ partials, int nblk, int C, long long T0, float eps,
                                   float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s = 0.0, q = 0.0;
  for (int b = 0; b < nblk; ++b) {
    s += partials[((long long)b * 2 + 0) * C + c];
    q += partials[((long long)b * 2 + 1) * C + c];
  }
  const double mean = s / (double)T0;
  const double var = fmax(q / (double)T0 - mean * mean, 0.0);
  mean_out[c] = (float)mean;
  rstd_out[c] = (float)(1.0 / sqrt(var + (double)eps));
}

// Pass 2: recompute the conv, normalise, affine, exact GELU -> bf16 [T0, C] channels-last.
__global__ void conv0_apply_kernel(const float* __restrict__ wav, long long n, const float* __restrict__ w, int C, int k,
                                   int stride, long long T0, const float* __restrict__ mean, const float* __restrict__ rstd,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   __nv_bfloat16* __restrict__ out) {
  extern __shared__ float s_wav[];
  const long long t0 = (long long)blockIdx.x * C0_TB;
  const int rows = (int)min((long long)C0_TB, T0 - t0);
  load_wave(wav, n, t0 * stride, rows * stride + k, s_wav);
  __syncthreads();
  const int c = threadIdx.x;
  float wr[C0_MAX_K];
#pragma unroll
  for (int j = 0; j < C0_MAX_K; ++j) wr[j] = j < k ? w[c * k + j] : 0.f;
  const float a = rstd[c] * gamma[c];
  const float b = beta[c] - mean[c] * a;
  for (int r = 0; r < rows; ++r) {
    const float* x = s_wav + r * stride;
    float v = 0.f;
#pragma unroll
    for (int j = 0; j < C0_MAX_K; ++j)
      if (j < k) v = fmaf(wr[j], x[j], v);
    out[(t0 + r) * C + c] = __float2bfloat16_rn(gelu_erf(fmaf(v, a, b)));
  }
}

// One block per output row: y[s] = LayerNorm((1 - l) x[i0] + l x[i1]) -> bf16, with the source index of
// F.interpolate(mode='linear', align_corners=True) computed in fp32 as torch does (scale = (T_in-1)/(S-1)).
__global__ void interp_layernorm_kernel(const float* __restrict__ x, int T_in, int C, int S, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ y) {
  extern __shared__ float s_row[];
  __shared__ float red[32];
  const int s = blockIdx.x;
  const float scale = S > 1 ? (float)(T_in - 1) / (float)(S - 1) : 0.f;
  const float src = scale * (float)s;
  int i0 = (int)src;
  if (i0 > T_in - 1) i0 = T_in - 1;
  const int i1 = i0 + (i0 < T_in - 1 ? 1 : 0);
  const float l1 = src - (float)i0, l0 = 1.f - l1;
  const float* x0 = x + (long long)i0 * C;
  const float* x1 = x + (long long)i1 * C;
  float sum = 0.f;
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    const float v = l0 * x0[i] + l1 * x1[i];
    s_row[i] = v;
    sum += v;
  }
  const float mu = block_sum(sum, red) / (float)C;
  float q = 0.f;
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    const float d = s_row[i] - mu;
    q += d * d;
  }
  const float rs = rsqrtf(block_sum(q, red) / (float)C + eps);
  __nv_bfloat16* yr = y + (long long)s * C;
  for (int i = threadIdx.x; i < C; i += blockDim.x) yr[i] = __float2bfloat16_rn((s_row[i] - mu) * rs * gamma[i] + beta[i]);
}

// Grouped positional convolution, one block = PC_TT output rows of one group; thread (tq, o): output channel o of the
// rows tq*PC_RPT .. +PC_RPT.  The input window [PC_TT + k - 1, cg] sits in shared memory (row pitch cg + 1: the rows of the
// two tq values a warp spans fall into different banks), the weights stream through in chunks of PC_JC taps.
constexpr int PC_TQ = 4;
constexpr int PC_RPT = 16;
constexpr int PC_TT = PC_TQ * PC_RPT;
constexpr int PC_JC = 4;
constexpr int PC_MAX_CG = 64;

__global__ void pos_conv_kernel(const float* __restrict__ x, int S, int D, int cg, int k, const float* __restrict__ w,
                                const float* __restrict__ bias, float* __restrict__ out) {
  extern __shared__ float sm[];
  const int xp = cg + 1;
  float* xs = sm;                                   // [PC_TT + k - 1][cg + 1]
  float* ws = xs + (PC_TT + k - 1) * xp;            // [PC_JC][cg][cg]
  const int g = blockIdx.y, t0 = blockIdx.x * PC_TT, pad = k / 2;
  const int win = PC_TT + k - 1;
  for (int i = threadIdx.x; i < win * cg; i += blockDim.x) {
    const int r = i / cg, c = i - r * cg;
    const int t = t0 + r - pad;
    xs[r * xp + c] = (t >= 0 && t < S) ? x[(long long)t * D + g * cg + c] : 0.f;
  }
  const int o = threadIdx.x % cg, tq = threadIdx.x / cg;
  float acc[PC_RPT];
#pragma unroll
  for (int i = 0; i < PC_RPT; ++i) acc[i] = 0.f;
  const float* wg = w + (long long)g * k * cg * cg;   // [k][cg in][cg out]
  for (int j0 = 0; j0 < k; j0 += PC_JC) {
    const int nj = min(PC_JC, k - j0);
    __syncthreads();
    for (int i = threadIdx.x; i < nj * cg * cg; i += blockDim.x) ws[i] = wg[(long long)j0 * cg * cg + i];
    __syncthreads();
    for (int jj = 0; jj < nj; ++jj) {
      const float* xr = xs + (tq * PC_RPT + j0 + jj) * xp;
      const float* wr = ws + jj * cg * cg + o;
      for (int c = 0; c < cg; ++c) {
        const float wv = wr[c * cg];
#pragma unroll
        for (int i = 0; i < PC_RPT; ++i) acc[i] = fmaf(xr[i * xp + c], wv, acc[i]);
      }
    }
  }
  const float b = bias[g * cg + o];
#pragma unroll
  for (int i = 0; i < PC_RPT; ++i) {
    const int t = t0 + tq * PC_RPT + i;
    if (t < S) {
      const long long idx = (long long)t * D + g * cg + o;
      out[idx] = x[idx] + gelu_erf(acc[i] + b);
    }
  }
}

// y = LayerNorm(x) * gamma + beta -> f32 (row pitch ldy) and bf16 (contiguous); y may alias x (same element, same thread).
__global__ void __launch_bounds__(256)
layernorm_f32x2_kernel(const float* x, long long ldx, int D, float eps, const float* __restrict__ gamma,
                       const float* __restrict__ beta, float* y, long long ldy, __nv_bfloat16* __restrict__ yb) {
  __shared__ float red[32];
  const float* xr = x + (long long)blockIdx.x * ldx;
  float s = 0.f;
  for (int i = threadIdx.x; i < D; i += 256) s += xr[i];
  const float mean = block_sum(s, red) / (float)D;
  float q = 0.f;
  for (int i = threadIdx.x; i < D; i += 256) {
    const float c = xr[i] - mean;
    q += c * c;
  }
  const float rstd = rsqrtf(block_sum(q, red) / (float)D + eps);
  float* yr = y + (long long)blockIdx.x * ldy;
  __nv_bfloat16* br = yb + (long long)blockIdx.x * D;
  for (int i = threadIdx.x; i < D; i += 256) {
    const float v = (xr[i] - mean) * rstd * gamma[i] + beta[i];
    yr[i] = v;
    br[i] = __float2bfloat16_rn(v);
  }
}

inline long long conv0_rows(long long n, int k, int stride) { return n >= k ? (n - k) / stride + 1 : 0; }
inline size_t conv0_ws(long long n, int C, int k, int stride) {
  const long long nblk = (conv0_rows(n, k, stride) + C0_TB - 1) / C0_TB;
  return (size_t)2 * C * sizeof(float) + 256 + (size_t)nblk * 2 * C * sizeof(double);
}

}  // namespace audio
}  // namespace svi

extern "C" size_t svi_audio_conv0_workspace_bytes(int64_t n_samples, int32_t C, int32_t k, int32_t stride) {
  if (n_samples <= 0 || C <= 0 || k <= 0 || stride <= 0) return 0;
  return svi::audio::conv0_ws(n_samples, C, k, stride);
}

extern "C" int svi_audio_conv0_gn_gelu(const float* wav, int64_t n_samples, const float* w, int32_t C, int32_t k,
                                       int32_t stride, const float* gamma, const float* beta, float eps, void* out_bf16,
                                       void* workspace, size_t workspace_bytes, void* stream) {
  using namespace svi;
  SVI_REQUIRE(wav && w && gamma && beta && out_bf16 && workspace, "svi_audio_conv0_gn_gelu: null pointer");
  SVI_REQUIRE(C > 0 && C <= 1024 && C % 32 == 0, "svi_audio_conv0_gn_gelu: C must be a multiple of 32 in [32, 1024] (got %d)", C);
  SVI_REQUIRE(k > 0 && k <= audio::C0_MAX_K && stride > 0, "svi_audio_conv0_gn_gelu: need 0 < k <= 16, stride > 0");
  const long long T0 = audio::conv0_rows(n_samples, k, stride);
  SVI_REQUIRE(T0 > 0, "svi_audio_conv0_gn_gelu: %lld samples give no output row", (long long)n_samples);
  SVI_REQUIRE(workspace_bytes >= audio::conv0_ws(n_samples, C, k, stride) && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
              "svi_audio_conv0_gn_gelu: workspace too small or not 16-byte aligned (svi_audio_conv0_workspace_bytes)");
  const long long nblk = (T0 + audio::C0_TB - 1) / audio::C0_TB;
  SVI_REQUIRE(nblk < (1LL << 31), "svi_audio_conv0_gn_gelu: input too long");
  float* mean = static_cast<float*>(workspace);
  float* rstd = mean + C;
  double* partials = reinterpret_cast<double*>(static_cast<char*>(workspace) + ((2 * C * sizeof(float) + 255) / 256) * 256);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t smem = sizeof(float) * ((size_t)audio::C0_TB * stride + k);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(audio::conv0_partials_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(audio::conv0_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_set = true;
  }
  SVI_REQUIRE(smem <= 200 * 1024, "svi_audio_conv0_gn_gelu: stride too large");
  audio::conv0_partials_kernel<<<(unsigned)nblk, C, smem, st>>>(wav, n_samples, w, C, k, stride, T0, partials);
  SVI_CUDA_LAUNCH_CHECK("svi_audio_conv0_gn_gelu (partials)");
  audio::conv0_stats_kernel<<<(C + 127) / 128, 128, 0, st>>>(partials, (int)nblk, C, T0, eps, mean, rstd);
  SVI_CUDA_LAUNCH_CHECK("svi_audio_conv0_gn_gelu (stats)");
  audio::conv0_apply_kernel<<<(unsigned)nblk, C, smem, st>>>(wav, n_samples, w, C, k, stride, T0, mean, rstd, gamma, beta,
                                                            reinterpret_cast<__nv_bfloat16*>(out_bf16));
  SVI_CUDA_LAUNCH_CHECK("svi_audio_conv0_gn_gelu (apply)");
  return SVI_OK;
}

extern "C" int svi_audio_interp_layernorm(const float* x, int32_t T_in, int32_t C, int32_t S, const float* gamma,
                                          const float* beta, float eps, void* y_bf16, void* stream) {
  using namespace svi;
  SVI_REQUIRE(x && gamma && beta && y_bf16 && T_in > 0 && S > 0 && C > 0 && C <= 8192,
              "svi_audio_interp_layernorm: bad arguments");
  audio::interp_layernorm_kernel<<<S, 128, sizeof(float) * C, static_cast<cudaStream_t>(stream)>>>(
      x, T_in, C, S, gamma, beta, eps, reinterpret_cast<__nv_bfloat16*>(y_bf16));
  SVI_CUDA_LAUNCH_CHECK("svi_audio_interp_layernorm");
  return SVI_OK;
}

extern "C" int svi_audio_pos_conv(const float* x, int32_t S, int32_t D, int32_t groups, int32_t k, const float* w_packed,
                                  const float* bias, float* out, void* stream) {
  using namespace svi;
  SVI_REQUIRE(x && w_packed && bias && out && S > 0 && groups > 0 && D % groups == 0, "svi_audio_pos_conv: bad arguments");
  const int cg = D / groups;
  SVI_REQUIRE(cg <= audio::PC_MAX_CG && (cg * audio::PC_TQ) % 32 == 0, "svi_audio_pos_conv: D / groups must be a multiple of 8 and <= 64");
  SVI_REQUIRE(k > 0 && k % 2 == 0 && k <= 256, "svi_audio_pos_conv: k must be even and <= 256");
  SVI_REQUIRE(x != out, "svi_audio_pos_conv: out must not alias x");
  const size_t smem = sizeof(float) * ((size_t)(audio::PC_TT + k - 1) * (cg + 1) + (size_t)audio::PC_JC * cg * cg);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(audio::pos_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_set = true;
  }
  dim3 grid((S + audio::PC_TT - 1) / audio::PC_TT, groups);
  audio::pos_conv_kernel<<<grid, cg * audio::PC_TQ, smem, static_cast<cudaStream_t>(stream)>>>(x, S, D, cg, k, w_packed, bias, out);
  SVI_CUDA_LAUNCH_CHECK("svi_audio_pos_conv");
  return SVI_OK;
}

extern "C" int svi_layernorm_f32x2(const float* x, int64_t ldx, int32_t M, int32_t D, float eps, const float* gamma,
                                   const float* beta, float* y, int64_t ldy, void* y_bf16, void* stream) {
  using namespace svi;
  SVI_REQUIRE(x && gamma && beta && y && y_bf16 && M > 0 && D > 0 && ldx >= D && ldy >= D, "svi_layernorm_f32x2: bad arguments");
  audio::layernorm_f32x2_kernel<<<M, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, ldx, D, eps, gamma, beta, y, ldy, reinterpret_cast<__nv_bfloat16*>(y_bf16));
  SVI_CUDA_LAUNCH_CHECK("svi_layernorm_f32x2");
  return SVI_OK;
}
