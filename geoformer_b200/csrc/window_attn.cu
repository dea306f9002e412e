// LoFTR full attention at the fine level (loftr_module/linear_attention.py:54-85 with `fine.attention: 'full'`):
// every token of a 25-token window attends to the 25 tokens of the paired window, softmax(Q K^T / sqrt(16)) V per head,
// heads x 16.  One warp per (window, head): lane t < tokens owns query token t; the head's K and V rows of the window
// (25 x 16 each) sit in shared memory and are read as broadcasts.  Q / K / V are fp16 (OUT16 projection, product mode)
// or fp32 (accurate mode); the arithmetic and the message are fp32.
#include "common.cuh"

#include <atomic>
#include <cuda_fp16.h>

namespace gf {
extern std::atomic<int64_t> g_launches;

namespace wa {
constexpr int kDim = 16;
constexpr int kMaxTokens = 32;
constexpr int kWarps = 4;
}  // namespace wa

__device__ __forceinline__ void load16(const float* p, float (&x)[wa::kDim]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p) + i);
    x[4 * i] = a.x; x[4 * i + 1] = a.y; x[4 * i + 2] = a.z; x[4 * i + 3] = a.w;
  }
}
__device__ __forceinline__ void load16(const __half* p, float (&x)[wa::kDim]) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p) + i);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
      x[8 * i + 2 * j] = f.x; x[8 * i + 2 * j + 1] = f.y;
    }
  }
}

// grid ceil(n_windows * heads / 4), 128 threads; out [n_windows * tokens, heads * 16] fp32
template <typename T>
__global__ void __launch_bounds__(32 * wa::kWarps)
window_full_attention_kernel(const T* __restrict__ q, int ldq, const T* __restrict__ k, int ldk, const T* __restrict__ v,
                             int ldv, float* __restrict__ out, int64_t n_windows, int tokens, int heads, float scale) {
  using namespace wa;
  __shared__ float ks[kWarps][kMaxTokens][kDim];
  __shared__ float vs[kWarps][kMaxTokens][kDim];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t item = (int64_t)blockIdx.x * kWarps + warp;                  // (window, head)
  if (item >= n_windows * heads) return;                                      // whole warps leave together
  const int64_t m = item / heads;
  const int h = (int)(item - m * heads);
  const int64_t row = m * tokens + lane;
  float x[kDim];
  if (lane < tokens) {
    load16(k + row * ldk + h * kDim, x);
#pragma unroll
    for (int d = 0; d < kDim; ++d) ks[warp][lane][d] = x[d];
    load16(v + row * ldv + h * kDim, x);
#pragma unroll
    for (int d = 0; d < kDim; ++d) vs[warp][lane][d] = x[d];
    load16(q + row * ldq + h * kDim, x);
  }
  __syncwarp();
  if (lane >= tokens) return;
  // two passes over the keys (the 16-term dots are recomputed bit-identically rather than held in 32 registers)
  auto score = [&](int j) {
    float dot = 0.f;
#pragma unroll
    for (int d = 0; d < kDim; ++d) dot = fmaf(x[d], ks[warp][j][d], dot);
    return dot * scale;
  };
  float mx = -INFINITY;
#pragma unroll 5
  for (int j = 0; j < tokens; ++j) mx = fmaxf(mx, score(j));
  float den = 0.f, acc[kDim];
#pragma unroll
  for (int d = 0; d < kDim; ++d) acc[d] = 0.f;
#pragma unroll 5
  for (int j = 0; j < tokens; ++j) {
    const float p = expf(score(j) - mx);
    den += p;
#pragma unroll
    for (int d = 0; d < kDim; ++d) acc[d] = fmaf(p, vs[warp][j][d], acc[d]);
  }
  const float inv = 1.f / den;
  float4* dst = reinterpret_cast<float4*>(out + row * (int64_t)(heads * kDim) + h * kDim);
#pragma unroll
  for (int i = 0; i < 4; ++i) dst[i] = make_float4(acc[4 * i] * inv, acc[4 * i + 1] * inv, acc[4 * i + 2] * inv, acc[4 * i + 3] * inv);
}

template <typename T>
static int launch_window_full_attention(const T* q, int ldq, const T* k, int ldk, const T* v, int ldv, float* out,
                                        int64_t n_windows, int tokens, int heads, int dim, gf_stream_t stream,
                                        const char* name) {
  constexpr int align = 16 / (int)sizeof(T);
  if (n_windows <= 0 || tokens <= 0 || tokens > wa::kMaxTokens || heads <= 0 || dim != wa::kDim || (ldq % align) ||
      (ldk % align) || (ldv % align))
    return gf_set_error(GF_ERR_ARG, name);
  const int64_t items = n_windows * heads;
  window_full_attention_kernel<T><<<gf_cdiv(items, wa::kWarps), 32 * wa::kWarps, 0, (cudaStream_t)stream>>>(
      q, ldq, k, ldk, v, ldv, out, n_windows, tokens, heads, 1.f / sqrtf((float)dim));
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

}  // namespace gf

using namespace gf;

extern "C" int gf_full_attention_window(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* out,
                                        int64_t n_windows, int tokens, int heads, int dim, gf_stream_t stream) {
  return launch_window_full_attention(q, ldq, k, ldk, v, ldv, out, n_windows, tokens, heads, dim, stream,
                                      "gf_full_attention_window: needs dim 16, <= 32 tokens, 16-byte rows");
}

extern "C" int gf_full_attention_window_f16(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, float* out,
                                            int64_t n_windows, int tokens, int heads, int dim, gf_stream_t stream) {
  return launch_window_full_attention((const __half*)q, ldq, (const __half*)k, ldk, (const __half*)v, ldv, out, n_windows,
                                      tokens, heads, dim, stream,
                                      "gf_full_attention_window_f16: needs dim 16, <= 32 tokens, 16-byte rows");
}
