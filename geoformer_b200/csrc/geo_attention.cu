// Geometrized attention kernels (model/geo_module.py:51-94, utils/common_utils.py:65-91,166-181,
// utils/homography.py:86-105, model/geo_transformer/transformer.py:111-139, geo_attention.py:72-100).
#include "common.cuh"

#include <atomic>
#include <cuda_fp16.h>

namespace gf {
extern std::atomic<int64_t> g_launches;

// ---------------------------------------------------------------------------------------------
// window token table.  One thread per (sample, source token).
//   centre = H * (x, y, 1) with x = col*scale, y = row*scale (fp32, z==0 -> 1e-6)
//   slot w = r*window + c : (kx, ky) = centre + ((c-half)*scale, (r-half)*scale)
//   out of [0,W) x [0,H)  -> -1 ;  else token = (int(ky)/scale) * w_dst_c + int(kx)/scale
// ---------------------------------------------------------------------------------------------
__global__ void geo_window_table_kernel(const float* __restrict__ hmat, const int* __restrict__ has_h, int n, int l,
                                        int w_src_c, int h_dst_px, int w_dst_px, int w_dst_c, int scale, int window,
                                        int* __restrict__ widx) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n * l) return;
  const int b = (int)(idx / l);
  const int tok = (int)(idx - (int64_t)b * l);
  int* out = widx + idx * window * window;
  if (!has_h[b]) {
    for (int w = 0; w < window * window; ++w) out[w] = -1;
    return;
  }
  const float* H = hmat + b * 9;
  const float x = (float)((tok % w_src_c) * scale), y = (float)((tok / w_src_c) * scale);
  // k = 0,1,2 accumulation order of a 3-term sgemm dot product
  float wx = __fmaf_rn(H[2], 1.f, __fmaf_rn(H[1], y, __fmul_rn(H[0], x)));
  float wy = __fmaf_rn(H[5], 1.f, __fmaf_rn(H[4], y, __fmul_rn(H[3], x)));
  float wz = __fmaf_rn(H[8], 1.f, __fmaf_rn(H[7], y, __fmul_rn(H[6], x)));
  if (wz == 0.f) wz = 1e-6f;
  const float cx = __fdiv_rn(wx, wz), cy = __fdiv_rn(wy, wz);
  const int half = window / 2;
  for (int r = 0; r < window; ++r) {
    for (int c = 0; c < window; ++c) {
      const float kx = __fadd_rn(cx, (float)((c - half) * scale));
      const float ky = __fadd_rn(cy, (float)((r - half) * scale));
      const bool oob = (kx < 0.f) | (ky < 0.f) | (kx >= (float)w_dst_px) | (ky >= (float)h_dst_px) | !(kx == kx) | !(ky == ky);
      int t = -1;
      if (!oob) t = ((int)ky / scale) * w_dst_c + ((int)kx / scale);
      out[r * window + c] = t;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// self attention against anchor tokens: flash-style online softmax, fp32 FFMA.
// grid (ceil(l/64), heads, n); 256 threads as 16x16, each thread owns a 4x4 block of the 64x64 score tile
// and a 4 x (D/16) block of the 64 x D output tile (head dim D = 64).
// DENSE: every query attends to all s key rows of its sample (LoFTR full attention, linear_attention.py:54-85; D = 32
// at the coarse level) instead of the anchor rows of its own image.
// ---------------------------------------------------------------------------------------------
constexpr int kSA = 64;          // queries per CTA == keys per tile
constexpr int kSAPad = kSA + 4;

template <int D>
constexpr size_t self_attention_smem_bytes() { return (size_t)(kSA * D + D * kSAPad + kSA * (D + 4) + kSA * kSAPad) * sizeof(float); }

template <int D, bool DENSE>
__global__ void __launch_bounds__(256)
geo_self_attention_kernel(const float* __restrict__ q, int ldq, const float* __restrict__ k, int ldk,
                          const float* __restrict__ v, int ldv, float* __restrict__ out, int l, int s, int heads,
                          const int* __restrict__ anchor_idx, const int* __restrict__ anchor_cnt, int anchor_cap,
                          float softmax_scale) {
  constexpr int CW = D / 16;              // output columns per thread
  constexpr int VP = D + 4;
  extern __shared__ float sh[];
  float* Qs = sh;                         // [64][D]
  float* Kt = Qs + kSA * D;               // [D][68 keys]
  float* Vs = Kt + D * kSAPad;            // [64 keys][D + 4]
  float* Ps = Vs + kSA * VP;              // [64 q][68]
  const int n = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * kSA;
  const int cnt = DENSE ? s : anchor_cnt[n];
  const int c = heads * D;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  if (cnt == 0) {
    for (int e = tid; e < kSA * D; e += 256) {
      const int r = e / D, d = e % D;
      if (q0 + r < l) out[((int64_t)n * l + q0 + r) * c + h * D + d] = 0.f;
    }
    return;
  }
  for (int e = tid; e < kSA * D; e += 256) {
    const int r = e / D, d = e % D;
    Qs[e] = (q0 + r < l) ? q[((int64_t)n * l + q0 + r) * ldq + h * D + d] : 0.f;
  }
  float m_run[4], l_run[4], o[4][CW];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m_run[i] = -INFINITY; l_run[i] = 0.f;
#pragma unroll
    for (int j = 0; j < CW; ++j) o[i][j] = 0.f;
  }
  const int* aidx = DENSE ? nullptr : anchor_idx + (int64_t)n * anchor_cap;
  for (int k0 = 0; k0 < cnt; k0 += kSA) {
    __syncthreads();   // previous tile fully consumed (also covers the Qs fill on the first iteration)
    for (int e = tid; e < kSA * D; e += 256) {
      const int r = e / D, d = e % D;
      float kv = 0.f, vv = 0.f;
      if (k0 + r < cnt) {
        const int64_t tok = DENSE ? (int64_t)n * s + k0 + r : (int64_t)n * l + aidx[k0 + r];
        kv = k[tok * ldk + h * D + d];
        vv = v[tok * ldv + h * D + d];
      }
      Kt[d * kSAPad + r] = kv;
      Vs[r * VP + d] = vv;
    }
    __syncthreads();
    float s_[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s_[i][j] = 0.f;
#pragma unroll 8
    for (int d = 0; d < D; ++d) {
      const float4 kk = *reinterpret_cast<const float4*>(&Kt[d * kSAPad + 4 * tx]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float qv = Qs[(4 * ty + i) * D + d];
        s_[i][0] = fmaf(qv, kk.x, s_[i][0]); s_[i][1] = fmaf(qv, kk.y, s_[i][1]);
        s_[i][2] = fmaf(qv, kk.z, s_[i][2]); s_[i][3] = fmaf(qv, kk.w, s_[i][3]);
      }
    }
    float alpha[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s_[i][j] = (k0 + 4 * tx + j < cnt) ? s_[i][j] * softmax_scale : -INFINITY;
        mx = fmaxf(mx, s_[i][j]);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float m_new = fmaxf(m_run[i], mx);      // finite: every tile has >= 1 live key
      alpha[i] = expf(m_run[i] - m_new);
      float rs = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) { s_[i][j] = expf(s_[i][j] - m_new); rs += s_[i][j]; }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, off);
      l_run[i] = l_run[i] * alpha[i] + rs;
      m_run[i] = m_new;
      *reinterpret_cast<float4*>(&Ps[(4 * ty + i) * kSAPad + 4 * tx]) = make_float4(s_[i][0], s_[i][1], s_[i][2], s_[i][3]);
#pragma unroll
      for (int j = 0; j < CW; ++j) o[i][j] *= alpha[i];
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < kSA; ++kk) {
      float vv[CW];
      if constexpr (CW == 4) {
        const float4 t = *reinterpret_cast<const float4*>(&Vs[kk * VP + 4 * tx]);
        vv[0] = t.x; vv[1] = t.y; vv[2] = t.z; vv[3] = t.w;
      } else {
        const float2 t = *reinterpret_cast<const float2*>(&Vs[kk * VP + 2 * tx]);
        vv[0] = t.x; vv[1] = t.y;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float pv = Ps[(4 * ty + i) * kSAPad + kk];
#pragma unroll
        for (int j = 0; j < CW; ++j) o[i][j] = fmaf(pv, vv[j], o[i][j]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = q0 + 4 * ty + i;
    if (r < l) {
      const float inv = 1.f / l_run[i];
      float* dst = &out[((int64_t)n * l + r) * c + h * D + CW * tx];
      if constexpr (CW == 4) *reinterpret_cast<float4*>(dst) = make_float4(o[i][0] * inv, o[i][1] * inv, o[i][2] * inv, o[i][3] * inv);
      else *reinterpret_cast<float2*>(dst) = make_float2(o[i][0] * inv, o[i][1] * inv);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// cross attention: one warp per query token, all heads; lane owns 8 consecutive channels
// (heads*dim == 256, dim == 64 -> 8 lanes per head).  Keys/values are gathered rows of the
// once-projected K/V of the other image (project-then-gather; the reference gathers-then-projects,
// which is the same arithmetic per row but 25x the FLOPs).
// ---------------------------------------------------------------------------------------------
// T = float, or __half when Q|K|V come from the OUT16 projection (the message is then fp16 too and feeds the fp16 merge)
__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const __half* p, float (&v)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
    v[2 * i] = f.x; v[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(__half* p, const float (&v)[8]) {
  uint4 u;
  __half2 h;
  h = __floats2half2_rn(v[0], v[1]); u.x = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2half2_rn(v[2], v[3]); u.y = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2half2_rn(v[4], v[5]); u.z = *reinterpret_cast<uint32_t*>(&h);
  h = __floats2half2_rn(v[6], v[7]); u.w = *reinterpret_cast<uint32_t*>(&h);
  *reinterpret_cast<uint4*>(p) = u;
}

template <typename T>
__global__ void geo_cross_attention_kernel(const T* __restrict__ q, int ldq, const T* __restrict__ kp, int ldk,
                                           const T* __restrict__ vp, int ldv, T* __restrict__ out, int n, int l,
                                           int s, const int* __restrict__ widx, int window2, float softmax_scale) {
  const int64_t tok = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (tok >= (int64_t)n * l) return;
  const int b = (int)(tok / l);
  const int* wi = widx + tok * window2;
  float qv[8];
  load8(q + tok * ldq + lane * 8, qv);
  float sc[25];
  int id[25];
  float mx = -INFINITY;
  int live = 0;
#pragma unroll
  for (int w = 0; w < 25; ++w) {
    const int t = w < window2 ? wi[w] : -1;
    id[w] = t;
    float d = 0.f;
    if (t >= 0) {
      float kv[8];
      load8(kp + ((int64_t)b * s + t) * ldk + lane * 8, kv);
      d = qv[0] * kv[0] + qv[1] * kv[1] + qv[2] * kv[2] + qv[3] * kv[3] + qv[4] * kv[4] + qv[5] * kv[5] + qv[6] * kv[6] + qv[7] * kv[7];
      ++live;
    }
    d += __shfl_xor_sync(0xffffffffu, d, 1);
    d += __shfl_xor_sync(0xffffffffu, d, 2);
    d += __shfl_xor_sync(0xffffffffu, d, 4);
    // masked_fill_(~mask, -1e8) happens BEFORE the 1/sqrt(D) temperature (geo_attention.py:83-91)
    sc[w] = (t >= 0 ? d : -1e8f) * softmax_scale;
    if (w < window2) mx = fmaxf(mx, sc[w]);
  }
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (live > 0) {          // all-masked rows are zeroed (geo_attention.py:98-100)
    float den = 0.f;
#pragma unroll
    for (int w = 0; w < 25; ++w) {
      if (w < window2) { sc[w] = expf(sc[w] - mx); den += sc[w]; }
    }
    const float inv = 1.f / den;
#pragma unroll
    for (int w = 0; w < 25; ++w) {
      if (w < window2 && id[w] >= 0) {
        const float p = sc[w] * inv;
        float vv[8];
        load8(vp + ((int64_t)b * s + id[w]) * ldv + lane * 8, vv);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = fmaf(p, vv[i], acc[i]);
      }
    }
  }
  store8(out + tok * 256 + lane * 8, acc);
}

// ---------------------------------------------------------------------------------------------
// tensor-core path of the self attention: anchor K rows gathered per head (K-major for Q K^T) and
// anchor V rows gathered transposed (K-major for P V), masked row soft-max in between.
//   kg[h][n][s_pad][dim]   vt[h][n][dim][s_pad]   (zero beyond anchor_cnt[n])
// ---------------------------------------------------------------------------------------------
__global__ void gather_anchor_kv_kernel(const float* __restrict__ k, int ldk, const float* __restrict__ v, int ldv,
                                        int n, int l, int heads, int dim, const int* __restrict__ anchor_idx,
                                        const int* __restrict__ anchor_cnt, int anchor_cap, int s_pad,
                                        float* __restrict__ kg, float* __restrict__ vt) {
  const int c = heads * dim;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;     // over n * s_pad * c
  if (idx >= (int64_t)n * s_pad * c) return;
  const int ch = (int)(idx % c);
  const int64_t r = idx / c;
  const int s = (int)(r % s_pad), b = (int)(r / s_pad);
  const int h = ch / dim, d = ch - h * dim;
  float kv = 0.f, vv = 0.f;
  if (s < anchor_cnt[b]) {
    const int64_t tok = (int64_t)b * l + anchor_idx[(int64_t)b * anchor_cap + s];
    kv = k[tok * ldk + ch];
    vv = v[tok * ldv + ch];
  }
  kg[(((int64_t)h * n + b) * s_pad + s) * dim + d] = kv;
  vt[(((int64_t)h * n + b) * dim + d) * s_pad + s] = vv;
}

// fp16 variant for the fused flash kernel; the same launch also converts the query rows: q16[n*l][c]
__global__ void gather_anchor_kv_f16_kernel(const float* __restrict__ q, int ldq, const float* __restrict__ k, int ldk,
                                            const float* __restrict__ v, int ldv, int n, int l, int heads, int dim,
                                            const int* __restrict__ anchor_idx, const int* __restrict__ anchor_cnt,
                                            int anchor_cap, int s_pad, __half* __restrict__ q16, __half* __restrict__ kg,
                                            __half* __restrict__ vt) {
  const int c = heads * dim;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_kv = (int64_t)n * s_pad * c, n_q = (int64_t)n * l * c;
  if (idx < n_kv) {
    const int ch = (int)(idx % c);
    const int64_t r = idx / c;
    const int s = (int)(r % s_pad), b = (int)(r / s_pad);
    const int h = ch / dim, d = ch - h * dim;
    float kv = 0.f, vv = 0.f;
    if (s < anchor_cnt[b]) {
      const int64_t tok = (int64_t)b * l + anchor_idx[(int64_t)b * anchor_cap + s];
      kv = k[tok * ldk + ch];
      vv = v[tok * ldv + ch];
    }
    kg[(((int64_t)h * n + b) * s_pad + s) * dim + d] = __float2half_rn(kv);
    vt[(((int64_t)h * n + b) * dim + d) * s_pad + s] = __float2half_rn(vv);
  } else if (idx < n_kv + n_q) {
    const int64_t e = idx - n_kv;
    const int64_t row = e / c;
    q16[e] = __float2half_rn(q[row * ldq + (e - row * c)]);
  }
}

// Same gather from fp16 K / V rows (the OUT16 projection): kg rows are copied as 16-byte chunks, the V tile of 64
// anchors is transposed through shared memory so that vt rows leave as 16-byte vectors too.  grid (s_pad / 64, n),
// 256 threads; heads * D == 256.  DENSE: key j of sample b is row b * s + j of K / V (all s rows, no anchor list), and
// block (0, b) also writes key_cnt[b] = s for the flash kernel.
template <int D, bool DENSE>
__global__ void __launch_bounds__(256)
gather_anchor_kv_h16_kernel(const __half* __restrict__ k, int ldk, const __half* __restrict__ v, int ldv, int n, int l,
                            const int* __restrict__ anchor_idx, const int* __restrict__ anchor_cnt, int anchor_cap,
                            int s_pad, __half* __restrict__ kg, __half* __restrict__ vt, int* __restrict__ key_cnt) {
  constexpr int C = 256, PITCH = C + 8, CH = D / 8;           // CH: 16-byte chunks per head row
  __shared__ __align__(16) __half vs[64 * PITCH];
  const int b = blockIdx.y, s0 = blockIdx.x * 64, t = threadIdx.x;
  const int cnt = DENSE ? l : anchor_cnt[b];                  // dense: l is the key count s of every sample
  if (DENSE && blockIdx.x == 0 && t == 0) key_cnt[b] = cnt;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int e = t + 256 * i, r = e >> 5, q = e & 31;       // anchor row r of the tile, 16-byte chunk q of its 512 B
    const int s = s0 + r;
    uint4 kq = make_uint4(0u, 0u, 0u, 0u), vq = kq;
    if (s < cnt) {
      const int64_t tok = DENSE ? (int64_t)b * l + s : (int64_t)b * l + anchor_idx[(int64_t)b * anchor_cap + s];
      kq = __ldg(reinterpret_cast<const uint4*>(k + tok * ldk) + q);
      vq = __ldg(reinterpret_cast<const uint4*>(v + tok * ldv) + q);
    }
    if (s < s_pad) {
      const int h = q / CH;
      *reinterpret_cast<uint4*>(kg + (((int64_t)h * n + b) * s_pad + s) * D + (q % CH) * 8) = kq;
    }
    *reinterpret_cast<uint4*>(vs + r * PITCH + q * 8) = vq;
  }
  __syncthreads();
  const int h = t / D, d = t % D;                             // thread == channel
  __half* dst = vt + (((int64_t)h * n + b) * D + d) * s_pad + s0;
#pragma unroll
  for (int g8 = 0; g8 < 8; ++g8) {
    if (s0 + 8 * g8 >= s_pad) break;
    __half tmp[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) tmp[j] = vs[(8 * g8 + j) * PITCH + t];
    *reinterpret_cast<uint4*>(dst + 8 * g8) = *reinterpret_cast<const uint4*>(tmp);
  }
}

// rows of [heads][n][l][s_pad]: p = softmax(x[0:cnt]) (x is already scaled), zeros beyond cnt.  One warp per row.
// PER_LANE > 0: the whole row (s_pad <= 32 * PER_LANE) lives in registers -> one read and one write of the block.
template <int PER_LANE>
__global__ void masked_softmax_rows_kernel(float* __restrict__ x, int64_t rows, int n, int l, int s_pad,
                                           const int* __restrict__ cnt_per_sample) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int b = (int)((row / l) % n);
  const int cnt = cnt_per_sample[b];
  float* p = x + row * s_pad;
  if constexpr (PER_LANE > 0) {
    float v[PER_LANE];
    float m = -INFINITY;
#pragma unroll
    for (int i = 0; i < PER_LANE; ++i) {
      const int j = lane + 32 * i;
      v[i] = j < cnt ? p[j] : -INFINITY;
      m = fmaxf(m, v[i]);
    }
    m = warp_max(m);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < PER_LANE; ++i) { v[i] = (lane + 32 * i < cnt) ? expf(v[i] - m) : 0.f; sum += v[i]; }
    sum = warp_sum(sum);
    const float inv = cnt > 0 ? 1.f / sum : 0.f;
#pragma unroll
    for (int i = 0; i < PER_LANE; ++i) {
      const int j = lane + 32 * i;
      if (j < s_pad) p[j] = v[i] * inv;
    }
  } else {
    float m = -INFINITY;
    for (int j = lane; j < cnt; j += 32) m = fmaxf(m, p[j]);
    m = warp_max(m);
    float sum = 0.f;
    for (int j = lane; j < cnt; j += 32) sum += expf(p[j] - m);
    sum = warp_sum(sum);
    const float inv = cnt > 0 ? 1.f / sum : 0.f;
    for (int j = lane; j < s_pad; j += 32) p[j] = j < cnt ? expf(p[j] - m) * inv : 0.f;
  }
}

}  // namespace gf

using namespace gf;
#define STREAM ((cudaStream_t)stream)

extern "C" int gf_geo_window_table(const float* hmat, const int* has_h, int n, int h_src_c, int w_src_c, int h_dst_px,
                                   int w_dst_px, int w_dst_c, int scale, int window, int* widx, gf_stream_t stream) {
  if (n <= 0 || h_src_c <= 0 || w_src_c <= 0 || scale <= 0 || window <= 0 || window > 5)
    return gf_set_error(GF_ERR_ARG, "gf_geo_window_table: bad shape");
  const int l = h_src_c * w_src_c;
  geo_window_table_kernel<<<gf_cdiv((int64_t)n * l, 128), 128, 0, STREAM>>>(hmat, has_h, n, l, w_src_c, h_dst_px, w_dst_px,
                                                                          w_dst_c, scale, window, widx);
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

extern "C" int gf_geo_self_attention(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                                     float* out, int n, int l, int heads, int dim, const int* anchor_idx,
                                     const int* anchor_cnt, int anchor_cap, gf_stream_t stream) {
  if (n <= 0 || l <= 0 || heads <= 0 || dim != 64) return gf_set_error(GF_ERR_ARG, "gf_geo_self_attention: dim must be 64");
  constexpr size_t smem = self_attention_smem_bytes<64>();
  GF_SMEM_OPTIN((geo_self_attention_kernel<64, false>), smem);
  geo_self_attention_kernel<64, false><<<dim3(gf_cdiv(l, kSA), heads, n), 256, smem, STREAM>>>(
      q, ldq, k, ldk, v, ldv, out, l, l, heads, anchor_idx, anchor_cnt, anchor_cap, 1.f / sqrtf((float)dim));
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

extern "C" int gf_geo_cross_attention(const float* q, int ldq, const float* kproj, int ldk, const float* vproj, int ldv,
                                      float* out, int n, int l, int s, int heads, int dim, const int* widx, int window2,
                                      gf_stream_t stream) {
  if (n <= 0 || l <= 0 || s <= 0 || heads * dim != 256 || dim != 64 || window2 <= 0 || window2 > 25)
    return gf_set_error(GF_ERR_ARG, "gf_geo_cross_attention: needs heads*dim == 256, dim == 64, window <= 25");
  geo_cross_attention_kernel<float><<<gf_cdiv((int64_t)n * l, 4), 128, 0, STREAM>>>(q, ldq, kproj, ldk, vproj, ldv, out, n, l, s,
                                                                                   widx, window2, 1.f / sqrtf((float)dim));
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

extern "C" int gf_geo_cross_attention_f16(const void* q, int ldq, const void* kproj, int ldk, const void* vproj, int ldv,
                                          void* out, int n, int l, int s, int heads, int dim, const int* widx, int window2,
                                          gf_stream_t stream) {
  if (n <= 0 || l <= 0 || s <= 0 || heads * dim != 256 || dim != 64 || window2 <= 0 || window2 > 25 || (ldq % 8) || (ldk % 8) || (ldv % 8))
    return gf_set_error(GF_ERR_ARG, "gf_geo_cross_attention_f16: needs heads*dim == 256, dim == 64, window <= 25, 16-byte rows");
  geo_cross_attention_kernel<__half><<<gf_cdiv((int64_t)n * l, 4), 128, 0, STREAM>>>(
      (const __half*)q, ldq, (const __half*)kproj, ldk, (const __half*)vproj, ldv, (__half*)out, n, l, s, widx, window2,
      1.f / sqrtf((float)dim));
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

extern "C" int gf_gather_anchor_kv(const float* k, int ldk, const float* v, int ldv, int n, int l, int heads, int dim,
                                   const int* anchor_idx, const int* anchor_cnt, int anchor_cap, int s_pad, float* kg,
                                   float* vt, gf_stream_t stream) {
  if (n <= 0 || l <= 0 || heads <= 0 || dim <= 0 || s_pad <= 0) return gf_set_error(GF_ERR_ARG, "gf_gather_anchor_kv: bad shape");
  const int64_t total = (int64_t)n * s_pad * heads * dim;
  gather_anchor_kv_kernel<<<gf_cdiv(total, 256), 256, 0, STREAM>>>(k, ldk, v, ldv, n, l, heads, dim, anchor_idx, anchor_cnt,
                                                                   anchor_cap, s_pad, kg, vt);
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

extern "C" int gf_gather_anchor_kv_f16(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, int n,
                                       int l, int heads, int dim, const int* anchor_idx, const int* anchor_cnt,
                                       int anchor_cap, int s_pad, void* q16, void* kg, void* vt, gf_stream_t stream) {
  if (n <= 0 || l <= 0 || heads <= 0 || dim <= 0 || s_pad <= 0) return gf_set_error(GF_ERR_ARG, "gf_gather_anchor_kv_f16: bad shape");
  const int64_t total = (int64_t)n * (s_pad + l) * heads * dim;
  gather_anchor_kv_f16_kernel<<<gf_cdiv(total, 256), 256, 0, STREAM>>>(q, ldq, k, ldk, v, ldv, n, l, heads, dim, anchor_idx,
                                                                       anchor_cnt, anchor_cap, s_pad, (__half*)q16, (__half*)kg,
                                                                       (__half*)vt);
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

extern "C" int gf_gather_anchor_kv_h16(const void* k, int ldk, const void* v, int ldv, int n, int l, int heads, int dim,
                                       const int* anchor_idx, const int* anchor_cnt, int anchor_cap, int s_pad, void* kg,
                                       void* vt, gf_stream_t stream) {
  if (n <= 0 || l <= 0 || heads * dim != 256 || dim != 64 || s_pad <= 0 || (s_pad % 8) || (ldk % 8) || (ldv % 8))
    return gf_set_error(GF_ERR_ARG, "gf_gather_anchor_kv_h16: needs 4 heads of dim 64, s_pad % 8 == 0, 16-byte aligned rows");
  gather_anchor_kv_h16_kernel<64, false><<<dim3(gf_cdiv(s_pad, 64), n), 256, 0, STREAM>>>(
      (const __half*)k, ldk, (const __half*)v, ldv, n, l, anchor_idx, anchor_cnt, anchor_cap, s_pad, (__half*)kg, (__half*)vt,
      nullptr);
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

// LoFTR full attention (linear_attention.py:54-85) over dense keys, fp32 FFMA: out[n*l, heads*32] from the query rows
// q [n*l] and the key / value rows k, v [n*s] (row strides ldq / ldk / ldv floats); scale 1/sqrt(32).
extern "C" int gf_full_attention(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* out,
                                 int n, int l, int s, int heads, int dim, gf_stream_t stream) {
  if (n <= 0 || l <= 0 || s <= 0 || heads <= 0 || dim != 32) return gf_set_error(GF_ERR_ARG, "gf_full_attention: dim must be 32");
  constexpr size_t smem = self_attention_smem_bytes<32>();
  GF_SMEM_OPTIN((geo_self_attention_kernel<32, true>), smem);
  geo_self_attention_kernel<32, true><<<dim3(gf_cdiv(l, kSA), heads, n), 256, smem, STREAM>>>(
      q, ldq, k, ldk, v, ldv, out, l, s, heads, nullptr, nullptr, 0, 1.f / sqrtf((float)dim));
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

// Dense K / V^T tiles of gf_full_attention_tc from fp16 K / V rows [n*s] (8 heads of dim 32):
// kg[h][n][s_pad][32], vt[h][n][32][s_pad] (zero for keys >= s) and key_cnt[n] = s.
extern "C" int gf_dense_kv_h16(const void* k, int ldk, const void* v, int ldv, int n, int s, int heads, int dim, int s_pad,
                               void* kg, void* vt, int* key_cnt, gf_stream_t stream) {
  if (n <= 0 || s <= 0 || heads * dim != 256 || dim != 32 || s_pad < s || (s_pad % 64) || (ldk % 8) || (ldv % 8))
    return gf_set_error(GF_ERR_ARG, "gf_dense_kv_h16: needs 8 heads of dim 32, s <= s_pad, s_pad % 64 == 0, 16-byte rows");
  gather_anchor_kv_h16_kernel<32, true><<<dim3(s_pad / 64, n), 256, 0, STREAM>>>(
      (const __half*)k, ldk, (const __half*)v, ldv, n, s, nullptr, nullptr, 0, s_pad, (__half*)kg, (__half*)vt, key_cnt);
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

extern "C" int gf_masked_softmax_rows(float* x, int heads, int n, int l, int s_pad, const int* cnt_per_sample,
                                      gf_stream_t stream) {
  if (heads <= 0 || n <= 0 || l <= 0 || s_pad <= 0) return gf_set_error(GF_ERR_ARG, "gf_masked_softmax_rows: bad shape");
  const int64_t rows = (int64_t)heads * n * l;
  if (s_pad <= 512)       masked_softmax_rows_kernel<16><<<gf_cdiv(rows, 8), 256, 0, STREAM>>>(x, rows, n, l, s_pad, cnt_per_sample);
  else if (s_pad <= 1024) masked_softmax_rows_kernel<32><<<gf_cdiv(rows, 8), 256, 0, STREAM>>>(x, rows, n, l, s_pad, cnt_per_sample);
  else if (s_pad <= 2048) masked_softmax_rows_kernel<64><<<gf_cdiv(rows, 8), 256, 0, STREAM>>>(x, rows, n, l, s_pad, cnt_per_sample);
  else                    masked_softmax_rows_kernel<0><<<gf_cdiv(rows, 8), 256, 0, STREAM>>>(x, rows, n, l, s_pad, cnt_per_sample);
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}
