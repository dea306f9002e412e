// Fused geo self-attention on tcgen05 (model/geo_transformer/transformer.py:111-124 + geo_attention.py:72-97):
// every token of an image attends to that image's anchor (RANSAC-inlier) tokens, full softmax, heads x 64.
//
// One CTA = 128 queries of one (sample, head); key tiles of 64 anchors stream through shared memory by TMA; two CTAs are
// resident per SM (256 TMEM columns, 192 threads, ~70 KB of shared memory each) and fill each other's pipeline bubbles.
// r02 redesign (the r01 kernel made two passes over the keys with Q and P as shared-memory operands: 20.9 % tensor pipe;
// an N = 64 MMA with a shared-memory A operand reads 6 KB per 32 cycles, more than the 128 B/clk port delivers):
//   * BOTH A operands live in tensor memory (tcgen05.mma ".ts" form): Q is written there once per CTA, P is written by
//     the softmax warps straight over the first 32 columns of the score buffer it was computed from; shared memory only
//     feeds the K and V^T tiles (2 KB per MMA);
//   * ONE pass over the keys: S_t = Q K_t^T (TMEM, double buffered); softmax warps (thread == query row) keep a
//     reference maximum m in the log2 domain that is raised LAZILY - only when a tile's maximum exceeds it by more
//     than 8 (P <= 2^8 stays far inside fp16's range); only then is the accumulator rescaled (tcgen05.ld -> scale ->
//     tcgen05.st, warp-uniform, after the previous P V retired); P = 2^(s c2 - m): one FFMA + one MUFU.EX2 per element,
//     pairs packed to fp16 (ex2.approx.f16x2 is half rate on sm_100a: it compiles to two MUFU.EX2.F16);
//   * O += P_t V_t  and  l += P_t 1  (a second N = 16 MMA against a constant ones tile: the row sums accumulate in fp32 on
//     the tensor core instead of 64 FADDs per row and tile);  out = O / l.
// Operands are fp16 (kind::f16, fp32 accumulate).  The score matrix never touches HBM.
// Roles: warp 0 TMA producer, warp 1 MMA issuer (+TMEM alloc), warps 2..5 softmax / epilogue.
//
// The same body runs LoFTR's full attention (loftr_module/linear_attention.py:54-85, `attention: 'full'`) at the coarse
// level: heads x 32, dense keys (every query attends to all s tokens of its sample's source).  Per score the softmax work
// is the same; the K tile shrinks to 64-byte rows (64B swizzle), the Q K^T MMA to two K = 16 steps and P V to N = 32.
#include "common.cuh"
#include "ptx.cuh"

#include <atomic>
#include <cuda_fp16.h>

namespace gf {
extern std::atomic<int64_t> g_launches;

namespace fa {
constexpr int kBQ = 128;       // queries per CTA
constexpr int kBK = 64;        // keys per tile
constexpr int kRing = 4;       // K / V^T smem stages
constexpr int kOnesBytes = 16 * 128;            // B operand of the row-sum MMA: [16][64 keys] fp16, row 0 = 1
constexpr int kSoftWarps = 4;
constexpr int kThreads = 64 + 32 * kSoftWarps;
constexpr int kTmemCols = 256;                  // S / P: 2 x 64 | O: D | l: 16 | Q: D / 2
constexpr float kLazy = 8.f;                    // log2 units the reference maximum may lag behind
// head dim 64 (geo self attention over anchors) or 32 (LoFTR coarse full attention over dense keys)
template <int D>
struct Cfg {
  static_assert(D == 64 || D == 32, "head dim 64 or 32");
  static constexpr int kKBytes = kBK * D * 2;   // 64 keys x D dims (fp16): 128 B rows (128B swizzle) or 64 B rows (64B)
  static constexpr int kVBytes = D * 128;       // V^T tile: D dim rows x 64 keys (fp16)
  static constexpr int kRingBytes = kRing * (kKBytes + kVBytes);   // the epilogue stages the output here (D x 512 B)
  static constexpr int kSmem = kRingBytes + kOnesBytes + 1024 + 256;
  static constexpr int kColO = 128, kColL = kColO + D, kColQ = kColL + 16;
  static constexpr uint32_t kKDescHi = D == 64 ? ptx::kDescHiSw128 : ptx::kDescHiSw64;
  static_assert(2 * kSmem <= 227 * 1024, "two CTAs per SM");
  static_assert(kColQ + D / 2 <= kTmemCols, "tensor memory budget");
};
}  // namespace fa

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t ex2_h2(float a, float b) {      // (2^a, 2^b) as packed fp16, a in the low half
  uint32_t y;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(y) : "f"(ex2_approx(b)), "f"(ex2_approx(a)));   // first source -> upper half
  return y;
}

// One CTA = (128-query tile, head, sample) over the first key_cnt[b] keys of the sample's K / V^T tiles (0: zeros).
// D = 64: geo self attention over gathered anchors; D = 32: LoFTR full attention, key_cnt[b] = s for every sample.
template <int D>
__global__ void __launch_bounds__(fa::kThreads, 2)
geo_flash_attn_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                      const __grid_constant__ CUtensorMap tmO, const __half* __restrict__ q16, int ldq,
                      float* __restrict__ out, const int* __restrict__ key_cnt, int n_samples, int l, int heads,
                      float scale) {
  using namespace fa;
  using C = Cfg<D>;
  constexpr int kD = D, kKBytes = C::kKBytes, kVBytes = C::kVBytes, kColO = C::kColO, kColL = C::kColL, kColQ = C::kColQ;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = sK + kRing * kKBytes;
  uint8_t* sOnes = sV + kRing * kVBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOnes + kOnesBytes);
  uint64_t* q_ready = bars;                // 1 (count: softmax warps)
  uint64_t* k_full = bars + 1;             // kRing
  uint64_t* k_empty = k_full + kRing;
  uint64_t* v_full = k_empty + kRing;
  uint64_t* v_empty = v_full + kRing;
  uint64_t* s_full = v_empty + kRing;      // 2
  uint64_t* p_full = s_full + 2;           // 2 (count: softmax warps)
  uint64_t* pv_done = p_full + 2;          // 2
  uint64_t* o_full = pv_done + 2;          // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * kBQ, h = blockIdx.y, b = blockIdx.z;
  const int c = heads * kD;
  const int cnt = key_cnt[b];
  if (cnt <= 0) {   // no anchors: the layer is skipped for this sample (caller restores the features); emit zeros
    for (int e = threadIdx.x; e < kBQ * (kD / 4); e += blockDim.x) {
      const int r = e / (kD / 4), q = e - r * (kD / 4);
      if (q0 + r < l) reinterpret_cast<float4*>(out + ((int64_t)b * l + q0 + r) * c + h * kD)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    return;
  }
  const int T = (cnt + kBK - 1) / kBK;
  const int hb = h * n_samples + b;        // batch coordinate of the gathered K / V^T tensors

  if (warp == 0 && lane == 0) { ptx::prefetch_tmap(&tmK); ptx::prefetch_tmap(&tmV); ptx::prefetch_tmap(&tmO); }
  // ones tile (K-major, 128B rows; row 0 = 1.0, rows 1..15 = 0): every 16-byte chunk of a row holds the same value, so
  // the 128B swizzle does not change it
  for (int e = threadIdx.x; e < kOnesBytes / 16; e += blockDim.x) {
    const uint32_t w = (e < 8) ? 0x3C003C00u : 0u;
    reinterpret_cast<uint4*>(sOnes)[e] = make_uint4(w, w, w, w);
  }
  ptx::fence_proxy_async();
  if (warp == 1) {
    if (lane == 0) {
      ptx::mbar_init(q_ready, kSoftWarps);
      for (int i = 0; i < kRing; ++i) {
        ptx::mbar_init(&k_full[i], 1); ptx::mbar_init(&k_empty[i], 1);
        ptx::mbar_init(&v_full[i], 1); ptx::mbar_init(&v_empty[i], 1);
      }
      for (int i = 0; i < 2; ++i) {
        ptx::mbar_init(&s_full[i], 1); ptx::mbar_init(&p_full[i], kSoftWarps); ptx::mbar_init(&pv_done[i], 1);
      }
      ptx::mbar_init(o_full, 1);
      ptx::fence_barrier_init();
    }
    __syncwarp();
    ptx::tmem_alloc(tmem_slot, kTmemCols);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------ TMA producer ------------------------------------
    if (lane == 0) {
      for (int t = 0; t < T; ++t) {
        const int s = t % kRing; const uint32_t ph = (t / kRing) & 1;
        ptx::mbar_wait(&k_empty[s], ph ^ 1);
        ptx::mbar_expect_tx(&k_full[s], kKBytes);
        ptx::tma_load_3d(sK + s * kKBytes, &tmK, &k_full[s], 0, t * kBK, hb);
        ptx::mbar_wait(&v_empty[s], ph ^ 1);
        ptx::mbar_expect_tx(&v_full[s], kVBytes);
        ptx::tma_load_3d(sV + s * kVBytes, &tmV, &v_full[s], t * kBK, 0, hb);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------ MMA issuer ------------------------------------
    // issue order S0, S1, P V0, S2, P V1, ...: S(t) lands in the buffer whose first 32 columns held P(t-2); the tensor
    // core executes in issue order, so it is written only after P V(t-2) has read them
    // (whole warp converged, one elected lane issues: operands stay in uniform registers - see conv_tc.cu)
    {
      constexpr uint32_t idesc = ptx::umma_idesc(0 /*f16*/, kBQ, 64);
      constexpr uint32_t idesc_o = ptx::umma_idesc(0 /*f16*/, kBQ, kD);
      constexpr uint32_t idesc_l = ptx::umma_idesc(0 /*f16*/, kBQ, 16);
      ptx::mbar_wait(q_ready, 0);
      ptx::tc_fence_after();
      const uint32_t smem0 = __shfl_sync(0xffffffffu, ptx::smem_addr(smem), 0);
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t bar0 = smem0 + (uint32_t)((uint8_t*)bars - smem);
      auto bar_addr = [&](const uint64_t* b) -> uint32_t { return bar0 + (uint32_t)((const uint8_t*)b - (const uint8_t*)bars); };
      const uint32_t ones_lo = ptx::umma_desc_lo(smem0 + (uint32_t)(sOnes - smem));
      const uint32_t sK0 = smem0, sV0 = smem0 + kRing * kKBytes;
      for (int t = 0; t <= T; ++t) {
        if (t < T) {
          const int ks = t % kRing; const uint32_t kph = (t / kRing) & 1;
          const int sb = t & 1;
          ptx::mbar_wait(&k_full[ks], kph);
          ptx::tc_fence_after();
          const uint32_t b_lo = ptx::umma_desc_lo(sK0 + ks * kKBytes);
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < kD / 16; ++k) ptx::umma_ts_f16_lo(tb + sb * 64, tb + kColQ + 8 * k, b_lo + 2 * k, C::kKDescHi, idesc, k ? 1u : 0u);
            ptx::umma_commit_addr(bar_addr(&k_empty[ks]));
            ptx::umma_commit_addr(bar_addr(&s_full[sb]));
          }
        }
        if (t > 0) {
          const int u = t - 1;
          const int pb = u & 1; const uint32_t pph = (u >> 1) & 1;
          const int vs = u % kRing; const uint32_t vph = (u / kRing) & 1;
          ptx::mbar_wait(&p_full[pb], pph);
          ptx::mbar_wait(&v_full[vs], vph);
          ptx::tc_fence_after();
          const uint32_t b_lo = ptx::umma_desc_lo(sV0 + vs * kVBytes);
          const uint32_t acc0 = u > 0 ? 1u : 0u;
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) ptx::umma_ts_f16_lo(tb + kColO, tb + pb * 64 + 8 * k, b_lo + 2 * k, ptx::kDescHiSw128, idesc_o, k ? 1u : acc0);
#pragma unroll
            for (int k = 0; k < 4; ++k) ptx::umma_ts_f16_lo(tb + kColL, tb + pb * 64 + 8 * k, ones_lo + 2 * k, ptx::kDescHiSw128, idesc_l, k ? 1u : acc0);
            ptx::umma_commit_addr(bar_addr(&v_empty[vs]));
            ptx::umma_commit_addr(bar_addr(&pv_done[pb]));
          }
        }
      }
      if (ptx::elect_one()) ptx::umma_commit_addr(bar_addr(o_full));
    }
  } else {
    // ------------------------------------ softmax / epilogue (warps 2..5) ------------------------------------
    const int quad = warp & 3;                                     // TMEM lane quadrant (hardware: warp id % 4)
    const int row = quad * 32 + lane;                              // query row inside the CTA tile
    const uint32_t t_lane = tmem_base + (uint32_t(quad * 32) << 16);
    {   // Q row -> tensor memory (A operand of every S MMA): D halves = D / 2 columns, two consecutive dims per column
      uint4 qv[kD / 8];
#pragma unroll
      for (int j = 0; j < kD / 8; ++j) qv[j] = make_uint4(0u, 0u, 0u, 0u);
      if (q0 + row < l) {
        const uint4* qg = reinterpret_cast<const uint4*>(q16 + ((int64_t)b * l + q0 + row) * ldq + h * kD);
#pragma unroll
        for (int j = 0; j < kD / 8; ++j) qv[j] = __ldg(qg + j);
      }
      if constexpr (kD == 64) ptx::tmem_st_32x32(t_lane + kColQ, reinterpret_cast<const float*>(qv));
      else ptx::tmem_st_32x16(t_lane + kColQ, reinterpret_cast<const float*>(qv));
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(q_ready);
    }
    const float c2 = scale * 1.4426950408889634f;                  // logits -> log2 domain
    float m2 = -INFINITY;                                          // reference maximum (log2 domain), raised lazily
    for (int t = 0; t < T; ++t) {
      const int sb = t & 1;
      ptx::mbar_wait(&s_full[sb], (t >> 1) & 1);
      ptx::tc_fence_after();
      float v[64];
      ptx::tmem_ld_32x32(t_lane + sb * 64, v);
      ptx::tmem_ld_32x32(t_lane + sb * 64 + 32, v + 32);
      ptx::tmem_ld_wait();
      const int live = min(kBK, cnt - t * kBK);
      if (live != kBK) {                                           // keys beyond the sample's anchor count
#pragma unroll
        for (int j = 0; j < 64; ++j) if (j >= live) v[j] = -INFINITY;
      }
      float x0 = fmaxf(fmaxf(v[0], v[1]), v[2]), x1 = fmaxf(fmaxf(v[3], v[4]), v[5]);
      float x2 = fmaxf(fmaxf(v[6], v[7]), v[8]), x3 = fmaxf(fmaxf(v[9], v[10]), v[11]);
#pragma unroll
      for (int j = 12; j < 60; j += 8) {
        x0 = fmaxf(fmaxf(x0, v[j]), v[j + 1]); x1 = fmaxf(fmaxf(x1, v[j + 2]), v[j + 3]);
        x2 = fmaxf(fmaxf(x2, v[j + 4]), v[j + 5]); x3 = fmaxf(fmaxf(x3, v[j + 6]), v[j + 7]);
      }
      x0 = fmaxf(fmaxf(x0, v[60]), v[61]); x1 = fmaxf(fmaxf(x1, v[62]), v[63]);
      const float tm2 = fmaxf(fmaxf(x0, x1), fmaxf(x2, x3)) * c2;  // c2 > 0
      // lazy reference maximum: the first tile sets it; later tiles raise it only when they exceed it by > kLazy
      const bool raise = tm2 > m2 + kLazy;                         // (m2 = -inf on the first tile: always true there)
      const float m2_new = raise ? tm2 : m2;
      const bool rescale = __any_sync(0xffffffffu, raise) && t > 0;   // warp-uniform: tcgen05.ld / .st are collective
      const float factor = raise ? ex2_approx(m2 - m2_new) : 1.f;     // 2^(-inf) = 0 can only occur at t == 0 (unused)
      m2 = m2_new;
      uint32_t pk[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) pk[j] = ex2_h2(fmaf(v[2 * j], c2, -m2), fmaf(v[2 * j + 1], c2, -m2));   // -inf -> 0
      if (rescale) {
        // every earlier P V must have retired before the accumulator is touched (P V(t-2) has: S(t) was issued behind it)
        ptx::mbar_wait(&pv_done[(t - 1) & 1], ((t - 1) >> 1) & 1);
        ptx::tc_fence_after();
        float o[32];
#pragma unroll
        for (int hcol = 0; hcol < kD / 32; ++hcol) {
          ptx::tmem_ld_32x32(t_lane + kColO + 32 * hcol, o);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] *= factor;
          ptx::tmem_st_32x32(t_lane + kColO + 32 * hcol, o);
        }
        ptx::tmem_ld_32x16(t_lane + kColL, o);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) o[j] *= factor;
        ptx::tmem_st_32x16(t_lane + kColL, o);
      }
      // P over the first 32 columns of the score buffer it came from (A operand of the P V MMAs)
      ptx::tmem_st_32x32(t_lane + sb * 64, reinterpret_cast<const float*>(pk));
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&p_full[sb]);
    }
    // epilogue: O / l -> D / 32 swizzled 32x32 fp32 boxes per warp (in the idle K / V ring) -> TMA store
    ptx::mbar_wait(o_full, 0);
    ptx::tc_fence_after();
    float lsum[16];
    ptx::tmem_ld_32x16(t_lane + kColL, lsum);
    ptx::tmem_ld_wait();
    const float inv = 1.f / lsum[0];
    uint8_t* wst = smem + (warp - 2) * (kD / 32) * 4096;
#pragma unroll
    for (int hcol = 0; hcol < kD / 32; ++hcol) {
      float o[32];
      ptx::tmem_ld_32x32(t_lane + kColO + 32 * hcol, o);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float4*>(wst + hcol * 4096 + lane * 128 + ((j ^ (lane & 7)) << 4)) =
            make_float4(o[4 * j] * inv, o[4 * j + 1] * inv, o[4 * j + 2] * inv, o[4 * j + 3] * inv);
    }
    ptx::fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
#pragma unroll
      for (int hcol = 0; hcol < kD / 32; ++hcol) ptx::tma_store_3d(&tmO, wst + hcol * 4096, h * kD + 32 * hcol, q0 + quad * 32, b);
      ptx::bulk_commit();
      ptx::bulk_wait<0>();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, fa::kTmemCols);
  }
}

}  // namespace gf

using namespace gf;

namespace gf {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn();
}  // namespace gf

// K tiles of head dim 32: dims {32, s_pad, heads * n} fp16, box {32 = 64 B, 64 keys, 1}, 64B swizzle
static int make_k32_tmap(CUtensorMap* m, const void* kg, int64_t s_pad, int64_t batches) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return gf_set_error(GF_ERR_DRIVER, "gf_init() was not called");
  cuuint64_t dims[3] = {32, (cuuint64_t)s_pad, (cuuint64_t)batches};
  cuuint64_t strides[2] = {64, (cuuint64_t)s_pad * 64};
  cuuint32_t box[3] = {32, (cuuint32_t)fa::kBK, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(kg), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return gf_set_error(GF_ERR_DRIVER, "cuTensorMapEncodeTiled(k32) failed");
  return GF_OK;
}

// fp16 operands from gf_gather_anchor_kv_f16: q16 [n*l, heads*64] (head h at columns [h*64, h*64+64)),
// kg [heads][n][s_pad][64], vt [heads][n][64][s_pad]; out fp32 [n*l, heads*64].
extern "C" int gf_geo_self_attention_tc(const void* q16, int ldq, const void* kg, const void* vt, float* out, int n, int l,
                                        int heads, int dim, int s_pad, const int* anchor_cnt, gf_stream_t stream) {
  using C = fa::Cfg<64>;
  const int c = heads * dim;
  if (n <= 0 || l <= 0 || heads <= 0 || dim != 64 || s_pad <= 0 || (s_pad % 8) || ldq < c || (ldq % 8))
    return gf_set_error(GF_ERR_ARG, "gf_geo_self_attention_tc: dim must be 64, s_pad % 8 == 0, ldq % 8 == 0");
  CUtensorMap tk, tv, to;
  int rc;
  if ((rc = make_tmap(&tk, kg, 2, dim, s_pad, (int64_t)heads * n, dim, (int64_t)s_pad * dim, fa::kBK))) return rc;
  if ((rc = make_tmap(&tv, vt, 2, s_pad, dim, (int64_t)heads * n, s_pad, (int64_t)dim * s_pad, 64))) return rc;
  if ((rc = make_out_tmap(&to, out, c, l, n, c, (int64_t)l * c))) return rc;
  GF_SMEM_OPTIN(geo_flash_attn_kernel<64>, C::kSmem);
  geo_flash_attn_kernel<64><<<dim3(gf_cdiv(l, fa::kBQ), heads, n), fa::kThreads, C::kSmem, (cudaStream_t)stream>>>(
      tk, tv, to, (const __half*)q16, ldq, out, anchor_cnt, n, l, heads, 1.f / sqrtf((float)dim));
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}

// fp16 operands from gf_dense_kv_h16: q16 rows [n*l] with stride ldq (head h at columns [h*32, h*32+32)),
// kg [heads][n][s_pad][32], vt [heads][n][32][s_pad] (zero for keys >= s); key_cnt [n] int32 on the device, every entry
// s (written by gf_dense_kv_h16); out fp32 [n*l, heads*32].
extern "C" int gf_full_attention_tc(const void* q16, int ldq, const void* kg, const void* vt, const int* key_cnt, float* out,
                                    int n, int l, int s, int heads, int dim, int s_pad, gf_stream_t stream) {
  using C = fa::Cfg<32>;
  const int c = heads * dim;
  if (n <= 0 || l <= 0 || s <= 0 || heads <= 0 || dim != 32 || s_pad < s || (s_pad % fa::kBK) || ldq < c || (ldq % 8))
    return gf_set_error(GF_ERR_ARG, "gf_full_attention_tc: dim must be 32, s <= s_pad, s_pad % 64 == 0, ldq % 8 == 0");
  CUtensorMap tk, tv, to;
  int rc;
  if ((rc = make_k32_tmap(&tk, kg, s_pad, (int64_t)heads * n))) return rc;
  if ((rc = make_tmap(&tv, vt, 2, s_pad, dim, (int64_t)heads * n, s_pad, (int64_t)dim * s_pad, 32))) return rc;
  if ((rc = make_out_tmap(&to, out, c, l, n, c, (int64_t)l * c))) return rc;
  GF_SMEM_OPTIN(geo_flash_attn_kernel<32>, C::kSmem);
  geo_flash_attn_kernel<32><<<dim3(gf_cdiv(l, fa::kBQ), heads, n), fa::kThreads, C::kSmem, (cudaStream_t)stream>>>(
      tk, tv, to, (const __half*)q16, ldq, out, key_cnt, n, l, heads, 1.f / sqrtf((float)dim));
  g_launches++;
  GF_CHECK_LAUNCH();
  return GF_OK;
}
