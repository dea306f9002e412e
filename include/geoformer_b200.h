/* libgeoformer_sm100.so — C ABI of the B200-native GeoFormer matching hot path.
 *
 * The reference (ruc-aimc-lab/GeoFormer) is pure Python/PyTorch and has no FFI; these entry
 * points replace the ATen call sites of model/full_model.py::GeoFormer.forward (SURVEY.md §2.2,
 * K2..K16).  Each function cites the reference lines whose arithmetic it implements.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller (PyTorch) owns every buffer, including workspaces;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return 0 on success, a negative GF_ERR_* otherwise; never throws, never exits;
 *     gf_last_error() returns a thread-local message for the last failure;
 *   - token features are row-major [rows, C] fp32; index outputs are int64 where the reference
 *     returns int64 tensors.
 */
#ifndef GEOFORMER_B200_H_
#define GEOFORMER_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GF_ABI_VERSION 1

#define GF_OK 0
#define GF_ERR_ARG (-1)      /* invalid argument / unsupported shape */
#define GF_ERR_LAUNCH (-2)   /* CUDA launch or runtime error */
#define GF_ERR_DRIVER (-3)   /* driver entry point (cuTensorMapEncodeTiled) unavailable */
#define GF_ERR_DEVICE (-4)   /* not an sm_100 device */

/* epilogue flags for gf_linear_* (applied in this order):
 *   acc -> +bias[col] -> +rowbias[row / rowbias_group][col] -> activation -> LayerNorm -> +residual[row][col] */
#define GF_EPI_RELU 1        /* all columns */
#define GF_EPI_TANH 2        /* all columns */
#define GF_EPI_ELU1 4        /* elu(x)+1 on columns [0, act_cols) only */
#define GF_EPI_LN 8          /* LayerNorm over the full row (requires N == 128 or 256), eps 1e-5 */

typedef void* gf_stream_t;

int gf_abi_version(void);
const char* gf_last_error(void);
/* Verifies that `device` is sm_100 and resolves the TMA descriptor encoder.  Does NOT change the calling thread's
 * current device: every launch goes to the current device of the calling thread, which must own `stream` and the
 * buffers (per-device kernel attributes are set lazily on first launch per device). */
int gf_init(int device);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t gf_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Linear layers (nn.Linear call sites: loftr_module/transformer.py:49-58, geo_transformer/
 * transformer.py:52-64, fine_preprocess.py:60-72).
 *   Y[M,N] = epilogue( [A | A2][M, K1+K2] * W[N, K1+K2]^T )
 * A2/K2 implement `torch.cat([x, message], dim=2)` (transformer.py:57) without materialising it.
 * gf_linear_tf32: TMA -> tcgen05.mma kind::tf32 -> TMEM -> fused epilogue.  N % 128 == 0, K % 32 == 0.
 * gf_linear_ref : plain fp32 FFMA kernel with the same contract (accuracy reference / debugging).
 * m_dev (optional): device int32 holding the live row count (<= M); tiles beyond it are skipped.
 */
int gf_linear_tf32(const float* A, const float* A2, const float* W, float* Y, int64_t M, int N, int K1, int K2,
                   int epi, int act_cols, const float* bias, const float* rowbias, int rowbias_group,
                   const float* gamma, const float* beta, const float* residual, const int* m_dev,
                   gf_stream_t stream);
/* Same GEMM with fp16 storage on either side (tensor-core path only).  in_f16: A, A2 and W are fp16 (tcgen05 kind::f16,
 * K % 64 == 0), else fp32 (kind::tf32).  out_f16: Y is fp16 (lean epilogue: scale / bias / activation only), else fp32.
 * Used for the intermediates of a transformer layer that feed only MMAs or the linear-attention kernels (projected
 * Q/K/V, attention message, MLP hidden): these GEMMs are bound by their HBM streams, the residual stream stays fp32. */
int gf_linear_mixed(const void* A, const void* A2, const void* W, void* Y, int in_f16, int out_f16, int64_t M, int N,
                    int K1, int K2, int epi, int act_cols, const float* bias, const float* rowbias, int rowbias_group,
                    const float* gamma, const float* beta, const float* residual, const int* m_dev, gf_stream_t stream);
int gf_linear_ref(const float* A, const float* A2, const float* W, float* Y, int64_t M, int N, int K1, int K2,
                  int epi, int act_cols, const float* bias, const float* rowbias, int rowbias_group,
                  const float* gamma, const float* beta, const float* residual, const int* m_dev,
                  gf_stream_t stream);

/* Backbone 3x3 / stride 1 / pad 1 convolution with folded BatchNorm (resnet_fpn.py:32-40,70-82) as a tcgen05
 * implicit GEMM over NHWC fp16 (fp32 accumulation; outputs saturate at +-65504):  y = act(conv(x, wt) + bias (+ residual)).
 *   x [b,h,w,cin_p] fp16; wt [cout_p][9][cin_k] fp16 (tap-major, cin_k = cin_p rounded up to 64, zero padded);
 *   bias fp32 [cout_p]; residual (optional) and y [b,h,w,cout_p] fp16.  act: 0 none, 1 ReLU, 2 LeakyReLU(0.01). */
int gf_conv3x3_f16(const void* x, const void* wt, const float* bias, const void* residual, void* y, int batch, int h,
                    int w, int cin_p, int cout_p, int cin_k, int act, gf_stream_t stream);
/* Generalisation used for the rest of the backbone: ksize 3 (pad 1) or 1 (pad 0), stride 1 or 2 (the stride-2 entry
 * convolutions and 1x1 downsample / FPN lateral convolutions of resnet_fpn.py:18-29, 62-82).  h, w are the INPUT sizes;
 * y is [batch, (h-1)/stride+1, (w-1)/stride+1, cout_p].  wt: [cout_p][ksize*ksize][cin_k] fp16. */
int gf_conv_f16(const void* x, const void* wt, const float* bias, const void* residual, void* y, int batch, int h, int w,
                 int cin_p, int cout_p, int cin_k, int ksize, int stride, int act, gf_stream_t stream);

/* Backbone stem (resnet_fpn.py:58-60,102): 7x7 / stride 2 / pad 3 conv of the 1-channel fp32 image + folded BN +
 * ReLU -> NHWC fp16 [b, h/2, w/2, 128].  wperm = folded weights as [49 taps][128 channels] fp32. */
int gf_stem_conv7x7_f16(const float* img, const float* wperm, const float* bias, void* out, int batch, int h, int w,
                         gf_stream_t stream);
/* FPN top-down merge (resnet_fpn.py:108-115): out = lateral + bilinear(src -> h x w, align_corners=True); NHWC fp16 */
int gf_upsample_add_f16(const void* lateral, const void* src, void* out, int batch, int h, int w, int hs, int ws,
                         int c, gf_stream_t stream);
/* fp32 FFMA versions of the backbone operators for the accurate mode (golden-match parity runs): the same layers
 * (resnet_fpn.py:15-40, 58-118) on NHWC fp32, any channel count (the 1-channel 7x7 stem included).
 *   gf_conv_ref: ksize 1 / 3 / 7 (pad = ksize / 2), stride 1 / 2; x [b,h,w,cin]; wt [ksize*ksize][cin][cout] fp32 (BN
 *   folded); bias fp32 [cout] or null; residual / y [b,ho,wo,cout] with ho = (h + 2 pad - ksize) / stride + 1;
 *   act as gf_conv_f16.  gf_upsample_add_ref: as gf_upsample_add_f16 on fp32. */
int gf_conv_ref(const float* x, const float* wt, const float* bias, const float* residual, float* y, int batch, int h,
                int w, int cin, int cout, int ksize, int stride, int act, gf_stream_t stream);
int gf_upsample_add_ref(const float* lateral, const float* src, float* out, int batch, int h, int w, int hs, int ws,
                        int c, gf_stream_t stream);

/* out[n,l,c] = x[n,l,c] + pe[l,c]  (position_encoding.py:42 on the NHWC-flattened coarse map) */
int gf_add_posenc(const float* x, const float* pe, float* out, int n, int64_t l, int c, gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Linear attention (loftr_module/linear_attention.py:33-49).  Q and K arrive already mapped through
 * elu(x)+1 (fused into the projection epilogue).  Row strides (ldq/ldk/ldv, in floats) let the caller
 * point into a fused [rows, 3C] projection buffer.
 *   reduce: KV[n,h,d,v] = sum_s K[n,s,h,d] * (V[n,s,h,v] / S);  Ksum[n,h,d] = sum_s K[n,s,h,d]
 *           (two deterministic stages; `partial` is a workspace of gf_linattn_partial_floats())
 *   apply : out[n,l,h,v] = (sum_d Q[n,l,h,d] KV[n,h,d,v]) / (Q[n,l,h,:].Ksum[n,h,:] + 1e-6) * S
 */
int64_t gf_linattn_partial_floats(int n, int s, int heads, int dim);
int gf_linattn_reduce(const float* K, int ldk, const float* V, int ldv, int n, int s, int heads, int dim,
                      float* partial, float* KV, float* Ksum, gf_stream_t stream);
int gf_linattn_apply(const float* Q, int ldq, const float* KV, const float* Ksum, float* out, int n, int l, int s,
                     int heads, int dim, gf_stream_t stream);
/* Fine-level variant (25 tokens, 8 heads x 16, one CTA per match; both phases fused). src_offset lets
 * the cross layer pair match m of the query tensor with match m of the source tensor. */
int gf_linattn_window(const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv, float* out,
                      int64_t n_windows, int tokens, int heads, int dim, gf_stream_t stream);
/* fp16-storage variants: Q/K/V (written by gf_linear_mixed out_f16) and the message are fp16; KV, Ksum and all
 * arithmetic stay fp32.  gf_linattn_window_f16 needs 25-token windows and 8 heads of dim 16. */
int gf_linattn_reduce_f16(const void* K, int ldk, const void* V, int ldv, int n, int s, int heads, int dim,
                          float* partial, float* KV, float* Ksum, gf_stream_t stream);
int gf_linattn_apply_f16(const void* Q, int ldq, const float* KV, const float* Ksum, void* out, int n, int l, int s,
                         int heads, int dim, gf_stream_t stream);
int gf_linattn_window_f16(const void* Q, int ldq, const void* K, int ldk, const void* V, int ldv, void* out,
                          int64_t n_windows, int tokens, int heads, int dim, gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * LoFTR full attention (`attention: 'full'`, loftr_module/linear_attention.py:54-85):
 *   out[n,l,h,:] = softmax_s(Q[n,l,h,:] . K[n,s,h,:] / sqrt(dim)) V[n,s,h,:]
 * on the plain projections (no elu+1 map).  Row strides ldq/ldk/ldv in elements; the message is fp32 [rows, heads*dim].
 */
/* coarse level, fp32 FFMA (accurate mode): q rows [n*l], k / v rows [n*s]; dim 32 */
int gf_full_attention(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* out, int n, int l,
                      int s, int heads, int dim, gf_stream_t stream);
/* coarse level, tensor cores (fp16 operands, fp32 accumulate): gf_dense_kv_h16 lays the fp16 K / V rows [n*s]
 * (8 heads of dim 32, 16-byte rows) out as kg[heads][n][s_pad][dim] and vt[heads][n][dim][s_pad] (zero for keys >= s,
 * s_pad % 64 == 0) and sets key_cnt[n] = s; gf_full_attention_tc (dim 32) then runs the flash kernel of
 * gf_geo_self_attention_tc over all s keys, reading the fp16 query rows in place through ldq. */
int gf_dense_kv_h16(const void* k, int ldk, const void* v, int ldv, int n, int s, int heads, int dim, int s_pad, void* kg,
                    void* vt, int* key_cnt, gf_stream_t stream);
int gf_full_attention_tc(const void* q16, int ldq, const void* kg, const void* vt, const int* key_cnt, float* out, int n,
                         int l, int s, int heads, int dim, int s_pad, gf_stream_t stream);
/* fine level: windows of `tokens` (<= 32) rows attend to the paired window of the same index, heads x 16; one warp per
 * (window, head).  Q / K / V fp32 or (_f16) fp16; the message is fp32 either way. */
int gf_full_attention_window(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* out,
                             int64_t n_windows, int tokens, int heads, int dim, gf_stream_t stream);
int gf_full_attention_window_f16(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, float* out,
                                 int64_t n_windows, int tokens, int heads, int dim, gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Coarse matching (utils/coarse_matching.py:110-125 and 161-212).
 * Split-fp16 operands: x*scale = hi + lo (fp16 each); role 0 (left operand) packs [hi | hi | lo],
 * role 1 (right operand) packs [hi | lo | hi] so that one K=3C fp16 tensor-core GEMM evaluates
 * hi*hi + hi*lo + lo*hi with fp32 accumulation (max-abs error on the logits <= 1e-3).
 */
int gf_pack_split_f16(const float* x, void* out_f16, int64_t rows, int c, float scale, int role, gf_stream_t stream);
/* sim[n,l,s] = (A3[n,l,:] . B3[n,s,:]) * out_scale   — batched tcgen05 kind::f16 GEMM, K = c3 */
int gf_similarity_f16x3(const void* a3, const void* b3, float* sim, int n, int l, int s, int c3, float out_scale,
                        gf_stream_t stream);
/* sim from fp32 features with plain FFMA (accuracy reference) */
int gf_similarity_ref(const float* f0, const float* f1, float* sim, int n, int l, int s, int c, float in_scale,
                      float out_scale, gf_stream_t stream);
/* row (dim=2) and column (dim=1) soft-max statistics of sim: max and sum(exp(x-max)).  With a workspace of
 * gf_dual_softmax_workspace_floats() floats both are produced from ONE read of sim (tile partials + merge);
 * workspace == NULL selects the two-sweep kernels. */
int64_t gf_dual_softmax_workspace_floats(int n, int l, int s);
int gf_dual_softmax_stats(const float* sim, int n, int l, int s, float* row_max, float* row_sum, float* col_max,
                          float* col_sum, float* workspace, gf_stream_t stream);
/* conf = softmax(sim,1)*softmax(sim,2), written in place over sim; also emits per-row / per-column max of conf */
int gf_dual_softmax_conf(float* sim_conf, int n, int l, int s, const float* row_max, const float* row_sum,
                         const float* col_max, const float* col_sum, float* conf_row_max, float* conf_col_max,
                         gf_stream_t stream);
/* per-row / per-column max of an existing confidence matrix (used when conf comes from outside) */
int gf_conf_row_col_max(const float* conf, int n, int l, int s, float* conf_row_max, float* conf_col_max,
                        gf_stream_t stream);
/* mutual-nearest + threshold + border selection; match_j[n,l] = first j with
 * conf>thr && conf==rowmax && conf==colmax && in-border, else -1 (coarse_matching.py:161-188) */
int gf_mnn_select(const float* conf, int n, int l, int s, float thr, int border, int h0c, int w0c, int h1c, int w1c,
                  const float* conf_row_max, const float* conf_col_max, int* match_j, float* match_conf,
                  gf_stream_t stream);
/* Fused inference path of the whole coarse-matching stage: two tcgen05 passes over the packed operands (statistics,
 * then confidences + per-row / per-column bests), never materialising the L x S matrix; then the mutual / threshold /
 * border test on vectors.  Fills match_j / match_conf [n*l] exactly like gf_mnn_select (feed gf_compact_coarse),
 * including the reference's tie order (first j that is row maximum AND column maximum AND inside the border,
 * coarse_matching.py:176-188): rows whose maximum is attained more than once and whose smallest-j candidate is rejected
 * are re-scanned exactly by a third, normally empty, tensor pass (see sim_fused.cu).  The kernels run as 2-CTA clusters. */
int64_t gf_coarse_match_fused_workspace_bytes(int n, int l, int s);
int gf_coarse_match_fused(const void* a3, const void* b3, int n, int l, int s, int c3, float out_scale, float thr,
                          int border, int h0c, int w0c, int h1c, int w1c, void* workspace, int* match_j,
                          float* match_conf, gf_stream_t stream);
/* profiling hook: launch only tensor pass 0 (statistics) or 1 (confidences) of the fused path on a workspace that a
 * full gf_coarse_match_fused call has already populated */
int gf_coarse_match_fused_pass(const void* a3, const void* b3, int n, int l, int s, int c3, float out_scale,
                               void* workspace, int pass, gf_stream_t stream);
/* ordered compaction (row-major (b,i), as torch.where) into the reference's output tensors
 * (coarse_matching.py:186-210).  counts[n] per sample, total[1]; capacity = max rows of the outputs. */
int gf_compact_coarse(const int* match_j, const float* match_conf, int n, int l, int w0c, int w1c, float scale,
                      int64_t* b_ids, int64_t* i_ids, int64_t* j_ids, float* mconf, float* mkpts0_c, float* mkpts1_c,
                      int* counts, int* total, int64_t capacity, gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Geometrized attention (model/geo_module.py:51-94, utils/common_utils.py:65-91,166-181,
 * utils/homography.py:86-105, geo_transformer/transformer.py:111-139, geo_attention.py:72-100).
 */
/* window token table: for each grid token of the source image (w_src_c columns), project its pixel
 * centre with hmat[n] (row-major 3x3 fp32) and list the 25 tokens of the other image around it.
 * widx[n,l,25] = token index, or -1 when the window sample falls outside the other image or has_h[n]==0. */
int gf_geo_window_table(const float* hmat, const int* has_h, int n, int h_src_c, int w_src_c, int h_dst_px, int w_dst_px,
                        int w_dst_c, int scale, int window, int* widx, gf_stream_t stream);
/* self attention against anchor (RANSAC inlier) tokens: full softmax, heads x dim, scale 1/sqrt(dim).
 * q [n,l,*] rows with stride ldq; k/v rows of the same image with strides ldk/ldv, gathered through
 * anchor_idx[n, anchor_cap] (first anchor_cnt[n] entries valid).  anchor_cnt[n]==0 leaves out[n] untouched
 * by writing zeros and setting skipped[n]=1 (the caller keeps the layer input for such samples). */
int gf_geo_self_attention(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* out,
                          int n, int l, int heads, int dim, const int* anchor_idx, const int* anchor_cnt,
                          int anchor_cap, gf_stream_t stream);
/* Tensor-core path of the same self attention, as three steps over materialised per-head score blocks:
 *   gf_gather_anchor_kv   : kg[h][n][s_pad][dim] (K rows) and vt[h][n][dim][s_pad] (V rows, transposed), 0 beyond cnt
 *   gf_gemm_tf32_batched  : scores[h][n][l][s_pad] = Q_h Kg_h^T / sqrt(dim)   (tcgen05 kind::tf32)
 *   gf_masked_softmax_rows: row soft-max over the first anchor_cnt[n] entries, zeros beyond
 *   gf_gemm_tf32_batched  : out[:, h*dim:(h+1)*dim] = P_h Vt_h^T */
int gf_gather_anchor_kv(const float* k, int ldk, const float* v, int ldv, int n, int l, int heads, int dim,
                        const int* anchor_idx, const int* anchor_cnt, int anchor_cap, int s_pad, float* kg, float* vt,
                        gf_stream_t stream);
int gf_masked_softmax_rows(float* x, int heads, int n, int l, int s_pad, const int* cnt_per_sample, gf_stream_t stream);
/* Fused version of the three steps above: one tcgen05 kernel per call, 128 queries of one (sample, head) per CTA,
 * ONE pass over 64-key tiles (running reference maximum raised lazily, accumulator rescaled only then; Q and P are
 * tensor-memory operands, the row sums accumulate on the tensor core), scores never leave the SM.  Operands are
 * fp16 (kind::f16, fp32 accumulate) prepared by gf_gather_anchor_kv_f16: q16 [n*l, heads*dim] (converted query rows),
 * kg [heads][n][s_pad][dim], vt [heads][n][dim][s_pad] (zero beyond anchor_cnt[n]); s_pad % 64 == 0. */
int gf_gather_anchor_kv_f16(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, int n, int l,
                            int heads, int dim, const int* anchor_idx, const int* anchor_cnt, int anchor_cap, int s_pad,
                            void* q16, void* kg, void* vt, gf_stream_t stream);
/* same gather when K / V are already fp16 (Q|K|V written by gf_linear_mixed out_f16; 4 heads of dim 64): no query copy
 * is needed, gf_geo_self_attention_tc reads the query rows in place through ldq */
int gf_gather_anchor_kv_h16(const void* k, int ldk, const void* v, int ldv, int n, int l, int heads, int dim,
                            const int* anchor_idx, const int* anchor_cnt, int anchor_cap, int s_pad, void* kg, void* vt,
                            gf_stream_t stream);
int gf_geo_self_attention_tc(const void* q16, int ldq, const void* kg, const void* vt, float* out, int n, int l,
                             int heads, int dim, int s_pad, const int* anchor_cnt, gf_stream_t stream);
/* Y[b] = out_scale * A[b] (M x K, row stride lda) * B[b]^T (N x K, row stride ldb); strides in floats */
int gf_gemm_tf32_batched(const float* A, int64_t lda, int64_t a_batch_stride, const float* B, int64_t ldb,
                         int64_t b_batch_stride, float* Y, int64_t ldy, int64_t y_batch_stride, int M, int N, int K,
                         int batches, float out_scale, gf_stream_t stream);

/* cross attention: one query token against its 25-token window of the other image (projected K/V rows
 * kproj/vproj [n, s, heads*dim]); masked entries filled with -1e8, all-masked rows give 0. */
int gf_geo_cross_attention(const float* q, int ldq, const float* kproj, int ldk, const float* vproj, int ldv,
                           float* out, int n, int l, int s, int heads, int dim, const int* widx, int window2,
                           gf_stream_t stream);
/* fp16-storage variant (Q|K|V from gf_linear_mixed out_f16; the message is fp16 and feeds the fp16-operand merge) */
int gf_geo_cross_attention_f16(const void* q, int ldq, const void* kproj, int ldk, const void* vproj, int ldv, void* out,
                               int n, int l, int s, int heads, int dim, const int* widx, int window2, gf_stream_t stream);
/* rows of samples whose flag[n]==0 are restored from src (layers skipped per sample) */
int gf_select_rows(float* dst, const float* src, const int* flag, int n, int64_t l, int c, gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Fine level (loftr_module/fine_preprocess.py:41-72, model/fine_matching2.py:52-126).
 */
/* One whole LoFTR encoder layer of the fine level (loftr_module/transformer.py:28-60 + linear_attention.py:33-49) as
 * one persistent tcgen05 kernel: 25-token windows, d_model 128, 8 heads.  x/src [windows*25, 128] fp32 (src == x for a
 * 'self' layer), y likewise (must not alias x/src).  wpack: the layer's weights as 30 operand blocks [30][128][128 B] in
 * streaming order (12 fp32 blocks Wq|Wk|Wv, 8 fp32 mlp.0[:, :128], 2 fp16 merge, 4 fp16 mlp.0[:, 128:], 4 fp16 mlp.2;
 * geoformer_b200/engine.py::pack_fine_layer).  Intermediates never leave the SM. */
int gf_fine_layer(const float* x, const float* src, const void* wpack, const float* gamma1, const float* beta1,
                  const float* gamma2, const float* beta2, float* y, int64_t windows, gf_stream_t stream);
/* 5x5 (stride 4, pad 2) windows of the NHWC fine map around coarse tokens: out[m, w*w, c] */
int gf_fine_gather(const float* fine_nhwc, int hf, int wf, int c, const int64_t* b_ids, const int64_t* tok_ids,
                   int64_t m, int wc, int stride, int window, float* out, gf_stream_t stream);
/* same, reading an fp16 NHWC fine map (native output of the tcgen05 backbone) */
int gf_fine_gather_f16(const void* fine_nhwc, int hf, int wf, int c, const int64_t* b_ids, const int64_t* tok_ids,
                        int64_t m, int wc, int stride, int window, float* out, gf_stream_t stream);
/* same, windows written as fp16 (a copy): A operand of the fp16 merge_feat GEMM */
int gf_fine_gather_f16_f16(const void* fine_nhwc, int hf, int wf, int c, const int64_t* b_ids, const int64_t* tok_ids,
                            int64_t m, int wc, int stride, int window, void* out, gf_stream_t stream);
/* rows out[m,:] = feat[b_ids[m], tok_ids[m], :] */
int gf_gather_rows(const float* feat, int64_t l, int c, const int64_t* b_ids, const int64_t* tok_ids, int64_t m,
                   float* out, gf_stream_t stream);
/* per match: 25x25 similarity, dual softmax, global arg-max, threshold.  sel[m] = 1 if kept;
 * fi/fj window cells; fconf confidence; optional fine_matrix [m,25,25]. */
int gf_fine_match(const float* f0, const float* f1, int64_t m, int ww, int c, float temperature, float thr,
                  int* sel, int* fi, int* fj, float* fconf, float* fine_matrix, gf_stream_t stream);
/* ordered compaction of kept fine matches into mkpts0_f/mkpts1_f/mconf/m_bids (fine_matching2.py:92-124) */
int gf_compact_fine(const int* sel, const int* fi, const int* fj, const float* fconf, const float* mkpts0_c,
                    const float* mkpts1_c, const int64_t* b_ids, int64_t m, int window, float coarse_scale,
                    float c2f_scale, float fine_scale, float* mkpts0_f, float* mkpts1_f, float* mconf,
                    int64_t* m_bids, int* total, gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Image ingest, the step before the path (eval_tool/immatch/utils/data_io.py:48-62): OpenCV's 8-bit INTER_LINEAR
 * cv2.resize reproduced bit-exactly + torchvision to_tensor (/255).  src: uint8 [ho, wo]; dst: fp32 [ht, wt].
 */
int gf_resize_gray_u8(const void* src, int ho, int wo, float* dst, int ht, int wt, gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Optional GPU RANSAC (replaces the host cv2.findHomography(kp0, kp1, cv2.RANSAC, 8.0) of model/geo_module.py:45-52
 * when GeoFormer.ransac == "gpu"; NOT bit-identical to OpenCV, so cv2 stays the default).  hyps % 8 == 0.
 * k0/k1 [m,2] fp32 first-pass coarse matches grouped by sample, counts[n] (device).  Outputs: hmat/hinv [n,9]
 * fp32 row-major, has_h[n] (0 when <= 8 matches or degenerate, geo_module.py:47), inlier[m], boolean token maps
 * map0 [n,l0] / map1 [n,l1] and the ascending anchor lists anchor_idx{0,1} [n,cap] + anchor_cnt{0,1}[n]
 * (all first-pass matches when has_h == 0, geo_module.py:76-88).
 */
int64_t gf_ransac_workspace_bytes(int n, int hyps);
int gf_ransac_homography(const float* k0, const float* k1, const int64_t* b_ids, const int* counts, int64_t m, int n,
                         int hyps, float thr, unsigned seed, int scale, int l0, int w0c, int l1, int w1c,
                         void* workspace, float* hmat, float* hinv, int* has_h, int* inlier, int* map0, int* map1,
                         int* anchor_idx0, int* anchor_cnt0, int* anchor_idx1, int* anchor_cnt1, int cap,
                         gf_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Optional padding masks data['mask0'] / data['mask1'] (zero-padded batches, model/full_model.py:79-83).  mask*: one
 * byte per token, 0 = padded (a torch.bool tensor as is).
 *   gf_mask_rows    : the `Q * q_mask`, `K * kv_mask`, `values * kv_mask` products of
 *                     loftr_module/linear_attention.py:37-43, in place on the projection buffer: for every row r with
 *                     mask[r] == 0 the elements buf[r*ld + col0 .. col0 + cols) are cleared (a product with a 0/1 mask).
 *                     elem_bytes 2 (fp16 storage) or 4 (fp32); ld, col0, cols in elements, each a multiple of 4 bytes.
 *   gf_mask_fill_sim: `sim_matrix.masked_fill_(~(mask_c0[..., None] * mask_c1[:, None]), -INF)` of
 *                     utils/coarse_matching.py:120-124, in place on sim [n, l, s] (fill = -1e9 in the reference),
 *                     between gf_similarity_* and gf_dual_softmax_stats.
 */
int gf_mask_rows(void* buf, int elem_bytes, int64_t rows, int64_t ld, int64_t col0, int64_t cols, const uint8_t* mask,
                 gf_stream_t stream);
int gf_mask_fill_sim(float* sim, int n, int l, int s, const uint8_t* mask0, const uint8_t* mask1, float fill,
                     gf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GEOFORMER_B200_H_ */
