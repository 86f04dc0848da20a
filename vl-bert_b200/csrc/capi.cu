// extern "C" entry points of libvlbert_b200.so (declared in include/vlbert_b200.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../include/vlbert_b200.h"
#include "common.cuh"
#include "gemm_sm100.cuh"
#include "ops.cuh"

namespace vlb {

namespace {
thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};
}  // namespace

void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_last_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  return VLB_ERR_CUDA;
}

static std::atomic<int> g_sm_limit{-1};
int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  int lim = g_sm_limit.load(std::memory_order_relaxed);
  if (lim < 0) {  // first call: environment default
    const char* v = getenv("VLB_SM_LIMIT");
    lim = v ? atoi(v) : 0;
    g_sm_limit.store(lim);
  }
  return (lim > 0 && lim < n) ? lim : n;
}

namespace {
struct ProfRec { cudaEvent_t a, b; int cat; double work; };
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
std::vector<cudaEvent_t> g_event_pool;
cudaEvent_t prof_event() {
  if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
}  // namespace

ProfScope::ProfScope(int cat, double work, cudaStream_t stream) : idx_(-1), stream_(stream) {
  if (!g_prof_on) return;
  ProfRec r; r.a = prof_event(); r.b = prof_event(); r.cat = cat; r.work = work;
  cudaEventRecord(r.a, stream);
  idx_ = (int)g_prof.size();
  g_prof.push_back(r);
}
ProfScope::~ProfScope() {
  if (idx_ >= 0) cudaEventRecord(g_prof[idx_].b, stream_);
}

bool pdl_enabled() {
  static const bool on = [] { const char* v = getenv("VLB_PDL"); return v ? atoi(v) != 0 : true; }();
  return on;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
void gemm_debug_override(uint32_t mn_lbo, uint32_t mn_sbo, uint32_t mn_kadv);
int bert_layer_forward(const VlbLayerWeights& w, const void* x, const VlbResidual* x_resid, const float* add_mask, const VlbLayerActs& a,
                       int B, int S, int H, int heads, int I, float eps, const VlbLayerDropout* drop, cudaStream_t st);
int64_t bert_layer_backward_workspace(int M, int H, int I);
int bert_layer_backward(const VlbLayerWeights& w, const VlbLayerActs& a, const void* x, const float* add_mask, const void* dy16,
                        const float* dy32, void* dx, float* dx_f32, const VlbLayerGrads& g, void* workspace, int64_t ws_bytes, int B, int S,
                        int H, int heads, int I, const VlbLayerDropout* drop, cudaStream_t st);

}  // namespace vlb

using namespace vlb;

extern "C" {

int vlb_abi_version(void) { return 2; }
int vlb_streamk_compiled(void) { return gemm_streamk_compiled() ? 1 : 0; }
void vlb_set_sm_limit(int sms) { g_sm_limit.store(sms > 0 ? sms : 0); }
const char* vlb_last_error_string(void) { return g_err; }
int64_t vlb_launch_count(void) { return g_launches.load(); }

int vlb_gemm_bf16(int mode, int M, int N, int K, const void* A, int lda, const void* B, int ldb, void* out,
                  int ldo, int out_kind, const float* bias, const void* resid, int ldr, int resid_kind, int act,
                  void* aux, int ld_aux, float alpha, int split_k, int force_bn, void* stream) {
  GemmEpilogue e;
  e.out = out; e.ldo = ldo; e.out_kind = out_kind;
  e.bias = bias;
  e.resid = resid; e.ldr = ldr; e.resid_kind = resid_kind;
  e.act = act; e.aux = aux; e.ld_aux = ld_aux; e.alpha = alpha;
  int rc = gemm_bf16(mode, M, N, K, A, lda, B, ldb, e, split_k, force_bn, static_cast<cudaStream_t>(stream));
  if (rc == VLB_OK) count_launch(1);
  return rc;
}

int vlb_gemm_bf16_dropout(int mode, int M, int N, int K, const void* A, int lda, const void* B, int ldb, void* out,
                          int ldo, int out_kind, const float* bias, const void* resid, int ldr, int resid_kind, int act,
                          void* aux, int ld_aux, float alpha, int split_k, int force_bn, const VlbDropout* drop, void* stream) {
  if (!drop_valid(drop)) { set_last_error("vlb_gemm_bf16_dropout: bad dropout configuration"); return VLB_ERR_INVALID; }
  GemmEpilogue e;
  e.out = out; e.ldo = ldo; e.out_kind = out_kind;
  e.bias = bias;
  e.resid = resid; e.ldr = ldr; e.resid_kind = resid_kind;
  e.act = act; e.aux = aux; e.ld_aux = ld_aux; e.alpha = alpha;
  e.drop = make_drop(drop);
  int rc = gemm_bf16(mode, M, N, K, A, lda, B, ldb, e, split_k, force_bn, static_cast<cudaStream_t>(stream));
  if (rc == VLB_OK) count_launch(1);
  return rc;
}

int vlb_gemm_bias_residual_f32(int M, int N, int K, const void* A, int lda, const void* W, int ldw, float* out, int ldo, const float* bias,
                               const VlbResidual* resid, const VlbDropout* drop, int force_bn, void* stream) {
  if (!resid || !resid->x_f32 || !drop_valid(drop)) { set_last_error("vlb_gemm_bias_residual_f32: bad residual / dropout arguments"); return VLB_ERR_INVALID; }
  GemmEpilogue e;
  e.out = out; e.ldo = ldo; e.out_kind = OUT_F32; e.bias = bias;
  e.resid = resid->x_f32; e.ldr = N; e.resid_kind = RESID_LN_F32;
  e.ln_mean = resid->mean; e.ln_rstd = resid->rstd; e.ln_gamma = resid->gamma; e.ln_beta = resid->beta;
  e.drop = make_drop(drop);
  int rc = gemm_bf16(GEMM_NT, M, N, K, A, lda, W, ldw, e, 1, force_bn, static_cast<cudaStream_t>(stream));
  if (rc == VLB_OK) count_launch(1);
  return rc;
}

int vlb_gemm_grouped_tn(int count, const VlbGroupedProblem* problems, int K, int split_k, int accumulate, int bn, void* stream) {
  if (count < 1 || count > 4 || !problems) { set_last_error("vlb_gemm_grouped_tn: bad arguments"); return VLB_ERR_INVALID; }
  GroupedProblem q[4];
  for (int i = 0; i < count; ++i) {
    q[i].M = problems[i].M; q[i].N = problems[i].N; q[i].A = problems[i].A; q[i].lda = problems[i].lda;
    q[i].B = problems[i].B; q[i].ldb = problems[i].ldb; q[i].out = problems[i].out; q[i].ldo = problems[i].ldo;
  }
  int rc = gemm_grouped_tn(count, q, K, split_k, accumulate != 0, bn, static_cast<cudaStream_t>(stream));
  if (rc == VLB_OK) count_launch(1);
  return rc;
}

void vlb_debug_gemm_desc(uint32_t mn_lbo, uint32_t mn_sbo, uint32_t mn_kadv) {
  gemm_debug_override(mn_lbo, mn_sbo, mn_kadv);
}

void vlb_debug_gemm_trace(void* buf) { gemm_debug_trace(static_cast<unsigned long long*>(buf)); }

void vlb_profile_enable(int on) { g_prof_on = on != 0; }
int vlb_profile_collect(double* ms, double* work, int64_t* launches) {
  for (int i = 0; i < PROF_NUM; ++i) { ms[i] = 0; work[i] = 0; launches[i] = 0; }
  for (auto& r : g_prof) {
    cudaError_t e = cudaEventSynchronize(r.b);
    if (e != cudaSuccess) return cuda_fail(e, "cudaEventSynchronize");
    float t = 0;
    e = cudaEventElapsedTime(&t, r.a, r.b);
    if (e != cudaSuccess) return cuda_fail(e, "cudaEventElapsedTime");
    ms[r.cat] += t; work[r.cat] += r.work; launches[r.cat] += 1;
    g_event_pool.push_back(r.a); g_event_pool.push_back(r.b);
  }
  g_prof.clear();
  return VLB_OK;
}

#define ST static_cast<cudaStream_t>(stream)
#define COUNTED(n, call) do { int _rc = (call); if (_rc == VLB_OK) count_launch(n); return _rc; } while (0)

int vlb_mhsa_forward(const void* qkv, const float* add_mask, void* ctx, float* lse, int B, int S, int H, int heads,
                     void* stream) {
  COUNTED(1, mhsa_forward(qkv, add_mask, ctx, lse, B, S, H, heads, ST));
}
int vlb_mhsa_backward(const void* qkv, const float* add_mask, const void* ctx, const float* lse, const void* dctx, void* dqkv,
                      float* scratch_f32, int B, int S, int H, int heads, void* stream) {
  COUNTED(1, mhsa_backward(qkv, add_mask, ctx, lse, dctx, dqkv, scratch_f32, B, S, H, heads, ST));
}
int vlb_mhsa_forward_dropout(const void* qkv, const float* add_mask, void* ctx, float* lse, int B, int S, int H, int heads,
                             const VlbDropout* drop, void* stream) {
  COUNTED(1, mhsa_forward(qkv, add_mask, ctx, lse, B, S, H, heads, ST, drop));
}
int vlb_mhsa_backward_dropout(const void* qkv, const float* add_mask, const void* ctx, const float* lse, const void* dctx,
                              void* dqkv, float* scratch_f32, int B, int S, int H, int heads, float* dbias_qkv, const VlbDropout* drop,
                              void* stream) {
  COUNTED(1, mhsa_backward(qkv, add_mask, ctx, lse, dctx, dqkv, scratch_f32, B, S, H, heads, ST, drop, dbias_qkv));
}
int vlb_layernorm_forward_dropout(const float* x, int ldx, const float* gamma, const float* beta, void* y_bf16, float* y_f32,
                                  float* mean, float* rstd, int M, int H, float eps, const VlbDropout* out_drop, void* stream) {
  COUNTED(1, layernorm_forward(x, ldx, gamma, beta, y_bf16, y_f32, mean, rstd, M, H, eps, ST, out_drop));
}
int vlb_layernorm_backward_dropout(const void* dy_bf16, const float* dy_f32, const float* x, int ldx, const float* mean,
                                   const float* rstd, const float* gamma, void* dx_bf16, float* dx_f32, int ld_dx, float* dgamma,
                                   float* dbeta, float* dcolsum, int M, int H, const VlbDropout* in_drop, void* dx_bf16_drop,
                                   const VlbDropout* out_drop, void* stream) {
  COUNTED(1, layernorm_backward(dy_bf16, dy_f32, x, ldx, mean, rstd, gamma, dx_bf16, dx_f32, ld_dx, dgamma, dbeta, dcolsum, M, H, ST,
                                in_drop, dx_bf16_drop, out_drop));
}
int vlb_layernorm_forward(const float* x, int ldx, const float* gamma, const float* beta, void* y_bf16, float* y_f32,
                          float* mean, float* rstd, int M, int H, float eps, void* stream) {
  COUNTED(1, layernorm_forward(x, ldx, gamma, beta, y_bf16, y_f32, mean, rstd, M, H, eps, ST));
}
int vlb_layernorm_backward(const void* dy_bf16, const float* dy_f32, const float* x, int ldx, const float* mean,
                           const float* rstd, const float* gamma, void* dx_bf16, float* dx_f32, int ld_dx, float* dgamma,
                           float* dbeta, float* dcolsum, int M, int H, void* stream) {
  COUNTED(1, layernorm_backward(dy_bf16, dy_f32, x, ldx, mean, rstd, gamma, dx_bf16, dx_f32, ld_dx, dgamma, dbeta, dcolsum, M, H, ST));
}
int vlb_colsum_bf16(const void* x, int ld, float* out, int M, int N, void* stream) {
  COUNTED(1, colsum_bf16(x, ld, out, M, N, ST));
}
int vlb_cast_f32_to_bf16(const float* in, void* out, int64_t n, void* stream) {
  COUNTED(1, cast_f32_to_bf16(in, out, (size_t)n, ST));
}
int vlb_cast_bf16_to_f32(const void* in, float* out, int64_t n, void* stream) {
  COUNTED(1, cast_bf16_to_f32(in, out, (size_t)n, ST));
}
int vlb_multi_cast(const VlbCastDesc* descs_device, int count, int blocks_per_tensor, void* stream) {
  COUNTED(1, multi_cast(descs_device, count, blocks_per_tensor, ST));
}
int vlb_pack_index(const uint8_t* text_mask, const uint8_t* object_mask, const int64_t* text_type_ids, int B, int T, int R,
                   int S, int pos_offset, int32_t* kind, int32_t* src, int32_t* pos_id, int32_t* type_id, float* add_mask,
                   int32_t* obj_row, int32_t* lens, int32_t* err, void* stream) {
  COUNTED(1, pack_index(text_mask, object_mask, text_type_ids, B, T, R, S, pos_offset, kind, src, pos_id, type_id, add_mask,
                        obj_row, lens, err, ST));
}
int vlb_pack_forward(const int32_t* kind, const int32_t* src, const int32_t* pos_id, const int32_t* type_id, const int64_t* ids,
                     const float* word_emb, const float* end_emb, const float* pos_emb, const float* type_emb,
                     const float* text_vis_ln, const float* obj_vis_ln, const float* object_vl, int ld_obj, int lin_off, float* e,
                     int B, int T, int R, int S, int H, int vocab, int max_pos, int32_t* err, void* stream) {
  COUNTED(1, pack_forward(kind, src, pos_id, type_id, ids, word_emb, end_emb, pos_emb, type_emb, text_vis_ln, obj_vis_ln,
                          object_vl, ld_obj, lin_off, e, B, T, R, S, H, vocab, max_pos, err, ST));
}
int vlb_pack_backward(const int32_t* kind, const int32_t* src, const int32_t* pos_id, const int32_t* type_id, const int64_t* ids,
                      const float* de, float* d_word, float* d_end, float* d_pos, float* d_type, float* d_text_vl,
                      float* d_obj_vl, int B, int T, int R, int S, int H, int vocab, int max_pos, int pos_offset, void* stream) {
  COUNTED(1, pack_backward(kind, src, pos_id, type_id, ids, de, d_word, d_end, d_pos, d_type, d_text_vl, d_obj_vl, B, T, R, S,
                           H, vocab, max_pos, pos_offset, ST));
}
int vlb_gather_rows(const void* in, int in_is_bf16, int ld_in, const int32_t* idx, void* out, int out_is_bf16, int ld_out,
                    int n_out, int H, void* stream) {
  COUNTED(1, gather_rows(in, in_is_bf16, ld_in, idx, out, out_is_bf16, ld_out, n_out, H, ST));
}
int vlb_scatter_rows_add(const void* in, int in_is_bf16, int ld_in, const int32_t* idx, float* out, int ld_out, int n_in, int H,
                         void* stream) {
  COUNTED(1, scatter_rows_add(in, in_is_bf16, ld_in, idx, out, ld_out, n_in, H, ST));
}
int vlb_roi_align_forward(const float* input, const float* rois, float* out, int K, int C, int H, int W, int pooled_h,
                          int pooled_w, float spatial_scale, int sampling_ratio, void* stream) {
  COUNTED(1, roi_align_forward(input, rois, out, K, C, H, W, pooled_h, pooled_w, spatial_scale, sampling_ratio, ST));
}
int vlb_roi_align_backward(const float* grad_out, const float* rois, float* grad_in, int K, int N, int C, int H, int W,
                           int pooled_h, int pooled_w, float spatial_scale, int sampling_ratio, void* stream) {
  COUNTED(1, roi_align_backward(grad_out, rois, grad_in, K, N, C, H, W, pooled_h, pooled_w, spatial_scale, sampling_ratio, ST));
}
int vlb_region_operand(const float* boxes, int ld_box, const uint8_t* box_mask, const float* im_info, int ld_info,
                       const int64_t* mvrc_ops, const float* mask_visual_embed, void* A, int32_t* gather_idx, int B, int R,
                       int feat_dim, void* stream) {
  COUNTED(2, region_operand(boxes, ld_box, box_mask, im_info, ld_info, mvrc_ops, mask_visual_embed, A, gather_idx, B, R,
                            feat_dim, ST));
}
int vlb_region_operand_dropout(const float* boxes, int ld_box, const uint8_t* box_mask, const float* im_info, int ld_info,
                               const int64_t* mvrc_ops, const float* mask_visual_embed, void* A, int32_t* gather_idx, int B, int R,
                               int feat_dim, const VlbDropout* drop, void* stream) {
  COUNTED(2, region_operand(boxes, ld_box, box_mask, im_info, ld_info, mvrc_ops, mask_visual_embed, A, gather_idx, B, R,
                            feat_dim, ST, drop));
}
int vlb_im2col_nhwc(const void* x, void* col, int N, int H, int W, int C, int kh, int kw, int stride, int pad, int dil, int Ho,
                    int Wo, int Kp, void* stream) {
  COUNTED(1, im2col_nhwc(x, col, N, H, W, C, kh, kw, stride, pad, dil, Ho, Wo, Kp, ST));
}
int vlb_col2im_nhwc(const void* dcol, const void* add, void* dx, int N, int H, int W, int C, int kh, int kw, int stride, int pad,
                    int dil, int Ho, int Wo, int Kp, void* stream) {
  COUNTED(1, col2im_nhwc(dcol, add, dx, N, H, W, C, kh, kw, stride, pad, dil, Ho, Wo, Kp, ST));
}
int vlb_conv_gemm(const void* col, int ld_col, const void* w, int ld_w, void* y, int P, int Cout, int K, const float* scale,
                  const float* shift, const void* resid, int relu_mode, void* stream) {
  GemmEpilogue e;
  e.out = y; e.ldo = Cout; e.out_kind = OUT_BF16;
  e.colscale = scale; e.bias = shift;
  if (resid) { e.resid = resid; e.ldr = Cout; e.resid_kind = RESID_BF16; }
  e.act = relu_mode == 1 ? ACT_RELU : (relu_mode == 2 ? ACT_RELU_POST : ACT_NONE);
  COUNTED(1, gemm_bf16(GEMM_NT, P, Cout, K, col, ld_col, w, ld_w, e, 1, 0, ST));
}
int vlb_label_compact(const int64_t* labels, int n, int64_t ignore_index, int32_t* idx, int32_t* lab, int cap, int32_t* count, void* stream) {
  COUNTED(1, label_compact(labels, n, ignore_index, idx, lab, cap, count, ST));
}
int vlb_mlm_ce_forward(const void* logits_bf16, int ld, int V, const int32_t* lab, const int32_t* count, int rows, float* lse,
                       float* loss_sum, int32_t* correct, void* stream) {
  COUNTED(1, mlm_ce_forward(logits_bf16, ld, V, lab, count, rows, lse, loss_sum, correct, ST));
}
int vlb_mlm_ce_backward(void* logits_bf16, int ld, int V, const int32_t* lab, const int32_t* count, int rows, const float* lse,
                        const float* gscale, void* stream) {
  COUNTED(1, mlm_ce_backward(logits_bf16, ld, V, lab, count, rows, lse, gscale, ST));
}
int vlb_soft_target_rows(const float* targets, int n, int C, int ld_t, int64_t* arg, void* stream) {
  COUNTED(1, soft_target_rows(targets, n, C, ld_t, arg, ST));
}
int vlb_soft_ce_forward(const void* logits_bf16, int ld, int C, const float* targets, int ld_t, const int32_t* idx,
                        const int32_t* lab, const int32_t* count, int rows, float* lse, float* row_loss, int32_t* correct,
                        void* stream) {
  COUNTED(1, soft_ce_forward(logits_bf16, ld, C, targets, ld_t, idx, lab, count, rows, lse, row_loss, correct, ST));
}
int vlb_soft_ce_backward(void* logits_bf16, int ld, int C, const float* targets, int ld_t, const int32_t* idx,
                         const int32_t* count, int rows, const float* lse, const float* w, void* stream) {
  COUNTED(1, soft_ce_backward(logits_bf16, ld, C, targets, ld_t, idx, count, rows, lse, w, ST));
}
int vlb_grad_sqnorm(const VlbAdamWTensor* descs_device, int count, float* sq, void* stream) {
  COUNTED(1, grad_sqnorm(descs_device, count, sq, ST));
}
int vlb_adamw_step(const VlbAdamWTensor* descs_device, const float* hyper_device, int count, double beta1, double beta2, double eps,
                   const float* sq, float max_norm, void* stream) {
  COUNTED(1, adamw_step(descs_device, hyper_device, count, beta1, beta2, eps, sq, max_norm, ST));
}
int vlb_dropout_mask(uint8_t* keep, int64_t n, float p, uint64_t seed, uint32_t site, uint32_t step, void* stream) {
  COUNTED(1, dropout_mask(keep, n, p, seed, site, step, ST));
}
int vlb_dropout_mask_2d(uint8_t* keep, int64_t rows, int cols, float p, uint64_t seed, uint32_t site, uint32_t step, void* stream) {
  COUNTED(1, dropout_mask_2d(keep, rows, cols, p, seed, site, step, ST));
}
int64_t vlb_dropout_bits_words(int64_t rows, int cols) { return dropout_bits_words(rows, cols); }
int vlb_dropout_bits(uint32_t* bits, int64_t rows, int cols, const VlbDropout* drop, void* stream) {
  COUNTED(1, dropout_bits(bits, rows, cols, drop, ST));
}
int vlb_dropout_2d(const void* x, int ldx, void* y, int ldy, int64_t rows, int cols, int col_offset, int total_cols, int is_bf16,
                   const VlbDropout* drop, void* stream) {
  COUNTED(1, dropout_2d(x, ldx, y, ldy, rows, cols, col_offset, total_cols, is_bf16, drop, ST));
}
int vlb_dropout(const void* x, void* y, int64_t n, int is_bf16, float p, uint64_t seed, uint32_t site, uint32_t step, void* stream) {
  COUNTED(1, dropout_apply(x, y, n, is_bf16, p, seed, site, step, ST));
}
static ConvGeom to_geom(const VlbConvGeom* g) {
  ConvGeom c{g->N, g->H, g->W, g->C, g->Ho, g->Wo, g->kh, g->kw, g->stride, g->pad, g->dil, g->kh * g->kw * g->C};
  return c;
}
static int check_geom(const VlbConvGeom* g) {
  if (!g || g->N < 1 || g->C < 1 || g->kh < 1 || g->kw < 1 || g->stride < 1 || g->dil < 1 || g->pad < 0 ||
      g->Ho != (g->H + 2 * g->pad - g->dil * (g->kh - 1) - 1) / g->stride + 1 ||
      g->Wo != (g->W + 2 * g->pad - g->dil * (g->kw - 1) - 1) / g->stride + 1) {
    set_last_error("conv: inconsistent geometry");
    return VLB_ERR_INVALID;
  }
  return VLB_OK;
}
int vlb_conv_fprop(const void* x, const VlbConvGeom* g, const void* w, int ld_w, void* y, int Cout, const float* scale,
                   const float* shift, const void* resid, int relu_mode, void* stream) {
  if (int rc = check_geom(g)) return rc;
  const ConvGeom cg = to_geom(g);
  GemmEpilogue e;
  e.out = y; e.ldo = Cout; e.out_kind = OUT_BF16;
  e.colscale = scale; e.bias = shift;
  if (resid) { e.resid = resid; e.ldr = Cout; e.resid_kind = RESID_BF16; }
  e.act = relu_mode == 1 ? ACT_RELU : (relu_mode == 2 ? ACT_RELU_POST : ACT_NONE);
  const long P = (long)g->N * g->Ho * g->Wo;
  COUNTED(1, gemm_bf16(GEMM_NT, (int)P, Cout, cg.Kp, x, cg.C, w, ld_w, e, 1, 0, ST, &cg, 1));
}
int vlb_conv_wgrad(const void* x, const VlbConvGeom* g, const void* dy, int Cout, float* dw, int ld_dw, int split_k, void* stream) {
  if (int rc = check_geom(g)) return rc;
  const ConvGeom cg = to_geom(g);
  GemmEpilogue e;
  e.out = dw; e.ldo = ld_dw; e.out_kind = OUT_F32_ATOMIC;
  const long P = (long)g->N * g->Ho * g->Wo;
  COUNTED(1, gemm_bf16(GEMM_TN, Cout, cg.Kp, (int)P, dy, Cout, x, cg.C, e, split_k, 0, ST, &cg, 2));
}
int vlb_relu_bn_backward(const void* dy, const void* dy2, const void* y_mask, const float* scale, void* d_pre, void* d_conv,
                         int64_t rows, int C, void* stream) {
  COUNTED(1, relu_bn_backward(dy, dy2, y_mask, scale, d_pre, d_conv, rows, C, ST));
}
int vlb_maxpool3x3s2_nhwc(const void* x, void* y, int N, int H, int W, int C, void* stream) {
  COUNTED(1, maxpool3x3s2_nhwc(x, y, N, H, W, C, ST));
}
int vlb_avgpool_forward(const void* x, float* y, int K, int HW, int C, void* stream) { COUNTED(1, avgpool_forward(x, y, K, HW, C, ST)); }
int vlb_avgpool_backward(const float* dy, void* dx, int K, int HW, int C, void* stream) { COUNTED(1, avgpool_backward(dy, dx, K, HW, C, ST)); }
int vlb_nchw_f32_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W, void* stream) {
  COUNTED(1, nchw_f32_to_nhwc_bf16(x, y, N, C, H, W, ST));
}
int vlb_nhwc_bf16_to_nchw_f32(const void* x, float* y, int N, int C, int H, int W, void* stream) {
  COUNTED(1, nhwc_bf16_to_nchw_f32(x, y, N, C, H, W, ST));
}
int vlb_roi_align_nhwc_forward(const void* feat, const float* rois, void* out, int K, int C, int H, int W, int ph, int pw,
                               float spatial_scale, int sampling_ratio, void* stream) {
  COUNTED(1, roi_align_nhwc_forward(feat, rois, out, K, C, H, W, ph, pw, spatial_scale, sampling_ratio, ST));
}
int vlb_roi_align_nhwc_backward(const void* grad_out, const float* rois, float* grad_feat, int K, int N, int C, int H, int W, int ph,
                                int pw, float spatial_scale, int sampling_ratio, void* stream) {
  COUNTED(1, roi_align_nhwc_backward(grad_out, rois, grad_feat, K, N, C, H, W, ph, pw, spatial_scale, sampling_ratio, ST));
}
int vlb_bert_layer_forward(const VlbLayerWeights* w, const void* x_bf16, const VlbResidual* x_resid, const float* add_mask,
                           const VlbLayerActs* acts, int B, int S, int H, int heads, int I, float eps, const VlbLayerDropout* drop,
                           void* stream) {
  if (!w || !acts || !x_bf16) { set_last_error("vlb_bert_layer_forward: null pointer"); return VLB_ERR_INVALID; }
  return bert_layer_forward(*w, x_bf16, x_resid, add_mask, *acts, B, S, H, heads, I, eps, drop, ST);
}
int vlb_layer_dropout_bits(const VlbLayerActs* acts, int B, int S, int H, int heads, const VlbLayerDropout* drop, void* stream) {
  if (!acts || !drop || !drop->rng) { set_last_error("vlb_layer_dropout_bits: null pointer"); return VLB_ERR_INVALID; }
  COUNTED(1, layer_dropout_bits(acts->keep_attn, acts->keep_self_out, acts->keep_out, B, S, H, heads, *drop, ST));
}
int64_t vlb_bert_layer_backward_workspace(int M, int H, int I) { return bert_layer_backward_workspace(M, H, I); }
int vlb_bert_layer_backward(const VlbLayerWeights* w, const VlbLayerActs* acts, const void* x_bf16, const float* add_mask,
                            const void* dy_bf16, const float* dy_f32, void* dx_bf16, float* dx_f32, const VlbLayerGrads* grads, void* workspace,
                            int64_t workspace_bytes, int B, int S, int H, int heads, int I, const VlbLayerDropout* drop,
                            void* stream) {
  if (!w || !acts || !x_bf16 || !grads || !workspace || !dx_bf16 || (!dy_bf16 && !dy_f32)) {
    set_last_error("vlb_bert_layer_backward: null pointer");
    return VLB_ERR_INVALID;
  }
  return bert_layer_backward(*w, *acts, x_bf16, add_mask, dy_bf16, dy_f32, dx_bf16, dx_f32, *grads, workspace, workspace_bytes, B, S, H,
                             heads, I, drop, ST);
}

}  // extern "C"
