// Internal host-side declarations of the kernels' launchers (definitions in the .cu files).
#pragma once
#include "common.cuh"
#include "gemm_sm100.cuh"

namespace vlb {

void count_launch(int n);

// mhsa_sm100.cu
int mhsa_forward(const void* qkv, const float* add_mask, void* ctx, float* lse, int B, int S, int H, int heads,
                 cudaStream_t stream, const VlbDropout* drop = nullptr);
int mhsa_backward(const void* qkv, const float* add_mask, const void* ctx, const float* lse, const void* dctx, void* dqkv,
                  float* scratch_f32, int B, int S, int H, int heads, cudaStream_t stream, const VlbDropout* drop = nullptr,
                  float* dbias_qkv = nullptr);

// rowops.cu
int layernorm_forward(const float* x, int ldx, const float* gamma, const float* beta, void* y_bf16, float* y_f32, float* mean,
                      float* rstd, int M, int H, float eps, cudaStream_t stream, const VlbDropout* out_drop = nullptr);
int layernorm_backward(const void* dy_bf16, const float* dy_f32, const float* x, int ldx, const float* mean, const float* rstd,
                       const float* gamma, void* dx_bf16, float* dx_f32, int ld_dx, float* dgamma, float* dbeta, float* dcolsum,
                       int M, int H, cudaStream_t stream, const VlbDropout* in_drop = nullptr, void* dx_bf16_drop = nullptr,
                       const VlbDropout* out_drop = nullptr);
int colsum_bf16(const void* x, int ld, float* out, int M, int N, cudaStream_t stream);
int cast_f32_to_bf16(const float* in, void* out, size_t n, cudaStream_t stream);
int cast_bf16_to_f32(const void* in, float* out, size_t n, cudaStream_t stream);
int multi_cast(const VlbCastDesc* descs_device, int count, int blocks_per_tensor, cudaStream_t stream);

// embed.cu
int pack_index(const uint8_t* text_mask, const uint8_t* object_mask, const int64_t* text_type_ids, int B, int T, int R, int S,
               int pos_offset, int32_t* kind, int32_t* src, int32_t* pos_id, int32_t* type_id, float* add_mask,
               int32_t* obj_row, int32_t* lens, int32_t* err, cudaStream_t stream);
int pack_forward(const int32_t* kind, const int32_t* src, const int32_t* pos_id, const int32_t* type_id, const int64_t* ids,
                 const float* word_emb, const float* end_emb, const float* pos_emb, const float* type_emb,
                 const float* text_vis_ln, const float* obj_vis_ln, const float* object_vl, int ld_obj, int lin_off, float* e,
                 int B, int T, int R, int S, int H, int vocab, int max_pos, int32_t* err, cudaStream_t stream);
int pack_backward(const int32_t* kind, const int32_t* src, const int32_t* pos_id, const int32_t* type_id, const int64_t* ids,
                  const float* de, float* d_word, float* d_end, float* d_pos, float* d_type, float* d_text_vl, float* d_obj_vl,
                  int B, int T, int R, int S, int H, int vocab, int max_pos, int pos_offset, cudaStream_t stream);
int gather_rows(const void* in, int in_is_bf16, int ld_in, const int32_t* idx, void* out, int out_is_bf16, int ld_out, int n_out,
                int H, cudaStream_t stream);
int scatter_rows_add(const void* in, int in_is_bf16, int ld_in, const int32_t* idx, float* out, int ld_out, int n_in, int H,
                     cudaStream_t stream);

// roi_align.cu
int roi_align_forward(const float* input, const float* rois, float* out, int K, int C, int H, int W, int ph, int pw,
                      float spatial_scale, int sampling_ratio, cudaStream_t stream);
int roi_align_backward(const float* grad_out, const float* rois, float* grad_in, int K, int N, int C, int H, int W, int ph,
                       int pw, float spatial_scale, int sampling_ratio, cudaStream_t stream);
int region_operand(const float* boxes, int ld_box, const uint8_t* box_mask, const float* im_info, int ld_info,
                   const int64_t* mvrc_ops, const float* mask_visual_embed, void* A, int32_t* gather_idx, int B, int R,
                   int feat_dim, cudaStream_t stream, const VlbDropout* drop = nullptr);

// conv.cu
int im2col_nhwc(const void* x, void* col, int N, int H, int W, int C, int kh, int kw, int stride, int pad, int dil, int Ho, int Wo,
                int Kp, cudaStream_t stream);
int col2im_nhwc(const void* dcol, const void* add, void* dx, int N, int H, int W, int C, int kh, int kw, int stride, int pad, int dil,
                int Ho, int Wo, int Kp, cudaStream_t stream);
int relu_bn_backward(const void* dy, const void* dy2, const void* y_mask, const float* scale, void* d_pre, void* d_conv, int64_t rows,
                     int C, cudaStream_t stream);
int maxpool3x3s2_nhwc(const void* x, void* y, int N, int H, int W, int C, cudaStream_t stream);
int avgpool_forward(const void* x, float* y, int K, int HW, int C, cudaStream_t stream);
int avgpool_backward(const float* dy, void* dx, int K, int HW, int C, cudaStream_t stream);
int nchw_f32_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W, cudaStream_t stream);
int nhwc_bf16_to_nchw_f32(const void* x, float* y, int N, int C, int H, int W, cudaStream_t stream);
int roi_align_nhwc_forward(const void* feat, const float* rois, void* out, int K, int C, int H, int W, int ph, int pw, float scale,
                           int sampling_ratio, cudaStream_t stream);
int roi_align_nhwc_backward(const void* grad_out, const float* rois, float* grad_feat, int K, int N, int C, int H, int W, int ph, int pw,
                            float scale, int sampling_ratio, cudaStream_t stream);

// heads.cu
int label_compact(const int64_t* labels, int n, int64_t ignore_index, int32_t* idx, int32_t* lab, int cap, int32_t* count,
                  cudaStream_t stream);
int mlm_ce_forward(const void* logits, int ld, int V, const int32_t* lab, const int32_t* count, int rows, float* lse, float* loss_sum,
                   int32_t* correct, cudaStream_t stream);
int mlm_ce_backward(void* logits, int ld, int V, const int32_t* lab, const int32_t* count, int rows, const float* lse,
                    const float* gscale, cudaStream_t stream);
int soft_target_rows(const float* targets, int n, int C, int ld_t, int64_t* arg, cudaStream_t stream);
int soft_ce_forward(const void* logits, int ld, int C, const float* targets, int ld_t, const int32_t* idx, const int32_t* lab,
                    const int32_t* count, int rows, float* lse, float* row_loss, int32_t* correct, cudaStream_t stream);
int soft_ce_backward(void* logits, int ld, int C, const float* targets, int ld_t, const int32_t* idx, const int32_t* count, int rows,
                     const float* lse, const float* w, cudaStream_t stream);

int grad_sqnorm(const VlbAdamWTensor* descs_device, int count, float* sq, cudaStream_t stream);
int adamw_step(const VlbAdamWTensor* descs_device, const float* hyper_device, int count, double beta1, double beta2, double eps,
               const float* sq, float max_norm, cudaStream_t stream);

int dropout_mask(uint8_t* keep, int64_t n, float p, uint64_t seed, uint32_t site, uint32_t step, cudaStream_t stream);
int dropout_mask_2d(uint8_t* keep, int64_t rows, int cols, float p, uint64_t seed, uint32_t site, uint32_t step, cudaStream_t stream);
int64_t dropout_bits_words(int64_t rows, int cols);
int dropout_bits(uint32_t* bits, int64_t rows, int cols, const VlbDropout* drop, cudaStream_t stream);
int layer_dropout_bits(uint32_t* keep_attn, uint32_t* keep_self_out, uint32_t* keep_out, int B, int S, int H, int heads,
                       const VlbLayerDropout& d, cudaStream_t stream);
int dropout_2d(const void* x, int ldx, void* y, int ldy, int64_t rows, int cols, int col_offset, int total_cols, int is_bf16,
               const VlbDropout* drop, cudaStream_t stream);
int dropout_apply(const void* x, void* y, int64_t n, int is_bf16, float p, uint64_t seed, uint32_t site, uint32_t step, cudaStream_t stream);

}  // namespace vlb
