/*
 * vlbert_b200 -- C ABI of the B200-native VL-BERT hot path (libvlbert_b200.so).
 *
 * Drop-in boundary for the path BASELINE.json's north_star names: the visual-linguistic transformer
 * encoder (reference: common/visual_linguistic_bert.py, external/pytorch_pretrained_bert/modeling.py)
 * and the region-feature front end (reference: common/fast_rcnn.py, common/lib/roi_pooling).
 *
 * Conventions (all entry points):
 *   - plain C: raw DEVICE pointers, sizes and leading dimensions in ELEMENTS; no torch types.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Work is only
 *     ENQUEUED on that stream; nothing synchronises and nothing is allocated behind the caller's
 *     back -- workspaces are passed in (the reference's native op enqueues on the current stream,
 *     common/lib/roi_pooling/cuda/ROIAlign_cuda.cu:273).
 *   - return value: 0 on success, negative on error (VLB_ERR_*); never throws.  The message of the
 *     last error on the calling thread is available from vlb_last_error_string() (the reference
 *     raises RuntimeError through AT_ASSERTM / THCudaCheck, ROIAlign_cuda.cu:262-264,297; the
 *     Python binding turns a negative return into the same RuntimeError).
 *   - "bf16" = __nv_bfloat16 storage, row-major; "f32" = float.
 *   - there is NO CPU fallback: every entry point needs an sm_100a device.
 */
#ifndef VLBERT_B200_H_
#define VLBERT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VLB_OK 0
#define VLB_ERR_INVALID (-1)
#define VLB_ERR_CUDA (-2)
#define VLB_ERR_UNSUPPORTED (-3)

/* ---- library ------------------------------------------------------------------------------- */
int vlb_abi_version(void);
const char* vlb_last_error_string(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t vlb_launch_count(void);
/* Size the persistent grids (GEMM, grouped wgrad) for `sms` SMs instead of the whole device (0 = all).  Used when a
 * concurrent NCCL collective owns some SMs: a persistent grid larger than the free SMs would run in two waves.
 * Environment default: VLB_SM_LIMIT. */
void vlb_set_sm_limit(int sms);
/* 1 if the experimental stream-K tail of the GEMM was compiled in (-DVLB_ENABLE_STREAMK=1; off by default: no gain measured). */
int vlb_streamk_compiled(void);

/* Per-launch device timing for bench.py's roofline.  While enabled, GEMM / attention / LayerNorm launchers bracket
 * their kernel with CUDA events on the launch stream.  vlb_profile_collect() waits for the recorded events and
 * returns, per category (0 gemm NT, 1 gemm NN, 2 gemm TN, 3 mhsa fwd, 4 mhsa bwd, 5 LN fwd, 6 LN bwd, 7 other, 8 im2col,
 * 9 col2im, 10 conv elementwise backward, 11 NHWC RoIAlign; arrays of VLB_PROFILE_CATEGORIES = 12), the summed
 * milliseconds, algorithmic work (FLOPs for 0-4, bytes for 5-6 and 8-11) and launch count, then resets. */
#define VLB_PROFILE_CATEGORIES 12
void vlb_profile_enable(int on);
int vlb_profile_collect(double* ms, double* work, int64_t* launches);

/* ---- dropout configuration of a fused call site ---------------------------------------------------
 * The reference applies nn.Dropout at six kinds of call sites of the path (modeling.py:283 embedding -- in VL-BERT
 * common/visual_linguistic_bert.py:75,239 --, :310 attention probabilities, :331 / :376 the two dense outputs of a layer,
 * common/fast_rcnn.py:106 obj_downsample input).  The fused kernels regenerate the keep-mask from a counter-based stream
 * (Philox4x32-10, see "dropout contract" below) instead of storing it: `rng` points to DEVICE memory holding
 * {uint64 seed, uint64 step}, read by the kernel when it RUNS (a CUDA-graph replay therefore sees the current step);
 * `site` numbers the call site.  p == 0 or a NULL VlbDropout* means no dropout (eval mode). */
typedef struct VlbDropout {
  float p;             /* drop probability, 0 <= p < 1 */
  uint32_t site;       /* call-site id (counter word 2) */
  const uint64_t* rng; /* device: {seed, step} */
  /* Optional (REQUIRED by the attention, GEMM-epilogue and LayerNorm-backward `out_drop` consumers): the keep flags of this
   * site as a device bit array written by vlb_dropout_bits from the same (p, site, rng): bit (c % 32) of word
   * r * ceil(cols / 32) + c / 32 = element (r, c) is kept.  Same mask as the inline evaluation; generated once, read by the
   * forward and the backward kernels (ten Philox rounds per four elements made the attention kernels instruction-bound). */
  const uint32_t* keep_bits;
} VlbDropout;

/* ---- GEMM (tcgen05) --------------------------------------------------------------------------
 * Replaces the torch.nn.Linear / F.linear calls of the encoder layer and their autograd backward
 * (modeling.py:291-293, :330, :362, :375; common/fast_rcnn.py:105-109 obj_downsample).
 *   mode 0 (NT): C[M,N] = A[M,K] B[N,K]^T   forward   y = x W^T
 *   mode 1 (NN): C[M,N] = A[M,K] B[K,N]     dgrad     dx = dy W
 *   mode 2 (TN): C[M,N] = A[K,M]^T B[K,N]   wgrad     dW = dy^T x
 * Epilogue: x = alpha*acc; x += bias[col]; activation; x += resid[row,col]; store.
 *   out_kind   0 bf16, 1 f32, 2 f32 atomic accumulate (required when split_k > 1)
 *   resid_kind 0 none, 1 bf16, 2 f32
 *   act        0 none, 1 erf-GELU (GELU'(pre-activation) stored to aux as bf16 if non-null, for backward), 2 ReLU,
 *              3 multiply by aux (the saved GELU'), 4 multiply by [aux > 0]
 *   force_bn   0 = the library picks the kernel and tile (always correct; every other value is a measurement aid and is
 *              rejected with VLB_ERR_INVALID when the shape does not allow it): 64 / 128 / 192 / 256 single-CTA tile width;
 *              1128 / 1256 cta_group::2 pairs of 256 rows; 2128 / 2256 two-CTA clusters with a multicast B tile;
 *              3192 / 3256 CTA pairs with 192-row tiles (NT / NN, N % width == 0); 4192 the 16-warp GELU epilogue (act 1).
 */
int vlb_gemm_bf16(int mode, int M, int N, int K, const void* A, int lda, const void* B, int ldb,
                  void* out, int ldo, int out_kind, const float* bias, const void* resid, int ldr,
                  int resid_kind, int act, void* aux, int ld_aux, float alpha, int split_k,
                  int force_bn, void* stream);
/* Same, with dropout applied to the [M,N] value after bias + activation and BEFORE the residual add
 * (BertSelfOutput / BertOutput: LayerNorm(dropout(dense(x)) + input), modeling.py:330-333,375-378). */
int vlb_gemm_bf16_dropout(int mode, int M, int N, int K, const void* A, int lda, const void* B, int ldb,
                          void* out, int ldo, int out_kind, const float* bias, const void* resid, int ldr,
                          int resid_kind, int act, void* aux, int ld_aux, float alpha, int split_k,
                          int force_bn, const VlbDropout* drop, void* stream);

/* Grouped weight-gradient GEMM: out_i[M_i,N_i] (+)= A_i[K,M_i]^T B_i[K,N_i], i < count <= 4, same K, ONE launch
 * (the four wgrad GEMMs of a BertLayer backward).  accumulate != 0: fp32 atomic "+=" (required for split_k > 1);
 * bn = 128 or 256 (tile width). */
typedef struct VlbGroupedProblem {
  int M, N;
  const void* A; int lda;
  const void* B; int ldb;
  float* out; int ldo;
} VlbGroupedProblem;
/* "dense + dropout + residual" of BertSelfOutput / BertOutput (modeling.py:329-333, :374-378) with the residual stream in fp32:
 *   out f32 [M,N] = dropout(A[M,K] W[N,K]^T + bias) + R,   R = resid->x_f32 (mean == NULL) or LayerNorm(resid->x_f32) recomputed
 * from its row statistics (see VlbResidual below).  drop may be NULL; otherwise drop->keep_bits is required. */
struct VlbResidual;
int vlb_gemm_bias_residual_f32(int M, int N, int K, const void* A, int lda, const void* W, int ldw, float* out, int ldo,
                               const float* bias, const struct VlbResidual* resid, const VlbDropout* drop, int force_bn,
                               void* stream);

int vlb_gemm_grouped_tn(int count, const VlbGroupedProblem* problems, int K, int split_k, int accumulate, int bn,
                        void* stream);

/* bring-up aid: override the MN-major shared-memory descriptor geometry (0 = default). */
void vlb_debug_gemm_desc(uint32_t mn_lbo, uint32_t mn_sbo, uint32_t mn_kadv);
/* timing aid (tools/gemm_trace.py): the CTA-pair GEMM kernel writes 8 %globaltimer stamps per CTA into buf
 * (device memory, >= 296 * 8 uint64); NULL switches it off. */
void vlb_debug_gemm_trace(void* buf);

/* ---- fused multi-head self-attention ---------------------------------------------------------
 * Replaces BertSelfAttention.forward after the three Linear layers (modeling.py:295-315):
 *   ctx[b*S+s, h*64:(h+1)*64] = softmax(q k^T / 8 + add_mask[b, :]) v        head size 64, S <= 256
 * (S <= 128: one tile per (batch, head); 128 < S <= 256: two query tiles x two key tiles, the backward then
 * accumulates partial dQ/dK/dV in scratch_f32 [B*S, 3H] (fp32, required only in that case) before converting).
 * qkv: bf16 [B*S, 3H] (q | k | v column blocks, the output of one fused QKV GEMM); add_mask: f32 [B,S]
 * additive (0 / -10000, common/visual_linguistic_bert.py:119-127) or NULL; ctx: bf16 [B*S, H];
 * lse: f32 [B, heads, S] log-sum-exp of the masked scaled scores (saved for backward; may be NULL
 * in forward-only use).  Backward writes dqkv bf16 [B*S, 3H] from dctx bf16 [B*S, H].
 */
int vlb_mhsa_forward(const void* qkv, const float* add_mask, void* ctx, float* lse, int B, int S, int H,
                     int heads, void* stream);
int vlb_mhsa_backward(const void* qkv, const float* add_mask, const void* ctx, const float* lse,
                      const void* dctx, void* dqkv, float* scratch_f32, int B, int S, int H, int heads,
                      void* stream);
/* With dropout on the attention probabilities (modeling.py:310): ctx = dropout(softmax(..)) v.  The mask is indexed as a
 * [B*heads*S, S] matrix (row = (b, head, query), column = key) under the 2-D contract below; lse is of the UNdropped
 * probabilities.  The backward must be given the same VlbDropout (and the same *rng contents) as the forward. */
int vlb_mhsa_forward_dropout(const void* qkv, const float* add_mask, void* ctx, float* lse, int B, int S, int H,
                             int heads, const VlbDropout* drop, void* stream);
/* dbias_qkv (optional, f32 [3H]): += column sums of dqkv = the bias gradients of the query / key / value Linear layers
 * (modeling.py:277-279), reduced inside the kernel's store phase instead of a separate pass over dqkv. */
int vlb_mhsa_backward_dropout(const void* qkv, const float* add_mask, const void* ctx, const float* lse,
                              const void* dctx, void* dqkv, float* scratch_f32, int B, int S, int H, int heads,
                              float* dbias_qkv, const VlbDropout* drop, void* stream);

/* ---- LayerNorm (TF style, eps inside the sqrt) -----------------------------------------------
 * Replaces BertLayerNorm.forward (modeling.py:231-235) and its autograd backward.
 * forward : x f32 [M, H] (row stride ldx) -> y bf16 and/or f32 [M, H]; mean / rstd f32 [M] (optional)
 * backward: dy = dy_bf16 (+ dy_f32), either may be NULL; dx to bf16 [M,H] and/or f32 (row stride ld_dx);
 *           dgamma / dbeta / dcolsum f32 [H] are ACCUMULATED (+=), each optional.
 *           dcolsum = sum over rows of dx = bias gradient of the Linear that produced x.
 */
int vlb_layernorm_forward(const float* x, int ldx, const float* gamma, const float* beta, void* y_bf16,
                          float* y_f32, float* mean, float* rstd, int M, int H, float eps, void* stream);
int vlb_layernorm_backward(const void* dy_bf16, const float* dy_f32, const float* x, int ldx,
                           const float* mean, const float* rstd, const float* gamma, void* dx_bf16,
                           float* dx_f32, int ld_dx, float* dgamma, float* dbeta, float* dcolsum, int M,
                           int H, void* stream);
/* LayerNorm followed by dropout on its output (the embedding: dropout(LayerNorm(e)), visual_linguistic_bert.py:237-239);
 * mask indexed over the [M, H] output. */
int vlb_layernorm_forward_dropout(const float* x, int ldx, const float* gamma, const float* beta, void* y_bf16,
                                  float* y_f32, float* mean, float* rstd, int M, int H, float eps,
                                  const VlbDropout* out_drop, void* stream);
/* Backward with the dropout sites either side of a LayerNorm:
 *   in_drop  : dy is first multiplied by the keep-mask / (1-p) of `in_drop`   (LayerNorm output was dropped: embedding)
 *   out_drop : a second bf16 output dx_bf16_drop = dx * keep-mask / (1-p) is written and dcolsum sums THAT tensor
 *              (LayerNorm input was dropout(dense(.)) + residual: the dense branch sees the masked gradient, the
 *              residual branch the plain dx).  Either may be NULL. */
int vlb_layernorm_backward_dropout(const void* dy_bf16, const float* dy_f32, const float* x, int ldx,
                                   const float* mean, const float* rstd, const float* gamma, void* dx_bf16,
                                   float* dx_f32, int ld_dx, float* dgamma, float* dbeta, float* dcolsum, int M,
                                   int H, const VlbDropout* in_drop, void* dx_bf16_drop, const VlbDropout* out_drop,
                                   void* stream);
/* out[n] += sum_m x[m, n]   (x bf16 [M, N], ld in elements) -- bias gradients */
int vlb_colsum_bf16(const void* x, int ld, float* out, int M, int N, void* stream);
int vlb_cast_f32_to_bf16(const float* in, void* out, int64_t n, void* stream);
int vlb_cast_bf16_to_f32(const void* in, float* out, int64_t n, void* stream);
/* Many casts/copies in one launch (the fp32 master weights -> bf16 operand copies of a whole encoder).
 * `descs_device` is a DEVICE array of `count` descriptors; src is f32, 16-byte aligned when bf16 dst. */
typedef struct VlbCastDesc {
  const void* src;     /* f32 */
  void* dst;           /* bf16 if dst_is_bf16 else f32 */
  int64_t n;           /* elements */
  int64_t dst_is_bf16;
} VlbCastDesc;
int vlb_multi_cast(const VlbCastDesc* descs_device, int count, int blocks_per_tensor, void* stream);

/* ---- embedding gather / sequence packing -----------------------------------------------------
 * Replaces VisualLinguisticBert.embedding (common/visual_linguistic_bert.py:173-241) index math and
 * gathers, and the output un-packing (:146-159).
 * vlb_pack_index: masks are uint8 [B,T] / [B,R]; S = caller's max_length (>= max_b(text_end+object_end)+1).
 *   kind/src/pos_id/type_id int32 [B,S]; add_mask f32 [B,S]; obj_row int32 [B,R]; lens int32 [B,2];
 *   err int32[1] is OR-ed with 1 (S too small), 2 (position id out of range), 4 (token id out of range), 8 (token type
 *   id outside 0..2); offending ids are remapped to row 0 so the kernels never read out of bounds -- the CALLER must check
 *   err (the reference raises an IndexError in these cases).
 *   pos_offset = position_padding_idx + 1.
 * vlb_pack_forward: e f32 [B*S, H] = vl + position_emb + token_type_emb (pre-LayerNorm sum).
 *   text_vis_ln f32 [B*T,H] / obj_vis_ln f32 [B*R,H] are the already LayerNorm-ed visual streams;
 *   object_vl f32 [B*R, ld_obj], its linguistic half starts at column lin_off.
 * vlb_pack_backward: scatters de f32 [B*S,H] into the embedding-table gradients (atomic +=, optional)
 *   and into dense d_text_vl [B*T,H] / d_obj_vl [B*R,H] (plain stores; caller zero-fills).
 */
int vlb_pack_index(const uint8_t* text_mask, const uint8_t* object_mask, const int64_t* text_type_ids,
                   int B, int T, int R, int S, int pos_offset, int32_t* kind, int32_t* src, int32_t* pos_id,
                   int32_t* type_id, float* add_mask, int32_t* obj_row, int32_t* lens, int32_t* err,
                   void* stream);
int vlb_pack_forward(const int32_t* kind, const int32_t* src, const int32_t* pos_id, const int32_t* type_id,
                     const int64_t* ids, const float* word_emb, const float* end_emb, const float* pos_emb,
                     const float* type_emb, const float* text_vis_ln, const float* obj_vis_ln,
                     const float* object_vl, int ld_obj, int lin_off, float* e, int B, int T, int R, int S,
                     int H, int vocab, int max_pos, int32_t* err, void* stream);
int vlb_pack_backward(const int32_t* kind, const int32_t* src, const int32_t* pos_id, const int32_t* type_id,
                      const int64_t* ids, const float* de, float* d_word, float* d_end, float* d_pos,
                      float* d_type, float* d_text_vl, float* d_obj_vl, int B, int T, int R, int S, int H,
                      int vocab, int max_pos, int pos_offset, void* stream);
/* out[i,:] = idx[i] >= 0 ? in[idx[i],:] : 0     /    out[idx[i],:] += in[i,:] (idx[i] >= 0, out f32) */
int vlb_gather_rows(const void* in, int in_is_bf16, int ld_in, const int32_t* idx, void* out, int out_is_bf16,
                    int ld_out, int n_out, int H, void* stream);
int vlb_scatter_rows_add(const void* in, int in_is_bf16, int ld_in, const int32_t* idx, float* out, int ld_out,
                         int n_in, int H, void* stream);

/* ---- RoIAlign ---------------------------------------------------------------------------------
 * Replaces the reference's only native extension, pybind11 module C_ROIPooling
 * (common/lib/roi_pooling/vision.cpp:6-11):
 *   roi_align_forward (Tensor input[N,C,H,W], Tensor rois[K,5], float spatial_scale, int pooled_h,
 *                      int pooled_w, int sampling_ratio) -> Tensor[K,C,ph,pw]        (ROIAlign.h:11-25)
 *   roi_align_backward(Tensor grad[K,C,ph,pw], rois, spatial_scale, ph, pw, batch_size, channels, height,
 *                      width, sampling_ratio) -> Tensor[N,C,H,W]                     (ROIAlign.h:27-45)
 * fp32, NCHW, contiguous (the reference forces .float() and .contiguous(), roi_align.py:69,
 * ROIAlign_cuda.cu:286,294).  K == 0 is a no-op (ROIAlign_cuda.cu:278-281).  Backward zero-fills grad_in.
 * roi_pool_* of the same module is dead code on the hot path (ROIPool is never instantiated,
 * common/fast_rcnn.py:10,66) and is not provided.
 */
int vlb_roi_align_forward(const float* input, const float* rois, float* out, int K, int C, int H, int W,
                          int pooled_h, int pooled_w, float spatial_scale, int sampling_ratio, void* stream);
int vlb_roi_align_backward(const float* grad_out, const float* rois, float* grad_in, int K, int N, int C, int H,
                           int W, int pooled_h, int pooled_w, float spatial_scale, int sampling_ratio,
                           void* stream);
/* Precomputed-feature path of FastRCNN.forward (common/fast_rcnn.py:140-142,170-174 + bbox.py:33-65):
 * builds the bf16 operand A [B*R, 2048 + feat_dim] = [coordinate embedding | feature] for the
 * obj_downsample GEMM (all-zero rows where box_mask == 0) and the pad_sequence gather index
 * (gather_idx int32 [B*R]: slot k of sample b <- k-th valid box, else -1).  boxes f32 [B*R, ld_box]
 * with (x1,y1,x2,y2,feat...); im_info f32 [B, ld_info] = (W, H, ...); mvrc_ops int64 [B*R] and
 * mask_visual_embed f32 [feat_dim] optional (NULL). */
int vlb_region_operand(const float* boxes, int ld_box, const uint8_t* box_mask, const float* im_info,
                       int ld_info, const int64_t* mvrc_ops, const float* mask_visual_embed, void* A,
                       int32_t* gather_idx, int B, int R, int feat_dim, void* stream);
/* Same with the Dropout(0.1) that heads obj_downsample (common/fast_rcnn.py:104-109) applied to A (mask indexed over the
 * [B*R, 2048 + feat_dim] slot layout; rows of invalid boxes stay zero). */
int vlb_region_operand_dropout(const float* boxes, int ld_box, const uint8_t* box_mask, const float* im_info,
                               int ld_info, const int64_t* mvrc_ops, const float* mask_visual_embed, void* A,
                               int32_t* gather_idx, int B, int R, int feat_dim, const VlbDropout* drop, void* stream);

/* ---- convolution front end (ResNet-101 C4 + res5 RoI head), NHWC bf16 ------------------------------
 * Replaces the nn.Conv2d / BatchNorm2d(eval, frozen) / ReLU / residual stack of Bottleneck.forward
 * (common/backbone/resnet/resnet.py:98-118) and the stem (:175-179): a convolution is lowered to vlb_conv_gemm (the
 * tcgen05 GEMM with the BN scale/shift, residual add and ReLU in its epilogue) on an im2col matrix; 1x1 stride-1
 * convolutions need no lowering.  col rows are output pixels (n, ho, wo), columns (r, s, c) tap-major, padded to Kp.
 */
int vlb_im2col_nhwc(const void* x_bf16, void* col_bf16, int N, int H, int W, int C, int kh, int kw, int stride,
                    int pad, int dil, int Ho, int Wo, int Kp, void* stream);
/* adjoint of im2col in gather form (no atomics): dx = col2im(dcol) (+ add, optional bf16 [N,H,W,C]) */
int vlb_col2im_nhwc(const void* dcol_bf16, const void* add_bf16, void* dx_bf16, int N, int H, int W, int C, int kh,
                    int kw, int stride, int pad, int dil, int Ho, int Wo, int Kp, void* stream);
/* y[P,Cout] = act(col[P,K] W[Cout,K]^T * scale[co] + shift[co] (+ resid[P,Cout])); relu_mode 0 none, 1 ReLU,
 * 2 ReLU after the residual add.  All matrices bf16 row-major; scale/shift f32 [Cout] (shift may be NULL). */
int vlb_conv_gemm(const void* col, int ld_col, const void* w, int ld_w, void* y, int P, int Cout, int K,
                  const float* scale, const float* shift, const void* resid, int relu_mode, void* stream);
/* Implicit-GEMM forms of the same convolution: the producer warp of the GEMM gathers the filter taps itself with TMA
 * im2col-mode loads from the NHWC tensor (no col matrix in HBM).  Needs C % 64 == 0; w is bf16 [Cout, kh*kw*C] tap-major.
 * vlb_conv_fprop also serves the data gradient of a stride-1 convolution: x := dY [N,Ho,Wo,Cout], w := the filter flipped
 * and transposed to [C, kh*kw*Cout], pad := dil*(k-1) - pad, scale = shift = NULL. */
typedef struct VlbConvGeom {
  int N, H, W, C;   /* input tensor, NHWC */
  int Ho, Wo;       /* output spatial size */
  int kh, kw, stride, pad, dil;
} VlbConvGeom;
int vlb_conv_fprop(const void* x, const VlbConvGeom* g, const void* w, int ld_w, void* y, int Cout, const float* scale,
                   const float* shift, const void* resid, int relu_mode, void* stream);
/* dw[Cout, kh*kw*C] (f32, ld_dw) += dy[P, Cout]^T im2col(x)[P, kh*kw*C]   (split_k > 1 splits the pixel reduction) */
int vlb_conv_wgrad(const void* x, const VlbConvGeom* g, const void* dy, int Cout, float* dw, int ld_dw, int split_k,
                   void* stream);
/* d_pre = (dy (+ dy2)) * [y_mask > 0] ; d_conv = d_pre * scale[c]  (either output may be NULL; y_mask NULL = no ReLU) */
int vlb_relu_bn_backward(const void* dy, const void* dy2, const void* y_mask, const float* scale, void* d_pre,
                         void* d_conv, int64_t rows, int C, void* stream);
int vlb_maxpool3x3s2_nhwc(const void* x, void* y, int N, int H, int W, int C, void* stream);
int vlb_avgpool_forward(const void* x_bf16, float* y, int K, int HW, int C, void* stream);
int vlb_avgpool_backward(const float* dy, void* dx_bf16, int K, int HW, int C, void* stream);
int vlb_nchw_f32_to_nhwc_bf16(const float* x, void* y, int N, int C, int H, int W, void* stream);
int vlb_nhwc_bf16_to_nchw_f32(const void* x, float* y, int N, int C, int H, int W, void* stream);
/* RoIAlign on an NHWC bf16 feature map [N,H,W,C] -> [K,ph,pw,C] bf16 (same sampling rules as vlb_roi_align_forward);
 * backward accumulates into grad_feat f32 [N,H,W,C] (zero-filled here). */
int vlb_roi_align_nhwc_forward(const void* feat, const float* rois, void* out, int K, int C, int H, int W, int ph,
                               int pw, float spatial_scale, int sampling_ratio, void* stream);
int vlb_roi_align_nhwc_backward(const void* grad_out, const float* rois, float* grad_feat, int K, int N, int C, int H,
                                int W, int ph, int pw, float spatial_scale, int sampling_ratio, void* stream);

/* ---- masked-language-model loss head (SURVEY 8(f) rank 1) ---------------------------------------------
 * Replaces, for the LOSS path, BertLMPredictionHead + F.cross_entropy(ignore_index=-1) of the pre-training task
 * (modeling.py:456-472; pretrain/modules/resnet_vlbert_for_pretraining.py:165-189).  The reference computes fp32 logits for
 * every text position ([B*T, 30522]) although only the labelled ~15 % enter the loss; here:
 *   vlb_label_compact : idx[k] = flat position of the k-th label != ignore_index (ascending), lab[k] = that label, k < cap;
 *                       -1 beyond the count; count[0] = number of labelled positions (device scalar, no host sync).
 *   (caller: gather those rows with vlb_gather_rows, transform + decoder GEMMs with vlb_gemm_bf16 on `cap` rows;
 *    the decoder's N is padded to a multiple of 8 with a bias of -30000 in the padding columns)
 *   vlb_mlm_ce_forward: per compacted row < count: lse[row] = log-sum-exp over the first V logits (bf16 [rows, ld]);
 *                       loss_sum[0] += lse - logit[label]; correct[0] += (argmax == label)   (accuracy metric of the trainer)
 *   vlb_mlm_ce_backward: overwrites the logits IN PLACE with d loss / d logits = (softmax - onehot) * gscale[0] / count
 *                       (rows >= count and padding columns: 0), ready to be the operand of the dgrad / wgrad GEMMs.
 */
int vlb_label_compact(const int64_t* labels, int n, int64_t ignore_index, int32_t* idx, int32_t* lab, int cap, int32_t* count,
                      void* stream);
int vlb_mlm_ce_forward(const void* logits_bf16, int ld, int V, const int32_t* lab, const int32_t* count, int rows, float* lse,
                       float* loss_sum, int32_t* correct, void* stream);
int vlb_mlm_ce_backward(void* logits_bf16, int ld, int V, const int32_t* lab, const int32_t* count, int rows, const float* lse,
                        const float* gscale, void* stream);

/* ---- masked visual region classification (MVRC) loss head ----------------------------------------------
 * Replaces, for the LOSS path, VisualLinguisticBertMVRCHead + soft_cross_entropy of the pre-training task
 * (common/visual_linguistic_bert.py:473-502; common/utils/misc.py:124-151; pretrain/modules/resnet_vlbert_for_pretraining.py:
 * 191-203).  A region row is valid when its fp32 soft target sums to 1 within 0.1; only those (~15 %) enter the loss.
 *   vlb_soft_target_rows: targets f32 [n, C] (row stride ld_t, rows only 4-byte aligned is fine): arg[row] (int64) = first
 *                       index of the row's maximum target if |sum - 1| < 0.1, else -1.  Feed arg to vlb_label_compact with
 *                       ignore_index = -1: idx = valid rows (ascending), lab = their target arg-max, count = their number.
 *   (caller: gather those rows with vlb_gather_rows; transform GEMM (+ bias + erf-GELU, act 1) and classifier GEMM with
 *    vlb_gemm_bf16 on `rows` rows into bf16 logits [rows, ld], ld = C padded to 8, padding columns biased to -30000)
 *   vlb_soft_ce_forward: per compacted row < count, reading targets[idx[row]] in place: lse[row] = log-sum-exp of the first
 *                       C logits; row_loss[row] = S lse - sum_c t_c x_c (= -sum_c t_c log_softmax(x)_c, S = sum_c t_c);
 *                       correct[0] += (logit arg-max == lab[row])  (what MVRCAccuracy counts).  Rows >= count: row_loss 0.
 *   vlb_soft_ce_backward: overwrites the logits IN PLACE with d loss / d logits = (S softmax(x) - t) * w[row], w = the
 *                       per-row DEVICE weight d loss / d row_loss (rows >= count and padding columns: 0).
 * No host synchronisation: count stays on the device.
 */
int vlb_soft_target_rows(const float* targets, int n, int C, int ld_t, int64_t* arg, void* stream);
int vlb_soft_ce_forward(const void* logits_bf16, int ld, int C, const float* targets, int ld_t, const int32_t* idx,
                        const int32_t* lab, const int32_t* count, int rows, float* lse, float* row_loss, int32_t* correct,
                        void* stream);
int vlb_soft_ce_backward(void* logits_bf16, int ld, int C, const float* targets, int ld_t, const int32_t* idx,
                         const int32_t* count, int rows, const float* lse, const float* w, void* stream);

/* ---- optimizer step after the path (SURVEY 8(f) rank 2) ---------------------------------------------
 * Replaces AdamW.step (common/nlp/bert/optimization.py:129-187: Adam moments, bias-corrected step size, decoupled weight decay
 * applied AFTER the update) and torch.nn.utils.clip_grad_norm_ of the trainer (common/trainer.py:139-147) for all parameter
 * tensors at once.  `descs_device` is a DEVICE array of `count` descriptors (fp32 tensors); `hyper_device` a DEVICE array
 * [count][4] f32 = (lr, lr * weight_decay, step_size, 0) per tensor for this step, 16-byte aligned.
 * vlb_grad_sqnorm writes sum(g^2) over all tensors to sq[0]; vlb_adamw_step scales every gradient by
 * min(1, max_norm / (sqrt(sq[0]) + 1e-6)) when sq != NULL and max_norm > 0 (gradients themselves are left untouched). */
typedef struct VlbAdamWTensor {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t n;
} VlbAdamWTensor;
int vlb_grad_sqnorm(const VlbAdamWTensor* descs_device, int count, float* sq, void* stream);
int vlb_adamw_step(const VlbAdamWTensor* descs_device, const float* hyper_device, int count, double beta1, double beta2,
                   double eps, const float* sq, float max_norm, void* stream);

/* ---- dropout contract -----------------------------------------------------------------------------
 * Counter-based masks (Philox4x32-10): element i of a row-major tensor is kept iff word (i % 4) of
 * philox(counter = (i/4 lo, i/4 hi, site, step), key = (seed lo, seed hi)) >= floor(p * 2^32); kept values are scaled by
 * 1/(1-p).  `site` numbers the nn.Dropout call sites of the reference (modeling.py:283,316,334,379,
 * common/visual_linguistic_bert.py:75, common/fast_rcnn.py:104), `step` the training step: forward and backward regenerate
 * the same mask, nothing is stored, and oracle/philox.py reproduces it on the CPU.  The reference's own masks come from
 * torch's global generator and cannot be reproduced by any implementation; this is the contract the fused kernels are
 * specified against.  vlb_dropout_mask writes the keep flags (uint8), vlb_dropout applies them to a bf16 / f32 tensor. */
int vlb_dropout_mask(uint8_t* keep, int64_t n, float p, uint64_t seed, uint32_t site, uint32_t step, void* stream);
/* 2-D form used by every fused site: element (r, c) of a [rows, cols] tensor belongs to Philox group
 * r * ceil(cols / 4) + c / 4, word c % 4 -- identical to the linear contract when cols % 4 == 0; rows of the attention
 * probabilities (cols = S keys) are padded to a multiple of four so that a row never shares a Philox call. */
int vlb_dropout_mask_2d(uint8_t* keep, int64_t rows, int cols, float p, uint64_t seed, uint32_t site, uint32_t step,
                        void* stream);
/* The same flags as a bit array for VlbDropout.keep_bits: bits uint32 [rows, ceil(cols / 32)], (seed, step) read from
 * drop->rng on the device.  vlb_dropout_bits_words(rows, cols) = number of uint32 words. */
int64_t vlb_dropout_bits_words(int64_t rows, int cols);
int vlb_dropout_bits(uint32_t* bits, int64_t rows, int cols, const VlbDropout* drop, void* stream);
/* y[r, c] = x[r, c] * keep(r, col_offset + c) / (1-p) for a [rows, cols] window (leading dimensions ldx / ldy, elements) of a tensor
 * whose mask is indexed over [rows, total_cols]; (seed, step) are read from drop->rng on the device.  cols, col_offset and
 * total_cols must be multiples of 4.  Stand-alone form of what the fused sites do (used for the gradient wrt the region
 * features behind obj_downsample's dropout and by the tests). */
int vlb_dropout_2d(const void* x, int ldx, void* y, int ldy, int64_t rows, int cols, int col_offset, int total_cols,
                   int is_bf16, const VlbDropout* drop, void* stream);
int vlb_dropout(const void* x, void* y, int64_t n, int is_bf16, float p, uint64_t seed, uint32_t site, uint32_t step, void* stream);

/* ---- one BertLayer, forward and backward -------------------------------------------------------
 * Replaces BertLayer.forward (modeling.py:388-397) = BertAttention + BertIntermediate + BertOutput and
 * its autograd backward, as a fixed sequence of the kernels above on `stream`
 * M = B*S rows.  ABI version 2: the trailing VlbLayerDropout* (same contents in forward and backward).
 */
typedef struct VlbLayerWeights {
  const void* w_qkv;   /* bf16 [3H, H]  rows: query | key | value weights (modeling.py:277-279) */
  const float* b_qkv;  /* f32 [3H] */
  const void* w_o;     /* bf16 [H, H]   attention.output.dense */
  const float* b_o;
  const float* ln1_g;  /* attention.output.LayerNorm */
  const float* ln1_b;
  const void* w_1;     /* bf16 [I, H]   intermediate.dense */
  const float* b_1;
  const void* w_2;     /* bf16 [H, I]   output.dense */
  const float* b_2;
  const float* ln2_g;  /* output.LayerNorm */
  const float* ln2_b;
} VlbLayerWeights;

typedef struct VlbLayerActs { /* saved activations of one layer, caller-allocated */
  void* qkv;       /* bf16 [M, 3H] */
  void* ctx;       /* bf16 [M, H]  */
  float* lse;      /* f32 [B, heads, S] */
  float* a;        /* f32 [M, H]   dense(ctx) + x, input of LayerNorm 1 */
  float* ln1_mean; /* f32 [M] */
  float* ln1_rstd;
  void* h;         /* bf16 [M, H]  attention output */
  void* z;         /* bf16 [M, I]  GELU'(pre-activation), saved for backward */
  void* u;         /* bf16 [M, I]  GELU output */
  float* y0;       /* f32 [M, H]   dense(u) + h, input of LayerNorm 2 */
  float* ln2_mean;
  float* ln2_rstd;
  void* y;         /* bf16 [M, H]  layer output */
  float* y_f32;    /* optional f32 copy of the layer output (NULL to skip) */
  /* dropout keep flags of the layer's three sites (VlbDropout.keep_bits layout), WRITTEN by the forward and read by the
   * backward; required where the corresponding probability is > 0, else NULL: */
  uint32_t* keep_attn;      /* [B*heads*S, ceil(S/32)] words */
  uint32_t* keep_self_out;  /* [M, ceil(H/32)] */
  uint32_t* keep_out;       /* [M, ceil(H/32)] */
} VlbLayerActs;

/* fp32 residual stream: the layer input x (bf16, the GEMM operand) described a second time for the residual add.
 * mean == NULL: x_f32 is x itself in fp32 [M, H] (the embedding output).  Otherwise x is the output of a LayerNorm that is
 * not stored in fp32: x_f32 is that LayerNorm's fp32 INPUT [M, H], mean / rstd [M] its row statistics and gamma / beta [H]
 * its parameters (for layer l > 0: acts(l-1).y0, ln2_mean, ln2_rstd, weights(l-1).ln2_g, ln2_b) -- the epilogue recomputes
 * the fp32 LayerNorm output instead of reading a stored copy. */
typedef struct VlbResidual {
  const float* x_f32;
  const float* mean;
  const float* rstd;
  const float* gamma;
  const float* beta;
} VlbResidual;

typedef struct VlbLayerGrads { /* f32, ACCUMULATED (+=); caller zero-fills or passes existing .grad */
  float* dw_qkv; float* db_qkv; float* dw_o; float* db_o; float* dln1_g; float* dln1_b;
  float* dw_1; float* db_1; float* dw_2; float* db_2; float* dln2_g; float* dln2_b;
} VlbLayerGrads;

/* Dropout of one BertLayer: attention probabilities (p_attn, modeling.py:310) and the two dense outputs (p_hidden,
 * :331 and :376).  NULL or both p == 0: the layer runs without dropout. */
typedef struct VlbLayerDropout {
  float p_attn;
  float p_hidden;
  uint32_t site_attn, site_self_out, site_out;   /* 1+3l, 2+3l, 3+3l for layer l */
  const uint64_t* rng;                           /* device: {seed, step} */
  /* 0: vlb_bert_layer_forward writes acts->keep_* itself (one extra launch at the head of the layer).  1: the caller has
   * already done so with vlb_layer_dropout_bits -- typically for all layers on a side stream at the start of the step, where
   * the instruction-bound Philox work overlaps the tensor-bound GEMMs instead of sitting in the layer's dependency chain. */
  int keep_bits_ready;
} VlbLayerDropout;

/* writes acts->keep_attn / keep_self_out / keep_out for one layer (the sites whose probability is > 0) */
int vlb_layer_dropout_bits(const VlbLayerActs* acts, int B, int S, int H, int heads, const VlbLayerDropout* drop, void* stream);

/* x_resid: NULL = the residual add uses x_bf16 (all-bf16 residual stream); else the fp32 residual stream (see VlbResidual). */
int vlb_bert_layer_forward(const VlbLayerWeights* w, const void* x_bf16, const VlbResidual* x_resid, const float* add_mask,
                           const VlbLayerActs* acts, int B, int S, int H, int heads, int I, float eps,
                           const VlbLayerDropout* drop, void* stream);
/* bytes of scratch vlb_bert_layer_backward needs */
int64_t vlb_bert_layer_backward_workspace(int M, int H, int I);
/* dy = dy_bf16 (+ dy_f32), either may be NULL.  dx_f32 == NULL: dx_bf16 [M, H] receives the whole gradient wrt x.
 * dx_f32 != NULL (fp32 residual stream): the gradient wrt x is dx_bf16 (the GEMM part) + dx_f32 (the residual part, fp32
 * [M, H]); hand both to the layer below as its dy_bf16 / dy_f32. */
int vlb_bert_layer_backward(const VlbLayerWeights* w, const VlbLayerActs* acts, const void* x_bf16,
                            const float* add_mask, const void* dy_bf16, const float* dy_f32, void* dx_bf16, float* dx_f32,
                            const VlbLayerGrads* grads, void* workspace, int64_t workspace_bytes, int B, int S,
                            int H, int heads, int I, const VlbLayerDropout* drop, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VLBERT_B200_H_ */
