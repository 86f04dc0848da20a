// Loss-head kernels after the encoder (SURVEY 8(f) rank 1): the masked-language-model cross-entropy of the pre-training task
// (reference: BertLMPredictionHead, external/pytorch_pretrained_bert/modeling.py:456-472; the loss itself
// pretrain/modules/resnet_vlbert_for_pretraining.py:165-189: F.cross_entropy(mlm_logits.view(-1, V), labels.view(-1),
// ignore_index=-1)).  The reference materialises logits for EVERY text position ([B*T, 30522] fp32 = 500 MB at config 2)
// although only the ~15 % labelled positions enter the loss.  Here the labelled rows are compacted on the device first
// (label_compact_kernel), the transform + decoder GEMMs run on those rows only (the library GEMM), and the cross-entropy is one
// pass over the bf16 logits (mlm_ce_forward_kernel: online log-sum-exp, label logit, arg-max for the accuracy metric) with the
// gradient written in place by mlm_ce_backward_kernel.
// The masked-region-classification loss of the same task (soft_cross_entropy, common/utils/misc.py:124-151, on the region
// classifier VisualLinguisticBertMVRCHead, common/visual_linguistic_bert.py:473-502) follows the same plan: its valid rows
// (target sum within 0.1 of 1) are found by soft_target_rows_kernel and compacted by label_compact_kernel, and the soft-target
// cross-entropy reads the fp32 targets in place (soft_ce_forward_kernel / soft_ce_backward_kernel).
#include "ops.cuh"

namespace vlb {

namespace {

// idx[k] = flat position of the k-th position whose label != ignore (k < cap), -1 beyond the count; count[0] = number found.
// One block: n is B*T (a few thousand).  Deterministic (ascending) order.
__global__ void __launch_bounds__(1024)
label_compact_kernel(const int64_t* __restrict__ labels, int n, int64_t ignore, int32_t* __restrict__ idx, int32_t* __restrict__ lab,
                     int cap, int32_t* __restrict__ count) {
  __shared__ int warp_tot[32];
  __shared__ int base_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) base_s = 0;
  __syncthreads();
  for (int start = 0; start < n; start += blockDim.x) {
    const int i = start + tid;
    const int64_t l = i < n ? labels[i] : ignore;
    const bool on = l != ignore;
    const unsigned m = __ballot_sync(0xffffffffu, on);
    const int before = __popc(m & ((1u << lane) - 1u));
    if (lane == 0) warp_tot[warp] = __popc(m);
    __syncthreads();
    int off = base_s;
    for (int w = 0; w < warp; ++w) off += warp_tot[w];
    if (on) {
      const int k = off + before;
      if (k < cap) { idx[k] = i; lab[k] = (int32_t)l; }
    }
    __syncthreads();
    if (tid == 0) {
      int t = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += warp_tot[w];
      base_s += t;
    }
    __syncthreads();
  }
  const int total = base_s;
  for (int k = total + tid; k < cap; k += blockDim.x) { idx[k] = -1; lab[k] = -1; }
  if (tid == 0) count[0] = total;
}

__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = red[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = fmaxf(r, red[w]);
  return r;
}
__device__ __forceinline__ float block_add(float v, float* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = 0.0f;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += red[w];
  return r;
}

// One block per compacted row: lse[row] = log sum_v exp(logit[row, v]) over v < V, picked[row] = logit[row, label],
// arg-max (first maximum) for the accuracy metric; loss_sum += lse - picked, correct += (argmax == label) over rows < count.
__global__ void __launch_bounds__(256)
mlm_ce_forward_kernel(const __nv_bfloat16* __restrict__ logits, int ld, int V, const int32_t* __restrict__ lab,
                      const int32_t* __restrict__ count, float* __restrict__ lse, float* __restrict__ loss_sum,
                      int32_t* __restrict__ correct) {
  __shared__ float red[8];
  __shared__ int redi[8];
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x;
  if (row >= count[0]) return;
  const __nv_bfloat16* __restrict__ lr = logits + (size_t)row * ld;
  const int nvec = V >> 3;
  float m = -INFINITY;
  int am = 0;
  for (int v = threadIdx.x; v < nvec; v += blockDim.x) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(lr + v * 8));
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a = bf16lo(w[j]), b = bf16hi(w[j]);
      if (a > m) { m = a; am = v * 8 + 2 * j; }
      if (b > m) { m = b; am = v * 8 + 2 * j + 1; }
    }
  }
  for (int c = (nvec << 3) + threadIdx.x; c < V; c += blockDim.x) {
    const float a = __bfloat162float(lr[c]);
    if (a > m) { m = a; am = c; }
  }
  const float gmax = block_max(m, red);
  // first index attaining the maximum (torch.argmax semantics on ties are unspecified; the smallest index is used here)
  int cand = (m == gmax) ? am : 0x7fffffff;
  for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) redi[threadIdx.x >> 5] = cand;
  __syncthreads();
  int best = redi[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = min(best, redi[w]);
  float s = 0.0f;
  for (int v = threadIdx.x; v < nvec; v += blockDim.x) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(lr + v * 8));
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) s += __expf(bf16lo(w[j]) - gmax) + __expf(bf16hi(w[j]) - gmax);
  }
  for (int c = (nvec << 3) + threadIdx.x; c < V; c += blockDim.x) s += __expf(__bfloat162float(lr[c]) - gmax);
  const float tot = block_add(s, red);
  if (threadIdx.x == 0) {
    const float l = gmax + __logf(tot);
    lse[row] = l;
    const int y = lab[row];
    const float picked = __bfloat162float(lr[y]);
    atomicAdd(loss_sum, l - picked);
    if (best == y) atomicAdd(correct, 1);
  }
}

// dlogits[row, v] = (exp(logit - lse[row]) - [v == label]) * gscale[0] / count   for rows < count, v < V; zero elsewhere
// (rows >= count and the padding columns V .. ld-1), written IN PLACE over the logits.
__global__ void __launch_bounds__(256)
mlm_ce_backward_kernel(__nv_bfloat16* __restrict__ logits, int ld, int V, const int32_t* __restrict__ lab,
                       const int32_t* __restrict__ count, const float* __restrict__ lse, const float* __restrict__ gscale) {
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x;
  const int n = count[0];
  __nv_bfloat16* __restrict__ lr = logits + (size_t)row * ld;
  const int nvec = ld >> 3;
  if (row >= n) {
    for (int v = threadIdx.x; v < nvec; v += blockDim.x) *reinterpret_cast<uint4*>(lr + v * 8) = make_uint4(0u, 0u, 0u, 0u);
    return;
  }
  const float l = lse[row];
  const float sc = gscale[0] / (float)n;
  const int y = lab[row];
  for (int v = threadIdx.x; v < nvec; v += blockDim.x) {
    const uint4 u = *reinterpret_cast<const uint4*>(lr + v * 8);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    float o[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      o[2 * j] = __expf(bf16lo(w[j]) - l);
      o[2 * j + 1] = __expf(bf16hi(w[j]) - l);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = v * 8 + j;
      o[j] = c < V ? (o[j] - (c == y ? 1.0f : 0.0f)) * sc : 0.0f;
    }
    uint4 pk;
    pk.x = pack_bf16x2(o[0], o[1]); pk.y = pack_bf16x2(o[2], o[3]);
    pk.z = pack_bf16x2(o[4], o[5]); pk.w = pack_bf16x2(o[6], o[7]);
    *reinterpret_cast<uint4*>(lr + v * 8) = pk;
  }
}

// ---- masked visual region classification (MVRC) ---------------------------------------------------------------------------
// soft_cross_entropy of common/utils/misc.py:124-151 on the regions whose fp32 target row sums to 1 +- 0.1.

__device__ __forceinline__ void argmax_step(float v, int c, float& m, int& am) {
  if (v > m) { m = v; am = c; }
}

// One warp per target row: arg[row] = first index of the row's maximum when |sum - 1| < 0.1, else -1 (the int64 label array
// label_compact_kernel takes, with ignore = -1).  Rows are C fp32 at stride ld_t and only 4-byte aligned (C = 1601): the
// unaligned head and the tail are read as scalars, the middle as float4.  Each lane sees its indices in ascending order, so
// its strict '>' keeps the first maximum; the lane merge takes the smallest index among equal maxima.
__global__ void __launch_bounds__(256)
soft_target_rows_kernel(const float* __restrict__ t, int n, int C, int ld_t, int64_t* __restrict__ arg) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const float* __restrict__ tr = t + (size_t)row * ld_t;
  const int head = min(C, (int)(((16u - (reinterpret_cast<uintptr_t>(tr) & 15u)) & 15u) >> 2));
  const int nvec = (C - head) >> 2;
  const int tail0 = head + (nvec << 2);
  float s = 0.0f, m = -INFINITY;
  int am = 0x7fffffff;
  if (lane < head) {
    const float v = __ldg(tr + lane);
    s += v;
    argmax_step(v, lane, m, am);
  }
  const float4* __restrict__ tv = reinterpret_cast<const float4*>(tr + head);
  for (int v = lane; v < nvec; v += 32) {
    const float4 q = __ldg(tv + v);
    const int c = head + (v << 2);
    s += (q.x + q.y) + (q.z + q.w);
    argmax_step(q.x, c, m, am);
    argmax_step(q.y, c + 1, m, am);
    argmax_step(q.z, c + 2, m, am);
    argmax_step(q.w, c + 3, m, am);
  }
  if (tail0 + lane < C) {
    const float v = __ldg(tr + tail0 + lane);
    s += v;
    argmax_step(v, tail0 + lane, m, am);
  }
  s = warp_sum(s);
  const float gm = warp_max(m);
  int cand = (m == gm) ? am : 0x7fffffff;
  for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
  if (lane == 0) arg[row] = fabsf(s - 1.0f) < 0.1f ? (int64_t)cand : (int64_t)-1;
}

// One block per compacted row < count: the bf16 logits row (ld, padding columns biased to -30000) and the fp32 target row
// targets[idx[row]] read in place.  lse[row] = log sum_c exp(x_c), row_loss[row] = S lse - sum_c t_c x_c
// (= -sum_c t_c log_softmax(x)_c, S = sum_c t_c), correct += (logit arg-max == lab[row]).  Rows >= count: row_loss = 0.
__global__ void __launch_bounds__(256)
soft_ce_forward_kernel(const __nv_bfloat16* __restrict__ logits, int ld, int C, const float* __restrict__ targets, int ld_t,
                       const int32_t* __restrict__ idx, const int32_t* __restrict__ lab, const int32_t* __restrict__ count,
                       float* __restrict__ lse, float* __restrict__ row_loss, int32_t* __restrict__ correct) {
  __shared__ float red[8];
  __shared__ int redi[8];
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x;
  if (row >= count[0]) {
    if (threadIdx.x == 0) { row_loss[row] = 0.0f; lse[row] = 0.0f; }
    return;
  }
  const __nv_bfloat16* __restrict__ lr = logits + (size_t)row * ld;
  const float* __restrict__ tr = targets + (size_t)idx[row] * ld_t;
  float m = -INFINITY, dot = 0.0f, s = 0.0f;
  int am = 0x7fffffff;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float x = __bfloat162float(lr[c]);
    const float tc = __ldg(tr + c);
    argmax_step(x, c, m, am);
    dot = fmaf(tc, x, dot);
    s += tc;
  }
  const float gmax = block_max(m, red);
  int cand = (m == gmax) ? am : 0x7fffffff;
  for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) redi[threadIdx.x >> 5] = cand;
  __syncthreads();
  int best = redi[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = min(best, redi[w]);
  float e = 0.0f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) e += __expf(__bfloat162float(lr[c]) - gmax);
  const float tot = block_add(e, red);
  const float dsum = block_add(dot, red);
  const float ssum = block_add(s, red);
  if (threadIdx.x == 0) {
    const float l = gmax + __logf(tot);
    lse[row] = l;
    row_loss[row] = ssum * l - dsum;
    if (best == lab[row]) atomicAdd(correct, 1);
  }
}

// IN PLACE over the logits: d[row, c] = (S exp(x_c - lse[row]) - t_c) * w[row] for rows < count, c < C, with S the row's own
// target sum (valid rows sum to anything in (0.9, 1.1)); 0 for rows >= count and the padding columns C .. ld-1.
__global__ void __launch_bounds__(256)
soft_ce_backward_kernel(__nv_bfloat16* __restrict__ logits, int ld, int C, const float* __restrict__ targets, int ld_t,
                        const int32_t* __restrict__ idx, const int32_t* __restrict__ count, const float* __restrict__ lse,
                        const float* __restrict__ w) {
  __shared__ float red[8];
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x;
  __nv_bfloat16* __restrict__ lr = logits + (size_t)row * ld;
  if (row >= count[0]) {
    const int nvec = ld >> 3;
    for (int v = threadIdx.x; v < nvec; v += blockDim.x) *reinterpret_cast<uint4*>(lr + v * 8) = make_uint4(0u, 0u, 0u, 0u);
    return;
  }
  const float* __restrict__ tr = targets + (size_t)idx[row] * ld_t;
  float s = 0.0f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s += __ldg(tr + c);
  const float S = block_add(s, red);
  const float l = lse[row], wr = w[row];
  for (int c = threadIdx.x; c < ld; c += blockDim.x) {
    float d = 0.0f;
    if (c < C) d = (S * __expf(__bfloat162float(lr[c]) - l) - __ldg(tr + c)) * wr;
    lr[c] = __float2bfloat16_rn(d);
  }
}

}  // namespace

int label_compact(const int64_t* labels, int n, int64_t ignore_index, int32_t* idx, int32_t* lab, int cap, int32_t* count,
                  cudaStream_t stream) {
  VLB_REQUIRE(labels && idx && lab && count && n > 0 && cap > 0, "label_compact: bad arguments");
  label_compact_kernel<<<1, 1024, 0, stream>>>(labels, n, ignore_index, idx, lab, cap, count);
  VLB_CHECK_LAUNCH();
  return VLB_OK;
}

int mlm_ce_forward(const void* logits, int ld, int V, const int32_t* lab, const int32_t* count, int rows, float* lse, float* loss_sum,
                   int32_t* correct, cudaStream_t stream) {
  VLB_REQUIRE(logits && lab && count && lse && loss_sum && correct && rows > 0 && V > 0 && ld >= V && ld % 8 == 0,
              "mlm_ce_forward: bad arguments");
  VLB_CHECK_CUDA(launch_pdl(mlm_ce_forward_kernel, dim3(rows), dim3(256), 0, stream, static_cast<const __nv_bfloat16*>(logits), ld, V, lab,
                            count, lse, loss_sum, correct));
  return VLB_OK;
}

int mlm_ce_backward(void* logits, int ld, int V, const int32_t* lab, const int32_t* count, int rows, const float* lse,
                    const float* gscale, cudaStream_t stream) {
  VLB_REQUIRE(logits && lab && count && lse && gscale && rows > 0 && V > 0 && ld >= V && ld % 8 == 0, "mlm_ce_backward: bad arguments");
  VLB_CHECK_CUDA(launch_pdl(mlm_ce_backward_kernel, dim3(rows), dim3(256), 0, stream, static_cast<__nv_bfloat16*>(logits), ld, V, lab, count,
                            lse, gscale));
  return VLB_OK;
}

int soft_target_rows(const float* targets, int n, int C, int ld_t, int64_t* arg, cudaStream_t stream) {
  VLB_REQUIRE(targets && arg && n > 0 && C > 0 && ld_t >= C, "soft_target_rows: bad arguments (n=%d C=%d ld_t=%d)", n, C, ld_t);
  VLB_CHECK_CUDA(launch_pdl(soft_target_rows_kernel, dim3((n + 7) / 8), dim3(256), 0, stream, targets, n, C, ld_t, arg));
  return VLB_OK;
}

int soft_ce_forward(const void* logits, int ld, int C, const float* targets, int ld_t, const int32_t* idx, const int32_t* lab,
                    const int32_t* count, int rows, float* lse, float* row_loss, int32_t* correct, cudaStream_t stream) {
  VLB_REQUIRE(logits && targets && idx && lab && count && lse && row_loss && correct && rows > 0 && C > 0 && ld >= C && ld % 8 == 0 &&
              ld_t >= C, "soft_ce_forward: bad arguments (rows=%d C=%d ld=%d ld_t=%d)", rows, C, ld, ld_t);
  VLB_CHECK_CUDA(launch_pdl(soft_ce_forward_kernel, dim3(rows), dim3(256), 0, stream, static_cast<const __nv_bfloat16*>(logits), ld, C,
                            targets, ld_t, idx, lab, count, lse, row_loss, correct));
  return VLB_OK;
}

int soft_ce_backward(void* logits, int ld, int C, const float* targets, int ld_t, const int32_t* idx, const int32_t* count, int rows,
                     const float* lse, const float* w, cudaStream_t stream) {
  VLB_REQUIRE(logits && targets && idx && count && lse && w && rows > 0 && C > 0 && ld >= C && ld % 8 == 0 && ld_t >= C,
              "soft_ce_backward: bad arguments (rows=%d C=%d ld=%d ld_t=%d)", rows, C, ld, ld_t);
  VLB_CHECK_CUDA(launch_pdl(soft_ce_backward_kernel, dim3(rows), dim3(256), 0, stream, static_cast<__nv_bfloat16*>(logits), ld, C,
                            targets, ld_t, idx, count, lse, w));
  return VLB_OK;
}

}  // namespace vlb
