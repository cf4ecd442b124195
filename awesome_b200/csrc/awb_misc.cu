// Integer reductions around the fit loop: mask IoU counts for the in-loop "proper prior fit"
// check (MIOU(average="binary", invert=True), awesome/measures/miou.py:29-48 used at
// awesome/model/path_connected_net.py:964-982) and fg/bg pixel counts for the weighted
// losses (torch.unique(target >= 0.5, return_counts=True),
// awesome/measures/unaries_weighted_loss.py:38-40).  Exact integer arithmetic.
#include <math.h>

#include "awb_internal.cuh"

namespace awb {

__global__ void __launch_bounds__(256) k_iou_counts(const float* __restrict__ pred, const float* __restrict__ target,
                                                    int64_t N, int pred_is_logit, unsigned long long* counts) {
  int o = blockIdx.y;
  const float* p = pred + (int64_t)o * N;
  const float* t = target + (int64_t)o * N;
  unsigned inter = 0, pf = 0, tf = 0;
  for (int64_t n = (int64_t)blockIdx.x * 256 + threadIdx.x; n < N; n += (int64_t)gridDim.x * 256) {
    // foreground = (1 - mask) with mask = value > 0.5  <=>  value <= 0.5 ; sigmoid(y) > 0.5 <=> y > 0
    bool a = pred_is_logit ? !(p[n] > 0.f) : !(p[n] > 0.5f);
    bool b = !(t[n] > 0.5f);
    inter += (a && b); pf += a; tf += b;
  }
  __shared__ unsigned s[3][8];
  for (int off = 16; off > 0; off >>= 1) {
    inter += __shfl_xor_sync(0xffffffffu, inter, off);
    pf += __shfl_xor_sync(0xffffffffu, pf, off);
    tf += __shfl_xor_sync(0xffffffffu, tf, off);
  }
  int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { s[0][w] = inter; s[1][w] = pf; s[2][w] = tf; }
  __syncthreads();
  if (threadIdx.x < 3) {
    unsigned long long a = 0;
    for (int i = 0; i < 8; i++) a += s[threadIdx.x][i];
    atomicAdd(&counts[o * 4 + threadIdx.x], a);
  }
  if (threadIdx.x == 3 && blockIdx.x == 0) counts[o * 4 + 3] = (unsigned long long)N;
}

// IGN: pixels whose target equals ignore_value count in neither class (awb_target_counts_ignore)
template <bool IGN>
__global__ void __launch_bounds__(256) k_target_counts(const float* __restrict__ target, int64_t N, int cls_rule,
                                                       unsigned long long* counts, float ignore_value) {
  int o = blockIdx.y;
  const float* t = target + (int64_t)o * N;
  unsigned fg = 0, bg = 0;
  for (int64_t n = (int64_t)blockIdx.x * 256 + threadIdx.x; n < N; n += (int64_t)gridDim.x * 256) {
    if (IGN && t[n] == ignore_value) continue;
    bool f = cls_rule == AWB_CLS_UNARY_LT_HALF ? (t[n] < 0.5f) : (t[n] != 1.0f);
    fg += f; bg += !f;
  }
  __shared__ unsigned s[2][8];
  for (int off = 16; off > 0; off >>= 1) {
    fg += __shfl_xor_sync(0xffffffffu, fg, off);
    bg += __shfl_xor_sync(0xffffffffu, bg, off);
  }
  int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { s[0][w] = fg; s[1][w] = bg; }
  __syncthreads();
  if (threadIdx.x < 2) {
    unsigned long long a = 0;
    for (int i = 0; i < 8; i++) a += s[threadIdx.x][i];
    atomicAdd(&counts[o * 2 + threadIdx.x], a);
  }
}

}  // namespace awb

using namespace awb;

extern "C" {

int awb_mask_iou_counts(const float* pred, const float* target, int64_t N, int32_t O, int32_t pred_is_logit,
                        long long* counts, void* stream) {
  if (!pred || !target || !counts || N < 1 || O < 1) { set_error("bad argument"); return AWB_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  AWB_CUDA(cudaMemsetAsync(counts, 0, sizeof(long long) * 4 * O, st));
  int blocks = (int)((N + 255) / 256 < 592 ? (N + 255) / 256 : 592);
  k_iou_counts<<<dim3(blocks, O), 256, 0, st>>>(pred, target, N, pred_is_logit, (unsigned long long*)counts);
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int awb_target_counts(const float* target, int64_t N, int32_t O, int32_t cls_rule, long long* counts, void* stream) {
  if (!target || !counts || N < 1 || O < 1) { set_error("bad argument"); return AWB_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  AWB_CUDA(cudaMemsetAsync(counts, 0, sizeof(long long) * 2 * O, st));
  int blocks = (int)((N + 255) / 256 < 592 ? (N + 255) / 256 : 592);
  k_target_counts<false><<<dim3(blocks, O), 256, 0, st>>>(target, N, cls_rule, (unsigned long long*)counts, 0.f);
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

int awb_target_counts_ignore(const float* target, int64_t N, int32_t O, int32_t cls_rule, int32_t ignore_enabled,
                             float ignore_value, long long* counts, void* stream) {
  if (!target || !counts || N < 1 || O < 1) { set_error("bad argument"); return AWB_ERR_INVALID; }
  if (ignore_enabled && !isfinite(ignore_value)) { set_error("ignore_value must be finite"); return AWB_ERR_INVALID; }
  cudaStream_t st = (cudaStream_t)stream;
  AWB_CUDA(cudaMemsetAsync(counts, 0, sizeof(long long) * 2 * O, st));
  int blocks = (int)((N + 255) / 256 < 592 ? (N + 255) / 256 : 592);
  if (ignore_enabled)
    k_target_counts<true><<<dim3(blocks, O), 256, 0, st>>>(target, N, cls_rule, (unsigned long long*)counts, ignore_value);
  else
    k_target_counts<false><<<dim3(blocks, O), 256, 0, st>>>(target, N, cls_rule, (unsigned long long*)counts, 0.f);
  AWB_CUDA(cudaGetLastError());
  return AWB_OK;
}

}  // extern "C"
