// Row softmax (+argmax) and the evaluators (loss gradient + metrics).
// Parity: /root/reference/cuda/all2all/softmax.cu:14 (apply_exp), cuda/evaluator.jcu:21
// (evaluate_softmax), cuda/evaluator_mse.jcu:19, cuda/mse_find_closest.jcu:30.
// One warp per row, many CTAs (the reference evaluators are a single CTA and fill the
// confusion matrix serially on thread 0). Runtime batch size / multiplier come from a device
// scalar pair so the kernels can live in a captured CUDA graph.
#include "common.cuh"

namespace zn {

// in: logits [rows, cols] (bf16 or fp32, leading dim = cols); out: probabilities fp32
template <typename T>
__global__ void softmax_rows_k(const T* __restrict__ in, float* __restrict__ out,
                               int* __restrict__ max_idx, int rows, int cols) {
  pdl_wait();
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const T* r = in + (size_t)warp * cols;
  float m = -3.0e38f; int mi = 0;
  for (int c = lane; c < cols; c += 32) { float v = ldf(r + c); if (v > m) { m = v; mi = c; } }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float om = __shfl_xor_sync(0xffffffffu, m, o); int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
  }
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += __expf(ldf(r + c) - m);
  s = warp_sum(s);
  float inv = 1.f / s;
  float* o = out + (size_t)warp * cols;
  for (int c = lane; c < cols; c += 32) o[c] = __expf(ldf(r + c) - m) * inv;
  if (lane == 0) max_idx[warp] = mi;
}

// bp[0] = batch size (as float), bp[1] = multiplier
template <typename TE>
__global__ void evaluate_softmax_k(const float* __restrict__ y, const int* __restrict__ max_idx,
                                   const int* __restrict__ labels, TE* __restrict__ err,
                                   const float* __restrict__ bp, int rows, int cols,
                                   int* __restrict__ n_err, int* __restrict__ confusion,
                                   float* __restrict__ max_err_sum) {
  pdl_wait();
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  int batch = (int)bp[0]; float mult = bp[1];
  TE* e = err + (size_t)warp * cols;
  int label = warp < batch ? labels[warp] : -1;
  if (label < 0) {
    for (int c = lane; c < cols; c += 32) stf(e + c, 0.f);
    return;
  }
  const float* r = y + (size_t)warp * cols;
  float asum = 0.f;
  for (int c = lane; c < cols; c += 32) {
    float v = (r[c] - (c == label ? 1.f : 0.f)) * mult;
    stf(e + c, v);
    asum += fabsf(v);
  }
  asum = warp_sum(asum);
  if (lane == 0) {
    int mi = max_idx[warp];
    if (mi != label) atomicAdd(n_err, 1);
    atomicAdd(n_err + 1, 1);
    if (confusion) atomicAdd(confusion + (size_t)mi * cols + label, 1);
    atomicMax(reinterpret_cast<int*>(max_err_sum), __float_as_int(asum));  // asum >= 0
  }
}

template <typename TY, typename TE>
__global__ void evaluate_mse_k(const TY* __restrict__ y, const TY* __restrict__ target,
                               TE* __restrict__ err, const float* __restrict__ bp, int rows, int cols,
                               const float* __restrict__ denorm_mul, int root,
                               float* __restrict__ metrics, float* __restrict__ mse) {
  pdl_wait();
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  int batch = (int)bp[0]; float mult = bp[1];
  TE* e = err + (size_t)warp * cols;
  if (warp >= batch) {
    for (int c = lane; c < cols; c += 32) stf(e + c, 0.f);
    if (lane == 0) mse[warp] = 0.f;
    return;
  }
  const TY* r = y + (size_t)warp * cols;
  const TY* t = target + (size_t)warp * cols;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) {
    float d = ldf(r + c) - ldf(t + c);
    stf(e + c, d * mult);
    float dd = denorm_mul ? d * denorm_mul[c] : d;   // affine denormalisation: offsets cancel
    s += dd * dd;
  }
  s = warp_sum(s) / (float)cols;
  if (root) s = sqrtf(s);
  if (lane == 0) {
    mse[warp] = s;
    atomicAdd(metrics, s);
    atomicMax(reinterpret_cast<int*>(metrics + 1), __float_as_int(s));
    atomicMin(reinterpret_cast<int*>(metrics + 2), __float_as_int(s));
  }
}

// nearest class target (squared L2) vs label -> n_err
template <typename TY>
__global__ void mse_find_closest_k(const TY* __restrict__ y, const float* __restrict__ class_targets,
                                   const int* __restrict__ labels, const float* __restrict__ bp,
                                   int rows, int cols, int n_targets, int* __restrict__ n_err) {
  pdl_wait();
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows || warp >= (int)bp[0]) return;
  const TY* r = y + (size_t)warp * cols;
  float best = 3.0e38f; int bi = 0;
  for (int t = 0; t < n_targets; ++t) {
    const float* ct = class_targets + (size_t)t * cols;
    float s = 0.f;
    for (int c = lane; c < cols; c += 32) { float d = ldf(r + c) - ct[c]; s += d * d; }
    s = warp_sum(s);
    if (s < best) { best = s; bi = t; }
  }
  if (lane == 0) {
    if (bi != labels[warp]) atomicAdd(n_err, 1);
    atomicAdd(n_err + 1, 1);
  }
}

void launch_softmax_rows(const void* in, bool in_bf16, float* out, int* max_idx, int rows, int cols,
                         cudaStream_t st) {
  int grid = cdiv((long long)rows * 32, 128);
  if (in_bf16) launch_k(softmax_rows_k<__nv_bfloat16>, grid, 128, 0, st, (const __nv_bfloat16*)in, out, max_idx, rows, cols);
  else launch_k(softmax_rows_k<float>, grid, 128, 0, st, (const float*)in, out, max_idx, rows, cols);
}
void launch_evaluate_softmax(const float* y, const int* max_idx, const int* labels, void* err,
                             bool err_bf16, const float* bp, int rows, int cols, int* n_err,
                             int* confusion, float* max_err_sum, cudaStream_t st) {
  int grid = cdiv((long long)rows * 32, 128);
  if (err_bf16) launch_k(evaluate_softmax_k<__nv_bfloat16>, grid, 128, 0, st, y, max_idx, labels, (__nv_bfloat16*)err, bp, rows, cols, n_err, confusion, max_err_sum);
  else launch_k(evaluate_softmax_k<float>, grid, 128, 0, st, y, max_idx, labels, (float*)err, bp, rows, cols, n_err, confusion, max_err_sum);
}
void launch_evaluate_mse(const void* y, const void* target, bool y_bf16, void* err, bool err_bf16,
                         const float* bp, int rows, int cols, const float* denorm_mul, int root,
                         float* metrics, float* mse, cudaStream_t st) {
  int grid = cdiv((long long)rows * 32, 128);
  if (y_bf16) {
    if (err_bf16) launch_k(evaluate_mse_k<__nv_bfloat16, __nv_bfloat16>, grid, 128, 0, st, (const __nv_bfloat16*)y, (const __nv_bfloat16*)target, (__nv_bfloat16*)err, bp, rows, cols, denorm_mul, root, metrics, mse);
    else launch_k(evaluate_mse_k<__nv_bfloat16, float>, grid, 128, 0, st, (const __nv_bfloat16*)y, (const __nv_bfloat16*)target, (float*)err, bp, rows, cols, denorm_mul, root, metrics, mse);
  } else {
    if (err_bf16) launch_k(evaluate_mse_k<float, __nv_bfloat16>, grid, 128, 0, st, (const float*)y, (const float*)target, (__nv_bfloat16*)err, bp, rows, cols, denorm_mul, root, metrics, mse);
    else launch_k(evaluate_mse_k<float, float>, grid, 128, 0, st, (const float*)y, (const float*)target, (float*)err, bp, rows, cols, denorm_mul, root, metrics, mse);
  }
}
void launch_mse_find_closest(const void* y, bool y_bf16, const float* class_targets, const int* labels,
                             const float* bp, int rows, int cols, int n_targets, int* n_err,
                             cudaStream_t st) {
  int grid = cdiv((long long)rows * 32, 128);
  if (y_bf16) launch_k(mse_find_closest_k<__nv_bfloat16>, grid, 128, 0, st, (const __nv_bfloat16*)y, class_targets, labels, bp, rows, cols, n_targets, n_err);
  else launch_k(mse_find_closest_k<float>, grid, 128, 0, st, (const float*)y, class_targets, labels, bp, rows, cols, n_targets, n_err);
}

}  // namespace zn
