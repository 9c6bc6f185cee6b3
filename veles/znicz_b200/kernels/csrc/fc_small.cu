// Fully connected layers with a handful of outputs (n_out <= 16: the 10-class softmax head of the
// CIFAR/MNIST nets, Wine's 3 classes, the 7-segment targets of Mnist7 ...).
//
// A 128x16 tcgen05 tile wastes > 90 % of the tensor-core tile for N = 10 and the generic SIMT GEMM
// is latency bound at 16 CTAs, so these shapes get two purpose-built kernels:
//
//   fc_small_forward_k   one CTA per batch row: dot products against all outputs, bias, activation
//                        and (for All2AllSoftmax) the row softmax + arg-max in the same launch
//                        (replaces GEMM + bias/activation + softmax_rows of the reference:
//                        /root/reference/all2all.py:236-255, cuda/all2all/softmax.cu)
//   fc_small_backward_k  one launch for the whole GD step of the layer
//                        (/root/reference/gd.py:506-549): err_output *= f'(y); err_input =
//                        alpha * err_output . W + beta * err_input; gradW partials (split over the
//                        batch, summed by the update kernel) and bias-gradient partials.
#include "common.cuh"

namespace zn {

constexpr int FCS_MAX_OUT = 16;

// Optional fused softmax evaluator (workflow/fusion.py::fuse_evaluator): the loss gradient
// err = (p - onehot) * mult, the error counters, the confusion matrix and max |err| row sum are
// produced by the warp that already holds the row's probabilities - the stand-alone
// evaluate_softmax launch (softmax_eval.cu, /root/reference/cuda/evaluator.jcu:21) disappears.
struct EvalArgs {
  const int* labels; void* err; int err_bf16; const float* bp;   // bp[0] = batch size, bp[1] = mult
  int* n_err; int* confusion; float* max_err_sum;
};

template <typename T>
__global__ void __launch_bounds__(128)
fc_small_forward_k(const T* __restrict__ x, const float* __restrict__ w,
                   const float* __restrict__ bias, T* __restrict__ out_t, float* __restrict__ out_f,
                   int* __restrict__ max_idx, int n_in, int n_out, int act, int softmax, EvalArgs ev) {
  pdl_wait();
  __shared__ float red[4][FCS_MAX_OUT];
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const T* xr = x + (size_t)row * n_in;
  float acc[FCS_MAX_OUT];
#pragma unroll
  for (int o = 0; o < FCS_MAX_OUT; ++o) acc[o] = 0.f;
  // rows >= n_out re-read the last valid row (result ignored): branch-free, all 16 loads of an
  // iteration are independent; 8 iterations are unrolled so that (for n_in <= 1024) every load of
  // the thread is in flight at once: one memory round trip instead of one per iteration
  const int last = n_out - 1;
#pragma unroll 8
  for (int k = tid; k < n_in; k += 128) {
    const float xv = ldf(xr + k);
#pragma unroll
    for (int o = 0; o < FCS_MAX_OUT; ++o)
      acc[o] = fmaf(xv, __ldg(w + (size_t)min(o, last) * n_in + k), acc[o]);
  }
#pragma unroll
  for (int o = 0; o < FCS_MAX_OUT; ++o) {
    if (o < n_out) {
      const float s = warp_sum(acc[o]);
      if (lane == 0) red[wid][o] = s;
    }
  }
  __syncthreads();
  if (wid != 0) return;
  float v = -3.0e38f;
  if (lane < n_out) {
    v = (red[0][lane] + red[1][lane]) + (red[2][lane] + red[3][lane]);
    if (bias) v += bias[lane];
    if (!softmax) v = act_fwd5(act, v);
  }
  if (softmax) {
    float m = v; int mi = lane < n_out ? lane : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float om = __shfl_xor_sync(0xffffffffu, m, o);
      const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
      if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
    }
    float e = lane < n_out ? __expf(v - m) : 0.f;
    const float s = warp_sum(e);
    v = e / s;
    if (lane == 0 && max_idx) max_idx[row] = mi;
    if (ev.labels) {
      const int batch = (int)ev.bp[0];
      const float mult = ev.bp[1];
      const int label = row < batch ? ev.labels[row] : -1;
      float d = 0.f;
      if (label >= 0 && lane < n_out) d = (v - (lane == label ? 1.f : 0.f)) * mult;
      if (lane < n_out) {
        if (ev.err_bf16) reinterpret_cast<__nv_bfloat16*>(ev.err)[(size_t)row * n_out + lane] = __float2bfloat16_rn(d);
        else reinterpret_cast<float*>(ev.err)[(size_t)row * n_out + lane] = d;
      }
      // |err| of the value as stored (the stand-alone kernel sums what it wrote in fp32)
      const float asum = warp_sum(fabsf(d));
      if (lane == 0 && label >= 0) {
        if (mi != label) atomicAdd(ev.n_err, 1);
        atomicAdd(ev.n_err + 1, 1);
        if (ev.confusion) atomicAdd(ev.confusion + (size_t)mi * n_out + label, 1);
        atomicMax(reinterpret_cast<int*>(ev.max_err_sum), __float_as_int(asum));   // asum >= 0
      }
    }
  }
  if (lane < n_out) {
    if (out_f) out_f[(size_t)row * n_out + lane] = v;
    if (out_t) stf(out_t + (size_t)row * n_out + lane, v);
  }
}

// grid = (ceil(n_in / 128), bsplit); thread = one input index k, a contiguous batch range.
template <typename T>
__global__ void __launch_bounds__(128)
fc_small_backward_k(const T* __restrict__ err, const T* __restrict__ y, const T* __restrict__ x,
                    const float* __restrict__ w, T* __restrict__ err_in,
                    float* __restrict__ gw_parts, float* __restrict__ gb_parts, int batch, int n_in,
                    int n_out, int act, float alpha, float beta, int need_ei, int need_gw) {
  pdl_wait();
  extern __shared__ float s_err[];       // [rows_here][FCS_MAX_OUT]
  const int bs = gridDim.y, part = blockIdx.y;
  const int per = (batch + bs - 1) / bs;
  const int b0 = part * per, b1 = min(batch, b0 + per);
  const int rows = max(0, b1 - b0);
  const int tid = threadIdx.x;
  // stage err_output * f'(y) of this batch range
  for (int i = tid; i < rows * FCS_MAX_OUT; i += 128) {
    const int r = i / FCS_MAX_OUT, o = i - r * FCS_MAX_OUT;
    float e = 0.f;
    if (o < n_out) {
      const size_t idx = (size_t)(b0 + r) * n_out + o;
      e = ldf(err + idx);
      // err_output itself is left untouched (the reference scales it in place, but nothing
      // downstream reads it and an in-place write would race with the other CTAs' reads)
      if (act != ACT_LINEAR) e *= act_deriv(act, 0.f, ldf(y + idx));
    }
    s_err[i] = e;
  }
  __syncthreads();
  if (gb_parts && blockIdx.x == 0 && tid < n_out) {   // bias gradient partial of this batch range
    float s = 0.f;
    for (int r = 0; r < rows; ++r) s += s_err[r * FCS_MAX_OUT + tid];
    gb_parts[(size_t)part * n_out + tid] = s;
  }
  const int k = blockIdx.x * 128 + tid;
  if (k >= n_in) return;
  float wv[FCS_MAX_OUT], g[FCS_MAX_OUT];
#pragma unroll
  for (int o = 0; o < FCS_MAX_OUT; ++o) {
    wv[o] = (need_ei && o < n_out) ? w[(size_t)o * n_in + k] : 0.f;
    g[o] = 0.f;
  }
#pragma unroll 4
  for (int r = 0; r < rows; ++r) {
    const float* e = s_err + r * FCS_MAX_OUT;
    const size_t xi = (size_t)(b0 + r) * n_in + k;
    if (need_gw) {
      const float xv = ldf(x + xi);
#pragma unroll
      for (int o = 0; o < FCS_MAX_OUT; ++o) g[o] = fmaf(e[o], xv, g[o]);
    }
    if (need_ei) {
      float s = 0.f;
#pragma unroll
      for (int o = 0; o < FCS_MAX_OUT; ++o) s = fmaf(e[o], wv[o], s);
      s *= alpha;
      if (beta != 0.f) s += beta * ldf(err_in + xi);
      stf(err_in + xi, s);
    }
  }
  if (need_gw) {
    float* gp = gw_parts + (size_t)part * n_out * n_in;
#pragma unroll
    for (int o = 0; o < FCS_MAX_OUT; ++o)
      if (o < n_out) gp[(size_t)o * n_in + k] = g[o];
  }
}

int fc_small_max_out() { return FCS_MAX_OUT; }

void launch_fc_small_forward(const void* x, bool bf16, const float* w, const float* bias, void* out_t,
                             float* out_f, int* max_idx, int batch, int n_in, int n_out, int act,
                             int softmax, const int* ev_labels, void* ev_err, int ev_err_bf16,
                             const float* ev_bp, int* ev_n_err, int* ev_confusion, float* ev_max_err,
                             cudaStream_t st) {
  EvalArgs ev{ev_labels, ev_err, ev_err_bf16, ev_bp, ev_n_err, ev_confusion, ev_max_err};
  if (bf16)
    launch_k(fc_small_forward_k<__nv_bfloat16>, batch, 128, 0, st, 
        (const __nv_bfloat16*)x, w, bias, (__nv_bfloat16*)out_t, out_f, max_idx, n_in, n_out, act, softmax, ev);
  else
    launch_k(fc_small_forward_k<float>, batch, 128, 0, st, (const float*)x, w, bias, (float*)out_t, out_f,
                                                     max_idx, n_in, n_out, act, softmax, ev);
}

void launch_fc_small_backward(void* err, const void* y, const void* x, bool bf16, const float* w,
                              void* err_in, float* gw_parts, float* gb_parts, int batch, int n_in,
                              int n_out, int act, float alpha, float beta, int bsplit, cudaStream_t st) {
  dim3 grid((n_in + 127) / 128, bsplit);
  const int per = (batch + bsplit - 1) / bsplit;
  const size_t smem = (size_t)per * FCS_MAX_OUT * sizeof(float);
  const int need_ei = err_in != nullptr, need_gw = gw_parts != nullptr;
  if (bf16)
    launch_k(fc_small_backward_k<__nv_bfloat16>, grid, 128, smem, st, 
        (const __nv_bfloat16*)err, (const __nv_bfloat16*)y, (const __nv_bfloat16*)x, w, (__nv_bfloat16*)err_in,
        gw_parts, gb_parts, batch, n_in, n_out, act, alpha, beta, need_ei, need_gw);
  else
    launch_k(fc_small_backward_k<float>, grid, 128, smem, st, (const float*)err, (const float*)y, (const float*)x, w,
                                                        (float*)err_in, gw_parts, gb_parts, batch, n_in,
                                                        n_out, act, alpha, beta, need_ei, need_gw);
}

}  // namespace zn
