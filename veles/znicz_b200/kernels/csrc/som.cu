// Kohonen self-organising map kernels — the reference has only OpenCL kernels for this op
// (/root/reference/ocl/kohonen.cl:19,59,139,161,182: calculate_distances, calculate_argmin,
// set_total, compute_gravity, apply_gradient); this is a CUDA design for sm_100a:
//   som_winners_k : one CTA per sample, warp-shuffle argmin of ||w_n - x||^2, winners histogram
//   som_update_k  : one thread per (neuron, feature); sums gravity * (x - w) over the batch and
//                   applies the step (batch semantics identical to the numpy oracle)
#include "common.cuh"

namespace zn {

__global__ void som_winners_k(const float* __restrict__ x, const float* __restrict__ w,
                              int* __restrict__ argmins, int* __restrict__ winners, int neurons,
                              int len, int count_winners) {
  pdl_wait();
  const int s = blockIdx.x;
  const float* xs = x + (size_t)s * len;
  float best = 3.0e38f; int bi = 0x7fffffff;
  for (int n = threadIdx.x; n < neurons; n += blockDim.x) {
    const float* wn = w + (size_t)n * len;
    float d = 0.f;
    for (int k = 0; k < len; ++k) { float t = wn[k] - xs[k]; d = fmaf(t, t, d); }
    if (d < best || (d == best && n < bi)) { best = d; bi = n; }
  }
  __shared__ float sb[32]; __shared__ int si[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ob = __shfl_xor_sync(0xffffffffu, best, o); int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) { sb[warp] = best; si[warp] = bi; }
  __syncthreads();
  if (warp == 0) {
    best = lane < nw ? sb[lane] : 3.0e38f; bi = lane < nw ? si[lane] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(0xffffffffu, best, o); int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    if (lane == 0) {
      argmins[s] = bi;
      if (count_winners) atomicAdd(winners + bi, 1);
    }
  }
}

__global__ void som_update_k(const float* __restrict__ x, float* __restrict__ w,
                             const float* __restrict__ coords, const int* __restrict__ argmins,
                             int batch, int neurons, int len, float sigma, float gmult) {
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= neurons * len) return;
  const int n = i / len, k = i - n * len;
  const float cx = coords[2 * n], cy = coords[2 * n + 1];
  const float inv = -1.f / (2.f * sigma * sigma);
  const float wv = w[i];
  float g = 0.f;
  for (int s = 0; s < batch; ++s) {
    const int win = argmins[s];
    const float dx = cx - coords[2 * win], dy = cy - coords[2 * win + 1];
    g += __expf((dx * dx + dy * dy) * inv) * (x[(size_t)s * len + k] - wv);
  }
  w[i] = wv + g * gmult;
}

// ------------------------------------------------------------------------------------------
// GEMM formulation (the reference's calculate_distances is its tiled matmul with a custom
// MULTIPLY, /root/reference/ocl/kohonen.cl:19-36). ||w_n - x_s||^2 = |x_s|^2 - 2 x_s.w_n + |w_n|^2,
// so the winners are argmin_n (|w_n|^2 - 2 x_s.w_n): one [batch x neurons x len] GEMM on the
// tcgen05 kernel. fp32 operands are split into bf16 hi + lo parts and the three significant
// products (hi*hi + hi*lo + lo*hi) are folded into ONE GEMM by concatenating along K:
//   A' = [x_hi | x_hi | x_lo],  B' = [w_hi | w_lo | w_hi]   (K' = 3 * roundup(len, 8))
// which keeps ~16 bits of every product - enough for the argmin to agree with the fp32 oracle
// except on numerical ties. The batch update  w += gm * (G.x - rowsum(G) o w)  is a second GEMM
// (K = batch) with the same trick (parts stacked along the rows of x).
// ------------------------------------------------------------------------------------------
// dst part p of element (row, k) lives at dst[p * part_stride + row * ld + k]; pattern 0 = the
// A-side order (hi, hi, lo), 1 = the B-side order (hi, lo, hi). Columns len..kp-1 are zeroed.
__global__ void som_split_k(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int rows,
                            int len, int kp, long long ld, long long part_stride, int pattern,
                            float* __restrict__ norm_out) {
  pdl_wait();
  const int row = blockIdx.x;
  if (row >= rows) return;
  const float* s = src + (size_t)row * len;
  float nrm = 0.f;
  for (int k = threadIdx.x; k < kp; k += blockDim.x) {
    const float v = k < len ? s[k] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    __nv_bfloat16* d = dst + (size_t)row * ld + k;
    d[0] = hi;
    d[part_stride] = pattern ? lo : hi;
    d[2 * part_stride] = pattern ? hi : lo;
    nrm = fmaf(v, v, nrm);
  }
  if (norm_out) {
    __shared__ float red[32];
    nrm = warp_sum(nrm);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = nrm;
    __syncthreads();
    if (threadIdx.x < 32) {
      float t = threadIdx.x < ((blockDim.x + 31) >> 5) ? red[threadIdx.x] : 0.f;
      t = warp_sum(t);
      if (threadIdx.x == 0) norm_out[row] = t;
    }
  }
}

// winners from the dot products: argmin_n (wnorm[n] - 2 dots[s][n]), ties -> lowest index
__global__ void som_argmin_k(const float* __restrict__ dots, const float* __restrict__ wnorm,
                             int* __restrict__ argmins, int* __restrict__ winners, int neurons,
                             int count_winners) {
  pdl_wait();
  const int s = blockIdx.x;
  const float* d = dots + (size_t)s * neurons;
  float best = 3.0e38f; int bi = 0x7fffffff;
  for (int n = threadIdx.x; n < neurons; n += blockDim.x) {
    const float v = fmaf(-2.f, d[n], wnorm[n]);
    if (v < best || (v == best && n < bi)) { best = v; bi = n; }
  }
  __shared__ float sb[32]; __shared__ int si[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ob = __shfl_xor_sync(0xffffffffu, best, o); int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) { sb[warp] = best; si[warp] = bi; }
  __syncthreads();
  if (warp == 0) {
    best = lane < nw ? sb[lane] : 3.0e38f; bi = lane < nw ? si[lane] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ob = __shfl_xor_sync(0xffffffffu, best, o); int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    if (lane == 0) {
      argmins[s] = bi;
      if (count_winners) atomicAdd(winners + bi, 1);
    }
  }
}

// G[n][s] = exp(-|c_n - c_win(s)|^2 / (2 sigma^2)) written as the split A operand
// [G_hi | G_hi | G_lo] (row pitch 3 * bp) plus rowsum[n] = sum_s G[n][s]; one CTA per neuron.
__global__ void som_gravity_split_k(const float* __restrict__ coords, const int* __restrict__ argmins,
                                    __nv_bfloat16* __restrict__ dst, float* __restrict__ rowsum,
                                    int batch, int bp, float sigma) {
  pdl_wait();
  const int n = blockIdx.x;
  const float cx = coords[2 * n], cy = coords[2 * n + 1];
  const float inv = -1.f / (2.f * sigma * sigma);
  __nv_bfloat16* d = dst + (size_t)n * 3 * bp;
  float acc = 0.f;
  for (int s = threadIdx.x; s < bp; s += blockDim.x) {
    float g = 0.f;
    if (s < batch) {
      const int win = argmins[s];
      const float dx = cx - coords[2 * win], dy = cy - coords[2 * win + 1];
      g = __expf((dx * dx + dy * dy) * inv);
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(g);
    d[s] = hi; d[bp + s] = hi; d[2 * bp + s] = __float2bfloat16_rn(g - __bfloat162float(hi));
    acc += g;
  }
  __shared__ float red[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < ((blockDim.x + 31) >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) rowsum[n] = t;
  }
}

// w[n][k] += gmult * (M[n][k] - rowsum[n] * w[n][k])
__global__ void som_apply_k(float* __restrict__ w, const float* __restrict__ m,
                            const float* __restrict__ rowsum, long long total, int len, float gmult) {
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float wv = w[i];
  w[i] = wv + gmult * (m[i] - rowsum[i / len] * wv);
}

void launch_som_split(const float* src, __nv_bfloat16* dst, int rows, int len, int kp, long long ld,
                      long long part_stride, int pattern, float* norm_out, cudaStream_t st) {
  launch_k(som_split_k, rows, 128, 0, st, src, dst, rows, len, kp, ld, part_stride, pattern, norm_out);
}
void launch_som_argmin(const float* dots, const float* wnorm, int* argmins, int* winners, int batch,
                       int neurons, cudaStream_t st) {
  int threads = neurons >= 256 ? 256 : ((neurons + 31) / 32) * 32;
  launch_k(som_argmin_k, batch, threads, 0, st, dots, wnorm, argmins, winners, neurons, winners ? 1 : 0);
}
void launch_som_gravity_split(const float* coords, const int* argmins, __nv_bfloat16* dst, float* rowsum,
                              int neurons, int batch, int bp, float sigma, cudaStream_t st) {
  launch_k(som_gravity_split_k, neurons, 128, 0, st, coords, argmins, dst, rowsum, batch, bp, sigma);
}
void launch_som_apply(float* w, const float* m, const float* rowsum, int neurons, int len, float gmult,
                      cudaStream_t st) {
  const long long total = (long long)neurons * len;
  launch_k(som_apply_k, (int)((total + 255) / 256), 256, 0, st, w, m, rowsum, total, len, gmult);
}

void launch_som_winners(const float* x, const float* w, int* argmins, int* winners, int batch,
                        int neurons, int len, int count_winners, cudaStream_t st) {
  int threads = neurons >= 256 ? 256 : ((neurons + 31) / 32) * 32;
  launch_k(som_winners_k, batch, threads, 0, st, x, w, argmins, winners, neurons, len, count_winners);
}
void launch_som_update(const float* x, float* w, const float* coords, const int* argmins, int batch,
                       int neurons, int len, float sigma, float gmult, cudaStream_t st) {
  int total = neurons * len;
  launch_k(som_update_k, (total + 255) / 256, 256, 0, st, x, w, coords, argmins, batch, neurons, len, sigma, gmult);
}

}  // namespace zn
