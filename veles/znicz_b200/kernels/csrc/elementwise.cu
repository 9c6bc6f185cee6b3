// Elementwise / data-movement kernels: activations fwd/bwd, err_y *= f'(y) with fused
// bias-gradient column sums, dropout, mul/add, crop, axpby, gather, mask, casts.
// Parity targets: /root/reference/cuda/activation.cu, gradient_descent_{tanh,sigmoid,
// relu,strict_relu}.cu, dropout.cu, multiplier.cu, summator.cu, cutter.cu,
// weights_zerofilling.cu. All kernels: grid-stride, 16-byte vector path when aligned.
#include "common.cuh"
#include <cuda_fp8.h>

namespace zn {

template <typename T>
__global__ void act_forward_k(const T* __restrict__ x, T* __restrict__ y, long long n, int act,
                              float factor) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) stf(y + i, act_fwd(act, ldf(x + i), factor, (int)(i & 1)));
}

template <typename T>
__global__ void act_backward_k(const T* __restrict__ err_y, const T* __restrict__ x,
                               const T* __restrict__ y, T* __restrict__ err_x, long long n,
                               int act, float factor) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float xv = x ? ldf(x + i) : 0.f;
    float yv = y ? ldf(y + i) : 0.f;
    stf(err_x + i, ldf(err_y + i) * act_deriv(act, xv, yv, factor, (int)(i & 1)));
  }
}

// err_y[r, c] *= f'(y[r, c]) in place and col_sum[c] = sum_r err_y[r, c] (bias gradient),
// one pass. Block = 32 x 8 threads; each block owns 32 columns and a slice of rows, then
// one atomicAdd per column per block (deterministic variant: partial[blockIdx.y][c]).
template <typename T>
__global__ void err_act_colsum_k(T* __restrict__ err_y, const T* __restrict__ y, int rows, int cols,
                                 int act, float* __restrict__ partial /*[gridDim.y][cols]*/) {
  pdl_wait();
  __shared__ float red[8][33];
  int c = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
  if (c < cols) {
    for (int r = blockIdx.y * 8 + threadIdx.y; r < rows; r += gridDim.y * 8) {
      size_t o = (size_t)r * cols + c;
      float e = ldf(err_y + o);
      if (act != ACT_LINEAR) {
        e *= act_deriv(act, 0.f, ldf(y + o));
        stf(err_y + o, e);
      }
      acc += e;
    }
  }
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols && partial) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += red[j][threadIdx.x];
    partial[(size_t)blockIdx.y * cols + c] = s;
  }
}

// Vectorised variant for cols % 8 == 0: 256 threads = (256/groups) row lanes x groups of 8
// columns; 16-byte loads/stores; per-block partial sums -> partial[blockIdx.x][cols].
template <typename T>
__global__ void __launch_bounds__(256) err_act_colsum_vec_k(T* __restrict__ err_y, const T* __restrict__ y,
                                                         int rows, int cols, int act,
                                                         float* __restrict__ partial) {
  pdl_wait();
  __shared__ float red[256][9];
  const int groups = cols >> 3;                 // <= 256
  const int lanes = 256 / groups;
  const int g = threadIdx.x % groups, lane = threadIdx.x / groups;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (lane < lanes) {
    for (int r = blockIdx.x * lanes + lane; r < rows; r += gridDim.x * lanes) {
      size_t o = (size_t)r * cols + g * 8;
      float e[8];
      ld8(err_y + o, e);
      if (act != ACT_LINEAR) {
        float yv[8];
        ld8(y + o, yv);
#pragma unroll
        for (int j = 0; j < 8; ++j) e[j] *= act_deriv(act, 0.f, yv[j]);
        st8(err_y + o, e);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += e[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[threadIdx.x][j] = acc[j];
  __syncthreads();
  if (partial && threadIdx.x < cols) {
    const int c = threadIdx.x, gg = c >> 3, j = c & 7;
    float s = 0.f;
    for (int l = 0; l < lanes; ++l) s += red[l * groups + gg][j];
    partial[(size_t)blockIdx.x * cols + c] = s;
  }
}

template <typename T>
__global__ void dropout_forward_k(const T* __restrict__ x, T* __restrict__ y, T* __restrict__ mask,
                                  long long n, const int* __restrict__ rng, uint32_t threshold,
                                  float scale) {
  pdl_wait();
  uint32_t seed = (uint32_t)rng[0], counter = (uint32_t)rng[1];
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float m = hash_u32(seed, counter, (uint64_t)i) >= threshold ? scale : 0.f;
    stf(mask + i, m);
    stf(y + i, ldf(x + i) * m);
  }
}

template <typename T>
__global__ void mul_k(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ o, long long n) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) stf(o + i, ldf(a + i) * ldf(b + i));
}
template <typename T>
__global__ void add_k(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ o, long long n) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) stf(o + i, ldf(a + i) + ldf(b + i));
}
template <typename T>
__global__ void mul_backward_k(const T* __restrict__ x, const T* __restrict__ y,
                               const T* __restrict__ e, T* __restrict__ ex, T* __restrict__ ey,
                               long long n) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float ev = ldf(e + i);
    stf(ex + i, ev * ldf(y + i));
    stf(ey + i, ev * ldf(x + i));
  }
}

// dst[r, doff + c] = alpha * src[r, soff + c] + beta * dst[r, doff + c], c < len
template <typename T>
__global__ void axpby_2d_k(const T* __restrict__ src, int src_ld, int soff, T* __restrict__ dst,
                           int dst_ld, int doff, int rows, int len, float alpha, float beta) {
  pdl_wait();
  long long n = (long long)rows * len;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    int r = (int)(i / len), c = (int)(i % len);
    T* d = dst + (size_t)r * dst_ld + doff + c;
    float v = alpha * ldf(src + (size_t)r * src_ld + soff + c);
    if (beta != 0.f) v += beta * ldf(d);
    stf(d, v);
  }
}

// dst[(j * A + i), doff + c] = src[(i * Bn + j), soff + c]  (i < A, j < Bn, c < len): swaps the two
// leading axes of a [A][Bn][len] block while re-basing the rows - [batch][time] <-> [time][batch]
// for the whole sequence in ONE launch (the LSTM sequence unit issued one strided copy per step)
template <typename T>
__global__ void swap01_2d_k(const T* __restrict__ src, int src_ld, int soff, T* __restrict__ dst,
                            int dst_ld, int doff, int A, int Bn, int len) {
  pdl_wait();
  const long long n = (long long)A * Bn * len;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
    const int c = (int)(q % len);
    const long long r = q / len;              // destination row = j * A + i
    const int i = (int)(r % A), j = (int)(r / A);
    dst[(size_t)r * dst_ld + doff + c] = src[((size_t)i * Bn + j) * src_ld + soff + c];
  }
}

// NHWC crop: out[n, y, x, c] = in[n, y + top, x + left, c]; backward pastes into zeros.
template <typename T>
__global__ void crop_nhwc_k(const T* __restrict__ in, T* __restrict__ out, int N, int H, int W, int C,
                            int oh, int ow, int top, int left, int backward) {
  pdl_wait();
  if (!backward) {
    long long n = (long long)N * oh * ow * C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
      int c = (int)(i % C); long long t = i / C;
      int x = (int)(t % ow); t /= ow; int y = (int)(t % oh); int b = (int)(t / oh);
      out[i] = in[(((size_t)b * H + y + top) * W + x + left) * C + c];
    }
  } else {  // in = err_output [N, oh, ow, C], out = err_input [N, H, W, C]
    long long n = (long long)N * H * W * C;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
      int c = (int)(i % C); long long t = i / C;
      int x = (int)(t % W); t /= W; int y = (int)(t % H); int b = (int)(t / H);
      int yy = y - top, xx = x - left;
      T v; stf(&v, 0.f);
      if (yy >= 0 && yy < oh && xx >= 0 && xx < ow) v = in[(((size_t)b * oh + yy) * ow + xx) * C + c];
      out[i] = v;
    }
  }
}

// rows gather: dst[i, :] = src[idx[i], :] for i < count, zero for the tail rows
template <typename TS, typename TD>
__global__ void gather_rows_k(const TS* __restrict__ src, const int* __restrict__ idx,
                              TD* __restrict__ dst, int count, int max_rows, long long row) {
  pdl_wait();
  long long n = (long long)max_rows * row;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    int r = (int)(i / row); long long c = i % row;
    float v = 0.f;
    if (r < count) v = ldf(src + (size_t)idx[r] * row + c);
    stf(dst + i, v);
  }
}
__global__ void gather_labels_k(const int* __restrict__ src, const int* __restrict__ idx,
                                int* __restrict__ dst, int count, int max_rows) {
  pdl_wait();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < max_rows) dst[i] = i < count ? src[idx[i]] : -1;
}

// hdr = [count, class, epoch, pad, idx0, idx1, ...]; dst rows >= count are zero / label -1
template <typename TS, typename TD>
__global__ void gather_minibatch_k(const TS* __restrict__ src, const int* __restrict__ labels_src,
                                   const int* __restrict__ hdr, TD* __restrict__ dst,
                                   int* __restrict__ labels_dst, int max_rows, int row8,
                                   TD* __restrict__ dst_pad, int C, int CP) {
  pdl_wait();
  const int count = hdr[0];
  const int* idx = hdr + 4;
  const int total = max_rows * row8;
  if (dst_pad) {
    // second copy with the channels padded C -> CP (= 8): the first conv layer's tcgen05 gather
    // then moves whole 16-byte pixels (replaces a separate pad_channels launch)
    const int pixels = row8 * 8 / C;
    const int ptotal = max_rows * pixels;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < ptotal; i += gridDim.x * blockDim.x) {
      const int r = i / pixels, px = i - r * pixels;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
      if (r < count) {
        const TS* s = src + (size_t)idx[r] * row8 * 8 + (size_t)px * C;
        for (int j = 0; j < C; ++j) v[j] = ldf(s + j);
      }
      st8(dst_pad + (size_t)i * 8, v);
    }
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int r = i / row8, c = i - r * row8;
    float v[8];
    if (r < count) {
      ld8(src + ((size_t)idx[r] * row8 + c) * 8, v);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
    st8(dst + (size_t)i * 8, v);
  }
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (labels_dst && t < max_rows) labels_dst[t] = t < count ? labels_src[idx[t]] : -1;
}

// [P][C] -> [P][CP] (CP = 8-padded, zeros in the padding): first-layer channel padding so the
// implicit-GEMM gather can use 16-byte chunks
template <typename T>
__global__ void pad_channels_k(const T* __restrict__ x, T* __restrict__ y, int pixels, int C, int CP) {
  pdl_wait();
  const int total = pixels * CP;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int p = i / CP, c = i - p * CP;
    T v; stf(&v, 0.f);
    if (c < C) v = x[(size_t)p * C + c];
    y[i] = v;
  }
}

template <typename T>
__global__ void mask_mul_k(T* __restrict__ w, const T* __restrict__ mask, long long n) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) stf(w + i, ldf(w + i) * ldf(mask + i));
}

template <typename TS, typename TD>
__global__ void cast_k(const TS* __restrict__ s, TD* __restrict__ d, long long n) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) stf(d + i, ldf(s + i));
}

// depooling: out[offs[i]] = in[i] (out pre-zeroed by the caller via memsetAsync)
template <typename T>
__global__ void scatter_offsets_k(const T* __restrict__ in, const int* __restrict__ offs,
                                  T* __restrict__ out, long long n, int accumulate) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) out[offs[i]] = in[i];
}

static inline int grid_for(long long n, int block = 256) {
  long long g = (n + block - 1) / block;
  const long long cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

// ----------------------------------------------------------------------------- launchers
#define DISPATCH_T(bf16, ...)                                  \
  if (bf16) { using T = __nv_bfloat16; __VA_ARGS__; } else { using T = float; __VA_ARGS__; }

void launch_act_forward(const void* x, void* y, long long n, int act, float factor, bool bf16,
                        cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(act_forward_k<T>, grid_for(n), 256, 0, st, (const T*)x, (T*)y, n, act, factor));
}
void launch_act_backward(const void* ey, const void* x, const void* y, void* ex, long long n, int act,
                         float factor, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(act_backward_k<T>, grid_for(n), 256, 0, st, 
      (const T*)ey, (const T*)x, (const T*)y, (T*)ex, n, act, factor));
}
int err_act_colsum_slices(int rows) { int s = (rows + 63) / 64; return s < 1 ? 1 : (s > 128 ? 128 : s); }
void launch_err_act_colsum(void* err_y, const void* y, int rows, int cols, int act, float* partial,
                           int slices, bool bf16, cudaStream_t st) {
  if (cols % 8 == 0 && cols <= 256 && (((uintptr_t)err_y) & 15) == 0 &&
      (y == nullptr || (((uintptr_t)y) & 15) == 0)) {
    DISPATCH_T(bf16, launch_k(err_act_colsum_vec_k<T>, slices, 256, 0, st, (T*)err_y, (const T*)y, rows,
                                                                       cols, act, partial));
    return;
  }
  dim3 grid((cols + 31) / 32, slices), block(32, 8);
  DISPATCH_T(bf16, launch_k(err_act_colsum_k<T>, grid, block, 0, st, (T*)err_y, (const T*)y, rows, cols, act,
                                                              partial));
}
void launch_dropout_forward(const void* x, void* y, void* mask, long long n, const int* rng,
                            uint32_t threshold, float scale, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(dropout_forward_k<T>, grid_for(n), 256, 0, st, 
      (const T*)x, (T*)y, (T*)mask, n, rng, threshold, scale));
}
void launch_binary(const void* a, const void* b, void* o, long long n, int op, bool bf16,
                   cudaStream_t st) {
  if (op == 0) { DISPATCH_T(bf16, launch_k(mul_k<T>, grid_for(n), 256, 0, st, (const T*)a, (const T*)b, (T*)o, n)); }
  else { DISPATCH_T(bf16, launch_k(add_k<T>, grid_for(n), 256, 0, st, (const T*)a, (const T*)b, (T*)o, n)); }
}
void launch_mul_backward(const void* x, const void* y, const void* e, void* ex, void* ey, long long n,
                         bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(mul_backward_k<T>, grid_for(n), 256, 0, st, 
      (const T*)x, (const T*)y, (const T*)e, (T*)ex, (T*)ey, n));
}
void launch_axpby_2d(const void* src, int src_ld, int soff, void* dst, int dst_ld, int doff, int rows,
                     int len, float alpha, float beta, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(axpby_2d_k<T>, grid_for((long long)rows * len), 256, 0, st, 
      (const T*)src, src_ld, soff, (T*)dst, dst_ld, doff, rows, len, alpha, beta));
}
void launch_swap01_2d(const void* src, int src_ld, int soff, void* dst, int dst_ld, int doff, int A,
                      int Bn, int len, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(swap01_2d_k<T>, grid_for((long long)A * Bn * len), 256, 0, st,
      (const T*)src, src_ld, soff, (T*)dst, dst_ld, doff, A, Bn, len));
}
void launch_crop_nhwc(const void* in, void* out, int N, int H, int W, int C, int oh, int ow, int top,
                      int left, int backward, bool bf16, cudaStream_t st) {
  long long n = backward ? (long long)N * H * W * C : (long long)N * oh * ow * C;
  DISPATCH_T(bf16, launch_k(crop_nhwc_k<T>, grid_for(n), 256, 0, st, (const T*)in, (T*)out, N, H, W, C, oh, ow,
                                                              top, left, backward));
}
void launch_gather_rows(const void* src, bool src_bf16, const int* idx, void* dst, bool dst_bf16,
                        int count, int max_rows, long long row, cudaStream_t st) {
  long long n = (long long)max_rows * row;
  int g = grid_for(n);
  if (!src_bf16 && !dst_bf16) launch_k(gather_rows_k<float, float>, g, 256, 0, st, (const float*)src, idx, (float*)dst, count, max_rows, row);
  else if (!src_bf16 && dst_bf16) launch_k(gather_rows_k<float, __nv_bfloat16>, g, 256, 0, st, (const float*)src, idx, (__nv_bfloat16*)dst, count, max_rows, row);
  else if (src_bf16 && dst_bf16) launch_k(gather_rows_k<__nv_bfloat16, __nv_bfloat16>, g, 256, 0, st, (const __nv_bfloat16*)src, idx, (__nv_bfloat16*)dst, count, max_rows, row);
  else launch_k(gather_rows_k<__nv_bfloat16, float>, g, 256, 0, st, (const __nv_bfloat16*)src, idx, (float*)dst, count, max_rows, row);
}
// Host -> device "pull": the SMs read a pinned (mapped) host buffer directly over PCIe and write
// device memory. Used instead of cudaMemcpyAsync for the per-step loader uploads: on this platform
// every switch between the copy engine and compute work in one stream costs ~100 us (measured,
// profiles/host_vs_device_r1.md), a kernel reading host memory costs one PCIe round trip.
// ld.global.cv: never serve a slot the host has rewritten since from a cached line.
__global__ void pull_from_host_k(const uint4* __restrict__ src, uint4* __restrict__ dst, long long n16,
                                 const unsigned char* __restrict__ src_b, unsigned char* __restrict__ dst_b,
                                 int tail) {
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride)
    dst[i] = __ldcv(src + i);
  if (blockIdx.x == 0 && (int)threadIdx.x < tail) dst_b[threadIdx.x] = __ldcv(src_b + threadIdx.x);
}
void launch_pull_from_host(const void* src_dev_alias, void* dst, long long nbytes, cudaStream_t st) {
  const long long n16 = nbytes / 16;
  const int tail = (int)(nbytes - n16 * 16);
  long long blocks = (n16 + 255) / 256;
  if (blocks > 592) blocks = 592;
  if (blocks < 1) blocks = 1;
  launch_k(pull_from_host_k, (int)blocks, 256, 0, st, (const uint4*)src_dev_alias, (uint4*)dst, n16,
           (const unsigned char*)src_dev_alias + n16 * 16, (unsigned char*)dst + n16 * 16, tail);
}

// channel padding, CP % 8 == 0: thread = (pixel, group of 8 output channels) -> one 16/32-byte
// store (the element-wise kernel above spent 104 us on AlexNet's 128 x 227 x 227 x 3 -> 8 input)
template <typename T>
__global__ void pad_channels_vec_k(const T* __restrict__ x, T* __restrict__ y, long long groups, int C,
                                   int CP8) {
  pdl_wait();
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < groups; i += stride) {
    const long long p = i / CP8;
    const int c0 = (int)(i - p * CP8) * 8;
    const T* src = x + p * C + c0;
    float v[8];
    if (c0 + 8 <= C && ((reinterpret_cast<uintptr_t>(src) & (sizeof(T) * 8 - 1)) == 0)) {
      ld8(src, v);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (c0 + j < C) ? ldf(src + j) : 0.f;
    }
    st8(y + i * 8, v);
  }
}

// ---- fp8 (e4m3) per-tensor quantisation: q = sat(x * 448 / amax) -------------------------------
template <typename T>
__global__ void absmax_k(const T* __restrict__ x, long long n, float* __restrict__ amax) {
  pdl_wait();
  float m = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    m = fmaxf(m, fabsf(ldf(x + i)));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(amax), __float_as_int(m));   // m >= 0
}
template <typename T>
__global__ void quant_e4m3_k(const T* __restrict__ x, unsigned char* __restrict__ q, long long n,
                             const float* __restrict__ amax) {
  pdl_wait();
  const float scale = 448.f / fmaxf(*amax, 1e-12f);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    q[i] = (unsigned char)__nv_cvt_float_to_fp8(ldf(x + i) * scale, __NV_SATFINITE, __NV_E4M3);
}
void launch_fp8_absmax(const void* x, bool bf16, long long n, float* amax, cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(absmax_k<T>, grid_for(n), 256, 0, st, (const T*)x, n, amax));
}
void launch_fp8_quantize(const void* x, bool bf16, unsigned char* q, long long n, const float* amax,
                         cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(quant_e4m3_k<T>, grid_for(n), 256, 0, st, (const T*)x, q, n, amax));
}

void launch_pull_from_host_bytes(const void* src, void* dst, int nbytes, cudaStream_t st) {
  launch_k(pull_from_host_k, 1, 256, 0, st, (const uint4*)nullptr, (uint4*)nullptr, 0LL,
           (const unsigned char*)src, (unsigned char*)dst, nbytes);
}

void launch_gather_minibatch(const void* src, bool src_bf16, const int* labels_src, const int* hdr,
                             void* dst, bool dst_bf16, int* labels_dst, int max_rows, long long row,
                             void* dst_pad, int C, int CP, cudaStream_t st) {
  int row8 = (int)(row / 8);
  int g = grid_for((long long)max_rows * row8);
  if (g * 256 < max_rows) g = (max_rows + 255) / 256;
  if (!src_bf16 && dst_bf16) launch_k(gather_minibatch_k<float, __nv_bfloat16>, g, 256, 0, st, (const float*)src, labels_src, hdr, (__nv_bfloat16*)dst, labels_dst, max_rows, row8, (__nv_bfloat16*)dst_pad, C, CP);
  else if (!src_bf16) launch_k(gather_minibatch_k<float, float>, g, 256, 0, st, (const float*)src, labels_src, hdr, (float*)dst, labels_dst, max_rows, row8, (float*)dst_pad, C, CP);
  else if (dst_bf16) launch_k(gather_minibatch_k<__nv_bfloat16, __nv_bfloat16>, g, 256, 0, st, (const __nv_bfloat16*)src, labels_src, hdr, (__nv_bfloat16*)dst, labels_dst, max_rows, row8, (__nv_bfloat16*)dst_pad, C, CP);
  else launch_k(gather_minibatch_k<__nv_bfloat16, float>, g, 256, 0, st, (const __nv_bfloat16*)src, labels_src, hdr, (float*)dst, labels_dst, max_rows, row8, (float*)dst_pad, C, CP);
}
void launch_gather_labels(const int* src, const int* idx, int* dst, int count, int max_rows,
                          cudaStream_t st) {
  launch_k(gather_labels_k, (max_rows + 255) / 256, 256, 0, st, src, idx, dst, count, max_rows);
}
void launch_pad_channels(const void* x, void* y, int pixels, int C, int CP, bool bf16, cudaStream_t st) {
  if (CP % 8 == 0 && (reinterpret_cast<uintptr_t>(y) & 31) == 0) {
    const long long groups = (long long)pixels * (CP / 8);
    DISPATCH_T(bf16, launch_k(pad_channels_vec_k<T>, grid_for(groups), 256, 0, st, (const T*)x, (T*)y, groups, C, CP / 8));
    return;
  }
  DISPATCH_T(bf16, launch_k(pad_channels_k<T>, grid_for((long long)pixels * CP), 256, 0, st, (const T*)x, (T*)y, pixels, C, CP));
}
void launch_mask_mul(void* w, const void* mask, long long n, bool bf16, cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(mask_mul_k<T>, grid_for(n), 256, 0, st, (T*)w, (const T*)mask, n));
}
void launch_cast(const void* s, bool s_bf16, void* d, bool d_bf16, long long n, cudaStream_t st) {
  int g = grid_for(n);
  if (s_bf16 && !d_bf16) launch_k(cast_k<__nv_bfloat16, float>, g, 256, 0, st, (const __nv_bfloat16*)s, (float*)d, n);
  else if (!s_bf16 && d_bf16) launch_k(cast_k<float, __nv_bfloat16>, g, 256, 0, st, (const float*)s, (__nv_bfloat16*)d, n);
  else if (s_bf16) launch_k(cast_k<__nv_bfloat16, __nv_bfloat16>, g, 256, 0, st, (const __nv_bfloat16*)s, (__nv_bfloat16*)d, n);
  else launch_k(cast_k<float, float>, g, 256, 0, st, (const float*)s, (float*)d, n);
}
void launch_scatter_offsets(const void* in, const int* offs, void* out, long long n, bool bf16,
                            cudaStream_t st) {
  DISPATCH_T(bf16, launch_k(scatter_offsets_k<T>, grid_for(n), 256, 0, st, (const T*)in, offs, (T*)out, n, 0));
}

}  // namespace zn

// ------------------------------------------------------------------------------------------
// LSTM sequence cell kernels (ops/lstm_seq.py). Gate pre-activations z = [i | f | g | o]
// (each H wide, fp32) come from one GEMM per time step; the cell update is one fused launch:
//   i = sigma(z_i), f = sigma(z_f), g = A tanh(B z_g), o = sigma(z_o)
//   c = i * g + f * c_prev ;  h = o * A tanh(B c)          (A = 1.7159, B = 0.6666: the
//   reference's scaled tanh, /root/reference/lstm.py:75-108 + all2all.py:271-296)
// h is written twice: to the output sequence slot and into the [x | h] operand of step t + 1.
namespace zn {

template <typename T>
__global__ void lstm_cell_fwd_k(const float* __restrict__ z, const float* __restrict__ c_prev,
                                float* __restrict__ c, float* __restrict__ gates,
                                T* __restrict__ h_out, long long ldh, T* __restrict__ h_next,
                                long long ldn, int batch, int H) {
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch * H) return;
  const int b = i / H, j = i - b * H;
  const float* zr = z + (size_t)b * 4 * H;
  const float ig = 1.f / (1.f + __expf(-zr[j]));
  const float fg = 1.f / (1.f + __expf(-zr[H + j]));
  const float gg = 1.7159f * tanhf(0.6666f * zr[2 * H + j]);
  const float og = 1.f / (1.f + __expf(-zr[3 * H + j]));
  const float cv = ig * gg + fg * (c_prev ? c_prev[i] : 0.f);
  const float tc = 1.7159f * tanhf(0.6666f * cv);
  const float hv = og * tc;
  c[i] = cv;
  float* gr = gates + (size_t)b * 4 * H;
  gr[j] = ig; gr[H + j] = fg; gr[2 * H + j] = gg; gr[3 * H + j] = og;
  stf(h_out + (size_t)b * ldh + j, hv);
  if (h_next) stf(h_next + (size_t)b * ldn + j, hv);
}

// dh = err_h (from above, may be null) + dh_rec (from step t + 1 through W_h, may be null)
// dz (fp32 + compute-dtype copy for the GEMMs), dc_prev = dc * f
template <typename T>
__global__ void lstm_cell_bwd_k(const T* __restrict__ err_h, long long lde,
                                const T* __restrict__ dh_rec, long long ldr,
                                const float* __restrict__ dc_next, const float* __restrict__ gates,
                                const float* __restrict__ c, const float* __restrict__ c_prev,
                                float* __restrict__ dc_prev, T* __restrict__ dz, int batch, int H) {
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch * H) return;
  const int b = i / H, j = i - b * H;
  float dh = 0.f;
  if (err_h) dh += ldf(err_h + (size_t)b * lde + j);
  if (dh_rec) dh += ldf(dh_rec + (size_t)b * ldr + j);
  const float* gr = gates + (size_t)b * 4 * H;
  const float ig = gr[j], fg = gr[H + j], gg = gr[2 * H + j], og = gr[3 * H + j];
  const float tc = 1.7159f * tanhf(0.6666f * c[i]);
  const float dtc = tc * tc * (-0.388484177f) + 1.14381894f;     // d(A tanh(B c)) / dc
  float dc = dh * og * dtc + (dc_next ? dc_next[i] : 0.f);
  const float cp = c_prev ? c_prev[i] : 0.f;
  T* dr = dz + (size_t)b * 4 * H;
  stf(dr + j, dc * gg * ig * (1.f - ig));
  stf(dr + H + j, dc * cp * fg * (1.f - fg));
  stf(dr + 2 * H + j, dc * ig * (gg * gg * (-0.388484177f) + 1.14381894f));
  stf(dr + 3 * H + j, dh * tc * og * (1.f - og));
  dc_prev[i] = dc * fg;
}

void launch_lstm_cell_fwd(const float* z, const float* c_prev, float* c, float* gates, void* h_out,
                          long long ldh, void* h_next, long long ldn, int batch, int H, bool bf16,
                          cudaStream_t st) {
  const int g = (batch * H + 255) / 256;
  DISPATCH_T(bf16, launch_k(lstm_cell_fwd_k<T>, g, 256, 0, st, z, c_prev, c, gates, (T*)h_out, ldh,
                                                         (T*)h_next, ldn, batch, H));
}
void launch_lstm_cell_bwd(const void* err_h, long long lde, const void* dh_rec, long long ldr,
                          const float* dc_next, const float* gates, const float* c,
                          const float* c_prev, float* dc_prev, void* dz, int batch, int H, bool bf16,
                          cudaStream_t st) {
  const int g = (batch * H + 255) / 256;
  DISPATCH_T(bf16, launch_k(lstm_cell_bwd_k<T>, g, 256, 0, st, (const T*)err_h, lde, (const T*)dh_rec, ldr,
                                                         dc_next, gates, c, c_prev, dc_prev, (T*)dz,
                                                         batch, H));
}

}  // namespace zn
