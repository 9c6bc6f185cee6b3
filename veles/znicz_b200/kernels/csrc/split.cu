// fp32 -> bf16 hi/lo part splitter for the "fp32 on the tensor cores" path (kernels/fp32x.py).
//
// x = hi + lo with hi = bf16(x), lo = bf16(x - hi) carries 16 mantissa bits; the product of two
// split operands  x.w ~= hi.hi + hi.lo + lo.hi (+ lo.lo)  is evaluated by ONE bf16 tcgen05 GEMM whose
// reduction dimension holds the parts side by side:
//     A side, pattern 0: [hi | hi | lo | lo]      B side, pattern 1: [hi | lo | hi | lo]
// (3 parts drop the lo.lo term: 2^-18 relative). The fp32 accumulator of the tensor core adds the
// partial products, so no extra pass is needed. Parts are either concatenated along the columns of
// the destination (part_stride = padded length) or stacked along its rows (part_stride = rows * ld).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include "common.cuh"

namespace zn {

struct SplitDst {
  __nv_bfloat16* p;
  long long ld, part_stride;
  int kp, nparts, pattern;
};

__device__ __forceinline__ void split_store(const SplitDst& d, long long row, int k, __nv_bfloat16 hi,
                                            __nv_bfloat16 lo) {
  if (d.p == nullptr || k >= d.kp) return;
  __nv_bfloat16* o = d.p + row * d.ld + k;
#pragma unroll 4
  for (int p = 0; p < d.nparts; ++p) {
    const bool is_lo = d.pattern ? (p & 1) : (p >= 2);
    o[p * d.part_stride] = is_lo ? lo : hi;
  }
}

// one fp32 source [rows][len] -> up to two split destinations (e.g. the column-concatenated operand
// of dgrad and the row-stacked operand of wgrad from the same err_output)
__global__ void split_parts_k(const float* __restrict__ src, long long rows, int len, int kmax,
                              SplitDst a, SplitDst b) {
  pdl_wait();
  const long long total = rows * kmax;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / kmax;
    const int k = (int)(i - row * kmax);
    const float v = k < len ? src[row * len + k] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    split_store(a, row, k, hi, lo);
    split_store(b, row, k, hi, lo);
  }
}

// conv weights fp32 [F][taps][C] -> the dgrad operand [taps][nparts * Fp][Cp] (parts along F)
__global__ void split_conv_wt_k(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst, int F,
                                int taps, int C, int Fp, int Cp, int nparts, int pattern) {
  pdl_wait();
  const long long total = (long long)taps * Fp * Cp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % Cp);
    const int f = (int)((i / Cp) % Fp);
    const int tap = (int)(i / ((long long)Cp * Fp));
    const float v = (f < F && c < C) ? w[((long long)f * taps + tap) * C + c] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    for (int p = 0; p < nparts; ++p) {
      const bool is_lo = pattern ? (p & 1) : (p >= 2);
      dst[(((long long)tap * nparts + p) * Fp + f) * Cp + c] = is_lo ? lo : hi;
    }
  }
}

void launch_split_parts(const float* src, long long rows, int len, __nv_bfloat16* a, long long a_ld,
                        long long a_stride, int a_kp, int a_parts, int a_pattern, __nv_bfloat16* b,
                        long long b_ld, long long b_stride, int b_kp, int b_parts, int b_pattern,
                        cudaStream_t st) {
  SplitDst da{a, a_ld, a_stride, a_kp, a_parts, a_pattern};
  SplitDst db{b, b_ld, b_stride, b_kp, b_parts, b_pattern};
  const int kmax = (b && b_kp > a_kp) ? b_kp : a_kp;
  const long long total = rows * kmax;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  launch_k(split_parts_k, (int)blocks, 256, 0, st, src, rows, len, kmax, da, db);
}

void launch_split_conv_wt(const float* w, __nv_bfloat16* dst, int F, int taps, int C, int Fp, int Cp,
                          int nparts, int pattern, cudaStream_t st) {
  const long long total = (long long)taps * Fp * Cp;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  launch_k(split_conv_wt_k, (int)blocks, 256, 0, st, w, dst, F, taps, C, Fp, Cp, nparts, pattern);
}

}  // namespace zn
