// Space-to-depth form of a strided first-layer convolution (AlexNet conv1: 11 x 11, stride 4, C = 3).
//
// A stride-s convolution over [N][H][W][C] equals a stride-1 convolution with a ceil(k / s) kernel
// over the space-to-depth tensor [N][H / s][W / s][s * s * C]:
//     xs[n][y'][x'][(dy * s + dx) * C + c] = x[n][y' * s + dy - pad_t][x' * s + dx - pad_l][c]
//     ws[f][ty][tx][(dy * s + dx) * C + c] = w[f][ty * s + dy][tx * s + dx][c]   (0 outside k x k)
// The implicit-GEMM gather then moves 9 taps x 128 bytes per output pixel instead of 121 taps x 16
// bytes (the gather instruction count, not the FLOPs, bound that layer: 340 us fprop + 519 us wgrad
// per step), and with the channels padded to 64 the tensor qualifies for the TMA im2col path.
#include "common.cuh"

namespace zn {

template <typename T>
__global__ void space_to_depth_k(const T* __restrict__ x, __nv_bfloat16* __restrict__ xs, int N, int H, int W,
                                 int C, int s, int pad_t, int pad_l, int Hs, int Ws, int Cp) {
  pdl_wait();
  const long long total = (long long)N * Hs * Ws * Cp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int cc = (int)(i % Cp);
    long long t = i / Cp;
    const int xq = (int)(t % Ws); t /= Ws;
    const int yq = (int)(t % Hs);
    const int n = (int)(t / Hs);
    float v = 0.f;
    if (cc < s * s * C) {
      const int c = cc % C, d = cc / C, dx = d % s, dy = d / s;
      const int y = yq * s + dy - pad_t, xx = xq * s + dx - pad_l;
      if (y >= 0 && y < H && xx >= 0 && xx < W) v = ldf(x + (((long long)n * H + y) * W + xx) * C + c);
    }
    xs[i] = __float2bfloat16_rn(v);
  }
}

// fp32 master weights [F][ky][kx][C] -> bf16 [F][kyp][kxp][Cp] in the space-to-depth tap order
__global__ void s2d_pack_weights_k(const float* __restrict__ w, __nv_bfloat16* __restrict__ ws, int F, int ky,
                                   int kx, int C, int s, int kyp, int kxp, int Cp) {
  pdl_wait();
  const long long total = (long long)F * kyp * kxp * Cp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int cc = (int)(i % Cp);
    long long t = i / Cp;
    const int tx = (int)(t % kxp); t /= kxp;
    const int ty = (int)(t % kyp);
    const int f = (int)(t / kyp);
    float v = 0.f;
    if (cc < s * s * C) {
      const int c = cc % C, d = cc / C, dx = d % s, dy = d / s;
      const int yy = ty * s + dy, xx = tx * s + dx;
      if (yy < ky && xx < kx) v = w[(((long long)f * ky + yy) * kx + xx) * C + c];
    }
    ws[i] = __float2bfloat16_rn(v);
  }
}

// gradient partials in the space-to-depth layout [parts][Fr][kyp][kxp][Cp] -> [parts][F][ky][kx][C]
__global__ void s2d_unpack_grad_k(const float* __restrict__ gs, float* __restrict__ g, int parts, int F, int Fr,
                                  int ky, int kx, int C, int s, int kyp, int kxp, int Cp) {
  pdl_wait();
  const long long total = (long long)parts * F * ky * kx * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long long t = i / C;
    const int xx = (int)(t % kx); t /= kx;
    const int yy = (int)(t % ky); t /= ky;
    const int f = (int)(t % F);
    const int p = (int)(t / F);
    const int ty = yy / s, dy = yy % s, tx = xx / s, dx = xx % s;
    g[i] = gs[((((long long)p * Fr + f) * kyp + ty) * kxp + tx) * Cp + (dy * s + dx) * C + c];
  }
}

static int grid_of(long long total) {
  long long b = (total + 255) / 256;
  if (b > 148 * 32) b = 148 * 32;
  return (int)(b < 1 ? 1 : b);
}

void launch_space_to_depth(const void* x, bool x_bf16, void* xs, int N, int H, int W, int C, int s, int pad_t,
                           int pad_l, int Hs, int Ws, int Cp, cudaStream_t st) {
  const long long total = (long long)N * Hs * Ws * Cp;
  if (x_bf16)
    launch_k(space_to_depth_k<__nv_bfloat16>, grid_of(total), 256, 0, st, (const __nv_bfloat16*)x,
             (__nv_bfloat16*)xs, N, H, W, C, s, pad_t, pad_l, Hs, Ws, Cp);
  else
    launch_k(space_to_depth_k<float>, grid_of(total), 256, 0, st, (const float*)x, (__nv_bfloat16*)xs, N, H, W, C,
             s, pad_t, pad_l, Hs, Ws, Cp);
}
void launch_s2d_pack_weights(const float* w, void* ws, int F, int ky, int kx, int C, int s, int kyp, int kxp, int Cp,
                             cudaStream_t st) {
  launch_k(s2d_pack_weights_k, grid_of((long long)F * kyp * kxp * Cp), 256, 0, st, w, (__nv_bfloat16*)ws, F, ky, kx,
           C, s, kyp, kxp, Cp);
}
void launch_s2d_unpack_grad(const float* gs, float* g, int parts, int F, int Fr, int ky, int kx, int C, int s, int kyp,
                            int kxp, int Cp, cudaStream_t st) {
  launch_k(s2d_unpack_grad_k, grid_of((long long)parts * F * ky * kx * C), 256, 0, st, gs, g, parts, F, Fr, ky, kx, C,
           s, kyp, kxp, Cp);
}

}  // namespace zn
