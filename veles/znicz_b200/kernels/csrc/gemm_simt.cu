// Exact-fp32 SIMT implicit-GEMM family (fallback + reference-equivalent baseline path).
// Used when a shape cannot go through the tcgen05 kernels (TMA alignment: leading dims that are
// not multiples of 8 elements, e.g. MNIST conv2 F=87 / FC K=791) and for fp32-exact numerics
// tests. Tile 64x64x16, 256 threads, 4x4 outputs per thread; operands are fetched through
// functors so dense GEMM (all transposes), conv fprop, conv dgrad and conv wgrad share one
// kernel. Parity of the math: /root/reference/all2all.py:239-243, gd.py:514-546,
// conv.py:278-297, gd_conv.py:333-423 (im2col/col2im expressed as index functors).
#include "common.cuh"

namespace zn {

struct ConvGeom {
  int N, H, W, C;          // input NHWC
  int OH, OW, F;           // output
  int KY, KX, SY, SX;      // kernel, stride
  int PT, PL;              // top / left padding
};

template <typename T> struct DenseA {   // A(m, k)
  const T* p; long long ld; int trans;
  __device__ __forceinline__ float operator()(int m, int k) const {
    return trans ? ldf(p + (long long)k * ld + m) : ldf(p + (long long)m * ld + k);
  }
};
template <typename T> struct DenseB {   // B(k, n)
  const T* p; long long ld; int trans;  // trans=0: stored [K][N]; trans=1: stored [N][K]
  __device__ __forceinline__ float operator()(int k, int n) const {
    return trans ? ldf(p + (long long)n * ld + k) : ldf(p + (long long)k * ld + n);
  }
};
// im2col(x)(pixel, kidx) with kidx = (ky*KX + kx)*C + c
template <typename T> struct Im2col {
  const T* x; ConvGeom g;
  __device__ __forceinline__ float at(int pix, int kidx) const {
    int c = kidx % g.C; int t = kidx / g.C; int kx = t % g.KX; int ky = t / g.KX;
    int ox = pix % g.OW; int t2 = pix / g.OW; int oy = t2 % g.OH; int n = t2 / g.OH;
    int iy = oy * g.SY - g.PT + ky, ix = ox * g.SX - g.PL + kx;
    if (iy < 0 || iy >= g.H || ix < 0 || ix >= g.W) return 0.f;
    return ldf(x + (((long long)n * g.H + iy) * g.W + ix) * g.C + c);
  }
};
template <typename T> struct Im2colA { Im2col<T> f; __device__ __forceinline__ float operator()(int m, int k) const { return f.at(m, k); } };
template <typename T> struct Im2colB { Im2col<T> f; __device__ __forceinline__ float operator()(int k, int n) const { return f.at(k, n); } };
// dgrad gather: A(input pixel, k=(tap, f)) = err_out[n, (iy+PT-ky)/SY, (ix+PL-kx)/SX, f]
template <typename T> struct DgradA {
  const T* e; ConvGeom g;
  __device__ __forceinline__ float operator()(int m, int k) const {
    int f = k % g.F; int tap = k / g.F; int kx = tap % g.KX; int ky = tap / g.KX;
    int ix = m % g.W; int t2 = m / g.W; int iy = t2 % g.H; int n = t2 / g.H;
    int ty = iy + g.PT - ky, tx = ix + g.PL - kx;
    if (ty < 0 || tx < 0 || ty % g.SY || tx % g.SX) return 0.f;
    int oy = ty / g.SY, ox = tx / g.SX;
    if (oy >= g.OH || ox >= g.OW) return 0.f;
    return ldf(e + (((long long)n * g.OH + oy) * g.OW + ox) * g.F + f);
  }
};
// B(k=(tap, f), n=c) = W[f][tap*C + c]   (W stored [F][KY*KX*C], optionally transposed storage)
template <typename T> struct DgradB {
  const T* w; ConvGeom g; long long ld; int trans;
  __device__ __forceinline__ float operator()(int k, int n) const {
    int f = k % g.F; int tap = k / g.F;
    long long col = (long long)tap * g.C + n;
    return trans ? ldf(w + col * ld + f) : ldf(w + (long long)f * ld + col);
  }
};

struct Epilogue {
  void* out; int out_bf16; long long ld;   // C stored [M][ld] (or transposed when out_trans)
  int out_trans;
  const float* bias;                       // per-n bias (may be null)
  int act;
  float alpha, beta;                       // out = alpha * v + beta * out  (beta path reads out)
  long long split_stride;                  // >0: fp32 partials, out + blockIdx.z * split_stride
};

template <typename AL, typename BL>
__global__ void __launch_bounds__(256) gemm_simt_k(AL A, BL B, Epilogue ep, int M, int N, int K,
                                                   int k_chunk) {
  pdl_wait();
  __shared__ float As[16][65];
  __shared__ float Bs[16][65];
  int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  int kb = blockIdx.z * k_chunk, ke = min(K, kb + k_chunk);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = kb; k0 < ke; k0 += 16) {
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      int e = threadIdx.x + l * 256;           // 0..1023 -> (kk, mm)
      int kk = e % 16, mm = e / 16;
      int m = m0 + mm, k = k0 + kk;
      As[kk][mm] = (m < M && k < ke) ? A(m, k) : 0.f;
      int nn = e % 64, kk2 = e / 64;
      int n = n0 + nn, k2 = k0 + kk2;
      Bs[kk2][nn] = (n < N && k2 < ke) ? B(k2, n) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j];
      long long o = ep.out_trans ? (long long)n * ep.ld + m : (long long)m * ep.ld + n;
      if (ep.split_stride > 0) {
        reinterpret_cast<float*>(ep.out)[(long long)blockIdx.z * ep.split_stride + o] = v;
        continue;
      }
      v *= ep.alpha;                       // act(alpha * acc + bias), same as the tcgen05 epilogue
      if (ep.bias) v += ep.bias[n];
      v = act_fwd5(ep.act, v);
      if (ep.out_bf16) {
        __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(ep.out) + o;
        if (ep.beta != 0.f) v += ep.beta * __bfloat162float(*p);
        *p = __float2bfloat16_rn(v);
      } else {
        float* p = reinterpret_cast<float*>(ep.out) + o;
        if (ep.beta != 0.f) v += ep.beta * *p;
        *p = v;
      }
    }
  }
}

template <typename AL, typename BL>
static void run(AL a, BL b, const Epilogue& ep, int M, int N, int K, int splits, cudaStream_t st) {
  int k_chunk = (K + splits - 1) / splits;
  k_chunk = ((k_chunk + 15) / 16) * 16;
  dim3 grid((N + 63) / 64, (M + 63) / 64, splits);
  launch_k(gemm_simt_k<AL, BL>, grid, 256, 0, st, a, b, ep, M, N, K, k_chunk);
}

// C[M,N] = act(alpha * opA(A) opB(B) + bias) (+ beta*C); a/b dtype selected independently
void launch_gemm_simt(const void* a, bool a_bf16, long long lda, int transa, const void* b, bool b_bf16,
                      long long ldb, int transb, void* c, bool c_bf16, long long ldc, int out_trans,
                      int M, int N, int K, const float* bias, int act, float alpha, float beta,
                      int splits, long long split_stride, cudaStream_t st) {
  Epilogue ep{c, c_bf16 ? 1 : 0, ldc, out_trans, bias, act, alpha, beta, split_stride};
  if (a_bf16 && b_bf16) run(DenseA<__nv_bfloat16>{(const __nv_bfloat16*)a, lda, transa}, DenseB<__nv_bfloat16>{(const __nv_bfloat16*)b, ldb, transb}, ep, M, N, K, splits, st);
  else if (a_bf16) run(DenseA<__nv_bfloat16>{(const __nv_bfloat16*)a, lda, transa}, DenseB<float>{(const float*)b, ldb, transb}, ep, M, N, K, splits, st);
  else if (b_bf16) run(DenseA<float>{(const float*)a, lda, transa}, DenseB<__nv_bfloat16>{(const __nv_bfloat16*)b, ldb, transb}, ep, M, N, K, splits, st);
  else run(DenseA<float>{(const float*)a, lda, transa}, DenseB<float>{(const float*)b, ldb, transb}, ep, M, N, K, splits, st);
}

// out[pix, f] = act(sum_k im2col(x)[pix, k] * W[f, k] + bias[f])
void launch_conv_fprop_simt(const void* x, bool x_bf16, const float* w, long long ldw, int w_trans,
                            const float* bias, void* out, bool out_bf16, ConvGeom g, int act,
                            cudaStream_t st) {
  int M = g.N * g.OH * g.OW, N = g.F, K = g.KY * g.KX * g.C;
  Epilogue ep{out, out_bf16 ? 1 : 0, (long long)g.F, 0, bias, act, 1.f, 0.f, 0};
  DenseB<float> b{w, ldw, w_trans ? 0 : 1};   // W stored [F][K] => B(k,n)=W[n][k] => trans=1
  if (x_bf16) run(Im2colA<__nv_bfloat16>{{(const __nv_bfloat16*)x, g}}, b, ep, M, N, K, 1, st);
  else run(Im2colA<float>{{(const float*)x, g}}, b, ep, M, N, K, 1, st);
}
// err_in[ipix, c] = alpha * sum_{tap,f} err_out[..] * W[f, tap, c] + beta * err_in
void launch_conv_dgrad_simt(const void* err_out, bool e_bf16, const float* w, long long ldw, int w_trans,
                            void* err_in, bool ei_bf16, ConvGeom g, float alpha, float beta,
                            cudaStream_t st) {
  int M = g.N * g.H * g.W, N = g.C, K = g.KY * g.KX * g.F;
  Epilogue ep{err_in, ei_bf16 ? 1 : 0, (long long)g.C, 0, nullptr, 0, alpha, beta, 0};
  DgradB<float> b{w, g, ldw, w_trans};
  if (e_bf16) run(DgradA<__nv_bfloat16>{(const __nv_bfloat16*)err_out, g}, b, ep, M, N, K, 1, st);
  else run(DgradA<float>{(const float*)err_out, g}, b, ep, M, N, K, 1, st);
}
// gradW partials [split][F][K] = sum_{pix in split} err_out[pix, f] * im2col(x)[pix, k]
void launch_conv_wgrad_simt(const void* err_out, bool e_bf16, const void* x, bool x_bf16, float* partials,
                            int splits, ConvGeom g, int out_trans, cudaStream_t st) {
  int M = g.F, N = g.KY * g.KX * g.C, K = g.N * g.OH * g.OW;
  long long ld = out_trans ? (long long)M : (long long)N;
  Epilogue ep{partials, 0, ld, out_trans, nullptr, 0, 1.f, 0.f, (long long)M * N};
  if (e_bf16) {
    DenseA<__nv_bfloat16> a{(const __nv_bfloat16*)err_out, (long long)g.F, 1};
    if (x_bf16) run(a, Im2colB<__nv_bfloat16>{{(const __nv_bfloat16*)x, g}}, ep, M, N, K, splits, st);
    else run(a, Im2colB<float>{{(const float*)x, g}}, ep, M, N, K, splits, st);
  } else {
    DenseA<float> a{(const float*)err_out, (long long)g.F, 1};
    if (x_bf16) run(a, Im2colB<__nv_bfloat16>{{(const __nv_bfloat16*)x, g}}, ep, M, N, K, splits, st);
    else run(a, Im2colB<float>{{(const float*)x, g}}, ep, M, N, K, splits, st);
  }
}

}  // namespace zn

// raw-geometry wrappers for the binding layer (geometry = int[13]:
// N,H,W,C,OH,OW,F,KY,KX,SY,SX,PT,PL)
namespace zn {
static ConvGeom geom_from(const int* g) {
  ConvGeom c; c.N = g[0]; c.H = g[1]; c.W = g[2]; c.C = g[3]; c.OH = g[4]; c.OW = g[5]; c.F = g[6];
  c.KY = g[7]; c.KX = g[8]; c.SY = g[9]; c.SX = g[10]; c.PT = g[11]; c.PL = g[12];
  return c;
}
void launch_conv_fprop_simt_raw(const void* x, bool x_bf16, const float* w, long long ldw, int w_trans,
                                const float* bias, void* out, bool out_bf16, const int* g, int act,
                                cudaStream_t st) {
  launch_conv_fprop_simt(x, x_bf16, w, ldw, w_trans, bias, out, out_bf16, geom_from(g), act, st);
}
void launch_conv_dgrad_simt_raw(const void* e, bool e_bf16, const float* w, long long ldw, int w_trans,
                                void* ei, bool ei_bf16, const int* g, float alpha, float beta,
                                cudaStream_t st) {
  launch_conv_dgrad_simt(e, e_bf16, w, ldw, w_trans, ei, ei_bf16, geom_from(g), alpha, beta, st);
}
void launch_conv_wgrad_simt_raw(const void* e, bool e_bf16, const void* x, bool x_bf16, float* partials,
                                int splits, const int* g, int out_trans, cudaStream_t st) {
  launch_conv_wgrad_simt(e, e_bf16, x, x_bf16, partials, splits, geom_from(g), out_trans, st);
}
}  // namespace zn
