// Pooling forward/backward + depooling for NHWC tensors (ceil-mode partial windows).
// Parity: /root/reference/cuda/pooling.cu (max :22, avg :77, stochastic :151, pool+depool
// :248), gradient_descent_pooling.cu (:24,:56), depooling.cu:4. One thread per (pixel, channel)
// with channels fastest => coalesced. Backward kernels are *gather* formulations (each input
// element inspects the windows that cover it): no memset, no atomics, deterministic.
#include "common.cuh"

namespace zn {

enum PoolMode { POOL_MAX = 0, POOL_MAXABS = 1, POOL_AVG = 2, POOL_STOCH = 3, POOL_STOCH_ABS = 4,
                POOL_STOCH_DEPOOL = 5, POOL_STOCH_ABS_DEPOOL = 6 };

// act: activation fused behind the pooling (0 = none; forward applies f, backward multiplies the
// incoming error by f'(y) with y = the pooled+activated output)
struct PoolGeom { int N, H, W, C, OH, OW, KY, KX, SY, SX; int act; int in_act; };
// in_act (backward only): derivative of the PRODUCER's activation, applied to err_input through the
// pooling input x (= the producer's output y): err_input *= f'(x). Saves the conv / FC layer below a
// separate err_output *= f'(y) pass (/root/reference/gd_conv.py:645-750 runs one per layer).

template <typename T>
__global__ void pool_forward_k(const T* __restrict__ in, T* __restrict__ out, int* __restrict__ offs,
                               PoolGeom g, int mode, const int* __restrict__ rng) {
  pdl_wait();
  long long total = (long long)g.N * g.OH * g.OW * g.C;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % g.C); long long t = i / g.C;
  int ox = (int)(t % g.OW); t /= g.OW; int oy = (int)(t % g.OH); int n = (int)(t / g.OH);
  int y1 = oy * g.SY, x1 = ox * g.SX;
  int y2 = min(y1 + g.KY, g.H), x2 = min(x1 + g.KX, g.W);
  const T* base = in + (size_t)n * g.H * g.W * g.C + c;
  if (mode == POOL_AVG) {
    float s = 0.f;
    for (int y = y1; y < y2; ++y)
      for (int x = x1; x < x2; ++x) s += ldf(base + ((size_t)y * g.W + x) * g.C);
    stf(out + i, act_fwd5(g.act, s / (float)((y2 - y1) * (x2 - x1))));
    return;
  }
  bool use_abs = (mode == POOL_MAXABS || mode == POOL_STOCH_ABS || mode == POOL_STOCH_ABS_DEPOOL);
  int best_off = 0; float best_v = 0.f;
  if (mode == POOL_MAX || mode == POOL_MAXABS) {
    float best_key = -3.0e38f;
    for (int y = y1; y < y2; ++y)
      for (int x = x1; x < x2; ++x) {
        size_t o = ((size_t)y * g.W + x) * g.C;
        float v = ldf(base + o);
        float key = use_abs ? fabsf(v) : v;
        if (key > best_key) { best_key = key; best_v = v; best_off = (int)(o); }
      }
  } else {
    // stochastic: P(index) ~ max(v,0) (or |v|); 16-bit random per output element
    uint32_t rnd = hash_u32((uint32_t)rng[0], (uint32_t)rng[1], (uint64_t)i) >> 16;
    float vsum = 0.f; int cnt = (y2 - y1) * (x2 - x1);
    for (int y = y1; y < y2; ++y)
      for (int x = x1; x < x2; ++x) {
        float v = ldf(base + ((size_t)y * g.W + x) * g.C);
        vsum += use_abs ? fabsf(v) : fmaxf(v, 0.f);
      }
    bool found = false;
    if (vsum == 0.f) {
      int pick = (int)(((unsigned long long)rnd * (unsigned)cnt) >> 16);
      int k = 0;
      for (int y = y1; y < y2 && !found; ++y)
        for (int x = x1; x < x2; ++x, ++k)
          if (k == pick) { size_t o = ((size_t)y * g.W + x) * g.C; best_off = (int)o; best_v = ldf(base + o); found = true; break; }
    } else {
      float pos = (float)rnd * vsum / 65536.f, acc = 0.f;
      for (int y = y1; y < y2 && !found; ++y)
        for (int x = x1; x < x2; ++x) {
          size_t o = ((size_t)y * g.W + x) * g.C;
          float v = ldf(base + o);
          acc += use_abs ? fabsf(v) : fmaxf(v, 0.f);
          if (pos <= acc) { best_off = (int)o; best_v = v; found = true; break; }
        }
      if (!found) {  // rounding at the very end of the window
        size_t o = ((size_t)(y2 - 1) * g.W + (x2 - 1)) * g.C; best_off = (int)o; best_v = ldf(base + o);
      }
    }
  }
  int flat = (int)((size_t)n * g.H * g.W * g.C + c) + best_off;
  offs[i] = flat;
  if (mode == POOL_STOCH_DEPOOL || mode == POOL_STOCH_ABS_DEPOOL) {
    // in-place pool+depool (non-overlapping windows): keep the winner, zero the rest
    T* wbase = const_cast<T*>(base);
    for (int y = y1; y < y2; ++y)
      for (int x = x1; x < x2; ++x) {
        size_t o = ((size_t)y * g.W + x) * g.C;
        if ((int)o != best_off) stf(wbase + o, 0.f);
      }
  } else {
    stf(out + i, act_fwd5(g.act, best_v));
  }
}

// err_in[n,y,x,c] = sum over windows covering (y,x) of err_out[window] * [offs[window]==self]
template <typename T>
__global__ void pool_backward_max_k(const T* __restrict__ err_out, const int* __restrict__ offs,
                                    T* __restrict__ err_in, PoolGeom g, const T* __restrict__ yact,
                                    const T* __restrict__ xin) {
  pdl_wait();
  long long total = (long long)g.N * g.H * g.W * g.C;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % g.C); long long t = i / g.C;
  int x = (int)(t % g.W); t /= g.W; int y = (int)(t % g.H); int n = (int)(t / g.H);
  int oy_hi = min(y / g.SY, g.OH - 1), ox_hi = min(x / g.SX, g.OW - 1);
  int oy_lo = max(0, (y - g.KY + g.SY) / g.SY), ox_lo = max(0, (x - g.KX + g.SX) / g.SX);
  if (y - g.KY + 1 <= 0) oy_lo = 0;
  if (x - g.KX + 1 <= 0) ox_lo = 0;
  float s = 0.f;
  for (int oy = oy_lo; oy <= oy_hi; ++oy)
    for (int ox = ox_lo; ox <= ox_hi; ++ox) {
      size_t o = (((size_t)n * g.OH + oy) * g.OW + ox) * g.C + c;
      if (offs[o] == (int)i)
        s += ldf(err_out + o) * (g.act ? act_deriv(g.act, 0.f, ldf(yact + o)) : 1.f);
    }
  if (g.in_act) s *= act_deriv(g.in_act, 0.f, ldf(xin + i));
  stf(err_in + i, s);
}

template <typename T>
__global__ void pool_backward_avg_k(const T* __restrict__ err_out, T* __restrict__ err_in, PoolGeom g,
                                    const T* __restrict__ yact, const T* __restrict__ xin) {
  pdl_wait();
  long long total = (long long)g.N * g.H * g.W * g.C;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = (int)(i % g.C); long long t = i / g.C;
  int x = (int)(t % g.W); t /= g.W; int y = (int)(t % g.H); int n = (int)(t / g.H);
  int oy_hi = min(y / g.SY, g.OH - 1), ox_hi = min(x / g.SX, g.OW - 1);
  int oy_lo = (y - g.KY + 1 <= 0) ? 0 : (y - g.KY + g.SY) / g.SY;
  int ox_lo = (x - g.KX + 1 <= 0) ? 0 : (x - g.KX + g.SX) / g.SX;
  float s = 0.f;
  for (int oy = oy_lo; oy <= oy_hi; ++oy) {
    int hy = min(oy * g.SY + g.KY, g.H) - oy * g.SY;
    for (int ox = ox_lo; ox <= ox_hi; ++ox) {
      int hx = min(ox * g.SX + g.KX, g.W) - ox * g.SX;
      const size_t o = (((size_t)n * g.OH + oy) * g.OW + ox) * g.C + c;
      s += ldf(err_out + o) * (g.act ? act_deriv(g.act, 0.f, ldf(yact + o)) : 1.f) / (float)(hy * hx);
    }
  }
  if (g.in_act) s *= act_deriv(g.in_act, 0.f, ldf(xin + i));
  stf(err_in + i, s);
}


// ------------------------------------------------------------------ vectorised (C % 8 == 0)
// thread = (output pixel, group of 8 channels): 16-byte loads, 32-bit index math.
template <typename T>
__global__ void pool_forward_vec_k(const T* __restrict__ in, T* __restrict__ out, int* __restrict__ offs,
                                   PoolGeom g, int mode) {
  pdl_wait();
  const int C8 = g.C >> 3;
  const int total = g.N * g.OH * g.OW * C8;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cg = i % C8; int t = i / C8;
  const int ox = t % g.OW; t /= g.OW; const int oy = t % g.OH; const int n = t / g.OH;
  const int y1 = oy * g.SY, x1 = ox * g.SX;
  const int y2 = min(y1 + g.KY, g.H), x2 = min(x1 + g.KX, g.W);
  const int img = n * g.H * g.W * g.C + cg * 8;
  float best[8]; int boff[8]; float key[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { best[j] = 0.f; boff[j] = 0; key[j] = -3.0e38f; }
  for (int y = y1; y < y2; ++y)
    for (int x = x1; x < x2; ++x) {
      const int o = img + (y * g.W + x) * g.C;
      float v[8];
      ld8(in + o, v);
      if (mode == POOL_AVG) {
#pragma unroll
        for (int j = 0; j < 8; ++j) best[j] += v[j];
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float k = (mode == POOL_MAXABS) ? fabsf(v[j]) : v[j];
          if (k > key[j]) { key[j] = k; best[j] = v[j]; boff[j] = o + j; }
        }
      }
    }
  if (mode == POOL_AVG) {
    const float inv = 1.f / (float)((y2 - y1) * (x2 - x1));
#pragma unroll
    for (int j = 0; j < 8; ++j) best[j] *= inv;
  } else {
    int4* po = reinterpret_cast<int4*>(offs + (size_t)i * 8);
    po[0] = make_int4(boff[0], boff[1], boff[2], boff[3]);
    po[1] = make_int4(boff[4], boff[5], boff[6], boff[7]);
  }
  if (g.act) {
#pragma unroll
    for (int j = 0; j < 8; ++j) best[j] = act_fwd5(g.act, best[j]);
  }
  st8(out + (size_t)i * 8, best);
}

template <typename T>
__global__ void pool_backward_vec_k(const T* __restrict__ err_out, const int* __restrict__ offs,
                                    T* __restrict__ err_in, PoolGeom g, int is_avg,
                                    const T* __restrict__ yact, const T* __restrict__ xin) {
  pdl_wait();
  const int C8 = g.C >> 3;
  const int total = g.N * g.H * g.W * C8;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cg = i % C8; int t = i / C8;
  const int x = t % g.W; t /= g.W; const int y = t % g.H; const int n = t / g.H;
  const int oy_hi = min(y / g.SY, g.OH - 1), ox_hi = min(x / g.SX, g.OW - 1);
  const int oy_lo = (y - g.KY + 1 <= 0) ? 0 : (y - g.KY + g.SY) / g.SY;
  const int ox_lo = (x - g.KX + 1 <= 0) ? 0 : (x - g.KX + g.SX) / g.SX;
  const int self = i * 8;     // flat element index of channel 0 of this group
  float s[8], xv[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { s[j] = 0.f; xv[j] = 0.f; }
  if (g.in_act) ld8(xin + (size_t)i * 8, xv);     // issued first: overlaps the window loads
  for (int oy = oy_lo; oy <= oy_hi; ++oy) {
    const int hy = min(oy * g.SY + g.KY, g.H) - oy * g.SY;
    for (int ox = ox_lo; ox <= ox_hi; ++ox) {
      const int o = (((n * g.OH + oy) * g.OW + ox) * C8 + cg) * 8;
      float e[8];
      ld8(err_out + o, e);
      if (g.act) {
        float yv[8];
        ld8(yact + o, yv);
#pragma unroll
        for (int j = 0; j < 8; ++j) e[j] *= act_deriv(g.act, 0.f, yv[j]);
      }
      if (is_avg) {
        const int hx = min(ox * g.SX + g.KX, g.W) - ox * g.SX;
        const float inv = 1.f / (float)(hy * hx);
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] += e[j] * inv;
      } else {
        const int4* po = reinterpret_cast<const int4*>(offs + o);
        const int4 a = po[0], b = po[1];
        const int of[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) if (of[j] == self + j) s[j] += e[j];
      }
    }
  }
  if (g.in_act) {
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] *= act_deriv(g.in_act, 0.f, xv[j]);
  }
  st8(err_in + (size_t)i * 8, s);
}

// LRN, thread = (pixel, 8-channel group); needs 2*half <= 8
template <typename T, int half>
__global__ void lrn_vec_k(const T* __restrict__ x, const T* __restrict__ ey, T* __restrict__ out,
                          int pixels, int C, float alpha, float beta, float k, int backward) {
  pdl_wait();
  const int C8 = C >> 3;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pixels * C8) return;
  const int cg = i % C8; const int pix = i / C8;
  const T* px = x + (size_t)pix * C;
  float xv[24], ev[24];
#pragma unroll
  for (int q = 0; q < 24; ++q) { xv[q] = 0.f; ev[q] = 0.f; }
  // local window [cg*8 - 8, cg*8 + 16)
#pragma unroll
  for (int b = 0; b < 3; ++b) {
    const int c0 = (cg - 1 + b) * 8;
    if (c0 >= 0 && c0 < C) {
      float tmp[8];
      ld8(px + c0, tmp);
#pragma unroll
      for (int j = 0; j < 8; ++j) xv[b * 8 + j] = tmp[j];
      if (backward) {
        ld8(ey + (size_t)pix * C + c0, tmp);
#pragma unroll
        for (int j = 0; j < 8; ++j) ev[b * 8 + j] = tmp[j];
      }
    }
  }
  // s[q] for local positions q in [8 - half, 16 + half): window clipped to [0, C) == zeros outside
  // backward: bit 0 = backward pass, bits 8.. = activation code of the PRODUCER whose derivative
  // is folded in (err_input *= f'(x), x = this unit's input = the producer's output; see PoolGeom)
  const int in_act = backward >> 8;
  backward &= 1;
  float res[8];
  if (!backward) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float s = 0.f;
#pragma unroll
      for (int d = -half; d <= half; ++d) { const float v = xv[8 + j + d]; s += v * v; }
      res[j] = xv[8 + j] * __powf(k + alpha * s, -beta);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float acc = 0.f, si = 1.f;
#pragma unroll
      for (int d = -half; d <= half; ++d) {
        const int q = 8 + j + d;
        const int cabs = cg * 8 + j + d;
        if (cabs < 0 || cabs >= C) continue;
        float s = 0.f;
#pragma unroll
        for (int d2 = -half; d2 <= half; ++d2) { const float v = xv[q + d2]; s += v * v; }
        s = k + alpha * s;
        if (d == 0) si = s;
        acc += ev[q] * xv[q] * __powf(s, -beta - 1.f);
      }
      res[j] = ev[8 + j] * __powf(si, -beta) - 2.f * alpha * beta * xv[8 + j] * acc;
      if (in_act) res[j] *= act_deriv(in_act, 0.f, xv[8 + j]);
    }
  }
  st8(out + (size_t)i * 8, res);
}

// ------------------------------------------------------------ fixed-window vectorised kernels
// The generic kernels above walk the window with run-time trip counts, so every window position
// is a separate global-memory round trip (ncu: long_scoreboard-bound, 4-18 us for the CIFAR
// layers). With the window shape a template parameter (3x3 stride 2 and 2x2 stride 2 cover every
// sample config) all loads of a thread are issued before the first use.
template <typename T> struct Raw8;
template <> struct Raw8<__nv_bfloat16> {
  uint4 r;
  __device__ __forceinline__ void load(const __nv_bfloat16* p) { r = *reinterpret_cast<const uint4*>(p); }
  __device__ __forceinline__ void zero() { r = make_uint4(0, 0, 0, 0); }
  __device__ __forceinline__ void unpack(float (&v)[8]) const {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
  }
};
template <> struct Raw8<float> {
  float4 a, b;
  __device__ __forceinline__ void load(const float* p) {
    a = *reinterpret_cast<const float4*>(p); b = *reinterpret_cast<const float4*>(p + 4);
  }
  __device__ __forceinline__ void zero() { a = make_float4(0, 0, 0, 0); b = a; }
  __device__ __forceinline__ void unpack(float (&v)[8]) const {
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
};

template <typename T, int KY, int KX, int SY, int SX>
__global__ void __launch_bounds__(256)
pool_forward_win_k(const T* __restrict__ in, T* __restrict__ out, int* __restrict__ offs, PoolGeom g,
                   int mode) {
  pdl_wait();
  const int C8 = g.C >> 3;
  const int total = g.N * g.OH * g.OW * C8;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cg = i % C8; int t = i / C8;
  const int ox = t % g.OW; t /= g.OW; const int oy = t % g.OH; const int n = t / g.OH;
  const int y1 = oy * SY, x1 = ox * SX;
  const int img = n * g.H * g.W * g.C + cg * 8;
  Raw8<T> raw[KY * KX];
#pragma unroll
  for (int ky = 0; ky < KY; ++ky)
#pragma unroll
    for (int kx = 0; kx < KX; ++kx) {
      const bool ok = (y1 + ky < g.H) && (x1 + kx < g.W);
      if (ok) raw[ky * KX + kx].load(in + img + ((y1 + ky) * g.W + x1 + kx) * g.C);
      else raw[ky * KX + kx].zero();
    }
  float best[8]; int boff[8]; float key[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { best[j] = 0.f; boff[j] = 0; key[j] = -3.0e38f; }
#pragma unroll
  for (int ky = 0; ky < KY; ++ky)
#pragma unroll
    for (int kx = 0; kx < KX; ++kx) {
      if ((y1 + ky < g.H) && (x1 + kx < g.W)) {
        const int o = img + ((y1 + ky) * g.W + x1 + kx) * g.C;
        float v[8];
        raw[ky * KX + kx].unpack(v);
        if (mode == POOL_AVG) {
#pragma unroll
          for (int j = 0; j < 8; ++j) best[j] += v[j];
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float k = (mode == POOL_MAXABS) ? fabsf(v[j]) : v[j];
            if (k > key[j]) { key[j] = k; best[j] = v[j]; boff[j] = o + j; }
          }
        }
      }
    }
  if (mode == POOL_AVG) {
    const int y2 = min(y1 + KY, g.H), x2 = min(x1 + KX, g.W);
    const float inv = 1.f / (float)((y2 - y1) * (x2 - x1));
#pragma unroll
    for (int j = 0; j < 8; ++j) best[j] *= inv;
  } else {
    int4* po = reinterpret_cast<int4*>(offs + (size_t)i * 8);
    po[0] = make_int4(boff[0], boff[1], boff[2], boff[3]);
    po[1] = make_int4(boff[4], boff[5], boff[6], boff[7]);
  }
  if (g.act) {
#pragma unroll
    for (int j = 0; j < 8; ++j) best[j] = act_fwd5(g.act, best[j]);
  }
  st8(out + (size_t)i * 8, best);
}

// Per-kernel ncu timing on B200 (CIFAR layers, bf16): the fixed-window forward kernel is faster
// than the generic one (3.7-4.2 us vs 5.2-5.9 us, pool1 7.1 vs 7.7 us) and is the default;
// ZNICZ_POOL_WIN=0 selects the generic one. A fixed-window backward kernel was slower (pool1 27 us
// vs 17.5 us: 4 positions x (err + offsets + output) held in registers cost more occupancy than
// the serialised round trips it removed), so backward always takes the generic kernel.
static bool pool_win_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("ZNICZ_POOL_WIN"); on = (e && atoi(e) == 0) ? 0 : 1; }
  return on != 0;
}

void launch_pool_forward(const void* in, void* out, int* offs, int N, int H, int W, int C, int OH, int OW,
                         int KY, int KX, int SY, int SX, int mode, const int* rng, bool bf16, int act,
                         cudaStream_t st) {
  PoolGeom g{N, H, W, C, OH, OW, KY, KX, SY, SX, act};
  long long total = (long long)N * OH * OW * C;
  if (mode <= POOL_AVG && C % 8 == 0 && (long long)N * H * W * C < (1LL << 31) &&
      (((uintptr_t)in | (uintptr_t)out | (uintptr_t)offs) & 15) == 0) {
    int gridv = cdiv(total / 8, 256);
    typedef __nv_bfloat16 bf;
    if (pool_win_enabled() && KY == 3 && KX == 3 && SY == 2 && SX == 2) {
      if (bf16) launch_k(pool_forward_win_k<bf, 3, 3, 2, 2>, gridv, 256, 0, st, (const bf*)in, (bf*)out, offs, g, mode);
      else launch_k(pool_forward_win_k<float, 3, 3, 2, 2>, gridv, 256, 0, st, (const float*)in, (float*)out, offs, g, mode);
    } else if (pool_win_enabled() && KY == 2 && KX == 2 && SY == 2 && SX == 2) {
      if (bf16) launch_k(pool_forward_win_k<bf, 2, 2, 2, 2>, gridv, 256, 0, st, (const bf*)in, (bf*)out, offs, g, mode);
      else launch_k(pool_forward_win_k<float, 2, 2, 2, 2>, gridv, 256, 0, st, (const float*)in, (float*)out, offs, g, mode);
    } else if (bf16) launch_k(pool_forward_vec_k<__nv_bfloat16>, gridv, 256, 0, st, (const __nv_bfloat16*)in, (__nv_bfloat16*)out, offs, g, mode);
    else launch_k(pool_forward_vec_k<float>, gridv, 256, 0, st, (const float*)in, (float*)out, offs, g, mode);
    return;
  }
  int grid = cdiv(total, 256);
  if (bf16) launch_k(pool_forward_k<__nv_bfloat16>, grid, 256, 0, st, (const __nv_bfloat16*)in, (__nv_bfloat16*)out, offs, g, mode, rng);
  else launch_k(pool_forward_k<float>, grid, 256, 0, st, (const float*)in, (float*)out, offs, g, mode, rng);
}
void launch_pool_backward(const void* err_out, const int* offs, void* err_in, int N, int H, int W, int C,
                          int OH, int OW, int KY, int KX, int SY, int SX, int is_avg, bool bf16,
                          const void* yact, int act, const void* xin, int in_act, cudaStream_t st) {
  PoolGeom g{N, H, W, C, OH, OW, KY, KX, SY, SX, yact ? act : 0, xin ? in_act : 0};
  long long total = (long long)N * H * W * C;
  typedef __nv_bfloat16 bf;
  if (C % 8 == 0 && total < (1LL << 31) &&
      (((uintptr_t)err_out | (uintptr_t)err_in | (uintptr_t)offs | (uintptr_t)yact | (uintptr_t)xin) & 15) == 0) {
    int gridv = cdiv(total / 8, 256);
    if (bf16) launch_k(pool_backward_vec_k<bf>, gridv, 256, 0, st, (const bf*)err_out, offs, (bf*)err_in, g, is_avg, (const bf*)yact, (const bf*)xin);
    else launch_k(pool_backward_vec_k<float>, gridv, 256, 0, st, (const float*)err_out, offs, (float*)err_in, g, is_avg, (const float*)yact, (const float*)xin);
    return;
  }
  int grid = cdiv(total, 256);
  if (is_avg) {
    if (bf16) launch_k(pool_backward_avg_k<bf>, grid, 256, 0, st, (const bf*)err_out, (bf*)err_in, g, (const bf*)yact, (const bf*)xin);
    else launch_k(pool_backward_avg_k<float>, grid, 256, 0, st, (const float*)err_out, (float*)err_in, g, (const float*)yact, (const float*)xin);
  } else {
    if (bf16) launch_k(pool_backward_max_k<bf>, grid, 256, 0, st, (const bf*)err_out, offs, (bf*)err_in, g, (const bf*)yact, (const bf*)xin);
    else launch_k(pool_backward_max_k<float>, grid, 256, 0, st, (const float*)err_out, offs, (float*)err_in, g, (const float*)yact, (const float*)xin);
  }
}

// ------------------------------------------------------------------------------------ LRN
// y_i = x_i * (k + alpha * sum_{j in win(i)} x_j^2)^-beta  (/root/reference/cuda/normalization.cu)
template <typename T>
__global__ void lrn_forward_k(const T* __restrict__ x, T* __restrict__ y, long long pixels, int C,
                              int half, float alpha, float beta, float k) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pixels * C) return;
  int c = (int)(i % C);
  const T* px = x + (i - c);
  int lo = max(0, c - half), hi = min(C - 1, c + half);
  float s = 0.f;
  for (int j = lo; j <= hi; ++j) { float v = ldf(px + j); s += v * v; }
  s = k + alpha * s;
  stf(y + i, ldf(px + c) * __powf(s, -beta));
}
// eh_i = ey_i s_i^-b - 2ab x_i sum_{j in win(i)} ey_j x_j s_j^(-b-1)
template <typename T>
__global__ void lrn_backward_k(const T* __restrict__ ey, const T* __restrict__ x, T* __restrict__ eh,
                               long long pixels, int C, int half, float alpha, float beta, float k,
                               int in_act) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pixels * C) return;
  int c = (int)(i % C);
  const T* px = x + (i - c);
  const T* pe = ey + (i - c);
  int lo = max(0, c - half), hi = min(C - 1, c + half);
  // sliding subsums for the (up to) 2*half+1 neighbours: recompute (C and n are small)
  float xi = ldf(px + c);
  float acc = 0.f, si = 0.f;
  for (int j = lo; j <= hi; ++j) {
    int jlo = max(0, j - half), jhi = min(C - 1, j + half);
    float s = 0.f;
    for (int q = jlo; q <= jhi; ++q) { float v = ldf(px + q); s += v * v; }
    s = k + alpha * s;
    if (j == c) si = s;
    acc += ldf(pe + j) * ldf(px + j) * __powf(s, -beta - 1.f);
  }
  float r = ldf(pe + c) * __powf(si, -beta) - 2.f * alpha * beta * xi * acc;
  if (in_act) r *= act_deriv(in_act, 0.f, xi);
  stf(eh + i, r);
}

void launch_lrn_forward(const void* x, void* y, long long pixels, int C, int n, float alpha, float beta,
                        float k, bool bf16, cudaStream_t st) {
  if (C % 8 == 0 && (n / 2 == 1 || n / 2 == 2) && pixels * C < (1LL << 31) &&
      (((uintptr_t)x | (uintptr_t)y) & 15) == 0) {
    int gridv = cdiv(pixels * C / 8, 256);
    if (n / 2 == 1) {
      if (bf16) launch_k(lrn_vec_k<__nv_bfloat16, 1>, gridv, 256, 0, st, (const __nv_bfloat16*)x, nullptr, (__nv_bfloat16*)y, (int)pixels, C, alpha, beta, k, 0);
      else launch_k(lrn_vec_k<float, 1>, gridv, 256, 0, st, (const float*)x, nullptr, (float*)y, (int)pixels, C, alpha, beta, k, 0);
    } else {
      if (bf16) launch_k(lrn_vec_k<__nv_bfloat16, 2>, gridv, 256, 0, st, (const __nv_bfloat16*)x, nullptr, (__nv_bfloat16*)y, (int)pixels, C, alpha, beta, k, 0);
      else launch_k(lrn_vec_k<float, 2>, gridv, 256, 0, st, (const float*)x, nullptr, (float*)y, (int)pixels, C, alpha, beta, k, 0);
    }
    return;
  }
  int grid = cdiv(pixels * C, 256);
  if (bf16) launch_k(lrn_forward_k<__nv_bfloat16>, grid, 256, 0, st, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, pixels, C, n / 2, alpha, beta, k);
  else launch_k(lrn_forward_k<float>, grid, 256, 0, st, (const float*)x, (float*)y, pixels, C, n / 2, alpha, beta, k);
}
void launch_lrn_backward(const void* ey, const void* x, void* eh, long long pixels, int C, int n,
                         float alpha, float beta, float k, bool bf16, int in_act, cudaStream_t st) {
  const int bw = 1 | (in_act << 8);
  if (C % 8 == 0 && (n / 2 == 1 || n / 2 == 2) && pixels * C < (1LL << 31) &&
      (((uintptr_t)x | (uintptr_t)ey | (uintptr_t)eh) & 15) == 0) {
    int gridv = cdiv(pixels * C / 8, 256);
    if (n / 2 == 1) {
      if (bf16) launch_k(lrn_vec_k<__nv_bfloat16, 1>, gridv, 256, 0, st, (const __nv_bfloat16*)x, (const __nv_bfloat16*)ey, (__nv_bfloat16*)eh, (int)pixels, C, alpha, beta, k, bw);
      else launch_k(lrn_vec_k<float, 1>, gridv, 256, 0, st, (const float*)x, (const float*)ey, (float*)eh, (int)pixels, C, alpha, beta, k, bw);
    } else {
      if (bf16) launch_k(lrn_vec_k<__nv_bfloat16, 2>, gridv, 256, 0, st, (const __nv_bfloat16*)x, (const __nv_bfloat16*)ey, (__nv_bfloat16*)eh, (int)pixels, C, alpha, beta, k, bw);
      else launch_k(lrn_vec_k<float, 2>, gridv, 256, 0, st, (const float*)x, (const float*)ey, (float*)eh, (int)pixels, C, alpha, beta, k, bw);
    }
    return;
  }
  int grid = cdiv(pixels * C, 256);
  if (bf16) launch_k(lrn_backward_k<__nv_bfloat16>, grid, 256, 0, st, (const __nv_bfloat16*)ey, (const __nv_bfloat16*)x, (__nv_bfloat16*)eh, pixels, C, n / 2, alpha, beta, k, in_act);
  else launch_k(lrn_backward_k<float>, grid, 256, 0, st, (const float*)ey, (const float*)x, (float*)eh, pixels, C, n / 2, alpha, beta, k, in_act);
}

}  // namespace zn
