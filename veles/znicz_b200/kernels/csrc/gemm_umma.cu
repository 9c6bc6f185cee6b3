// tcgen05 / TMEM / TMA GEMM family for sm_100a (bf16 operands, fp32 accumulate in TMEM).
//
//   D[M, N] = sum_k A[m, k] * B[n, k]      (one 128 x BLOCK_N tile per CTA, optional split-K)
//
// Operand sources (template):
//   A_TMA_K   A stored [M][K] (K contiguous)  -> TMA box {64, 128}, K-major SW128 descriptor
//   A_TMA_MN  A stored [K][M] (M contiguous)  -> TMA boxes {64, 64}, MN-major SW128 descriptor
//   A_GATHER_K / A_GATHER_MN: implicit-GEMM convolution; producer warps gather NHWC patches
//   (im2col of x, or the dgrad gather of err_out) as 16-byte chunks straight into the swizzled
//   shared-memory tile — no im2col buffer in HBM (the reference unpacks 16 images at a time into
//   a temp buffer and calls cuBLAS, /root/reference/conv.py:268-297, gd_conv.py:313-423).
//   A_IM2COL_K: the A_GATHER_K operand fetched by TMA in im2col mode instead (see below).
//   B_TMA_K   B stored [N][K];  B_TMA_MN  B stored [K][N].
//
// Warp roles (192 threads): warps 0-3 = gather producers (if any) then epilogue (TMEM -> regs ->
// bias/activation/alpha-beta -> global); warp 4 = TMA producer; warp 5 = TMEM allocator + the
// single thread that issues tcgen05.mma and commits to mbarriers. 4-stage smem ring (3 stages for
// short reductions, see launch_cfg).
//
// This covers: FC forward (TMA_K x TMA_K, fused bias+activation), FC dgrad (TMA_K x TMA_MN,
// alpha/beta), FC wgrad (TMA_MN x TMA_MN), conv fprop (GATHER_K x TMA_K, fused bias+act),
// conv dgrad (GATHER_K x TMA_MN, no atomics), conv wgrad (GATHER_MN x TMA_MN, split-K partials
// that the fused update kernel sums in fixed order).
#include "common.cuh"
#include "umma.cuh"
#include <stdlib.h>

namespace zn {

using namespace umma;

// A_IM2COL_K: the same implicit-GEMM operand as A_GATHER_K, but fetched by TMA in im2col mode
// (one instruction per [128 pixels x 64 channels] block instead of a 128-thread LDGSTS gather) -
// channel counts that are multiples of 64 only.
enum { A_TMA_K = 0, A_TMA_MN = 1, A_GATHER_K = 2, A_GATHER_MN = 3, A_IM2COL_K = 4 };
enum { B_TMA_K = 0, B_TMA_MN = 1 };
enum { G_NONE = 0, G_IM2COL = 1, G_DGRAD = 2 };

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;          // bf16 elements = 128 bytes = one SW128 row
constexpr int STAGES_DEFAULT = 4;   // 3-stage variant for short reductions: see launch_cfg
constexpr int A_BYTES = BLOCK_M * 128;

struct ConvGeomU {
  int N, H, W, C, OH, OW, F, KY, KX, SY, SX, PT, PL;
  int vec;   // 1 when 16-byte chunks never straddle a tap (C % 8 == 0 resp. F % 8 == 0)
  // tap mode (GVEC == 2): a 64-wide block of the reduction index covers ``tpk`` whole taps
  // (inner = 64 / tpk channels each) or a 64-channel slice of one tap (tpk == 1, inner % 64 == 0)
  int tpk, ntaps, inner;
  // wgrad only: 16 bytes holding bf16 {1, 0, 0, 0, 0, 0, 0, 0}. The gathered im2col operand gets a
  // "ones" row at reduction-weight index Kw (first padding row of the last M tile), so that
  // row Kw of the product is sum_pixels err[pixel][f] = the bias gradient - for free.
  const __nv_bfloat16* ones;
};

struct GemmParams {
  int M, N, K;                 // logical GEMM sizes (K = reduction)
  int k_blocks_per_split;      // in BLOCK_K units
  // epilogue
  void* out; int out_bf16; long long ldo; int out_trans;
  const float* bias; int act; float alpha, beta;
  float* bias_out;             // wgrad: row M of the product -> bias_out[blockIdx.z][N] (see ones)
  const __nv_bfloat16* dmul;   // dgrad: out *= f'(dmul[row][col]) - the producer layer's activation
  int dact;                    //        derivative (dmul = this layer's input, same layout as out)
  long long split_stride;      // > 0: fp32 partial [blockIdx.z][...]
  // gather source
  const __nv_bfloat16* gsrc; ConvGeomU g; int gather_kind;
  int gK;                      // valid extent of the gathered K (fprop/dgrad) or M (wgrad) index
  int ktab_n;                  // entries of the gather lookup table (dynamic shared memory)
};

// ---- gather: 8 consecutive "inner" indices of one "pixel" -> 16 bytes ------------------------
// All div/mod of the reduction index is hoisted into a per-CTA shared-memory table built once:
// vec mode   : ktab[k / 8] = (ky << 24) | (kx << 16) | c0     (16-byte chunks never straddle a tap)
// scalar mode: ktab[k]     = (ky << 24) | (kx << 16) | c
constexpr int KTAB = 4096;

struct PixCtx { const __nv_bfloat16* base; int y, x, valid; };

__device__ __forceinline__ PixCtx decode_out_pixel(const __nv_bfloat16* src, const ConvGeomU& g,
                                                   int pix, int limit) {
  // im2col source = x [N,H,W,C]; (y, x) = top-left input coordinate of the patch
  PixCtx c; c.valid = pix < limit;
  const int p = c.valid ? pix : 0;
  const int ox = p % g.OW; const int t = p / g.OW; const int oy = t % g.OH; const int n = t / g.OH;
  c.y = oy * g.SY - g.PT; c.x = ox * g.SX - g.PL;
  c.base = src + (long long)n * g.H * g.W * g.C;
  return c;
}
__device__ __forceinline__ PixCtx decode_in_pixel(const __nv_bfloat16* src, const ConvGeomU& g,
                                                  int pix, int limit) {
  // dgrad source = err_out [N,OH,OW,F]; (y, x) = input pixel + padding
  PixCtx c; c.valid = pix < limit;
  const int p = c.valid ? pix : 0;
  const int ix = p % g.W; const int t = p / g.W; const int iy = t % g.H; const int n = t / g.H;
  c.y = iy + g.PT; c.x = ix + g.PL;
  c.base = src + (long long)n * g.OH * g.OW * g.F;
  return c;
}
__device__ __forceinline__ void build_ktab(int* ktab, const ConvGeomU& g, int kind, int klimit) {
  if (g.tpk > 0) {                                // tap mode: ktab[tap] = (ky << 8) | kx
    for (int e = threadIdx.x; e < g.ntaps; e += blockDim.x)
      ktab[e] = ((e / g.KX) << 8) | (e % g.KX);
    return;
  }
  const int inner = (kind == 1) ? g.C : g.F;      // G_IM2COL : G_DGRAD
  const int step = g.vec ? 8 : 1;
  const int n = min(KTAB, (klimit + step - 1) / step);
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int k = e * step;
    const int c = k % inner; const int tap = k / inner;
    const int kx = tap % g.KX; const int ky = tap / g.KX;
    ktab[e] = (ky << 24) | (kx << 16) | c;
  }
}
__device__ __forceinline__ const __nv_bfloat16* im2col_addr(const ConvGeomU& g, const PixCtx& c, int e) {
  const int iy = c.y + (e >> 24), ix = c.x + ((e >> 16) & 0xff);
  if ((unsigned)iy >= (unsigned)g.H || (unsigned)ix >= (unsigned)g.W) return nullptr;
  return c.base + (iy * g.W + ix) * g.C + (e & 0xffff);
}
__device__ __forceinline__ const __nv_bfloat16* dgrad_addr(const ConvGeomU& g, const PixCtx& c, int e) {
  int ty = c.y - (e >> 24), tx = c.x - ((e >> 16) & 0xff);
  if (g.SY != 1 || g.SX != 1) {
    if (ty < 0 || tx < 0 || (ty % g.SY) || (tx % g.SX)) return nullptr;
    ty /= g.SY; tx /= g.SX;
  }
  if ((unsigned)ty >= (unsigned)g.OH || (unsigned)tx >= (unsigned)g.OW) return nullptr;
  return c.base + (ty * g.OW + tx) * g.F + (e & 0xffff);
}
template <int KIND, int VEC>
__device__ __forceinline__ uint4 gather_chunk(const int* ktab, const ConvGeomU& g, const PixCtx& c,
                                              int k0, int klimit) {
  uint4 z = make_uint4(0, 0, 0, 0);
  if (!c.valid || k0 >= klimit) return z;
  if (VEC) {
    const __nv_bfloat16* p = (KIND == 1) ? im2col_addr(g, c, ktab[k0 >> 3]) : dgrad_addr(g, c, ktab[k0 >> 3]);
    return p ? *reinterpret_cast<const uint4*>(p) : z;
  }
  __nv_bfloat16 v[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int k = k0 + j;
    const __nv_bfloat16* p = nullptr;
    if (k < klimit) p = (KIND == 1) ? im2col_addr(g, c, ktab[k]) : dgrad_addr(g, c, ktab[k]);
    v[j] = p ? *p : __float2bfloat16_rn(0.f);
  }
  return *reinterpret_cast<uint4*>(v);
}

// Tap-mode gather: the 8 chunks (64 reduction indices starting at k0, k0 % 64 == 0) of one pixel.
// One table lookup + one bounds check + one address per *tap*; the chunks of a tap are
// consecutive 16-byte loads. ~6 instructions per chunk instead of ~100 for the generic path.
template <int KIND, int TPK>
__device__ __forceinline__ void gather_taps(uint4 (&nv)[8], const int* ttab, const ConvGeomU& g,
                                            const PixCtx& c, int k0) {
  constexpr int CPT = 8 / TPK;
  int tap0, c0;
  if (TPK == 1) { tap0 = k0 / g.inner; c0 = k0 - tap0 * g.inner; }
  else { tap0 = (k0 >> 6) * TPK; c0 = 0; }
  const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int j = 0; j < TPK; ++j) {
    const int tap = tap0 + j;
    bool ok = c.valid && tap < g.ntaps;
    const int e = ttab[ok ? tap : 0];
    const int ky = e >> 8, kx = e & 0xff;
    int off;
    if (KIND == G_IM2COL) {
      const int iy = c.y + ky, ix = c.x + kx;
      ok = ok && (unsigned)iy < (unsigned)g.H && (unsigned)ix < (unsigned)g.W;
      off = (iy * g.W + ix) * g.C;
    } else {                                      // dgrad, unit stride only
      const int ty = c.y - ky, tx = c.x - kx;
      ok = ok && (unsigned)ty < (unsigned)g.OH && (unsigned)tx < (unsigned)g.OW;
      off = (ty * g.OW + tx) * g.F;
    }
    const uint4* ptr = reinterpret_cast<const uint4*>(c.base + (ok ? off + c0 : 0));
#pragma unroll
    for (int q = 0; q < CPT; ++q) nv[j * CPT + q] = ok ? ptr[q] : z;
  }
}
// Asynchronous variant: the same taps, but every 16-byte chunk is an LDGSTS (cp.async) straight
// into its swizzled shared-memory slot (row_base + ((c8 ^ sw) << 4)); out-of-image chunks are
// zero-filled by the copy itself. No registers are staged and the thread never waits for global
// memory: the stage's full-barrier gets this thread's arrival when its copies have landed, so
// up to STAGES k-blocks of gathers are in flight per thread.
template <int KIND, int TPK, bool ONES = false>
__device__ __forceinline__ void gather_taps_async(uint32_t row_base, int sw, const int* ttab,
                                                  const ConvGeomU& g, const PixCtx& c, int k0) {
  constexpr int CPT = 8 / TPK;
  int tap0, c0;
  if (TPK == 1) { tap0 = k0 / g.inner; c0 = k0 - tap0 * g.inner; }
  else { tap0 = (k0 >> 6) * TPK; c0 = 0; }
#pragma unroll
  for (int j = 0; j < TPK; ++j) {
    const int tap = tap0 + j;
    bool ok = c.valid && tap < g.ntaps;
    const int e = ttab[ok ? tap : 0];
    const int ky = e >> 8, kx = e & 0xff;
    int off;
    if (KIND == G_IM2COL) {
      const int iy = c.y + ky, ix = c.x + kx;
      ok = ok && (unsigned)iy < (unsigned)g.H && (unsigned)ix < (unsigned)g.W;
      off = (iy * g.W + ix) * g.C;
    } else {
      const int ty = c.y - ky, tx = c.x - kx;
      ok = ok && (unsigned)ty < (unsigned)g.OH && (unsigned)tx < (unsigned)g.OW;
      off = (ty * g.OW + tx) * g.F;
    }
    // ONES: this 64-wide block holds reduction-weight index Kw (see ConvGeomU::ones) - only the
    // wgrad kernel instantiates it, and only for the one block of the last M tile that needs it
    const bool one = ONES && c.valid && tap == g.ntaps && c0 == 0;
    const __nv_bfloat16* ptr = one ? g.ones : c.base + (ok ? off + c0 : 0);
    const uint32_t nbytes = ok ? 16u : 0u;
#pragma unroll
    for (int q = 0; q < CPT; ++q) {
      const int c8 = j * CPT + q;
      cp_async_16(row_base + (uint32_t)((c8 ^ sw) << 4), one ? ptr : ptr + q * 8,
                  (one && q == 0) ? 16u : nbytes);
    }
  }
}
template <int KIND, bool ONES = false>
__device__ __forceinline__ void gather_row_async(uint32_t row_base, int sw, const int* ktab,
                                                 const ConvGeomU& g, const PixCtx& c, int k0) {
  switch (g.tpk) {
    case 1: gather_taps_async<KIND, 1, ONES>(row_base, sw, ktab, g, c, k0); break;
    case 2: gather_taps_async<KIND, 2, ONES>(row_base, sw, ktab, g, c, k0); break;
    case 4: gather_taps_async<KIND, 4, ONES>(row_base, sw, ktab, g, c, k0); break;
    default: gather_taps_async<KIND, 8, ONES>(row_base, sw, ktab, g, c, k0); break;
  }
}

template <int KIND, int GVEC>
__device__ __forceinline__ void gather_row(uint4 (&nv)[8], const int* ktab, const ConvGeomU& g,
                                           const PixCtx& c, int k0, int klimit) {
  if (GVEC == 2) {
    switch (g.tpk) {
      case 1: gather_taps<KIND, 1>(nv, ktab, g, c, k0); break;
      case 2: gather_taps<KIND, 2>(nv, ktab, g, c, k0); break;
      case 4: gather_taps<KIND, 4>(nv, ktab, g, c, k0); break;
      default: gather_taps<KIND, 8>(nv, ktab, g, c, k0); break;
    }
  } else {
#pragma unroll
    for (int c8 = 0; c8 < 8; ++c8) nv[c8] = gather_chunk<KIND, GVEC>(ktab, g, c, k0 + c8 * 8, klimit);
  }
}

template <int BLOCK_N, int B_MODE>
__host__ __device__ constexpr int b_bytes() {
  return B_MODE == B_TMA_K ? BLOCK_N * 128 : ((BLOCK_N + 63) / 64) * 8192;
}

// generic (rare) epilogue element: split-K partials, transposed / fp32 / alpha-beta outputs.
// Deliberately not inlined: keeps the unrolled epilogue small.
__device__ __noinline__ void epi_store_slow(const GemmParams& p, int row, int n, float v, int z) {
  const long long o = p.out_trans ? (long long)n * p.ldo + row : (long long)row * p.ldo + n;
  if (p.split_stride > 0) {
    reinterpret_cast<float*>(p.out)[(long long)z * p.split_stride + o] = v;
    return;
  }
  v *= p.alpha;
  if (p.bias) v += p.bias[n];
  v = act_fwd5(p.act, v);
  if (p.out_bf16) {
    __nv_bfloat16* q = reinterpret_cast<__nv_bfloat16*>(p.out) + o;
    if (p.beta != 0.f) v += p.beta * __bfloat162float(*q);
    *q = __float2bfloat16_rn(v);
  } else {
    float* q = reinterpret_cast<float*>(p.out) + o;
    if (p.beta != 0.f) v += p.beta * *q;
    *q = v;
  }
}

template <int BLOCK_N, int B_MODE, int STAGES>
__host__ __device__ constexpr int min_ctas() {
  return (2 * (STAGES * (A_BYTES + b_bytes<BLOCK_N, B_MODE>()) + 2048) <= 227 * 1024) ? 2 : 1;
}

// FP8: operands are e4m3 bytes (TMA / TMA, both K-major): the byte geometry of a stage is the
// same (128-byte swizzled rows), a k-block is 128 elements and every MMA consumes 32 of them.
template <int BLOCK_N, int A_MODE, int B_MODE, int GKIND, int GVEC, int STAGES, bool FP8 = false>
__global__ void __launch_bounds__(192, (min_ctas<BLOCK_N, B_MODE, STAGES>()))
gemm_umma_k(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
            const GemmParams p) {
  constexpr int B_BYTES = b_bytes<BLOCK_N, B_MODE>();
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr bool A_GATHER = (A_MODE == A_GATHER_K || A_MODE == A_GATHER_MN);
  constexpr bool A_MN = (A_MODE == A_TMA_MN || A_MODE == A_GATHER_MN);
  constexpr bool B_MN = (B_MODE == B_TMA_MN);
  constexpr uint32_t TMEM_COLS = BLOCK_N < 32 ? 32 : BLOCK_N;
  constexpr uint32_t IDESC = FP8 ? make_idesc_e4m3(BLOCK_M, BLOCK_N)
                                 : make_idesc_bf16(BLOCK_M, BLOCK_N, A_MN ? 1 : 0, B_MN ? 1 : 0);
  constexpr int KBLK = FP8 ? 2 * BLOCK_K : BLOCK_K;      // elements per k-block (128 bytes per row)
  static_assert(!FP8 || (A_MODE == A_TMA_K && B_MODE == B_TMA_K), "fp8: TMA K-major operands only");
  constexpr uint32_t TX_BYTES = (A_GATHER ? 0 : A_BYTES) + B_BYTES;

  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[STAGES];
  __shared__ __align__(8) uint64_t empty_bar[STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_base_smem;

  // 1024-byte aligned tile area (SWIZZLE_128B atoms are 1024 B)
  uint8_t* tiles = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  // behind the ring: the gather lookup table (only as many entries as this geometry needs - a
  // fixed-size table cost the BLOCK_N = 64 conv kernels their second CTA per SM) and the tile's
  // bias slice (the epilogue would otherwise wait on one L2 round trip per 8 columns)
  int* const ktab = reinterpret_cast<int*>(tiles + (size_t)STAGES * STAGE_BYTES);
  float* const s_bias = reinterpret_cast<float*>(ktab + ((p.ktab_n + 3) & ~3));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * BLOCK_M, n0 = blockIdx.x * BLOCK_N;
  const int total_kb = (p.K + KBLK - 1) / KBLK;
  const int kb_begin = blockIdx.z * p.k_blocks_per_split;
  const int kb_end = min(total_kb, kb_begin + p.k_blocks_per_split);
  const int num_kb = max(0, kb_end - kb_begin);

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], (A_GATHER ? 128u : 0u) + 1u);
      mbar_init(&empty_bar[s], 1u);
    }
    mbar_init(&tmem_full_bar, 1u);
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) {
    if (!A_GATHER) tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 5) {
    tmem_alloc(&tmem_base_smem, TMEM_COLS);
    tmem_relinquish();
  }
  if (A_GATHER) build_ktab(ktab, p.g, GKIND, p.gK);
  pdl_wait();      // everything above overlapped the previous kernel's tail; global reads start here
  if (threadIdx.x < BLOCK_N) {
    const int n = blockIdx.x * BLOCK_N + threadIdx.x;
    s_bias[threadIdx.x] = (p.bias && n < p.N) ? __ldg(p.bias + n) : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (warp == 4) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      for (int i = 0; i < num_kb; ++i) {
        const int s = i % STAGES; const uint32_t ph = (i / STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        uint8_t* sa = tiles + (size_t)s * STAGE_BYTES;
        uint8_t* sb = sa + A_BYTES;
        const int k0 = (kb_begin + i) * KBLK;
        mbar_arrive_expect_tx(&full_bar[s], TX_BYTES);
        if (A_MODE == A_IM2COL_K) {
          // conv fprop / stride-1 dgrad: tile rows = pixels m0 .. m0 + 127, k-block = 64
          // channels of ONE filter tap
          const ConvGeomU& g = p.g;
          const int tap = k0 / g.inner, c0 = k0 - tap * g.inner;
          const int ky = tap / g.KX, kx = tap - ky * g.KX;
          int w0, h0, n, ow, oh;
          if (GKIND == G_IM2COL) {
            const int q = m0 % g.OW; const int t2 = m0 / g.OW;
            const int pr = t2 % g.OH; n = t2 / g.OH;
            w0 = q * g.SX - g.PL; h0 = pr * g.SY - g.PT; ow = kx; oh = ky;
          } else {                                   // dgrad: correlation with the flipped filter
            const int ix = m0 % g.W; const int t2 = m0 / g.W;
            const int iy = t2 % g.H; n = t2 / g.H;
            w0 = ix - (g.KX - 1 - g.PL); h0 = iy - (g.KY - 1 - g.PT);
            ow = g.KX - 1 - kx; oh = g.KY - 1 - ky;
          }
          tma_load_im2col_4d(sa, &tmap_a, &full_bar[s], c0, w0, h0, n, (uint16_t)ow, (uint16_t)oh);
        } else if (A_MODE == A_TMA_K) {
          tma_load_2d(sa, &tmap_a, &full_bar[s], k0, m0);
        } else if (A_MODE == A_TMA_MN) {
          tma_load_2d(sa, &tmap_a, &full_bar[s], m0, k0);
          tma_load_2d(sa + 8192, &tmap_a, &full_bar[s], m0 + 64, k0);
        }
        if (B_MODE == B_TMA_K) {
          tma_load_2d(sb, &tmap_b, &full_bar[s], k0, n0);
        } else {
#pragma unroll
          for (int j = 0; j < (BLOCK_N + 63) / 64; ++j)
            tma_load_2d(sb + j * 8192, &tmap_b, &full_bar[s], n0 + j * 64, k0);
        }
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      for (int i = 0; i < num_kb; ++i) {
        const int s = i % STAGES; const uint32_t ph = (i / STAGES) & 1;
        mbar_wait(&full_bar[s], ph);
        if (A_GATHER && GVEC == 2) fence_proxy_async_smem();   // LDGSTS data -> async proxy
        tc_fence_after();
        const uint32_t sa = smem_u32(tiles + (size_t)s * STAGE_BYTES);
        const uint32_t sb = sa + A_BYTES;
#pragma unroll
        for (int k = 0; k < BLOCK_K / 16; ++k) {
          // K-major: 16 bf16 = 32 B along the swizzled row. MN-major: 16 k-rows = 2 atoms.
          const uint64_t da = A_MN ? make_smem_desc(sa + k * 2048, 8192, 1024)
                                   : make_smem_desc(sa + k * 32, 16, 1024);
          const uint64_t db = B_MN ? make_smem_desc(sb + k * 2048, 8192, 1024)
                                   : make_smem_desc(sb + k * 32, 16, 1024);
          if (FP8) mma_f8(tmem_base, da, db, IDESC, (i > 0 || k > 0) ? 1u : 0u);
          else mma_f16(tmem_base, da, db, IDESC, (i > 0 || k > 0) ? 1u : 0u);
        }
        mma_commit(&empty_bar[s]);          // smem slot reusable once these MMAs retire
        if (i == num_kb - 1) mma_commit(&tmem_full_bar);   // the accumulator is complete
      }
    }
  } else {
    // ===================== gather producers (if any), then epilogue (warps 0-3) ================
    if (A_GATHER) {
      const int t = threadIdx.x;            // 0..127
      if (A_MODE == A_GATHER_K) {
        // tile row r = t is GEMM row m0 + t (a pixel); chunks run over the reduction index
        const PixCtx ctx = (GKIND == G_IM2COL) ? decode_out_pixel(p.gsrc, p.g, m0 + t, p.M)
                                               : decode_in_pixel(p.gsrc, p.g, m0 + t, p.M);
        if (GVEC == 2) {
          // asynchronous gather: issue the LDGSTS of a stage as soon as its slot is free; the
          // stage's full barrier is armed by the copies themselves
#pragma unroll 1
          for (int i = 0; i < num_kb; ++i) {
            const int s = i % STAGES; const uint32_t ph = (i / STAGES) & 1;
            mbar_wait(&empty_bar[s], ph ^ 1);
            const uint32_t row_base = smem_u32(tiles + (size_t)s * STAGE_BYTES) + t * 128;
            gather_row_async<GKIND>(row_base, t & 7, ktab, p.g, ctx, (kb_begin + i) * BLOCK_K);
            cp_async_mbar_arrive_noinc(&full_bar[s]);
          }
        } else {
        uint4 v[8], nv[8];
        // software pipeline with ONE load site: iteration i issues the global loads of stage
        // i + 1 and then publishes stage i (whose loads were issued one iteration earlier)
#pragma unroll 1
        for (int i = -1; i < num_kb; ++i) {
          if (i + 1 < num_kb) {
            const int k0 = (kb_begin + i + 1) * BLOCK_K;
            gather_row<GKIND, GVEC>(nv, ktab, p.g, ctx, k0, p.gK);
          }
          if (i >= 0) {
            const int s = i % STAGES; const uint32_t ph = (i / STAGES) & 1;
            mbar_wait(&empty_bar[s], ph ^ 1);
            uint8_t* sa = tiles + (size_t)s * STAGE_BYTES;
#pragma unroll
            for (int c8 = 0; c8 < 8; ++c8)
              *reinterpret_cast<uint4*>(sa + t * 128 + ((c8 ^ (t & 7)) << 4)) = v[c8];
            fence_proxy_async_smem();
            mbar_arrive(&full_bar[s]);
          }
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8) v[c8] = nv[c8];
        }
        }
      } else {
        // A_GATHER_MN (conv wgrad): tile = [64 reduction rows (pixels)][128 m (kidx)];
        // thread -> reduction row kr = t % 64, 64-wide m block = t / 64 (8 chunks of 8 kidx)
        const int kr = t & 63, mblk = t >> 6;
        // only the 64-wide m block that contains index Kw carries the bias "ones" row
        const int kk0 = m0 + mblk * 64;
        const bool has_one = p.g.ones != nullptr && kk0 <= p.gK && p.gK < kk0 + 64;
        if (GVEC == 2) {
#pragma unroll 1
          for (int i = 0; i < num_kb; ++i) {
            const int s = i % STAGES; const uint32_t ph = (i / STAGES) & 1;
            mbar_wait(&empty_bar[s], ph ^ 1);
            const int pix = (kb_begin + i) * BLOCK_K + kr;
            const PixCtx ctx = decode_out_pixel(p.gsrc, p.g, pix, p.K);
            const uint32_t row_base =
                smem_u32(tiles + (size_t)s * STAGE_BYTES) + mblk * 8192 + kr * 128;
            if (has_one) gather_row_async<G_IM2COL, true>(row_base, kr & 7, ktab, p.g, ctx, kk0);
            else gather_row_async<G_IM2COL, false>(row_base, kr & 7, ktab, p.g, ctx, kk0);
            cp_async_mbar_arrive_noinc(&full_bar[s]);
          }
        } else {
        uint4 v[8], nv[8];
#pragma unroll 1
        for (int i = -1; i < num_kb; ++i) {
          if (i + 1 < num_kb) {
            const int pix = (kb_begin + i + 1) * BLOCK_K + kr;
            const PixCtx ctx = decode_out_pixel(p.gsrc, p.g, pix, p.K);
            gather_row<G_IM2COL, GVEC>(nv, ktab, p.g, ctx, m0 + mblk * 64, p.gK);
          }
          if (i >= 0) {
            const int s = i % STAGES; const uint32_t ph = (i / STAGES) & 1;
            mbar_wait(&empty_bar[s], ph ^ 1);
            uint8_t* sa = tiles + (size_t)s * STAGE_BYTES;
#pragma unroll
            for (int c8 = 0; c8 < 8; ++c8)
              *reinterpret_cast<uint4*>(sa + mblk * 8192 + kr * 128 + ((c8 ^ (kr & 7)) << 4)) = v[c8];
            fence_proxy_async_smem();
            mbar_arrive(&full_bar[s]);
          }
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8) v[c8] = nv[c8];
        }
        }
      }
    }
    // ===================== epilogue =====================
    if (num_kb > 0) {
      mbar_wait(&tmem_full_bar, 0);
      tc_fence_after();
    }
    // The epilogue runs once per tile, so every instruction of it is an instruction-cache miss:
    // the former 32-column unrolled version (4-5 K SASS instructions) cost ~10 us per tile on
    // fetch stalls alone. This one is a rolled loop over 8-column chunks - TMEM loads double
    // buffered (the next chunk is in flight while this one is stored) - with the output mode
    // decided once per thread; the loop body is a few hundred instructions, fetched once.
    enum { EPI_BF16, EPI_RAW_T, EPI_RAW, EPI_SLOW, EPI_NONE, EPI_BIASROW, EPI_F32 };
    const int row = m0 + warp * 32 + lane;
    const bool raw32 = !p.out_bf16 && p.beta == 0.f && p.alpha == 1.f && !p.bias && p.act == 0;
    float* const rbase = reinterpret_cast<float*>(p.out) +
                         (p.split_stride > 0 ? (long long)blockIdx.z * p.split_stride : 0LL);
    int mode;
    if (row >= p.M) mode = (p.bias_out && row == p.M) ? EPI_BIASROW : EPI_NONE;
    else if (p.split_stride == 0 && !p.out_trans && p.out_bf16 && p.beta == 0.f) mode = EPI_BF16;
    else if (p.split_stride == 0 && !p.out_trans && !p.out_bf16 && p.beta == 0.f && !raw32)
      mode = EPI_F32;        // fp32 row-major with bias / activation (LSTM gate pre-activations,
                             // softmax logits): same inline path as bf16, fp32 stores
    else if (raw32 && p.out_trans) mode = EPI_RAW_T;
    else if (raw32 && (p.ldo & 3) == 0 && (reinterpret_cast<uintptr_t>(rbase) & 15) == 0)
      mode = EPI_RAW;
    else mode = EPI_SLOW;
    const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);

    auto emit = [&](const uint32_t (&r)[8], int c0) {
      const int nb = n0 + c0;
      if (mode == EPI_NONE) return;
      if (mode == EPI_BIASROW) {       // product row M = column sums of err (see ConvGeomU::ones)
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (nb + j < p.N) p.bias_out[(long long)blockIdx.z * p.N + nb + j] = __uint_as_float(r[j]);
        return;
      }
      if (mode == EPI_BF16 || mode == EPI_F32) {
        float v[8];
        {
          const float4 b0 = *reinterpret_cast<const float4*>(s_bias + c0);
          const float4 b1 = *reinterpret_cast<const float4*>(s_bias + c0 + 4);
          v[0] = b0.x; v[1] = b0.y; v[2] = b0.z; v[3] = b0.w;
          v[4] = b1.x; v[5] = b1.y; v[6] = b1.z; v[7] = b1.w;
        }
        // activation selected once per chunk (not per element): the executed path stays short
        switch (p.act) {
          // out = act(alpha * acc + bias): alpha is the operand de-scaling of the fp8 path and the
          // err_input_alpha of dgrad (no bias, linear); every other caller passes alpha = 1
          case ACT_LINEAR:
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaf(__uint_as_float(r[j]), p.alpha, v[j]);
            break;
          case ACT_STRICT_RELU:
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(__uint_as_float(r[j]), p.alpha, v[j]), 0.f);
            break;
          case ACT_TANH:
#pragma unroll
            for (int j = 0; j < 8; ++j)
              v[j] = 1.7159f * tanh_approx(0.6666f * fmaf(__uint_as_float(r[j]), p.alpha, v[j]));
            break;
          default:
#pragma unroll
            for (int j = 0; j < 8; ++j)
              v[j] = act_fwd5_fast(p.act, fmaf(__uint_as_float(r[j]), p.alpha, v[j]));
        }
        if (p.dmul != nullptr && mode == EPI_BF16) {
          // err_input *= f'(x): x has the layout of the output (row pitch ldo)
          const __nv_bfloat16* dx = p.dmul + (long long)row * p.ldo + nb;
          if (nb + 8 <= p.N && (p.ldo & 7) == 0) {
            float xv[8];
            ld8(dx, xv);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] *= act_deriv(p.dact, 0.f, xv[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (nb + j < p.N) v[j] *= act_deriv(p.dact, 0.f, __bfloat162float(dx[j]));
          }
        }
        if (mode == EPI_F32) {
          float* qf = reinterpret_cast<float*>(p.out) + (long long)row * p.ldo + nb;
          if (nb + 8 <= p.N && (p.ldo & 3) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0) {
            reinterpret_cast<float4*>(qf)[0] = make_float4(v[0], v[1], v[2], v[3]);
            reinterpret_cast<float4*>(qf)[1] = make_float4(v[4], v[5], v[6], v[7]);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (nb + j < p.N) qf[j] = v[j];
          }
          return;
        }
        // bf16 pack: one 16-byte store per 8 outputs
        __nv_bfloat16* q = reinterpret_cast<__nv_bfloat16*>(p.out) + (long long)row * p.ldo + nb;
        if (nb + 8 <= p.N && (p.ldo & 7) == 0) {
          st8(q, v);
        } else {                       // ragged last chunk / row pitch not a multiple of 16 bytes
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (nb + j < p.N) q[j] = __float2bfloat16_rn(v[j]);
        }
      } else if (mode == EPI_RAW_T) {
        // raw fp32 (split-K partials / FC weight gradients), transposed: for a fixed column the
        // 32 lanes hold consecutive rows = one coalesced 128-byte store per column
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (nb + j < p.N) rbase[(long long)(nb + j) * p.ldo + row] = __uint_as_float(r[j]);
      } else if (mode == EPI_RAW && nb + 8 <= p.N) {
        float4* q = reinterpret_cast<float4*>(rbase + (long long)row * p.ldo + nb);
        q[0] = make_float4(__uint_as_float(r[0]), __uint_as_float(r[1]), __uint_as_float(r[2]),
                           __uint_as_float(r[3]));
        q[1] = make_float4(__uint_as_float(r[4]), __uint_as_float(r[5]), __uint_as_float(r[6]),
                           __uint_as_float(r[7]));
      } else if (raw32) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (nb + j < p.N) rbase[(long long)row * p.ldo + nb + j] = __uint_as_float(r[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)     // (static indices: r stays in registers)
          if (nb + j < p.N) epi_store_slow(p, row, nb + j, __uint_as_float(r[j]), blockIdx.z);
      }
    };

    // rb receives the TMEM load of the next chunk while the current one (ra) is converted and
    // stored; a single copy of the emit code serves every chunk
    uint32_t ra[8], rb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) rb[j] = 0u;
    if (num_kb > 0) tmem_ld_32x8(trow, rb);
#pragma unroll 1
    for (int c0 = 0; c0 < BLOCK_N; c0 += 8) {
      if (n0 + c0 >= p.N) break;     // chunk beyond the last column
      if (num_kb > 0) tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 8; ++j) ra[j] = rb[j];
      if (num_kb > 0 && c0 + 8 < BLOCK_N) tmem_ld_32x8(trow + c0 + 8, rb);
      emit(ra, c0);
    }
    if (num_kb > 0) tmem_ld_wait();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p)
      return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D bf16 tensor map: inner dim `inner` (contiguous), outer dim `outer`, row pitch ld elements,
// box {64, box_rows}, SWIZZLE_128B, OOB -> zeros.
static int make_map(CUtensorMap* m, const void* ptr, long long inner, long long outer, long long ld,
                    int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return -1;
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)(ld * 2)};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}

// ---- im2col-mode tensor map over an NHWC bf16 tensor [N][H][W][C] --------------------------------
// Filter-window base positions along w run from lower_w to W + upper_w (exclusive) in steps of the
// traversal stride; upper_* are chosen by the callers so that exactly OW x OH positions exist.
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeIm2colFn get_encode_im2col() {
  static EncodeIm2colFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &q) != cudaSuccess || !p)
      return nullptr;
    fn = reinterpret_cast<EncodeIm2colFn>(p);
  }
  return fn;
}
static int make_map_im2col(CUtensorMap* m, const void* ptr, int N, int H, int W, int C, int lower_w,
                           int lower_h, int upper_w, int upper_h, int stride_w, int stride_h, int pixels) {
  EncodeIm2colFn enc = get_encode_im2col();
  if (!enc) return -1;
  if (lower_w < -128 || lower_h < -128 || upper_w < -128 || upper_h < -128 || lower_w > 127 ||
      lower_h > 127 || upper_w > 127 || upper_h > 127 || stride_w > 8 || stride_h > 8)
    return -7;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  int lower[2] = {lower_w, lower_h};
  int upper[2] = {upper_w, upper_h};
  cuuint32_t estr[4] = {1u, (cuuint32_t)stride_w, (cuuint32_t)stride_h, 1u};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, lower,
                   upper, 64u, (cuuint32_t)pixels, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}
static long long g_im2col_launches = 0;
long long im2col_tma_launches() { return g_im2col_launches; }
// ZNICZ_IM2COL_TMA=0 keeps the LDGSTS gather producers (A/B measurements, fallback)
static bool im2col_tma_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("ZNICZ_IM2COL_TMA"); on = (e && atoi(e) == 0) ? 0 : 1; }
  return on != 0;
}

template <int BN, int AM, int BM, int GK, int GV, int NS>
static int launch_stages(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p_in, dim3 grid,
                         cudaStream_t st) {
  constexpr int ring = NS * (A_BYTES + b_bytes<BN, BM>()) + 1024;
  constexpr bool gather = (AM == A_GATHER_K || AM == A_GATHER_MN);
  constexpr int smem_max = ring + (gather ? KTAB * 4 : 0) + BN * 4 + 16;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_umma_k<BN, AM, BM, GK, GV, NS>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  GemmParams p = p_in;
  p.ktab_n = 0;
  if (gather) {       // must match build_ktab()
    const int step = p.g.vec ? 8 : 1;
    p.ktab_n = p.g.tpk > 0 ? p.g.ntaps : std::min(KTAB, (p.gK + step - 1) / step);
  }
  const int smem = ring + ((p.ktab_n + 3) & ~3) * 4 + BN * 4;
  launch_k(gemm_umma_k<BN, AM, BM, GK, GV, NS>, grid, 192, smem, st, ta, tb, p);
  return (int)cudaGetLastError();
}

template <int BN, int AM, int BM, int GK, int GV>
static int launch_cfg(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, int splits,
                      cudaStream_t st) {
  dim3 grid((p.N + BN - 1) / BN, (p.M + BLOCK_M - 1) / BLOCK_M, splits);
  // Short reductions (K <= 4 k-blocks, e.g. a 5x5 first layer on 8 padded channels) in grids of
  // several waves: a 3-stage ring already holds almost the whole K and is small enough for a
  // third CTA per SM (ncu: these kernels are latency-bound at 15 % warp occupancy).
  if constexpr (AM == A_GATHER_K && GV == 2 && BN <= 64) {
    const long long ctas = (long long)grid.x * grid.y * grid.z;
    static int s3 = -1;
    if (s3 < 0) { const char* e = getenv("ZNICZ_UMMA_S3"); s3 = e ? atoi(e) : 1; }
    if (s3 && p.k_blocks_per_split <= 4 && ctas > 2 * 148)
      return launch_stages<BN, AM, BM, GK, GV, 3>(ta, tb, p, grid, st);
  }
  return launch_stages<BN, AM, BM, GK, GV, STAGES_DEFAULT>(ta, tb, p, grid, st);
}

// B K-major: BLOCK_N in {16, 32, 64, 128}; B MN-major: {64, 128}
template <int AM, int BM, int GK, int GV>
static int launch_bn(int bn, const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p,
                     int splits, cudaStream_t st) {
  if constexpr (BM == B_TMA_K) {
    switch (bn) {
      case 16: return launch_cfg<16, AM, BM, GK, GV>(ta, tb, p, splits, st);
      case 32: return launch_cfg<32, AM, BM, GK, GV>(ta, tb, p, splits, st);
      case 64: return launch_cfg<64, AM, BM, GK, GV>(ta, tb, p, splits, st);
      case 128: return launch_cfg<128, AM, BM, GK, GV>(ta, tb, p, splits, st);
      default: return -2;
    }
  } else {
    switch (bn) {
      case 64: return launch_cfg<64, AM, BM, GK, GV>(ta, tb, p, splits, st);
      case 128: return launch_cfg<128, AM, BM, GK, GV>(ta, tb, p, splits, st);
      default: return -2;
    }
  }
}

static int pick_bn(int N) { return N <= 16 ? 16 : (N <= 32 ? 32 : (N <= 64 ? 64 : 128)); }

int pair_wgrad_splits(int, int, int, int);      // gemm_pair.cu

int umma_pick_splits(int M, int N, int K, int max_splits) {
  {
    // conv wgrad shapes served by the 2-CTA kernel (gemm_pair.cu) want ~74 work items
    const int sp = pair_wgrad_splits(M, N, K, max_splits);
    if (sp > 0) return sp;
  }
  int bn = pick_bn(N);
  if (bn < 64) bn = 64;
  long long tiles = (long long)((M + BLOCK_M - 1) / BLOCK_M) * ((N + bn - 1) / bn);
  int kb = (K + BLOCK_K - 1) / BLOCK_K;
  int s = (int)((148 + tiles - 1) / tiles);
  if (s > kb) s = kb;
  if (s > max_splits) s = max_splits;
  return s < 1 ? 1 : s;
}

// Dense GEMM. a_mn = 0: A stored [M][lda] (K contiguous); 1: A stored [K][lda] (M contiguous).
// b_mn = 0: B stored [N][ldb] (K contiguous); 1: B stored [K][ldb] (N contiguous).
// Returns 0 on success; non-zero = not launched (caller must fall back loudly).
int launch_gemm_umma(const void* a, long long lda, int a_mn, const void* b, long long ldb, int b_mn,
                     void* out, int out_bf16, long long ldo, int out_trans, int M, int N, int K,
                     const float* bias, int act, float alpha, float beta, int splits,
                     long long split_stride, cudaStream_t st) {
  if ((lda % 8) || (ldb % 8) || ((uintptr_t)a & 15) || ((uintptr_t)b & 15)) return -3;
  CUtensorMap ta, tb;
  int bn = pick_bn(N);
  if (b_mn && bn < 64) bn = 64;
  int r;
  if (a_mn) r = make_map(&ta, a, M, K, lda, 64); else r = make_map(&ta, a, K, M, lda, BLOCK_M);
  if (r) return r;
  if (b_mn) r = make_map(&tb, b, N, K, ldb, 64); else r = make_map(&tb, b, K, N, ldb, bn);
  if (r) return r;
  GemmParams p{};
  p.M = M; p.N = N; p.K = K;
  int total_kb = (K + BLOCK_K - 1) / BLOCK_K;
  if (splits < 1) splits = 1;
  p.k_blocks_per_split = (total_kb + splits - 1) / splits;
  splits = (total_kb + p.k_blocks_per_split - 1) / p.k_blocks_per_split;
  p.out = out; p.out_bf16 = out_bf16; p.ldo = ldo; p.out_trans = out_trans;
  p.bias = bias; p.act = act; p.alpha = alpha; p.beta = beta; p.split_stride = split_stride;
  p.gather_kind = G_NONE;
  if (!a_mn && !b_mn) return launch_bn<A_TMA_K, B_TMA_K, 0, 0>(bn, ta, tb, p, splits, st);
  // MN-major B tiles are built from 64-wide swizzle atoms: never go below UMMA_N = 64 there
  if (!a_mn && b_mn) return launch_bn<A_TMA_K, B_TMA_MN, 0, 0>(bn, ta, tb, p, splits, st);
  if (a_mn && !b_mn) return launch_bn<A_TMA_MN, B_TMA_K, 0, 0>(bn, ta, tb, p, splits, st);
  return launch_bn<A_TMA_MN, B_TMA_MN, 0, 0>(bn, ta, tb, p, splits, st);
}

// ---- fp8 (e4m3 x e4m3 -> fp32 accumulate) GEMM: out = act(alpha * a . b^T + bias) -------------
static int make_map_u8(CUtensorMap* m, const void* ptr, long long inner, long long outer, long long ld,
                       int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return -1;
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)ld};
  cuuint32_t box[2] = {128u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(ptr), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}
template <int BN>
static int launch_fp8_bn(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, dim3 grid,
                         cudaStream_t st) {
  constexpr int ring = STAGES_DEFAULT * (A_BYTES + b_bytes<BN, B_TMA_K>()) + 1024;
  constexpr int smem = ring + BN * 4 + 16;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_umma_k<BN, A_TMA_K, B_TMA_K, 0, 0, STAGES_DEFAULT, true>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  launch_k(gemm_umma_k<BN, A_TMA_K, B_TMA_K, 0, 0, STAGES_DEFAULT, true>, grid, 192, smem, st, ta, tb, p);
  return (int)cudaGetLastError();
}
// a [M][lda] e4m3, b [N][ldb] e4m3 (both K-major, ld % 16 == 0); alpha carries 1/(scale_a*scale_b)
int launch_gemm_fp8(const void* a, long long lda, const void* b, long long ldb, void* out, int out_bf16,
                    long long ldo, int M, int N, int K, const float* bias, int act, float alpha,
                    cudaStream_t st) {
  if ((lda % 16) || (ldb % 16) || ((uintptr_t)a & 15) || ((uintptr_t)b & 15)) return -3;
  CUtensorMap ta, tb;
  const int bn = pick_bn(N);
  int r = make_map_u8(&ta, a, K, M, lda, BLOCK_M);
  if (r) return r;
  r = make_map_u8(&tb, b, K, N, ldb, bn);
  if (r) return r;
  GemmParams p{};
  p.M = M; p.N = N; p.K = K;
  p.k_blocks_per_split = (K + 2 * BLOCK_K - 1) / (2 * BLOCK_K);
  p.out = out; p.out_bf16 = out_bf16; p.ldo = ldo; p.out_trans = 0;
  p.bias = bias; p.act = act; p.alpha = alpha; p.beta = 0.f; p.split_stride = 0;
  p.gather_kind = G_NONE;
  dim3 grid((N + bn - 1) / bn, (M + BLOCK_M - 1) / BLOCK_M, 1);
  switch (bn) {
    case 16: return launch_fp8_bn<16>(ta, tb, p, grid, st);
    case 32: return launch_fp8_bn<32>(ta, tb, p, grid, st);
    case 64: return launch_fp8_bn<64>(ta, tb, p, grid, st);
    default: return launch_fp8_bn<128>(ta, tb, p, grid, st);
  }
}

static ConvGeomU geom(int N, int H, int W, int C, int OH, int OW, int F, int KY, int KX, int SY, int SX,
                      int PT, int PL, int vec) {
  ConvGeomU g{N, H, W, C, OH, OW, F, KY, KX, SY, SX, PT, PL, vec, 0, KY * KX, 0};
  return g;
}
// Enable the tap-mode gather when the inner (channel) extent tiles a 64-wide reduction block.
static bool set_tap_mode(ConvGeomU& g, int inner, bool dgrad) {
  g.tpk = 0; g.inner = inner;
  if (!g.vec || (inner % 8) || g.KY * g.KX > KTAB) return false;
  if (dgrad && (g.SY != 1 || g.SX != 1)) return false;
  if (inner >= 64) { if (inner % 64) return false; g.tpk = 1; return true; }
  if (64 % inner) return false;
  g.tpk = 64 / inner;
  return true;
}

int launch_conv_fprop_pair(const void*, const void*, long long, const float*, void*, int, int, int, int, int,
                           int, int, int, int, int, int, int, int, int, cudaStream_t);
int launch_conv_dgrad_pair(const void*, const void*, long long, void*, int, int, int, int, int, int, int, int,
                           int, int, int, float, const void*, int, cudaStream_t);
int launch_conv_wgrad_pair(const void*, const void*, float*, int, int, int, int, int, int, int, int, int, int,
                           int, int, int, int, cudaStream_t);
int pair_wgrad_splits(int, int, int, int);
static long long g_pair_conv_launches = 0;
long long conv_pair_launches() { return g_pair_conv_launches; }

// out[pix, f] = act(im2col(x)[pix, :] . w_lp[f, :] + bias[f]); w_lp stored [F][ldw] bf16 (ldw % 8 == 0)
int launch_conv_fprop_umma(const void* x, const void* w_lp, long long ldw, const float* bias, void* out,
                           int out_bf16, int N, int H, int W, int C, int OH, int OW, int F, int KY, int KX,
                           int SY, int SX, int PT, int PL, int act, cudaStream_t st) {
  if ((ldw % 8) || ((uintptr_t)w_lp & 15) || ((uintptr_t)x & 15)) return -3;
  if (out_bf16 && launch_conv_fprop_pair(x, w_lp, ldw, bias, out, N, H, W, C, OH, OW, F, KY, KX, SY, SX, PT,
                                         PL, act, st) == 0) {
    ++g_pair_conv_launches;        // large layer: 2-CTA persistent kernel, A by TMA im2col
    return 0;
  }
  int Kw = KY * KX * C;
  if ((C % 8 == 0 ? (Kw + 7) / 8 : Kw) > KTAB || KY > 255 || KX > 255) return -4;
  CUtensorMap ta, tb;
  int bn = pick_bn(F);
  int r = make_map(&tb, w_lp, ldw, F, ldw, bn);
  if (r) return r;
  ta = tb;
  GemmParams p{};
  p.M = N * OH * OW; p.N = F; p.K = Kw;
  p.k_blocks_per_split = (Kw + BLOCK_K - 1) / BLOCK_K;
  p.out = out; p.out_bf16 = out_bf16; p.ldo = F; p.out_trans = 0;
  p.bias = bias; p.act = act; p.alpha = 1.f; p.beta = 0.f; p.split_stride = 0;
  p.gsrc = (const __nv_bfloat16*)x; p.g = geom(N, H, W, C, OH, OW, F, KY, KX, SY, SX, PT, PL, C % 8 == 0);
  p.gather_kind = G_IM2COL; p.gK = Kw;
  if (C % 64 == 0 && im2col_tma_enabled()) {
    // A operand by TMA im2col: window bases -PL .. W + upper_w, OW x OH of them
    CUtensorMap ti;
    if (make_map_im2col(&ti, x, N, H, W, C, -PL, -PT, (OW - 1) * SX + 1 - PL - W,
                        (OH - 1) * SY + 1 - PT - H, SX, SY, BLOCK_M) == 0) {
      p.g.inner = C;
      ++g_im2col_launches;
      return launch_bn<A_IM2COL_K, B_TMA_K, G_IM2COL, 0>(bn, ti, tb, p, 1, st);
    }
  }
  if (set_tap_mode(p.g, C, false)) return launch_bn<A_GATHER_K, B_TMA_K, G_IM2COL, 2>(bn, ta, tb, p, 1, st);
  if (C % 8 == 0) return launch_bn<A_GATHER_K, B_TMA_K, G_IM2COL, 1>(bn, ta, tb, p, 1, st);
  return launch_bn<A_GATHER_K, B_TMA_K, G_IM2COL, 0>(bn, ta, tb, p, 1, st);
}

// err_in[ipix, c] = alpha * sum_{tap,f} gather(err_out) * wd_lp[(tap,f), c] + beta * err_in
// wd_lp stored [KY*KX*F][ldc] bf16 (ldc % 8 == 0, zero padded columns)
int launch_conv_dgrad_umma(const void* err_out, const void* wd_lp, long long ldc, void* err_in,
                           int ei_bf16, int N, int H, int W, int C, int OH, int OW, int F, int KY, int KX,
                           int SY, int SX, int PT, int PL, float alpha, float beta, const void* dmul,
                           int dact, cudaStream_t st) {
  // the folded derivative needs the inline bf16 epilogue mode (row-major bf16 output, no beta)
  if (dmul && (!ei_bf16 || beta != 0.f || ((uintptr_t)dmul & 15))) return -5;
  if ((ldc % 8) || ((uintptr_t)wd_lp & 15) || ((uintptr_t)err_out & 15)) return -3;
  if (ei_bf16 && beta == 0.f && SY == 1 && SX == 1 &&
      launch_conv_dgrad_pair(err_out, wd_lp, ldc, err_in, N, H, W, C, OH, OW, F, KY, KX, PT, PL, alpha, dmul,
                             dact, st) == 0) {
    ++g_pair_conv_launches;
    return 0;
  }
  int Kd = KY * KX * F;
  if ((F % 8 == 0 ? (Kd + 7) / 8 : Kd) > KTAB || KY > 255 || KX > 255) return -4;
  CUtensorMap ta, tb;
  int bn = pick_bn(C);
  if (bn < 64) bn = 64;
  int r = make_map(&tb, wd_lp, ldc, Kd, ldc, 64);
  if (r) return r;
  ta = tb;
  GemmParams p{};
  p.M = N * H * W; p.N = C; p.K = Kd;
  p.k_blocks_per_split = (Kd + BLOCK_K - 1) / BLOCK_K;
  p.out = err_in; p.out_bf16 = ei_bf16; p.ldo = C; p.out_trans = 0;
  p.bias = nullptr; p.act = 0; p.alpha = alpha; p.beta = beta; p.split_stride = 0;
  p.gsrc = (const __nv_bfloat16*)err_out;
  p.g = geom(N, H, W, C, OH, OW, F, KY, KX, SY, SX, PT, PL, F % 8 == 0);
  p.gather_kind = G_DGRAD; p.gK = Kd;
  p.dmul = (const __nv_bfloat16*)dmul; p.dact = dmul ? dact : 0;
  if (F % 64 == 0 && SY == 1 && SX == 1 && im2col_tma_enabled()) {
    // unit stride: dgrad is a correlation of err_out with the flipped filter; W x H window bases
    // starting at -(K - 1 - pad) over the [N][OH][OW][F] tensor
    CUtensorMap ti;
    const int lw = -(KX - 1 - PL), lh = -(KY - 1 - PT);
    if (make_map_im2col(&ti, err_out, N, OH, OW, F, lw, lh, W + lw - OW, H + lh - OH, 1, 1,
                        BLOCK_M) == 0) {
      p.g.inner = F;
      ++g_im2col_launches;
      return launch_bn<A_IM2COL_K, B_TMA_MN, G_DGRAD, 0>(bn, ti, tb, p, 1, st);
    }
  }
  if (set_tap_mode(p.g, F, true)) return launch_bn<A_GATHER_K, B_TMA_MN, G_DGRAD, 2>(bn, ta, tb, p, 1, st);
  if (F % 8 == 0) return launch_bn<A_GATHER_K, B_TMA_MN, G_DGRAD, 1>(bn, ta, tb, p, 1, st);
  return launch_bn<A_GATHER_K, B_TMA_MN, G_DGRAD, 0>(bn, ta, tb, p, 1, st);
}

// partials[z][f][kidx] = sum_{pix in split z} err_out[pix, f] * im2col(x)[pix, kidx]
// (computed as D[kidx, f] with the im2col operand on the 128-wide M side, stored transposed)
__device__ __align__(16) unsigned short zn_ones_bf16[8] = {0x3F80, 0, 0, 0, 0, 0, 0, 0};

// Returns 0, or 1 when ``bias_parts`` [splits][F] was filled with the per-split column sums of
// err_out as well (tap-mode gather and Kw % 128 != 0, i.e. the last M tile has a spare row).
int launch_conv_wgrad_umma(const void* err_out, const void* x, float* partials, int splits, int N, int H,
                           int W, int C, int OH, int OW, int F, int KY, int KX, int SY, int SX, int PT,
                           int PL, float* bias_parts, cudaStream_t st) {
  if ((F % 8) || ((uintptr_t)err_out & 15) || ((uintptr_t)x & 15)) return -3;
  if (launch_conv_wgrad_pair(err_out, x, partials, splits, N, H, W, C, OH, OW, F, KY, KX, SY, SX, PT, PL,
                             st) == 0) {
    ++g_pair_conv_launches;        // (no bias row: the caller falls back to the column-sum kernel)
    return 0;
  }
  int Kw = KY * KX * C, P = N * OH * OW;
  if ((C % 8 == 0 ? (Kw + 7) / 8 : Kw) > KTAB || KY > 255 || KX > 255) return -4;
  CUtensorMap ta, tb;
  int bn = pick_bn(F);
  if (bn < 64) bn = 64;
  int r = make_map(&tb, err_out, F, P, F, 64);
  if (r) return r;
  ta = tb;
  GemmParams p{};
  p.M = Kw; p.N = F; p.K = P;
  int total_kb = (P + BLOCK_K - 1) / BLOCK_K;
  if (splits < 1) splits = 1;
  p.k_blocks_per_split = (total_kb + splits - 1) / splits;
  p.out = partials; p.out_bf16 = 0; p.ldo = Kw; p.out_trans = 1;
  p.bias = nullptr; p.act = 0; p.alpha = 1.f; p.beta = 0.f; p.split_stride = (long long)F * Kw;
  p.gsrc = (const __nv_bfloat16*)x; p.g = geom(N, H, W, C, OH, OW, F, KY, KX, SY, SX, PT, PL, C % 8 == 0);
  p.gather_kind = G_IM2COL; p.gK = Kw;
  if (set_tap_mode(p.g, C, false)) {
    bool row = bias_parts != nullptr && (Kw % BLOCK_M) != 0;
    if (row) {
      static void* ones = nullptr;
      if (!ones && cudaGetSymbolAddress(&ones, zn_ones_bf16) != cudaSuccess) ones = nullptr;
      row = ones != nullptr;
      if (row) { p.g.ones = (const __nv_bfloat16*)ones; p.bias_out = bias_parts; }
    }
    r = launch_bn<A_GATHER_MN, B_TMA_MN, G_IM2COL, 2>(bn, ta, tb, p, splits, st);
    return (r == 0 && row) ? 1 : r;
  }
  if (C % 8 == 0) return launch_bn<A_GATHER_MN, B_TMA_MN, G_IM2COL, 1>(bn, ta, tb, p, splits, st);
  return launch_bn<A_GATHER_MN, B_TMA_MN, G_IM2COL, 0>(bn, ta, tb, p, splits, st);
}

}  // namespace zn
