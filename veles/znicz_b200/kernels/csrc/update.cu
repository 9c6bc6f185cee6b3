// Fused SGD step (+ cross-GPU gradient reduction over peer memory).
//
// One kernel replaces the reference's weights_update / bias_update / compute_col_sums kernels
// (/root/reference/cuda/all2all/gradient_descent/weights_update.cu:10, bias_update.cu:18,
// cuda/weights_ortho.cu:14,41, cuda/gradient_descent.store_output.cu) AND the slave->master /
// master->slave gradient and weight messages of the reference's data parallelism
// (/root/reference/nn_units.py:644-694):
//
//   g    = sum over ranks r (fixed order) of sum over split-K partials p of grad[r][p][idx]
//   gd   = -lr * (g + wd * ((1 - l1) * w + 0.5 * l1 * sign(w)) + ortho / rows * (colsum[col] - w))
//   acc  = acc_beta * acc + acc_alpha * gd ; gd = gd_beta * gd + gd_alpha * acc      (optional)
//   gd  += moment * vel ; vel = gd                                                     (optional)
//   w   += gd                                                                          (optional)
//   + bf16 shadow copies of w in the layouts the tcgen05 GEMM/conv kernels consume.
//
// In data-parallel mode grad[r] are *peer pointers* into the other GPUs' HBM (symmetric
// memory over NVLink5/NVSwitch): every rank reads all ranks' gradient tiles in the same order,
// so all replicas compute bit-identical weights with no NCCL call and no broadcast.
// Cross-GPU ordering uses per-block flag words in symmetric memory (st.release.sys /
// ld.acquire.sys), with the epoch counter kept in device memory so CUDA-graph replays work.
#include "common.cuh"
#include <string.h>

namespace zn {

struct GradSources {
  const float* ptr[8];   // per-rank base pointers (ptr[0] = local when nranks == 1)
  int nranks;
  int nparts;            // split-K partials per rank
  long long part_stride; // elements between partials
  int g_cpad;            // > 0: gradient rows are [tap][g_cpad] channel-padded (first conv layer)
  float gscale;          // multiplies the cross-rank sum (1 / world_size: data-parallel mean)
};

struct ShadowSpec {
  __nv_bfloat16* lp;       // [rows][ld] bf16 copy of w (row-major as w), may be null
  int ld;
  int lp_cpad;             // > 0: lp rows are [tap][lp_cpad] channel-padded
  __nv_bfloat16* lp_conv;  // conv dgrad operand [tap][f_pad = roundup(rows, 8)][c_pad], may be null
  int taps, C, c_pad;
};

struct PeerSync {
  uint32_t* flags[8];      // flags[r] = rank r's flag array [max_blocks][8]
  uint32_t* epoch;         // local [max_blocks]
  int rank, nranks;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// A peer that never arrives (crashed rank, protocol bug) must not hang the box: trap after
// ZN_PEER_TIMEOUT_NS of wall time (the host then sees a launch failure on every rank).
#ifndef ZN_PEER_TIMEOUT_NS
#define ZN_PEER_TIMEOUT_NS 20000000000ULL
#endif

// Block-level barrier across ranks: thread t < nranks signals rank t and waits for rank t.
__device__ __forceinline__ void peer_barrier(const PeerSync& ps, uint32_t value) {
  __syncthreads();
  if ((int)threadIdx.x < ps.nranks) {
    int peer = threadIdx.x;
    st_release_sys(ps.flags[peer] + (size_t)blockIdx.x * 8 + ps.rank, value);
    const uint32_t* mine = ps.flags[ps.rank] + (size_t)blockIdx.x * 8 + peer;
    if ((int)(ld_acquire_sys(mine) - value) < 0) {
      const unsigned long long t0 = globaltimer_ns();
      unsigned spins = 0;
      while ((int)(ld_acquire_sys(mine) - value) < 0) {
        if ((++spins & 1023u) == 0 && globaltimer_ns() - t0 > ZN_PEER_TIMEOUT_NS) { __trap(); }
      }
    }
  }
  __syncthreads();
}

// ---- NVLS: loads / stores on the MULTICAST mapping of a symmetric buffer. A multimem load with
// .add is reduced inside the NVSwitch over every rank's copy; a multimem store lands in every
// rank's copy (one write on this GPU's link instead of N - 1).
__device__ __forceinline__ float4 mm_ld_reduce_f4(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ float mm_ld_reduce_f1(const float* mc) {
  float v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.f32 %0, [%1];" : "=f"(v) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ void mm_st_f4(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x),
               "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// hyper layout: see GradientDescentBase.HYPER_FIELDS
template <bool MULTI>
__global__ void fused_update_k(float* __restrict__ w, GradSources gs, float* __restrict__ grad_out,
                               float* __restrict__ acc, float* __restrict__ vel,
                               const float* __restrict__ hyper, const float* __restrict__ col_sums,
                               int flags, int is_bias, long long size, int rows, int cols,
                               ShadowSpec sh, PeerSync ps) {
  pdl_wait();
  __shared__ uint32_t s_epoch;
  uint32_t epoch = 0;
  if (MULTI) {
    if (threadIdx.x == 0) s_epoch = ps.epoch[blockIdx.x] + 1;
    __syncthreads();
    epoch = s_epoch;
    peer_barrier(ps, 2 * epoch - 1);   // every rank's gradient is complete and visible
  }
  const float lr = hyper[is_bias ? 9 : 0], wd = hyper[is_bias ? 10 : 1];
  const float l1 = hyper[is_bias ? 11 : 2], moment = hyper[is_bias ? 12 : 3];
  const float acc_alpha = hyper[4], acc_beta = hyper[5], gd_alpha = hyper[6], gd_beta = hyper[7];
  const float ortho = hyper[8];
  const bool apply = flags & 1, use_moment = flags & 2, use_acc = flags & 4;
  const bool use_ortho = (flags & 8) && col_sums != nullptr;
  const bool transposed = flags & 16;

  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < size; i += stride) {
    long long gi = i;
    if (gs.g_cpad > 0) {
      const int r_ = (int)(i / cols), c_ = (int)(i % cols);
      const int tap_ = c_ / sh.C, ch_ = c_ - tap_ * sh.C;
      gi = ((long long)r_ * sh.taps + tap_) * gs.g_cpad + ch_;
    }
    float g = 0.f;
    for (int r = 0; r < gs.nranks; ++r) {        // fixed rank order => bit-identical replicas
      const float* base = gs.ptr[r] + gi;
      float g0 = 0.f, g1 = 0.f, g2 = 0.f, g3 = 0.f;
      int p = 0;
      for (; p + 4 <= gs.nparts; p += 4) {       // 4 loads in flight per rank
        g0 += base[(long long)(p + 0) * gs.part_stride];
        g1 += base[(long long)(p + 1) * gs.part_stride];
        g2 += base[(long long)(p + 2) * gs.part_stride];
        g3 += base[(long long)(p + 3) * gs.part_stride];
      }
      for (; p < gs.nparts; ++p) g0 += base[(long long)p * gs.part_stride];
      g += (g0 + g1) + (g2 + g3);
    }
    g *= gs.gscale;
    if (grad_out) grad_out[i] = g;
    float wv = w[i];
    float sgn = wv > 0.f ? 1.f : (wv < 0.f ? -1.f : 0.f);
    float reg = wd * ((1.f - l1) * wv + 0.5f * l1 * sgn);
    if (use_ortho) {
      // weights [rows=Y][cols=H] (or stored transposed [H][Y]); col index = input index
      int col = transposed ? (int)(i / rows) : (int)(i % cols);
      int n_rows = transposed ? cols : rows;
      reg += ortho / (float)(transposed ? rows : rows) * (col_sums[col] - wv);
      (void)n_rows;
    }
    float gd = -lr * (g + reg);
    if (use_acc) {
      float a = (acc_beta != 0.f ? acc_beta * acc[i] : 0.f) + acc_alpha * gd;
      acc[i] = a;
      gd = gd * gd_beta + gd_alpha * a;
    }
    if (use_moment) { gd += vel[i] * moment; vel[i] = gd; }
    if (apply) { wv += gd; w[i] = wv; }
    if (sh.lp) {
      int r = (int)(i / cols), c = (int)(i % cols);
      int lc = c;
      if (sh.lp_cpad > 0) { int tap = c / sh.C; lc = tap * sh.lp_cpad + (c - tap * sh.C); }
      sh.lp[(size_t)r * sh.ld + lc] = __float2bfloat16_rn(wv);
      if (sh.lp_conv) {
        int tap = c / sh.C, ch = c % sh.C;      // w[f=r][tap][ch]
        sh.lp_conv[((size_t)tap * ((rows + 7) & ~7) + r) * sh.c_pad + ch] = __float2bfloat16_rn(wv);
      }
    }
  }
  if (MULTI) {
    peer_barrier(ps, 2 * epoch);       // nobody still reads my gradient buffer
    if (threadIdx.x == 0) ps.epoch[blockIdx.x] = epoch;
  }
}

// column sums of W (pre-update) for the orthogonality regulariser: out[col] = sum_row w[row, col]
__global__ void col_sums_k(const float* __restrict__ w, float* __restrict__ out, int rows, int cols,
                           int transposed) {
  pdl_wait();
  // logical matrix [rows=Y][cols=H]; when transposed the storage is [H][Y]
  int col = blockIdx.x * blockDim.y + threadIdx.y;
  if (col >= cols) return;
  float s = 0.f;
  for (int r = threadIdx.x; r < rows; r += 32)
    s += transposed ? w[(size_t)col * rows + r] : w[(size_t)r * cols + col];
  s = warp_sum(s);
  if (threadIdx.x == 0) out[col] = s;
}

// shadow refresh without an update step (initialisation, rollback, weights from a snapshot)
__global__ void refresh_shadows_k(const float* __restrict__ w, long long size, int rows, int cols,
                                  ShadowSpec sh) {
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < size; i += stride) {
    float wv = w[i];
    int r = (int)(i / cols), c = (int)(i % cols);
    int lc = c;
    if (sh.lp_cpad > 0) { int tap = c / sh.C; lc = tap * sh.lp_cpad + (c - tap * sh.C); }
    if (sh.lp) sh.lp[(size_t)r * sh.ld + lc] = __float2bfloat16_rn(wv);
    if (sh.lp_conv) {
      int tap = c / sh.C, ch = c % sh.C;
      sh.lp_conv[((size_t)tap * ((rows + 7) & ~7) + r) * sh.c_pad + ch] = __float2bfloat16_rn(wv);
    }
  }
}


// ------------------------------------------------------------------------------------------
// Whole-network step: ONE launch applies the (cross-GPU reduced) SGD step to every parameter
// tensor of the model. Replaces ~2 launches per layer (weights, bias) + the col_sums launches
// with a single persistent kernel, and in data-parallel mode pays ONE cross-GPU flag barrier
// per training step instead of one per tensor.
//
//   phase 0  signal peers "my gradients are complete" (they are: stream order)
//   phase 1  column sums of the pre-update weights for tensors with the ortho regulariser
//   ------   grid barrier (generation counter in device memory; graph-replay safe)
//   phase 2  wait for the peers' signals, then tiles of 256 elements round-robin over blocks:
//            sum over ranks and split-K partials (LANES threads cooperate per element when the
//            partial count is large and the tensor small), SGD step, bf16 shadows
//   phase 3  peer barrier "nobody still reads my gradient buffers"
// ------------------------------------------------------------------------------------------
struct TensorDesc {
  float* w; float* grad_out; float* acc; float* vel;
  const float* hyper; float* col_sums;
  const float* grad[8];
  long long part_stride, size;
  int nparts, g_cpad, flags, is_bias, rows, cols, lanes, enabled;
  ShadowSpec sh;
  int tile_begin, n_tiles;
  int ept;                    // elements per thread (lanes == 1 only): 4 for large tensors
  int vec4;                   // ept == 4 and every array / stride is 16-byte aligned: float4 path
  long long red_off;          // offset of this tensor in the cross-GPU reduction buffer
};

struct GridSync { unsigned* count; unsigned* gen; };
// half > 0: the reduction buffer is double buffered (slot parity alternates every step), which
// makes the trailing cross-GPU barrier unnecessary; chunks = launches per step
// algo: how phase B gets the cross-rank sum of an element
//   ALGO_ONESHOT_PEER  every rank loads all N slots over NVLink ((N - 1) * P floats in per rank)
//   ALGO_TWOSHOT       tile owners reduce their 1/N of the tiles and broadcast the sums into every
//                      rank's ``sum`` buffer (reduce-scatter + all-gather: ~2 * P floats per rank,
//                      one more flag barrier); with mc_red / mc_sum the reduce is ONE
//                      multimem.ld_reduce per float4 (in-switch, NVLS) and the broadcast ONE
//                      multimem.st, otherwise N peer loads and N peer stores per float4.
//                      The owner computes each sum once => replicas stay bit-identical whatever
//                      order the switch adds in.
//   ALGO_ONESHOT_NVLS  every rank multimem.ld_reduce-s every element itself (single barrier;
//                      bit-identical replicas only if the switch reduction is order-stable)
enum { ALGO_ONESHOT_PEER = 0, ALGO_TWOSHOT = 1, ALGO_ONESHOT_NVLS = 2 };
struct RedBufs {
  float* ptr[8]; int nranks, rank; long long half; int chunks;
  float* sum[8];            // two-shot: reduced gradients, sum[rank] is the local copy
  float* mc_red;            // multicast address of the slot buffer (null: no NVLS)
  float* mc_sum;            // multicast address of the sum buffer
  int algo;
  float gscale;             // multiplies the cross-rank gradient sum (1 / world: mean over the
                            // global batch, so N ranks x batch b == one process at batch N * b)
};
constexpr int MU_MAX_TENSORS = 48;
constexpr int MU_MAX_PEER_BLOCKS = 592;     // size of the cross-GPU flag / epoch arrays

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void grid_barrier(GridSync gs) {
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned my_gen = ld_acquire_gpu(gs.gen);   // cannot advance before I arrive
    __threadfence();
    const unsigned old = atomicAdd(gs.count, 1u);
    if (old == gridDim.x - 1) {
      *gs.count = 0u;
      __threadfence();
      atomicAdd(gs.gen, 1u);
    } else {
      long long spins = 0;
      while (ld_acquire_gpu(gs.gen) == my_gen) {
        if (++spins > (1LL << 31)) { __trap(); }
      }
    }
  }
  __syncthreads();
}

// ``base`` rotates the block -> work mapping so that consecutive tensors land on different
// blocks (the column-block lists of all tensors together are shorter than the grid).
__device__ __forceinline__ int multi_col_sums(const TensorDesc& d, int base) {
  // logical matrix [rows = Y][cols = H]; out[col] = sum over rows. 256 threads.
  __shared__ float red[8][33];
  const int tid = threadIdx.x;
  const int vb = (int)((blockIdx.x + gridDim.x - (unsigned)base % gridDim.x) % gridDim.x);
  if (d.flags & 16) {          // stored transposed [H][Y]: a warp per column, lanes over rows
    const int lane = tid & 31, wib = tid >> 5;
    for (int col = vb * 8 + wib; col < d.cols; col += gridDim.x * 8) {
      float s = 0.f;
      for (int r = lane; r < d.rows; r += 32) s += d.w[(size_t)col * d.rows + r];
      s = warp_sum(s);
      if (lane == 0) d.col_sums[col] = s;
    }
    return (d.cols + 7) / 8;
  }
  const int cx = tid & 31, ry = tid >> 5;
  const int n_cb = (d.cols + 31) / 32;
  for (int cb = vb; cb < n_cb; cb += gridDim.x) {
    const int col = cb * 32 + cx;
    float s0 = 0.f, s1 = 0.f;
    if (col < d.cols) {
      int r = ry;
      for (; r + 8 < d.rows; r += 16) {
        s0 += d.w[(size_t)r * d.cols + col];
        s1 += d.w[(size_t)(r + 8) * d.cols + col];
      }
      if (r < d.rows) s0 += d.w[(size_t)r * d.cols + col];
    }
    red[ry][cx] = s0 + s1;
    __syncthreads();
    if (ry == 0 && col < d.cols) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) s += red[k][cx];     // fixed order
      d.col_sums[col] = s;
    }
    __syncthreads();
  }
  return n_cb;
}

// MODE 0: single GPU (partials -> update). Data-parallel runs split the tile in two so that only
// ONE fp32 value per element crosses NVLink instead of every split-K partial of every rank:
// MODE 1: sum this rank's partials into its slot of the symmetric reduction buffer;
// MODE 2 (after the cross-GPU flag barrier): sum the ranks' slots in fixed order and update.
template <int MODE>
__device__ __forceinline__ void multi_elem(const TensorDesc& d, long long i, bool valid, int lane,
                                           const RedBufs& rb, long long poff);

__device__ __forceinline__ float4 f4add(float4 a, float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

// four consecutive elements i0 .. i0 + 3 (i0 % 4 == 0, all valid, no channel-padded gradient)
template <int MODE>
__device__ __forceinline__ void multi_elem4(const TensorDesc& d, const long long i0, const RedBufs& rb,
                                            const long long poff) {
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 g4 = z4;
  if (MODE == 2 && rb.algo == ALGO_TWOSHOT) {
    g4 = *reinterpret_cast<const float4*>(rb.sum[rb.rank] + poff + d.red_off + i0);
  } else if (MODE == 2 && rb.algo == ALGO_ONESHOT_NVLS) {
    g4 = mm_ld_reduce_f4(rb.mc_red + poff + d.red_off + i0);
  } else if (MODE == 2) {
    // all peer loads in flight at once (a run-time loop issues them one NVLink round trip after
    // the other), then a fixed-order sum: replicas stay bit-identical
    float4 v[8];
#pragma unroll
    for (int r = 0; r < 8; ++r)
      v[r] = (r < rb.nranks) ? *reinterpret_cast<const float4*>(rb.ptr[r] + poff + d.red_off + i0) : z4;
#pragma unroll
    for (int r = 0; r < 8; ++r) g4 = f4add(g4, v[r]);
  } else {
    const float* base = d.grad[0] + i0;
    const long long st = d.part_stride;
    float4 a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = z4;
    // same accumulator assignment and final tree as the scalar path (bit-identical sums)
    for (int p = 0; p < d.nparts; p += 8) {
      const int left = d.nparts - p;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < left) a[k] = f4add(a[k], *reinterpret_cast<const float4*>(base + (long long)(p + k) * st));
    }
    g4 = f4add(f4add(f4add(a[0], a[1]), f4add(a[2], a[3])), f4add(f4add(a[4], a[5]), f4add(a[6], a[7])));
  }
  if (MODE == 1) { *reinterpret_cast<float4*>(rb.ptr[rb.rank] + poff + d.red_off + i0) = g4; return; }
  g4.x *= rb.gscale; g4.y *= rb.gscale; g4.z *= rb.gscale; g4.w *= rb.gscale;

  const int is_bias = d.is_bias;
  const float* hyper = d.hyper;
  const float lr = hyper[is_bias ? 9 : 0], wd = hyper[is_bias ? 10 : 1];
  const float l1 = hyper[is_bias ? 11 : 2], moment = hyper[is_bias ? 12 : 3];
  const float acc_alpha = hyper[4], acc_beta = hyper[5], gd_alpha = hyper[6], gd_beta = hyper[7];
  const float ortho = hyper[8];
  const int flags = d.flags;
  const bool apply = flags & 1, use_moment = flags & 2, use_acc = flags & 4;
  const bool use_ortho = (flags & 8) && d.col_sums != nullptr;
  const bool transposed = flags & 16;
  const int rows = d.rows, cols = d.cols;
  // ---- every load first ----
  const float4 w4 = *reinterpret_cast<const float4*>(d.w + i0);
  const float4 v4 = use_moment ? *reinterpret_cast<const float4*>(d.vel + i0) : z4;
  const float4 c4 = (use_acc && acc_beta != 0.f) ? *reinterpret_cast<const float4*>(d.acc + i0) : z4;
  float cs[4] = {0.f, 0.f, 0.f, 0.f};
  if (use_ortho) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long i = i0 + j;
      cs[j] = d.col_sums[transposed ? (int)(i / rows) : (int)(i % cols)];
    }
  }
  const float g[4] = {g4.x, g4.y, g4.z, g4.w};
  float wv[4] = {w4.x, w4.y, w4.z, w4.w};
  float vv[4] = {v4.x, v4.y, v4.z, v4.w};
  float av[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float sgn = wv[j] > 0.f ? 1.f : (wv[j] < 0.f ? -1.f : 0.f);
    float reg = wd * ((1.f - l1) * wv[j] + 0.5f * l1 * sgn);
    if (use_ortho) reg += ortho / (float)rows * (cs[j] - wv[j]);
    float gd = -lr * (g[j] + reg);
    if (use_acc) {
      const float a = (acc_beta != 0.f ? acc_beta * av[j] : 0.f) + acc_alpha * gd;
      av[j] = a;
      gd = gd * gd_beta + gd_alpha * a;
    }
    if (use_moment) { gd += vv[j] * moment; vv[j] = gd; }
    if (apply) wv[j] += gd;
  }
  // ---- then every store ----
  if (d.grad_out) *reinterpret_cast<float4*>(d.grad_out + i0) = g4;
  if (use_acc) *reinterpret_cast<float4*>(d.acc + i0) = make_float4(av[0], av[1], av[2], av[3]);
  if (use_moment) *reinterpret_cast<float4*>(d.vel + i0) = make_float4(vv[0], vv[1], vv[2], vv[3]);
  if (apply) *reinterpret_cast<float4*>(d.w + i0) = make_float4(wv[0], wv[1], wv[2], wv[3]);
  const ShadowSpec& sh = d.sh;
  if (sh.lp) {
    const int r = (int)(i0 / cols), c = (int)(i0 % cols);
    if (sh.lp_cpad == 0 && !sh.lp_conv && c + 3 < cols && ((sh.ld | c) & 3) == 0) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(wv[0], wv[1]), hi = __floats2bfloat162_rn(wv[2], wv[3]);
      uint2 pk;
      pk.x = *reinterpret_cast<unsigned*>(&lo); pk.y = *reinterpret_cast<unsigned*>(&hi);
      *reinterpret_cast<uint2*>(sh.lp + (size_t)r * sh.ld + c) = pk;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const long long i = i0 + j;
        const int rj = (int)(i / cols), cj = (int)(i % cols);
        int lc = cj;
        if (sh.lp_cpad > 0) { const int tap = cj / sh.C; lc = tap * sh.lp_cpad + (cj - tap * sh.C); }
        sh.lp[(size_t)rj * sh.ld + lc] = __float2bfloat16_rn(wv[j]);
        if (sh.lp_conv) {
          const int tap = cj / sh.C, ch = cj % sh.C;
          sh.lp_conv[((size_t)tap * ((rows + 7) & ~7) + rj) * sh.c_pad + ch] = __float2bfloat16_rn(wv[j]);
        }
      }
    }
  }
}

template <int MODE>
__device__ __forceinline__ void multi_tile(const TensorDesc& d, int tile, const RedBufs& rb,
                                           long long poff) {
  const int L = d.lanes;                         // power of two, <= 32
  const int tid = threadIdx.x;
  if (d.ept > 1 && d.vec4) {
    // large tensors (AlexNet FC6: 37.7 M weights): one float4 chunk per thread, every input of
    // the chunk loaded before the first store. The element-at-a-time form below cannot overlap
    // its loads (the compiler must assume the stores alias them): ~12 dependent HBM round trips
    // per tile, 1.2 ms for the AlexNet step where the traffic (1.6 GB) needs 0.25 ms.
    const long long i0 = (long long)tile * (256 * 4) + (long long)tid * 4;
    if (i0 + 3 < d.size) { multi_elem4<MODE>(d, i0, rb, poff); return; }
#pragma unroll 1
    for (int k = 0; k < 4; ++k) multi_elem<MODE>(d, i0 + k, i0 + k < d.size, 0, rb, poff);
    return;
  }
  if (d.ept > 1) {
    // 4 independent elements per thread (stride 256 keeps every access coalesced)
    const long long base = (long long)tile * (256 * 4) + tid;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long i = base + k * 256;
      multi_elem<MODE>(d, i, i < d.size, 0, rb, poff);
    }
    return;
  }
  const int lane = tid & (L - 1);
  const int ept = 256 / L;                       // elements per tile
  const long long i = (long long)tile * ept + tid / L;
  multi_elem<MODE>(d, i, i < d.size, lane, rb, poff);
}

// gradient of element i: sum of the split-K partials (this rank) or of the ranks' slots; the
// result is valid on lane 0 of the element's lane group. Loads only - no stores - so the caller
// may issue it for the next tile before the current tile's update has been written.
template <int MODE>
__device__ __forceinline__ float multi_grad(const TensorDesc& d, const long long i, const bool valid,
                                            const int lane, const RedBufs& rb, long long poff) {
  const int L = d.ept > 1 ? 1 : d.lanes;
  float g = 0.f;
  if (MODE == 2 && rb.algo == ALGO_TWOSHOT) {
    if (valid && lane == 0) g = rb.sum[rb.rank][poff + d.red_off + i];
  } else if (MODE == 2 && rb.algo == ALGO_ONESHOT_NVLS) {
    if (valid && lane == 0) g = mm_ld_reduce_f1(rb.mc_red + poff + d.red_off + i);
  } else if (MODE == 2) {
    if (valid && lane == 0) {
      // every peer load in flight at once, then a fixed-order sum (bit-identical replicas)
      float v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) v[r] = (r < rb.nranks) ? rb.ptr[r][poff + d.red_off + i] : 0.f;
#pragma unroll
      for (int r = 0; r < 8; ++r) g += v[r];
    }
  } else if (valid) {
    long long gi = i;
    if (d.g_cpad > 0) {
      const int r_ = (int)(i / d.cols), c_ = (int)(i % d.cols);
      const int tap_ = c_ / d.sh.C, ch_ = c_ - tap_ * d.sh.C;
      gi = ((long long)r_ * d.sh.taps + tap_) * d.g_cpad + ch_;
    }
    const float* base = d.grad[0] + gi;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f, a5 = 0.f, a6 = 0.f, a7 = 0.f;
    // 8 predicated loads in flight per round (the remainder is not serialised: out-of-range
    // slots load nothing and add 0, the summation order stays fixed)
    for (int p = lane; p < d.nparts; p += 8 * L) {
      const long long st = d.part_stride;
      const float* b = base + (long long)p * st;
      const int left = d.nparts - p;
      a0 += b[0];
      a1 += (1 * L < left) ? b[(long long)(1 * L) * st] : 0.f;
      a2 += (2 * L < left) ? b[(long long)(2 * L) * st] : 0.f;
      a3 += (3 * L < left) ? b[(long long)(3 * L) * st] : 0.f;
      a4 += (4 * L < left) ? b[(long long)(4 * L) * st] : 0.f;
      a5 += (5 * L < left) ? b[(long long)(5 * L) * st] : 0.f;
      a6 += (6 * L < left) ? b[(long long)(6 * L) * st] : 0.f;
      a7 += (7 * L < left) ? b[(long long)(7 * L) * st] : 0.f;
    }
    g = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  }
  if (MODE != 2)
    for (int o = L >> 1; o > 0; o >>= 1) g += __shfl_xor_sync(0xffffffffu, g, o);
  return MODE == 1 ? g : g * rb.gscale;
}

template <int MODE>
__device__ __forceinline__ void multi_apply(const TensorDesc& d, const long long i, const bool valid,
                                            const int lane, const float g, const RedBufs& rb,
                                            long long poff) {
  const int is_bias = d.is_bias;
  if (!valid || lane != 0) return;
  if (MODE == 1) { rb.ptr[rb.rank][poff + d.red_off + i] = g; return; }

  const float* hyper = d.hyper;
  const float lr = hyper[is_bias ? 9 : 0], wd = hyper[is_bias ? 10 : 1];
  const float l1 = hyper[is_bias ? 11 : 2], moment = hyper[is_bias ? 12 : 3];
  const float acc_alpha = hyper[4], acc_beta = hyper[5], gd_alpha = hyper[6], gd_beta = hyper[7];
  const float ortho = hyper[8];
  const int flags = d.flags;
  const bool apply = flags & 1, use_moment = flags & 2, use_acc = flags & 4;
  const bool use_ortho = (flags & 8) && d.col_sums != nullptr;
  const bool transposed = flags & 16;
  const int rows = d.rows, cols = d.cols;

  if (d.grad_out) d.grad_out[i] = g;
  float wv = d.w[i];
  const float sgn = wv > 0.f ? 1.f : (wv < 0.f ? -1.f : 0.f);
  float reg = wd * ((1.f - l1) * wv + 0.5f * l1 * sgn);
  if (use_ortho) {
    const int col = transposed ? (int)(i / rows) : (int)(i % cols);
    reg += ortho / (float)rows * (d.col_sums[col] - wv);
  }
  float gd = -lr * (g + reg);
  if (use_acc) {
    const float a = (acc_beta != 0.f ? acc_beta * d.acc[i] : 0.f) + acc_alpha * gd;
    d.acc[i] = a;
    gd = gd * gd_beta + gd_alpha * a;
  }
  if (use_moment) { gd += d.vel[i] * moment; d.vel[i] = gd; }
  if (apply) { wv += gd; d.w[i] = wv; }
  const ShadowSpec& sh = d.sh;
  if (sh.lp) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    int lc = c;
    if (sh.lp_cpad > 0) { const int tap = c / sh.C; lc = tap * sh.lp_cpad + (c - tap * sh.C); }
    sh.lp[(size_t)r * sh.ld + lc] = __float2bfloat16_rn(wv);
    if (sh.lp_conv) {
      const int tap = c / sh.C, ch = c % sh.C;
      sh.lp_conv[((size_t)tap * ((rows + 7) & ~7) + r) * sh.c_pad + ch] = __float2bfloat16_rn(wv);
    }
  }
}

template <int MODE>
__device__ __forceinline__ void multi_elem(const TensorDesc& d, const long long i, const bool valid,
                                           const int lane, const RedBufs& rb, long long poff) {
  multi_apply<MODE>(d, i, valid, lane, multi_grad<MODE>(d, i, valid, lane, rb, poff), rb, poff);
}

// Two-shot, owner side: reduce one tile's slots over the ranks and broadcast the sums.
// The tile's slot range is float4-aligned and padded to a multiple of 4 (multi_update_table).
__device__ __forceinline__ void multi_reduce_bcast(const TensorDesc& d, int tile_local, const RedBufs& rb,
                                                   long long poff) {
  const long long n_tile = d.ept > 1 ? 1024 : 256 / d.lanes;
  const long long e0 = (long long)tile_local * n_tile;
  long long n = d.size - e0;
  if (n > n_tile) n = n_tile;
  n = (n + 3) & ~3LL;
  const long long o = poff + d.red_off + e0;
  for (long long c = (long long)threadIdx.x * 4; c < n; c += 256 * 4) {
    float4 g;
    if (rb.mc_red != nullptr) {
      g = mm_ld_reduce_f4(rb.mc_red + o + c);
      mm_st_f4(rb.mc_sum + o + c, g);
    } else {
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 v[8];
#pragma unroll
      for (int r = 0; r < 8; ++r)
        v[r] = (r < rb.nranks) ? *reinterpret_cast<const float4*>(rb.ptr[r] + o + c) : z4;
      g = z4;
#pragma unroll
      for (int r = 0; r < 8; ++r) g = f4add(g, v[r]);       // fixed rank order
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < rb.nranks) *reinterpret_cast<float4*>(rb.sum[r] + o + c) = g;
    }
  }
}

__global__ void __launch_bounds__(256, 4)
multi_update_k(const TensorDesc* __restrict__ table, int n, int total_tiles, int has_ortho,
               PeerSync ps, GridSync gsync, RedBufs rb) {
  __shared__ uint32_t s_epoch;
  __shared__ TensorDesc s_table[MU_MAX_TENSORS];     // the whole table: no dependent global loads
  const bool multi = ps.nranks > 1;
  uint32_t epoch = 0;
  {
    // the descriptor table is written by the host when the step is built, never by a kernel:
    // staging it may overlap the tail of the preceding (last wgrad) kernel
    const int words = n * (int)(sizeof(TensorDesc) / 4);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(table);
    uint32_t* dst = reinterpret_cast<uint32_t*>(s_table);
    for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
  }
  pdl_wait();
  if (multi) {
    if (threadIdx.x == 0) s_epoch = ps.epoch[blockIdx.x] + 1;
  }
  __syncthreads();
  if (multi) epoch = s_epoch;
  const long long poff =
      (multi && rb.half > 0 && (((epoch - 1) / (uint32_t)max(rb.chunks, 1)) & 1u)) ? rb.half : 0;
  if (has_ortho) {
    int cs_base = 0;
    for (int t = 0; t < n; ++t) {
      const TensorDesc& d = s_table[t];
      if (!d.enabled || d.is_bias || !(d.flags & 8) || !d.col_sums) continue;
      cs_base += multi_col_sums(d, cs_base);
    }
  }
  if (multi) {
    // phase A: this block's tiles, local split-K reduction -> my slot of the reduction buffer
    int t = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      while (t + 1 < n && tile >= s_table[t].tile_begin + s_table[t].n_tiles) ++t;
      const TensorDesc& d = s_table[t];
      if (d.enabled) multi_tile<1>(d, tile - d.tile_begin, rb, poff);
    }
    // every rank maps tile -> block identically, so block b only needs block b of each peer:
    // publish (release, after the CTA barrier inside peer_barrier) and wait
    peer_barrier(ps, 2 * epoch - 1);
    if (rb.algo == ALGO_TWOSHOT) {
      // reduce-scatter + all-gather over tile owners. Tile t belongs to block t % grid on every
      // rank, so the owner's block index equals the reader's: the per-block flag barrier below
      // is all the synchronisation the broadcast needs.
      int t = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        while (t + 1 < n && tile >= s_table[t].tile_begin + s_table[t].n_tiles) ++t;
        const TensorDesc& d = s_table[t];
        if (!d.enabled) continue;
        if ((int)(((unsigned)(tile / (int)gridDim.x) + (unsigned)tile) % (unsigned)rb.nranks) != rb.rank) continue;
        multi_reduce_bcast(d, tile - d.tile_begin, rb, poff);
      }
      __threadfence_system();              // my broadcast stores before my flag
      peer_barrier(ps, 2 * epoch);         // every owner's sums have landed in my sum buffer
    }
  }
  if (has_ortho) grid_barrier(gsync);    // col_sums of all tensors complete before any update
  if (!multi) {
    // single GPU: software-pipelined tile loop - the partial sums of the CTA's next tile are
    // loaded (multi_grad: loads only) while the current tile is being updated; small tensors
    // (one element per lane group) only, the float4 / 4-element tiles keep their own path
    int t = 0;
    int tile = blockIdx.x;
    float g_next = 0.f;
    bool have_next = false;
    auto locate = [&](int tl) {
      while (t + 1 < n && tl >= s_table[t].tile_begin + s_table[t].n_tiles) ++t;   // uniform
      return t;
    };
    auto elem_of = [&](const TensorDesc& d, int tl, long long& i, int& lane) {
      const int L = d.lanes;
      lane = threadIdx.x & (L - 1);
      i = (long long)(tl - d.tile_begin) * (256 / L) + threadIdx.x / L;
    };
    while (tile < total_tiles) {
      const int tc = locate(tile);
      const TensorDesc& d = s_table[tc];
      const int nxt = tile + gridDim.x;
      if (!d.enabled) { tile = nxt; have_next = false; continue; }
      if (d.ept > 1) { multi_tile<0>(d, tile - d.tile_begin, rb, poff); tile = nxt; have_next = false; continue; }
      long long i; int lane;
      elem_of(d, tile, i, lane);
      const bool valid = i < d.size;
      const float g = have_next ? g_next : multi_grad<0>(d, i, valid, lane, rb, poff);
      have_next = false;
      if (nxt < total_tiles) {
        const int tn = locate(nxt);           // t advances monotonically; d stays a valid reference
        const TensorDesc& dn = s_table[tn];
        if (dn.enabled && dn.ept <= 1) {
          long long in_; int ln;
          elem_of(dn, nxt, in_, ln);
          g_next = multi_grad<0>(dn, in_, in_ < dn.size, ln, rb, poff);
          have_next = true;
        }
      }
      multi_apply<0>(d, i, valid, lane, g, rb, poff);
      tile = nxt;
    }
  } else {
    int t = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      while (t + 1 < n && tile >= s_table[t].tile_begin + s_table[t].n_tiles) ++t;   // uniform
      const TensorDesc& d = s_table[t];
      if (!d.enabled) continue;
      multi_tile<2>(d, tile - d.tile_begin, rb, poff);
    }
  }
  if (multi) {
    // single-buffered slots: wait until nobody still reads mine. Double-buffered slots need no
    // trailing barrier: a rank can be at most one step ahead (the phase barrier of step k + 1
    // is passed only after every peer finished reading step k), and step k + 1 uses the other half.
    if (rb.half <= 0 && rb.algo != ALGO_TWOSHOT) peer_barrier(ps, 2 * epoch);
    if (threadIdx.x == 0) ps.epoch[blockIdx.x] = epoch;
  }
}

// Data-parallel gradient scale (set once by parallel/data_parallel.py): the step kernels multiply
// the cross-rank gradient sum by it. 1 = plain sum.
static float g_dp_gscale = 1.f;
void set_dp_gradient_scale(float s) { g_dp_gscale = s; }
float get_dp_gradient_scale() { return g_dp_gscale; }

size_t multi_update_desc_size() { return sizeof(TensorDesc); }
int multi_update_max_tensors() { return MU_MAX_TENSORS; }

// fields: see ext.cpp::multi_update_table. Returns the number of tiles.
int multi_update_pack(const long long* f, int n_fields, void* out, int tile_begin, long long red_off) {
  TensorDesc d{};
  d.w = (float*)f[0]; d.grad_out = (float*)f[1]; d.acc = (float*)f[2]; d.vel = (float*)f[3];
  d.hyper = (const float*)f[4]; d.col_sums = (float*)f[5];
  for (int r = 0; r < 8; ++r) d.grad[r] = (const float*)f[6 + r];
  d.part_stride = f[14]; d.size = f[15];
  d.nparts = (int)f[16]; d.g_cpad = (int)f[17]; d.flags = (int)f[18]; d.is_bias = (int)f[19];
  d.rows = (int)f[20]; d.cols = (int)f[21]; d.lanes = (int)f[22]; d.enabled = (int)f[23];
  d.sh.lp = (__nv_bfloat16*)f[24]; d.sh.ld = (int)f[25]; d.sh.lp_cpad = (int)f[26];
  d.sh.lp_conv = (__nv_bfloat16*)f[27]; d.sh.taps = (int)f[28]; d.sh.C = (int)f[29];
  d.sh.c_pad = (int)f[30];
  if (d.lanes < 1) d.lanes = 1;
  d.ept = (d.lanes == 1 && d.size >= (1LL << 20)) ? 4 : 1;
  {
    uintptr_t al = (uintptr_t)d.w | (uintptr_t)d.grad_out | (uintptr_t)d.acc | (uintptr_t)d.vel |
                   (uintptr_t)d.grad[0];
    d.vec4 = (d.ept == 4 && d.g_cpad == 0 && (al & 15) == 0 &&
              (d.nparts <= 1 || (d.part_stride & 3) == 0) && (red_off & 3) == 0) ? 1 : 0;
  }
  const int ept = d.ept > 1 ? 1024 : 256 / d.lanes;
  d.tile_begin = tile_begin;
  d.n_tiles = (int)((d.size + ept - 1) / ept);
  d.red_off = red_off;
  memcpy(out, &d, sizeof(d));
  (void)n_fields;
  return d.n_tiles;
}

void launch_multi_update(const void* table, int n, int total_tiles, int has_ortho, int nranks,
                         uint32_t* const* peer_flags, uint32_t* epoch, int rank, unsigned* gridsync,
                         float* const* red_ptrs, long long red_half, int chunks,
                         float* const* sum_ptrs, float* mc_red, float* mc_sum, int algo, int max_blocks,
                         cudaStream_t st) {
  PeerSync ps{};
  ps.rank = rank; ps.nranks = (peer_flags && nranks > 1) ? nranks : 1; ps.epoch = epoch;
  if (peer_flags) for (int r = 0; r < nranks; ++r) ps.flags[r] = peer_flags[r];
  GridSync gs{gridsync, gridsync + 1};
  // latency-bound kernel: 4 CTAs of 256 threads per SM (all co-resident: the grid barrier needs it)
  int blocks = total_tiles < 592 ? total_tiles : 592;
  if (ps.nranks > 1 && blocks > MU_MAX_PEER_BLOCKS) blocks = MU_MAX_PEER_BLOCKS;
  if (blocks < 1) blocks = 1;
  RedBufs rb{};
  rb.nranks = ps.nranks; rb.rank = rank; rb.half = red_half; rb.chunks = chunks;
  if (red_ptrs) for (int r = 0; r < nranks; ++r) rb.ptr[r] = red_ptrs[r];
  if (sum_ptrs) for (int r = 0; r < nranks; ++r) rb.sum[r] = sum_ptrs[r];
  rb.mc_red = mc_red; rb.mc_sum = mc_sum;
  rb.algo = ps.nranks > 1 ? algo : ALGO_ONESHOT_PEER;
  rb.gscale = g_dp_gscale;
  if (max_blocks > 0 && blocks > max_blocks) blocks = max_blocks;   // (fake-peer tests share one GPU)
  launch_k(multi_update_k, blocks, 256, 0, st, (const TensorDesc*)table, n, total_tiles, has_ortho, ps, gs, rb);
}

int fused_update_blocks(long long size) {
  long long b = (size + 255) / 256;     // one element per thread up to one CTA per SM
  if (b < 1) b = 1;
  if (b > 148) b = 148;
  return (int)b;
}

void launch_fused_update(float* w, const float* const* grad_ptrs, int nranks, int nparts,
                         long long part_stride, float* grad_out, float* acc, float* vel,
                         const float* hyper, const float* col_sums, int flags, int is_bias,
                         long long size, int rows, int cols, __nv_bfloat16* lp, int ld,
                         __nv_bfloat16* lp_conv, int taps, int C, int c_pad,
                         uint32_t* const* peer_flags, uint32_t* epoch, int rank, int blocks,
                         int lp_cpad, int g_cpad, cudaStream_t st) {
  GradSources gs{};
  for (int r = 0; r < nranks; ++r) gs.ptr[r] = grad_ptrs[r];
  gs.nranks = nranks; gs.nparts = nparts; gs.part_stride = part_stride; gs.g_cpad = g_cpad;
  gs.gscale = g_dp_gscale;
  ShadowSpec sh{lp, ld, lp_cpad, lp_conv, taps, C, c_pad};
  PeerSync ps{};
  ps.rank = rank; ps.nranks = nranks; ps.epoch = epoch;
  if (peer_flags) for (int r = 0; r < nranks; ++r) ps.flags[r] = peer_flags[r];
  if (blocks <= 0) blocks = fused_update_blocks(size);
  if (peer_flags && nranks > 1)
    launch_k(fused_update_k<true>, blocks, 256, 0, st, w, gs, grad_out, acc, vel, hyper, col_sums, flags,
                                                  is_bias, size, rows, cols, sh, ps);
  else
    launch_k(fused_update_k<false>, blocks, 256, 0, st, w, gs, grad_out, acc, vel, hyper, col_sums, flags,
                                                   is_bias, size, rows, cols, sh, ps);
}
void launch_col_sums(const float* w, float* out, int rows, int cols, int transposed, cudaStream_t st) {
  dim3 block(32, 8);
  launch_k(col_sums_k, (cols + 7) / 8, block, 0, st, w, out, rows, cols, transposed);
}
void launch_refresh_shadows(const float* w, long long size, int rows, int cols, __nv_bfloat16* lp, int ld,
                            __nv_bfloat16* lp_conv, int taps, int C, int c_pad, int lp_cpad,
                            cudaStream_t st) {
  ShadowSpec sh{lp, ld, lp_cpad, lp_conv, taps, C, c_pad};
  long long b = (size + 255) / 256; if (b > 592) b = 592; if (b < 1) b = 1;
  launch_k(refresh_shadows_k, (int)b, 256, 0, st, w, size, rows, cols, sh);
}

// ---- epoch-end metric reduction over the same peer-memory mechanism -------------------------------------
// Each rank's metrics (error counts, confusion matrix, maxima; packed as doubles, sums first) sit in a
// symmetric buffer with two slots (epoch parity); one block per rank publishes, waits for every
// peer with the flag barrier of the gradient kernels and reduces in fixed rank order - every rank
// ends with bit-identical totals and no library collective is involved.
struct MetricSrc { const double* p[8]; };

__global__ void metric_reduce_k(PeerSync ps, MetricSrc src, double* __restrict__ out, int n_sum, int n_max,
                                int slot) {
  __shared__ uint32_t s_epoch;
  if (threadIdx.x == 0) s_epoch = ++ps.epoch[blockIdx.x];
  __syncthreads();
  const int n = n_sum + n_max;
  peer_barrier(ps, s_epoch);                  // every rank's slot is written and visible
  const size_t off = (size_t)slot * n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double acc = src.p[0][off + i];
    for (int r = 1; r < ps.nranks; ++r) {
      const double v = src.p[r][off + i];
      acc = i < n_sum ? acc + v : (v > acc ? v : acc);
    }
    out[i] = acc;
  }
  // no trailing barrier: the host alternates the slot, and a rank only gets to overwrite a slot two
  // calls later - after it passed the next call's barrier, which every peer enters (block 0 exists
  // in every call) after its previous kernel, i.e. these reads, completed
}

void launch_metric_reduce(const double* const* src, int nranks, int rank, uint32_t* const* peer_flags,
                          uint32_t* epoch, double* out, int n_sum, int n_max, int slot, cudaStream_t st) {
  PeerSync ps{};
  ps.rank = rank; ps.nranks = nranks; ps.epoch = epoch;
  MetricSrc ms{};
  for (int r = 0; r < nranks; ++r) { ps.flags[r] = peer_flags[r]; ms.p[r] = src[r]; }
  int blocks = (n_sum + n_max + 1023) / 1024;
  blocks = blocks < 1 ? 1 : (blocks > 64 ? 64 : blocks);
  metric_reduce_k<<<blocks, 256, 0, st>>>(ps, ms, out, n_sum, n_max, slot);
}

}  // namespace zn
