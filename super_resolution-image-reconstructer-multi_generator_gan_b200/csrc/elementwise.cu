// Memory-bound kernels of the SR-GAN hot path: BatchNorm statistics / apply / backward, LeakyReLU backward,
// 9x9 unfold, weight packing, Adam, ReconstructionLoss and the relativistic tanh loss.
// All loads/stores on activations are 128-bit (8 bf16 channels); reductions are warp-shuffle + fixed-order
// partial sums (run-to-run deterministic, no float atomics).
#include "elementwise.cuh"

#include <cuda_bf16.h>
#include <stdlib.h>
#include <string.h>

#include "conv_gemm.cuh"
#include "launch.cuh"
#include "ptx.cuh"

namespace srg {

#define SRG_LAUNCH_CHECK(name)                                                    \
  do {                                                                            \
    cudaError_t e_ = cudaGetLastError();                                          \
    if (e_ != cudaSuccess) {                                                      \
      set_error("%s launch: %s", name, cudaGetErrorString(e_));                   \
      return int(e_);                                                             \
    }                                                                             \
    count_launch();                                                               \
  } while (0)

__device__ __forceinline__ float blo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bhi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t bpack(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void unpack8(const uint4& r, float (&f)[8]) {
  f[0] = blo(r.x); f[1] = bhi(r.x); f[2] = blo(r.y); f[3] = bhi(r.y);
  f[4] = blo(r.z); f[5] = bhi(r.z); f[6] = blo(r.w); f[7] = bhi(r.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 o;
  o.x = bpack(f[0], f[1]); o.y = bpack(f[2], f[3]); o.z = bpack(f[4], f[5]); o.w = bpack(f[6], f[7]);
  return o;
}

// ------------------------------------------------------------------------------------------------
// per-channel reductions: thread = (pixel lane, channel group of 8)
// ------------------------------------------------------------------------------------------------
static int env_int(const char* name, int dflt) {
  const char* ev = getenv(name);
  return (ev != nullptr && ev[0] != '\0') ? atoi(ev) : dflt;
}
// developer knobs (read once): CTAs per SM of the elementwise / reduction passes.  Fewer CTAs leave HBM bandwidth to a
// tensor-core kernel of another graph branch running beside them (profiles/r02_notes.md)
static int red_per_sm() { static int v = -1; if (v < 0) v = env_int("SRG_RED_PER_SM", 2); return v < 1 ? 1 : v; }
static int ew_per_sm() { static int v = -1; if (v < 0) v = env_int("SRG_EW_PER_SM", 4); return v < 1 ? 1 : v; }
static int fin_per_sm() { static int v = -1; if (v < 0) v = env_int("SRG_FIN_PER_SM", 2); return v < 1 ? 1 : v; }
// L2 eviction priorities (SRG_L2_HINTS: 0 none, 1 BatchNorm chain, 2 + conv outputs / aux tiles, 3 (default) + conv operands
// and the block-input read, 4 + weight-gradient and generic-kernel operands).  Per trunk layer the three generators
// stream ~450 MB through a 126 MB L2; without hints the tensors with a near reuse (the conv output the reduction and the
// apply pass read next, the apply output the next conv reads) are evicted by data that is dead after its access.
int l2_hints() { static int v = -1; if (v < 0) v = env_int("SRG_L2_HINTS", 3); return v; }
static int red_threads() { static int v = -1; if (v < 0) v = env_int("SRG_RED_THREADS", 512) == 256 ? 256 : 512; return v; }
int reduce_blocks(int64_t pixels) {
  int64_t b = (pixels + 32 * 8 - 1) / (32 * 8);
  if (b < 1) b = 1;
  const int cap = red_per_sm() * sm_budget() < kRedBlocksMax ? red_per_sm() * sm_budget() : kRedBlocksMax;
  if (b > cap) {
    // every block the same number of 128-pixel rounds (4 pixels of a thread in flight per round): no block runs a tail of
    // single-pixel rounds after the others have finished (cfg2: 288 blocks x 4 rounds instead of 296 x 3 + up to 3 singles)
    const int64_t per_round = red_threads() / 2;      // T / 8 pixels x 4 in flight
    const int64_t rounds = (pixels + per_round - 1) / per_round;
    const int64_t per_block = (rounds + cap - 1) / cap;
    b = (rounds + per_block - 1) / per_block;
  }
  return int(b);
}

// T threads per block = T / 8 pixels per round-slot.  T = 512 (two blocks per SM) keeps 32 warps x 8 loads in flight per SM:
// at cfg2 every block then runs 2 dependent rounds instead of 4 (the pass is bound by the latency of its rounds).
template <bool TWO, int T>
__global__ void __launch_bounds__(T) chan_reduce_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b,
                                                        int64_t pixels, float* __restrict__ partials, uint64_t pol) {
  constexpr int PR = T / 8;       // pixels per round-slot
  __shared__ float red[PR][129];
  pdl_trigger();
  pdl_wait();
  const int cg = threadIdx.x & 7;
  const int lane_p = threadIdx.x >> 3;
  float s1[8], s2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) s1[e] = s2[e] = 0.f;
  // four pixels of a thread in flight per round (8 x 128-bit loads): the kernel is latency-bound otherwise (measured
  // 2.9 TB/s with one pixel per round); the accumulation order per thread is unchanged
  const int64_t stride = int64_t(gridDim.x) * PR;
  int64_t p = int64_t(blockIdx.x) * PR + lane_p;
  for (; p + 3 * stride < pixels; p += 4 * stride) {
    uint4 ra[4], rb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      ra[u] = ldg_hint_u4(a + (p + u * stride) * 8 + cg, pol);
      if (TWO) rb[u] = ldg_hint_u4(b + (p + u * stride) * 8 + cg, pol);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float fa[8], fb[8];
      unpack8(ra[u], fa);
      if (TWO) unpack8(rb[u], fb);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        s1[e] += fa[e];
        s2[e] += TWO ? fa[e] * fb[e] : fa[e] * fa[e];
      }
    }
  }
  for (; p < pixels; p += stride) {
    float fa[8], fb[8];
    unpack8(a[p * 8 + cg], fa);
    if (TWO) unpack8(b[p * 8 + cg], fb);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      s1[e] += fa[e];
      s2[e] += TWO ? fa[e] * fb[e] : fa[e] * fa[e];
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    red[lane_p][cg * 8 + e] = s1[e];
    red[lane_p][64 + cg * 8 + e] = s2[e];
  }
  __syncthreads();
  if (threadIdx.x < 128) {
    float acc = 0.f;
#pragma unroll 8
    for (int l = 0; l < PR; ++l) acc += red[l][threadIdx.x];
    partials[size_t(blockIdx.x) * 128 + threadIdx.x] = acc;
  }
}

// ---- fused reduction + finalize: the last block to finish (atomic ticket) sums the block partials in a fixed order
// and runs the per-channel finalize in the same launch (3 launches -> 1 when no cross-GPU all-reduce sits in between).
__device__ __forceinline__ void finalize_channels(const ReduceFinalize& f, int c, double s1, double s2) {
  if (f.mode == RF_BN_FWD) {
    const double mean = s1 / f.count;
    double var = s2 / f.count - mean * mean;
    if (var < 0.0) var = 0.0;
    const float inv = float(1.0 / sqrt(var + double(f.eps)));
    const float sc = f.gamma[c] * inv;
    f.out0[c] = sc;                                 // scale
    f.out1[c] = f.beta[c] - float(mean) * sc;       // shift
    f.out2[c] = float(mean);                        // save_mean
    f.out3[c] = inv;                                // save_inv
    if (f.running_mean != nullptr) {
      const double unbiased = f.count > 1.0 ? var * (f.count / (f.count - 1.0)) : var;
      f.running_mean[c] = (1.f - f.momentum) * f.running_mean[c] + f.momentum * float(mean);
      f.running_var[c] = (1.f - f.momentum) * f.running_var[c] + f.momentum * float(unbiased);
    }
  } else if (f.mode == RF_BN_BWD) {
    const double mean = f.save_mean[c], inv = f.save_inv[c];
    const double dg = inv * (s2 - mean * s1);
    const double db = s1;
    if (f.dgamma) f.dgamma[c] = float(dg);
    if (f.dbeta) f.dbeta[c] = float(db);
    const double sc = double(f.gamma[c]) * inv;
    f.out0[c] = float(sc);
    f.out1[c] = float(-sc * inv * dg / f.count);
    f.out2[c] = float(-sc * db / f.count + sc * inv * mean * dg / f.count);
  } else if (f.mode == RF_BN_BWD_FROZEN) {
    // y_hat = (y - running_mean) * inv does not depend on the batch: dy = gamma * inv * dz
    const double rm = f.save_mean[c], inv = f.save_inv[c];
    const double sc = double(f.gamma[c]) * inv;
    if (f.dgamma) f.dgamma[c] = float(inv * (s2 - rm * s1));
    if (f.dbeta) f.dbeta[c] = float(s1);
    if (f.dbias) f.dbias[c] = float(sc * s1);
    f.out0[c] = float(sc);
    f.out1[c] = 0.f;
    f.out2[c] = 0.f;
  } else {
    f.out0[c] = float(s1);                          // RF_SUM: bias gradient
  }
}

template <bool TWO, int T>
__global__ void __launch_bounds__(T) chan_reduce_final_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b,
                                                                int64_t pixels, float* __restrict__ partials,
                                                                unsigned int* __restrict__ ticket, const ReduceFinalize f,
                                                                uint64_t pol) {
  constexpr int PR = T / 8;       // pixels per round-slot (as chan_reduce_kernel)
  constexpr int RL = T / 32;      // row lanes of the last block's fixed-order sum
  __shared__ float red[PR][129];
  __shared__ bool is_last;
  static_assert(sizeof(float) * PR * 129 >= sizeof(double) * RL * 128, "the fp64 staging reuses the float rows");
  pdl_trigger();
  pdl_wait();
  const int cg = threadIdx.x & 7;
  const int lane_p = threadIdx.x >> 3;
  float s1[8], s2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) s1[e] = s2[e] = 0.f;
  const int64_t stride = int64_t(gridDim.x) * PR;
  int64_t p = int64_t(blockIdx.x) * PR + lane_p;
  for (; p + 3 * stride < pixels; p += 4 * stride) {      // same loop (and per-thread accumulation order) as chan_reduce_kernel
    uint4 ra[4], rb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      ra[u] = ldg_hint_u4(a + (p + u * stride) * 8 + cg, pol);
      if (TWO) rb[u] = ldg_hint_u4(b + (p + u * stride) * 8 + cg, pol);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float fa[8], fb[8];
      unpack8(ra[u], fa);
      if (TWO) unpack8(rb[u], fb);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        s1[e] += fa[e];
        s2[e] += TWO ? fa[e] * fb[e] : fa[e] * fa[e];
      }
    }
  }
  for (; p < pixels; p += stride) {
    float fa[8], fb[8];
    unpack8(a[p * 8 + cg], fa);
    if (TWO) unpack8(b[p * 8 + cg], fb);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      s1[e] += fa[e];
      s2[e] += TWO ? fa[e] * fb[e] : fa[e] * fa[e];
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    red[lane_p][cg * 8 + e] = s1[e];
    red[lane_p][64 + cg * 8 + e] = s2[e];
  }
  __syncthreads();
  if (threadIdx.x < 128) {
    float acc = 0.f;
#pragma unroll 8
    for (int l = 0; l < PR; ++l) acc += red[l][threadIdx.x];
    partials[size_t(blockIdx.x) * 128 + threadIdx.x] = acc;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  // the last block to finish: fixed-order fp64 sum of every block's row (RL row lanes x 32 column quads), then the finalize
  __threadfence();
  double* dred = reinterpret_cast<double*>(&red[0][0]);        // [RL][128] doubles over the dead float rows
  const int c4 = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const float4* src = reinterpret_cast<const float4*>(partials) + c4;
  const int rows = int(gridDim.x);
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int r = rl;
  for (; r + 4 * RL < rows; r += 5 * RL) {
    const float4 v0 = __ldcg(src + size_t(r) * 32), v1 = __ldcg(src + size_t(r + RL) * 32), v2 = __ldcg(src + size_t(r + 2 * RL) * 32);
    const float4 v3 = __ldcg(src + size_t(r + 3 * RL) * 32), v4 = __ldcg(src + size_t(r + 4 * RL) * 32);
    a0 += double(v0.x); a1 += double(v0.y); a2 += double(v0.z); a3 += double(v0.w);
    a0 += double(v1.x); a1 += double(v1.y); a2 += double(v1.z); a3 += double(v1.w);
    a0 += double(v2.x); a1 += double(v2.y); a2 += double(v2.z); a3 += double(v2.w);
    a0 += double(v3.x); a1 += double(v3.y); a2 += double(v3.z); a3 += double(v3.w);
    a0 += double(v4.x); a1 += double(v4.y); a2 += double(v4.z); a3 += double(v4.w);
  }
  for (; r < rows; r += RL) {
    const float4 v = __ldcg(src + size_t(r) * 32);
    a0 += double(v.x); a1 += double(v.y); a2 += double(v.z); a3 += double(v.w);
  }
  __syncthreads();
  dred[rl * 128 + c4 * 4 + 0] = a0; dred[rl * 128 + c4 * 4 + 1] = a1;
  dred[rl * 128 + c4 * 4 + 2] = a2; dred[rl * 128 + c4 * 4 + 3] = a3;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 128) {
#pragma unroll
    for (int i = 0; i < RL; ++i) t += dred[i * 128 + threadIdx.x];
  }
  __syncthreads();
  if (threadIdx.x < 128) dred[threadIdx.x] = t;
  __syncthreads();
  if (threadIdx.x < 64) finalize_channels(f, threadIdx.x, dred[threadIdx.x], dred[64 + threadIdx.x]);
  if (threadIdx.x == 0) *ticket = 0u;
}

// partials [rows][128] -> fixed-order column sums (8 row lanes x 128 columns, 4 independent accumulators per thread) ->
// per-channel finalize, one 1024-thread block.
__global__ void __launch_bounds__(1024) partials_finalize_kernel(const float* __restrict__ partials, int rows,
                                                                 const ReduceFinalize f, double* __restrict__ sums_out) {
  __shared__ double red[8][128];
  pdl_trigger();
  pdl_wait();
  const int col = threadIdx.x & 127, rl = threadIdx.x >> 7;
  red[rl][col] = partials_lane_sum(partials, rows, col, rl);
  __syncthreads();
  if (rl == 0) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][col];
    red[0][col] = t;
    if (sums_out != nullptr) sums_out[col] = t;
  }
  __syncthreads();
  if (sums_out == nullptr && threadIdx.x < 64) finalize_channels(f, threadIdx.x, red[0][threadIdx.x], red[0][64 + threadIdx.x]);
}
int launch_partials_finalize(const float* partials, int rows, const ReduceFinalize& f, cudaStream_t st) {
  launch_pdl(partials_finalize_kernel, dim3(1), dim3(1024), 0, st, partials, rows, f, static_cast<double*>(nullptr));
  SRG_LAUNCH_CHECK("partials_finalize");
  return 0;
}
int launch_partials_sums(const float* partials, int rows, double* sums, cudaStream_t st) {
  ReduceFinalize f;
  memset(&f, 0, sizeof(f));
  partials_finalize_kernel<<<1, 1024, 0, st>>>(partials, rows, f, sums);
  SRG_LAUNCH_CHECK("partials_sums");
  return 0;
}

int launch_chan_reduce_final(const void* a, const void* b, int64_t pixels, float* partials, unsigned int* ticket,
                             const ReduceFinalize& f, cudaStream_t st) {
  const int blocks = reduce_blocks(pixels);
  const uint64_t pol = (b && l2_hints()) ? kL2EvictLast : kL2EvictNormal;
  const uint4* aa = reinterpret_cast<const uint4*>(a);
  const uint4* bb = reinterpret_cast<const uint4*>(b);
  if (red_threads() == 512) {
    if (b) launch_pdl(chan_reduce_final_kernel<true, 512>, dim3(blocks), dim3(512), 0, st, aa, bb, pixels, partials, ticket, f, pol);
    else launch_pdl(chan_reduce_final_kernel<false, 512>, dim3(blocks), dim3(512), 0, st, aa, bb, pixels, partials, ticket, f, pol);
  } else {
    if (b) launch_pdl(chan_reduce_final_kernel<true, 256>, dim3(blocks), dim3(256), 0, st, aa, bb, pixels, partials, ticket, f, pol);
    else launch_pdl(chan_reduce_final_kernel<false, 256>, dim3(blocks), dim3(256), 0, st, aa, bb, pixels, partials, ticket, f, pol);
  }
  SRG_LAUNCH_CHECK("chan_reduce_final");
  return 0;
}

int launch_chan_reduce(const void* a, const void* b, int64_t pixels, float* partials, cudaStream_t st) {
  const int blocks = reduce_blocks(pixels);
  const uint64_t pol = (b && l2_hints()) ? kL2EvictLast : kL2EvictNormal;
  const uint4* aa = reinterpret_cast<const uint4*>(a);
  const uint4* bb = reinterpret_cast<const uint4*>(b);
  if (red_threads() == 512) {
    if (b) launch_pdl(chan_reduce_kernel<true, 512>, dim3(blocks), dim3(512), 0, st, aa, bb, pixels, partials, pol);
    else launch_pdl(chan_reduce_kernel<false, 512>, dim3(blocks), dim3(512), 0, st, aa, bb, pixels, partials, pol);
  } else {
    if (b) launch_pdl(chan_reduce_kernel<true, 256>, dim3(blocks), dim3(256), 0, st, aa, bb, pixels, partials, pol);
    else launch_pdl(chan_reduce_kernel<false, 256>, dim3(blocks), dim3(256), 0, st, aa, bb, pixels, partials, pol);
  }
  SRG_LAUNCH_CHECK("chan_reduce");
  return 0;
}

__global__ void partials_to_sums_kernel(const float* __restrict__ partials, int blocks, double* __restrict__ sums) {
  // 128 columns x 8 row-lanes; fixed order => deterministic
  __shared__ double red[8][128];
  const int col = threadIdx.x & 127, rl = threadIdx.x >> 7;
  double acc = 0.0;
  for (int b = rl; b < blocks; b += 8) acc += double(partials[size_t(b) * 128 + col]);
  red[rl][col] = acc;
  __syncthreads();
  if (rl == 0) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][col];
    sums[col] = t;
  }
}
int launch_partials_to_sums(const float* partials, int blocks, double* sums, cudaStream_t st) {
  partials_to_sums_kernel<<<1, 1024, 0, st>>>(partials, blocks, sums);
  SRG_LAUNCH_CHECK("partials_to_sums");
  return 0;
}

__global__ void bn_finalize_kernel(const double* __restrict__ sums, double count, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, float* running_mean,
                                   float* running_var, float* scale, float* shift, float* save_mean, float* save_inv) {
  const int c = threadIdx.x;
  if (c >= 64) return;
  const double mean = sums[c] / count;
  double var = sums[64 + c] / count - mean * mean;
  if (var < 0.0) var = 0.0;
  const float inv = float(1.0 / sqrt(var + double(eps)));
  const float sc = gamma[c] * inv;
  scale[c] = sc;
  shift[c] = beta[c] - float(mean) * sc;
  save_mean[c] = float(mean);
  save_inv[c] = inv;
  if (running_mean != nullptr) {
    const double unbiased = count > 1.0 ? var * (count / (count - 1.0)) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * float(mean);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * float(unbiased);
  }
}
int launch_bn_finalize(const double* sums, double count, const float* gamma, const float* beta, float eps,
                       float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                       float* save_mean, float* save_inv, cudaStream_t st) {
  bn_finalize_kernel<<<1, 64, 0, st>>>(sums, count, gamma, beta, eps, momentum, running_mean, running_var, scale, shift,
                                       save_mean, save_inv);
  SRG_LAUNCH_CHECK("bn_finalize");
  return 0;
}

__global__ void bn_eval_coeffs_kernel(const float* gamma, const float* beta, const float* rm, const float* rv, float eps,
                                      const float* conv_bias, float* scale, float* shift) {
  const int c = threadIdx.x;
  const float sc = gamma[c] * rsqrtf(rv[c] + eps);
  scale[c] = sc;
  // conv_bias != null: the shift absorbs the producing conv's bias, bn(conv + b) = conv * sc + (beta + (b - mean) * sc)
  shift[c] = beta[c] + ((conv_bias != nullptr ? conv_bias[c] : 0.f) - rm[c]) * sc;
}
int launch_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                          float eps, float* scale, float* shift, cudaStream_t st, const float* conv_bias) {
  bn_eval_coeffs_kernel<<<1, 64, 0, st>>>(gamma, beta, running_mean, running_var, eps, conv_bias, scale, shift);
  SRG_LAUNCH_CHECK("bn_eval_coeffs");
  return 0;
}

// every eval-mode BatchNorm of a generator in ONE launch, issued before the first conv of the forward: the convs are
// launched with programmatic dependent launch and read their folded coefficients in the prologue, BEFORE
// griddepcontrol.wait, so the coefficients must not come from the immediately preceding kernel (launch.cuh)
__global__ void bn_eval_coeffs_all_kernel(const float* __restrict__ master, const float* __restrict__ buffers,
                                          const int4* __restrict__ tab, float eps, float* __restrict__ coef) {
  const int l = blockIdx.x, c = threadIdx.x;
  const int4 t = tab[l];                      // {gamma, beta, running_mean, conv bias} offsets
  const float* rm = buffers + t.z;
  const float sc = master[t.x + c] * rsqrtf(rm[64 + c] + eps);
  coef[size_t(l) * 256 + c] = sc;
  coef[size_t(l) * 256 + 64 + c] = master[t.y + c] + (master[t.w + c] - rm[c]) * sc;
}
int launch_bn_eval_coeffs_all(const float* master, const float* buffers, const void* tab, int n_bn, float eps, float* coef,
                              cudaStream_t st) {
  if (n_bn <= 0) return 0;
  bn_eval_coeffs_all_kernel<<<n_bn, 64, 0, st>>>(master, buffers, reinterpret_cast<const int4*>(tab), eps, coef);
  SRG_LAUNCH_CHECK("bn_eval_coeffs_all");
  return 0;
}

// frozen BatchNorm (eval-mode statistics on the training workspace): the convs keep their own bias, so the shift does not
// absorb it; running_mean and inv go to the save_mean / save_inv slots the backward reads
__global__ void bn_frozen_coeffs_all_kernel(const float* __restrict__ master, const float* __restrict__ buffers,
                                            const int4* __restrict__ tab, float eps, float* __restrict__ coef) {
  const int l = blockIdx.x, c = threadIdx.x;
  const int4 t = tab[l];                      // {gamma, beta, running_mean, (conv bias: unused)} offsets
  const float* rm = buffers + t.z;
  const float inv = 1.f / sqrtf(rm[64 + c] + eps);
  const float sc = master[t.x + c] * inv;
  float* o = coef + size_t(l) * 256;
  o[c] = sc;
  o[64 + c] = master[t.y + c] - rm[c] * sc;
  o[128 + c] = rm[c];
  o[192 + c] = inv;
}
int launch_bn_frozen_coeffs_all(const float* master, const float* buffers, const void* tab, int n_bn, float eps, float* coef,
                                cudaStream_t st) {
  if (n_bn <= 0) return 0;
  bn_frozen_coeffs_all_kernel<<<n_bn, 64, 0, st>>>(master, buffers, reinterpret_cast<const int4*>(tab), eps, coef);
  SRG_LAUNCH_CHECK("bn_frozen_coeffs_all");
  return 0;
}

template <bool RELU, bool SKIP>
__global__ void __launch_bounds__(256) bn_apply_kernel(const uint4* __restrict__ y, const float* __restrict__ scale,
                                                       const float* __restrict__ shift, const uint4* __restrict__ skip,
                                                       uint4* __restrict__ out, int64_t n_vec, uint64_t pol_y, uint64_t pol_out,
                                                       uint64_t pol_skip, int late) {
  if (!late) pdl_trigger();
  pdl_wait();
  const int cg = threadIdx.x & 7;  // blockDim is a multiple of 8 and the grid stride too
  float sc[8], sh[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    sc[e] = scale[cg * 8 + e];
    sh[e] = shift[cg * 8 + e];
  }
  // U vectors of a thread in flight per round, the last round predicated (the pass is latency-bound with one vector per
  // round: 4.1 TB/s at cfg2)
  constexpr int U = SKIP ? 2 : 4;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec; i += U * stride) {
    uint4 ry[U], rk[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i + u * stride < n_vec) {
        ry[u] = ldg_hint_u4(y + i + u * stride, pol_y);
        if (SKIP) rk[u] = ldg_hint_u4(skip + i + u * stride, pol_skip);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i + u * stride < n_vec) {
        float f[8], k[8];
        unpack8(ry[u], f);
        if (SKIP) unpack8(rk[u], k);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float v = fmaf(f[e], sc[e], sh[e]);
          if (RELU) v = fmaxf(v, 0.f);
          if (SKIP) v += k[e];
          f[e] = v;
        }
        stg_hint_u4(out + i + u * stride, pack8(f), pol_out);
      }
    }
  }
  if (late) pdl_trigger();
}
static int ew_blocks(int64_t n_vec) {
  int64_t b = (n_vec + 255) / 256;
  if (b > sm_budget() * ew_per_sm()) b = sm_budget() * ew_per_sm();
  if (b < 1) b = 1;
  return int(b);
}
// grid of a pass whose threads take U vectors per round: every block the same number of rounds (cfg2: 576 blocks x 2 or 4
// full rounds instead of 592 blocks with a mostly-empty last round)
static int ew_blocks_rounds(int64_t n_vec, int U) {
  const int64_t cap = int64_t(sm_budget()) * ew_per_sm();
  const int64_t rounds = (n_vec + 256 * U - 1) / (256 * U);
  if (rounds <= cap) return int(rounds < 1 ? 1 : rounds);
  const int64_t per_block = (rounds + cap - 1) / cap;
  return int((rounds + per_block - 1) / per_block);
}
int launch_bn_apply(const void* y, const float* scale, const float* shift, const void* skip, int relu, void* out,
                    int64_t pixels, cudaStream_t st) {
  const int64_t n_vec = pixels * 8;
  const int blocks = ew_blocks_rounds(n_vec, skip ? 2 : 4);
  const uint4* yy = reinterpret_cast<const uint4*>(y);
  const uint4* kk = reinterpret_cast<const uint4*>(skip);
  uint4* oo = reinterpret_cast<uint4*>(out);
  // y is not read again before the backward pass (evict first); the output is the next convolution's operand (keep)
  const uint64_t py = l2_hints() ? kL2EvictFirst : kL2EvictNormal, po = l2_hints() ? kL2EvictLast : kL2EvictNormal;
  const uint64_t pk = l2_hints() >= 3 ? kL2EvictFirst : kL2EvictNormal;      // the block input: last read of the forward pass
  if (relu && skip) launch_pdl(bn_apply_kernel<true, true>, dim3(blocks), dim3(256), 0, st, yy, scale, shift, kk, oo, n_vec, py, po, pk, pdl_ew_late());
  else if (relu) launch_pdl(bn_apply_kernel<true, false>, dim3(blocks), dim3(256), 0, st, yy, scale, shift, kk, oo, n_vec, py, po, pk, pdl_ew_late());
  else if (skip) launch_pdl(bn_apply_kernel<false, true>, dim3(blocks), dim3(256), 0, st, yy, scale, shift, kk, oo, n_vec, py, po, pk, pdl_ew_late());
  else launch_pdl(bn_apply_kernel<false, false>, dim3(blocks), dim3(256), 0, st, yy, scale, shift, kk, oo, n_vec, py, po, pk, pdl_ew_late());
  SRG_LAUNCH_CHECK("bn_apply");
  return 0;
}

__global__ void bn_bwd_finalize_kernel(const double* __restrict__ sums, double count, const float* __restrict__ gamma,
                                       const float* __restrict__ save_mean, const float* __restrict__ save_inv,
                                       float* dgamma, float* dbeta, float* coefA, float* coefB, float* coefC,
                                       float param_grad_scale) {
  const int c = threadIdx.x;
  if (c >= 64) return;
  const double sd = sums[c], sdy = sums[64 + c];
  const double mean = save_mean[c], inv = save_inv[c];
  const double dg = inv * (sdy - mean * sd);  // sum dout * xhat
  const double db = sd;
  // under SyncBatchNorm the sums are global: every rank then holds d(sum of rank losses)/d(gamma); scaling by
  // 1/world makes the rank-mean of the (identical) values the gradient of the MEAN loss, like DDP + SyncBatchNorm
  if (dgamma) dgamma[c] = float(dg) * param_grad_scale;
  if (dbeta) dbeta[c] = float(db) * param_grad_scale;
  const double sc = double(gamma[c]) * inv;
  // dy = sc * (dout - db/M - xhat * dg/M),  xhat = (y - mean) * inv
  coefA[c] = float(sc);
  coefB[c] = float(-sc * inv * dg / count);
  coefC[c] = float(-sc * db / count + sc * inv * mean * dg / count);
}
int launch_bn_bwd_finalize(const double* sums, double count, const float* gamma, const float* save_mean,
                           const float* save_inv, float* dgamma, float* dbeta, float* coefA, float* coefB,
                           float* coefC, float param_grad_scale, cudaStream_t st) {
  bn_bwd_finalize_kernel<<<1, 64, 0, st>>>(sums, count, gamma, save_mean, save_inv, dgamma, dbeta, coefA, coefB, coefC,
                                           param_grad_scale);
  SRG_LAUNCH_CHECK("bn_bwd_finalize");
  return 0;
}

__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const uint4* __restrict__ dout, const uint4* __restrict__ y,
                                                           const float* __restrict__ cA, const float* __restrict__ cB,
                                                           const float* __restrict__ cC, uint4* __restrict__ dy,
                                                           int64_t n_vec, uint64_t pol_in, uint64_t pol_out, int late) {
  if (!late) pdl_trigger();
  pdl_wait();
  const int cg = threadIdx.x & 7;
  float a[8], b[8], c[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    a[e] = cA[cg * 8 + e];
    b[e] = cB[cg * 8 + e];
    c[e] = cC[cg * 8 + e];
  }
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec; i += 2 * stride) {
    // two vectors of each tensor in flight per thread, the second predicated
    const bool two = i + stride < n_vec;
    const uint4 rd0 = ldg_hint_u4(dout + i, pol_in), ry0 = ldg_hint_u4(y + i, pol_in);
    uint4 rd1 = rd0, ry1 = ry0;
    if (two) { rd1 = ldg_hint_u4(dout + i + stride, pol_in); ry1 = ldg_hint_u4(y + i + stride, pol_in); }
    float d[8], v[8];
    unpack8(rd0, d);
    unpack8(ry0, v);
#pragma unroll
    for (int e = 0; e < 8; ++e) d[e] = fmaf(a[e], d[e], fmaf(b[e], v[e], c[e]));
    stg_hint_u4(dy + i, pack8(d), pol_out);
    if (two) {
      unpack8(rd1, d);
      unpack8(ry1, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) d[e] = fmaf(a[e], d[e], fmaf(b[e], v[e], c[e]));
      stg_hint_u4(dy + i + stride, pack8(d), pol_out);
    }
  }
  if (late) pdl_trigger();
}
int launch_bn_bwd_apply(const void* dout, const void* y, const float* coefA, const float* coefB, const float* coefC,
                        void* dy, int64_t pixels, cudaStream_t st) {
  const int64_t n_vec = pixels * 8;
  launch_pdl(bn_bwd_apply_kernel, dim3(ew_blocks_rounds(n_vec, 2)), dim3(256), 0, st, reinterpret_cast<const uint4*>(dout),
             reinterpret_cast<const uint4*>(y), coefA, coefB, coefC, reinterpret_cast<uint4*>(dy), n_vec,
             // dz and y are (all but) dead after this pass.  Measured: keeping bn2's dz, which the block's conv1 dgrad reads
             // once more as the skip gradient, at high priority costs 0.15 ms per step, and discarding the dead bn1 dz lines
             // (discard.global.L2) buys nothing (profiles/r02_notes.md)
             l2_hints() ? kL2EvictFirst : kL2EvictNormal,
             l2_hints() ? kL2EvictLast : kL2EvictNormal,       // dy is the next dgrad's operand
             pdl_ew_late());
  SRG_LAUNCH_CHECK("bn_bwd_apply");
  return 0;
}

// ---- BatchNorm apply / backward apply with the statistics finalize folded in ---------------------------------------
// The separate one-block finalize launch between the producer of the [rows][128] partial sums and the apply pass is pure
// latency on the per-generator dependency chain (measured in the replayed graph: ~5 us of execution + ~5 us of
// dependent-launch gaps per BatchNorm layer and direction).  Here every CTA of the apply pass re-reduces the partial rows
// itself (<= 296 x 512 B, L2-resident, fixed order => every CTA and every run gets bit-identical sums), computes the
// per-channel coefficients into shared memory and goes straight on to the elementwise pass; CTA 0 also writes what
// later kernels need (coefficients, saved mean / inv-std, running statistics, weight / bias gradients).
constexpr int kFinThreads = 512;
__device__ __forceinline__ void block_partial_sums(const float* __restrict__ partials, int rows, double (*red)[128],
                                                   double* sums) {
  // 512 threads = 16 row lanes x 32 column quads; row lane rl sums rows rl, rl+16, ... in order (fp64)
  const int c4 = threadIdx.x & 31, rl = threadIdx.x >> 5;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  const float4* src = reinterpret_cast<const float4*>(partials) + c4;
  int r = rl;
  for (; r + 48 < rows; r += 64) {
    const float4 v0 = __ldcg(src + size_t(r) * 32), v1 = __ldcg(src + size_t(r + 16) * 32);
    const float4 v2 = __ldcg(src + size_t(r + 32) * 32), v3 = __ldcg(src + size_t(r + 48) * 32);
    a0 += double(v0.x); a1 += double(v0.y); a2 += double(v0.z); a3 += double(v0.w);
    a0 += double(v1.x); a1 += double(v1.y); a2 += double(v1.z); a3 += double(v1.w);
    a0 += double(v2.x); a1 += double(v2.y); a2 += double(v2.z); a3 += double(v2.w);
    a0 += double(v3.x); a1 += double(v3.y); a2 += double(v3.z); a3 += double(v3.w);
  }
  for (; r < rows; r += 16) {
    const float4 v = __ldcg(src + size_t(r) * 32);
    a0 += double(v.x); a1 += double(v.y); a2 += double(v.z); a3 += double(v.w);
  }
  red[rl][c4 * 4 + 0] = a0; red[rl][c4 * 4 + 1] = a1; red[rl][c4 * 4 + 2] = a2; red[rl][c4 * 4 + 3] = a3;
  __syncthreads();
  if (threadIdx.x < 128) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) t += red[i][threadIdx.x];
    sums[threadIdx.x] = t;
  }
  __syncthreads();
}

template <bool RELU, bool SKIP>
__global__ void __launch_bounds__(kFinThreads) bn_apply_fin_kernel(const uint4* __restrict__ y, const float* __restrict__ partials,
                                                                   int rows, const ReduceFinalize f,
                                                                   const uint4* __restrict__ skip, uint4* __restrict__ out,
                                                                   int64_t n_vec) {
  __shared__ double red[16][128];
  __shared__ double sums[128];
  __shared__ float coef[2][64];
  pdl_trigger();
  pdl_wait();
  block_partial_sums(partials, rows, red, sums);
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    const double mean = sums[c] / f.count;
    double var = sums[64 + c] / f.count - mean * mean;
    if (var < 0.0) var = 0.0;
    const float inv = float(1.0 / sqrt(var + double(f.eps)));
    const float sc = f.gamma[c] * inv;
    const float sh = f.beta[c] - float(mean) * sc;
    coef[0][c] = sc;
    coef[1][c] = sh;
    if (blockIdx.x == 0) {
      f.out0[c] = sc; f.out1[c] = sh; f.out2[c] = float(mean); f.out3[c] = inv;
      if (f.running_mean != nullptr) {
        const double unbiased = f.count > 1.0 ? var * (f.count / (f.count - 1.0)) : var;
        f.running_mean[c] = (1.f - f.momentum) * f.running_mean[c] + f.momentum * float(mean);
        f.running_var[c] = (1.f - f.momentum) * f.running_var[c] + f.momentum * float(unbiased);
      }
    }
  }
  __syncthreads();
  const int cg = threadIdx.x & 7;
  float sc[8], sh[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { sc[e] = coef[0][cg * 8 + e]; sh[e] = coef[1][cg * 8 + e]; }
  const int64_t stride = int64_t(gridDim.x) * kFinThreads;
  int64_t i = int64_t(blockIdx.x) * kFinThreads + threadIdx.x;
  for (; i + 3 * stride < n_vec; i += 4 * stride) {
    uint4 ry[4], rk[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      ry[u] = y[i + u * stride];
      if (SKIP) rk[u] = skip[i + u * stride];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float v[8], k[8];
      unpack8(ry[u], v);
      if (SKIP) unpack8(rk[u], k);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float o = fmaf(v[e], sc[e], sh[e]);
        if (RELU) o = fmaxf(o, 0.f);
        if (SKIP) o += k[e];
        v[e] = o;
      }
      out[i + u * stride] = pack8(v);
    }
  }
  for (; i < n_vec; i += stride) {
    float v[8], k[8];
    unpack8(y[i], v);
    if (SKIP) unpack8(skip[i], k);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float o = fmaf(v[e], sc[e], sh[e]);
      if (RELU) o = fmaxf(o, 0.f);
      if (SKIP) o += k[e];
      v[e] = o;
    }
    out[i] = pack8(v);
  }
}
static int fin_blocks(int64_t n_vec) {
  int64_t b = (n_vec + kFinThreads - 1) / kFinThreads;
  if (b > fin_per_sm() * sm_budget()) b = fin_per_sm() * sm_budget();
  if (b < 1) b = 1;
  return int(b);
}
int launch_bn_apply_fin(const void* y, const float* partials, int rows, const ReduceFinalize& f, const void* skip, int relu,
                        void* out, int64_t pixels, cudaStream_t st) {
  if (f.mode != RF_BN_FWD) { set_error("bn_apply_fin: needs an RF_BN_FWD finalize descriptor"); return -40; }
  const int64_t n_vec = pixels * 8;
  const dim3 grid(fin_blocks(n_vec)), block(kFinThreads);
  const uint4* yy = reinterpret_cast<const uint4*>(y);
  const uint4* kk = reinterpret_cast<const uint4*>(skip);
  uint4* oo = reinterpret_cast<uint4*>(out);
  if (relu && skip) launch_pdl(bn_apply_fin_kernel<true, true>, grid, block, 0, st, yy, partials, rows, f, kk, oo, n_vec);
  else if (relu) launch_pdl(bn_apply_fin_kernel<true, false>, grid, block, 0, st, yy, partials, rows, f, kk, oo, n_vec);
  else if (skip) launch_pdl(bn_apply_fin_kernel<false, true>, grid, block, 0, st, yy, partials, rows, f, kk, oo, n_vec);
  else launch_pdl(bn_apply_fin_kernel<false, false>, grid, block, 0, st, yy, partials, rows, f, kk, oo, n_vec);
  SRG_LAUNCH_CHECK("bn_apply_fin");
  return 0;
}

__global__ void __launch_bounds__(kFinThreads) bn_bwd_apply_fin_kernel(const uint4* __restrict__ dout, const uint4* __restrict__ y,
                                                                       const float* __restrict__ partials, int rows,
                                                                       const ReduceFinalize f, uint4* __restrict__ dy,
                                                                       int64_t n_vec) {
  __shared__ double red[16][128];
  __shared__ double sums[128];
  __shared__ float coef[3][64];
  pdl_trigger();
  pdl_wait();
  block_partial_sums(partials, rows, red, sums);
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    const double s1 = sums[c], s2 = sums[64 + c];
    const double mean = f.save_mean[c], inv = f.save_inv[c];
    const double dg = inv * (s2 - mean * s1);
    const double db = s1;
    const double sc = double(f.gamma[c]) * inv;
    const float cA = float(sc), cB = float(-sc * inv * dg / f.count);
    const float cC = float(-sc * db / f.count + sc * inv * mean * dg / f.count);
    coef[0][c] = cA; coef[1][c] = cB; coef[2][c] = cC;
    if (blockIdx.x == 0) {
      if (f.dgamma) f.dgamma[c] = float(dg);
      if (f.dbeta) f.dbeta[c] = float(db);
      f.out0[c] = cA; f.out1[c] = cB; f.out2[c] = cC;
    }
  }
  __syncthreads();
  const int cg = threadIdx.x & 7;
  float a[8], b[8], c[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { a[e] = coef[0][cg * 8 + e]; b[e] = coef[1][cg * 8 + e]; c[e] = coef[2][cg * 8 + e]; }
  const int64_t stride = int64_t(gridDim.x) * kFinThreads;
  int64_t i = int64_t(blockIdx.x) * kFinThreads + threadIdx.x;
  for (; i + 3 * stride < n_vec; i += 4 * stride) {
    uint4 rd[4], ry[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { rd[u] = dout[i + u * stride]; ry[u] = y[i + u * stride]; }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float d[8], v[8];
      unpack8(rd[u], d);
      unpack8(ry[u], v);
#pragma unroll
      for (int e = 0; e < 8; ++e) d[e] = fmaf(a[e], d[e], fmaf(b[e], v[e], c[e]));
      dy[i + u * stride] = pack8(d);
    }
  }
  for (; i < n_vec; i += stride) {
    float d[8], v[8];
    unpack8(dout[i], d);
    unpack8(y[i], v);
#pragma unroll
    for (int e = 0; e < 8; ++e) d[e] = fmaf(a[e], d[e], fmaf(b[e], v[e], c[e]));
    dy[i] = pack8(d);
  }
}
int launch_bn_bwd_apply_fin(const void* dout, const void* y, const float* partials, int rows, const ReduceFinalize& f, void* dy,
                            int64_t pixels, cudaStream_t st) {
  if (f.mode != RF_BN_BWD) { set_error("bn_bwd_apply_fin: needs an RF_BN_BWD finalize descriptor"); return -40; }
  const int64_t n_vec = pixels * 8;
  launch_pdl(bn_bwd_apply_fin_kernel, dim3(fin_blocks(n_vec)), dim3(kFinThreads), 0, st, reinterpret_cast<const uint4*>(dout),
             reinterpret_cast<const uint4*>(y), partials, rows, f, reinterpret_cast<uint4*>(dy), n_vec);
  SRG_LAUNCH_CHECK("bn_bwd_apply_fin");
  return 0;
}

__global__ void __launch_bounds__(256) lrelu_bwd_add2_kernel(const uint4* __restrict__ ga, const uint4* __restrict__ gb,
                                                             const uint4* __restrict__ post, float slope,
                                                             uint4* __restrict__ dpre, int64_t n_vec) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_vec; i += int64_t(gridDim.x) * blockDim.x) {
    float a[8], b[8], p[8];
    unpack8(ga[i], a);
    if (gb) unpack8(gb[i], b);
    unpack8(post[i], p);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float g = gb ? a[e] + b[e] : a[e];
      a[e] = p[e] > 0.f ? g : g * slope;
    }
    dpre[i] = pack8(a);
  }
}
int launch_lrelu_bwd_add2(const void* ga, const void* gb, const void* post, float slope, void* dpre, int64_t pixels,
                          cudaStream_t st) {
  const int64_t n_vec = pixels * 8;
  lrelu_bwd_add2_kernel<<<ew_blocks(n_vec), 256, 0, st>>>(reinterpret_cast<const uint4*>(ga),
                                                          reinterpret_cast<const uint4*>(gb),
                                                          reinterpret_cast<const uint4*>(post), slope,
                                                          reinterpret_cast<uint4*>(dpre), n_vec);
  SRG_LAUNCH_CHECK("lrelu_bwd_add2");
  return 0;
}

__global__ void sums_to_float_kernel(const double* sums, float* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = float(sums[i]);
}
int launch_sums_to_float(const double* sums, float* out, int n, cudaStream_t st) {
  sums_to_float_kernel<<<(n + 127) / 128, 128, 0, st>>>(sums, out, n);
  SRG_LAUNCH_CHECK("sums_to_float");
  return 0;
}

// One block per image row of the pixel-shuffled gradient: 256 threads = 16 pixel lanes x (j, channel group).
__global__ void __launch_bounds__(256) ps_row_sums_kernel(const uint4* __restrict__ g, int W2, float* __restrict__ scratch) {
  __shared__ float red[16][129];
  const int64_t row = blockIdx.x;
  const int slot = threadIdx.x & 15;   // (j, cg): j = slot >> 3
  const int lane_p = threadIdx.x >> 4; // pixel-pair lane
  float s[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) s[e] = 0.f;
  const int n_slots = W2 * 8;          // uint4 per row; slot index within a pixel pair = (w&1)*8 + cg
  for (int i = lane_p * 16 + slot; i < n_slots; i += 256) {
    float f[8];
    unpack8(g[row * n_slots + i], f);
#pragma unroll
    for (int e = 0; e < 8; ++e) s[e] += f[e];
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) red[lane_p][slot * 8 + e] = s[e];
  __syncthreads();
  if (threadIdx.x < 128) {
    float acc = 0.f;
#pragma unroll
    for (int l = 0; l < 16; ++l) acc += red[l][threadIdx.x];
    scratch[row * 128 + threadIdx.x] = acc;  // [j*64 + c]
  }
}
// dbias[4c + 2i + j] = sum over rows with (row & 1) == i of scratch[row][j*64 + c]; one block per output, fixed-order tree
__global__ void __launch_bounds__(256) ps_bias_finalize_kernel(const float* __restrict__ scratch, int64_t rows, float* __restrict__ dbias) {
  __shared__ double sh[256];
  const int o = blockIdx.x;  // 256 = i(2) x j(2) x c(64)
  const int i = o >> 7, j = (o >> 6) & 1, c = o & 63;
  double acc = 0.0;
  for (int64_t r = i + 2 * int64_t(threadIdx.x); r < rows; r += 512) acc += double(scratch[r * 128 + j * 64 + c]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) dbias[4 * c + 2 * i + j] = float(sh[0]);
}
int launch_ps_bias_grad(const void* g, int N, int H2, int W2, float* scratch, float* dbias, cudaStream_t st) {
  if ((H2 & 1) || (W2 & 1)) { set_error("ps_bias_grad: odd extent"); return -1; }
  const int64_t rows = int64_t(N) * H2;
  ps_row_sums_kernel<<<unsigned(rows), 256, 0, st>>>(reinterpret_cast<const uint4*>(g), W2, scratch);
  SRG_LAUNCH_CHECK("ps_row_sums");
  ps_bias_finalize_kernel<<<256, 256, 0, st>>>(scratch, rows, dbias);
  SRG_LAUNCH_CHECK("ps_bias_finalize");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// unfold9: one thread per (pixel of the H+1 row grid, channel group of 8)
// ------------------------------------------------------------------------------------------------
// Where row hh (0 <= hh < H) of channel c of item n starts (row) and the value of its column ww (at): a dense [N,3,H,W]
// fp32 batch or a window of larger fp32 frames (launch_unfold9_windows), or the same two forms of 8-bit NHWC frames
// (launch_unfold9_u8 / launch_unfold9_windows_u8).  Both kernels below read their source through one of these.
struct PlainRows {
  const float* src;
  int64_t plane;
  int W;
  __device__ __forceinline__ const float* row(int n, int c, int hh) const {
    return src + (int64_t(n) * 3 + c) * plane + int64_t(hh) * W;
  }
  __device__ __forceinline__ float at(const float* r, int ww) const { return __ldg(r + ww); }
};
struct WindowRows {
  const float* src;
  WindowGather g;
  __device__ __forceinline__ const float* row(int n, int c, int hh) const {
    return src + g.base[n] + c * g.plane + int64_t(hh) * g.pitch;
  }
  __device__ __forceinline__ float at(const float* r, int ww) const { return __ldg(r + ww); }
};
// 8-bit pixels are 3 bytes (no alignment); a byte v becomes v / 255 with the same fp32 division as ToTensor
// (resample.cu), so conv1's bf16 operand, and every later bit, equals the fp32 path's for to_tensor(frames)
__device__ __forceinline__ float u8_to_unit(const uint8_t* p) { return __fdiv_rn(float(__ldg(p)), 255.f); }
struct PlainRowsU8 {
  const uint8_t* src;       // [N][H][W][3]
  int H, W;
  __device__ __forceinline__ const uint8_t* row(int n, int c, int hh) const {
    return src + ((int64_t(n) * H + hh) * W) * 3 + c;
  }
  __device__ __forceinline__ float at(const uint8_t* r, int ww) const { return u8_to_unit(r + 3 * ww); }
};
struct WindowRowsU8 {
  const uint8_t* src;
  WindowGather g;           // byte offsets: plane = 1 (channel stride), pitch = 3 x frame width
  __device__ __forceinline__ const uint8_t* row(int n, int c, int hh) const {
    return src + g.base[n] + c * g.plane + int64_t(hh) * g.pitch;
  }
  __device__ __forceinline__ float at(const uint8_t* r, int ww) const { return u8_to_unit(r + 3 * ww); }
};

template <class Rows>
__global__ void __launch_bounds__(256) unfold9_kernel(const __grid_constant__ Rows rows, int N, int H, int W, float scale,
                                                      uint4* __restrict__ dst) {
  // one thread per (n, h', w): gathers the 2 x 9 x 3 neighbourhood once and writes the pixel's 128-byte row
  const int64_t total = int64_t(N) * (H + 1) * W;
  for (int64_t pix = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; pix < total; pix += int64_t(gridDim.x) * blockDim.x) {
    const int w = int(pix % W);
    const int64_t t = pix / W;
    const int hp = int(t % (H + 1));
    const int n = int(t / (H + 1));
    float f[64];
#pragma unroll
    for (int ch = 54; ch < 64; ++ch) f[ch] = 0.f;
#pragma unroll
    for (int dr = 0; dr < 2; ++dr) {
      const int hh = hp - 1 + dr;
      const bool row_ok = hh >= 0 && hh < H;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const auto* row = rows.row(n, c, row_ok ? hh : 0);
#pragma unroll
        for (int sft = 0; sft < 9; ++sft) {
          const int ww = w + sft - 4;
          f[dr * 27 + sft * 3 + c] = (row_ok && ww >= 0 && ww < W) ? rows.at(row, ww) * scale : 0.f;
        }
      }
    }
    uint4* o = dst + pix * 8;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      uint4 v;
      v.x = bpack(f[8 * g + 0], f[8 * g + 1]); v.y = bpack(f[8 * g + 2], f[8 * g + 3]);
      v.z = bpack(f[8 * g + 4], f[8 * g + 5]); v.w = bpack(f[8 * g + 6], f[8 * g + 7]);
      o[g] = v;
    }
  }
}
// Same result for W % 128 == 0 (every training / inference size): one block = 128 consecutive pixels of one image row.  The
// two source rows x three planes (+4 halo pixels each side) are read ONCE into shared memory with coalesced loads, every
// thread assembles its pixel's 54 values from there, and the 16 KB of output go out as fully coalesced 16-byte vectors
// (the per-thread form issues 54 global loads per pixel and writes 128-byte rows with a 128-byte lane stride).
template <class Rows>
__global__ void __launch_bounds__(128) unfold9_tile_kernel(const __grid_constant__ Rows rows, int N, int H, int W, float scale,
                                                           uint4* __restrict__ dst) {
  __shared__ float tile[6][136];             // [dr * 3 + c][4 + 128 + 4]
  __shared__ uint4 stage[128 * 8];
  const int segs = W / 128;
  const int64_t total = int64_t(N) * (H + 1) * segs;
  const int tp = threadIdx.x;
  for (int64_t blk = blockIdx.x; blk < total; blk += gridDim.x) {
    const int seg = int(blk % segs);
    const int64_t t = blk / segs;
    const int hp = int(t % (H + 1));
    const int n = int(t / (H + 1));
    const int w0 = seg * 128;
    for (int i = tp; i < 6 * 136; i += 128) {
      const int r = i / 136, x = i - r * 136;
      const int dr = r / 3, c = r - dr * 3;
      const int hh = hp - 1 + dr, ww = w0 + x - 4;
      tile[r][x] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? rows.at(rows.row(n, c, hh), ww) * scale : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      float f[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int ch = 8 * g + e;                        // ch = dr * 27 + sft * 3 + c
        f[e] = ch < 54 ? tile[(ch / 27) * 3 + (ch % 27) % 3][tp + (ch % 27) / 3] : 0.f;
      }
      uint4 v;
      v.x = bpack(f[0], f[1]); v.y = bpack(f[2], f[3]); v.z = bpack(f[4], f[5]); v.w = bpack(f[6], f[7]);
      stage[tp * 8 + (g ^ (tp & 7))] = v;               // XOR swizzle: the 8 lanes of a quarter-warp hit 8 different columns
    }
    __syncthreads();
    uint4* o = dst + ((int64_t(n) * (H + 1) + hp) * W + w0) * 8;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int l = k * 128 + tp;                       // linear 16-byte index inside the block's 16 KB
      const int pp = l >> 3, g = l & 7;
      o[l] = stage[pp * 8 + (g ^ (pp & 7))];
    }
    __syncthreads();
  }
}
template <class Rows>
static int launch_unfold9_rows(const Rows& rows, int N, int H, int W, float scale, void* dst, cudaStream_t st) {
  const int64_t total = int64_t(N) * (H + 1) * W;
  if (W % 128 == 0) {
    int64_t blocks = int64_t(N) * (H + 1) * (W / 128);
    if (blocks > int64_t(sm_budget()) * 16) blocks = int64_t(sm_budget()) * 16;
    unfold9_tile_kernel<Rows><<<int(blocks), 128, 0, st>>>(rows, N, H, W, scale, reinterpret_cast<uint4*>(dst));
  } else {
    unfold9_kernel<Rows><<<ew_blocks(total), 256, 0, st>>>(rows, N, H, W, scale, reinterpret_cast<uint4*>(dst));
  }
  SRG_LAUNCH_CHECK("unfold9");
  return 0;
}
int launch_unfold9(const float* src, int N, int H, int W, float scale, void* dst, cudaStream_t st) {
  const PlainRows rows{src, int64_t(H) * W, W};
  return launch_unfold9_rows(rows, N, H, W, scale, dst, st);
}
int launch_unfold9_windows(const float* frames, const WindowGather& wg, int H, int W, void* dst, cudaStream_t st) {
  if (wg.n < 1 || wg.n > kMaxWindows) { set_error("unfold9_windows: 1..%d windows", kMaxWindows); return -1; }
  WindowRows rows;
  rows.src = frames;
  rows.g = wg;
  return launch_unfold9_rows(rows, wg.n, H, W, 1.f, dst, st);
}
int launch_unfold9_u8(const uint8_t* src, int N, int H, int W, void* dst, cudaStream_t st) {
  const PlainRowsU8 rows{src, H, W};
  return launch_unfold9_rows(rows, N, H, W, 1.f, dst, st);
}
int launch_unfold9_windows_u8(const uint8_t* frames, const WindowGather& wg, int H, int W, void* dst, cudaStream_t st) {
  if (wg.n < 1 || wg.n > kMaxWindows) { set_error("unfold9_windows_u8: 1..%d windows", kMaxWindows); return -1; }
  WindowRowsU8 rows;
  rows.src = frames;
  rows.g = wg;
  return launch_unfold9_rows(rows, wg.n, H, W, 1.f, dst, st);
}

// ------------------------------------------------------------------------------------------------
// window gather / scatter-add of the frozen-tiles backward: one thread per (item, channel, row, column) of the window
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t window_elem(const WindowTable& t, int i, int c, int h, int w) {
  return ((int64_t(t.frame[i]) * 3 + c) * t.fh + t.y0[i] + h) * t.fw + t.x0[i] + w;
}

__global__ void __launch_bounds__(256) crop_masked_gather_kernel(const float* __restrict__ frames,
                                                                 const __grid_constant__ WindowTable t, int H, int W,
                                                                 float* __restrict__ dst) {
  const int64_t total = int64_t(t.n) * 3 * H * W;
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += int64_t(gridDim.x) * blockDim.x) {
    const int w = int(e % W);
    const int64_t r = e / W;
    const int h = int(r % H);
    const int ic = int(r / H);
    const int i = ic / 3, c = ic - 3 * i;
    const bool in = h >= t.h_lo[i] && h < t.h_hi[i] && w >= t.w_lo[i] && w < t.w_hi[i];
    dst[e] = in ? __ldg(frames + window_elem(t, i, c, h, w)) : 0.f;
  }
}

__global__ void __launch_bounds__(256) window_scatter_add_kernel(const float* __restrict__ src,
                                                                 const __grid_constant__ WindowTable t, int H, int W,
                                                                 float* __restrict__ frames) {
  const int64_t total = int64_t(t.n) * 3 * H * W;
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += int64_t(gridDim.x) * blockDim.x) {
    const int w = int(e % W);
    const int64_t r = e / W;
    const int h = int(r % H);
    const int ic = int(r / H);
    const int i = ic / 3, c = ic - 3 * i;
    const int f = t.frame[i], y = t.y0[i] + h, x = t.x0[i] + w;
    auto covers = [&](int j) {
      return t.frame[j] == f && y >= t.y0[j] && y < t.y0[j] + H && x >= t.x0[j] && x < t.x0[j] + W;
    };
    // the first window that contains this frame element owns it; later ones are added by the owner, in order
    bool owner = true;
    for (int j = 0; j < i && owner; ++j) owner = !covers(j);
    if (!owner) continue;
    const int64_t o = window_elem(t, i, c, h, w);
    float acc = frames[o] + src[e];
    for (int j = i + 1; j < t.n; ++j)
      if (covers(j)) acc += src[((int64_t(j) * 3 + c) * H + (y - t.y0[j])) * W + (x - t.x0[j])];
    frames[o] = acc;
  }
}

int launch_crop_masked_gather(const float* frames, const WindowTable& wt, int H, int W, float* dst, cudaStream_t st) {
  if (wt.n < 1 || wt.n > kMaxWindows) { set_error("crop_masked_gather: 1..%d windows", kMaxWindows); return -1; }
  crop_masked_gather_kernel<<<ew_blocks(int64_t(wt.n) * 3 * H * W), 256, 0, st>>>(frames, wt, H, W, dst);
  SRG_LAUNCH_CHECK("crop_masked_gather");
  return 0;
}
int launch_window_scatter_add(const float* src, const WindowTable& wt, int H, int W, float* frames, cudaStream_t st) {
  if (wt.n < 1 || wt.n > kMaxWindows) { set_error("window_scatter_add: 1..%d windows", kMaxWindows); return -1; }
  window_scatter_add_kernel<<<ew_blocks(int64_t(wt.n) * 3 * H * W), 256, 0, st>>>(src, wt, H, W, frames);
  SRG_LAUNCH_CHECK("window_scatter_add");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// parameters
// ------------------------------------------------------------------------------------------------
__global__ void pack_bf16_kernel(const float* __restrict__ src, const int* __restrict__ idx, __nv_bfloat16* __restrict__ dst,
                                 int64_t n) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int j = idx[i];
    dst[i] = __float2bfloat16_rn(j >= 0 ? src[j] : 0.f);
  }
}
int launch_pack_bf16(const float* src, const int* idx, void* dst, int64_t n, cudaStream_t st) {
  if (n <= 0) return 0;
  pack_bf16_kernel<<<ew_blocks(n), 256, 0, st>>>(src, idx, reinterpret_cast<__nv_bfloat16*>(dst), n);
  SRG_LAUNCH_CHECK("pack_bf16");
  return 0;
}
__global__ void gather_f32_kernel(const float* __restrict__ src, const int* __restrict__ idx, float* __restrict__ dst, int64_t n) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int j = idx[i];
    dst[i] = j >= 0 ? src[j] : 0.f;
  }
}
int launch_gather_f32(const float* src, const int* idx, float* dst, int64_t n, cudaStream_t st) {
  if (n <= 0) return 0;
  gather_f32_kernel<<<ew_blocks(n), 256, 0, st>>>(src, idx, dst, n);
  SRG_LAUNCH_CHECK("gather_f32");
  return 0;
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, int64_t n, float lr_over_bc1, float beta1,
                                                   float beta2, float eps, float inv_sqrt_bc2, float grad_scale) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const float gi = g[i] * grad_scale;
    const float mi = m[i] + (gi - m[i]) * (1.f - beta1);          // torch: exp_avg.lerp_(grad, 1-beta1)
    const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;       // exp_avg_sq.mul_(b2).addcmul_(g, g, 1-b2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;           // (sqrt(v)/sqrt(bc2)).add_(eps)
    p[i] -= lr_over_bc1 * (mi / denom);                            // addcdiv_(m, denom, -lr/bc1)
  }
}
int launch_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                int step, float grad_scale, cudaStream_t st) {
  if (n <= 0) return 0;
  const double bc1 = 1.0 - pow(double(beta1), double(step));
  const double bc2 = 1.0 - pow(double(beta2), double(step));
  adam_kernel<<<ew_blocks(n), 256, 0, st>>>(p, g, m, v, n, float(double(lr) / bc1), beta1, beta2, eps,
                                            float(1.0 / sqrt(bc2)), grad_scale);
  SRG_LAUNCH_CHECK("adam");
  return 0;
}

// Graph-capturable variant: learning rate and step count live in device memory, so a captured launch stays valid while
// the host scheduler changes the LR and the step advances (bias corrections are computed on the device).
__global__ void __launch_bounds__(256) adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                       float* __restrict__ v, int64_t n, const float* __restrict__ lr_dev,
                                                       float beta1, float beta2, float eps, const int* __restrict__ step_dev,
                                                       float grad_scale) {
  const int t = *step_dev + 1;
  const double bc1 = 1.0 - pow(double(beta1), double(t));
  const double bc2 = 1.0 - pow(double(beta2), double(t));
  const float lr_over_bc1 = float(double(*lr_dev) / bc1);
  const float inv_sqrt_bc2 = float(1.0 / sqrt(bc2));
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const float gi = g[i] * grad_scale;
    const float mi = m[i] + (gi - m[i]) * (1.f - beta1);
    const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
    p[i] -= lr_over_bc1 * (mi / denom);
  }
}
__global__ void step_inc_kernel(int* step_dev) { *step_dev += 1; }
int launch_adam_dev(float* p, const float* g, float* m, float* v, int64_t n, const float* lr_dev, float beta1, float beta2,
                    float eps, int* step_dev, float grad_scale, cudaStream_t st) {
  if (n <= 0) return 0;
  adam_dev_kernel<<<ew_blocks(n), 256, 0, st>>>(p, g, m, v, n, lr_dev, beta1, beta2, eps, step_dev, grad_scale);
  SRG_LAUNCH_CHECK("adam_dev");
  step_inc_kernel<<<1, 1, 0, st>>>(step_dev);
  SRG_LAUNCH_CHECK("adam_step_inc");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// ReconstructionLoss
// ------------------------------------------------------------------------------------------------
constexpr int kLossBlocks = 1184;  // 8 x 148
constexpr int kLossHdr = 16;
int loss_scratch_doubles() { return kLossHdr + 3 * kLossBlocks + 64; }

__device__ __forceinline__ double block_sum_256(double v, double* sh) {
  // warp shuffle, then 8 warp totals in shared memory (fixed order)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[w] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) t += sh[i];
  return t;
}

// Row-wise helpers: r0/r1/r2 = rows h-1, h, h+1 of one image plane (nullptr when outside), zero padding.
struct Rows3 {
  const float* r0;
  const float* r1;
  const float* r2;
};
__device__ __forceinline__ Rows3 rows3(const float* __restrict__ plane_base, int h, int H, int W) {
  Rows3 r;
  r.r1 = plane_base + int64_t(h) * W;
  r.r0 = h > 0 ? r.r1 - W : nullptr;
  r.r2 = h + 1 < H ? r.r1 + W : nullptr;
  return r;
}
__device__ __forceinline__ float ldz(const float* __restrict__ row, int w, int W) {
  return (row != nullptr && w >= 0 && w < W) ? __ldg(row + w) : 0.f;
}
// E0 = max(|Px * x|, |Py * x|), Prewitt x5, zero padding (src/utils.py:180-186, 200-209)
__device__ __forceinline__ float edge0(const Rows3& r, int w, int W) {
  const float a = ldz(r.r0, w - 1, W), b = ldz(r.r0, w, W), c = ldz(r.r0, w + 1, W);
  const float d = ldz(r.r1, w - 1, W), f = ldz(r.r1, w + 1, W);
  const float g = ldz(r.r2, w - 1, W), i = ldz(r.r2, w, W), j = ldz(r.r2, w + 1, W);
  const float gx = 5.f * ((c - a) + (f - d) + (j - g));
  const float gy = 5.f * ((g - a) + (i - b) + (j - c));
  return fmaxf(fabsf(gx), fabsf(gy));
}
// L * x with L = [[-1/8 x3],[-1/8, 1, -1/8],[-1/8 x3]] (src/utils.py:190-192)
__device__ __forceinline__ float lap8(const Rows3& r, int w, int W) {
  const float nb = ldz(r.r0, w - 1, W) + ldz(r.r0, w, W) + ldz(r.r0, w + 1, W) + ldz(r.r1, w - 1, W) + ldz(r.r1, w + 1, W) +
                   ldz(r.r2, w - 1, W) + ldz(r.r2, w, W) + ldz(r.r2, w + 1, W);
  return __ldg(r.r1 + w) - 0.125f * nb;
}
// 4 consecutive pixels of a row plus their left / right neighbours: v[0] = x[w-1], v[1..4] = x[w..w+3], v[5] = x[w+4]
struct Row6 { float v[6]; };
__device__ __forceinline__ Row6 load_row6(const float* __restrict__ row, int w, int W) {
  Row6 r;
  if (row == nullptr) {
#pragma unroll
    for (int i = 0; i < 6; ++i) r.v[i] = 0.f;
    return r;
  }
  const float4 c = __ldg(reinterpret_cast<const float4*>(row + w));     // w % 4 == 0, W % 4 == 0, row 16-byte aligned
  r.v[1] = c.x; r.v[2] = c.y; r.v[3] = c.z; r.v[4] = c.w;
  r.v[0] = w > 0 ? __ldg(row + w - 1) : 0.f;
  r.v[5] = w + 4 < W ? __ldg(row + w + 4) : 0.f;
  return r;
}
__device__ __forceinline__ float edge0_v(const Row6& a, const Row6& b, const Row6& c, int i) {   // pixel i (0..3) of the quad
  const float gx = 5.f * ((a.v[i + 2] - a.v[i]) + (b.v[i + 2] - b.v[i]) + (c.v[i + 2] - c.v[i]));
  const float gy = 5.f * ((c.v[i] - a.v[i]) + (c.v[i + 1] - a.v[i + 1]) + (c.v[i + 2] - a.v[i + 2]));
  return fmaxf(fabsf(gx), fabsf(gy));
}
__device__ __forceinline__ float lap8_v(const Row6& a, const Row6& b, const Row6& c, int i) {
  const float nb = a.v[i] + a.v[i + 1] + a.v[i + 2] + b.v[i] + b.v[i + 2] + c.v[i] + c.v[i + 1] + c.v[i + 2];
  return b.v[i + 1] - 0.125f * nb;
}
constexpr int kLossThreads = 128;
__device__ __forceinline__ double block_sum_any(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < nw; ++i) t += sh[i];
  return t;
}

// All three passes walk image rows: block -> rows (grid stride), thread -> columns; no per-element divisions.
// Passes 1 and 2 take STRIPS of consecutive rows of one plane per iteration when W % 4 == 0: every input row of a strip is
// loaded once for the up to three output rows that use it, and all of a strip's loads are independent of its arithmetic, so
// a thread has 6 (pass 1) / 8 (pass 2) row loads in flight instead of 3 / 6 per dependent round (the row-by-row form was
// bound by one DRAM round trip per row: 28 MB in 21 us).  Each row's fp32 partial sums are formed exactly as before and
// added in double, so only the order of the double additions differs from the row-by-row form.
constexpr int kLossStrip1 = 4;
constexpr int kLossStrip2 = 2;
__global__ void __launch_bounds__(kLossThreads) loss_pass1_kernel(const float* __restrict__ hr, int rows_total, int H, int W,
                                                                  double* __restrict__ scratch) {
  __shared__ double sh[8];
  double s1 = 0.0, s2 = 0.0;
  if ((W & 3) == 0) {
    const int strips_per_plane = (H + kLossStrip1 - 1) / kLossStrip1;
    const int strips_total = (rows_total / H) * strips_per_plane;
    for (int strip = blockIdx.x; strip < strips_total; strip += gridDim.x) {
      const int pl = strip / strips_per_plane, h0 = (strip - pl * strips_per_plane) * kLossStrip1;
      const float* plane = hr + int64_t(pl) * H * W;
      for (int w = threadIdx.x * 4; w < W; w += kLossThreads * 4) {
        Row6 r[kLossStrip1 + 2];
#pragma unroll
        for (int i = 0; i < kLossStrip1 + 2; ++i) {
          const int h = h0 - 1 + i;
          r[i] = load_row6((h >= 0 && h < H) ? plane + int64_t(h) * W : nullptr, w, W);
        }
#pragma unroll
        for (int i = 0; i < kLossStrip1; ++i) {
          if (h0 + i < H) {
            float a1 = 0.f, a2 = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float e0 = edge0_v(r[i], r[i + 1], r[i + 2], k);
              a1 += e0;
              a2 += e0 * e0;
            }
            s1 += double(a1);
            s2 += double(a2);
          }
        }
      }
    }
  } else {
    for (int row = blockIdx.x; row < rows_total; row += gridDim.x) {
      const int pl = row / H, h = row - pl * H;
      const Rows3 r = rows3(hr + int64_t(pl) * H * W, h, H, W);
      float a1 = 0.f, a2 = 0.f;
      for (int w = threadIdx.x; w < W; w += kLossThreads) {
        const float e0 = edge0(r, w, W);
        a1 += e0;
        a2 += e0 * e0;
      }
      s1 += double(a1);
      s2 += double(a2);
    }
  }
  s1 = block_sum_any(s1, sh);
  s2 = block_sum_any(s2, sh);
  if (threadIdx.x == 0) {
    scratch[kLossHdr + blockIdx.x] = s1;
    scratch[kLossHdr + kLossBlocks + blockIdx.x] = s2;
  }
}
// 256 threads; sums `cnt` arrays of kLossBlocks partials into hdr[dst0 ...]
__device__ void sum_partials(double* scratch, int which, int blocks, double* out, double* sh) {
  double acc = 0.0;
  for (int b = threadIdx.x; b < blocks; b += 256) acc += scratch[kLossHdr + which * kLossBlocks + b];
  acc = block_sum_256(acc, sh);
  if (threadIdx.x == 0) *out = acc;
}
__global__ void loss_stats_kernel(double* scratch, int blocks, double n) {
  __shared__ double sh[8];
  sum_partials(scratch, 0, blocks, &scratch[0], sh);
  sum_partials(scratch, 1, blocks, &scratch[1], sh);
  __syncthreads();
  if (threadIdx.x == 0) {
    const double mean = scratch[0] / n;
    double var = (scratch[1] - n * mean * mean) / (n - 1.0);  // torch.std: unbiased
    if (var < 0.0) var = 0.0;
    scratch[2] = mean;
    scratch[3] = sqrt(var);
  }
}
__global__ void __launch_bounds__(kLossThreads) loss_pass2_kernel(const float* __restrict__ hr, const float* __restrict__ sr,
                                                                  int rows_total, int H, int W, double* __restrict__ scratch,
                                                                  float* __restrict__ e_buf, float* __restrict__ g_buf) {
  __shared__ double sh[8];
  const float mean = float(scratch[2]), stdv = float(scratch[3]);
  double sE = 0.0, sL = 0.0, sT = 0.0;
  if ((W & 3) == 0) {
    const int strips_per_plane = (H + kLossStrip2 - 1) / kLossStrip2;
    const int strips_total = (rows_total / H) * strips_per_plane;
    for (int strip = blockIdx.x; strip < strips_total; strip += gridDim.x) {
      const int pl = strip / strips_per_plane, h0 = (strip - pl * strips_per_plane) * kLossStrip2;
      const int64_t pbase = int64_t(pl) * H * W;
      for (int w = threadIdx.x * 4; w < W; w += kLossThreads * 4) {
        Row6 hrow[kLossStrip2 + 2], srow[kLossStrip2 + 2];
#pragma unroll
        for (int i = 0; i < kLossStrip2 + 2; ++i) {
          const int h = h0 - 1 + i;
          const bool in = h >= 0 && h < H;
          hrow[i] = load_row6(in ? hr + pbase + int64_t(h) * W : nullptr, w, W);
          srow[i] = load_row6(in ? sr + pbase + int64_t(h) * W : nullptr, w, W);
        }
#pragma unroll
        for (int i = 0; i < kLossStrip2; ++i) {
          if (h0 + i < H) {
            const int64_t o = pbase + int64_t(h0 + i) * W;
            float aE = 0.f, aL = 0.f, aT = 0.f;
            float ev[4], gv[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float e0 = edge0_v(hrow[i], hrow[i + 1], hrow[i + 2], k);
              float e = (e0 - mean) / stdv * 0.2f + 1.f;                 // normalize(...)*0.2 + 1  (:213, :194-198)
              e = fminf(fmaxf(e, 0.f), 2.f);
              const float d = lap8_v(srow[i], srow[i + 1], srow[i + 2], k);
              const float om = 1.f - e;
              ev[k] = e;
              gv[k] = (d > 0.f ? om : (d < 0.f ? -om : 0.f));            // sign(D) * (1 - E)
              aE += e;
              aL += fabsf(hrow[i + 1].v[k + 1] - srow[i + 1].v[k + 1]) * e;
              aT += fabsf(d) * om;
            }
            *reinterpret_cast<float4*>(e_buf + o + w) = make_float4(ev[0], ev[1], ev[2], ev[3]);
            *reinterpret_cast<float4*>(g_buf + o + w) = make_float4(gv[0], gv[1], gv[2], gv[3]);
            sE += double(aE);
            sL += double(aL);
            sT += double(aT);
          }
        }
      }
    }
  } else {
    for (int row = blockIdx.x; row < rows_total; row += gridDim.x) {
      const int pl = row / H, h = row - pl * H;
      const int64_t pbase = int64_t(pl) * H * W;
      const Rows3 rh = rows3(hr + pbase, h, H, W);
      const Rows3 rs = rows3(sr + pbase, h, H, W);
      const int64_t o = pbase + int64_t(h) * W;
      float aE = 0.f, aL = 0.f, aT = 0.f;
      for (int w = threadIdx.x; w < W; w += kLossThreads) {
        const float e0 = edge0(rh, w, W);
        float e = (e0 - mean) / stdv * 0.2f + 1.f;                 // normalize(...)*0.2 + 1  (:213, :194-198)
        e = fminf(fmaxf(e, 0.f), 2.f);
        const float d = lap8(rs, w, W);
        const float om = 1.f - e;
        e_buf[o + w] = e;
        g_buf[o + w] = (d > 0.f ? om : (d < 0.f ? -om : 0.f));    // sign(D) * (1 - E)
        aE += e;
        aL += fabsf(__ldg(rh.r1 + w) - __ldg(rs.r1 + w)) * e;
        aT += fabsf(d) * om;
      }
      sE += double(aE);
      sL += double(aL);
      sT += double(aT);
    }
  }
  sE = block_sum_any(sE, sh);
  sL = block_sum_any(sL, sh);
  sT = block_sum_any(sT, sh);
  if (threadIdx.x == 0) {
    scratch[kLossHdr + blockIdx.x] = sE;
    scratch[kLossHdr + kLossBlocks + blockIdx.x] = sL;
    scratch[kLossHdr + 2 * kLossBlocks + blockIdx.x] = sT;
  }
}
__global__ void loss_final_kernel(double* scratch, int blocks, double n, float* losses) {
  __shared__ double sh[8];
  sum_partials(scratch, 0, blocks, &scratch[4], sh);
  sum_partials(scratch, 1, blocks, &scratch[5], sh);
  sum_partials(scratch, 2, blocks, &scratch[6], sh);
  __syncthreads();
  if (threadIdx.x == 0) {
    const double edge = scratch[5] / scratch[4];
    const double m = scratch[6] / n;
    scratch[7] = m;
    losses[0] = float(edge);
    losses[1] = float(m > 0.0 ? m : 0.0);
  }
}
__global__ void __launch_bounds__(kLossThreads) loss_pass3_kernel(const float* __restrict__ hr, const float* __restrict__ sr,
                                                                  const float* __restrict__ e_buf, const float* __restrict__ g_buf,
                                                                  int rows_total, int64_t total, int H, int W,
                                                                  const double* __restrict__ scratch,
                                                                  const float* __restrict__ w_edge, const float* __restrict__ w_tv,
                                                                  float* __restrict__ grad, float grad_scale) {
  // w_edge / w_tv: optional device scalars = d(objective)/d(edge_loss), d(objective)/d(tv_loss) (autograd inputs)
  const float inv_sum_e = float(1.0 / scratch[4]) * (w_edge ? *w_edge : 1.f);
  const float tv_k = scratch[7] > 0.0 ? float(1.0 / double(total)) * (w_tv ? *w_tv : 1.f) : 0.f;
  for (int row = blockIdx.x; row < rows_total; row += gridDim.x) {
    const int pl = row / H, h = row - pl * H;
    const int64_t pbase = int64_t(pl) * H * W;
    const Rows3 rg = rows3(g_buf + pbase, h, H, W);
    const int64_t o = pbase + int64_t(h) * W;
    if ((W & 3) == 0) {
      for (int w = threadIdx.x * 4; w < W; w += kLossThreads * 4) {
        const float4 s4 = __ldg(reinterpret_cast<const float4*>(sr + o + w));
        const float4 h4 = __ldg(reinterpret_cast<const float4*>(hr + o + w));
        const float4 e4 = __ldg(reinterpret_cast<const float4*>(e_buf + o + w));
        const float sv[4] = {s4.x, s4.y, s4.z, s4.w}, hv[4] = {h4.x, h4.y, h4.z, h4.w}, ev[4] = {e4.x, e4.y, e4.z, e4.w};
        float gout[4];
        Row6 ga, gb, gc;
        if (tv_k != 0.f) { ga = load_row6(rg.r0, w, W); gb = load_row6(rg.r1, w, W); gc = load_row6(rg.r2, w, W); }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float diff = sv[i] - hv[i];
          const float sg = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
          float g = sg * ev[i] * inv_sum_e;
          if (tv_k != 0.f) g += tv_k * lap8_v(ga, gb, gc, i);
          gout[i] = g * grad_scale;
        }
        *reinterpret_cast<float4*>(grad + o + w) = make_float4(gout[0], gout[1], gout[2], gout[3]);
      }
    } else
    for (int w = threadIdx.x; w < W; w += kLossThreads) {
      const float diff = sr[o + w] - hr[o + w];
      const float sg = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
      float g = sg * e_buf[o + w] * inv_sum_e;
      if (tv_k != 0.f) g += tv_k * lap8(rg, w, W);
      grad[o + w] = g * grad_scale;
    }
  }
}
// grid of pass `which` (0 / 1): min(work units, resident blocks of the current device, kLossBlocks partial-sum rows)
static int loss_grid(int which, int units) {
  int dev = 0, sms = 148, per_sm = 4;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (which == 0) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, loss_pass1_kernel, kLossThreads, 0);
  else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, loss_pass2_kernel, kLossThreads, 0);
  if (per_sm < 1) per_sm = 1;
  int blocks = sms * per_sm;
  if (blocks > kLossBlocks) blocks = kLossBlocks;
  if (blocks > units) blocks = units;
  return blocks < 1 ? 1 : blocks;
}
int launch_recon_loss_forward(const float* hr, const float* sr, int N, int C, int H, int W, double* scratch, float* e_buf,
                              float* g_buf, float* losses, cudaStream_t st) {
  const int64_t total = int64_t(N) * C * H * W;
  if (total <= 1) { set_error("recon_loss: need more than one element"); return -1; }
  const int64_t rows64 = int64_t(N) * C * H;
  if (rows64 > 0x7fffffff) { set_error("recon_loss: too many rows"); return -1; }
  const int rows = int(rows64);
  // one wave of resident blocks (the strip forms hold 72 / 92 registers per thread: 7 / 5 blocks of 128 threads per SM);
  // a block that found no work still writes its (zero) partial sums, so the finalize kernels sum exactly `blocks` rows
  const bool strips = (W & 3) == 0;
  const int units1 = strips ? (rows / H) * ((H + kLossStrip1 - 1) / kLossStrip1) : rows;
  const int units2 = strips ? (rows / H) * ((H + kLossStrip2 - 1) / kLossStrip2) : rows;
  const int blocks1 = loss_grid(0, units1), blocks2 = loss_grid(1, units2);
  loss_pass1_kernel<<<blocks1, kLossThreads, 0, st>>>(hr, rows, H, W, scratch);
  SRG_LAUNCH_CHECK("loss_pass1");
  loss_stats_kernel<<<1, 256, 0, st>>>(scratch, blocks1, double(total));
  SRG_LAUNCH_CHECK("loss_stats");
  loss_pass2_kernel<<<blocks2, kLossThreads, 0, st>>>(hr, sr, rows, H, W, scratch, e_buf, g_buf);
  SRG_LAUNCH_CHECK("loss_pass2");
  loss_final_kernel<<<1, 256, 0, st>>>(scratch, blocks2, double(total), losses);
  SRG_LAUNCH_CHECK("loss_final");
  return 0;
}
int launch_recon_loss_backward(const float* hr, const float* sr, int N, int C, int H, int W, const double* scratch,
                               const float* e_buf, const float* g_buf, const float* w_edge, const float* w_tv, float* grad,
                               float grad_scale, cudaStream_t st) {
  const int64_t total = int64_t(N) * C * H * W;
  const int rows = int(int64_t(N) * C * H);
  const int blocks = rows < kLossBlocks ? rows : kLossBlocks;
  loss_pass3_kernel<<<blocks, kLossThreads, 0, st>>>(hr, sr, e_buf, g_buf, rows, total, H, W, scratch, w_edge, w_tv, grad,
                                                    grad_scale);
  SRG_LAUNCH_CHECK("loss_pass3");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// evaluation path: ImageEnhancer (src/models.py:28-41) and the PSNR numerator (src/utils.py:141-144)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kLossThreads) enhance_kernel(const float* __restrict__ x, int rows_total, int H, int W,
                                                               float factor, float* __restrict__ out) {
  for (int row = blockIdx.x; row < rows_total; row += gridDim.x) {
    const int pl = row / H, h = row - pl * H;
    const int64_t pbase = int64_t(pl) * H * W;
    const Rows3 r = rows3(x + pbase, h, H, W);
    const int64_t o = pbase + int64_t(h) * W;
    for (int w = threadIdx.x; w < W; w += kLossThreads) {
      const float v = __ldg(r.r1 + w) + factor * lap8(r, w, W);     // x + factor * (L * x), zero padding
      out[o + w] = fminf(fmaxf(v, 0.f), 1.f);                        // torch.clamp(x, 0, 1)
    }
  }
}
int launch_image_enhance(const float* x, int N, int C, int H, int W, float factor, float* out, cudaStream_t st) {
  const int64_t rows64 = int64_t(N) * C * H;
  if (rows64 <= 0 || rows64 > 0x7fffffff) { set_error("image_enhance: bad shape"); return -1; }
  const int rows = int(rows64);
  enhance_kernel<<<rows < 8 * 1184 ? rows : 8 * 1184, kLossThreads, 0, st>>>(x, rows, H, W, factor, out);
  SRG_LAUNCH_CHECK("image_enhance");
  return 0;
}
__global__ void __launch_bounds__(256) sqdiff_kernel(const float* __restrict__ a, const float* __restrict__ b, int64_t n,
                                                     double* __restrict__ scratch) {
  __shared__ double sh[8];
  double acc = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * 256 + threadIdx.x; i < n; i += int64_t(gridDim.x) * 256) {
    const float d = a[i] - b[i];
    acc += double(d) * double(d);
  }
  acc = block_sum_256(acc, sh);
  if (threadIdx.x == 0) scratch[kLossHdr + blockIdx.x] = acc;
}
__global__ void sqdiff_final_kernel(double* scratch, int blocks, double n, double* out) {
  __shared__ double sh[8];
  sum_partials(scratch, 0, blocks, &scratch[9], sh);
  __syncthreads();
  if (threadIdx.x == 0) out[0] = scratch[9] / n;
}
int launch_mse(const float* a, const float* b, int64_t n, double* scratch, double* out, cudaStream_t st) {
  if (n <= 0) { set_error("mse: empty input"); return -1; }
  const int blocks = int((n + 255) / 256 < kLossBlocks ? (n + 255) / 256 : kLossBlocks);
  sqdiff_kernel<<<blocks, 256, 0, st>>>(a, b, n, scratch);
  SRG_LAUNCH_CHECK("sqdiff");
  sqdiff_final_kernel<<<1, 256, 0, st>>>(scratch, blocks, double(n), out);
  SRG_LAUNCH_CHECK("sqdiff_final");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// plain pixel losses named by the north_star (L1 / MSE) and the discriminator BCE: 128-bit vectorised
// mean reductions with the gradient written in the same pass (oracle: torch.nn.functional)
// ------------------------------------------------------------------------------------------------
template <int KIND>  // 0: L1 mean |a-b|, 1: MSE mean (a-b)^2, 2: BCE mean -(t log p + (1-t) log(1-p)), a = p, b = t
__device__ __forceinline__ void point_loss(float a, float b, float gk, float& val, float& ga) {
  if (KIND == 0) {
    const float d = a - b;
    val = fabsf(d);
    ga = (d > 0.f ? gk : (d < 0.f ? -gk : 0.f));
  } else if (KIND == 1) {
    const float d = a - b;
    val = d * d;
    ga = 2.f * d * gk;
  } else {
    const float lp = fmaxf(logf(a), -100.f), lq = fmaxf(logf(1.f - a), -100.f);     // torch clamps the logs at -100
    val = -(b * lp + (1.f - b) * lq);
    ga = (a - b) / fmaxf(a * (1.f - a), 1e-12f) * gk;                                 // torch: (p - t) / max(p(1-p), eps)
  }
}
template <int KIND>
__global__ void __launch_bounds__(256) point_loss_kernel(const float* __restrict__ a, const float* __restrict__ b, int64_t n,
                                                         double* __restrict__ scratch, float* __restrict__ grad_a, float gk) {
  __shared__ double sh[8];
  double acc = 0.0;
  const int64_t n4 = n >> 2;
  for (int64_t i = int64_t(blockIdx.x) * 256 + threadIdx.x; i < n4; i += int64_t(gridDim.x) * 256) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(a) + i), y = __ldg(reinterpret_cast<const float4*>(b) + i);
    float v0, v1, v2, v3;
    float4 g;
    point_loss<KIND>(x.x, y.x, gk, v0, g.x);
    point_loss<KIND>(x.y, y.y, gk, v1, g.y);
    point_loss<KIND>(x.z, y.z, gk, v2, g.z);
    point_loss<KIND>(x.w, y.w, gk, v3, g.w);
    acc += double((v0 + v1) + (v2 + v3));
    if (grad_a) reinterpret_cast<float4*>(grad_a)[i] = g;
  }
  if (blockIdx.x == 0 && threadIdx.x < int(n & 3)) {      // tail (n not a multiple of 4)
    const int64_t i = (n4 << 2) + threadIdx.x;
    float v, g;
    point_loss<KIND>(a[i], b[i], gk, v, g);
    acc += double(v);
    if (grad_a) grad_a[i] = g;
  }
  acc = block_sum_256(acc, sh);
  if (threadIdx.x == 0) scratch[kLossHdr + blockIdx.x] = acc;
}
__global__ void point_loss_final_kernel(double* scratch, int blocks, double n, float* out) {
  __shared__ double sh[8];
  sum_partials(scratch, 0, blocks, &scratch[10], sh);
  __syncthreads();
  if (threadIdx.x == 0) out[0] = float(scratch[10] / n);
}
int launch_point_loss(int kind, const float* a, const float* b, int64_t n, double* scratch, float* out, float* grad_a,
                      float grad_scale, cudaStream_t st) {
  if (n <= 0) { set_error("point_loss: empty input"); return -1; }
  if (((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(grad_a)) & 15) != 0) {
    set_error("point_loss: pointers must be 16-byte aligned"); return -2;
  }
  const int64_t n4 = (n + 3) / 4;
  const int blocks = int((n4 + 255) / 256 < kLossBlocks ? (n4 + 255) / 256 : kLossBlocks);
  const float gk = grad_scale / float(n);
  if (kind == 0) point_loss_kernel<0><<<blocks, 256, 0, st>>>(a, b, n, scratch, grad_a, gk);
  else if (kind == 1) point_loss_kernel<1><<<blocks, 256, 0, st>>>(a, b, n, scratch, grad_a, gk);
  else if (kind == 2) point_loss_kernel<2><<<blocks, 256, 0, st>>>(a, b, n, scratch, grad_a, gk);
  else { set_error("point_loss: kind must be 0 (L1), 1 (MSE) or 2 (BCE)"); return -3; }
  SRG_LAUNCH_CHECK("point_loss");
  point_loss_final_kernel<<<1, 256, 0, st>>>(scratch, blocks, double(n), out);
  SRG_LAUNCH_CHECK("point_loss_final");
  return 0;
}

// per-channel sums of NCHW fp32: grid = (chunks, N*C)
__global__ void __launch_bounds__(256) nchw_plane_sum_kernel(const float* __restrict__ x, int64_t plane, double* __restrict__ scratch) {
  __shared__ double sh[8];
  const float* pl = x + int64_t(blockIdx.y) * plane;
  double acc = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * 256 + threadIdx.x; i < plane; i += int64_t(gridDim.x) * 256) acc += double(pl[i]);
  acc = block_sum_256(acc, sh);
  if (threadIdx.x == 0) scratch[int64_t(blockIdx.y) * gridDim.x + blockIdx.x] = acc;
}
__global__ void __launch_bounds__(256) nchw_chan_final_kernel(const double* __restrict__ scratch, int N, int C, int chunks,
                                                              float* out, float scale) {
  // one block per channel; fixed-order tree over the N x chunks partial sums
  __shared__ double sh[256];
  const int c = blockIdx.x;
  const int total = N * chunks;
  double acc = 0.0;
  for (int i = threadIdx.x; i < total; i += 256) {
    const int n = i / chunks, k = i - n * chunks;
    acc += scratch[(int64_t(n) * C + c) * chunks + k];
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[c] = float(sh[0]) * scale;
}
int launch_nchw_chan_sum(const float* x, int N, int C, int64_t plane, double* scratch, float* out, float scale,
                         cudaStream_t st) {
  int chunks = int((plane + 256 * 16 - 1) / (256 * 16));
  if (chunks > 64) chunks = 64;
  if (chunks < 1) chunks = 1;
  // scratch needs N*C*chunks doubles; callers size it with loss_scratch_doubles() >= 16 + 3*1184 (N*C*chunks <= that)
  if (int64_t(N) * C * chunks > 3 * kLossBlocks) chunks = int(3 * kLossBlocks / (int64_t(N) * C)) > 0 ? int(3 * kLossBlocks / (int64_t(N) * C)) : 1;
  if (int64_t(N) * C * chunks > 3 * kLossBlocks) { set_error("nchw_chan_sum: batch too large for scratch"); return -1; }
  nchw_plane_sum_kernel<<<dim3(chunks, N * C), 256, 0, st>>>(x, plane, scratch + kLossHdr);
  SRG_LAUNCH_CHECK("nchw_plane_sum");
  nchw_chan_final_kernel<<<C, 256, 0, st>>>(scratch + kLossHdr, N, C, chunks, out, scale);
  SRG_LAUNCH_CHECK("nchw_chan_final");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// mean(tanh(sign * (a - b))) and its gradients
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tanh_mean_kernel(const float* __restrict__ a, const float* __restrict__ b, int64_t n,
                                                        float sign, double* __restrict__ scratch, float* da, float* db,
                                                        float gk) {
  __shared__ double sh[8];
  double acc = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * 256 + threadIdx.x; i < n; i += int64_t(gridDim.x) * 256) {
    const float t = tanhf(sign * (a[i] - b[i]));
    acc += double(t);
    const float g = sign * (1.f - t * t) * gk;
    if (da) da[i] = g;
    if (db) db[i] = -g;
  }
  acc = block_sum_256(acc, sh);
  if (threadIdx.x == 0) scratch[kLossHdr + blockIdx.x] = acc;
}
__global__ void tanh_mean_final_kernel(double* scratch, int blocks, double n, float* out) {
  __shared__ double sh[8];
  sum_partials(scratch, 0, blocks, &scratch[8], sh);
  __syncthreads();
  if (threadIdx.x == 0) out[0] = float(scratch[8] / n);
}
int launch_tanh_mean(const float* a, const float* b, int64_t n, float sign, double* scratch, float* out, float* da,
                     float* db, float gscale, cudaStream_t st) {
  if (n <= 0) { set_error("tanh_mean: empty input"); return -1; }
  int blocks = int((n + 255) / 256 < kLossBlocks ? (n + 255) / 256 : kLossBlocks);
  tanh_mean_kernel<<<blocks, 256, 0, st>>>(a, b, n, sign, scratch, da, db, gscale / float(n));
  SRG_LAUNCH_CHECK("tanh_mean");
  tanh_mean_final_kernel<<<1, 256, 0, st>>>(scratch, blocks, double(n), out);
  SRG_LAUNCH_CHECK("tanh_mean_final");
  return 0;
}

}  // namespace srg
