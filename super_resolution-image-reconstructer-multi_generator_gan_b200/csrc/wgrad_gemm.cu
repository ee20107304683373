// Weight-gradient implicit GEMM for sm_100a.
//
//   D_t[ci][co] = sum over pixels p of  x[p + shift_t][ci] * dy[p][co]          (one 64x64 block per tap t)
//
// The reduction (GEMM K) dimension is the pixel index, so both operands are "MN-major": a shared-memory row is
// one pixel's 64 channels (128 bytes, 128B-swizzled by TMA), exactly the tiles the forward kernel loads.  Two taps
// are paired into one M=128 MMA: the A descriptor's leading-dimension byte offset is the distance between the two
// taps' row-shifted views of the same input strips.  Every CTA keeps all tap accumulators resident in TMEM across
// its pixel tiles (split-K over CTAs) and writes one fp32 partial block at the end; wgrad_reduce_kernel sums the
// partials in a fixed order (deterministic) and scatters them into the OIHW gradient through an index map.
#include "conv_gemm.cuh"
#include "elementwise.cuh"
#include "launch.cuh"
#include "ptx.cuh"

#include <string.h>

namespace srg {

int encode_map_bf16(CUtensorMap* map, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box);

struct WgradKParams {
  CUtensorMap x_map;       // input activations (strips)
  CUtensorMap dy_map[4];   // output gradients: one view per n-block
  int N, H, W, TH, TW;
  int tiles_h, tiles_w, tiles_total;
  int n_strips, n_taps, strip_rows, strip_dh;   // n_taps = taps per strip
  int strip_dw[kMaxStrips];
  int tap_row[kMaxTaps];
  int n_pairs;             // ceil(n_strips*n_taps / 2)
  int n_blocks, splits;    // grid = n_blocks * splits
  int dy_c0_step;          // channel offset per n-block inside dy_map (0 when each n-block has its own view)
  uint32_t strip_bytes, stage_bytes;
  int n_stages;
  float* partials;         // [splits][n_blocks][n_pairs][128][64]
  uint64_t pol_in;         // L2 eviction priority of the operand loads (x and dy are dead after the weight gradient)
};

constexpr int kWgThreads = 192;  // warp 0 producer, warp 1 MMA, warps 2-5 epilogue
constexpr uint32_t kDyBytes = 128 * 128;

__global__ void __launch_bounds__(kWgThreads, 1) wgrad_gemm_kernel(const __grid_constant__ WgradKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __builtin_assume(__isShared(smem));
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  pdl_trigger();

  uint8_t* stages = smem;  // n_stages * stage_bytes; stage = [dy tile 16 KB][strip 0][strip 1]...
  uint64_t* bars = reinterpret_cast<uint64_t*>(stages + size_t(p.n_stages) * p.stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + 4;
  uint64_t* done = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int nblk = blockIdx.x % p.n_blocks;
  const int split = blockIdx.x / p.n_blocks;
  const int tiles_per_img = p.tiles_h * p.tiles_w;

  if (warp == 0 && elect_one()) {
    for (int i = 0; i < p.n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
    tma_prefetch_desc(&p.x_map);
    tma_prefetch_desc(&p.dy_map[nblk]);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      pdl_wait();      // x and dy come from the previous kernels
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = split; tile < p.tiles_total; tile += p.splits) {
        const int n = tile / tiles_per_img;
        const int rem = tile - n * tiles_per_img;
        const int h0 = (rem / p.tiles_w) * p.TH;
        const int w0 = (rem % p.tiles_w) * p.TW;
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* dst = stages + size_t(stage) * p.stage_bytes;
        mbar_expect_tx(&full[stage], p.stage_bytes);
        tma_load_4d_hint(dst, &p.dy_map[nblk], &full[stage], nblk * p.dy_c0_step, w0, h0, n, p.pol_in);
        for (int s = 0; s < p.n_strips; ++s)
          tma_load_4d_hint(dst + kDyBytes + size_t(s) * p.strip_bytes, &p.x_map, &full[stage], 0, w0 + p.strip_dw[s],
                      h0 + p.strip_dh, n, p.pol_in);
        if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(128, 64, 1, 1);  // both operands MN-major
    const uint64_t hi_common = (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    const int total_taps = p.n_strips * p.n_taps;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t accumulate = 0;
    for (int tile = split; tile < p.tiles_total; tile += p.splits) {
      mbar_wait(&full[stage], phase);
      tc_fence_after();
      const uint32_t base = smem_u32(stages + size_t(stage) * p.stage_bytes);
      const uint32_t b_lo = base >> 4;
      if (elect_one()) {
        for (int pr = 0; pr < p.n_pairs; ++pr) {
          const int t0 = 2 * pr, t1 = (2 * pr + 1 < total_taps) ? 2 * pr + 1 : 2 * pr;
          const uint32_t a0 = base + kDyBytes + uint32_t(t0 / p.n_taps) * p.strip_bytes +
                              uint32_t(p.tap_row[t0 % p.n_taps] * p.TW) * 128u;
          const uint32_t a1 = base + kDyBytes + uint32_t(t1 / p.n_taps) * p.strip_bytes +
                              uint32_t(p.tap_row[t1 % p.n_taps] * p.TW) * 128u;
          const uint32_t lbo = (t1 == t0) ? 1024u : (a1 - a0);   // unpaired last tap: second half is junk
          const uint64_t adesc = hi_common | (uint64_t((lbo >> 4) & 0x3FFF) << 16) | uint64_t(a0 >> 4);
          const uint64_t bdesc = hi_common | uint64_t(b_lo);
          const uint32_t d_tmem = tmem_base + uint32_t(pr * 64);
#pragma unroll
          for (int k = 0; k < 8; ++k)   // 16 pixels (= 2048 bytes of rows) per MMA
            umma_bf16(d_tmem, adesc + uint64_t(128 * k), bdesc + uint64_t(128 * k), idesc, (k > 0) ? 1u : accumulate);
        }
        umma_commit(&empty[stage]);
      }
      __syncwarp();
      accumulate = 1;
      if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  } else {
    // epilogue: once per CTA
    const int q = warp & 3;
    const int m = q * 32 + lane;
    pdl_wait();        // the split-K partial buffer is still being read by the previous layer's reduce kernel
    mbar_wait(done, 0);
    tc_fence_after();
    const bool any = split < p.tiles_total;
    float* dst = p.partials + ((size_t(split) * p.n_blocks + nblk) * p.n_pairs) * 128 * 64;
    for (int pr = 0; pr < p.n_pairs; ++pr) {
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t v[32];
        tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(pr * 64 + half * 32), v);
        tmem_ld_wait();
        float4* o = reinterpret_cast<float4*>(dst + (size_t(pr) * 128 + m) * 64 + half * 32);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          float4 f;
          f.x = any ? __uint_as_float(v[4 * g + 0]) : 0.f;
          f.y = any ? __uint_as_float(v[4 * g + 1]) : 0.f;
          f.z = any ? __uint_as_float(v[4 * g + 2]) : 0.f;
          f.w = any ? __uint_as_float(v[4 * g + 3]) : 0.f;
          o[g] = f;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// out[e] = sum_s partials[s][idx[e]]  (idx < 0 -> 0).  Fixed summation order => run-to-run deterministic.
__global__ void wgrad_reduce_kernel(const float* __restrict__ partials, const int* __restrict__ idx,
                                    float* __restrict__ out, int n_out, int splits, size_t split_stride,
                                    int accumulate_into) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_out) return;
  const int j = idx[e];
  float acc = 0.f;
  if (j >= 0) {
    const float* p = partials + j;
    for (int s = 0; s < splits; ++s) acc += p[size_t(s) * split_stride];
  }
  out[e] = accumulate_into ? out[e] + acc : acc;
}

// Same reduction driven from the PARTIAL side: thread = 4 consecutive partial elements (coalesced 16-byte loads), 8 warps
// of a block split the `splits` dimension, fixed-order combine, scatter through the inverse map (inv[j] = output element
// or -1).  Output elements no partial maps to are left untouched (the caller zero-fills the gradient buffer).
__global__ void __launch_bounds__(256) wgrad_reduce_inv_kernel(const float4* __restrict__ partials, const int* __restrict__ inv,
                                                               float* __restrict__ out, int n_part4, int splits,
                                                               size_t split_stride4) {
  __shared__ float4 sh[8][32];
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31, sg = threadIdx.x >> 5;
  const int j4 = blockIdx.x * 32 + lane;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (j4 < n_part4) {
    const float4* p = partials + j4;
#pragma unroll 4
    for (int s = sg; s < splits; s += 8) {
      const float4 v = __ldcs(p + size_t(s) * split_stride4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  sh[sg][lane] = acc;
  __syncthreads();
  if (sg == 0 && j4 < n_part4) {
    float4 t = sh[0][lane];
#pragma unroll
    for (int g = 1; g < 8; ++g) { t.x += sh[g][lane].x; t.y += sh[g][lane].y; t.z += sh[g][lane].z; t.w += sh[g][lane].w; }
    const int4 o = *reinterpret_cast<const int4*>(inv + 4 * j4);
    if (o.x >= 0) out[o.x] = t.x;
    if (o.y >= 0) out[o.y] = t.y;
    if (o.z >= 0) out[o.z] = t.z;
    if (o.w >= 0) out[o.w] = t.w;
  }
}
int launch_wgrad_reduce_inv(const float* partials, const int* inv, float* out, int n_part, int splits, size_t split_stride,
                            cudaStream_t stream) {
  if (n_part <= 0 || (n_part & 3) || (split_stride & 3)) { set_error("wgrad_reduce_inv: sizes must be multiples of 4"); return -1; }
  const int n4 = n_part / 4;
  cudaError_t e = launch_pdl(wgrad_reduce_inv_kernel, dim3((n4 + 31) / 32), dim3(256), 0, stream,
                             reinterpret_cast<const float4*>(partials), inv, out, n4, splits, split_stride / 4);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("wgrad_reduce_inv launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

int wgrad_partials_floats(const WgradArgs& a, int* splits_out);

// =====================================================================================================================
// 3x3 weight gradient with taps fused along BOTH GEMM dimensions (one MMA covers 6 of the 9 taps).
//
//   D_t[ci][co] = sum_{h', w} x[h'][w + kw - 1][ci] * dy[h' - kh + 1][w][co]            t = (kh, kw)
//
// The column shift kw selects one of three un-haloed 16-row x strips (A operand, MN-major); the row shift kh selects a
// window of ONE vertically haloed 18-row dy strip (B operand, MN-major).  Because the leading-dimension byte offset of an
// MN-major descriptor is free, M = 128 stacks two x strips (LBO = strip size) and N = 192 stacks the three dy windows
// (LBO = one image row): chain 1 = [kw0; kw1] x [kh2 | kh1 | kh0], chain 2 = [kw1; kw2] x same (its first half repeats
// kw1 and is dropped).  Per 16 pixels that is 2 MMAs of 96 cycles instead of 5 of 69 (tools/mma_probe.cu: an M128 x K16
// MMA costs max(~64, N/2) cycles), and one dy tile + three x tiles per 128 pixels instead of one dy + three haloed x.
// Partials: [split][n-block][kw 3][(2 - kh) * 64 + co][ci 64] fp32 (ci fastest: the lanes of a warp store contiguously).
// =====================================================================================================================
constexpr int kW3Elems = 3 * 192 * 64;          // one partial set: [kw 3][(2-kh)*64 + co 192][ci 64] fp32 (147 KB)
constexpr uint32_t kW3DyBytes = 18 * 8 * 128;   // 18 KB haloed dy strip
constexpr uint32_t kW3XBytes = 16 * 8 * 128;    // 16 KB x strip
constexpr uint32_t kW3Stage = kW3DyBytes + 3 * kW3XBytes;

__global__ void __launch_bounds__(kWgThreads, 1) wgrad3_kernel(const __grid_constant__ WgradKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __builtin_assume(__isShared(smem));
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  pdl_trigger();
  uint8_t* stages = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stages + size_t(p.n_stages) * kW3Stage);
  uint64_t* full = bars;
  uint64_t* empty = bars + 4;
  uint64_t* done = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  const int nblk = blockIdx.x % p.n_blocks;
  const int split = blockIdx.x / p.n_blocks;
  const int tiles_per_img = p.tiles_h * p.tiles_w;

  if (warp == 0 && elect_one()) {
    for (int i = 0; i < p.n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
    tma_prefetch_desc(&p.x_map);
    tma_prefetch_desc(&p.dy_map[nblk]);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      pdl_wait();
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = split; tile < p.tiles_total; tile += p.splits) {
        const int n = tile / tiles_per_img;
        const int rem = tile - n * tiles_per_img;
        const int h0 = (rem / p.tiles_w) * 16;
        const int w0 = (rem % p.tiles_w) * 8;
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* dst = stages + size_t(stage) * kW3Stage;
        mbar_expect_tx(&full[stage], kW3Stage);
        tma_load_4d_hint(dst, &p.dy_map[nblk], &full[stage], nblk * p.dy_c0_step, w0, h0 - 1, n, p.pol_in);
        for (int kw = 0; kw < 3; ++kw)
          tma_load_4d_hint(dst + kW3DyBytes + size_t(kw) * kW3XBytes, &p.x_map, &full[stage], 0, w0 + kw - 1, h0, n, p.pol_in);
        if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(128, 192, 1, 1);
    const uint64_t hi_common = (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    const uint64_t a_hi = hi_common | (uint64_t((kW3XBytes >> 4) & 0x3FFF) << 16);   // M atoms: two x strips
    const uint64_t b_hi = hi_common | (uint64_t((1024 >> 4) & 0x3FFF) << 16);        // N atoms: dy windows one row apart
    int stage = 0;
    uint32_t phase = 0;
    uint32_t accumulate = 0;
    for (int tile = split; tile < p.tiles_total; tile += p.splits) {
      mbar_wait(&full[stage], phase);
      tc_fence_after();
      const uint32_t base = smem_u32(stages + size_t(stage) * kW3Stage);
      if (elect_one()) {
        const uint64_t bdesc = b_hi | uint64_t(base >> 4);
        const uint64_t a1 = a_hi | uint64_t((base + kW3DyBytes) >> 4);               // [kw0; kw1]
        const uint64_t a2 = a_hi | uint64_t((base + kW3DyBytes + kW3XBytes) >> 4);   // [kw1; kw2]
#pragma unroll
        for (int k = 0; k < 8; ++k) {   // 16 pixels (2 image rows = 2048 bytes) per MMA
          umma_bf16(tmem_base, a1 + uint64_t(128 * k), bdesc + uint64_t(128 * k), idesc, (k > 0) ? 1u : accumulate);
          umma_bf16(tmem_base + 192, a2 + uint64_t(128 * k), bdesc + uint64_t(128 * k), idesc, (k > 0) ? 1u : accumulate);
        }
        umma_commit(&empty[stage]);
      }
      __syncwarp();
      accumulate = 1;
      if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  } else {
    // epilogue, once per CTA: lanes 0-63 of chain 1 = kw0, lanes 64-127 of chain 1 = kw1, lanes 64-127 of chain 2 = kw2
    const int q = warp & 3;
    const int m = q * 32 + lane;
    pdl_wait();
    mbar_wait(done, 0);
    tc_fence_after();
    float* dst = p.partials + (size_t(split) * p.n_blocks + nblk) * (3 * 64 * 192);
    for (int chain = 0; chain < 2; ++chain) {
      if (chain == 1 && q < 2) continue;
      const int kw = chain == 0 ? (m >> 6) : 2;
      float* col0 = dst + size_t(kw) * 192 * 64 + (m & 63);
#pragma unroll 1
      for (int c0 = 0; c0 < 192; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(chain * 192 + c0), v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) col0[size_t(c0 + j) * 64] = __uint_as_float(v[j]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

int wgrad3x3_partials_floats(const WgradArgs& a, int* splits_out) {
  int splits = 0;
  wgrad_partials_floats(a, &splits);      // same split policy: SMs / n_blocks, capped by the tile count
  if (splits_out) *splits_out = splits;
  return splits * a.n_blocks * 3 * 64 * 192;
}

int launch_wgrad3x3(const WgradArgs& a, cudaStream_t stream) {
  if (a.TH != 16 || a.TW != 8) { set_error("wgrad3x3: tile must be 16x8"); return -1; }
  if (a.n_blocks < 1 || a.n_blocks > 4) { set_error("wgrad3x3: n_blocks must be 1..4"); return -2; }
  if (a.in_H != a.H || a.in_W != a.W) { set_error("wgrad3x3: stride-1 'same' convolution only"); return -3; }
  WgradKParams p;
  memset(&p, 0, sizeof(p));
  p.N = a.N; p.H = a.H; p.W = a.W; p.TH = 16; p.TW = 8;
  p.tiles_h = (a.H + 15) / 16;
  p.tiles_w = (a.W + 7) / 8;
  p.tiles_total = a.N * p.tiles_h * p.tiles_w;
  if (p.tiles_total == 0) return 0;
  p.n_blocks = a.n_blocks;
  int splits = 0;
  wgrad3x3_partials_floats(a, &splits);
  p.splits = splits;
  p.n_stages = 3;
  p.partials = a.partials;
  p.pol_in = kL2EvictNormal;
  p.dy_c0_step = a.dy_views == 1 ? 64 : 0;
  {
    uint64_t dims[4] = {64, uint64_t(a.in_W), uint64_t(a.in_H), uint64_t(a.N)};
    uint64_t strides[3] = {uint64_t(a.x.stride_w) * 2, uint64_t(a.x.stride_h) * 2, uint64_t(a.x.stride_n) * 2};
    uint32_t box[4] = {64, 8, 16, 1};
    int rc = encode_map_bf16(&p.x_map, a.x.ptr, 4, dims, strides, box);
    if (rc) return rc;
  }
  for (int v = 0; v < 4; ++v) {
    const InView& dv = a.dy[v < a.dy_views ? v : 0];
    uint64_t dims[4] = {uint64_t(dv.channels), uint64_t(a.W), uint64_t(a.H), uint64_t(a.N)};
    uint64_t strides[3] = {uint64_t(dv.stride_w) * 2, uint64_t(dv.stride_h) * 2, uint64_t(dv.stride_n) * 2};
    uint32_t box[4] = {64, 8, 18, 1};
    int rc = encode_map_bf16(&p.dy_map[v], dv.ptr, 4, dims, strides, box);
    if (rc) return rc;
  }
  static DeviceOnce attr;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(wgrad3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return int(e); }
    attr = true;
  }
  const size_t smem_bytes = 1024 + size_t(p.n_stages) * kW3Stage + 256;
  cudaError_t e = launch_pdl(wgrad3_kernel, dim3(p.n_blocks * p.splits), dim3(kWgThreads), smem_bytes, stream, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("wgrad3x3 launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}


// =====================================================================================================================
// Batched 3x3 weight gradients: ALL same-shape layers (the generator trunk: 2 x 16 residual convs + conv2) in ONE launch.
//
// A trunk layer at training sizes is ~10 GFLOP: launched alone it needs all 148 SMs as split-K workers, i.e. 148 partial
// sets of 147 KB per layer (21.8 MB written and re-read by a reduce kernel) plus a launch ramp / TMEM drain / tail per
// layer that is as long as the MMA work itself.  Nothing consumes a weight gradient before the optimizer step, so the
// engine keeps every layer's output gradient (uniformly strided slots) and runs this kernel once at the end of the
// backward pass: the flattened (layer, pixel tile) space is cut into one contiguous range per CTA, a CTA drains its
// TMEM accumulators only when its range crosses a layer boundary, and a layer receives <= ceil(T/R)+1 partial sets
// (6 at cfg2 instead of 148).  Inputs and output gradients are addressed through two 5-D tensor maps whose last
// dimension is the layer.
// Partials: [layer][slot][kw 3][(2 - kh) * 64 + co][ci 64] fp32, slot = CTA - first CTA that touches the layer.
// =====================================================================================================================
struct WgradBatchKParams {
  CUtensorMap x_map;       // {64, W, H, N, layers}
  CUtensorMap dy_map;      // {64, W, H, N, layers}
  int tiles_h, tiles_w, tiles_per_img, tiles_per_layer;
  int n_layers, total_tiles, per_cta, max_slots;
  int n_stages;
  float* partials;
  uint64_t pol_in;
};

__device__ __forceinline__ void tma_load_5d_hint(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3,
                                                 int c4, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2], %8;" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3,
                                            int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

__global__ void __launch_bounds__(kWgThreads, 1) wgrad3_batched_kernel(const __grid_constant__ WgradBatchKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __builtin_assume(__isShared(smem));
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  pdl_trigger();
  uint8_t* stages = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stages + size_t(p.n_stages) * kW3Stage);
  uint64_t* full = bars;
  uint64_t* empty = bars + 4;
  uint64_t* done = bars + 8;       // MMA -> epilogue: the accumulators of one layer segment are complete
  uint64_t* drained = bars + 9;    // epilogue -> MMA: TMEM may be overwritten
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);
  const int begin = blockIdx.x * p.per_cta;
  const int end = min(begin + p.per_cta, p.total_tiles);

  if (warp == 0 && elect_one()) {
    for (int i = 0; i < p.n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(done, 1);
    mbar_init(drained, 128);
    fence_barrier_init();
    tma_prefetch_desc(&p.x_map);
    tma_prefetch_desc(&p.dy_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      pdl_wait();
      int stage = 0;
      uint32_t phase = 0;
      for (int flat = begin; flat < end; ++flat) {
        const int layer = flat / p.tiles_per_layer;
        const int tile = flat - layer * p.tiles_per_layer;
        const int n = tile / p.tiles_per_img;
        const int rem = tile - n * p.tiles_per_img;
        const int h0 = (rem / p.tiles_w) * 16;
        const int w0 = (rem % p.tiles_w) * 8;
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* dst = stages + size_t(stage) * kW3Stage;
        mbar_expect_tx(&full[stage], kW3Stage);
        tma_load_5d_hint(dst, &p.dy_map, &full[stage], 0, w0, h0 - 1, n, layer, p.pol_in);
        for (int kw = 0; kw < 3; ++kw)
          tma_load_5d_hint(dst + kW3DyBytes + size_t(kw) * kW3XBytes, &p.x_map, &full[stage], 0, w0 + kw - 1, h0, n, layer, p.pol_in);
        if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(128, 192, 1, 1);
    const uint64_t hi_common = (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    const uint64_t a_hi = hi_common | (uint64_t((kW3XBytes >> 4) & 0x3FFF) << 16);   // M atoms: two x strips
    const uint64_t b_hi = hi_common | (uint64_t((1024 >> 4) & 0x3FFF) << 16);        // N atoms: dy windows one row apart
    int stage = 0;
    uint32_t phase = 0, drained_phase = 0;
    uint32_t accumulate = 0;
    int cur_layer = begin / p.tiles_per_layer;
    for (int flat = begin; flat < end; ++flat) {
      const int layer = flat / p.tiles_per_layer;
      if (layer != cur_layer) {
        // layer boundary inside this CTA's range: hand the finished accumulators to the epilogue, wait for the drain
        if (elect_one()) umma_commit(done);
        __syncwarp();
        mbar_wait(drained, drained_phase);
        drained_phase ^= 1;
        tc_fence_after();
        accumulate = 0;
        cur_layer = layer;
      }
      mbar_wait(&full[stage], phase);
      tc_fence_after();
      const uint32_t base = smem_u32(stages + size_t(stage) * kW3Stage);
      if (elect_one()) {
        const uint64_t bdesc = b_hi | uint64_t(base >> 4);
        const uint64_t a1 = a_hi | uint64_t((base + kW3DyBytes) >> 4);               // [kw0; kw1]
        const uint64_t a2 = a_hi | uint64_t((base + kW3DyBytes + kW3XBytes) >> 4);   // [kw1; kw2]
#pragma unroll
        for (int k = 0; k < 8; ++k) {   // 16 pixels (2 image rows = 2048 bytes) per MMA
          umma_bf16(tmem_base, a1 + uint64_t(128 * k), bdesc + uint64_t(128 * k), idesc, (k > 0) ? 1u : accumulate);
          umma_bf16(tmem_base + 192, a2 + uint64_t(128 * k), bdesc + uint64_t(128 * k), idesc, (k > 0) ? 1u : accumulate);
        }
        umma_commit(&empty[stage]);
      }
      __syncwarp();
      accumulate = 1;
      if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  } else {
    // epilogue: one drain per layer segment of this CTA's range
    const int q = warp & 3;
    const int m = q * 32 + lane;
    pdl_wait();
    uint32_t done_phase = 0;
    const int first_layer = begin / p.tiles_per_layer;
    const int last_layer = (end - 1) / p.tiles_per_layer;
    for (int layer = first_layer; layer <= last_layer; ++layer) {
      mbar_wait(done, done_phase);
      done_phase ^= 1;
      tc_fence_after();
      const int slot = int(blockIdx.x) - (layer * p.tiles_per_layer) / p.per_cta;
      float* dst = p.partials + (size_t(layer) * p.max_slots + slot) * kW3Elems;
      for (int chain = 0; chain < 2; ++chain) {
        if (chain == 1 && q < 2) continue;
        const int kw = chain == 0 ? (m >> 6) : 2;
        float* col0 = dst + size_t(kw) * 192 * 64 + (m & 63);
#pragma unroll 1
        for (int c0 = 0; c0 < 192; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(chain * 192 + c0), v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) col0[size_t(c0 + j) * 64] = __uint_as_float(v[j]);
        }
      }
      tc_fence_before();
      mbar_arrive(drained);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// out[layer] element inv[j] = sum over the layer's slots of partial element j (fixed order => deterministic)
__global__ void __launch_bounds__(256) wgrad_reduce_batched_kernel(const float4* __restrict__ partials, const int* __restrict__ inv,
                                                                   float* __restrict__ grads, const long long* __restrict__ out_off,
                                                                   int n_part4, int tiles_per_layer, int per_cta, int max_slots) {
  pdl_trigger();
  pdl_wait();
  const int layer = blockIdx.y;
  const int j4 = blockIdx.x * blockDim.x + threadIdx.x;
  if (j4 >= n_part4) return;
  const int c_first = (layer * tiles_per_layer) / per_cta;
  const int c_last = ((layer + 1) * tiles_per_layer - 1) / per_cta;
  const float4* p = partials + size_t(layer) * max_slots * n_part4 + j4;
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s <= c_last - c_first; ++s) {
    const float4 v = __ldcs(p + size_t(s) * n_part4);
    t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
  }
  float* out = grads + out_off[layer];
  const int4 o = *reinterpret_cast<const int4*>(inv + 4 * j4);
  if (o.x >= 0) out[o.x] = t.x;
  if (o.y >= 0) out[o.y] = t.y;
  if (o.z >= 0) out[o.z] = t.z;
  if (o.w >= 0) out[o.w] = t.w;
}

void wgrad3_batched_plan(const WgradBatchArgs& a, int* tiles_per_layer, int* grid, int* per_cta, int* max_slots) {
  const int sms = sm_budget();
  const int T = a.N * ((a.H + 15) / 16) * ((a.W + 7) / 8);
  const long long total = (long long)T * a.n_layers;
  int per = int((total + sms - 1) / sms);
  if (per < 1) per = 1;
  const int g = int((total + per - 1) / per);
  *tiles_per_layer = T; *grid = g; *per_cta = per;
  *max_slots = (T + per - 1) / per + 1;
}

size_t wgrad3_batched_partials_floats(const WgradBatchArgs& a) {
  int T, g, per, ms;
  wgrad3_batched_plan(a, &T, &g, &per, &ms);
  return size_t(a.n_layers) * ms * kW3Elems;
}

int launch_wgrad3x3_batched(const WgradBatchArgs& a, cudaStream_t stream) {
  if (a.n_layers < 1 || a.N < 1 || a.H < 1 || a.W < 1) { set_error("wgrad3x3_batched: bad geometry"); return -1; }
  WgradBatchKParams p;
  memset(&p, 0, sizeof(p));
  int T, grid, per, ms;
  wgrad3_batched_plan(a, &T, &grid, &per, &ms);
  p.tiles_h = (a.H + 15) / 16;
  p.tiles_w = (a.W + 7) / 8;
  p.tiles_per_img = p.tiles_h * p.tiles_w;
  p.tiles_per_layer = T;
  p.n_layers = a.n_layers;
  p.total_tiles = T * a.n_layers;
  p.per_cta = per;
  p.max_slots = ms;
  p.n_stages = 3;
  p.partials = a.partials;
  p.pol_in = kL2EvictNormal;
  {
    uint64_t dims[5] = {64, uint64_t(a.W), uint64_t(a.H), uint64_t(a.N), uint64_t(a.n_layers)};
    uint64_t xs[4] = {128, uint64_t(a.W) * 128, uint64_t(a.H) * a.W * 128, uint64_t(a.x_layer_stride_bytes)};
    uint32_t xbox[5] = {64, 8, 16, 1, 1};
    int rc = encode_map_bf16(&p.x_map, a.x_base, 5, dims, xs, xbox);
    if (rc) return rc;
    uint64_t ds[4] = {128, uint64_t(a.W) * 128, uint64_t(a.H) * a.W * 128, uint64_t(a.dy_layer_stride_bytes)};
    uint32_t dbox[5] = {64, 8, 18, 1, 1};
    rc = encode_map_bf16(&p.dy_map, a.dy_base, 5, dims, ds, dbox);
    if (rc) return rc;
  }
  static DeviceOnce attr;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(wgrad3_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return int(e); }
    attr = true;
  }
  const size_t smem_bytes = 1024 + size_t(p.n_stages) * kW3Stage + 256;
  cudaError_t e = launch_pdl(wgrad3_batched_kernel, dim3(grid), dim3(kWgThreads), smem_bytes, stream, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("wgrad3x3_batched launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  // reduce: [layer][slot] partial sets -> OIHW gradients through the inverse index map shared by all layers
  const int n4 = kW3Elems / 4;
  e = launch_pdl(wgrad_reduce_batched_kernel, dim3((n4 + 255) / 256, a.n_layers), dim3(256), 0, stream,
                 reinterpret_cast<const float4*>(a.partials), a.inv, a.grads, a.out_off, n4, T, per, ms);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("wgrad_reduce_batched launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

int wgrad_partials_floats(const WgradArgs& a, int* splits_out) {
  const int sms = sm_budget();
  const int tiles = a.N * ((a.H + a.TH - 1) / a.TH) * ((a.W + a.TW - 1) / a.TW);
  int splits = sms / a.n_blocks;
  if (splits < 1) splits = 1;
  if (splits > tiles) splits = tiles;
  if (splits_out) *splits_out = splits;
  const int n_pairs = (a.n_strips * a.n_taps + 1) / 2;
  return splits * a.n_blocks * n_pairs * 128 * 64;
}

int launch_wgrad_gemm(const WgradArgs& a, cudaStream_t stream) {
  if (a.TH * a.TW != 128 || a.TW % 8 != 0) { set_error("wgrad: tile must be 128 pixels with TW%%8==0"); return -1; }
  if (a.n_blocks < 1 || a.n_blocks > 4) { set_error("wgrad: n_blocks must be 1..4"); return -2; }
  const int total_taps = a.n_strips * a.n_taps;
  if (total_taps < 1 || a.n_strips > kMaxStrips || a.n_taps > kMaxTaps) { set_error("wgrad: bad tap count"); return -3; }
  WgradKParams p;
  memset(&p, 0, sizeof(p));
  p.N = a.N; p.H = a.H; p.W = a.W; p.TH = a.TH; p.TW = a.TW;
  p.tiles_h = (a.H + a.TH - 1) / a.TH;
  p.tiles_w = (a.W + a.TW - 1) / a.TW;
  p.tiles_total = a.N * p.tiles_h * p.tiles_w;
  if (p.tiles_total == 0) return 0;
  p.n_strips = a.n_strips; p.n_taps = a.n_taps; p.strip_rows = a.strip_rows; p.strip_dh = a.strip_dh;
  for (int s = 0; s < a.n_strips; ++s) p.strip_dw[s] = a.strip_dw[s];
  for (int r = 0; r < a.n_taps; ++r) {
    if (a.tap_row[r] < 0 || a.tap_row[r] + a.TH > a.strip_rows) { set_error("wgrad: tap row outside strip"); return -4; }
    p.tap_row[r] = a.tap_row[r];
  }
  p.n_pairs = (total_taps + 1) / 2;
  if (p.n_pairs * 64 > 512) { set_error("wgrad: too many taps for TMEM"); return -5; }
  p.n_blocks = a.n_blocks;
  int splits = 0;
  wgrad_partials_floats(a, &splits);
  p.splits = splits;
  p.strip_bytes = uint32_t(a.strip_rows) * a.TW * 128u;
  p.stage_bytes = kDyBytes + uint32_t(a.n_strips) * p.strip_bytes;
  int stages = int((227u * 1024u - 2048u) / p.stage_bytes);
  if (stages > 4) stages = 4;
  if (stages < 1) { set_error("wgrad: stage does not fit in shared memory (%u B)", p.stage_bytes); return -6; }
  p.n_stages = stages;
  p.partials = a.partials;
  p.pol_in = kL2EvictNormal;
  p.dy_c0_step = a.dy_views == 1 ? 64 : 0;

  {
    uint64_t dims[4] = {64, uint64_t(a.in_W), uint64_t(a.in_H), uint64_t(a.N)};
    uint64_t strides[3] = {uint64_t(a.x.stride_w) * 2, uint64_t(a.x.stride_h) * 2, uint64_t(a.x.stride_n) * 2};
    uint32_t box[4] = {64, uint32_t(a.TW), uint32_t(a.strip_rows), 1};
    int rc = encode_map_bf16(&p.x_map, a.x.ptr, 4, dims, strides, box);
    if (rc) return rc;
  }
  for (int v = 0; v < 4; ++v) {
    const InView& dv = a.dy[v < a.dy_views ? v : 0];
    uint64_t dims[4] = {uint64_t(dv.channels), uint64_t(a.W), uint64_t(a.H), uint64_t(a.N)};
    uint64_t strides[3] = {uint64_t(dv.stride_w) * 2, uint64_t(dv.stride_h) * 2, uint64_t(dv.stride_n) * 2};
    uint32_t box[4] = {64, uint32_t(a.TW), uint32_t(a.TH), 1};
    int rc = encode_map_bf16(&p.dy_map[v], dv.ptr, 4, dims, strides, box);
    if (rc) return rc;
  }
  static DeviceOnce attr;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return int(e); }
    attr = true;
  }
  const size_t smem_bytes = 1024 + size_t(stages) * p.stage_bytes + 256;
  cudaError_t e = launch_pdl(wgrad_gemm_kernel, dim3(p.n_blocks * p.splits), dim3(kWgThreads), smem_bytes, stream, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("wgrad launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

int launch_wgrad_reduce(const float* partials, const int* idx, float* out, int n_out, int splits, size_t split_stride,
                        int accumulate_into, cudaStream_t stream) {
  if (n_out <= 0) return 0;
  wgrad_reduce_kernel<<<(n_out + 255) / 256, 256, 0, stream>>>(partials, idx, out, n_out, splits, split_stride,
                                                              accumulate_into);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("wgrad_reduce launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

}  // namespace srg
