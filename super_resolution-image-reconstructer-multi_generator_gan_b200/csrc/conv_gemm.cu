// Strip implicit-GEMM convolution for sm_100a: TMA -> shared (128B swizzle) -> tcgen05.mma -> TMEM -> epilogue.
//
// GEMM view: M = 128 output pixels (a TH x TW tile), N = 64 (or 32) output channels, K = 64 input channels per
// (strip, tap) k-block.  For every column shift s ("strip") the producer loads ONE box of (TH + span) input rows
// x TW pixels x 64 channels; the taps that share that column shift read it at different row offsets, so each
// input element crosses L2->SM  n_strips times instead of n_strips*n_taps times.  Because TW % 8 == 0 every tap's
// A operand starts on a 1024-byte swizzle-atom boundary: canonical K-major SWIZZLE_128B descriptors throughout.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-9 = epilogue.
// Persistent CTAs; two TMEM accumulator stages so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// Three kernels live in this file, all behind launch_conv_gemm():
//   conv_gemm_kernel<BLOCK_N, NT>  the generic strip kernel described above (one N = 64 / 32 MMA per tap and K-step);
//   conv3_il_kernel                plain 3x3 / 64-input-channel launches: row-interleaved accumulator blocks so that two
//                                  taps share one N = 128 MMA (the ~64-cycle floor of an M128 MMA makes that free);
//   conv9_rows_kernel              the 9x9 / 3-output-channel conv3: one image row per MMA feeding up to 8 output rows.
#include "conv_gemm.cuh"
#include "elementwise.cuh"
#include "launch.cuh"
#include "ptx.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>

namespace srg {

// ------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
const char* last_error() { return g_err; }
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static long long g_launch_total = 0;
void count_launch(int n) { __atomic_fetch_add(&g_launch_total, (long long)n, __ATOMIC_RELAXED); }
long long total_launches() { return __atomic_load_n(&g_launch_total, __ATOMIC_RELAXED); }

// ------------------------------------------------------- device parameters
struct ConvKParams {
  CUtensorMap in_map[kMaxInMaps];
  CUtensorMap w_map;
  CUtensorMap out_map[4];  // NHWC: [0]; pixel shuffle: one strided view of the HR tensor per n-block
  CUtensorMap aux_map;     // residual / mask tensor (same geometry as out_map[0])
  uint64_t pol_in;         // L2 eviction priority of the operand / aux loads
  int N, H, W, TH, TW;
  int tiles_h, tiles_w, tiles_total;
  int tile_step_w;  // TW, or TW-8 for the fold9 epilogue
  int tile_w_org;   // 0, or -4 for fold9
  int n_chunks, chunks_per_view;
  int n_strips, strip_rows, strip_dh;
  int strip_dw[kMaxStrips];
  int tap_row[kMaxTaps];
  int cout_total, n_blocks, ctas_per_block;
  int resident, n_stages;
  uint32_t strip_bytes, stage_bytes, w_resident_bytes;
  const float* bias;
  const float* scale;  // optional per-channel multiplier of the accumulator (folded eval-mode BatchNorm)
  int act;
  float slope;
  int aux_mode;  // 0 none, 1 add (residual), 2 mask (zero where aux <= 0)
  void* out;     // fold9 only (through the FoldScatter of ConvKParamsFold)
  int out_mode;
  float* stats;  // per-CTA channel sums / sums of squares (BatchNorm statistics fused into the epilogue)
  long long* prof;  // optional per-CTA role timers (debug)
};

// the fold9 instance also carries its store table (the other instances keep their parameter size)
struct ConvKParamsFold : ConvKParams {
  FoldScatter scatter;
};
template <int BLOCK_N> struct KParamsOf { using type = ConvKParams; };
template <> struct KParamsOf<32> { using type = ConvKParamsFold; };

constexpr int kThreads = 320;       // warp 0 producer, warp 1 MMA, warps 2..9 epilogue
constexpr int kEpiThreads = 256;
constexpr int kFoldPad = 33;
constexpr uint32_t kTileOutBytes = 128 * 128;  // 128 pixels x 64 bf16

template <int ACT>
__device__ __forceinline__ float apply_act(float x, float slope) {
  if (ACT == ACT_RELU) return fmaxf(x, 0.f);
  if (ACT == ACT_LRELU) return x > 0.f ? x : x * slope;
  return x;
}

// one output pixel of a fold9 epilogue through its FoldScatter.  The 8-bit store is torch's
// (sr.clamp(0, 1) * 255).round().to(uint8): fp32 multiply, round half to even; NaN stores 0 (fmaxf returns 0)
__device__ __forceinline__ uint8_t quantise_u8(float y) {
  return uint8_t(rintf(__fmul_rn(fminf(fmaxf(y, 0.f), 1.f), 255.f)));
}
__device__ __forceinline__ void fold9_store(const FoldScatter& s, void* out, int n, int h, int w, float o0, float o1,
                                            float o2) {
  const int64_t base = (s.n == 0 ? int64_t(n) * s.item : s.t[n].base) + int64_t(h) * s.pitch + int64_t(w) * s.px;
  if (s.u8) {
    uint8_t* o = reinterpret_cast<uint8_t*>(out) + base;
    o[0] = quantise_u8(o0);
    o[s.plane] = quantise_u8(o1);
    o[2 * s.plane] = quantise_u8(o2);
  } else {
    float* o = reinterpret_cast<float*>(out) + base;
    o[0] = o0;
    o[s.plane] = o1;
    o[2 * s.plane] = o2;
  }
}
// the plain fp32 NCHW store of an H x W launch that brings no FoldScatter
static FoldScatter fold9_nchw(int H, int W) {
  FoldScatter s;
  memset(&s, 0, sizeof(s));
  s.plane = int64_t(H) * W;
  s.item = 3 * s.plane;
  s.pitch = W;
  s.px = 1;
  return s;
}

template <int BLOCK_N, int NT>
__global__ void __launch_bounds__(kThreads, 1) conv_gemm_kernel(const __grid_constant__ typename KParamsOf<BLOCK_N>::type p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __builtin_assume(__isShared(smem));

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  constexpr bool kFold = (BLOCK_N == 32);
  pdl_trigger();   // let the next kernel's CTAs take this SM as soon as this CTA leaves it

  uint8_t* w_smem = smem;                                 // resident weights (may be empty)
  uint8_t* stages = smem + p.w_resident_bytes;            // n_stages * stage_bytes
  uint8_t* out_stage = stages + size_t(p.n_stages) * p.stage_bytes;      // 2 x 16 KB (not fold9)
  uint8_t* aux_stage = out_stage + (kFold ? 0 : 2 * kTileOutBytes);      // 2 x 16 KB (aux_mode != 0)
  uint8_t* tail = aux_stage + (p.aux_mode ? 2 * kTileOutBytes : 0);
  float* fold_buf = reinterpret_cast<float*>(tail);       // 128*33 floats (fold9 only)
  uint8_t* tail2 = tail + (kFold ? 128 * kFoldPad * 4 : 0);
  float* s_bias = reinterpret_cast<float*>(tail2);        // BLOCK_N floats bias, then BLOCK_N floats scale (128 + 128 B used of 512)
  float* s_scale = s_bias + 64;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail2 + 512);
  uint64_t* full = bars;                                  // [n_stages]
  uint64_t* empty = bars + 8;                             // [n_stages]
  uint64_t* wfull = bars + 16;
  uint64_t* tfull = bars + 17;                            // [2]
  uint64_t* tempty = bars + 19;                           // [2]
  uint64_t* auxfull = bars + 21;                          // [2]
  uint64_t* auxempty = bars + 23;                         // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 25);
  float* s_stats = reinterpret_cast<float*>(tail2 + 768);  // [8][128] floats (p.stats only)

  const int nblk = blockIdx.x % p.n_blocks;
  const int tile0 = blockIdx.x / p.n_blocks;
  const int tiles_per_img = p.tiles_h * p.tiles_w;
  constexpr uint32_t kBTile = BLOCK_N * 128;              // bytes of one weight k-block
  constexpr uint32_t kTmemCols = 2 * BLOCK_N < 32 ? 32 : 2 * BLOCK_N;
  constexpr int kEpiActive = kFold ? 128 : kEpiThreads;   // epilogue threads that touch TMEM
  const int kb_total = p.n_chunks * p.n_strips * NT;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < p.n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(wfull, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kEpiActive);
      mbar_init(&auxfull[i], 1);
      mbar_init(&auxempty[i], kEpiActive);
    }
    fence_barrier_init();
    for (int v = 0; v < kMaxInMaps; ++v) tma_prefetch_desc(&p.in_map[v]);
    tma_prefetch_desc(&p.w_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  if (warp >= 2) {
    const int t = threadIdx.x - 64;
    if (t < BLOCK_N) {
      float b = 0.f;
      if (p.bias != nullptr && !kFold) b = p.bias[nblk * BLOCK_N + t];
      s_bias[t] = b;
      s_scale[t] = (p.scale != nullptr && !kFold) ? p.scale[nblk * BLOCK_N + t] : 1.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  long long prof_acc[4] = {0, 0, 0, 0};
  const long long t_start = clock64();

  if (warp == 0) {
    // =============================================================== TMA producer
    if (elect_one()) {
      if (p.resident) {
        mbar_expect_tx(wfull, uint32_t(kb_total) * kBTile);
        for (int kb = 0; kb < kb_total; ++kb)
          tma_load_2d(w_smem + size_t(kb) * kBTile, &p.w_map, wfull, 0, kb * p.cout_total + nblk * BLOCK_N);
      }
      pdl_wait();      // the activations (and aux tensor) come from the previous kernel; the weights above do not
      int stage = 0, ab = 0;
      uint32_t phase = 0, aux_phase = 0;
      for (int tile = tile0; tile < p.tiles_total; tile += p.ctas_per_block) {
        const int n = tile / tiles_per_img;
        const int rem = tile - n * tiles_per_img;
        const int h0 = (rem / p.tiles_w) * p.TH;
        const int w0 = (rem % p.tiles_w) * p.tile_step_w + p.tile_w_org;
        if (p.aux_mode) {
          mbar_wait(&auxempty[ab], aux_phase ^ 1);
          mbar_expect_tx(&auxfull[ab], kTileOutBytes);
          tma_load_4d_hint(aux_stage + ab * kTileOutBytes, &p.aux_map, &auxfull[ab], nblk * BLOCK_N, w0, h0, n, p.pol_in);
          ab ^= 1;
          if (ab == 0) aux_phase ^= 1;
        }
        for (int c = 0; c < p.n_chunks; ++c) {
          const int view = c / p.chunks_per_view;
          const int coff = (c - view * p.chunks_per_view) * 64;
          for (int s = 0; s < p.n_strips; ++s) {
            { long long t0_ = clock64(); mbar_wait(&empty[stage], phase ^ 1); prof_acc[0] += clock64() - t0_; }
            uint8_t* dst = stages + size_t(stage) * p.stage_bytes;
            mbar_expect_tx(&full[stage], p.resident ? p.strip_bytes : p.stage_bytes);
            tma_load_4d_hint(dst, &p.in_map[view], &full[stage], coff, w0 + p.strip_dw[s], h0 + p.strip_dh, n, p.pol_in);
            if (!p.resident) {
              const int kb0 = (c * p.n_strips + s) * NT;
              for (int r = 0; r < NT; ++r)
                tma_load_2d(dst + p.strip_bytes + size_t(r) * kBTile, &p.w_map, &full[stage], 0,
                            (kb0 + r) * p.cout_total + nblk * BLOCK_N);
            }
            if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    // The whole warp runs this loop with warp-uniform values; only `leader` issues tcgen05 instructions.
    constexpr uint32_t idesc = make_idesc_bf16(128, BLOCK_N, 0, 0);
    const uint64_t desc_hi = (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    uint32_t tap_off[NT];
#pragma unroll
    for (int r = 0; r < NT; ++r) tap_off[r] = uint32_t(p.tap_row[r] * p.TW) * 8u;  // bytes >> 4
    const uint32_t stage0_lo = smem_u32(stages) >> 4;
    const uint32_t stage_lo_stride = p.stage_bytes >> 4;
    const uint32_t w_lo = smem_u32(w_smem) >> 4;
    const uint32_t strip_lo = p.strip_bytes >> 4;
    if (p.resident) mbar_wait(wfull, 0);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = tile0; tile < p.tiles_total; tile += p.ctas_per_block) {
      { long long t0_ = clock64(); mbar_wait(&tempty[acc], acc_phase ^ 1); prof_acc[1] += clock64() - t0_; }
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + uint32_t(acc * BLOCK_N);
      uint32_t accumulate = 0;
      uint32_t kb = 0;
      for (int c = 0; c < p.n_chunks; ++c) {
        for (int s = 0; s < p.n_strips; ++s) {
          { long long t0_ = clock64(); mbar_wait(&full[stage], phase); prof_acc[2] += clock64() - t0_; }
          tc_fence_after();
          const uint32_t a_lo = stage0_lo + uint32_t(stage) * stage_lo_stride;
          const uint32_t b_lo = p.resident ? w_lo + kb * (kBTile >> 4) : a_lo + strip_lo;
          if (elect_one()) {
#pragma unroll
            for (int r = 0; r < NT; ++r) {
              const uint64_t adesc = desc_hi | uint64_t(a_lo + tap_off[r]);
              const uint64_t bdesc = desc_hi | uint64_t(b_lo + uint32_t(r) * (kBTile >> 4));
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                umma_bf16(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc, accumulate);
                accumulate = 1;
              }
            }
            umma_commit(&empty[stage]);
          }
          __syncwarp();
          accumulate = 1;
          kb += NT;
          if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
        }
      }
      if (elect_one()) umma_commit(&tfull[acc]);
      __syncwarp();
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (!kFold || warp < 6) {
    // =================================================================== epilogue
    const int q = warp & 3;            // TMEM lane quadrant this warp may read
    const int m = q * 32 + lane;       // GEMM row == pixel within the tile
    const int hf = (warp - 2) >> 2;    // which 32-column half of the 64-wide tile (0 for fold9)
    const int etid = threadIdx.x - 64;
    int acc = 0, ob = 0, ab = 0;
    uint32_t acc_phase = 0, aux_phase = 0;
    float st_s0 = 0.f, st_s1 = 0.f, st_q0 = 0.f, st_q1 = 0.f;   // BatchNorm statistics of this thread's channel pair
    for (int tile = tile0; tile < p.tiles_total; tile += p.ctas_per_block) {
      const int n = tile / tiles_per_img;
      const int rem = tile - n * tiles_per_img;
      const int h0 = (rem / p.tiles_w) * p.TH;
      const int w0 = (rem % p.tiles_w) * p.tile_step_w + p.tile_w_org;
      { long long t0_ = clock64(); mbar_wait(&tfull[acc], acc_phase); prof_acc[3] += clock64() - t0_; }
      tc_fence_after();
      const uint32_t t_addr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * BLOCK_N + hf * 32);
      uint32_t v[32];
      tmem_ld32(t_addr, v);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&tempty[acc]);

      if constexpr (kFold) {
        // fold9: P[pixel][s*3+co] -> out[co][h][w] = bias + sum_s P[(h, w+s-4)][s*3+co]
        const int th = m / p.TW;
        const int tw = m - th * p.TW;
        const int h = h0 + th, w = w0 + tw;
#pragma unroll
        for (int j = 0; j < 32; ++j) fold_buf[m * kFoldPad + j] = __uint_as_float(v[j]);
        named_bar_sync(1, 128);
        const bool in_crop = p.scatter.n == 0 || (h >= p.scatter.t[n].h_lo && h < p.scatter.t[n].h_hi &&
                                                  w >= p.scatter.t[n].w_lo && w < p.scatter.t[n].w_hi);
        if (tw >= 4 && tw < p.TW - 4 && h < p.H && w >= 0 && w < p.W && in_crop) {
          float o0 = p.bias ? p.bias[0] : 0.f, o1 = p.bias ? p.bias[1] : 0.f, o2 = p.bias ? p.bias[2] : 0.f;
#pragma unroll
          for (int s = 0; s < 9; ++s) {
            const float* row = fold_buf + (m + s - 4) * kFoldPad + s * 3;
            o0 += row[0];
            o1 += row[1];
            o2 += row[2];
          }
          fold9_store(p.scatter, p.out, n, h, w, o0, o1, o2);
        }
        named_bar_sync(2, 128);
      } else {
        float f[32];
        {
          const float4* bp = reinterpret_cast<const float4*>(s_bias + hf * 32);
          const float4* sp4 = reinterpret_cast<const float4*>(s_scale + hf * 32);
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 b = bp[g];
            const float4 sc = sp4[g];
            f[4 * g + 0] = fmaf(__uint_as_float(v[4 * g + 0]), sc.x, b.x);
            f[4 * g + 1] = fmaf(__uint_as_float(v[4 * g + 1]), sc.y, b.y);
            f[4 * g + 2] = fmaf(__uint_as_float(v[4 * g + 2]), sc.z, b.z);
            f[4 * g + 3] = fmaf(__uint_as_float(v[4 * g + 3]), sc.w, b.w);
          }
        }
        if (p.act == ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = apply_act<ACT_RELU>(f[j], 0.f);
        } else if (p.act == ACT_LRELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = apply_act<ACT_LRELU>(f[j], p.slope);
        }
        if (p.out_mode == OUT_NHWC_F32) {
          // fp32 output: every thread owns 32 consecutive channels of one pixel (128 contiguous bytes)
          const int th = m / p.TW;
          const int h = h0 + th, w = w0 + (m - th * p.TW);
          if (h < p.H && w < p.W) {
            float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) +
                                                  ((size_t(n) * p.H + h) * p.W + w) * p.cout_total + nblk * BLOCK_N + hf * 32);
#pragma unroll
            for (int g = 0; g < 8; ++g) o[g] = make_float4(f[4 * g], f[4 * g + 1], f[4 * g + 2], f[4 * g + 3]);
          }
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
          continue;
        }
        const uint32_t row_off = uint32_t(m) * 128u;
        const uint32_t sw = uint32_t(m & 7);
        if (p.aux_mode) {
          mbar_wait(&auxfull[ab], aux_phase);
          const uint8_t* ap = aux_stage + ab * kTileOutBytes + row_off;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const uint4 r = *reinterpret_cast<const uint4*>(ap + (((uint32_t(hf * 4 + g)) ^ sw) << 4));
            const uint32_t ws[4] = {r.x, r.y, r.z, r.w};
            if (p.aux_mode == 1) {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                f[g * 8 + 2 * e] += bf16_lo(ws[e]);
                f[g * 8 + 2 * e + 1] += bf16_hi(ws[e]);
              }
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                if (!(bf16_lo(ws[e]) > 0.f)) f[g * 8 + 2 * e] = 0.f;
                if (!(bf16_hi(ws[e]) > 0.f)) f[g * 8 + 2 * e + 1] = 0.f;
              }
            }
          }
          mbar_arrive(&auxempty[ab]);
          ab ^= 1;
          if (ab == 0) aux_phase ^= 1;
        }
        // stage the bf16 tile in shared memory (128B-swizzled rows) and hand it to the TMA store engine
        if (etid == 0) tma_store_wait_read<1>();      // the store that used this buffer two tiles ago has drained
        named_bar_sync(1, kEpiThreads);
        uint8_t* op = out_stage + ob * kTileOutBytes + row_off;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 o;
          o.x = pack_bf16(f[g * 8 + 0], f[g * 8 + 1]);
          o.y = pack_bf16(f[g * 8 + 2], f[g * 8 + 3]);
          o.z = pack_bf16(f[g * 8 + 4], f[g * 8 + 5]);
          o.w = pack_bf16(f[g * 8 + 6], f[g * 8 + 7]);
          *reinterpret_cast<uint4*>(op + (((uint32_t(hf * 4 + g)) ^ sw) << 4)) = o;
        }
        fence_proxy_async_smem();
        named_bar_sync(2, kEpiThreads);
        if (etid == 0) {
          const bool ps = p.out_mode == OUT_PIXEL_SHUFFLE;
          tma_store_4d(&p.out_map[ps ? nblk : 0], out_stage + ob * kTileOutBytes, ps ? 0 : nblk * BLOCK_N, w0, h0, n);
          tma_store_commit();
        }
        if (p.stats != nullptr) {
          // column sums of the staged bf16 tile (exactly the values BatchNorm will normalise): thread = channel pair
          // c2 x 16-row part; rows outside the image (ragged tiles) are skipped
          const int c2 = etid & 31, part = etid >> 5;
          const uint8_t* sp = out_stage + ob * kTileOutBytes;
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            const int mm = part * 16 + r;
            const int th = mm >> 3;
            if (h0 + th < p.H && w0 + (mm & 7) < p.W) {
              const uint32_t v = *reinterpret_cast<const uint32_t*>(sp + mm * 128 + ((((c2 >> 2)) ^ (mm & 7)) << 4) + (c2 & 3) * 4);
              const float a0 = bf16_lo(v), a1 = bf16_hi(v);
              st_s0 += a0; st_s1 += a1;
              st_q0 = fmaf(a0, a0, st_q0); st_q1 = fmaf(a1, a1, st_q1);
            }
          }
        }
        ob ^= 1;
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (!kFold && etid == 0) tma_store_wait_all<0>();
    if (!kFold && p.stats != nullptr) {
      const int c2 = etid & 31, part = etid >> 5;
      s_stats[part * 128 + 2 * c2] = st_s0;
      s_stats[part * 128 + 2 * c2 + 1] = st_s1;
      s_stats[part * 128 + 64 + 2 * c2] = st_q0;
      s_stats[part * 128 + 64 + 2 * c2 + 1] = st_q1;
      named_bar_sync(3, kEpiThreads);
      if (etid < 128) {
        float t = 0.f;
#pragma unroll
        for (int g = 0; g < 8; ++g) t += s_stats[g * 128 + etid];
        p.stats[size_t(blockIdx.x) * 128 + etid] = t;
      }
    }
  }

  if (p.prof != nullptr && lane == 0 && (warp <= 2)) {
    long long* d = p.prof + (size_t(blockIdx.x) * 3 + warp) * 6;
    d[0] = prof_acc[0]; d[1] = prof_acc[1]; d[2] = prof_acc[2]; d[3] = prof_acc[3]; d[4] = clock64() - t_start; d[5] = t_start;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}


// =====================================================================================================================
// 3x3 stride-1 convolution, 64 input channels, with ROW-INTERLEAVED accumulator blocks ("conv3_il").
//
// Measured on B200 (tools/mma_probe.cu): an SS-mode M128 x K16 tcgen05.mma costs ~69 cycles for N = 64 AND for N = 128
// (a ~64-cycle floor per instruction), so the N = 64 MMAs of the generic kernel run the tensor pipe at 46 %.  Pairing
// two taps in one N = 128 MMA is free -- if both halves of the accumulator are complete outputs, i.e. nothing has to be
// re-aligned in registers afterwards.  This kernel gets there through the A descriptor instead of the epilogue:
//
//   * a tile is 32 image rows x 8 pixels; TMEM block E (64 columns) holds the EVEN rows h0+2g, block O (the next 64
//     columns) the ODD rows h0+2g+1, g = 0..15 = the MMA's 8-lane row groups;
//   * the input is loaded through two row-parity views, so a "half strip" is 17 dense rows of one parity;
//   * an A window starting at image row h0+rho (rho = -1..2, stepping 2 rows per lane group) contributes tap
//     kh = rho+1 to block E and tap kh = rho to block O:
//         rho = -1: E += W[kh0]                  (N = 64)       rho = 0: [E | O] += [W[kh1] | W[kh0]]   (N = 128)
//         rho =  1: [E | O] += [W[kh2] | W[kh1]] (N = 128)      rho = 2: O += W[kh2]                    (N = 64)
//     with the weights of one column shift resident in shared memory as 192 rows [kh2 ; kh1 ; kh0].
//
// 256 pixels x 9 taps cost 3 x 4 windows x 4 K-steps = 48 MMAs instead of 72, every accumulator lane is a finished
// output pixel, and the two blocks go to two independent 8-warp epilogue groups (the generic kernel's epilogue needs
// ~1600 cycles per 128 pixels, which would otherwise become the limiter).  Output / residual / mask tiles move through
// row-parity TMA views as well (16 rows x 8 pixels per block).
// =====================================================================================================================
struct IlKParams {
  // A launch may carry up to kIlMaxGroups independent problems of one geometry ("groups": the same layer of several
  // generators, each with its own tensors and filter).  CTA c works for group c % n_groups; with one group the arrays'
  // first entries are the whole launch.
  CUtensorMap in_map[2 * kIlMaxGroups];     // [group][image-row parity] 64-channel input view
  CUtensorMap w_map[kIlMaxGroups];
  CUtensorMap out_map[8];    // [n-block (pixel shuffle) or group][row parity]
  CUtensorMap aux_map[2 * kIlMaxGroups];    // [group][row parity] residual / mask tensor
  int n_groups;
  int N, H, W;
  int tiles_h, tiles_w, tiles_total;
  int strip_dw[3];
  int cout_total, n_blocks, ctas_per_block;
  int n_stages;
  const float* bias[kIlMaxGroups];
  const float* scale[kIlMaxGroups];   // optional per-channel multiplier of the accumulator (folded eval-mode BatchNorm)
  int act;
  float slope;
  int aux_mode;              // 0 none, 1 add (residual), 2 mask (zero where aux <= 0)
  int out_mode;
  float* stats[kIlMaxGroups];            // per-CTA channel sums / sums of squares (row = the CTA's index inside its group)
  uint64_t pol_out, pol_aux, pol_in; // L2 eviction priorities of the output store / the residual-mask tile loads / the operand strips
  int ramp;                  // 1: the first tile runs column shift by column shift (the filter streams in under the MMAs)
  long long* prof;
};

constexpr int kIlThreads = 64 + 512;            // warp 0 producer, warp 1 MMA, warps 2-9 block E, warps 10-17 block O
constexpr uint32_t kIlWBytes = 9 * 64 * 128;    // resident filter: [kw 3][kh2 ; kh1 ; kh0][64 cout][64 cin]
// ONE 10-pixel-wide half strip (17 rows x 10 pixels, row pitch 1280 B) serves all three column shifts: the A
// descriptor starts kw * 128 B into it with a stride (SBO) of 1280 B between 8-pixel row groups.  Measured on B200
// (tools/conv_probe il_* cases): the UMMA 128B swizzle is a function of the ABSOLUTE shared-memory address bits, exactly
// like the TMA write side, so a start address / group stride that is only 128-byte aligned reads the right data with
// base_offset = 0 (setting base_offset = (addr >> 7) & 7 gives wrong results).  One third of the L2->SM operand traffic
// and of the stage footprint of one 8-pixel half strip per column shift, so the same shared memory holds a 2x deeper
// prefetch.
constexpr uint32_t kIlWidePitch = 10 * 128;
constexpr uint32_t kIlWideStage = 22 * 1024;    // 17 x 1280 = 21760 B, rounded up to the 1024-byte swizzle period

// in-kernel stall counters of conv3_il (tools/conv_probe): compiled in only with -DSRG_IL_PROF, they cost ~10 registers
#ifdef SRG_IL_PROF
#define IL_PROF(...) __VA_ARGS__
#define IL_TIMED(slot, ...) { long long t0_ = clock64(); __VA_ARGS__ prof_acc[slot] += clock64() - t0_; }
#else
#define IL_PROF(...)
#define IL_TIMED(slot, ...) { __VA_ARGS__ }
#endif
// GROUPED: CTA c works for group c % n_groups (a run-time index into the per-group tensor maps / pointers).  Measured on one
// box: one body per group with a compile-time index (no spills, 3x the code) runs the grouped trunk launch in 38.5-40.9 us, the
// run-time index (8 bytes of spills) in 33.2 us (profiles/r02_ab_grouped.log), so the run-time index stays.
template <bool GROUPED>
__global__ void __launch_bounds__(kIlThreads, 1) conv3_il_kernel(const __grid_constant__ IlKParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __builtin_assume(__isShared(smem));      // the integer round-up hides the state space: keep LDS / STS instead of generic accesses
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  pdl_trigger();

  uint8_t* w_smem = smem;
  uint8_t* stages = w_smem + kIlWBytes;
  constexpr uint32_t kStage = kIlWideStage;
  uint8_t* out_stage = stages + size_t(p.n_stages) * kStage;             // [block 2][16 KB]
  uint8_t* aux_stage = out_stage + 2 * kTileOutBytes;                     // [block 2][16 KB] (aux_mode != 0)
  uint8_t* tail = aux_stage + (p.aux_mode ? 2 * kTileOutBytes : 0);
  float* s_bias = reinterpret_cast<float*>(tail);                         // 64 floats bias, 64 floats scale
  float* s_scale = s_bias + 64;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail + 512);
  uint64_t* full = bars;                                                  // [n_stages <= 8]
  uint64_t* empty = bars + 8;
  uint64_t* wfull = bars + 26;                                            // [kw 3]: the filter arrives per column shift
  uint64_t* tfull = bars + 17;                                            // [2]
  uint64_t* tempty = bars + 19;                                           // [2]
  uint64_t* auxfull = bars + 21;                                          // [block 2]
  uint64_t* auxempty = bars + 23;                                         // [block 2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 25);
  float* s_stats = reinterpret_cast<float*>(tail + 768);                  // [16][128] floats (p.stats only)

  // n_groups > 1 implies n_blocks == 1 (OUT_NHWC, 64 output channels)
  const int grp = GROUPED ? int(blockIdx.x) % p.n_groups : 0;
  const int nblk = GROUPED ? 0 : int(blockIdx.x) % p.n_blocks;
  const int tile0 = int(blockIdx.x) / (GROUPED ? p.n_groups : p.n_blocks);
  const CUtensorMap* const in_map = &p.in_map[2 * grp];
  const CUtensorMap* const w_map = &p.w_map[grp];
  const CUtensorMap* const aux_map = &p.aux_map[2 * grp];
  const CUtensorMap* const out_map = &p.out_map[GROUPED ? 2 * grp : 0];
  float* const stats = p.stats[grp];
  const int tiles_per_img = p.tiles_h * p.tiles_w;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < p.n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 3; ++i) mbar_init(&wfull[i], 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 512);
      mbar_init(&auxfull[i], 1);
      mbar_init(&auxempty[i], 256);
    }
    fence_barrier_init();
    tma_prefetch_desc(w_map);
    tma_prefetch_desc(&in_map[1]);
    tma_prefetch_desc(&in_map[0]);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  if (warp >= 2 && warp < 4) {
    const int t = threadIdx.x - 64;
    s_bias[t] = p.bias[grp] != nullptr ? p.bias[grp][nblk * 64 + t] : 0.f;
    s_scale[t] = p.scale[grp] != nullptr ? p.scale[grp][nblk * 64 + t] : 1.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  IL_PROF(long long prof_acc[4] = {0, 0, 0, 0}; const long long t_start = clock64();)

  if (warp == 0) {
    // =============================================================== TMA producer
    if (elect_one()) {
      // generic packing is k-block (kw*3 + kh); shared memory wants [kw][kh2 ; kh1 ; kh0]
      auto load_w = [&](int s) {
        mbar_expect_tx(&wfull[s], kIlWBytes / 3);
        for (int r = 0; r < 3; ++r)
          tma_load_2d(w_smem + size_t(s * 3 + (2 - r)) * 8192, w_map, &wfull[s], 0, (s * 3 + r) * p.cout_total + nblk * 64);
      };
      // ramp: only the first column shift's 24 KB go out ahead of the first tile's strips; the other two follow them.  All
      // CTAs start together and fetch the same 72 KB, so the ramp is bound by L2 bandwidth (148 x 72 KB): the first tile's
      // MMAs run column shift by column shift (see the MMA warp) and start after 45 KB instead of 115 KB have arrived.
      const bool ramp = p.ramp != 0;
      load_w(0);
      if (!ramp) { load_w(1); load_w(2); }
      pdl_wait();      // the activations (and aux tensor) come from the previous kernel; the weights above do not
      int stage = 0;
      uint32_t phase = 0;
      bool first = true;
      for (int tile = tile0; tile < p.tiles_total; tile += p.ctas_per_block) {
        const int n = tile / tiles_per_img;
        const int rem = tile - n * tiles_per_img;
        const int hh = (rem / p.tiles_w) * 16;       // tile origin in parity-view rows (h0 / 2)
        const int w0 = (rem % p.tiles_w) * 8;
#pragma unroll
        for (int par = 1; par >= 0; --par) {         // odd image rows h0-1+2j first, then even rows h0+2j (j = 0..16)
          IL_TIMED(0, mbar_wait(&empty[stage], phase ^ 1);)
          mbar_expect_tx(&full[stage], 17 * kIlWidePitch);
          tma_load_4d_hint(stages + size_t(stage) * kStage, &in_map[par], &full[stage], 0, w0 + p.strip_dw[0], hh - par, n, p.pol_in);
          if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
        }
        if (first) {
          if (ramp) { load_w(1); load_w(2); }
          if (p.aux_mode) {
            // the first tile's residual / mask blocks go out here, behind everything the first MMAs wait for (the TMA
            // engine fetches descriptors in order: an aux load issued first would hold the operands back)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
              mbar_expect_tx(&auxfull[b], kTileOutBytes);
              tma_load_4d_hint(aux_stage + b * kTileOutBytes, &aux_map[b], &auxfull[b], nblk * 64, w0, hh, n, p.pol_aux);
            }
          }
          first = false;
        }
        // the residual / mask tiles of the following tiles are loaded by the epilogue groups themselves (one buffer per group, the next tile's load
        // issued as soon as the group has read the current one): the operand prefetch never waits for an epilogue
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    constexpr uint32_t idesc64 = make_idesc_bf16(128, 64, 0, 0);
    constexpr uint32_t idesc128 = make_idesc_bf16(128, 128, 0, 0);
    const uint64_t desc_hi = (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    const uint32_t w_lo = smem_u32(w_smem) >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    bool w_ready = false;            // first tile: wait for each column shift's weights right before their first use
    for (int tile = tile0; tile < p.tiles_total; tile += p.ctas_per_block) {
      IL_TIMED(1, mbar_wait(&tempty[acc], acc_phase ^ 1);)
      tc_fence_after();
      const uint32_t d_e = tmem_base + uint32_t(acc * 128);
      const uint32_t d_o = d_e + 64;
      // descriptor high part: SBO = 1280 B between 8-pixel row groups, base_offset 0 (see kIlWidePitch)
      const uint64_t adesc_hi = (uint64_t(kIlWidePitch >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
      // the 16 MMAs of one (row parity, column shift) pair; a_base = the half strip's stage (1024-byte aligned)
      auto issue = [&](int par, int s, uint32_t a_base, bool fresh) {
        const uint32_t wb = w_lo + uint32_t(s) * (3 * 8192 >> 4);
        // window starting at half-strip row 0 / row 1, column shift s pixels
        const uint32_t st0 = a_base + uint32_t(s) * 128u, st1 = st0 + kIlWidePitch;
        const uint64_t a0 = adesc_hi | uint64_t((st0 & 0x3FFFFu) >> 4);
        const uint64_t a1 = adesc_hi | uint64_t((st1 & 0x3FFFFu) >> 4);
        if (par == 1) {
          const uint64_t b1 = desc_hi | uint64_t(wb);                         // rho = 1: E += kh2, O += kh1
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(d_e, a1 + uint64_t(2 * k), b1 + uint64_t(2 * k), idesc128, (!fresh || k > 0) ? 1u : 0u);
          const uint64_t b0 = desc_hi | uint64_t(wb + (2 * 8192 >> 4));       // rho = -1: E += kh0
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(d_e, a0 + uint64_t(2 * k), b0 + uint64_t(2 * k), idesc64, 1u);
        } else {
          const uint64_t b0 = desc_hi | uint64_t(wb + (8192 >> 4));           // rho = 0: E += kh1, O += kh0
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(d_e, a0 + uint64_t(2 * k), b0 + uint64_t(2 * k), idesc128, 1u);
          const uint64_t b1 = desc_hi | uint64_t(wb);                         // rho = 2: O += kh2
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(d_o, a1 + uint64_t(2 * k), b1 + uint64_t(2 * k), idesc64, 1u);
        }
      };
      if (!w_ready && p.ramp) {
        // first tile of a training launch: (kw0, odd) (kw0, even) | (kw1, odd) (kw2, odd) -> odd half strip released |
        // (kw1, even) (kw2, even): the MMAs start once the first 24 KB of the filter and the first half strip have landed
        // and the rest of the filter streams in underneath them.  Later tiles keep the strip-by-strip order (measured:
        // the interleaved order costs 4 % in the steady state).  Eval-mode (exclusive) launches never take this path, so an
        // output pixel's fp32 accumulation order does not depend on the tile slot that computes it and eval results stay
        // bit-identical between batch layouts.
        const int st1 = stage; const uint32_t ph1 = phase;
        if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
        const int st0 = stage; const uint32_t ph0 = phase;
        if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
        const uint32_t base1 = smem_u32(stages) + uint32_t(st1) * kStage, base0 = smem_u32(stages) + uint32_t(st0) * kStage;
        mbar_wait(&wfull[0], 0);
        IL_TIMED(2, mbar_wait(&full[st1], ph1);)
        IL_PROF(prof_acc[0] = clock64() - t_start;)     // ramp: launch -> first MMA issue
        tc_fence_after();
        if (elect_one()) issue(1, 0, base1, true);
        __syncwarp();
        IL_TIMED(2, mbar_wait(&full[st0], ph0);)
        tc_fence_after();
        if (elect_one()) issue(0, 0, base0, false);
        __syncwarp();
        mbar_wait(&wfull[1], 0);
        tc_fence_after();
        if (elect_one()) issue(1, 1, base1, false);
        __syncwarp();
        mbar_wait(&wfull[2], 0);
        tc_fence_after();
        if (elect_one()) {
          issue(1, 2, base1, false);
          umma_commit(&empty[st1]);
          issue(0, 1, base0, false);
          issue(0, 2, base0, false);
          umma_commit(&empty[st0]);
        }
        __syncwarp();
      } else {
#pragma unroll
        for (int par = 1; par >= 0; --par) {
          IL_TIMED(2, mbar_wait(&full[stage], phase);)
          tc_fence_after();
          const uint32_t a_base = smem_u32(stages) + uint32_t(stage) * kStage;     // 1024-byte aligned
          if (!w_ready) {           // first tile in the plain order: every column shift's weights before its first use
            mbar_wait(&wfull[0], 0); mbar_wait(&wfull[1], 0); mbar_wait(&wfull[2], 0);
            IL_PROF(if (par == 1) prof_acc[0] = clock64() - t_start;)
            tc_fence_after();
          }
          if (elect_one()) {
#pragma unroll
            for (int s = 0; s < 3; ++s) issue(par, s, a_base, s == 0 && par == 1);
            umma_commit(&empty[stage]);
          }
          __syncwarp();
          if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
        }
      }
      w_ready = true;
      if (elect_one()) umma_commit(&tfull[acc]);
      __syncwarp();
      IL_PROF(prof_acc[3] = clock64() - t_start;)                              // last commit issued
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    // =================================================================== epilogue: two independent 8-warp groups
    const int blk = (warp - 2) >> 3;           // 0: even rows (block E), 1: odd rows (block O)
    const int gw = (warp - 2) & 7;
    const int q = warp & 3;                    // TMEM lane quadrant this warp may read
    const int m = q * 32 + lane;               // GEMM row: lane group g = m >> 3 is image row h0 + 2g + blk
    const int hf = gw >> 2;                    // which 32-column half of the block's 64 columns
    const int gtid = gw * 32 + lane;           // thread index inside the group
    const int bar_a = 1 + 2 * blk, bar_b = 2 + 2 * blk;
    uint8_t* my_out = out_stage + blk * kTileOutBytes;
    const uint8_t* my_aux = aux_stage + blk * kTileOutBytes;
    int acc = 0;
    uint32_t acc_phase = 0, aux_phase = 0;
    // statistics: thread (c4 = gtid & 15, rp = gtid >> 4) owns channels 4*c4 .. 4*c4+3 of rows 8*rp .. 8*rp+7 of the block
    float st_s[4] = {0.f, 0.f, 0.f, 0.f}, st_q[4] = {0.f, 0.f, 0.f, 0.f};
    const int c4 = gtid & 15, rp = gtid >> 4;
    auto load_aux = [&](int tile) {           // one thread per group: this group's 16 KB of the residual / mask tile
      const int n = tile / tiles_per_img;
      const int rem = tile - n * tiles_per_img;
      mbar_expect_tx(&auxfull[blk], kTileOutBytes);
      tma_load_4d_hint(aux_stage + blk * kTileOutBytes, &aux_map[blk], &auxfull[blk], nblk * 64, (rem % p.tiles_w) * 8,
                       (rem / p.tiles_w) * 16, n, p.pol_aux);
    };
    for (int tile = tile0; tile < p.tiles_total; tile += p.ctas_per_block) {
      const int n = tile / tiles_per_img;
      const int rem = tile - n * tiles_per_img;
      const int hh = (rem / p.tiles_w) * 16;
      const int w0 = (rem % p.tiles_w) * 8;
      IL_TIMED(3, mbar_wait(&tfull[acc], acc_phase);) IL_PROF(prof_acc[0] = clock64() - t_start;)
      tc_fence_after();
      const uint32_t t_addr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * 128 + blk * 64 + hf * 32);
      uint32_t v[32];
      tmem_ld32(t_addr, v);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&tempty[acc]);

      float f[32];
      {
        const float4* bp = reinterpret_cast<const float4*>(s_bias + hf * 32);
        const float4* sp4 = reinterpret_cast<const float4*>(s_scale + hf * 32);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 b = bp[g];
          const float4 sc = sp4[g];
          f[4 * g + 0] = fmaf(__uint_as_float(v[4 * g + 0]), sc.x, b.x);
          f[4 * g + 1] = fmaf(__uint_as_float(v[4 * g + 1]), sc.y, b.y);
          f[4 * g + 2] = fmaf(__uint_as_float(v[4 * g + 2]), sc.z, b.z);
          f[4 * g + 3] = fmaf(__uint_as_float(v[4 * g + 3]), sc.w, b.w);
        }
      }
      if (p.act == ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = apply_act<ACT_RELU>(f[j], 0.f);
      } else if (p.act == ACT_LRELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = apply_act<ACT_LRELU>(f[j], p.slope);
      }
      const uint32_t row_off = uint32_t(m) * 128u;
      const uint32_t sw = uint32_t(m & 7);
      if (p.aux_mode) {
        mbar_wait(&auxfull[blk], aux_phase);
        const uint8_t* ap = my_aux + row_off;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const uint4 r = *reinterpret_cast<const uint4*>(ap + (((uint32_t(hf * 4 + g)) ^ sw) << 4));
          const uint32_t ws[4] = {r.x, r.y, r.z, r.w};
          if (p.aux_mode == 1) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              f[g * 8 + 2 * e] += bf16_lo(ws[e]);
              f[g * 8 + 2 * e + 1] += bf16_hi(ws[e]);
            }
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              if (!(bf16_lo(ws[e]) > 0.f)) f[g * 8 + 2 * e] = 0.f;
              if (!(bf16_hi(ws[e]) > 0.f)) f[g * 8 + 2 * e + 1] = 0.f;
            }
          }
        }
        aux_phase ^= 1;
      }
      // stage the bf16 block (128B-swizzled rows) and hand it to the TMA store engine; one staging buffer per group
      if (gtid == 0) tma_store_wait_read<0>();      // this group's previous store has drained the buffer
      named_bar_sync(bar_a, 256);                   // ... and every thread of the group has read its part of the aux tile
      if (p.aux_mode && gtid == 0 && tile + p.ctas_per_block < p.tiles_total) load_aux(tile + p.ctas_per_block);
      uint8_t* op = my_out + row_off;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 o;
        o.x = pack_bf16(f[g * 8 + 0], f[g * 8 + 1]);
        o.y = pack_bf16(f[g * 8 + 2], f[g * 8 + 3]);
        o.z = pack_bf16(f[g * 8 + 4], f[g * 8 + 5]);
        o.w = pack_bf16(f[g * 8 + 6], f[g * 8 + 7]);
        *reinterpret_cast<uint4*>(op + (((uint32_t(hf * 4 + g)) ^ sw) << 4)) = o;
      }
      fence_proxy_async_smem();
      // a tile whose 16 rows x 8 pixels all lie inside the image needs no bounds tests in the statistics loop
      const bool full_tile = 2 * (hh + 15) + blk < p.H && w0 + 7 < p.W;
      named_bar_sync(bar_b, 256);
      if (gtid == 0) {
        const bool ps = p.out_mode == OUT_PIXEL_SHUFFLE;
        tma_store_4d_hint(&out_map[(ps ? nblk : 0) * 2 + blk], my_out, ps ? 0 : nblk * 64, w0, hh, n, p.pol_out);
        tma_store_commit();
      }
      if (stats != nullptr) {
        // column sums of the staged bf16 block (exactly the values BatchNorm will normalise): 8 conflict-free 8-byte
        // reads per thread (a half warp covers one 128-byte row)
        const uint8_t* sp = my_out + rp * 1024 + (c4 & 1) * 8;
        const uint32_t cch = uint32_t(c4 >> 1);
        const bool row_ok = full_tile || 2 * (hh + rp) + blk < p.H;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          if (row_ok && (full_tile || w0 + r < p.W)) {
            const uint2 sv = *reinterpret_cast<const uint2*>(sp + r * 128 + ((cch ^ uint32_t(r)) << 4));
            const float a0 = bf16_lo(sv.x), a1 = bf16_hi(sv.x), a2 = bf16_lo(sv.y), a3 = bf16_hi(sv.y);
            st_s[0] += a0; st_s[1] += a1; st_s[2] += a2; st_s[3] += a3;
            st_q[0] = fmaf(a0, a0, st_q[0]); st_q[1] = fmaf(a1, a1, st_q[1]);
            st_q[2] = fmaf(a2, a2, st_q[2]); st_q[3] = fmaf(a3, a3, st_q[3]);
          }
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    IL_PROF(prof_acc[1] = clock64() - t_start;)  // last tile's store handed to the TMA engine (+ statistics loop)
    if (gtid == 0) tma_store_wait_all<0>();
    IL_PROF(prof_acc[2] = clock64() - t_start;)
    if (stats != nullptr) {
      // lanes l and l+16 hold the same channels of different rows: fold them, then one row of partials per warp
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        st_s[e] += __shfl_xor_sync(0xFFFFFFFFu, st_s[e], 16);
        st_q[e] += __shfl_xor_sync(0xFFFFFFFFu, st_q[e], 16);
      }
      const int part = blk * 8 + (gtid >> 5);
      if (lane < 16) {
        *reinterpret_cast<float4*>(s_stats + part * 128 + 4 * c4) = make_float4(st_s[0], st_s[1], st_s[2], st_s[3]);
        *reinterpret_cast<float4*>(s_stats + part * 128 + 64 + 4 * c4) = make_float4(st_q[0], st_q[1], st_q[2], st_q[3]);
      }
      named_bar_sync(5, 512);
      if (blk == 0 && gtid < 128) {
        float t = 0.f;
#pragma unroll
        for (int g = 0; g < 16; ++g) t += s_stats[g * 128 + gtid];
        stats[size_t(GROUPED ? tile0 : int(blockIdx.x)) * 128 + gtid] = t;
      }
    }
  }

#ifdef SRG_IL_PROF
  if (p.prof != nullptr && lane == 0 && (warp <= 2)) {
    long long* d = p.prof + (size_t(blockIdx.x) * 3 + warp) * 6;
    d[0] = prof_acc[0]; d[1] = prof_acc[1]; d[2] = prof_acc[2]; d[3] = prof_acc[3]; d[4] = clock64() - t_start; d[5] = t_start;
  }
#endif
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 256);
}

// =====================================================================================================================
// 9x9 convolution with 3 output channels (conv3 of the generator, the last layer at 4x resolution): "conv9_rows".
//
// The generic fold9 instance folds the 9 horizontal taps into N = 27 (+5) and issues one N = 32 MMA per row tap and
// K-step: with the ~64-cycle floor of an M128 MMA that is 4 % of the tensor rate.  Here one MMA consumes ONE image row
// segment (128 pixels x 64 channels) and feeds up to 8 output rows at once: TMEM block j (32 columns) is output row
// h0 + j, and the input row h0 + rho contributes row tap kh = rho - j + 4 to every block with 0 <= kh <= 8.  With the
// filter resident as 288 rows [kh8 ; kh7 ; ... ; kh0] (32 rows = 9 column taps x 3 channels each), the blocks a row
// touches are CONTIGUOUS in both the B operand and the accumulator, so one MMA of N = 32 x (number of blocks, <= 256)
// covers them: 16 input rows x 4 K-steps (+7 first-touch splits) = 71 MMAs per 8 x 120 output pixels instead of 360,
// 4.5x fewer tensor-pipe cycles.  The epilogue (two 4-warp groups, 4 blocks each) shift-accumulates the 9 column taps
// through shared memory and writes fp32 NCHW.  Tiles are 128 pixels wide with a 4-pixel halo on each side.
// =====================================================================================================================
struct C9KParams {
  CUtensorMap in_map;        // {64, W, H, N}, box {64, 128, 1, 1}
  CUtensorMap w_map;         // {64, 9*32}, box {64, 32}
  int N, H, W;
  int tiles_h, tiles_w, tiles_total, n_ctas;
  int n_stages;
  const float* bias;         // [3] or null
  void* out;                 // through `scatter`
  long long* prof;
  FoldScatter scatter;
};

constexpr int kC9Threads = 64 + 256;            // warp 0 producer, warp 1 MMA, warps 2-5 / 6-9 epilogue groups
constexpr uint32_t kC9Row = 128 * 128;          // one image-row segment: 128 pixels x 64 bf16
constexpr uint32_t kC9WBytes = 9 * 32 * 128;    // resident filter

__global__ void __launch_bounds__(kC9Threads, 1) conv9_rows_kernel(const __grid_constant__ C9KParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __builtin_assume(__isShared(smem));
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  pdl_trigger();

  uint8_t* w_smem = smem;                                   // 36 KB
  uint8_t* stages = w_smem + kC9WBytes;                     // n_stages x 16 KB
  float* fold_buf = reinterpret_cast<float*>(stages + size_t(p.n_stages) * kC9Row);   // [group 2][128][33]
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(fold_buf) + 2 * 128 * kFoldPad * 4);
  uint64_t* full = bars;                                    // [n_stages <= 10]
  uint64_t* empty = bars + 10;
  uint64_t* wfull = bars + 20;
  uint64_t* tfull = bars + 21;                              // [2]
  uint64_t* tempty = bars + 23;                             // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 25);
  const int tiles_per_img = p.tiles_h * p.tiles_w;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < p.n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(wfull, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 256);
    }
    fence_barrier_init();
    tma_prefetch_desc(&p.in_map);
    tma_prefetch_desc(&p.w_map);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  long long prof_acc[4] = {0, 0, 0, 0};
  const long long t_start = clock64();

  if (warp == 0) {
    // =============================================================== TMA producer: one image-row segment per stage
    if (elect_one()) {
      mbar_expect_tx(wfull, kC9WBytes);
      for (int r = 0; r < 9; ++r) tma_load_2d(w_smem + size_t(8 - r) * 4096, &p.w_map, wfull, 0, r * 32);
      pdl_wait();
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.tiles_total; tile += p.n_ctas) {
        const int n = tile / tiles_per_img;
        const int rem = tile - n * tiles_per_img;
        const int h0 = (rem / p.tiles_w) * 8;
        const int w0 = (rem % p.tiles_w) * 120 - 4;
        for (int ri = 0; ri < 16; ++ri) {
          { long long t0_ = clock64(); mbar_wait(&empty[stage], phase ^ 1); prof_acc[0] += clock64() - t0_; }
          mbar_expect_tx(&full[stage], kC9Row);
          tma_load_4d(stages + size_t(stage) * kC9Row, &p.in_map, &full[stage], 0, w0, h0 + ri - 4, n);
          if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    constexpr uint32_t idesc0 = make_idesc_bf16(128, 0, 0, 0);        // N field (bits 17-22) filled per MMA
    const uint64_t desc_hi = (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    const uint32_t stage0_lo = smem_u32(stages) >> 4;
    const uint32_t w_lo = smem_u32(w_smem) >> 4;
    mbar_wait(wfull, 0);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.tiles_total; tile += p.n_ctas) {
      { long long t0_ = clock64(); mbar_wait(&tempty[acc], acc_phase ^ 1); prof_acc[1] += clock64() - t0_; }
      tc_fence_after();
      const uint32_t d_base = tmem_base + uint32_t(acc * 256);
#pragma unroll 1
      for (int ri = 0; ri < 16; ++ri) {          // input row h0 + ri - 4
        { long long t0_ = clock64(); mbar_wait(&full[stage], phase); prof_acc[2] += clock64() - t0_; }
        tc_fence_after();
        const C9Window win = c9_window(ri);      // output rows (blocks) this input row reaches: kh = ri - j in [0, 8]
        const int jlo = win.jlo, jhi = win.jhi;
        const bool fresh = win.fresh != 0;       // block jhi = ri sees its first tap (kh = 0) here
        const uint64_t adesc = desc_hi | uint64_t(stage0_lo + uint32_t(stage) * (kC9Row >> 4));
        const uint64_t b_all = desc_hi | uint64_t(w_lo + uint32_t(win.slot_lo) * (4096 >> 4));     // slot of block jlo
        const uint64_t b_kh0 = desc_hi | uint64_t(w_lo + 8u * (4096 >> 4));
        if (elect_one()) {
          const uint32_t n_all = uint32_t(jhi - jlo + 1) * 32u;
          if (fresh) {
            // K-step 0: the fresh block must overwrite (accumulate = 0), the older blocks accumulate
            if (jhi > jlo) umma_bf16(d_base + uint32_t(jlo * 32), adesc, b_all, idesc0 | (((n_all - 32u) >> 3) << 17), 1u);
            umma_bf16(d_base + uint32_t(jhi * 32), adesc, b_kh0, idesc0 | ((32u >> 3) << 17), 0u);
          } else {
            umma_bf16(d_base + uint32_t(jlo * 32), adesc, b_all, idesc0 | ((n_all >> 3) << 17), 1u);
          }
#pragma unroll
          for (int k = 1; k < 4; ++k)
            umma_bf16(d_base + uint32_t(jlo * 32), adesc + uint64_t(2 * k), b_all + uint64_t(2 * k), idesc0 | ((n_all >> 3) << 17), 1u);
          umma_commit(&empty[stage]);
        }
        __syncwarp();
        if (++stage == p.n_stages) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(&tfull[acc]);
      __syncwarp();
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    // =================================================================== epilogue: two 4-warp groups, 4 blocks each
    const int grp = (warp - 2) >> 2;
    const int q = warp & 3;
    const int m = q * 32 + lane;               // pixel within the 128-wide tile
    float* fb = fold_buf + grp * 128 * kFoldPad;
    const float b0 = p.bias ? p.bias[0] : 0.f, b1 = p.bias ? p.bias[1] : 0.f, b2 = p.bias ? p.bias[2] : 0.f;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.tiles_total; tile += p.n_ctas) {
      const int n = tile / tiles_per_img;
      const int rem = tile - n * tiles_per_img;
      const int h0 = (rem / p.tiles_w) * 8;
      const int w0 = (rem % p.tiles_w) * 120 - 4;
      const int w = w0 + m;
      { long long t0_ = clock64(); mbar_wait(&tfull[acc], acc_phase); prof_acc[3] += clock64() - t0_; }
      tc_fence_after();
#pragma unroll 1
      for (int jj = 0; jj < 4; ++jj) {
        const int j = grp + 2 * jj;
        uint32_t v[32];
        tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(acc * 256 + j * 32), v);
        tmem_ld_wait();
        if (jj == 3) {
          tc_fence_before();
          mbar_arrive(&tempty[acc]);
        }
#pragma unroll
        for (int c = 0; c < 32; ++c) fb[m * kFoldPad + c] = __uint_as_float(v[c]);
        named_bar_sync(1 + 2 * grp, 128);
        const int h = h0 + j;
        const bool in_crop = p.scatter.n == 0 || (h >= p.scatter.t[n].h_lo && h < p.scatter.t[n].h_hi &&
                                                  w >= p.scatter.t[n].w_lo && w < p.scatter.t[n].w_hi);
        if (m >= 4 && m < 124 && h < p.H && w < p.W && in_crop) {
          float o0 = b0, o1 = b1, o2 = b2;
#pragma unroll
          for (int s = 0; s < 9; ++s) {
            const float* row = fb + (m + s - 4) * kFoldPad + s * 3;
            o0 += row[0];
            o1 += row[1];
            o2 += row[2];
          }
          fold9_store(p.scatter, p.out, n, h, w, o0, o1, o2);
        }
        named_bar_sync(2 + 2 * grp, 128);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }

  if (p.prof != nullptr && lane == 0 && (warp <= 2)) {
    long long* d = p.prof + (size_t(blockIdx.x) * 3 + warp) * 6;
    d[0] = prof_acc[0]; d[1] = prof_acc[1]; d[2] = prof_acc[2]; d[3] = prof_acc[3]; d[4] = clock64() - t_start; d[5] = t_start;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ----------------------------------------------------------- host launcher
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || sym == nullptr) return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

int encode_map_bf16(CUtensorMap* map, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
    return -100;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(ptr), dims, strides_bytes, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_ERROR_INVALID_CONTEXT || r == CUDA_ERROR_NOT_INITIALIZED) {
    // a thread that has not made a runtime call yet (e.g. autograd's backward worker) has no current driver context:
    // bind the device's primary context through the runtime and retry
    cudaFree(nullptr);
    r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(ptr), dims, strides_bytes, box, estr,
           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: CUresult %d (rank %d dims %llu,%llu box %u,%u)", int(r), rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    return -101;
  }
  return 0;
}

static int g_num_sms = 0;
int sm_budget() {
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

template <int BLOCK_N, int NT>
static int launch_instance(const typename KParamsOf<BLOCK_N>::type& p, dim3 grid, size_t smem_bytes, cudaStream_t stream) {
  static DeviceOnce attr_set;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_gemm_kernel<BLOCK_N, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         227 * 1024);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return int(e); }
    attr_set = true;
  }
  cudaError_t e = launch_pdl(conv_gemm_kernel<BLOCK_N, NT>, grid, dim3(kThreads), smem_bytes, stream, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("conv_gemm launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

static int g_variant_override = 0;
int set_conv_variant(int variant) {
  if (variant != 0 && variant != 1) { set_error("set_conv_variant: variant %d is not 0 (automatic) or 1 (generic)", variant); return -1; }
  const int old = g_variant_override;
  g_variant_override = variant;
  return old;
}
static int effective_variant(const ConvGemmArgs& a) { return a.variant != 0 ? a.variant : g_variant_override; }
// conv3_il applies to the plain 3x3 / 64-input-channel launches (trunk fprop + dgrad, up-conv fprop) whose three column
// shifts are -1, 0, +1 (one 10-pixel strip starting at w0 - 1); everything else (multi-view inputs, 9x9 row pairs, fold9,
// fp32 outputs) stays on the generic kernel.
static bool use_conv3_il(const ConvGemmArgs& a) {
  if (effective_variant(a) == 1) return false;
  return a.TH == 16 && a.TW == 8 && a.block_n == 64 && a.n_strips == 3 && a.n_taps == 3 && a.strip_dh == -1 &&
         a.strip_dw[0] == -1 && a.strip_dw[1] == 0 && a.strip_dw[2] == 1 &&
         a.strip_rows == 18 && a.tap_row[0] == 0 && a.tap_row[1] == 1 && a.tap_row[2] == 2 && a.n_views == 1 &&
         a.views[0].channels == 64 && a.in_H == a.H && a.in_W == a.W && a.H >= 2 &&
         (a.out_mode == OUT_NHWC || a.out_mode == OUT_PIXEL_SHUFFLE) &&
         a.cout_total % 64 == 0 && a.cout_total <= 256;
}

// row-parity view of a [N, H, W, C] tensor given by element strides: rows 2j + par
static int encode_parity_map(CUtensorMap* map, const void* base, int C, int W, int H, int N, int64_t stride_w,
                             int64_t stride_h, int64_t stride_n, int par, uint32_t box_rows, uint32_t box_w = 8) {
  const __nv_bfloat16* ptr = reinterpret_cast<const __nv_bfloat16*>(base) + size_t(par) * stride_h;
  uint64_t dims[4] = {uint64_t(C), uint64_t(W), uint64_t((H - par + 1) / 2), uint64_t(N)};
  uint64_t strides[3] = {uint64_t(stride_w) * 2, uint64_t(stride_h) * 4, uint64_t(stride_n) * 2};
  uint32_t box[4] = {64, box_w, box_rows, 1};
  return encode_map_bf16(map, ptr, 4, dims, strides, box);
}

// `as[0 .. n)`: one problem per group (n = 1: a plain launch).  Groups must agree in everything but the tensors, the filter,
// the bias / scale vectors and the statistics rows.
static int launch_conv3_il(const ConvGemmArgs* as, int n, cudaStream_t stream) {
  const ConvGemmArgs& a = as[0];
  if (n < 1 || n > kIlMaxGroups) { set_error("conv3_il: 1..%d groups", kIlMaxGroups); return -17; }
  for (int g = 1; g < n; ++g) {
    const ConvGemmArgs& o = as[g];
    if (o.N != a.N || o.H != a.H || o.W != a.W || o.in_H != a.in_H || o.in_W != a.in_W || o.cout_total != 64 || a.cout_total != 64 ||
        o.out_mode != OUT_NHWC || a.out_mode != OUT_NHWC || o.act != a.act || o.slope != a.slope || o.exclusive != a.exclusive ||
        (o.residual != nullptr) != (a.residual != nullptr) || (o.mask_src != nullptr) != (a.mask_src != nullptr) ||
        (o.stats != nullptr) != (a.stats != nullptr) ||
        o.views[0].stride_w != a.views[0].stride_w || o.views[0].stride_h != a.views[0].stride_h ||
        o.views[0].stride_n != a.views[0].stride_n || o.strip_dw[0] != a.strip_dw[0] || o.strip_dw[1] != a.strip_dw[1] ||
        o.strip_dw[2] != a.strip_dw[2] || effective_variant(o) != effective_variant(a) || a.prof != nullptr) {
      set_error("conv3_il: the problems of a grouped launch must share geometry, epilogue and layout (OUT_NHWC, 64 channels)");
      return -18;
    }
  }
  if (a.residual != nullptr && a.mask_src != nullptr) { set_error("conv_gemm: residual and mask are exclusive"); return -11; }
  const bool has_aux = a.residual != nullptr || a.mask_src != nullptr;
  if (has_aux && a.out_mode != OUT_NHWC) { set_error("conv_gemm: residual/mask need OUT_NHWC"); return -12; }
  if (a.out_mode == OUT_PIXEL_SHUFFLE && a.cout_total != 256) { set_error("conv_gemm: pixel shuffle needs cout 256"); return -13; }
  if (a.stats != nullptr && (a.out_mode != OUT_NHWC || a.cout_total != 64)) {
    set_error("conv_gemm: fused statistics need OUT_NHWC with 64 output channels"); return -16;
  }
  IlKParams p;
  memset(&p, 0, sizeof(p));
  p.N = a.N; p.H = a.H; p.W = a.W;
  p.tiles_h = (a.H + 31) / 32;
  p.tiles_w = (a.W + 7) / 8;
  p.tiles_total = a.N * p.tiles_h * p.tiles_w;
  if (p.tiles_total == 0) return 0;
  for (int s = 0; s < 3; ++s) p.strip_dw[s] = a.strip_dw[s];
  p.cout_total = a.cout_total;
  p.n_blocks = a.cout_total / 64;
  p.n_groups = n;
  p.ctas_per_block = sm_budget() / (p.n_blocks * n);      // CTAs per n-block, or per group
  if (p.ctas_per_block < 1) p.ctas_per_block = 1;
  if (p.ctas_per_block > p.tiles_total) p.ctas_per_block = p.tiles_total;
  p.aux_mode = a.residual ? 1 : (a.mask_src ? 2 : 0);
  const uint32_t fixed_bytes = kIlWBytes + 2 * kTileOutBytes + (has_aux ? 2 * kTileOutBytes : 0) + 768 +
                               (a.stats != nullptr ? 16 * 128 * 4 : 0);
  // Training launches leave 44 KB of the SM's shared memory to CTAs of other graph branches (chan_reduce, finalize, loss
  // passes need 8-18 KB): measured 11.27 -> 11.14 ms per cfg2 step; the shallower pipeline (3 / 2 stages) costs nothing
  // (profiles/r01_notes.md).  Launches with a residual / mask tile keep everything (they would be down to two stages: the
  // operand prefetch of the next tile could not start before half of the current tile's MMAs have retired; probe: 14.0 ->
  // 12.8 us at cfg2), and so do inference (exclusive) launches.
  constexpr int kIlSmemReserveKb = 44;
  const int reserve_kb = (a.exclusive || has_aux) ? 0 : kIlSmemReserveKb;
  int stages = int((227 * 1024 - reserve_kb * 1024 - 1024 - fixed_bytes) / kIlWideStage);
  if (stages > 8) stages = 8;      // full[] / empty[] hold 8 barriers
  if (stages < 2) stages = 2;
  p.n_stages = stages;
  const size_t smem_bytes = 1024 + fixed_bytes + size_t(stages) * kIlWideStage;

  for (int g = 0; g < n; ++g) {
    const ConvGemmArgs& ag = as[g];
    const InView& iv = ag.views[0];
    for (int par = 0; par < 2; ++par) {
      int rc = encode_parity_map(&p.in_map[2 * g + par], iv.ptr, 64, a.in_W, a.in_H, a.N, iv.stride_w, iv.stride_h, iv.stride_n, par, 17,
                                 10);
      if (rc) return rc;
    }
    {
      uint64_t dims[2] = {64, uint64_t(9) * a.cout_total};
      uint64_t strides[1] = {128};
      uint32_t box[2] = {64, 64};
      int rc = encode_map_bf16(&p.w_map[g], ag.weights, 2, dims, strides, box);
      if (rc) return rc;
    }
    if (a.out_mode == OUT_PIXEL_SHUFFLE) {       // n == 1
      // view q=(i,j) of the HR tensor [N,2H,2W,64]: pixel (2h+i, 2w+j)
      for (int q = 0; q < 4; ++q) {
        const int i = q >> 1, j = q & 1;
        const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(a.out) + (size_t(i) * 2 * a.W + j) * 64;
        for (int par = 0; par < 2; ++par) {
          int rc = encode_parity_map(&p.out_map[q * 2 + par], base, 64, a.W, a.H, a.N, 128, int64_t(4) * a.W * 64,
                                     int64_t(4) * a.H * a.W * 64, par, 16);
          if (rc) return rc;
        }
      }
      p.aux_map[0] = p.aux_map[1] = p.out_map[0];
    } else {
      const int64_t C = a.cout_total;
      for (int par = 0; par < 2; ++par) {
        int rc = encode_parity_map(&p.out_map[2 * g + par], ag.out, int(C), a.W, a.H, a.N, C, int64_t(a.W) * C, int64_t(a.H) * a.W * C, par, 16);
        if (rc) return rc;
        if (has_aux) {
          rc = encode_parity_map(&p.aux_map[2 * g + par], ag.residual ? ag.residual : ag.mask_src, int(C), a.W, a.H, a.N, C,
                                 int64_t(a.W) * C, int64_t(a.H) * a.W * C, par, 16);
          if (rc) return rc;
        } else {
          p.aux_map[2 * g + par] = p.out_map[2 * g + par];
        }
      }
      if (n == 1) for (int q = 2; q < 8; ++q) p.out_map[q] = p.out_map[q & 1];
    }
    p.bias[g] = ag.bias; p.scale[g] = ag.scale;
    p.stats[g] = ag.stats;
  }
  p.act = a.act; p.slope = a.slope;
  p.out_mode = a.out_mode;
  // training launches (not exclusive): the output is read by the statistics / apply passes right behind this kernel (keep
  // it in L2 ahead of streaming data); a mask / residual tile is dead after this read.  The operand tensor is not read again
  // before the weight gradients at the end of backward (neighbouring tiles re-read their halo within microseconds, long
  // before capacity pressure evicts it)
  p.pol_out = a.exclusive ? kL2EvictNormal : kL2EvictLast;
  p.pol_aux = a.exclusive ? kL2EvictNormal : kL2EvictFirst;
  p.pol_in = a.exclusive ? kL2EvictNormal : kL2EvictFirst;
  p.prof = reinterpret_cast<long long*>(a.prof);
  p.ramp = a.exclusive ? 0 : 1;
  static DeviceOnce attr_set;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv3_il_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3_il_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return int(e); }
    attr_set = true;
  }
  const dim3 grid(p.ctas_per_block * p.n_blocks * n);
  void (*const kernel)(IlKParams) = n > 1 ? conv3_il_kernel<true> : conv3_il_kernel<false>;
  cudaError_t e = a.exclusive ? launch_pdl_exclusive(kernel, grid, dim3(kIlThreads), smem_bytes, stream, p)
                              : launch_pdl(kernel, grid, dim3(kIlThreads), smem_bytes, stream, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("conv3_il launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

// conv9_rows replaces the fold9 instance of the generic kernel for the plain case (one 64-channel view, 9 row taps
// starting 4 rows above the tile); ConvGemmArgs::variant == 1 keeps the generic kernel.
static bool use_conv9_rows(const ConvGemmArgs& a) {
  const int variant = effective_variant(a);
  if (variant == 1 || a.out_mode != OUT_FOLD9_NCHW) return false;
  if (a.block_n != 32 || a.cout_total != 32 || a.n_strips != 1 || a.n_taps != 9 || a.strip_dh != -4 || a.strip_dw[0] != 0) return false;
  for (int r = 0; r < 9; ++r) if (a.tap_row[r] != r) return false;
  return a.n_views == 1 && a.views[0].channels == 64 && a.in_H == a.H && a.in_W == a.W && a.residual == nullptr &&
         a.mask_src == nullptr && a.stats == nullptr && a.act == ACT_NONE && a.scale == nullptr;
}

static int launch_conv9_rows(const ConvGemmArgs& a, cudaStream_t stream) {
  C9KParams p;
  memset(&p, 0, sizeof(p));
  p.N = a.N; p.H = a.H; p.W = a.W;
  p.tiles_h = (a.H + 7) / 8;
  p.tiles_w = (a.W + 119) / 120;
  p.tiles_total = a.N * p.tiles_h * p.tiles_w;
  if (p.tiles_total == 0) return 0;
  p.n_ctas = sm_budget() < p.tiles_total ? sm_budget() : p.tiles_total;
  const uint32_t fixed_bytes = kC9WBytes + 2 * 128 * kFoldPad * 4 + 512;
  int stages = int((227 * 1024 - 1024 - fixed_bytes) / kC9Row);
  if (stages > 10) stages = 10;
  p.n_stages = stages;
  const size_t smem_bytes = 1024 + fixed_bytes + size_t(stages) * kC9Row;
  {
    const InView& iv = a.views[0];
    uint64_t dims[4] = {64, uint64_t(a.in_W), uint64_t(a.in_H), uint64_t(a.N)};
    uint64_t strides[3] = {uint64_t(iv.stride_w) * 2, uint64_t(iv.stride_h) * 2, uint64_t(iv.stride_n) * 2};
    uint32_t box[4] = {64, 128, 1, 1};
    int rc = encode_map_bf16(&p.in_map, iv.ptr, 4, dims, strides, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {64, uint64_t(9) * 32};
    uint64_t strides[1] = {128};
    uint32_t box[2] = {64, 32};
    int rc = encode_map_bf16(&p.w_map, a.weights, 2, dims, strides, box);
    if (rc) return rc;
  }
  p.bias = a.bias;
  p.out = a.out;
  p.prof = reinterpret_cast<long long*>(a.prof);
  p.scatter = a.scatter != nullptr ? *a.scatter : fold9_nchw(a.H, a.W);
  static DeviceOnce attr_set;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv9_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return int(e); }
    attr_set = true;
  }
  cudaError_t e = launch_pdl(conv9_rows_kernel, dim3(p.n_ctas), dim3(kC9Threads), smem_bytes, stream, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("conv9_rows launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

int conv_gemm_grid(const ConvGemmArgs& a) {
  const bool fold = a.out_mode == OUT_FOLD9_NCHW;
  const int step_w = fold ? a.TW - 8 : a.TW;
  const int step_h = use_conv3_il(a) ? 32 : a.TH;
  const int tiles = a.N * ((a.H + step_h - 1) / step_h) * ((a.W + step_w - 1) / step_w);
  const int n_blocks = a.cout_total / a.block_n;
  int per = sm_budget() / n_blocks;
  if (per < 1) per = 1;
  if (per > tiles) per = tiles;
  return per * n_blocks;
}

// Grouped launch: the same 3x3 / 64 -> 64 layer of n <= 3 independent problems (one per generator) in ONE conv3_il launch.
// Every CTA works for one group (its filter stays resident); with 49 CTAs per group a cfg2 trunk layer is 12 tiles per CTA
// instead of 4, so the launch ramp, the 72 KB filter load and the last tile's epilogue are paid once per 12 tiles.
// The statistics rows of a group are its CTAs' rows: conv_gemm_grouped_rows().
int conv_gemm_grouped_rows(const ConvGemmArgs& a, int n) {
  const int tiles = a.N * ((a.H + 31) / 32) * ((a.W + 7) / 8);
  int per = sm_budget() / (n < 1 ? 1 : n);
  if (per < 1) per = 1;
  if (per > tiles) per = tiles;
  return per;
}
int launch_conv_gemm_grouped(const ConvGemmArgs* as, int n, cudaStream_t stream) {
  if (n == 1) return launch_conv_gemm(as[0], stream);
  for (int g = 0; g < n; ++g)
    if (!use_conv3_il(as[g]) || as[g].cout_total != 64) { set_error("grouped launch: every problem must be a plain 3x3 64 -> 64 layer"); return -19; }
  return launch_conv3_il(as, n, stream);
}

int launch_conv_gemm(const ConvGemmArgs& a, cudaStream_t stream) {
  if (a.scatter != nullptr && (a.out_mode != OUT_FOLD9_NCHW || a.scatter->n > kMaxTiles ||
                              (a.scatter->n != 0 && a.scatter->n != a.N))) {
    set_error("conv_gemm: a fold9 store table needs the fold9 output and none or one entry per item (at most %d)", kMaxTiles);
    return -20;
  }
  if (use_conv3_il(a)) return launch_conv3_il(&a, 1, stream);
  if (use_conv9_rows(a)) return launch_conv9_rows(a, stream);
  if (a.TH * a.TW != 128 || a.TW % 8 != 0) { set_error("conv_gemm: tile must be 128 pixels with TW%%8==0"); return -1; }
  if (a.block_n != 64 && a.block_n != 32) { set_error("conv_gemm: block_n must be 32 or 64"); return -2; }
  if (a.cout_total % a.block_n != 0) { set_error("conv_gemm: cout_total %% block_n != 0"); return -3; }
  if (a.n_views < 1 || a.n_views > kMaxInMaps) { set_error("conv_gemm: bad n_views"); return -4; }
  if (a.n_strips < 1 || a.n_strips > kMaxStrips || a.n_taps < 1 || a.n_taps > kMaxTaps) {
    set_error("conv_gemm: bad strip/tap count"); return -5;
  }
  const bool fold = a.out_mode == OUT_FOLD9_NCHW;
  if (fold != (a.block_n == 32)) { set_error("conv_gemm: fold9 <=> block_n 32"); return -6; }
  if (a.strip_rows > 256 || a.TW > 256) { set_error("conv_gemm: TMA box too large"); return -7; }
  if (a.residual != nullptr && a.mask_src != nullptr) { set_error("conv_gemm: residual and mask are exclusive"); return -11; }
  const bool has_aux = a.residual != nullptr || a.mask_src != nullptr;
  if (has_aux && a.out_mode != OUT_NHWC) { set_error("conv_gemm: residual/mask need OUT_NHWC"); return -12; }
  if (a.out_mode == OUT_PIXEL_SHUFFLE && a.cout_total != 256) { set_error("conv_gemm: pixel shuffle needs cout 256"); return -13; }

  ConvKParams p;
  memset(&p, 0, sizeof(p));
  p.N = a.N; p.H = a.H; p.W = a.W; p.TH = a.TH; p.TW = a.TW;
  p.tile_step_w = fold ? a.TW - 8 : a.TW;
  p.tile_w_org = fold ? -4 : 0;
  p.tiles_h = (a.H + a.TH - 1) / a.TH;
  p.tiles_w = (a.W + p.tile_step_w - 1) / p.tile_step_w;
  p.tiles_total = a.N * p.tiles_h * p.tiles_w;
  int total_ch = 0;
  for (int v = 0; v < a.n_views; ++v) {
    if (a.views[v].channels % 64 != 0 || a.views[v].channels != a.views[0].channels) {
      set_error("conv_gemm: view channels must be equal multiples of 64"); return -8;
    }
    total_ch += a.views[v].channels;
  }
  p.n_chunks = total_ch / 64;
  p.chunks_per_view = a.views[0].channels / 64;
  p.n_strips = a.n_strips; p.strip_rows = a.strip_rows; p.strip_dh = a.strip_dh;
  for (int s = 0; s < a.n_strips; ++s) p.strip_dw[s] = a.strip_dw[s];
  for (int r = 0; r < a.n_taps; ++r) {
    if (a.tap_row[r] < 0 || a.tap_row[r] + a.TH > a.strip_rows) { set_error("conv_gemm: tap row outside strip"); return -9; }
    p.tap_row[r] = a.tap_row[r];
  }
  p.cout_total = a.cout_total;
  p.n_blocks = a.cout_total / a.block_n;
  const int sms = sm_budget();
  p.ctas_per_block = sms / p.n_blocks;
  if (p.ctas_per_block < 1) p.ctas_per_block = 1;
  if (p.ctas_per_block > p.tiles_total) p.ctas_per_block = p.tiles_total;
  if (p.tiles_total == 0) return 0;

  const uint32_t btile = uint32_t(a.block_n) * 128u;
  const int kb_total = p.n_chunks * a.n_strips * a.n_taps;
  p.strip_bytes = uint32_t(a.strip_rows) * a.TW * 128u;
  const uint32_t w_all = uint32_t(kb_total) * btile;
  p.aux_mode = a.residual ? 1 : (a.mask_src ? 2 : 0);
  if (a.stats != nullptr && (a.out_mode != OUT_NHWC || a.cout_total != 64 || a.TW != 8)) {
    set_error("conv_gemm: fused statistics need OUT_NHWC with 64 output channels and 8-pixel-wide tiles"); return -16;
  }
  const uint32_t fixed_bytes = (fold ? 128 * kFoldPad * 4 : 2 * kTileOutBytes) + (has_aux ? 2 * kTileOutBytes : 0) + 512 + 256 +
                               (a.stats != nullptr ? 8 * 128 * 4 : 0);
  const uint32_t budget = 227 * 1024 - 1024 - fixed_bytes;
  p.resident = (w_all + 3 * p.strip_bytes <= budget) ? 1 : 0;
  p.w_resident_bytes = p.resident ? w_all : 0;
  p.stage_bytes = p.strip_bytes + (p.resident ? 0 : uint32_t(a.n_taps) * btile);
  int stages = int((budget - p.w_resident_bytes) / p.stage_bytes);
  if (stages > 8) stages = 8;
  if (stages < 2) { set_error("conv_gemm: shared memory too small for 2 stages (stage %u B)", p.stage_bytes); return -10; }
  p.n_stages = stages;
  const size_t smem_bytes = 1024 + p.w_resident_bytes + size_t(stages) * p.stage_bytes + fixed_bytes;

  for (int v = 0; v < a.n_views; ++v) {
    const InView& iv = a.views[v];
    uint64_t dims[4] = {uint64_t(iv.channels), uint64_t(a.in_W), uint64_t(a.in_H), uint64_t(a.N)};
    uint64_t strides[3] = {uint64_t(iv.stride_w) * 2, uint64_t(iv.stride_h) * 2, uint64_t(iv.stride_n) * 2};
    uint32_t box[4] = {64, uint32_t(a.TW), uint32_t(a.strip_rows), 1};
    int rc = encode_map_bf16(&p.in_map[v], iv.ptr, 4, dims, strides, box);
    if (rc) return rc;
  }
  for (int v = a.n_views; v < kMaxInMaps; ++v) p.in_map[v] = p.in_map[0];
  {
    uint64_t dims[2] = {64, uint64_t(kb_total) * a.cout_total};
    uint64_t strides[1] = {128};
    uint32_t box[2] = {64, uint32_t(a.block_n)};
    int rc = encode_map_bf16(&p.w_map, a.weights, 2, dims, strides, box);
    if (rc) return rc;
  }
  if (a.out_mode == OUT_NHWC_F32) {
    for (int q = 0; q < 4; ++q) p.out_map[q] = p.in_map[0];
    p.aux_map = p.in_map[0];
  } else if (!fold) {
    uint32_t box[4] = {64, uint32_t(a.TW), uint32_t(a.TH), 1};
    if (a.out_mode == OUT_PIXEL_SHUFFLE) {
      // view q=(i,j) of the HR tensor [N,2H,2W,64]: pixel (2h+i, 2w+j)
      for (int q = 0; q < 4; ++q) {
        const int i = q >> 1, j = q & 1;
        const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(a.out) + (size_t(i) * 2 * a.W + j) * 64;
        uint64_t dims[4] = {64, uint64_t(a.W), uint64_t(a.H), uint64_t(a.N)};
        uint64_t strides[3] = {128 * 2, uint64_t(4) * a.W * 64 * 2, uint64_t(4) * a.H * a.W * 64 * 2};
        int rc = encode_map_bf16(&p.out_map[q], base, 4, dims, strides, box);
        if (rc) return rc;
      }
    } else {
      uint64_t dims[4] = {uint64_t(a.cout_total), uint64_t(a.W), uint64_t(a.H), uint64_t(a.N)};
      uint64_t strides[3] = {uint64_t(a.cout_total) * 2, uint64_t(a.W) * a.cout_total * 2,
                             uint64_t(a.H) * a.W * a.cout_total * 2};
      int rc = encode_map_bf16(&p.out_map[0], a.out, 4, dims, strides, box);
      if (rc) return rc;
      for (int q = 1; q < 4; ++q) p.out_map[q] = p.out_map[0];
      if (has_aux) {
        rc = encode_map_bf16(&p.aux_map, a.residual ? a.residual : a.mask_src, 4, dims, strides, box);
        if (rc) return rc;
      }
    }
    if (!has_aux) p.aux_map = p.out_map[0];
  } else {
    for (int q = 0; q < 4; ++q) p.out_map[q] = p.in_map[0];
    p.aux_map = p.in_map[0];
  }
  p.bias = a.bias; p.scale = a.scale; p.act = a.act; p.slope = a.slope;
  p.pol_in = kL2EvictNormal;
  p.out = a.out; p.out_mode = a.out_mode;
  p.stats = a.stats;
  p.prof = reinterpret_cast<long long*>(a.prof);

  const dim3 grid(p.ctas_per_block * p.n_blocks);
  if (fold) {
    if (a.n_taps != 9) { set_error("conv_gemm: fold9 needs 9 row taps"); return -14; }
    ConvKParamsFold pf;
    memset(&pf, 0, sizeof(pf));
    static_cast<ConvKParams&>(pf) = p;
    pf.scatter = a.scatter != nullptr ? *a.scatter : fold9_nchw(a.H, a.W);
    return launch_instance<32, 9>(pf, grid, smem_bytes, stream);
  }
  switch (a.n_taps) {
    case 1: return launch_instance<64, 1>(p, grid, smem_bytes, stream);
    case 2: return launch_instance<64, 2>(p, grid, smem_bytes, stream);
    case 3: return launch_instance<64, 3>(p, grid, smem_bytes, stream);
    case 4: return launch_instance<64, 4>(p, grid, smem_bytes, stream);
    case 5: return launch_instance<64, 5>(p, grid, smem_bytes, stream);
    default: set_error("conv_gemm: unsupported tap count %d", a.n_taps); return -15;
  }
}

}  // namespace srg
