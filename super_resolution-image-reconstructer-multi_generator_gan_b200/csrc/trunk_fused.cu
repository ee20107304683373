// Persistent multi-layer trunk kernel ("trunk_fused"): the 2*n_res + 1 same-shape 3x3 / 64->64 convolutions of the
// generator's residual trunk (reference: src/models.py:10-25, :62-66, :82-84) run inside ONE cooperative launch per
// direction -- for up to 4 independent generators at once -- with training-mode BatchNorm fused between the layers.
//
// Why.  Per layer the cfg2 trunk is 10.9 GFLOP = ~8 us of tensor-pipe time, but as separate launches it cost a conv
// launch (ramp, 72 KB filter load, TMEM allocation, epilogue drain: 12-20 us) plus a statistics finalize launch plus a
// full HBM-bound BatchNorm-apply pass (forward) or a reduction pass + finalize + apply pass (backward).  BatchNorm needs
// the statistics of the WHOLE batch before any output element can be normalised, so inside one generator the chain
//   MMAs of layer l -> statistics -> grid-wide reduction -> apply -> halo exchange -> MMAs of layer l+1
// is strictly serial and its latency (measured: ~15 us on 148 SMs) cannot be hidden by that generator's own work.  The
// multi-generator GAN trains K independent generators on the same batch, so the kernel walks "slots" (layer l,
// generator g) in the order (0,0) (0,1) .. (0,K-1) (1,0) ..: while generator g waits for its statistics, the tensor pipe
// runs layer l of generator g+1.  With K = 1 the same kernel degenerates to the serial chain (still no launches and no
// separate BatchNorm passes).
//
// Per slot, per CTA (tile t of CTA c = c + t * grid, 32 rows x 8 pixels each):
//   MMA phase   conv3_il's schedule (row-interleaved accumulator blocks, two taps per N = 128 MMA, one 10-pixel-wide
//               half strip per row parity feeding all three column shifts) into a ring of 4 TMEM accumulators;
//   pass 1      (16 epilogue warps, overlapped with the MMAs of the next tile) v = bf16(acc [+ bias] [+ addend] [masked]),
//               staged in shared memory, TMA-stored as the layer's raw output (forward: the saved conv output y;
//               backward: the BatchNorm-output gradient), per-channel sums of v and v*v (forward) / v and v*y (backward)
//               from the staged tile; the CTA's partial sums go to global memory;
//   apply       (8 more warps, decoupled from the MMA / pass-1 pipeline) arrive on the generator's grid barrier; the LAST
//               CTA to arrive reduces the <= 148 partial rows in a fixed order (and, under data parallelism, exchanges the
//               128 sums with the peer GPUs through NVLink peer memory: SyncBatchNorm) and publishes them; every CTA then
//               computes the coefficients and transforms its own tiles from L2:
//                   out = relu(v * scale + shift) [+ block input]        (forward)
//                   out = A * v + B * y + C                              (backward, BatchNorm input gradient)
//               and publishes a per-tile release flag.
// The producer of a later slot polls the <= 9 flags of a tile's 3x3 neighbourhood before it loads the tile's strips; the
// next slot's filter is prefetched per column shift as soon as the last MMAs that read the old one have retired.
//
// Warp roles (896 threads, register budget re-balanced with setmaxnreg): warp 0 TMA producer (+ flag polling), warp 1
// MMA issuer, warps 2-3 store threads of the two epilogue groups, warps 4-11 epilogue group E (even image rows), warps
// 12-19 group O (odd rows), warps 20-27 apply.
// Every in-kernel wait is bounded in time and reports through *err instead of hanging the device.
#include "trunk_fused.cuh"

#include <stdlib.h>
#include <string.h>

#include "conv_gemm.cuh"
#include "launch.cuh"
#include "peer_sync.cuh"
#include "ptx.cuh"

namespace srg {

int encode_map_bf16(CUtensorMap* map, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box);

namespace {

constexpr int kTrThreads = 640;
constexpr int kTrEpi0 = 128;                    // first pass-1 thread
constexpr uint32_t kTrWBytes = 9 * 64 * 128;    // resident filter [kw 3][kh2 ; kh1 ; kh0][64][64] bf16
constexpr uint32_t kTrPitch = 10 * 128;         // 10-pixel-wide half strip row
constexpr uint32_t kTrStage = 22 * 1024;        // 17 x 1280 B rounded up to the 1024-byte swizzle period
constexpr uint32_t kTrTile = 128 * 128;         // one block (128 pixels x 64 bf16) staged for a TMA store
constexpr int kTrMaxLayers = 40;
constexpr uint32_t kTrTailBytes = 2 * 256 + 4 * 256 + 16 * 128 * 4 + 3 * 256 + 512 + kTrMaxLayers * 64;
static_assert(1024 + kTrWBytes + 2 * kTrStage + 6 * kTrTile + kTrTailBytes <= 227 * 1024, "backward instance exceeds the shared memory of an SM");
constexpr int kTraceBase = 148 * 18;            // role timers first, then the event trace [cta][slot 128][event 8]
constexpr int kTraceSlots = 128, kTraceEvents = 16;
constexpr int kProfWords = kTraceBase + 148 * kTraceSlots * kTraceEvents;

template <bool BWD> constexpr int tr_stages() { return BWD ? 2 : 3; }
template <bool BWD> constexpr size_t tr_smem_bytes() {
  return 1024 + kTrWBytes + size_t(tr_stages<BWD>()) * kTrStage + 4 * kTrTile + (BWD ? 2 * kTrTile : 0) + kTrTailBytes;
}

struct TrunkGenK {
  CUtensorMap ld_map[2];       // [row parity] 5-D {64, W, rows, N, buffer}, box {64, 10, 17, 1, 1}
  CUtensorMap st_map[2];       // [row parity] same tensor, box {64, 8, 16, 1, 1}
  CUtensorMap w_map;           // {64, weight rows}, box {64, 64}
  const uint8_t* act_base;
  const uint8_t* grad_base;
  const float* master;
  float* grads;
  float* bn_buffers;
  float* bncoef;
  float* gpart;
  unsigned int* sync;          // [0] grid barrier counter, [1] published sequence, [32 + tile] flags, then gsum
  unsigned int* err;
  double* gsum;                // [2][128] global sums published by the last CTA to arrive
  double* peers[8];            // SyncBatchNorm exchange buffers (world > 1)
  unsigned long long* peer_seq;
  int* peer_err;
};

struct TrunkKParams {
  TrunkGenK gen[kTrunkMaxGen];
  const TrunkLayer* layers;
  int n_layers, n_gen;
  int N, H, W, tiles_h, tiles_w, tiles_total;
  long long act_slot, grad_slot;
  double count;
  float eps, momentum;
  int update_running;
  float param_grad_scale;
  int world, rank;
  long long* prof;
};

__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3,
                                            int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_gpu(const unsigned int* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_u32(const unsigned int* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu_add(unsigned int* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t atom_add_acq_rel_gpu(unsigned int* p, uint32_t v) {
  uint32_t old;
  asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned int* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_acquire_cta_shared(const unsigned int* p) {
  uint32_t v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_cta_shared_add(unsigned int* p, uint32_t v) {
  asm volatile("red.release.cta.shared::cta.add.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
template <int N>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }

// Every wait in this kernel is bounded in TIME: a protocol bug or a lost peer sets *err (1: cross-CTA wait, 2: mbarrier,
// 4: peer GPU, 8: intra-CTA counter) and the waiter carries on with whatever data is there -- wrong numbers, reported by
// the host, never a hung GPU.  Once *err is set every later wait gives up after one probe, so the kernel drains quickly.
constexpr unsigned long long kWaitNs = 2000000000ull;
__device__ __forceinline__ unsigned long long gtimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void spin_ge(const unsigned int* p, uint32_t target, unsigned int* err) {
  if (ld_acquire_gpu(p) >= target) return;
  const unsigned long long t0 = gtimer_ns();
  int it = 0;
  while (ld_acquire_gpu(p) < target) {
    if ((++it & 63) == 0 && (ld_relaxed_u32(err) != 0u || gtimer_ns() - t0 > kWaitNs)) {
      atomicOr(err, 1u);
      return;
    }
    if (it > 32) __nanosleep(32);
  }
}
__device__ __forceinline__ void spin_shared_ge(const unsigned int* p, uint32_t target, unsigned int* err) {
  if (ld_acquire_cta_shared(p) >= target) return;
  const unsigned long long t0 = gtimer_ns();
  int it = 0;
  while (ld_acquire_cta_shared(p) < target) {
    if ((++it & 63) == 0 && (ld_relaxed_u32(err) != 0u || gtimer_ns() - t0 > kWaitNs)) {
      atomicOr(err, 8u);
      return;
    }
    __nanosleep(20);
  }
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, 0x989680;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_b(uint64_t* bar, uint32_t parity, unsigned int* err) {
  if (mbar_try_wait(bar, parity)) return;
  const unsigned long long t0 = gtimer_ns();
  int it = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++it & 15) == 0 && (ld_relaxed_u32(err) != 0u || gtimer_ns() - t0 > kWaitNs)) {
      atomicOr(err, 2u);
      return;
    }
  }
}

// 32 lanes x 16 columns of 32-bit words back into tensor memory (the mirror of tmem_ld16)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// asm volatile: the loads are PREFETCHES issued one tile ahead of their use; a plain __ldcg lets the compiler sink them
// next to the use to save registers, which puts the HBM latency back on the critical path
__device__ __forceinline__ uint4 ldg_cg_u4(const uint8_t* p) {
  uint4 v;
  asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void stg_u4(uint8_t* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }

struct TileCoord { int n, hh, w0; };
__device__ __forceinline__ TileCoord tile_coord(const TrunkKParams& p, int tile) {
  const int per = p.tiles_h * p.tiles_w;
  TileCoord c;
  c.n = tile / per;
  const int rem = tile - c.n * per;
  c.hh = (rem / p.tiles_w) * 16;       // tile origin in parity-view rows (h0 / 2)
  c.w0 = (rem % p.tiles_w) * 8;
  return c;
}

#define TR_EV(slot, ev)                                                                                             \
  do {                                                                                                              \
    if (p.prof != nullptr && (slot) < kTraceSlots)                                                                  \
      p.prof[kTraceBase + (size_t(cta) * kTraceSlots + (slot)) * kTraceEvents + (ev)] = clock64();                  \
  } while (0)

template <bool BWD>
__global__ void __launch_bounds__(kTrThreads, 1) trunk_kernel(const __grid_constant__ TrunkKParams p) {
  constexpr int kStages = BWD ? 2 : 3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __builtin_assume(__isShared(smem));
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  uint8_t* w_smem = smem;
  uint8_t* stages = w_smem + kTrWBytes;
  uint8_t* v_stage = stages + size_t(kStages) * kTrStage;                // [group 2][buffer 2][16 KB]
  uint8_t* y_stage = v_stage + 4 * kTrTile;                               // bwd: [group 2][16 KB]
  uint8_t* tail = y_stage + (BWD ? 2 * kTrTile : 0);
  float* s_bias = reinterpret_cast<float*>(tail);                         // [slot parity 2][64]   conv bias (fwd)
  float* s_mask = s_bias + 128;                                           // [slot parity 2][2][64] fwd scale / shift of the mask BatchNorm (bwd)
  float* s_stats = s_mask + 256;                                          // [16][128]
  float* s_coef = s_stats + 16 * 128;                                     // [3][64]  pass 2: scale, shift | A, B, C
  double* s_dred = reinterpret_cast<double*>(s_stats);                    // [4][128], aliases s_stats (dead once the partial row is out)
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_coef + 192);
  uint64_t* full = bars;                 // [kStages]
  uint64_t* empty = bars + 4;            // [kStages]
  uint64_t* wfull = bars + 8;            // [3]
  uint64_t* wfree = bars + 11;           // [3]
  uint64_t* tfull = bars + 14;           // [2]
  uint64_t* tempty = bars + 16;          // [2]
  uint64_t* staged = bars + 22;          // [group 2][buffer 2]
  uint64_t* freebuf = bars + 26;         // [group 2][buffer 2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 30);
  unsigned long long* seq_s = reinterpret_cast<unsigned long long*>(bars + 31);
  unsigned int* s_last = reinterpret_cast<unsigned int*>(bars + 32);
  int4* s_tile = reinterpret_cast<int4*>(bars + 34);                       // [4] {n, hh, w0, tile} of this CTA's tiles
  const uint8_t** s_base = reinterpret_cast<const uint8_t**>(bars + 42);   // [generator 4][2] activation / gradient region base
  TrunkLayer* s_layers = reinterpret_cast<TrunkLayer*>(bars + 64);         // [n_layers <= kTrMaxLayers] copy of the layer table
  static_assert(sizeof(TrunkLayer) == 64, "TrunkLayer is copied as 16 words");

  const int G = int(gridDim.x);
  const int cta = int(blockIdx.x);
  const int K = p.n_gen;
  const int n_slots = p.n_layers * K;
  int n_my = 0;
  for (int t = cta; t < p.tiles_total; t += G) ++n_my;                    // <= 4 (host-checked): one parked block per tile
  unsigned int* const err = p.gen[0].err;
  // pass 2 of a slot is interleaved, tile by tile, with pass 1 of the NEXT slot when that is another generator (K > 1);
  // with one generator the next slot consumes this slot's outputs, so pass 2 must complete first
  const bool interleave = K > 1;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 3; ++i) { mbar_init(&wfull[i], 1); mbar_init(&wfree[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 512); }
    for (int i = 0; i < 4; ++i) { mbar_init(&staged[i], 256); mbar_init(&freebuf[i], 1); }
    *s_last = 0u;
    {
      int ti = 0;
      for (int t = cta; t < p.tiles_total && ti < 4; t += G, ++ti) {
        const TileCoord c = tile_coord(p, t);
        s_tile[ti] = make_int4(c.n, c.hh, c.w0, t);
      }
    }
    fence_barrier_init();
    for (int g = 0; g < K; ++g) {
      tma_prefetch_desc(&p.gen[g].ld_map[0]);
      tma_prefetch_desc(&p.gen[g].ld_map[1]);
      tma_prefetch_desc(&p.gen[g].st_map[0]);
      tma_prefetch_desc(&p.gen[g].st_map[1]);
      tma_prefetch_desc(&p.gen[g].w_map);
    }
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  // hot, dynamically indexed launch constants go to shared memory once: the layer table and the region bases
  for (int i = threadIdx.x; i < p.n_layers * 16; i += kTrThreads)
    reinterpret_cast<int*>(s_layers)[i] = reinterpret_cast<const int*>(p.layers)[i];
  if (threadIdx.x < 2 * K) s_base[threadIdx.x] = (threadIdx.x & 1) ? p.gen[threadIdx.x >> 1].grad_base : p.gen[threadIdx.x >> 1].act_base;
  if (threadIdx.x >= kTrEpi0 && threadIdx.x < kTrEpi0 + 192) {
    // pass-1 coefficients of slot 0 (later slots: loaded one slot ahead)
    const int t = threadIdx.x - kTrEpi0;
    const TrunkLayer& L0 = p.layers[0];
    if (t < 64) {
      s_bias[t] = (!BWD && L0.bias_off >= 0) ? p.gen[0].master[L0.bias_off + t] : 0.f;
    } else if (BWD && L0.mask_bn >= 0) {
      s_mask[t - 64] = p.gen[0].bncoef[size_t(L0.mask_bn) * 256 + (t - 64)];      // scale [64] then shift [64]
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long t_start = clock64();

  if (warp == 0) {
    // =============================================================== TMA producer
    int stage = 0;
    uint32_t phase = 0;
    for (int slot = 0; slot < n_slots; ++slot) {
      const int j = slot / K, g = slot - j * K;
      const TrunkGenK& gp = p.gen[g];
      const int in_idx = s_layers[j].in_idx;
      const int w_row = s_layers[j].w_row;
      if (lane == 0) {
        // filter of this slot, one column shift at a time, as soon as the previous slot's last MMAs on that shift retired
        for (int s = 0; s < 3; ++s) {
          if (slot > 0) mbar_wait_b(&wfree[s], uint32_t(slot - 1) & 1u, err);
          mbar_expect_tx(&wfull[s], kTrWBytes / 3);
          for (int r = 0; r < 3; ++r)
            tma_load_2d(w_smem + size_t(s * 3 + (2 - r)) * 8192, &gp.w_map, &wfull[s], 0, w_row + (s * 3 + r) * 64);
        }
      }
      __syncwarp();
      unsigned int* g_flags = gp.sync + 32;
      int ti = 0;
      for (int tile = cta; tile < p.tiles_total; tile += G, ++ti) {
        const TileCoord c = tile_coord(p, tile);
        if (j > 0) {
          // inputs of this tile = pass-2 outputs of layer j-1 on the 3x3 tile neighbourhood (+2 per layer and tile)
          if (lane < 9) {
            const int th = c.hh / 16 + lane / 3 - 1, tw = c.w0 / 8 + lane % 3 - 1;
            if (th >= 0 && th < p.tiles_h && tw >= 0 && tw < p.tiles_w)
              spin_ge(g_flags + (c.n * p.tiles_h + th) * p.tiles_w + tw, uint32_t(2 * j), err);
          }
          __syncwarp();
        }
        if (ti == 0 && lane == 0) TR_EV(slot, 0);
        if (lane == 0) {
          fence_proxy_async_all();         // acquire (generic proxy) -> TMA reads (async proxy)
#pragma unroll
          for (int par = 1; par >= 0; --par) {   // odd image rows h0-1+2r first, then even rows h0+2r (r = 0..16)
            mbar_wait_b(&empty[stage], phase ^ 1, err);
            mbar_expect_tx(&full[stage], 17 * kTrPitch);
            tma_load_5d(stages + size_t(stage) * kTrStage, &gp.ld_map[par], &full[stage], 0, c.w0 - 1, c.hh - par, c.n, in_idx);
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    constexpr uint32_t idesc64 = make_idesc_bf16(128, 64, 0, 0);
    constexpr uint32_t idesc128 = make_idesc_bf16(128, 128, 0, 0);
    const uint64_t desc_hi = (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    const uint64_t adesc_hi = (uint64_t(kTrPitch >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
    const uint32_t w_lo = smem_u32(w_smem) >> 4;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t tcount = 0;                 // tiles issued so far: accumulator tcount & 1 (two 128-column accumulators)
    for (int slot = 0; slot < n_slots; ++slot) {
      for (int ti = 0; ti < n_my; ++ti, ++tcount) {
        const uint32_t r = tcount & 1u;
        mbar_wait_b(&tempty[r], ((tcount >> 1) & 1u) ^ 1u, err);
        tc_fence_after();
        const uint32_t d_e = tmem_base + r * 128u;
        const uint32_t d_o = d_e + 64;
        const bool last_tile = ti == n_my - 1;
#pragma unroll
        for (int par = 1; par >= 0; --par) {
          mbar_wait_b(&full[stage], phase, err);
          tc_fence_after();
          if (ti == 0 && par == 1 && lane == 0) TR_EV(slot, 1);
          const uint32_t a_base = smem_u32(stages) + uint32_t(stage) * kTrStage;
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            if (ti == 0 && par == 1) mbar_wait_b(&wfull[s], uint32_t(slot) & 1u, err);
            if (elect_one()) {
              const uint32_t wb = w_lo + uint32_t(s) * (3 * 8192 >> 4);
              const uint32_t st0 = a_base + uint32_t(s) * 128u, st1 = st0 + kTrPitch;
              const uint64_t a0 = adesc_hi | uint64_t((st0 & 0x3FFFFu) >> 4);
              const uint64_t a1 = adesc_hi | uint64_t((st1 & 0x3FFFFu) >> 4);
              if (par == 1) {
                const uint64_t b1 = desc_hi | uint64_t(wb);                         // rho = 1: E += kh2, O += kh1
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_bf16(d_e, a1 + uint64_t(2 * k), b1 + uint64_t(2 * k), idesc128, (s > 0 || k > 0) ? 1u : 0u);
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
                if (last_tile) umma_commit(&wfree[s]);    // this column shift's filter is dead: the next slot's may land
              }
              if (s == 2) umma_commit(&empty[stage]);
            }
            __syncwarp();
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit(&tfull[r]);
        __syncwarp();
        if (last_tile && lane == 0) TR_EV(slot, 2);
      }
    }
  } else if (warp < 4) {
    // ================================================================= store threads (one per epilogue group)
    // They replay the epilogue's job sequence: a job = one staged block -> one TMA store; pass-2 jobs additionally
    // publish the tile's flag once the store has COMPLETED (checked lazily, one job later, so nothing ever stalls).
    if (lane == 0) {
      const int blk = warp - 2;
      uint32_t jc = 0;                   // jobs so far: buffer jc & 1, its phase (jc >> 1) & 1
      // Nothing here blocks on a store that was issued less than two jobs ago: the staging buffer of job n-1 is handed
      // back after job n has been issued (wait_group.read 1), and the flag of a pass-2 job is published two jobs later
      // (wait_group 2), when its completion is no longer on anyone's critical path.
      unsigned int* pend_flag[2] = {nullptr, nullptr};   // flag of job jc-1 / jc-2 awaiting completion (index: job & 1)
      auto job = [&](int g, int idx, int ti, bool flag) {
        const int4 tc = s_tile[ti];
        TileCoord c; c.n = tc.x; c.hh = tc.y; c.w0 = tc.z;
        const int tile = tc.w;
        const uint32_t b = jc & 1u;
        mbar_wait_b(&staged[blk * 2 + b], (jc >> 1) & 1u, err);
        tma_store_5d(&p.gen[g].st_map[blk], v_stage + size_t(blk * 2 + b) * kTrTile, 0, c.w0, c.hh, c.n, idx);
        tma_store_commit();
        if (jc >= 1) {
          tma_store_wait_read<1>();          // job jc-1 has been read out of shared memory
          mbar_arrive(&freebuf[blk * 2 + (b ^ 1u)]);
        }
        if (pend_flag[b] != nullptr) {       // job jc-2 (same parity)
          tma_store_wait_all<2>();
          fence_proxy_async_all();
          red_release_gpu_add(pend_flag[b], 1u);
        }
        pend_flag[b] = flag ? p.gen[g].sync + 32 + tile : nullptr;
        ++jc;
      };
      // drain: every issued store complete, every pending flag published
      auto flush = [&]() {
        tma_store_wait_all<0>();
        fence_proxy_async_all();
        for (int i = 0; i < 2; ++i)
          if (pend_flag[i] != nullptr) { red_release_gpu_add(pend_flag[i], 1u); pend_flag[i] = nullptr; }
      };
      for (int slot = 0; slot < n_slots; ++slot) {
        const int j = slot / K, g = slot - j * K;
        const int st1 = s_layers[j].st1_idx;
        const int pslot = slot - 1;
        const int pj = pslot >= 0 ? pslot / K : 0, pg = pslot >= 0 ? pslot - pj * K : 0;
        const int pst2 = (interleave && pslot >= 0) ? s_layers[pj].st2_idx : -1;
        // no pass-2 job of the previous slot to interleave (it had no BatchNorm: the last layer of a direction): the flags
        // still pending would otherwise wait for this slot's own pass-1 jobs, whose MMAs may need them (K = 2: the last
        // generator's last layer reads the tiles of the pass-2 job issued one slot earlier)
        if (interleave && pst2 < 0) flush();
        for (int ti = 0; ti < n_my; ++ti) {
          if (pst2 >= 0) job(pg, pst2, ti, true);
          if (st1 >= 0) job(g, st1, ti, false);
        }
        if (!interleave && s_layers[j].st2_idx >= 0) {
          for (int ti = 0; ti < n_my; ++ti) job(g, s_layers[j].st2_idx, ti, true);
          flush();                           // one generator: the next slot needs these tiles now
        }
      }
      flush();
    }
  } else {
    // =================================================================== epilogue: two 8-warp groups
    const int ew = warp - 4;
    const int blk = ew >> 3;                   // 0: even image rows (block E), 1: odd rows (block O)
    const int gw = ew & 7;
    const int q = warp & 3;                    // TMEM lane quadrant this warp may access
    const int m = q * 32 + lane;               // GEMM row: lane group m >> 3 is image row h0 + 2 * (m >> 3) + blk
    const int hf = gw >> 2;                    // which 32-channel half of the block
    const int gtid = gw * 32 + lane;           // 0..255 inside the group
    const int etid = ew * 32 + lane;           // 0..511
    const int bar_a = 1 + 2 * blk, bar_b = 2 + 2 * blk;
    uint8_t* vb0 = v_stage + size_t(blk * 2) * kTrTile;
    uint8_t* yb = y_stage + size_t(blk) * kTrTile;
    uint64_t* my_staged = staged + blk * 2;
    uint64_t* my_free = freebuf + blk * 2;
    const uint32_t row_off = uint32_t(m) * 128u;
    const uint32_t sw = uint32_t(m & 7);
    const int cq = gtid & 7, rp4 = gtid >> 3;     // column-sum mapping: 8-channel chunk cq, staged rows rp4*4 .. +3
    const uint32_t lane_addr = tmem_base + (uint32_t(q * 32) << 16);
    const uint32_t park_col = 256u + uint32_t(blk * 32 + hf * 16);   // + 64 * tile index: 16 packed columns of this thread
    uint32_t tcount = 0;                         // accumulators consumed (MMA ring)
    uint32_t jc = 0;                             // store jobs issued (staging ring)

    // ---- pass 2 of one tile of slot (pj, pg): parked v -> out, staged for the store thread.  `xx` = this thread's 64
    // bytes of the second operand (forward: the block input added after BatchNorm; backward: the saved conv output y),
    // prefetched one tile ahead by load_x() so that its HBM latency never sits in front of the tensor-memory read.
    auto load_x = [&](int pj, int pg, int ti, uint4 (&xx)[4]) {
      const TrunkLayer& PL = s_layers[pj];
      const int4 tc = s_tile[ti];
      const int hr = 2 * (tc.y + (m >> 3)) + blk, wc = tc.z + (m & 7);
      const bool valid = hr < p.H && wc < p.W;
      const uint8_t* act = s_base[2 * pg];
      const uint8_t* xb = BWD ? act + size_t(PL.y_idx) * size_t(p.act_slot)
                              : (PL.aux2_idx >= 0 ? act + size_t(PL.aux2_idx) * size_t(p.act_slot) : nullptr);
      const size_t pix_off = ((size_t(tc.x) * p.H + hr) * p.W + wc) * 128 + size_t(hf) * 64;
#pragma unroll
      for (int i = 0; i < 4; ++i) xx[i] = (xb != nullptr && valid) ? ldg_cg_u4(xb + pix_off + i * 16) : make_uint4(0, 0, 0, 0);
    };
    auto pass2_tile = [&](int pj, int ti, const uint4 (&xx)[4]) {
      const TrunkLayer& PL = s_layers[pj];
      uint32_t pv[16];
      tmem_ld16(lane_addr + park_col + uint32_t(ti * 64), pv);
      tmem_ld_wait();
      const uint32_t b = jc & 1u;
      uint8_t* ob = vb0 + size_t(b) * kTrTile + row_off;
      if (jc >= 2) mbar_wait_b(&my_free[b], ((jc >> 1) - 1u) & 1u, err);
      ++jc;
      const bool relu = !BWD && PL.relu != 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {            // 8 channels per 16-byte chunk
        const uint32_t xw[4] = {xx[i].x, xx[i].y, xx[i].z, xx[i].w};
        const float4* kq = reinterpret_cast<const float4*>(s_coef + hf * 32 + i * 8);
        const float4 ka0 = kq[0], ka1 = kq[1], kb0 = kq[16], kb1 = kq[17];
        const float ka[8] = {ka0.x, ka0.y, ka0.z, ka0.w, ka1.x, ka1.y, ka1.z, ka1.w};
        const float kb[8] = {kb0.x, kb0.y, kb0.z, kb0.w, kb1.x, kb1.y, kb1.z, kb1.w};
        float kc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (BWD) {
          const float4 kc0 = kq[32], kc1 = kq[33];
          kc[0] = kc0.x; kc[1] = kc0.y; kc[2] = kc0.z; kc[3] = kc0.w; kc[4] = kc1.x; kc[5] = kc1.y; kc[6] = kc1.z; kc[7] = kc1.w;
        }
        uint32_t ow[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float v0 = bf16_lo(pv[i * 4 + e]), v1 = bf16_hi(pv[i * 4 + e]);
          const float x0 = bf16_lo(xw[e]), x1 = bf16_hi(xw[e]);
          float o0, o1;
          if (!BWD) {
            o0 = fmaf(v0, ka[2 * e], kb[2 * e]);
            o1 = fmaf(v1, ka[2 * e + 1], kb[2 * e + 1]);
            if (relu) { o0 = fmaxf(o0, 0.f); o1 = fmaxf(o1, 0.f); }
            o0 += x0; o1 += x1;                // x = 0 when the layer has no skip addend
          } else {
            o0 = fmaf(ka[2 * e], v0, fmaf(kb[2 * e], x0, kc[2 * e]));
            o1 = fmaf(ka[2 * e + 1], v1, fmaf(kb[2 * e + 1], x1, kc[2 * e + 1]));
          }
          ow[e] = pack_bf16(o0, o1);
        }
        *reinterpret_cast<uint4*>(ob + ((uint32_t(hf * 4 + i) ^ sw) << 4)) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
      }
      fence_proxy_async_smem();
      mbar_arrive(&my_staged[b]);
    };

    // ---- statistics of slot (pj, pg) are complete on every CTA: coefficients into shared memory
    auto finish_barrier = [&](int pslot, int pj, int pg) {
      const TrunkLayer& PL = s_layers[pj];
      const TrunkGenK& pp = p.gen[pg];
      const uint32_t seq = uint32_t(pj);
      double* gs = pp.gsum + size_t(seq & 1u) * 128;
      if (etid == 0) {
        spin_ge(pp.sync + 1, seq + 1u, err);
        TR_EV(pslot, 6);
      }
      named_bar_sync(5, 512);
      if (etid < 64) {
        const int ch = etid;
        const double s1 = __ldcg(gs + ch), s2 = __ldcg(gs + 64 + ch);
        float* coef = pp.bncoef + size_t(PL.bn) * 256;
        if (!BWD) {
          const double mean = s1 / p.count;
          double var = s2 / p.count - mean * mean;
          if (var < 0.0) var = 0.0;
          const float inv = float(1.0 / sqrt(var + double(p.eps)));
          const float sc = pp.master[PL.gamma_off + ch] * inv;
          const float sh = pp.master[PL.beta_off + ch] - float(mean) * sc;
          s_coef[ch] = sc;
          s_coef[64 + ch] = sh;
          if (cta == 0) {
            coef[ch] = sc; coef[64 + ch] = sh; coef[128 + ch] = float(mean); coef[192 + ch] = inv;
            if (p.update_running) {
              float* rm = pp.bn_buffers + PL.rm_off;
              const double unbiased = p.count > 1.0 ? var * (p.count / (p.count - 1.0)) : var;
              rm[ch] = (1.f - p.momentum) * rm[ch] + p.momentum * float(mean);
              rm[64 + ch] = (1.f - p.momentum) * rm[64 + ch] + p.momentum * float(unbiased);
            }
          }
        } else {
          const double mean = coef[128 + ch], inv = coef[192 + ch];
          const double dg = inv * (s2 - mean * s1);
          const double db = s1;
          const double sc = double(pp.master[PL.gamma_off + ch]) * inv;
          s_coef[ch] = float(sc);
          s_coef[64 + ch] = float(-sc * inv * dg / p.count);
          s_coef[128 + ch] = float(-sc * db / p.count + sc * inv * mean * dg / p.count);
          if (cta == 0 && pp.grads != nullptr) {     // null: input-gradient-only backward
            pp.grads[PL.gamma_off + ch] = float(dg) * p.param_grad_scale;
            pp.grads[PL.beta_off + ch] = float(db) * p.param_grad_scale;
          }
        }
      }
      named_bar_sync(5, 512);
      if (etid == 0) TR_EV(pslot, 7);
    };

    for (int slot = 0; slot < n_slots; ++slot) {
      const int j = slot / K, g = slot - j * K;
      const TrunkGenK& gp = p.gen[g];
      const TrunkLayer L = s_layers[j];
      const bool has_bn = L.bn >= 0;
      const uint8_t* aux1_base = L.aux1_idx >= 0 ? (BWD ? s_base[2 * g + 1] + size_t(L.aux1_idx) * size_t(p.grad_slot)
                                                        : s_base[2 * g] + size_t(L.aux1_idx) * size_t(p.act_slot))
                                                 : nullptr;
      const uint8_t* y_base = (BWD && L.y_idx >= 0) ? s_base[2 * g] + size_t(L.y_idx) * size_t(p.act_slot) : nullptr;
      const bool masked = BWD && L.mask_bn >= 0;
      const float* bias_s = s_bias + (slot & 1) * 64;
      const float* mask_s = s_mask + (slot & 1) * 128;
      float st_s[8], st_q[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) { st_s[e] = 0.f; st_q[e] = 0.f; }
      // previous slot (another generator when interleaving): its pass 2 runs here, one tile ahead of our pass 1
      const int pslot = slot - 1;
      const int pj = pslot >= 0 ? pslot / K : 0, pg = pslot >= 0 ? pslot - pj * K : 0;
      const bool prev_p2 = interleave && pslot >= 0 && s_layers[pj].bn >= 0;
      uint4 xq[4];
      if (prev_p2) {
        load_x(pj, pg, 0, xq);                 // in flight while we wait for the statistics
        finish_barrier(pslot, pj, pg);
      }

      for (int ti = 0; ti < n_my; ++ti, ++tcount) {
        const bool trt = etid == 0 && ti == 1;
        if (trt) TR_EV(slot, 8);
        if (prev_p2) {
          pass2_tile(pj, ti, xq);
          if (ti + 1 < n_my) load_x(pj, pg, ti + 1, xq);   // lands during this tile's pass 1
        }
        if (trt) TR_EV(slot, 9);
        TileCoord c;
        { const int4 tc = s_tile[ti]; c.n = tc.x; c.hh = tc.y; c.w0 = tc.z; }
        const int hr = 2 * (c.hh + (m >> 3)) + blk, wc = c.w0 + (m & 7);
        const bool valid = hr < p.H && wc < p.W;
        const size_t pix_off = ((size_t(c.n) * p.H + hr) * p.W + wc) * 128 + size_t(hf) * 64;
        const uint32_t r = tcount & 1u;
        const uint32_t b = jc & 1u;
        uint8_t* vb = vb0 + size_t(b) * kTrTile;
        uint8_t* yp = yb + row_off;
        named_bar_sync(bar_a, 256);            // the group has finished reading the previous tile's staged values
        if (BWD && y_base != nullptr) {
          // saved conv output y of this thread's pixel: global -> shared (same swizzled layout as the staged block); it is
          // the ReLU mask source and the second factor of the product sums
          uint4 yy[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) yy[i] = valid ? ldg_cg_u4(y_base + pix_off + i * 16) : make_uint4(0, 0, 0, 0);
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(yp + ((uint32_t(hf * 4 + i) ^ sw) << 4)) = yy[i];
        }
        uint4 a1[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a1[i] = make_uint4(0, 0, 0, 0);
        if (aux1_base != nullptr && valid) {
#pragma unroll
          for (int i = 0; i < 4; ++i) a1[i] = ldg_cg_u4(aux1_base + pix_off + i * 16);
        }
        if (trt) TR_EV(slot, 10);
        mbar_wait_b(&tfull[r], (tcount >> 1) & 1u, err);
        tc_fence_after();
        if (trt) TR_EV(slot, 11);
        if (jc >= 2) mbar_wait_b(&my_free[b], ((jc >> 1) - 1u) & 1u, err);   // the store of job jc-2 has read the buffer
        ++jc;
        if (trt) TR_EV(slot, 12);
        const uint32_t t_addr = lane_addr + r * 128u + uint32_t(blk * 64 + hf * 32);
        uint32_t park[16];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t v[16];
          tmem_ld16(t_addr + uint32_t(h * 16), v);
          tmem_ld_wait();
          if (h == 1) {
            tc_fence_before();
            mbar_arrive(&tempty[r]);            // accumulator read out: the MMA issuer may start the tile after next
          }
          float f[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) f[e] = __uint_as_float(v[e]);
          if (!BWD) {
            const float4* bp = reinterpret_cast<const float4*>(bias_s + hf * 32 + h * 16);
#pragma unroll
            for (int gq = 0; gq < 4; ++gq) {
              const float4 bq = bp[gq];
              f[4 * gq + 0] += bq.x; f[4 * gq + 1] += bq.y; f[4 * gq + 2] += bq.z; f[4 * gq + 3] += bq.w;
            }
          }
          if (aux1_base != nullptr) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const uint4 rr = a1[h * 2 + i];
              const uint32_t ws[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                f[i * 8 + 2 * e] += bf16_lo(ws[e]);
                f[i * 8 + 2 * e + 1] += bf16_hi(ws[e]);
              }
            }
          }
          if (masked) {
            const float* msc = mask_s + hf * 32 + h * 16;
            const float* msh = msc + 64;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const uint4 rr = *reinterpret_cast<const uint4*>(yp + ((uint32_t(hf * 4 + h * 2 + i) ^ sw) << 4));
              const uint32_t ws[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                if (!(fmaf(bf16_lo(ws[e]), msc[i * 8 + 2 * e], msh[i * 8 + 2 * e]) > 0.f)) f[i * 8 + 2 * e] = 0.f;
                if (!(fmaf(bf16_hi(ws[e]), msc[i * 8 + 2 * e + 1], msh[i * 8 + 2 * e + 1]) > 0.f)) f[i * 8 + 2 * e + 1] = 0.f;
              }
            }
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) park[h * 8 + e] = pack_bf16(f[2 * e], f[2 * e + 1]);
          uint8_t* op = vb + row_off;
          *reinterpret_cast<uint4*>(op + ((uint32_t(hf * 4 + h * 2) ^ sw) << 4)) =
              make_uint4(park[h * 8 + 0], park[h * 8 + 1], park[h * 8 + 2], park[h * 8 + 3]);
          *reinterpret_cast<uint4*>(op + ((uint32_t(hf * 4 + h * 2 + 1) ^ sw) << 4)) =
              make_uint4(park[h * 8 + 4], park[h * 8 + 5], park[h * 8 + 6], park[h * 8 + 7]);
        }
        if (has_bn) {
          // park the rounded values (two bf16 per 32-bit column) until the batch statistics are known
          tmem_st16(lane_addr + park_col + uint32_t(ti * 64), park);
          tmem_st_wait();
        }
        if (trt) TR_EV(slot, 13);
        fence_proxy_async_smem();
        mbar_arrive(&my_staged[b]);
        named_bar_sync(bar_b, 256);
        if (trt) TR_EV(slot, 14);
        if (has_bn) {
          // column sums over the staged block: sum v, and sum v*v (forward) or sum v*y (backward).  Thread = (8-channel
          // chunk cq, 4 consecutive staged rows): 128-bit shared loads, 16 running sums per thread.
          const int mm0 = rp4 * 4;
          const bool row_ok = 2 * (c.hh + (mm0 >> 3)) + blk < p.H;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int mm = mm0 + i;
            const uint32_t so = uint32_t(mm) * 128u + ((uint32_t(cq) ^ uint32_t(mm & 7)) << 4);
            uint4 a = *reinterpret_cast<const uint4*>(vb + so);
            if (!(row_ok && c.w0 + (mm & 7) < p.W)) a = make_uint4(0, 0, 0, 0);
            const uint32_t aw[4] = {a.x, a.y, a.z, a.w};
            uint32_t bw[4] = {a.x, a.y, a.z, a.w};
            if (BWD) {
              const uint4 bq = *reinterpret_cast<const uint4*>(yb + so);
              bw[0] = bq.x; bw[1] = bq.y; bw[2] = bq.z; bw[3] = bq.w;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float x0 = bf16_lo(aw[e]), x1 = bf16_hi(aw[e]);
              st_s[2 * e] += x0; st_s[2 * e + 1] += x1;
              st_q[2 * e] = fmaf(x0, bf16_lo(bw[e]), st_q[2 * e]);
              st_q[2 * e + 1] = fmaf(x1, bf16_hi(bw[e]), st_q[2 * e + 1]);
            }
          }
        }
        if (trt) TR_EV(slot, 15);
      }
      if (etid == 0) TR_EV(slot, 4);

      // ---------------------------------------------------- end of slot: partial sums out, next slot's coefficients in
      if (has_bn) {
        // lanes of a warp = 4 row groups x 8 chunks: fold the row groups, then one row of s_stats per warp
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          st_s[e] += __shfl_xor_sync(0xffffffffu, st_s[e], 8);
          st_q[e] += __shfl_xor_sync(0xffffffffu, st_q[e], 8);
          st_s[e] += __shfl_xor_sync(0xffffffffu, st_s[e], 16);
          st_q[e] += __shfl_xor_sync(0xffffffffu, st_q[e], 16);
        }
        if (lane < 8) {
          float* row = s_stats + (blk * 8 + gw) * 128;
#pragma unroll
          for (int e = 0; e < 8; ++e) { row[lane * 8 + e] = st_s[e]; row[64 + lane * 8 + e] = st_q[e]; }
        }
      }
      if (slot + 1 < n_slots && etid >= 256 && etid < 448) {
        const int t = etid - 256;
        const int j1 = (slot + 1) / K, g1 = (slot + 1) - j1 * K;
        const TrunkLayer& L1 = s_layers[j1];
        if (t < 64) {
          if (!BWD) s_bias[((slot + 1) & 1) * 64 + t] = L1.bias_off >= 0 ? p.gen[g1].master[L1.bias_off + t] : 0.f;
        } else if (BWD && L1.mask_bn >= 0) {
          s_mask[((slot + 1) & 1) * 128 + (t - 64)] = p.gen[g1].bncoef[size_t(L1.mask_bn) * 256 + (t - 64)];
        }
      }
      named_bar_sync(5, 512);
      if (!has_bn) continue;

      // ---- this generator's grid barrier: partial sums out, arrive; the LAST CTA to arrive reduces and publishes
      const uint32_t seq = uint32_t(j);           // BatchNorm layers of a chain are j = 0 .. n_layers-2
      float* gpart = gp.gpart + size_t(seq & 1u) * size_t(G) * 128;
      double* gs = gp.gsum + size_t(seq & 1u) * 128;
      if (etid < 128) {
        float t = 0.f;
#pragma unroll
        for (int gq = 0; gq < 16; ++gq) t += s_stats[gq * 128 + etid];
        gpart[size_t(cta) * 128 + etid] = t;
        __threadfence();
      }
      named_bar_sync(5, 512);
      if (etid == 0) {
        const uint32_t old = atom_add_acq_rel_gpu(gp.sync, 1u);
        *s_last = (old == (seq + 1u) * uint32_t(G) - 1u) ? 1u : 0u;
        TR_EV(slot, 5);
      }
      named_bar_sync(5, 512);
      if (*s_last != 0u) {
        // fixed-order reduction of the G partial rows: 4 row lanes x 128 columns, <= 37 loads per thread all in flight
        const int col = etid & 127, rp = etid >> 7;
        float pv[37];
#pragma unroll
        for (int i = 0; i < 37; ++i) {
          const int r = rp + 4 * i;
          pv[i] = r < G ? __ldcg(gpart + size_t(r) * 128 + col) : 0.f;
        }
        double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
        for (int i = 0; i < 36; i += 2) { acc0 += double(pv[i]); acc1 += double(pv[i + 1]); }
        acc0 += double(pv[36]);
        s_dred[rp * 128 + col] = acc0 + acc1;
        named_bar_sync(5, 512);
        if (p.world > 1) {
          // SyncBatchNorm: exchange the 128 local sums with every peer GPU through NVLink peer memory (protocol and
          // buffers of peer_finalize_kernel), rank-ordered total
          if (etid == 0) *seq_s = ++(*gp.peer_seq);
          named_bar_sync(5, 512);
          const unsigned long long pseq = *seq_s;
          const int ps = int(pseq % 4ull);
          constexpr int kSlotDoubles = 136;
          if (etid < 128) {
            const double t = (s_dred[col] + s_dred[128 + col]) + (s_dred[256 + col] + s_dred[384 + col]);
            for (int r = 0; r < p.world; ++r) gp.peers[r][(size_t(ps) * p.world + p.rank) * kSlotDoubles + col] = t;
            __threadfence_system();
          }
          named_bar_sync(5, 512);
          if (etid < p.world) {
            const int r = etid;
            st_release_sys_u64(reinterpret_cast<unsigned long long*>(gp.peers[r] + (size_t(ps) * p.world + p.rank) * kSlotDoubles + 128), pseq);
            const unsigned long long* flag =
                reinterpret_cast<const unsigned long long*>(gp.peers[p.rank] + (size_t(ps) * p.world + r) * kSlotDoubles + 128);
            long long spins = 0;
            while (ld_acquire_sys_u64(flag) != pseq) {
              if (++spins > (1ll << 22)) { *gp.peer_err = 1; atomicOr(err, 4u); break; }
              __nanosleep(64);
            }
          }
          named_bar_sync(5, 512);
          if (etid < 128) {
            double t = 0.0;
            for (int r = 0; r < p.world; ++r) {
              const double* src = gp.peers[p.rank] + (size_t(ps) * p.world + r) * kSlotDoubles + col;
              double x;
              asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(x) : "l"(src) : "memory");
              t += x;
            }
            gs[col] = t;
            __threadfence();
          }
        } else if (etid < 128) {
          gs[col] = (s_dred[col] + s_dred[128 + col]) + (s_dred[256 + col] + s_dred[384 + col]);
          __threadfence();
        }
        named_bar_sync(5, 512);
        if (etid == 0) st_release_gpu_u32(gp.sync + 1, seq + 1u);
      }
      if (!interleave) {
        // one generator: the next slot consumes this slot's outputs, so pass 2 runs now (serial chain)
        uint4 xs[4];
        load_x(j, g, 0, xs);
        finish_barrier(slot, j, g);
        for (int t2 = 0; t2 < n_my; ++t2) {
          pass2_tile(j, t2, xs);
          if (t2 + 1 < n_my) load_x(j, g, t2 + 1, xs);
        }
      }
    }
  }

  if (p.prof != nullptr && threadIdx.x == 0) {
    long long* d = p.prof + size_t(blockIdx.x) * 18;
    d[4] = clock64() - t_start; d[5] = t_start;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

int g_trunk_fused = 2;              // 0: off, 1: on, 2: automatic (set_trunk_fused)
long long* g_trunk_prof = nullptr;     // SRG_TRUNK_PROF=1: role timers + event trace of the last launch (debug)

}  // namespace

bool trunk_fused_enabled() { return g_trunk_fused != 0; }
// Measured on B200 (profiles/r02_notes.md): with at most one tile per SM and layer the step is launch-latency bound and
// the fused kernel wins (8x3x64x64: 2.21 vs 2.69 ms per eager generator step); at the cfg2 geometry (4 tiles per SM)
// its serial statistics -> barrier -> apply chain per layer loses to the per-layer launches, whose gaps the K
// generators' graph branches fill (12.6 vs 11.0 ms per 3-generator step).  Automatic mode picks accordingly;
// srg_set_trunk_fused(1) forces the fused kernel wherever it applies.
bool trunk_fused_preferred(int N, int H, int W) {
  const int mode = g_trunk_fused;
  if (mode != 2) return mode == 1;
  const int grid = trunk_grid(N, H, W);
  return grid > 0 && N * ((H + 31) / 32) * ((W + 7) / 8) <= grid;
}
int set_trunk_fused(int on) {
  const int old = g_trunk_fused;
  g_trunk_fused = on < 0 || on > 2 ? 2 : on;
  return old;
}

int trunk_prof_read(long long* host, int n) {
  if (g_trunk_prof == nullptr) return 0;
  if (n > kProfWords) n = kProfWords;
  if (cudaMemcpy(host, g_trunk_prof, size_t(n) * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return n;
}

static int trunk_tiles(int N, int H, int W) { return N * ((H + 31) / 32) * ((W + 7) / 8); }

int trunk_grid(int N, int H, int W) {
  if (H < 2) return 0;
  const int tiles = trunk_tiles(N, H, W);
  if (tiles < 1) return 0;
  const int sms = sm_budget();
  const int grid = tiles < sms ? tiles : sms;
  if ((tiles + grid - 1) / grid > 4) return 0;   // one parked tensor-memory block per tile of a layer: <= 4 tiles per CTA
  return grid;
}
static size_t trunk_sync_words(int N, int H, int W) { return (size_t(32 + trunk_tiles(N, H, W)) + 63) & ~size_t(63); }
size_t trunk_sync_bytes(int N, int H, int W) { return trunk_sync_words(N, H, W) * 4 + 2 * 128 * 8; }

int launch_trunk(const TrunkArgs& a, cudaStream_t stream) {
  const int grid = trunk_grid(a.N, a.H, a.W);
  if (grid == 0) { set_error("trunk_fused: unsupported geometry (more than 4 tiles of 32x8 pixels per SM and layer)"); return -60; }
  if (a.n_gen < 1 || a.n_gen > kTrunkMaxGen) { set_error("trunk_fused: 1..%d generators per launch", kTrunkMaxGen); return -62; }
  if (a.n_layers < 1) return 0;
  if (a.n_layers > kTrMaxLayers) { set_error("trunk_fused: at most %d layers per chain", kTrMaxLayers); return -67; }
  static TrunkKParams p;            // ~3 KB: keep it off the stack of small host threads; launches are serialized per process
  memset(&p, 0, sizeof(p));
  p.layers = a.layers; p.n_layers = a.n_layers; p.n_gen = a.n_gen;
  p.N = a.N; p.H = a.H; p.W = a.W;
  p.tiles_h = (a.H + 31) / 32; p.tiles_w = (a.W + 7) / 8; p.tiles_total = trunk_tiles(a.N, a.H, a.W);
  p.act_slot = a.act_slot; p.grad_slot = a.grad_slot;
  p.count = a.count; p.eps = a.eps; p.momentum = a.momentum;
  p.update_running = a.update_running; p.param_grad_scale = a.param_grad_scale;
  p.world = 1; p.rank = 0;
  {
    static int prof_on = -1;
    // SRG_TRUNK_PROF=1: trace every launch (the last one wins), 2: forward launches only, 3: backward launches only
    if (prof_on < 0) { const char* ev = getenv("SRG_TRUNK_PROF"); prof_on = (ev != nullptr && ev[0] >= '1' && ev[0] <= '3') ? ev[0] - '0' : 0; }
    if (prof_on && g_trunk_prof == nullptr && cudaMalloc(&g_trunk_prof, size_t(kProfWords) * sizeof(long long)) != cudaSuccess) g_trunk_prof = nullptr;
    if (prof_on == 1 || (prof_on == 2 && !a.bwd) || (prof_on == 3 && a.bwd)) p.prof = g_trunk_prof;
  }
  const size_t sync_words = trunk_sync_words(a.N, a.H, a.W);
  for (int g = 0; g < a.n_gen; ++g) {
    const TrunkGen& src = a.gen[g];
    TrunkGenK& dst = p.gen[g];
    dst.act_base = reinterpret_cast<const uint8_t*>(src.act_base);
    dst.grad_base = reinterpret_cast<const uint8_t*>(src.grad_base);
    dst.master = src.master; dst.grads = src.grads; dst.bn_buffers = src.bn_buffers; dst.bncoef = src.bncoef;
    dst.gpart = src.gpart; dst.sync = src.sync; dst.err = src.err;
    dst.gsum = reinterpret_cast<double*>(src.sync + sync_words);
    if ((src.peer != nullptr) != (a.gen[0].peer != nullptr)) { set_error("trunk_fused: mixed SyncBatchNorm settings"); return -63; }
    if (src.peer != nullptr) {
      PeerDeviceView v;
      int rc = peer_sync_device_view(src.peer, &v);
      if (rc) return rc;
      for (int r = 0; r < 8; ++r) dst.peers[r] = v.peers[r];
      dst.peer_seq = v.seq; dst.peer_err = v.err;
      if (g > 0 && (v.world != p.world || v.rank != p.rank)) { set_error("trunk_fused: generators on different communicators"); return -64; }
      p.world = v.world; p.rank = v.rank;
    }
    // 5-D row-parity views of the region the direction loads from / stores to: {64 ch, W, rows of one parity, N, buffer}
    const uint8_t* base = a.bwd ? dst.grad_base : dst.act_base;
    const int64_t slot = a.bwd ? a.grad_slot : a.act_slot;
    const int buffers = a.bwd ? a.grad_buffers : a.act_buffers;
    for (int par = 0; par < 2; ++par) {
      const uint8_t* ptr = base + size_t(par) * a.W * 128;
      uint64_t dims[5] = {64, uint64_t(a.W), uint64_t((a.H - par + 1) / 2), uint64_t(a.N), uint64_t(buffers)};
      uint64_t strides[4] = {128, uint64_t(a.W) * 256, uint64_t(a.H) * a.W * 128, uint64_t(slot)};
      uint32_t box_ld[5] = {64, 10, 17, 1, 1};
      uint32_t box_st[5] = {64, 8, 16, 1, 1};
      int rc = encode_map_bf16(&dst.ld_map[par], ptr, 5, dims, strides, box_ld);
      if (rc) return rc;
      rc = encode_map_bf16(&dst.st_map[par], ptr, 5, dims, strides, box_st);
      if (rc) return rc;
    }
    uint64_t wdims[2] = {64, uint64_t(a.weight_rows)};
    uint64_t wstrides[1] = {128};
    uint32_t wbox[2] = {64, 64};
    int rc = encode_map_bf16(&dst.w_map, src.weights, 2, wdims, wstrides, wbox);
    if (rc) return rc;
    if (cudaMemsetAsync(src.sync, 0, sync_words * 4, stream) != cudaSuccess) { set_error("trunk_fused: memset failed"); return -61; }
  }
  const size_t smem_bytes = a.bwd ? tr_smem_bytes<true>() : tr_smem_bytes<false>();
  static DeviceOnce attr_set;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(trunk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(tr_smem_bytes<false>()));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(trunk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(tr_smem_bytes<true>()));
    if (e != cudaSuccess) { set_error("trunk_fused cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return int(e); }
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kTrThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;     // all CTAs co-resident: the in-kernel grid barriers cannot deadlock
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = a.bwd ? cudaLaunchKernelEx(&cfg, trunk_kernel<true>, p) : cudaLaunchKernelEx(&cfg, trunk_kernel<false>, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("trunk_fused launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

}  // namespace srg
