// Programmatic dependent launch (PDL) helpers.
//
// A kernel launched through launch_pdl() may be scheduled while its stream predecessor is still running (as soon as
// every block of the predecessor has executed pdl_trigger(), or exited).  It MUST call pdl_wait() before it touches
// memory the predecessor writes: pdl_wait() returns once the predecessor grid has completed and flushed.  Everything a
// kernel does before pdl_wait() (barrier init, TMEM allocation, tensor-map prefetch, loading weights that were packed
// long before) overlaps the predecessor's tail; inside a captured CUDA graph the attribute becomes a programmatic edge.
// Only kernels that contain pdl_wait() are ever launched with the attribute.
#pragma once
#include <cuda_runtime.h>

#include <stdlib.h>

#include <atomic>
#include <utility>

namespace srg {

__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// cudaFuncSetAttribute() applies to the CURRENT device only, so "done once" is remembered per device ordinal (one bit
// each) and not per process: a process that drives a second GPU sets the attribute there too.  Used as
//   static DeviceOnce attr_set;  if (!attr_set) { ...cudaFuncSetAttribute...;  attr_set = true; }
struct DeviceOnce {
  std::atomic<unsigned long long> mask{0};
  static unsigned long long bit() {
    int d = 0;
    cudaGetDevice(&d);
    return 1ull << (d & 63);
  }
  bool operator!() const { return (mask.load(std::memory_order_acquire) & bit()) == 0; }
  DeviceOnce& operator=(bool done) {
    if (done) mask.fetch_or(bit(), std::memory_order_release);
    return *this;
  }
};

// Only grids of at most 8 blocks (the single-block finalize kernels) and inference (`exclusive`) convolutions start early: a
// big grid parked at griddepcontrol.wait holds registers / shared memory that a ready kernel of another stream could use.
// Measured on the cfg2 training step (profiles/r02_ab_pdl_grouped.log): 9.61-9.64 ms vs 9.69-9.74 ms with every launch_pdl()
// kernel starting early.
// SRG_PDL=0 (read once) is a diagnostic: plain stream-order launches everywhere, so that a kernel timeline shows each
// kernel's own duration instead of one that starts while the predecessor is still running.
inline bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("SRG_PDL"); return e == nullptr || atoi(e) != 0; }();
  return on;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_with_pdl_attr(bool early, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                        Args&&... args) {
  cudaLaunchConfig_t cfg;
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = early ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  const bool early = pdl_enabled() && grid.x * grid.y * grid.z <= 8;
  return launch_with_pdl_attr(early, kernel, grid, block, smem, st, std::forward<Args>(args)...);
}
// inference launches: a chain of SM-exclusive convolutions on one stream with nothing else to schedule -- early start pays
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_exclusive(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  return launch_with_pdl_attr(pdl_enabled(), kernel, grid, block, smem, st, std::forward<Args>(args)...);
}

// Column sum of a [rows][128] fp32 partial-sum table for row lane rl of 8 (rows rl, rl+8, ...), fp64, FIXED order: four
// accumulators take rows b, b+8, b+16, b+24 of every group of 32 rows in turn.  Shared by the local finalize
// (elementwise.cu) and the peer-memory finalize (peer_sync.cu), which must agree bit for bit.  Up to 12 independent loads are
// in flight per thread (the additions keep the 4-per-group order): the one-block finalize kernels sit on the dependency chain
// between a convolution and the BatchNorm pass behind it, and with 4 loads per round 288 rows were 9 L2 round trips.
__device__ __forceinline__ double partials_lane_sum(const float* __restrict__ partials, int rows, int col, int rl) {
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  const float* p = partials + col;
  int b = rl;
  for (; b + 88 < rows; b += 96) {
    float v[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) v[k] = p[size_t(b + 8 * k) * 128];
#pragma unroll
    for (int k = 0; k < 12; k += 4) { a0 += double(v[k]); a1 += double(v[k + 1]); a2 += double(v[k + 2]); a3 += double(v[k + 3]); }
  }
  for (; b + 24 < rows; b += 32) {
    const float v0 = p[size_t(b) * 128], v1 = p[size_t(b + 8) * 128], v2 = p[size_t(b + 16) * 128], v3 = p[size_t(b + 24) * 128];
    a0 += double(v0); a1 += double(v1); a2 += double(v2); a3 += double(v3);
  }
  // at most three rows are left: load them together (a missing row adds +0.0)
  const float t0 = b < rows ? p[size_t(b) * 128] : 0.f;
  const float t1 = b + 8 < rows ? p[size_t(b + 8) * 128] : 0.f;
  const float t2 = b + 16 < rows ? p[size_t(b + 16) * 128] : 0.f;
  a0 += double(t0); a0 += double(t1); a0 += double(t2);
  return (a0 + a1) + (a2 + a3);
}

}  // namespace srg
