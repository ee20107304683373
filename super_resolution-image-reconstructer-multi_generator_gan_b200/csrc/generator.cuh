// SRResNet generator engine: owns the launch sequence of one forward / backward pass over caller-provided
// device memory (reference: src/models.py:10-25 ResidualBlock, :44-87 SRResNet).  Internal C++ interface; the
// C ABI wrappers live in api.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

namespace srg {

struct ParamInfo {
  std::string name;      // state_dict key
  int64_t offset;        // element offset into the flat fp32 parameter / gradient buffers
  int64_t numel;
  int ndim;
  int shape[4];
};
struct BufferInfo {      // BatchNorm running statistics (flat fp32 buffer)
  std::string name;
  int64_t offset;
  int64_t numel;
};
struct TensorInfo {      // named intermediate inside the workspace (for per-layer parity tests)
  std::string name;
  int64_t byte_offset;
  int dims[4];           // NHWC
  int dtype;             // 0 = bf16 NHWC, 1 = fp32 NCHW
};

// Collective hook for SyncBatchNorm: sum `n` doubles in place across ranks, stream ordered.
typedef int (*AllreduceF64Fn)(void* ctx, double* buf, int n, cudaStream_t stream);

struct GeneratorEngine {
  int N, H, W, n_res, n_up;
  std::vector<ParamInfo> params;
  std::vector<BufferInfo> buffers;
  std::vector<TensorInfo> tensors;
  int64_t param_elems = 0, buffer_elems = 0;
  int64_t packed_elems = 0, bias_elems = 0;
  size_t workspace_bytes_train = 0, workspace_bytes_eval = 0;
  // device-resident constant index maps (owned)
  int* d_pack_idx = nullptr;
  int* d_bias_idx = nullptr;
  int* d_wg_idx_c3x3 = nullptr;   // 64->64 3x3
  int* d_wg_idx_up = nullptr;     // 64->256 3x3 (pixel-shuffle order)
  int* d_wg_idx_conv1 = nullptr;  // 9x9 3->64
  int* d_wg_idx_conv3 = nullptr;  // 9x9 64->3
  long long* d_wgb_off = nullptr; // gradient-buffer offsets of the trunk conv weights, layer order 2*block + conv, conv2 last
  // bound memory
  float* master = nullptr;
  float* grads = nullptr;
  float* bn_buffers = nullptr;
  uint8_t* ws = nullptr;
  size_t ws_bytes = 0;
  bool ws_training = false;
  // SyncBN
  AllreduceF64Fn allreduce = nullptr;
  void* allreduce_ctx = nullptr;
  struct PeerSync* peer = nullptr;   // NVLink peer-memory exchange fused with the finalize (preferred over `allreduce`)
  int world = 1;
  long long launches = 0;  // kernels launched so far (bench bookkeeping)
  // optional CUDA-event timing of the dominant kernel class (3x3 64->64 fprop/dgrad conv_gemm launches)
  bool fuse_bwd_stats = false;  // BatchNorm-backward sums in the dgrad epilogue instead of a separate pass (SRG_FUSE_BWD_STATS=1: on)
  // single GPU: BatchNorm statistics finalize inside the apply / backward-apply pass (SRG_FIN_FUSED=1).  Measured on B200
  // (profiles/r02_notes.md): one generator alone 3.94 -> 3.84 ms per step, but three generators as parallel graph branches
  // 11.08 -> 11.4-11.7 ms (the fatter apply CTAs take bandwidth from the other branches' tensor-core kernels), so it is off
  // by default
  bool fin_fused = false;
  // single GPU, backward: the BatchNorm-backward reduction's last block finalizes the coefficients (SRG_REDUCE_FINAL=1).
  // Measured: 96 fewer launches per 3-generator step, step time unchanged (10.69 vs 10.69-10.72 ms), so the two-launch form stays
  bool reduce_final = false;
  bool wgrad_batched = true;    // trunk weight gradients in one batched launch at the end of backward (SRG_WGRAD_BATCHED=0: off)
  bool keep_grads = false; // debug: keep every inter-layer gradient in its own named buffer (parity tests)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_events;   // pairs (start, stop)
  size_t prof_used = 0;
  int prof_layers = 1;     // trunk conv layers covered by one profiled launch (1: per-layer launches, 2*n_res+1: fused trunk kernel)

  virtual ~GeneratorEngine();
};

GeneratorEngine* generator_create(int N, int H, int W, int n_res, int n_up);
int generator_bind(GeneratorEngine* g, float* master, float* grads, float* bn_buffers, void* ws, size_t ws_bytes,
                   int training);
int generator_pack(GeneratorEngine* g, cudaStream_t st);
int generator_forward(GeneratorEngine* g, const float* lr_nchw, float* sr_nchw, int training, int update_running,
                      cudaStream_t st);
int generator_backward(GeneratorEngine* g, const float* dsr_nchw, cudaStream_t st);
// eval-mode (running-statistics) BatchNorm on a training-bound workspace, keeping what the backward needs
int generator_forward_frozen(GeneratorEngine* g, const float* lr_nchw, float* sr_nchw, cudaStream_t st);
// backward of the last forward (training or frozen); param_grads == 0: no parameter gradient is computed or written;
// dlr_nchw (optional) receives d(loss)/d(lr), fp32 N x 3 x H x W
int generator_backward_ex(GeneratorEngine* g, const float* dsr_nchw, int param_grads, float* dlr_nchw, cudaStream_t st);
// spatially tiled eval forward (srg_generator_forward_tiles): same layout as srg_tile_t, LR pixels
struct TileDesc { int32_t frame, y0, x0, crop_y0, crop_x0, crop_h, crop_w; };
int generator_tile_halo(int n_res, int n_up);
int generator_forward_tiles(GeneratorEngine* g, const float* frames_nchw, int F, int H, int W, const TileDesc* tiles, int n,
                            float* sr_nchw, cudaStream_t st);
// 8-bit frame I/O of the eval forward (srg_generator_forward_u8 / _tiles_u8): uint8 NHWC in, quantised uint8 NHWC out
int generator_forward_u8(GeneratorEngine* g, const uint8_t* lr_nhwc, uint8_t* sr_nhwc, cudaStream_t st);
int generator_forward_tiles_u8(GeneratorEngine* g, const uint8_t* frames_nhwc, int F, int H, int W, const TileDesc* tiles,
                               int n, uint8_t* sr_nhwc, cudaStream_t st);
// eval-mode autograd over windows (srg_generator_forward_frozen_tiles / srg_generator_backward_tiles): the frozen forward of
// n windows on a training workspace (sr_nchw may be NULL: activations only), then the backward of those windows
int generator_forward_frozen_tiles(GeneratorEngine* g, const float* frames_nchw, int F, int H, int W, const TileDesc* tiles,
                                   int n, float* sr_nchw, cudaStream_t st);
int generator_backward_tiles(GeneratorEngine* g, const float* dsr_nchw, int param_grads, float* dlr_nchw, cudaStream_t st);
// Split execution for the multi-generator step: PRE = everything before the residual trunk, TRUNK = the trunk itself,
// POST = everything after it (forward: conv1 | blocks + conv2 | upsample + conv3; backward: conv3 + upsample stages |
// trunk dgrad chain | conv1 gradients + the batched trunk weight gradients).  The TRUNK phases of several engines of equal
// geometry run as ONE interleaved launch through generators_trunk() (csrc/trunk_fused.cu).
enum GeneratorPhase : int { kPhasePre = 1, kPhaseTrunk = 2, kPhasePost = 4, kPhaseAll = 7 };
int generator_forward_phases(GeneratorEngine* g, const float* lr_nchw, float* sr_nchw, int training, int update_running,
                             int phases, cudaStream_t st);
int generator_backward_phases(GeneratorEngine* g, const float* dsr_nchw, int phases, cudaStream_t st);
int generators_trunk(GeneratorEngine* const* gs, int n, int bwd, int update_running, cudaStream_t st);
// dominant-kernel timing: enable/disable; read() synchronises on the recorded events, returns the summed duration
// (ms) and launch count since the last read and resets.
int generator_set_keep_grads(GeneratorEngine* g, int keep);
// non-zero if a bounded in-kernel wait of the fused trunk kernel ever gave up (synchronises the device)
int generator_trunk_error(GeneratorEngine* g);
int generator_prof_layers(const GeneratorEngine* g);
int generator_profile_enable(GeneratorEngine* g, int on);
int generator_profile_read(GeneratorEngine* g, double* ms_sum, long long* count);

}  // namespace srg
