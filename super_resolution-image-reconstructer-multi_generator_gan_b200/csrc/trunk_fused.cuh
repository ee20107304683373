// Persistent multi-layer kernel for the residual trunk of the generator (reference: src/models.py:10-25 ResidualBlock,
// :62-66 / :82-84 the 16-block trunk + conv2): ALL 3x3 / 64->64 convolutions of one direction (33 fprops, or 33 dgrads)
// of up to 4 independent generators run inside ONE cooperative launch, with training-mode BatchNorm (statistics -> grid
// barrier -> apply) fused between them.  Internal C++ interface; see trunk_fused.cu for the design.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace srg {

struct PeerSync;

constexpr int kTrunkMaxGen = 4;

// One layer of the chain.  "Buffer index" i addresses the dense NHWC bf16 tensor at region_base + i * region_slot_bytes;
// the forward direction loads / stores through the ACTIVATION region, the backward direction through the GRADIENT
// region; plain (non-TMA) reads may come from either region as noted.
struct TrunkLayer {
  int in_idx;      // conv input (TMA loads)
  int st1_idx;     // pass-1 store target:  fwd: y = bf16(conv + bias (+ aux1))   bwd: v = bf16(dgrad (+ aux1) (masked))
  int st2_idx;     // apply store target or -1 (-1 <=> the layer has no BatchNorm step: pass 1 is the whole layer)
  int aux1_idx;    // pass-1 addend or -1 (fwd: activation region, bwd: gradient region)
  int aux2_idx;    // fwd apply addend after BatchNorm (the block's input), activation region, or -1
  int y_idx;       // bwd: saved conv output y of the BatchNorm this layer differentiates through (activation region): second
                   // factor of the product statistics, B*y term of the apply, and the ReLU mask source when mask_bn >= 0
  int mask_bn;     // bwd: >= 0: v = 0 where fma(y, scale, shift) <= 0 with the FORWARD coefficients of BatchNorm `mask_bn`
  int bn;          // BatchNorm index (2*block + k) whose statistics this layer produces / consumes, or -1
  int relu;        // fwd apply: ReLU after BatchNorm
  int w_row;       // first row of the layer's packed filter in the weight tensor map
  int bias_off;    // fwd: float offset of the conv bias in `master`, or -1
  int gamma_off;   // float offset of the BatchNorm weight in master (and of its gradient in grads)
  int beta_off;
  int rm_off;      // float offset of running_mean in bn_buffers (running_var = +64)
  int pad0, pad1;
};

// per-generator memory (every generator of a launch has the same geometry, layer table and region layout)
struct TrunkGen {
  const void* act_base;          // activation region (buffer 0), dense [N,H,W,64] bf16 tensors `act_slot` bytes apart
  void* grad_base;               // gradient region
  const void* weights;           // packed bf16 filters, rows of 64: layer filter = 576 consecutive rows from w_row
  const float* master;
  float* grads;                  // bwd: BatchNorm weight / bias gradients are written here
  float* bn_buffers;             // fwd: running statistics (update_running)
  float* bncoef;                 // [bn][256] = scale, shift, save_mean, save_inv (written by fwd, read by bwd)
  float* gpart;                  // [2][grid][128] per-CTA partial sums (device scratch)
  unsigned int* sync;            // device scratch: trunk_sync_bytes(), zeroed by the launcher
  unsigned int* err;             // device word, OR-ed with a code if an in-kernel wait timed out (never reset by the launcher)
  PeerSync* peer;                // optional cross-GPU statistics exchange (SyncBatchNorm), else nullptr
};

struct TrunkArgs {
  int bwd;                       // 0: forward chain, 1: backward (dgrad) chain
  int N, H, W;
  int n_layers;
  const TrunkLayer* layers;      // DEVICE array [n_layers]
  int64_t act_slot;
  int act_buffers;
  int64_t grad_slot;
  int grad_buffers;
  int64_t weight_rows;
  double count;                  // elements per channel over which BatchNorm normalises (N*H*W * world)
  float eps, momentum;
  int update_running;
  float param_grad_scale;        // 1 / world under SyncBatchNorm
  int n_gen;
  TrunkGen gen[kTrunkMaxGen];
};

// number of CTAs a launch uses (0: unsupported geometry)
int trunk_grid(int N, int H, int W);
size_t trunk_sync_bytes(int N, int H, int W);   // device scratch behind TrunkGen::sync (barrier words, flags, published sums)
int launch_trunk(const TrunkArgs& a, cudaStream_t stream);
// process-wide switch: 0 = never, 1 = wherever the kernel applies, 2 = automatic (default):
// fused when a layer has at most one 32x8-pixel tile per SM (launch-latency bound sizes), per-layer launches otherwise
bool trunk_fused_enabled();
bool trunk_fused_preferred(int N, int H, int W);
int set_trunk_fused(int mode);   // returns the previous mode
// SRG_TRUNK_PROF=1: per-CTA role timers of the most recent launch (developer aid)
int trunk_prof_read(long long* host, int n);

}  // namespace srg
