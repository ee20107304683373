// Host-side description of one "strip" implicit-GEMM convolution launch (internal; the public
// C ABI in include/srgan_b200.h is a thin layer above this).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace srg {

constexpr int kMaxStrips = 9;
constexpr int kMaxTaps = 9;
constexpr int kMaxInMaps = 4;

enum ConvAct : int { ACT_NONE = 0, ACT_RELU = 1, ACT_LRELU = 2 };
enum ConvOutMode : int {
  OUT_NHWC = 0,          // bf16 [N,H,W,cout_total]
  OUT_PIXEL_SHUFFLE = 1, // bf16 [N,2H,2W,64]; GEMM n-block q=(i,j) -> pixel (2h+i, 2w+j)
  OUT_FOLD9_NCHW = 2,    // fp32 [N,3,H,W]; GEMM n = s*3+co partial sums, shift-accumulated over s (9x9, Cout=3)
  OUT_NHWC_F32 = 3,      // fp32 [N,H,W,cout_total] (direct 128-bit stores; discriminator conv outputs)
};

// Store of a fold9 (OUT_FOLD9_NCHW) launch: channel c of output pixel (h, w) of item i goes to element
// base_i + c * plane + h * pitch + w * px of `out`, with base_i = i * item (n == 0: whole frames) or t[i].base (a cropped
// scatter over n <= kMaxTiles windows, srg_generator_forward_tiles, which writes only h_lo <= h < h_hi, w_lo <= w < w_hi).
// fp32 NCHW: (plane, pitch, px) = (H x W, W, 1); uint8 NHWC (u8 = 1, quantised, srg_generator_forward_u8): (1, 3W, 3), in
// the units of the full frames.  A launch without one stores fp32 NCHW of its own geometry.  Passed by value in the
// kernel parameters; offsets are 64-bit.
constexpr int kMaxTiles = 64;
struct FoldTile {
  int64_t base;            // element offset of the window origin in channel 0 of its frame
  int h_lo, h_hi, w_lo, w_hi;
};
struct FoldScatter {
  int n;                   // 0: whole-frame store of the launch's N items
  int u8;                  // 1: uint8, y -> rint(255 * clamp(y, 0, 1)) (NaN -> 0); 0: fp32
  int64_t item, plane, pitch, px;  // element strides: item (n == 0), channel, row, pixel
  FoldTile t[kMaxTiles];
};

// One view of the (NHWC bf16) input that a K-chunk is loaded from. A plain tensor uses one view;
// the pixel-unshuffled gradient of an up-conv uses four strided views of the HR tensor.
struct InView {
  const void* ptr;       // base address (16-byte aligned)
  int64_t stride_w;      // in elements, multiple of 8
  int64_t stride_h;
  int64_t stride_n;
  int channels;          // channels visible through this view (multiple of 64)
};

struct ConvGemmArgs {
  // logical output grid (stride-1 conv: same grid as the input views)
  int N, H, W;
  int TH, TW;            // pixel tile, TH*TW == 128, TW % 8 == 0
  // input
  int n_views;
  InView views[kMaxInMaps];
  int in_H, in_W;        // extents of the input views (rows/cols outside are zero)
  // taps: n_strips column shifts, each with n_taps row offsets
  int n_strips, n_taps;
  int strip_dw[kMaxStrips];  // column offset of strip s relative to the tile origin
  int strip_dh;              // row offset of every strip's first row relative to the tile origin
  int strip_rows;            // rows loaded per strip (TH + vertical span)
  int tap_row[kMaxTaps];     // first strip row used by tap r
  // packed weights: bf16 [n_chunks*n_strips*n_taps][cout_total][64], k-block index ((c*S+s)*R+r)
  const void* weights;
  int cout_total;            // multiple of block_n
  int block_n;               // 32 (fold9 only) or 64
  // epilogue
  const float* bias;         // [cout_total] (GEMM n order) or nullptr; OUT_FOLD9: [3]
  const float* scale;        // optional [cout_total]: out = act(acc * scale + bias) (eval-mode BatchNorm folded into the
                             // epilogue: scale = gamma / sqrt(var + eps), bias = beta + (conv bias - mean) * scale)
  int act;
  float slope;
  const void* residual;      // bf16, same layout as out (OUT_NHWC only), added after activation
  const void* mask_src;      // bf16, same layout as out: out = (mask_src > 0) ? out : 0  (ReLU backward)
  void* out;
  int out_mode;
  int exclusive;             // 1: nothing else runs beside this launch (inference): conv3_il takes all shared memory for its
                             // pipeline instead of leaving 44 KB to co-resident CTAs of other graph branches
  int variant;               // 0: pick the kernel automatically (row-interleaved conv3_il for plain 3x3 / 64-channel launches,
                             // conv9_rows for the plain fold9 conv), 1: force the generic strip kernel (the reference the
                             // specialised kernels are tested against)
  float* stats;              // optional (OUT_NHWC, cout 64): per-CTA column sums of the STORED bf16 tile values,
                             // float [conv_gemm_grid(a)][128] = {sum over valid pixels [64], sum of squares [64]}
  void* prof;                // optional debug timers: int64 [grid][3][6]
  const FoldScatter* scatter;  // optional (OUT_FOLD9_NCHW only, host memory): the store layout (default fp32 NCHW)
  // fold9: tile columns overlap; valid output columns per tile = TW-8
};

// Returns 0 on success, cudaError_t (>0) or a negative argument-check code otherwise.
int launch_conv_gemm(const ConvGemmArgs& a, cudaStream_t stream);
constexpr int kIlMaxGroups = 3;
// one launch for the same 3x3 / 64 -> 64 layer of n <= kIlMaxGroups independent problems (see conv_gemm.cu); rows of statistics per group
int launch_conv_gemm_grouped(const ConvGemmArgs* as, int n, cudaStream_t stream);
int conv_gemm_grouped_rows(const ConvGemmArgs& a, int n);
// number of CTAs launch_conv_gemm uses for `a` (= rows written to a.stats)
int conv_gemm_grid(const ConvGemmArgs& a);

// Weight gradient: D_t[ci][co] = sum_p x[p + shift_t][ci] * dy[p][co] for every tap t = s*n_taps + r
// (strip-major), taps paired (2i, 2i+1) into 128-row accumulators.  Partials layout:
// [splits][n_blocks][n_pairs][128][64] fp32 with row = (t & 1)*64 + ci, column = co within the n-block.
struct WgradArgs {
  int N, H, W;               // output-gradient grid
  int TH, TW;
  InView x;                  // 64-channel input view (rows/cols outside in_H/in_W read as zero)
  int in_H, in_W;
  int dy_views;              // 1: one NHWC tensor with n_blocks*64 channels; 4: one 64-channel view per n-block
  InView dy[4];
  int n_blocks;
  int n_strips, n_taps, strip_rows, strip_dh;
  int strip_dw[kMaxStrips];
  int tap_row[kMaxTaps];
  float* partials;
};
int wgrad_partials_floats(const WgradArgs& a, int* splits_out);
int launch_wgrad_gemm(const WgradArgs& a, cudaStream_t stream);
// 3x3 stride-1 specialisation (taps fused along M and N): partials [splits][n_blocks][kw 3][(2-kh)*64 + co][ci 64]
int wgrad3x3_partials_floats(const WgradArgs& a, int* splits_out);
int launch_wgrad3x3(const WgradArgs& a, cudaStream_t stream);
// All same-shape 3x3 / 64->64 layers in one launch (+ one reduce launch).  Layer l reads x at x_base + l * x_layer_stride
// and dy at dy_base + l * dy_layer_stride (dense NHWC bf16 tensors [N,H,W,64]); its OIHW gradient is written to
// grads + out_off[l] through `inv` (partial element -> output element, the map launch_wgrad_reduce_inv uses).
struct WgradBatchArgs {
  int N, H, W, n_layers;
  const void* x_base;
  int64_t x_layer_stride_bytes;
  const void* dy_base;
  int64_t dy_layer_stride_bytes;
  float* partials;           // wgrad3_batched_partials_floats(a) floats
  const int* inv;            // device, 3*192*64 ints
  float* grads;
  const long long* out_off;  // device, n_layers element offsets into grads
};
// work split: tiles per layer, CTAs, flattened (layer, tile) indices per CTA, partial-set slots per layer (host arithmetic)
void wgrad3_batched_plan(const WgradBatchArgs& a, int* tiles_per_layer, int* grid, int* per_cta, int* max_slots);
size_t wgrad3_batched_partials_floats(const WgradBatchArgs& a);
int launch_wgrad3x3_batched(const WgradBatchArgs& a, cudaStream_t stream);
int launch_wgrad_reduce(const float* partials, const int* idx, float* out, int n_out, int splits, size_t split_stride,
                        int accumulate_into, cudaStream_t stream);

// conv9_rows schedule (shared by the kernel and by the host-side test entry srg_conv9_rows_window): input row `ri` of a tile
// (image row h0 + ri - 4, ri = 0..15) reaches the output rows (TMEM blocks) jlo..jhi with row tap kh = ri - j in [0, 8];
// block j reads filter slot 8 - kh of the resident [kh8 ; ... ; kh0] stack, so the blocks' slots are consecutive from
// slot_lo; `fresh`: block jhi sees its first tap (kh = 0) on this row and must overwrite instead of accumulate.
struct C9Window { int jlo, jhi, slot_lo, fresh; };
__host__ __device__ inline C9Window c9_window(int ri) {
  C9Window w;
  w.jlo = ri > 8 ? ri - 8 : 0;
  w.jhi = ri < 7 ? ri : 7;
  w.slot_lo = 8 - ri + w.jlo;
  w.fresh = ri <= 7 ? 1 : 0;
  return w;
}

// process-wide override of ConvGemmArgs::variant for launches that leave it 0 (parity tests): 0 or 1; returns the old
// value, or a negative code (set_error) for any other value, leaving the override unchanged
int set_conv_variant(int variant);

// SMs a persistent kernel sizes its grid for: the device's SM count
int sm_budget();

// total kernels launched by this library in this process (bench bookkeeping: "gpu_launches")
void count_launch(int n = 1);
long long total_launches();

// partial-side reduction: inv[j] = output element (or -1) for partial element j of one split; n_part % 4 == 0
int launch_wgrad_reduce_inv(const float* partials, const int* inv, float* out, int n_part, int splits, size_t split_stride,
                            cudaStream_t stream);

const char* last_error();
void set_error(const char* fmt, ...);

}  // namespace srg
