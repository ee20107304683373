// Memory-bound kernels of the SR-GAN hot path (internal launchers; the C ABI is in api.cu).
// All activations are NHWC bf16 with 64 channels per pixel (128 bytes), images are NCHW fp32.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace srg {

constexpr int kRedBlocksMax = 296;  // 2 x 148 SMs

// ---- per-channel reductions over [P pixels][64 ch] bf16 ------------------------------------------
// partials: float [blocks][128]  ([0,64) = sum a ; [64,128) = sum a*a (b == null) or sum a*b)
int reduce_blocks(int64_t pixels);
int launch_chan_reduce(const void* a, const void* b, int64_t pixels, float* partials, cudaStream_t st);
// Per-channel finalize of the fixed-order partial sums (launch_partials_finalize).
// RF_BN_BWD_FROZEN: backward of an eval-mode (running-statistics) BatchNorm; save_mean / save_inv hold running_mean and
// 1 / sqrt(running_var + eps), the coefficients are A = gamma * inv, B = C = 0 and `dbias` (optional) receives the
// gradient of the preceding conv's bias, A * sum(dz)
enum ReduceFinalizeMode : int { RF_BN_FWD = 0, RF_BN_BWD = 1, RF_SUM = 2, RF_BN_BWD_FROZEN = 3 };
struct ReduceFinalize {
  int mode;
  double count;                 // elements per channel
  float eps, momentum;
  const float* gamma;
  const float* beta;
  float* running_mean;          // RF_BN_FWD: optional
  float* running_var;
  const float* save_mean;       // RF_BN_BWD inputs
  const float* save_inv;
  float* dgamma;                // RF_BN_BWD outputs (optional)
  float* dbeta;
  float* out0;                  // FWD: scale | BWD: coefA | SUM: sums (float[64])
  float* out1;                  // FWD: shift | BWD: coefB
  float* out2;                  // FWD: save_mean | BWD: coefC
  float* out3;                  // FWD: save_inv
  float* dbias;                 // RF_BN_BWD_FROZEN: preceding conv's bias gradient (optional)
};
// Two-launch form used on the hot path: any producer of [rows][128] fp32 partials (launch_chan_reduce, or the conv
// epilogue's fused statistics) followed by ONE 1024-thread block that sums them in a fixed order and finalizes.
int launch_partials_finalize(const float* partials, int rows, const ReduceFinalize& f, cudaStream_t st);
// SyncBatchNorm path: only the fixed-order column sums (double[128]); the all-reduce and finalize follow.
int launch_partials_sums(const float* partials, int rows, double* sums, cudaStream_t st);
// sums[128] (double) = fixed-order sum of the block partials
int launch_partials_to_sums(const float* partials, int blocks, double* sums, cudaStream_t st);

// BatchNorm (training) finalize from sums = {sum y, sum y^2} over `count` elements per channel:
// scale = gamma*rsqrt(var+eps), shift = beta-mean*scale, saves mean / inv_std, updates running stats.
int launch_bn_finalize(const double* sums, double count, const float* gamma, const float* beta, float eps,
                       float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                       float* save_mean, float* save_inv, cudaStream_t st);
// eval mode: scale/shift from running statistics
// conv_bias (optional): fold the producing conv's bias into the shift, for the fused epilogue form
// out = act(acc * scale + shift) of ConvGemmArgs::scale
int launch_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean,
                          const float* running_var, float eps, float* scale, float* shift, cudaStream_t st,
                          const float* conv_bias = nullptr);
// all `n_bn` eval-mode BatchNorm layers of a model at once: tab[l] = int4{gamma, beta, running_mean (running_var = +64),
// conv bias} float offsets into master / buffers; coef[l][256] = {scale[64], shift[64] with the conv bias folded in, ...}
int launch_bn_eval_coeffs_all(const float* master, const float* buffers, const void* tab, int n_bn, float eps, float* coef,
                              cudaStream_t st);
// eval-mode BatchNorm on the training path (the conv adds its own bias): coef[l][256] = {scale = gamma * inv,
// shift = beta - running_mean * scale, running_mean, inv = 1 / sqrt(running_var + eps)}; tab as launch_bn_eval_coeffs_all
// (the conv-bias column is not read)
int launch_bn_frozen_coeffs_all(const float* master, const float* buffers, const void* tab, int n_bn, float eps, float* coef,
                                cudaStream_t st);
// out = act(scale*y + shift) (+ skip);  relu: 0/1
int launch_bn_apply(const void* y, const float* scale, const float* shift, const void* skip, int relu, void* out,
                    int64_t pixels, cudaStream_t st);
// BatchNorm backward finalize from sums = {sum dout, sum dout*y}: writes dgamma/dbeta and the
// per-channel coefficients of  dy = A*dout + B*y + C.
int launch_bn_bwd_finalize(const double* sums, double count, const float* gamma, const float* save_mean,
                           const float* save_inv, float* dgamma, float* dbeta, float* coefA, float* coefB,
                           float* coefC, float param_grad_scale, cudaStream_t st);
int launch_bn_bwd_apply(const void* dout, const void* y, const float* coefA, const float* coefB, const float* coefC,
                        void* dy, int64_t pixels, cudaStream_t st);
// d(pre-activation) of LeakyReLU from two incoming gradients: dpre = (ga + gb) * (post > 0 ? 1 : slope)
int launch_lrelu_bwd_add2(const void* ga, const void* gb, const void* post, float slope, void* dpre, int64_t pixels,
                          cudaStream_t st);
// out[c] = float(sums[c]) for c < n  (bias gradients)
int launch_sums_to_float(const double* sums, float* out, int n, cudaStream_t st);
// bias gradient of an up-conv whose output gradient lives in pixel-shuffled layout [N,2H,2W,64]:
// db[4c + 2i + j] = sum over (n,h,w) of g[n,2h+i,2w+j,c].  scratch: float [rows2][128], rows2 = N*2H.
int launch_ps_bias_grad(const void* g, int N, int H2, int W2, float* scratch, float* dbias, cudaStream_t st);

// ---- 9x9 / 3-channel helper: unfold an NCHW fp32 3-channel image into row-pair columns -----------
// dst bf16 [N][H+1][W][64]; channel (dr*27 + s*3 + c) of row h' holds src[n][c][h'-1+dr][w+s-4] (0 outside,
// channels 54..63 = 0).  `scale` multiplies the values (used to keep tiny loss gradients in bf16 range).
int launch_unfold9(const float* src, int N, int H, int W, float scale, void* dst, cudaStream_t st);
// Window gather form: item i of the same [N][H+1][W][64] operand is the H x W window whose origin (channel 0) is element
// base[i] of `frames` (NCHW fp32 frames of `plane` elements per channel and `pitch` per row), zero outside the window
// exactly as if the window had been cropped into its own tensor.  Passed by value in the kernel parameters.
constexpr int kMaxWindows = 64;
struct WindowGather {
  int n;
  int64_t plane, pitch;
  int64_t base[kMaxWindows];
};
int launch_unfold9_windows(const float* frames, const WindowGather& wg, int H, int W, void* dst, cudaStream_t st);
// 8-bit forms (srg_generator_forward_u8 / _tiles_u8): the same operand from uint8 NHWC frames, each byte v read as
// __fdiv_rn(v, 255) like ToTensor.  Dense: src [N][H][W][3].  Windows: base / plane / pitch of `wg` in bytes (plane = 1,
// pitch = 3 x frame width); any width, pixels need no alignment.
int launch_unfold9_u8(const uint8_t* src, int N, int H, int W, void* dst, cudaStream_t st);
int launch_unfold9_windows_u8(const uint8_t* frames, const WindowGather& wg, int H, int W, void* dst, cudaStream_t st);
// Windows of F x 3 x fh x fw fp32 frames for the backward of the frozen-tiles forward (srg_generator_backward_tiles), in
// the pixel units of the grid they index (HR for d(SR), LR for d(lr)).  Item i is the window of frame[i] at (y0[i], x0[i]);
// its crop is rows [h_lo, h_hi) x columns [w_lo, w_hi), window-relative.  Passed by value in the kernel parameters.
struct WindowTable {
  int n;
  int fh, fw;
  int frame[kMaxWindows], y0[kMaxWindows], x0[kMaxWindows];
  int h_lo[kMaxWindows], h_hi[kMaxWindows], w_lo[kMaxWindows], w_hi[kMaxWindows];
};
// Crop-masked gather: dst (n x 3 x H x W, H x W = the window) = the frames inside each item's crop, 0 elsewhere
int launch_crop_masked_gather(const float* frames, const WindowTable& wt, int H, int W, float* dst, cudaStream_t st);
// Ordered scatter-add: frames += src (n x 3 x H x W) over each item's whole window.  Where windows overlap, one thread adds
// every item's value in table order, ((f + src[i1]) + src[i2]) + ..., so the result is deterministic without atomics.
int launch_window_scatter_add(const float* src, const WindowTable& wt, int H, int W, float* frames, cudaStream_t st);

// ---- parameters ------------------------------------------------------------------------------------
// dst[i] = bf16(idx[i] >= 0 ? src[idx[i]] : 0)
int launch_pack_bf16(const float* src, const int* idx, void* dst, int64_t n, cudaStream_t st);
// dst[i] = idx[i] >= 0 ? src[idx[i]] : 0
int launch_gather_f32(const float* src, const int* idx, float* dst, int64_t n, cudaStream_t st);
// torch.optim.Adam (no weight decay, no amsgrad) over flat fp32 buffers; step = 1-based step count.
int launch_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                int step, float grad_scale, cudaStream_t st);

// same update with the learning rate and the (0-based, pre-increment) step count in DEVICE memory: CUDA-graph capturable
int launch_adam_dev(float* p, const float* g, float* m, float* v, int64_t n, const float* lr_dev, float beta1, float beta2,
                    float eps, int* step_dev, float grad_scale, cudaStream_t st);

// ---- ReconstructionLoss (reference src/utils.py:173-241) ------------------------------------------
// hr, sr: fp32 [N][3][H][W].  scratch doubles: >= loss_scratch_doubles().  e_buf, g_buf: fp32, same size as hr.
// losses[0] = edge_loss, losses[1] = tv_loss (forward); backward re-uses scratch / e_buf / g_buf of the forward call.
int loss_scratch_doubles();
int launch_recon_loss_forward(const float* hr, const float* sr, int N, int C, int H, int W, double* scratch, float* e_buf,
                              float* g_buf, float* losses, cudaStream_t st);
// grad = (w_edge * d edge/d sr + w_tv * d tv/d sr) * grad_scale; w_* are optional DEVICE scalars (null = 1)
int launch_recon_loss_backward(const float* hr, const float* sr, int N, int C, int H, int W, const double* scratch,
                               const float* e_buf, const float* g_buf, const float* w_edge, const float* w_tv, float* grad,
                               float grad_scale, cudaStream_t st);
// per-channel sums of an NCHW fp32 tensor: out[c] = scale * sum_{n,h,w} x[n][c][h][w]   (C <= 8)
int launch_nchw_chan_sum(const float* x, int N, int C, int64_t plane, double* scratch, float* out, float scale,
                         cudaStream_t st);

// ---- evaluation path ------------------------------------------------------------------------------
// ImageEnhancer.forward (src/models.py:36-41): out = clamp(x + factor * (L * x), 0, 1), L = Laplacian of the loss
int launch_image_enhance(const float* x, int N, int C, int H, int W, float factor, float* out, cudaStream_t st);
// out[0] (double, device) = mean((a - b)^2): the PSNR numerator of src/utils.py:141-144 (psnr = 10 log10(1 / mse))
int launch_mse(const float* a, const float* b, int64_t n, double* scratch, double* out, cudaStream_t st);

// plain mean losses (kind 0: L1, 1: MSE, 2: BCE with a = probabilities, b = targets); grad_a (optional) = d out / d a
// times grad_scale.  Vectorised 128-bit loads/stores, fixed-order reduction.
int launch_point_loss(int kind, const float* a, const float* b, int64_t n, double* scratch, float* out, float* grad_a,
                      float grad_scale, cudaStream_t st);

// relativistic tanh losses of the reference (src/train.py:190,218): out[0] = mean(tanh(sign*(a-b)));
// grads (optional): da = sign*(1-tanh^2)/n * gscale, db = -da
int launch_tanh_mean(const float* a, const float* b, int64_t n, float sign, double* scratch, float* out, float* da,
                     float* db, float gscale, cudaStream_t st);

}  // namespace srg
