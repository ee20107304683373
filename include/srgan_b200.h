/* srgan_b200.h -- C ABI of the B200-native SR-GAN hot path (libsrgan_b200.so).
 *
 * The reference (angelowxx/Super_resolution-Image-Reconstructer-Multi_Generator_GAN) has no FFI of its own: its
 * hot path is Python calling PyTorch ATen ops.  Each entry point below therefore replaces a *range of reference
 * Python lines*, cited per function (paths relative to the reference root).  The Python host side in
 * super_resolution-image-reconstructer-multi_generator_gan_b200/ binds these with ctypes and re-exposes the
 * reference's nn.Module / train-step interface.
 *
 * Conventions
 *  - every function returns 0 on success, a positive cudaError_t or a negative argument-check code otherwise; it
 *    never throws, exits or synchronises.  srg_last_error() returns a thread-local description of the last failure.
 *  - all pointers are DEVICE pointers unless stated otherwise; the caller owns every buffer; work is enqueued on
 *    `stream` (a cudaStream_t passed as void*), nothing is allocated on the hot path.
 *  - images are NCHW fp32 (the reference's tensors); parameters / gradients / Adam moments are flat fp32 buffers
 *    whose element offsets are reported by srg_generator_param_info().
 */
#ifndef SRGAN_B200_H_
#define SRGAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRG_ABI_VERSION 1

int srg_abi_version(void);
const char* srg_last_error(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Generator engine: SRResNet (src/models.py:44-87) built from ResidualBlock (src/models.py:10-25).
 * N x 3 x H x W fp32 in  ->  N x 3 x (H << n_up) x (W << n_up) fp32 out; n_up = int(upscale_factor // 2) stages.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct srg_generator srg_generator_t;

/* replaces SRResNet.__init__ (src/models.py:53-78): fixes geometry, builds weight-packing and scatter maps. */
int srg_generator_create(srg_generator_t** out, int N, int H, int W, int num_residuals, int num_upsample_stages);
void srg_generator_destroy(srg_generator_t* g);

/* parameter table in the reference's parameters() order / state_dict keys (SURVEY Appendix A) */
int srg_generator_num_params(const srg_generator_t* g);
int64_t srg_generator_param_elems(const srg_generator_t* g); /* length of the flat fp32 param / grad buffers */
int srg_generator_param_info(const srg_generator_t* g, int i, char* name, int name_cap, int64_t* offset,
                             int64_t* numel, int* ndim, int* shape4);
/* BatchNorm running_mean / running_var table (flat fp32 buffer) */
int srg_generator_num_buffers(const srg_generator_t* g);
int64_t srg_generator_buffer_elems(const srg_generator_t* g);
int srg_generator_buffer_info(const srg_generator_t* g, int i, char* name, int name_cap, int64_t* offset,
                              int64_t* numel);

size_t srg_generator_workspace_bytes(const srg_generator_t* g, int training);
/* binds caller-owned memory; `workspace` must be 1024-byte aligned; `grads` may be NULL when training == 0 */
int srg_generator_bind(srg_generator_t* g, float* params, float* grads, float* bn_buffers, void* workspace,
                       size_t workspace_bytes, int training);
/* fp32 master weights -> packed bf16 GEMM operands; call after every optimizer step / load_state_dict */
/* re-points the flat gradient buffer srg_generator_backward writes (same layout as `params`) */
int srg_generator_set_grads(srg_generator_t* g, float* grads);
int srg_generator_pack(srg_generator_t* g, void* stream);
/* replaces SRResNet.forward (src/models.py:80-87); training != 0 uses batch statistics (and keeps the
 * activations backward needs), update_running != 0 updates running_mean/var (momentum 0.1, unbiased var). */
int srg_generator_forward(srg_generator_t* g, const float* lr_nchw, float* sr_nchw, int training, int update_running,
                          void* stream);
/* replaces autograd through SRResNet inside g_loss.backward() (src/train.py:195): d(loss)/d(sr) in, every
 * parameter gradient out (written to the bound flat `grads`; biases feeding a training-mode BatchNorm get 0). */
int srg_generator_backward(srg_generator_t* g, const float* dsr_nchw, void* stream);
/* a fixed generator inside a larger differentiable pipeline (SRResNet in eval() fed an input that requires grad, whose
 * BatchNorm layers use their running statistics as in src/models.py:16,19 under model.eval()): eval-mode (running-
 * statistics) BatchNorm on a training-bound workspace, keeping what the backward needs; running statistics are read,
 * never updated and never exchanged across ranks.  The output differs from the eval-bound srg_generator_forward in bf16
 * rounding only (BatchNorm is a separate pass over the stored conv output instead of the conv epilogue). */
int srg_generator_forward_frozen(srg_generator_t* g, const float* lr_nchw, float* sr_nchw, void* stream);
/* backward of the last forward (training or frozen) through SRResNet (src/models.py:53-87), as autograd computes it for
 * the reference's nn.Module.  param_grads == 0: no parameter gradient is computed or written (the flat `grads` buffer
 * is not touched); dlr_nchw (may be NULL) receives d(loss)/d(lr) as fp32 N x 3 x H x W.  After a frozen forward the
 * biases of the trunk convs get their real gradient (a BatchNorm with fixed statistics passes it on).
 * srg_generator_backward(g, dsr, stream) == srg_generator_backward_ex(g, dsr, 1, NULL, stream).  Fails before any CUDA
 * call on a null engine or dsr_nchw, an unbound or eval-bound workspace, or param_grads == 0 with dlr_nchw == NULL. */
int srg_generator_backward_ex(srg_generator_t* g, const float* dsr_nchw, int param_grads, float* dlr_nchw, void* stream);

/* Spatially tiled eval forward: upscale frames larger than the engine, window by window, bit-identical to the whole-frame
 * eval forward.  srg_generator_tile_halo: the receptive radius in LR pixels (40 for 16 residual blocks and 2 upsample
 * stages): an output pixel depends on the input pixels at most that far away (-1 on negative arguments).
 * srg_generator_forward_tiles: the engine, created as (N, Hw, Ww) and bound to an EVAL workspace, runs n <= min(N,
 * SRG_MAX_TILES) windows of Hw x Ww LR pixels, taken from any of the F frames (NCHW fp32, F x 3 x H x W), in one eval pass:
 * window i is read from frames[tile.frame, :, y0 .. y0+Hw-1, x0 .. x0+Ww-1] (zero outside it, exactly as if it had been
 * cropped into its own tensor), and only the output pixels of its crop (crop_y0 .. crop_y0+crop_h-1 etc., window-relative,
 * times 2^n_up) are written, into sr_nchw (F x 3 x (H << n_up) x (W << n_up)) at their place in the frame.  A crop edge that
 * is not a frame edge must lie at least srg_generator_tile_halo() pixels inside its window for the output to equal the
 * whole-frame forward; window origins on even rows keep it bit-identical (conv3_il's even / odd row blocks accumulate the
 * three row taps in different orders).  `tiles` is a HOST array, copied into the kernel parameters: no allocation, upload
 * or synchronisation, so the call can be captured in a CUDA graph.  Every argument is checked before any CUDA call. */
typedef struct {
  int32_t frame, y0, x0, crop_y0, crop_x0, crop_h, crop_w; /* LR pixels; (y0, x0) = window origin in the frame, crop relative to the window */
} srg_tile_t;
#define SRG_MAX_TILES 64
int srg_generator_tile_halo(int num_residuals, int num_upsample_stages);
int srg_generator_forward_tiles(srg_generator_t* g, const float* frames_nchw, int F, int H, int W, const srg_tile_t* tiles,
                                int n, float* sr_nchw, void* stream);
/* 8-bit frame I/O of the eval forward, for frames as decoders produce them: uint8 RGB, channel-last.  Input byte v is read
 * as __fdiv_rn(v, 255) (ToTensor's fp32 division), output value y is stored as rint(255 * clamp(y, 0, 1)) (fp32 multiply,
 * round half to even; NaN stores 0), so the result equals (sr.clamp(0, 1) * 255).round().to(uint8) of the fp32 forward of
 * ToTensor(frames), bit for bit, with no fp32 copy of the input and no fp32 SR tensor.  The workspace is unchanged.
 * srg_generator_forward_u8: the eval forward (training = 0, no running-statistics update) of the engine's N frames,
 * lr_nhwc N x H x W x 3 -> sr_nhwc N x (H << n_up) x (W << n_up) x 3.
 * srg_generator_forward_tiles_u8: srg_generator_forward_tiles on F x H x W x 3 frames into F x (H << n_up) x (W << n_up)
 * x 3, with the same windows, checks and graph-capture guarantee.  Both check every argument before any CUDA call. */
int srg_generator_forward_u8(srg_generator_t* g, const uint8_t* lr_nhwc, uint8_t* sr_nhwc, void* stream);
int srg_generator_forward_tiles_u8(srg_generator_t* g, const uint8_t* frames_nhwc, int F, int H, int W,
                                   const srg_tile_t* tiles, int n, uint8_t* sr_nhwc, void* stream);
/* Eval-mode autograd over windows, for frames whose whole-frame frozen workspace is too large.  With running BatchNorm
 * statistics every layer is local, so for windows whose crops partition the frames (crop edges at least
 * srg_generator_tile_halo() inside the window, as for srg_generator_forward_tiles) the whole-frame gradients are sums of
 * window-local ones: x.grad adds up every window's input gradient over its whole window, a parameter gradient adds up the
 * windows' parameter gradients.
 * srg_generator_forward_frozen_tiles: srg_generator_forward_frozen over n <= min(N, SRG_MAX_TILES) windows, read from the
 * frames and written to sr_nchw (crops only) exactly as srg_generator_forward_tiles does, on an engine bound to a TRAINING
 * workspace.  It keeps every activation the backward reads and remembers the windows and the frames' H and W.  sr_nchw may be NULL:
 * the output conv is then skipped (a recompute for the backward).
 * srg_generator_backward_tiles: the backward of the last forward, which must be a frozen-tiles forward.  dsr_nchw is
 * F x 3 x (H << n_up) x (W << n_up); each window's backward sees it inside the window's crop and zero elsewhere.
 * param_grads != 0: the bound `grads` receive the sum over these windows (overwritten, as srg_generator_backward_ex does).
 * dlr_nchw (F x 3 x H x W, may be NULL) is ADDED to: every window's input gradient over its whole window, window by window
 * in table order, deterministic without atomics (the caller zeroes it once before the first call).  Windows of one call
 * may overlap.  param_grads == 0 with dlr_nchw == NULL fails.  Both check every argument before any CUDA call; tables
 * travel in kernel parameters.  srg_generator_backward / _ex refuse to run after a frozen-tiles forward. */
int srg_generator_forward_frozen_tiles(srg_generator_t* g, const float* frames_nchw, int F, int H, int W,
                                       const srg_tile_t* tiles, int n, float* sr_nchw, void* stream);
int srg_generator_backward_tiles(srg_generator_t* g, const float* dsr_nchw, int param_grads, float* dlr_nchw, void* stream);

/* named intermediates inside the workspace (per-layer parity checks): dtype 0 = bf16 NHWC, dims = N,H,W,C */
int srg_generator_num_tensors(const srg_generator_t* g);
int srg_generator_tensor_info(const srg_generator_t* g, int i, char* name, int name_cap, int64_t* byte_offset,
                              int* dims4, int* dtype);
/* parity-test aid: call before srg_generator_bind; every inter-layer gradient then gets its own named tensor
 * ("rb<i>.d_y2", "rb<i>.d_pre1", "rb<i>.d_y1", "rb<i>.d_in", "d_last", "d_pre_conv1") instead of rotating buffers. */
int srg_generator_set_keep_grads(srg_generator_t* g, int keep);
long long srg_generator_launch_count(const srg_generator_t* g); /* kernels enqueued so far by this engine */
long long srg_total_launches(void);                             /* kernels enqueued so far by the whole library */
/* parity-test / A-B aid: which convolution kernels later launches use.  0 = default (conv3_il for plain 3x3 / 64-channel
 * launches, conv9_rows for conv3; honours SRG_CONV_IL), 1 = the generic strip kernel for everything, 2 = conv3_il with one
 * 8-pixel strip per column shift, 3 = conv3_il with one 10-pixel strip.  Returns the previous value.  Affects kernels
 * enqueued afterwards (a captured CUDA graph keeps what it was captured with). */
int srg_set_conv_variant(int variant);
/* host-only: the work split of the batched trunk weight-gradient kernel for `layers` same-shape [N,H,W,64] layers
 * (no device work, usable without a GPU): CTA c owns flattened (layer, tile) indices [c * per_cta, (c + 1) * per_cta),
 * layer l = index / tiles_per_layer; its partial set for layer l goes to slot c - (l * tiles_per_layer) / per_cta, and
 * slot < max_slots.  Returns 0. */
/* host-only: the conv9_rows schedule (conv3, 9x9 / 3 output channels) for input row ri = 0..15 of a tile: the output rows
 * (TMEM blocks) jlo..jhi it feeds, the first filter slot (slot 8 - kh of the resident [kh8 ; ... ; kh0] stack, kh = ri - j)
 * and whether block jhi is touched for the first time.  The kernel evaluates the same inline function. */
int srg_conv9_rows_window(int ri, int* jlo, int* jhi, int* slot_lo, int* fresh);
int srg_wgrad_batched_plan(int N, int H, int W, int layers, int* tiles_per_layer, int* grid, int* per_cta, int* max_slots);
/* CUDA-event timing of the dominant kernel class (the 3x3 64->64 forward / data-gradient conv_gemm launches, 66 per
 * generator fwd+bwd): enable, run steps, then read the summed device time (ms) and launch count since the last read
 * (read synchronises on the recorded events and resets the counters). */
int srg_generator_profile_enable(srg_generator_t* g, int on);
int srg_generator_profile_read(srg_generator_t* g, double* ms_sum, long long* count);
/* Fused trunk kernel (csrc/trunk_fused.cu): the 2*n_res+1 3x3 / 64->64 convolutions of one direction of the residual trunk
 * (src/models.py:10-25 ResidualBlock x 16, :66 conv2) with their training-mode BatchNorm steps in ONE cooperative launch.
 * srg_set_trunk_fused(mode): 0 = one launch per layer, 1 = the fused kernel wherever it applies, 2 = automatic (default:
 * fused when a layer has at most one 32x8-pixel tile per SM, i.e. launch-latency-bound sizes; measured in
 * profiles/r02_notes.md).  SRG_TRUNK_FUSED=0/1 sets the initial mode.  Returns the previous mode.  srg_generator_trunk_layers: trunk conv layers covered by
 * the engine's last profiled launch (1 = per-layer launches).  srg_generator_trunk_error: non-zero if a bounded in-kernel
 * wait of the fused kernel ever gave up (bit 0 cross-CTA flag / barrier, bit 1 mbarrier, bit 2 peer GPU); synchronises. */
int srg_set_trunk_fused(int on);
/* Split execution of one generator pass, for the multi-generator step (readme.md:2-10: K generators trained on the same
 * batch): phases is a bit mask, 1 = PRE (forward: conv1 + LeakyReLU, src/models.py:81; backward: conv3 and the upsample
 * stages), 2 = TRUNK (the 16 residual blocks + conv2, src/models.py:82-84, forward or backward), 4 = POST (forward:
 * upsample + conv3, src/models.py:85-86; backward: conv1 gradients and the batched trunk weight gradients); 7 = the whole
 * pass (= srg_generator_forward / srg_generator_backward).  srg_generators_trunk runs the TRUNK phase of n <= 4 engines of
 * identical geometry jointly: where the fused trunk kernel is preferred, as ONE launch that interleaves their layers (the
 * BatchNorm barrier latency of one generator hides behind the tensor work of the others); otherwise layer by layer with ONE
 * grouped convolution launch per layer for up to three engines (csrc/conv_gemm.cu launch_conv_gemm_grouped: 49 CTAs per
 * engine, 3x the tiles per CTA) and each engine's BatchNorm passes on forked streams between two launches (internal side
 * streams that join `stream` again before the call returns; capturable).  srg_generator_trunk_layers reports 33 / n / 1 for
 * the fused / grouped / per-layer form of the last profiled launch.  Engines must be bound for training; split execution
 * needs the fused trunk kernel or the grouped path (batched trunk weight gradients, single GPU or the peer-memory
 * SyncBatchNorm transport, SRG_TRUNK_GROUPED != 0) -- otherwise these return an error and the caller uses the whole-pass
 * entry points. */
int srg_generator_forward_phases(srg_generator_t* g, const float* lr_nchw, float* sr_nchw, int training, int update_running,
                                 int phases, void* stream);
int srg_generator_backward_phases(srg_generator_t* g, const float* dsr_nchw, int phases, void* stream);
int srg_generators_trunk(srg_generator_t* const* gs, int n, int backward, int update_running, void* stream);
/* developer aid (SRG_TRUNK_PROF=1): cycle counters [cta][role: producer, MMA issuer, epilogue][6] of the last fused launch */
int srg_debug_trunk_prof(long long* host, int n);
int srg_generator_trunk_layers(const srg_generator_t* g);
int srg_generator_trunk_error(srg_generator_t* g);

/* SyncBatchNorm hook: called between the local per-channel sums and the BatchNorm finalize in forward and
 * backward with a device buffer of `n` doubles to be summed in place across `world` ranks on `stream`. */
typedef int (*srg_allreduce_f64_fn)(void* ctx, double* buf, int n, void* stream);
int srg_generator_set_allreduce(srg_generator_t* g, srg_allreduce_f64_fn fn, void* ctx, int world);

/* NCCL-backed implementation of the hook (libnccl is resolved with dlopen at first use).  Communicators are
 * explicit handles: one per model lets the models' steps run concurrently on separate streams / graph branches
 * without sharing a communicator.  srg_nccl_allreduce_f64 has the hook's signature (ctx = communicator). */
int srg_nccl_unique_id(void* out128); /* host buffer, 128 bytes */
int srg_nccl_comm_create(const void* unique_id128, int world, int rank, void** comm_out);
void srg_nccl_comm_destroy(void* comm);
int srg_nccl_allreduce_f64(void* comm, double* buf, int n, void* stream);
int srg_nccl_allreduce_f32(void* comm, float* buf, int64_t n, void* stream);
/* mean over ranks in one collective (ncclAvg): the DDP gradient all-reduce of src/train.py:195 without a scaling pass */
int srg_nccl_allreduce_mean_f32(void* comm, float* buf, int64_t n, void* stream); /* flat gradient all-reduce (sum) */
int srg_generator_use_nccl(srg_generator_t* g, void* comm, int world);

/* SyncBatchNorm over NVLink peer memory (preferred to the NCCL hook): the statistics reduction, the exchange with all
 * ranks (P2P stores into every peer's buffer + release flags through NVSwitch) and the BatchNorm finalize are ONE
 * kernel per BatchNorm layer and direction, CUDA-graph capturable.  Set-up: every rank creates its object, the 64-byte
 * IPC handles are all-gathered by the host (any transport), connect() maps the peers' buffers. */
typedef struct srg_peer_sync srg_peer_sync_t;
int srg_peer_sync_create(srg_peer_sync_t** out, int world, int rank);
int srg_peer_sync_handle(srg_peer_sync_t* ps, void* out64);
int srg_peer_sync_connect(srg_peer_sync_t* ps, const void* handles_world_x_64);
void srg_peer_sync_destroy(srg_peer_sync_t* ps);
int srg_peer_sync_error(srg_peer_sync_t* ps); /* 1 if a wait on a peer ever timed out (synchronises the device) */
int srg_generator_use_peer_sync(srg_generator_t* g, srg_peer_sync_t* ps);

/* ---------------------------------------------------------------------------------------------------------------
 * Discriminator engine (src/models.py:90-120): conv 8x8 s2 p2 (3->64), then 3 x conv 4x4 s2 p1 (64->128->256->512),
 * each followed by MaxPool2d(3,2), InstanceNorm2d (no affine, biased variance, eps 1e-5) and LeakyReLU(0.2); the last
 * stage ends in Sigmoid.  N x 3 x H x W fp32 in -> N x 512 x h x w fp32 out.  create() fails with the same conditions
 * that make the reference raise (a stage's conv output smaller than the 3x3 pooling window, or a final map of one
 * element: every HR axis >= 428 and one >= 684, SURVEY Appendix E).
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct srg_discriminator srg_discriminator_t;
int srg_discriminator_create(srg_discriminator_t** out, int N, int H, int W);
void srg_discriminator_destroy(srg_discriminator_t* d);
int srg_discriminator_output_hw(const srg_discriminator_t* d, int* h, int* w);
int srg_discriminator_num_params(const srg_discriminator_t* d);
int64_t srg_discriminator_param_elems(const srg_discriminator_t* d);
int srg_discriminator_param_info(const srg_discriminator_t* d, int i, char* name, int name_cap, int64_t* offset,
                                 int64_t* numel, int* ndim, int* shape4);
size_t srg_discriminator_workspace_bytes(const srg_discriminator_t* d, int training);
int srg_discriminator_bind(srg_discriminator_t* d, float* params, float* grads, void* workspace, size_t workspace_bytes,
                           int training);
int srg_discriminator_set_grads(srg_discriminator_t* d, float* grads);
int srg_discriminator_pack(srg_discriminator_t* d, void* stream);
/* replaces Discriminator.forward (src/models.py:117-119) */
int srg_discriminator_forward(srg_discriminator_t* d, const float* x_nchw, float* out_nchw, void* stream);
/* replaces autograd through the discriminator (src/train.py:195 in GAN mode, :222): dout = d(loss)/d(out).
 * param_grads != 0: every parameter gradient is written to the bound flat `grads`; dx_nchw (may be NULL) receives
 * d(loss)/d(input image), the path the generator's adversarial term back-propagates through. */
int srg_discriminator_backward(srg_discriminator_t* d, const float* dout_nchw, int param_grads, float* dx_nchw,
                               void* stream);
/* named intermediates (parity tests): dtype 0 = bf16, 1 = fp32; dims = N,H,W,C (channel-last) */
int srg_discriminator_num_tensors(const srg_discriminator_t* d);
int srg_discriminator_tensor_info(const srg_discriminator_t* d, int i, char* name, int name_cap, int64_t* byte_offset,
                                  int* dims4, int* dtype);

/* ---------------------------------------------------------------------------------------------------------------
 * Per-operator entry points for the HBM-bound BatchNorm passes (nn.BatchNorm2d(64) in training mode, src/models.py:16,19,
 * 23-24, and its autograd backward): the engines above call the same kernels; these exports let a caller (or bench.py's
 * HBM roofline leg) run them on its own [pixels][64] NHWC bf16 tensors.  All pointers are device pointers; every call
 * only enqueues on `stream`.
 *   srg_bn_stats          partials[rows][128] fp32 = per-block {sum a[64], sum a*a[64]} (b == NULL) or {sum a, sum a*b}
 *                         (BatchNorm backward: a = dout, b = y); rows = srg_bn_stats_rows(pixels) <= 296
 *   srg_bn_finalize       partial rows -> scale = gamma/sqrt(var+eps), shift = beta - mean*scale, save_mean, save_inv (biased
 *                         variance, fixed summation order, fp64); running_mean / running_var (may be NULL) updated with
 *                         `momentum` and the unbiased variance like torch
 *   srg_bn_apply          out = [relu](y*scale + shift) [+ skip]
 *   srg_bn_backward_finalize  partial rows of {sum dout, sum dout*y} -> dgamma, dbeta (may be NULL) and the coefficients of
 *                         dy = A*dout + B*y + C
 *   srg_bn_backward_apply dy = A*dout + B*y + C
 * ------------------------------------------------------------------------------------------------------------- */
int srg_bn_stats_rows(int64_t pixels);
int srg_bn_stats(const void* a_nhwc_bf16, const void* b_nhwc_bf16, int64_t pixels, float* partials, void* stream);
int srg_bn_finalize(const float* partials, int rows, double count, const float* gamma, const float* beta, float eps,
                    float momentum, float* running_mean, float* running_var, float* scale, float* shift, float* save_mean,
                    float* save_inv, void* stream);
int srg_bn_apply(const void* y_nhwc_bf16, const float* scale, const float* shift, const void* skip_nhwc_bf16, int relu,
                 void* out_nhwc_bf16, int64_t pixels, void* stream);
int srg_bn_backward_finalize(const float* partials, int rows, double count, const float* gamma, const float* save_mean,
                             const float* save_inv, float* dgamma, float* dbeta, float* coef_a, float* coef_b, float* coef_c,
                             void* stream);
int srg_bn_backward_apply(const void* dout_nhwc_bf16, const void* y_nhwc_bf16, const float* coef_a, const float* coef_b,
                          const float* coef_c, void* dy_nhwc_bf16, int64_t pixels, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Per-operator convolution (SURVEY 8b "conv2d_{fprop,dgrad,wgrad} ... workspace_bytes"): nn.Conv2d(cin, cout, ksize,
 * padding=ksize/2) (src/models.py:15,18,56,66,71,78 and the VGG19 stack of src/models.py:126) and its autograd backward
 * on NHWC bf16 activations [N][H][W][C] with C a multiple of 64; ksize 1 or 3 (wgrad: 3).  The engines above launch the
 * same tcgen05 kernels; these exports make topologies other than SRResNet / Discriminator reachable.
 *   srg_conv2d_pack_weights  fp32 OIHW -> the kernels' bf16 operand layout (srg_conv2d_packed_weight_bytes bytes);
 *                            for_dgrad != 0 packs the transposed, flipped copy the input-gradient launch convolves with
 *   srg_conv2d_fprop         out = act(conv(x) + bias) (+ residual); act: 0 none, 1 ReLU, 2 LeakyReLU(slope)
 *   srg_conv2d_dgrad         dx = conv^T(dy) (+ residual), or zeroed where relu_mask_src <= 0 (the ReLU that produced x)
 *   srg_conv2d_wgrad         dw (fp32 OIHW) = sum over pixels of x (x) dy per tap, dbias (may be NULL) = sum dy; workspace:
 *                            srg_conv2d_wgrad_workspace_bytes (caller-owned, nothing is allocated inside)
 * ------------------------------------------------------------------------------------------------------------- */
size_t srg_conv2d_packed_weight_bytes(int cout, int cin, int ksize);
int srg_conv2d_pack_weights(const float* w_oihw, int cout, int cin, int ksize, int for_dgrad, void* packed, void* stream);
int srg_conv2d_fprop(const void* x_nhwc_bf16, int N, int H, int W, int cin, const void* w_packed, int cout, int ksize,
                     const float* bias, int act, float slope, const void* residual_nhwc_bf16, void* out_nhwc_bf16,
                     void* stream);
int srg_conv2d_dgrad(const void* dy_nhwc_bf16, int N, int H, int W, int cout, const void* w_packed_dgrad, int cin, int ksize,
                     const void* relu_mask_src_nhwc_bf16, const void* residual_nhwc_bf16, void* dx_nhwc_bf16, void* stream);
size_t srg_conv2d_wgrad_workspace_bytes(int N, int H, int W, int cin, int cout);
int srg_conv2d_wgrad(const void* x_nhwc_bf16, const void* dy_nhwc_bf16, int N, int H, int W, int cin, int cout,
                     void* workspace, size_t workspace_bytes, float* dw_oihw, float* dbias, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * VGG19 perceptual loss (src/models.py:123-151 VGGFeatureExtractor, src/utils.py:154-166 perceptal_loss; listed in the
 * train_generator signature, src/train.py:175): the conv layers go through srg_conv2d_*; these are the passes between
 * them.  NHWC bf16 activations (C % 8 == 0), NCHW fp32 images.
 *   srg_unfold3x3_rgb      im2col of the 3-channel first layer: out[N][H][W][64], channel (kh*3 + kw)*3 + c (27 used), so
 *                          vgg19.features[0] becomes a 1x1 convolution over 64 channels
 *   srg_fold3x3_rgb        its adjoint: gradient of the unfolded tensor -> d(image) NCHW fp32 (times scale)
 *   srg_maxpool2x2_*       nn.MaxPool2d(2, 2) forward / backward (gradient to the first maximum, like torch; `add`
 *                          optionally adds a second gradient of dx's shape: a feature tapped before the pool)
 *   srg_l1_bf16            out1[0] (+)= weight * mean|a - b| (torch.nn.L1Loss); grad_a (may be NULL) = weight * grad_scale *
 *                          sign(a - b) / n, zeroed where relu_mask != 0 and a <= 0 (a is a ReLU output)
 * ------------------------------------------------------------------------------------------------------------- */
int srg_unfold3x3_rgb(const float* x_nchw, int N, int H, int W, void* out_nhwc64_bf16, void* stream);
int srg_fold3x3_rgb(const void* d_unfolded_nhwc64_bf16, int N, int H, int W, float scale, float* dx_nchw, void* stream);
int srg_maxpool2x2_forward(const void* x_nhwc_bf16, int N, int H, int W, int C, void* out_nhwc_bf16, void* stream);
int srg_maxpool2x2_backward(const void* x_nhwc_bf16, const void* dy_nhwc_bf16, const void* add_nhwc_bf16, int N, int H,
                            int W, int C, void* dx_nhwc_bf16, void* stream);
size_t srg_l1_bf16_scratch_bytes(void);
int srg_l1_bf16(const void* a_bf16, const void* b_bf16, int64_t n, float weight, int accumulate, float grad_scale,
                int relu_mask, void* grad_a_bf16, void* scratch, size_t scratch_bytes, float* out1, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Losses and optimiser
 * ------------------------------------------------------------------------------------------------------------- */
/* replaces ReconstructionLoss.forward (src/utils.py:173-241; called at src/train.py:189):
 * losses2[0] = edge-weighted L1 ("com_loss"), losses2[1] = Laplacian TV loss.  e_buf / g_buf: fp32 scratch of hr's
 * size, kept (with `scratch`) for the backward call. */
size_t srg_recon_loss_scratch_bytes(void);
int srg_recon_loss_forward(const float* hr_nchw, const float* sr_nchw, int N, int C, int H, int W, void* scratch,
                           size_t scratch_bytes, float* e_buf, float* g_buf, float* losses2, void* stream);
/* replaces autograd through ReconstructionLoss inside g_loss.backward() (src/train.py:195):
 * grad_sr = (w_edge * d losses2[0]/d sr + w_tv * d losses2[1]/d sr) * grad_scale, where w_edge / w_tv are optional
 * DEVICE scalars (NULL = 1; the reference's objective is com_loss + tv_loss, src/train.py:192). */
int srg_recon_loss_backward(const float* hr_nchw, const float* sr_nchw, int N, int C, int H, int W, const void* scratch,
                            const float* e_buf, const float* g_buf, const float* w_edge, const float* w_tv,
                            float* grad_sr, float grad_scale, void* stream);
/* replaces mean(tanh(fake - real)) / mean(tanh(real - fake)) (src/train.py:218, :190):
 * out[0] = mean(tanh(sign * (a - b))); da / db (may be NULL) receive the gradients times grad_scale. */
int srg_tanh_mean(const float* a, const float* b, int64_t n, float sign, void* scratch, size_t scratch_bytes,
                  float* out1, float* da, float* db, float grad_scale, void* stream);
/* Plain mean losses the scope statement names next to the reference's own objective (the reference code has no L1 / MSE
 * / BCE call on its hot path, SURVEY section 0; oracle: torch.nn.functional.l1_loss / mse_loss / binary_cross_entropy):
 * kind 0 = mean|a-b|, 1 = mean (a-b)^2, 2 = BCE with a = probabilities, b = targets (logs clamped at -100 like torch).
 * grad_a (may be NULL) receives d out / d a times grad_scale. */
int srg_point_loss(int kind, const float* a, const float* b, int64_t n, void* scratch, size_t scratch_bytes, float* out1,
                   float* grad_a, float grad_scale, void* stream);
/* replaces torch.optim.Adam.step with default betas/eps, no weight decay (src/train.py:61-62,196,223) on flat
 * buffers; `step` is the 1-based step count; gradients are multiplied by grad_scale first (1/world for DDP mean). */
int srg_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                  float beta1, float beta2, float eps, int step, float grad_scale, void* stream);

/* same update, CUDA-graph capturable: the learning rate and the number of steps taken so far live in device memory
 * (`*step_dev` is read as t-1 and incremented on the stream), so a captured step replays correctly under an LR
 * scheduler. */
int srg_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, const float* lr_dev,
                      float beta1, float beta2, float eps, int* step_dev, float grad_scale, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Evaluation path (src/evaluation.py:48-52)
 * ------------------------------------------------------------------------------------------------------------- */
/* replaces ImageEnhancer.forward (src/models.py:36-41): out = clamp(x + factor * Laplacian3x3(x), 0, 1), NCHW fp32 */
int srg_image_enhance(const float* x_nchw, int N, int C, int H, int W, float factor, float* out_nchw, void* stream);
/* out1[0] (DEVICE double) = mean((a - b)^2); calculate_psnr (src/utils.py:141-144) = 10 * log10(1 / mse) */
int srg_mse(const float* a, const float* b, int64_t n, void* scratch, size_t scratch_bytes, double* out1, void* stream);
/* replaces the per-image metric loop of compute_score (src/train.py:263-294) over calculate_psnr / calculate_ssim
 * (src/utils.py:141-151), for N images of 3 x H x W fp32 (NCHW) at once, both metrics in one pass over sr and hr:
 *   psnr_out[n] (DEVICE double) = 10 * log10(1 / mean((sr_n - hr_n)^2)), +inf for identical images (data_range 1)
 *   ssim_out[n] (DEVICE double) = skimage structural_similarity(sr_n, hr_n, win_size=3) with the array taken as a 3-D
 *                volume (channel_axis None): 3x3x3 uniform window, sample covariance (27/26), C1 = 1e-4, C2 = 9e-4, the
 *                map cropped by 1 on every axis = the mean of S over channel 1, rows 1..H-2, columns 1..W-2.
 * Needs C == 3, H >= 3, W >= 3, N >= 1 and scratch_bytes >= srg_image_metrics_scratch_bytes(N, H, W) (caller-owned,
 * 8-byte aligned); checked before any CUDA call.  An image's results do not depend on N or on its position in the batch.
 * Two kernel launches, no allocation, copy or synchronisation: capturable into a CUDA graph. */
size_t srg_image_metrics_scratch_bytes(int N, int H, int W); /* 0 for invalid sizes */
int srg_image_metrics(const float* sr, const float* hr, int N, int C, int H, int W, void* scratch, size_t scratch_bytes,
                      double* psnr_out, double* ssim_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Image-size transforms either side of the path (src/transformers.py:73-82, applied per image in src/utils.py:34-47):
 * transforms.Resize on PIL images = Pillow's ImagingResample (antialiased: the filter support scales with the reduction
 * factor; separable; 22-bit fixed-point coefficients; uint8 after each pass).  Bit-exact with Pillow for 8-bit RGB.
 *   srg_resize_plan_ksize  taps per output element for one axis (filter 0 = bilinear, 1 = bicubic), -1 on bad arguments
 *   srg_resize_plan        HOST arrays bounds[out][2] = (first input index, tap count), coeffs[out][ksize]
 *   srg_resize_u8          src uint8 [N][H][W][3] -> out_u8 [N][out_h][out_w][3] and / or out_f32 [N][3][out_h][out_w] =
 *                          v / 255 (ToTensor) + noise * sigma[n] (the degradation of downward_img_quality; both NULL: none).
 *                          bounds_* / coeffs_* are DEVICE copies of the plans; tmp: uint8 [N][H][out_w][3] when out_w != W
 * ------------------------------------------------------------------------------------------------------------- */
int srg_resize_plan_ksize(int in_size, int out_size, int filter);
int srg_resize_plan(int in_size, int out_size, int filter, int32_t* bounds_host, int32_t* coeffs_host);
int srg_resize_u8(const uint8_t* src_nhwc, int N, int H, int W, int out_h, int out_w, const int32_t* bounds_w,
                  const int32_t* coeffs_w, int ksize_w, const int32_t* bounds_h, const int32_t* coeffs_h, int ksize_h,
                  uint8_t* tmp, uint8_t* out_u8_nhwc, float* out_f32_nchw, const float* noise_nchw,
                  const float* sigma_per_image, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SRGAN_B200_H_ */
