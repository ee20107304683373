// Standalone GPU probe for the strip implicit-GEMM conv kernel (developer tool, not part of the product path).
// Builds random problems, runs launch_conv_gemm and compares with a scalar CPU evaluation of the same packed-GEMM
// definition.  Usage: conv_probe [timing_iters]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../super_resolution-image-reconstructer-multi_generator_gan_b200/csrc/conv_gemm.cuh"

using namespace srg;

static uint32_t rng_state = 12345u;
static float frand() {
  rng_state = rng_state * 1664525u + 1013904223u;
  return ((rng_state >> 8) & 0xFFFF) / 65536.0f - 0.5f;
}
static uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  uint32_t r = u + 0x7FFF + ((u >> 16) & 1);
  return uint16_t(r >> 16);
}
static float bf2f(uint16_t h) {
  uint32_t u = uint32_t(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
#define CK(x)                                                                  \
  do {                                                                         \
    cudaError_t e_ = (x);                                                      \
    if (e_ != cudaSuccess) {                                                   \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      exit(2);                                                                 \
    }                                                                          \
  } while (0)

struct Problem {
  const char* name;
  int N, H, W, TH, TW;
  int n_views, view_ch;      // input = n_views views of view_ch channels; stored as one [N,H,W,n_views*view_ch] tensor
  bool strided_views;        // views are the 4 pixel-shuffle phases of an HR tensor [N,2H,2W,64]
  int n_strips, n_taps, strip_rows, strip_dh;
  int strip_dw[9], tap_row[9];
  int cout_total, block_n;
  bool bias;
  int act;
  bool residual, mask;
  int out_mode;
  bool stats;                // exercise the fused BatchNorm-statistics epilogue (timing only)
  int variant;               // ConvGemmArgs::variant: 0 = specialised kernels (conv3_il, conv9_rows), 1 = generic strip kernel
};

static int run(const Problem& pr, int timing_iters) {
  const int Cin = pr.n_views * pr.view_ch;
  const int n_chunks = Cin / 64;
  const int KB = n_chunks * pr.n_strips * pr.n_taps;
  // input tensor, logical [N][H][W][Cin] (bf16)
  std::vector<uint16_t> x(size_t(pr.N) * pr.H * pr.W * Cin);
  for (auto& v : x) v = f2bf(frand());
  // physical layout
  std::vector<uint16_t> xphys(x.size());
  if (pr.strided_views) {
    // HR tensor [N][2H][2W][64]; view q=(i,j): pixel (2h+i, 2w+j)
    for (int n = 0; n < pr.N; ++n)
      for (int h = 0; h < pr.H; ++h)
        for (int w = 0; w < pr.W; ++w)
          for (int c = 0; c < Cin; ++c) {
            int q = c / 64, ch = c % 64, i = q >> 1, j = q & 1;
            size_t dst = ((size_t(n) * 2 * pr.H + 2 * h + i) * 2 * pr.W + 2 * w + j) * 64 + ch;
            xphys[dst] = x[((size_t(n) * pr.H + h) * pr.W + w) * Cin + c];
          }
  } else {
    xphys = x;
  }
  std::vector<uint16_t> wp(size_t(KB) * pr.cout_total * 64);
  for (auto& v : wp) v = f2bf(frand() * 0.25f);
  std::vector<float> bias(pr.cout_total);
  for (auto& v : bias) v = frand();
  const bool fold = pr.out_mode == OUT_FOLD9_NCHW;
  const bool ps = pr.out_mode == OUT_PIXEL_SHUFFLE;
  const size_t out_elems = fold ? size_t(pr.N) * 3 * pr.H * pr.W : size_t(pr.N) * pr.H * pr.W * pr.cout_total;
  std::vector<uint16_t> res(out_elems), msk(out_elems);
  for (auto& v : res) v = f2bf(frand());
  for (auto& v : msk) v = f2bf(frand());

  void *dx, *dw, *dout, *dres, *dmsk;
  float* dbias;
  CK(cudaMalloc(&dx, xphys.size() * 2));
  CK(cudaMalloc(&dw, wp.size() * 2));
  CK(cudaMalloc(&dout, out_elems * 4));
  CK(cudaMalloc(&dres, out_elems * 2));
  CK(cudaMalloc(&dmsk, out_elems * 2));
  CK(cudaMalloc(&dbias, bias.size() * 4));
  CK(cudaMemcpy(dx, xphys.data(), xphys.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dw, wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dres, res.data(), out_elems * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dmsk, msk.data(), out_elems * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dbias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(dout, 0xFF, out_elems * 4));

  ConvGemmArgs a;
  memset(&a, 0, sizeof(a));
  a.N = pr.N; a.H = pr.H; a.W = pr.W; a.TH = pr.TH; a.TW = pr.TW;
  a.n_views = pr.n_views;
  for (int v = 0; v < pr.n_views; ++v) {
    if (pr.strided_views) {
      int i = v >> 1, j = v & 1;
      a.views[v].ptr = (uint16_t*)dx + (size_t(i) * 2 * pr.W + j) * 64;
      a.views[v].stride_w = 128;
      a.views[v].stride_h = int64_t(4) * pr.W * 64;
      a.views[v].stride_n = int64_t(4) * pr.H * pr.W * 64;
    } else {
      a.views[v].ptr = (uint16_t*)dx + size_t(v) * pr.view_ch;
      a.views[v].stride_w = Cin;
      a.views[v].stride_h = int64_t(pr.W) * Cin;
      a.views[v].stride_n = int64_t(pr.H) * pr.W * Cin;
    }
    a.views[v].channels = pr.view_ch;
  }
  a.in_H = pr.H; a.in_W = pr.W;
  a.n_strips = pr.n_strips; a.n_taps = pr.n_taps; a.strip_rows = pr.strip_rows; a.strip_dh = pr.strip_dh;
  for (int s = 0; s < pr.n_strips; ++s) a.strip_dw[s] = pr.strip_dw[s];
  for (int r = 0; r < pr.n_taps; ++r) a.tap_row[r] = pr.tap_row[r];
  a.weights = dw; a.cout_total = pr.cout_total; a.block_n = pr.block_n;
  a.bias = pr.bias ? dbias : nullptr; a.act = pr.act; a.slope = 0.2f;
  a.residual = pr.residual ? dres : nullptr; a.mask_src = pr.mask ? dmsk : nullptr;
  a.out = dout; a.out_mode = pr.out_mode; a.variant = pr.variant;
  float* dstats = nullptr;
  if (pr.stats) { CK(cudaMalloc(&dstats, 148 * 128 * 4)); a.stats = dstats; }

  int rc = launch_conv_gemm(a, 0);
  if (rc != 0) { printf("[%s] launch rc=%d err=%s\n", pr.name, rc, last_error()); return 1; }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("[%s] kernel failed: %s\n", pr.name, cudaGetErrorString(e)); exit(3); }

  std::vector<uint8_t> outraw(out_elems * 4);
  CK(cudaMemcpy(outraw.data(), dout, out_elems * 4, cudaMemcpyDeviceToHost));

  // CPU reference on a sample of pixels (all pixels when small)
  const size_t npix = size_t(pr.N) * pr.H * pr.W;
  const size_t stride = npix > 6000 ? npix / 3000 : 1;
  double max_err = 0, max_ref = 0;
  size_t checked = 0, bad = 0;
  auto in_at = [&](int n, int h, int w, int c) -> float {
    if (h < 0 || h >= pr.H || w < 0 || w >= pr.W) return 0.f;
    return bf2f(x[((size_t(n) * pr.H + h) * pr.W + w) * Cin + c]);
  };
  auto gemm_at = [&](int n, int h, int w, int co) -> float {  // sum over all k-blocks
    double acc = 0;
    for (int c = 0; c < n_chunks; ++c)
      for (int s = 0; s < pr.n_strips; ++s)
        for (int r = 0; r < pr.n_taps; ++r) {
          const int kb = (c * pr.n_strips + s) * pr.n_taps + r;
          const int hh = h + pr.strip_dh + pr.tap_row[r], ww = w + pr.strip_dw[s];
          if (hh < 0 || hh >= pr.H || ww < 0 || ww >= pr.W) continue;
          const uint16_t* wrow = &wp[(size_t(kb) * pr.cout_total + co) * 64];
          const uint16_t* xrow = &x[((size_t(n) * pr.H + hh) * pr.W + ww) * Cin + c * 64];
          for (int k = 0; k < 64; ++k) acc += double(bf2f(xrow[k])) * bf2f(wrow[k]);
        }
    return float(acc);
  };
  (void)in_at;
  for (size_t pi = 0; pi < npix; pi += stride) {
    const int n = int(pi / (size_t(pr.H) * pr.W));
    const int h = int((pi / pr.W) % pr.H);
    const int w = int(pi % pr.W);
    if (fold) {
      for (int co = 0; co < 3; ++co) {
        double ref = pr.bias ? bias[co] : 0.0;
        for (int s = 0; s < 9; ++s) {
          const int ww = w + s - 4;
          if (ww < 0 || ww >= pr.W) continue;
          ref += gemm_at(n, h, ww, s * 3 + co);
        }
        const float got = reinterpret_cast<float*>(outraw.data())[((size_t(n) * 3 + co) * pr.H + h) * pr.W + w];
        const double err = fabs(got - ref);
        if (err > max_err) max_err = err;
        if (fabs(ref) > max_ref) max_ref = fabs(ref);
        if (!(err <= 0.02 + 0.01 * fabs(ref))) ++bad;
        ++checked;
      }
    } else {
      for (int co = 0; co < pr.cout_total; ++co) {
        float ref = gemm_at(n, h, w, co);
        if (pr.bias) ref += bias[co];
        if (pr.act == ACT_RELU) ref = ref > 0 ? ref : 0;
        if (pr.act == ACT_LRELU) ref = ref > 0 ? ref : 0.2f * ref;
        size_t oidx;
        if (ps) {
          const int q = co / 64, ch = co % 64, i = q >> 1, j = q & 1;
          oidx = ((size_t(n) * 2 * pr.H + 2 * h + i) * 2 * pr.W + 2 * w + j) * 64 + ch;
        } else {
          oidx = ((size_t(n) * pr.H + h) * pr.W + w) * pr.cout_total + co;
        }
        if (pr.residual) ref += bf2f(res[oidx]);
        if (pr.mask && !(bf2f(msk[oidx]) > 0.f)) ref = 0;
        const float got = bf2f(reinterpret_cast<uint16_t*>(outraw.data())[oidx]);
        const double err = fabs(got - ref);
        if (err > max_err) max_err = err;
        if (fabs(ref) > max_ref) max_ref = fabs(ref);
        if (!(err <= 0.02 + 0.01 * fabs(ref))) ++bad;
        ++checked;
      }
    }
  }
  printf("[%s] checked=%zu bad=%zu max_abs_err=%.5f max_ref=%.3f %s\n", pr.name, checked, bad, max_err, max_ref,
         bad == 0 ? "OK" : "FAIL");

  if (timing_iters > 0) {
    long long* dprof;
    CK(cudaMalloc(&dprof, 1024 * 18 * 8));
    CK(cudaMemset(dprof, 0, 1024 * 18 * 8));
    a.prof = dprof;
    static void* flush_buf = nullptr;
    const size_t flush_bytes = size_t(512) << 20;
    if (!flush_buf) CK(cudaMalloc(&flush_buf, flush_bytes));
    const bool cold = getenv("PROBE_COLD") != nullptr;
    if (cold) { CK(cudaMemsetAsync(flush_buf, 1, flush_bytes, 0)); CK(cudaDeviceSynchronize()); }
    launch_conv_gemm(a, 0);
    CK(cudaDeviceSynchronize());
    a.prof = nullptr;
    std::vector<long long> hp(1024 * 18);
    CK(cudaMemcpy(hp.data(), dprof, hp.size() * 8, cudaMemcpyDeviceToHost));
    for (int b = 0; b < 148; b += 49)
      printf("  cta %d: producer wait_empty=%lld total=%lld | mma wait_tempty=%lld wait_full=%lld total=%lld | epi wait_tfull=%lld total=%lld\n", b,
             hp[(b * 3 + 0) * 6 + 0], hp[(b * 3 + 0) * 6 + 4], hp[(b * 3 + 1) * 6 + 1], hp[(b * 3 + 1) * 6 + 2], hp[(b * 3 + 1) * 6 + 4],
             hp[(b * 3 + 2) * 6 + 3], hp[(b * 3 + 2) * 6 + 4]);
    {
      // averages over all CTAs (cycles): [producer wait_empty, mma wait_tempty, mma wait_full, epi(warp 2) wait_tfull], totals
      double acc[7] = {0, 0, 0, 0, 0, 0, 0};
      long long tmin = -1, tmax = 0;
      int nc = 0;
      for (int b = 0; b < 148; ++b) {
        if (hp[(b * 3 + 1) * 6 + 4] == 0) continue;
        ++nc;
        acc[0] += hp[(b * 3 + 0) * 6 + 0]; acc[1] += hp[(b * 3 + 1) * 6 + 1]; acc[2] += hp[(b * 3 + 1) * 6 + 2];
        acc[3] += hp[(b * 3 + 2) * 6 + 3]; acc[4] += hp[(b * 3 + 0) * 6 + 4]; acc[5] += hp[(b * 3 + 1) * 6 + 4]; acc[6] += hp[(b * 3 + 2) * 6 + 4];
        const long long t0 = hp[(b * 3 + 1) * 6 + 5], t1 = t0 + hp[(b * 3 + 2) * 6 + 4];
        if (tmin < 0 || t0 < tmin) tmin = t0;
        if (t1 > tmax) tmax = t1;
      }
      {
        double m0 = 0, m3 = 0, e0 = 0, e1 = 0, e2 = 0;
        for (int b = 0; b < 148; ++b) {
          m0 += hp[(b * 3 + 1) * 6 + 0]; m3 += hp[(b * 3 + 1) * 6 + 3];
          e0 += hp[(b * 3 + 2) * 6 + 0]; e1 += hp[(b * 3 + 2) * 6 + 1]; e2 += hp[(b * 3 + 2) * 6 + 2];
        }
        if (nc) printf("  timeline (cycles after the setup barrier): first MMA %.0f | last MMA commit %.0f | last accumulator ready %.0f | last store issued %.0f | store drained %.0f\n",
                       m0 / nc, m3 / nc, e0 / nc, e1 / nc, e2 / nc);
      }
      if (nc) printf("  %s avg over %d CTAs: prod wait_empty=%.0f (total %.0f) | mma wait_tempty=%.0f wait_full=%.0f (total %.0f) | epi wait_tfull=%.0f (total %.0f)\n",
                     cold ? "COLD" : "warm", nc, acc[0] / nc, acc[4] / nc, acc[1] / nc, acc[2] / nc, acc[5] / nc, acc[3] / nc, acc[6] / nc);
    }
    cudaFree(dprof);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    for (int i = 0; i < 3; ++i) launch_conv_gemm(a, 0);
    cudaEventRecord(e0);
    for (int i = 0; i < timing_iters; ++i) launch_conv_gemm(a, 0);
    cudaEventRecord(e1);
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    {
      // isolated launches: L2 flushed (512 MB memset) before each, no predecessor to overlap with
      float tot = 0;
      const int n_iso = 20;
      for (int i = 0; i < n_iso; ++i) {
        CK(cudaMemsetAsync(flush_buf, i, flush_bytes, 0));
        CK(cudaDeviceSynchronize());
        cudaEventRecord(e0);
        launch_conv_gemm(a, 0);
        cudaEventRecord(e1);
        CK(cudaEventSynchronize(e1));
        float t = 0; cudaEventElapsedTime(&t, e0, e1); tot += t;
      }
      float tot_h = 0;
      for (int i = 0; i < n_iso; ++i) {
        CK(cudaDeviceSynchronize());
        cudaEventRecord(e0);
        launch_conv_gemm(a, 0);
        cudaEventRecord(e1);
        CK(cudaEventSynchronize(e1));
        float t = 0; cudaEventElapsedTime(&t, e0, e1); tot_h += t;
      }
      printf("[%s] isolated launch: cold L2 %.2f us, warm L2 %.2f us (events around one launch)\n", pr.name, tot * 1000 / n_iso, tot_h * 1000 / n_iso);
    }
    const double flops = 2.0 * npix * double(KB) * 64 * pr.cout_total;
    printf("[%s] %.3f us/launch  %.1f TFLOP/s (MMA work incl. padding)\n", pr.name, ms * 1000 / timing_iters,
           flops / (ms / timing_iters * 1e-3) / 1e12);
  }
  cudaFree(dx); cudaFree(dw); cudaFree(dout); cudaFree(dres); cudaFree(dmsk); cudaFree(dbias);
  return bad == 0 ? 0 : 1;
}

static Problem conv3x3(const char* name, int N, int H, int W, int cout, bool ps) {
  Problem p;
  memset(&p, 0, sizeof(p));
  p.name = name; p.N = N; p.H = H; p.W = W; p.TH = 16; p.TW = 8;
  p.n_views = 1; p.view_ch = 64;
  p.n_strips = 3; p.n_taps = 3; p.strip_rows = 18; p.strip_dh = -1;
  for (int s = 0; s < 3; ++s) p.strip_dw[s] = s - 1;
  for (int r = 0; r < 3; ++r) p.tap_row[r] = r;
  p.cout_total = cout; p.block_n = 64; p.bias = true; p.act = ACT_NONE;
  p.out_mode = ps ? OUT_PIXEL_SHUFFLE : OUT_NHWC;
  p.variant = 1;
  return p;
}


// ------------------------------------------------------------------ wgrad probe
static int run_wgrad(const char* name, int N, int H, int W, int n_strips, int n_taps, int strip_rows, int strip_dh,
                     const int* strip_dw, const int* tap_row, int n_blocks, bool strided_dy, int iters, bool fused3 = false) {
  const int Cout = n_blocks * 64;
  std::vector<uint16_t> x(size_t(N) * H * W * 64), dy(size_t(N) * H * W * Cout);
  for (auto& v : x) v = f2bf(frand());
  for (auto& v : dy) v = f2bf(frand());
  std::vector<uint16_t> dyphys(dy.size());
  if (strided_dy) {
    for (int n = 0; n < N; ++n) for (int h = 0; h < H; ++h) for (int w = 0; w < W; ++w) for (int c = 0; c < Cout; ++c) {
      int q = c / 64, ch = c % 64, i = q >> 1, j = q & 1;
      dyphys[((size_t(n) * 2 * H + 2 * h + i) * 2 * W + 2 * w + j) * 64 + ch] = dy[((size_t(n) * H + h) * W + w) * Cout + c];
    }
  } else dyphys = dy;
  void *dx, *ddy; float* dpart; float* dout; int* didx;
  CK(cudaMalloc(&dx, x.size() * 2)); CK(cudaMalloc(&ddy, dy.size() * 2));
  CK(cudaMemcpy(dx, x.data(), x.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ddy, dyphys.data(), dy.size() * 2, cudaMemcpyHostToDevice));
  WgradArgs a; memset(&a, 0, sizeof(a));
  a.N = N; a.H = H; a.W = W; a.TH = 16; a.TW = 8;
  a.x.ptr = dx; a.x.stride_w = 64; a.x.stride_h = int64_t(W) * 64; a.x.stride_n = int64_t(H) * W * 64; a.x.channels = 64;
  a.in_H = H; a.in_W = W;
  if (strided_dy) {
    a.dy_views = 4;
    for (int v = 0; v < 4; ++v) {
      int i = v >> 1, j = v & 1;
      a.dy[v].ptr = (uint16_t*)ddy + (size_t(i) * 2 * W + j) * 64;
      a.dy[v].stride_w = 128; a.dy[v].stride_h = int64_t(4) * W * 64; a.dy[v].stride_n = int64_t(4) * H * W * 64; a.dy[v].channels = 64;
    }
  } else {
    a.dy_views = 1;
    a.dy[0].ptr = ddy; a.dy[0].stride_w = Cout; a.dy[0].stride_h = int64_t(W) * Cout; a.dy[0].stride_n = int64_t(H) * W * Cout; a.dy[0].channels = Cout;
  }
  a.n_blocks = n_blocks; a.n_strips = n_strips; a.n_taps = n_taps; a.strip_rows = strip_rows; a.strip_dh = strip_dh;
  for (int s = 0; s < n_strips; ++s) a.strip_dw[s] = strip_dw[s];
  for (int r = 0; r < n_taps; ++r) a.tap_row[r] = tap_row[r];
  int splits = 0;
  const int pf = fused3 ? wgrad3x3_partials_floats(a, &splits) : wgrad_partials_floats(a, &splits);
  if (fused3) printf("[%s] partial sets = %d\n", name, splits);
  CK(cudaMalloc(&dpart, size_t(pf) * 4));
  a.partials = dpart;
  const int T = n_strips * n_taps, n_pairs = (T + 1) / 2;
  // index map: out[t][ci][co_total]
  const int n_out = T * 64 * Cout;
  std::vector<int> idx(n_out);
  for (int t = 0; t < T; ++t) for (int ci = 0; ci < 64; ++ci) for (int co = 0; co < Cout; ++co) {
    const int nb = co / 64, pr = t / 2, row = (t & 1) * 64 + ci;
    idx[(t * 64 + ci) * Cout + co] = ((nb * n_pairs + pr) * 128 + row) * 64 + (co % 64);
    if (fused3) idx[(t * 64 + ci) * Cout + co] = ((nb * 3 + t / 3) * 192 + (2 - t % 3) * 64 + (co % 64)) * 64 + ci;
  }
  const size_t split_stride = fused3 ? size_t(n_blocks) * 3 * 64 * 192 : size_t(n_blocks) * n_pairs * 128 * 64;
  CK(cudaMalloc(&didx, n_out * 4)); CK(cudaMalloc(&dout, n_out * 4));
  CK(cudaMemcpy(didx, idx.data(), n_out * 4, cudaMemcpyHostToDevice));
  int rc = fused3 ? launch_wgrad3x3(a, 0) : launch_wgrad_gemm(a, 0);
  if (rc) { printf("[%s] launch rc=%d %s\n", name, rc, last_error()); return 1; }
  rc = launch_wgrad_reduce(dpart, didx, dout, n_out, splits, split_stride, 0, 0);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess || rc) { printf("[%s] kernel failed: %s\n", name, cudaGetErrorString(e)); exit(3); }
  std::vector<float> out(n_out);
  CK(cudaMemcpy(out.data(), dout, n_out * 4, cudaMemcpyDeviceToHost));
  // CPU reference on a sample of (t, ci, co)
  double max_err = 0, max_ref = 0; size_t bad = 0, checked = 0;
  for (int t = 0; t < T; ++t) {
    const int s = t / n_taps, r = t % n_taps;
    const int dh = strip_dh + tap_row[r], dw = strip_dw[s];
    for (int ci = (t * 7) % 5; ci < 64; ci += 13) for (int co = (t * 3) % 7; co < Cout; co += 29) {
      double acc = 0;
      for (int n = 0; n < N; ++n) for (int h = 0; h < H; ++h) {
        const int hh = h + dh; if (hh < 0 || hh >= H) continue;
        for (int w = 0; w < W; ++w) {
          const int ww = w + dw; if (ww < 0 || ww >= W) continue;
          acc += double(bf2f(x[((size_t(n) * H + hh) * W + ww) * 64 + ci])) * bf2f(dy[((size_t(n) * H + h) * W + w) * Cout + co]);
        }
      }
      const double got = out[(t * 64 + ci) * Cout + co];
      const double err = fabs(got - acc);
      if (err > max_err) max_err = err;
      if (fabs(acc) > max_ref) max_ref = fabs(acc);
      if (!(err <= 1e-2 + 2e-3 * fabs(acc))) ++bad;
      ++checked;
    }
  }
  printf("[%s] checked=%zu bad=%zu max_abs_err=%.5f max_ref=%.3f %s\n", name, checked, bad, max_err, max_ref, bad == 0 ? "OK" : "FAIL");
  if (iters > 0) {
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 3; ++i) { fused3 ? launch_wgrad3x3(a, 0) : launch_wgrad_gemm(a, 0); }
    cudaEventRecord(e0);
    for (int i = 0; i < iters; ++i) { fused3 ? launch_wgrad3x3(a, 0) : launch_wgrad_gemm(a, 0); }
    cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    printf("[%s] %.3f us/launch (gemm only)\n", name, ms * 1000 / iters);
    cudaEventRecord(e0);
    for (int i = 0; i < iters; ++i) { fused3 ? launch_wgrad3x3(a, 0) : launch_wgrad_gemm(a, 0); launch_wgrad_reduce(dpart, didx, dout, n_out, splits, split_stride, 0, 0); }
    cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * N * H * W * double(T) * 64 * Cout;
    printf("[%s] %.3f us/launch (gemm+reduce)  %.1f TFLOP/s useful\n", name, ms * 1000 / iters, flops / (ms / iters * 1e-3) / 1e12);
  }
  cudaFree(dx); cudaFree(ddy); cudaFree(dpart); cudaFree(dout); cudaFree(didx);
  return bad == 0 ? 0 : 1;
}

// ------------------------------------------------------------------ batched 3x3 wgrad probe (all layers in one launch)
static int run_wgrad_batched(const char* name, int L, int N, int H, int W, int iters) {
  const size_t S = size_t(N) * H * W * 64;            // elements per tensor
  const size_t xs = 2 * S + 512, ds = S + 1024;       // layer strides (elements): x two slots apart, padded
  std::vector<uint16_t> x(xs * L), dy(ds * L);
  for (auto& v : x) v = f2bf(frand());
  for (auto& v : dy) v = f2bf(frand());
  std::vector<int> inv(3 * 192 * 64);
  for (int kw = 0; kw < 3; ++kw) for (int kh = 0; kh < 3; ++kh) for (int co = 0; co < 64; ++co) for (int ci = 0; ci < 64; ++ci)
    inv[((kw * 192) + (2 - kh) * 64 + co) * 64 + ci] = ((co * 64 + ci) * 3 + kh) * 3 + kw;
  std::vector<long long> off(L);
  for (int l = 0; l < L; ++l) off[l] = (long long)l * 36864;
  void *dx, *ddy; int* dinv; long long* doff; float *dpart, *dgr;
  CK(cudaMalloc(&dx, x.size() * 2)); CK(cudaMalloc(&ddy, dy.size() * 2));
  CK(cudaMalloc(&dinv, inv.size() * 4)); CK(cudaMalloc(&doff, L * 8)); CK(cudaMalloc(&dgr, size_t(L) * 36864 * 4));
  CK(cudaMemcpy(dx, x.data(), x.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ddy, dy.data(), dy.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dinv, inv.data(), inv.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(doff, off.data(), L * 8, cudaMemcpyHostToDevice));
  CK(cudaMemset(dgr, 0, size_t(L) * 36864 * 4));
  WgradBatchArgs a; memset(&a, 0, sizeof(a));
  a.N = N; a.H = H; a.W = W; a.n_layers = L;
  a.x_base = dx; a.x_layer_stride_bytes = int64_t(xs) * 2; a.dy_base = ddy; a.dy_layer_stride_bytes = int64_t(ds) * 2;
  const size_t pf = wgrad3_batched_partials_floats(a);
  CK(cudaMalloc(&dpart, pf * 4));
  a.partials = dpart; a.inv = dinv; a.grads = dgr; a.out_off = doff;
  int rc = launch_wgrad3x3_batched(a, 0);
  cudaError_t e = cudaDeviceSynchronize();
  if (rc || e != cudaSuccess) { printf("[%s] failed rc=%d %s %s\n", name, rc, last_error(), cudaGetErrorString(e)); exit(3); }
  std::vector<float> g(size_t(L) * 36864);
  CK(cudaMemcpy(g.data(), dgr, g.size() * 4, cudaMemcpyDeviceToHost));
  size_t checked = 0, bad = 0; double max_err = 0, max_ref = 0;
  for (int l = 0; l < L; ++l)
    for (int s = 0; s < 40; ++s) {
      const int co = (s * 7 + l) % 64, ci = (s * 13 + 5 * l) % 64, kh = s % 3, kw = (s / 3) % 3;
      double ref = 0;
      for (int n = 0; n < N; ++n) for (int h = 0; h < H; ++h) for (int w = 0; w < W; ++w) {
        const int hi = h + kh - 1, wi = w + kw - 1;
        if (hi < 0 || hi >= H || wi < 0 || wi >= W) continue;
        ref += double(bf2f(x[xs * l + ((size_t(n) * H + hi) * W + wi) * 64 + ci])) * bf2f(dy[ds * l + ((size_t(n) * H + h) * W + w) * 64 + co]);
      }
      const double got = g[size_t(l) * 36864 + ((co * 64 + ci) * 3 + kh) * 3 + kw];
      const double err = fabs(got - ref);
      if (err > max_err) max_err = err;
      if (fabs(ref) > max_ref) max_ref = fabs(ref);
      if (err > 1e-3 * fabs(ref) + 5e-4 * sqrt(double(N) * H * W)) ++bad;   // fp32 accumulation over N*H*W products
      ++checked;
    }
  printf("[%s] checked=%zu bad=%zu max_abs_err=%.5f max_ref=%.3f %s\n", name, checked, bad, max_err, max_ref, bad == 0 ? "OK" : "FAIL");
  if (iters > 0) {
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 2; ++i) launch_wgrad3x3_batched(a, 0);
    cudaEventRecord(e0);
    for (int i = 0; i < iters; ++i) launch_wgrad3x3_batched(a, 0);
    cudaEventRecord(e1); CK(cudaEventSynchronize(e1));
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * L * N * H * W * 9.0 * 64 * 64;
    printf("[%s] %.3f us/launch (gemm+reduce, %d layers: %.3f us/layer)  %.1f TFLOP/s useful\n", name, ms * 1000 / iters, L,
           ms * 1000 / iters / L, flops / (ms / iters * 1e-3) / 1e12);
  }
  cudaFree(dx); cudaFree(ddy); cudaFree(dinv); cudaFree(doff); cudaFree(dpart); cudaFree(dgr);
  return bad == 0 ? 0 : 1;
}

int main(int argc, char** argv) {
  const int iters = argc > 1 ? atoi(argv[1]) : 0;
  int fails = 0;
  if (getenv("PROBE_IL_ONLY") != nullptr) {   // quick mode: the cfg2 trunk cases of the row-interleaved kernel only
    { Problem p = conv3x3("perf_il_trunk_16x96x96", 16, 96, 96, 64, false); p.variant = 0; fails += run(p, iters); }
    { Problem p = conv3x3("perf_il_trunk_stats", 16, 96, 96, 64, false); p.variant = 0; p.stats = true; fails += run(p, iters); }
    { Problem p = conv3x3("perf_il_trunk_mask", 16, 96, 96, 64, false); p.variant = 0; p.mask = true; p.bias = false; fails += run(p, iters); }
    { Problem p = conv3x3("perf_il_trunk_residual", 16, 96, 96, 64, false); p.variant = 0; p.residual = true; p.bias = false; fails += run(p, iters); }
    { Problem p = conv3x3("perf_il_trunk_mask_stats", 16, 96, 96, 64, false); p.variant = 0; p.mask = true; p.bias = false; p.stats = true; fails += run(p, iters); }
    { Problem p = conv3x3("perf_il_trunk_48x96x96", 48, 96, 96, 64, false); p.variant = 0; fails += run(p, iters); }
    printf("PROBE %s (%d failing cases)\n", fails == 0 ? "PASS" : "FAIL", fails);
    return fails == 0 ? 0 : 1;
  }
  {
    const int dw3[3] = {-1, 0, 1}, tr3[3] = {0, 1, 2};
    fails += run_wgrad("wg3x3_small", 2, 32, 24, 3, 3, 18, -1, dw3, tr3, 1, false, 0);
    fails += run_wgrad("wg3x3_ragged", 3, 40, 20, 3, 3, 18, -1, dw3, tr3, 1, false, 0);
    fails += run_wgrad("wg3x3_cout256_ps", 2, 32, 16, 3, 3, 18, -1, dw3, tr3, 4, true, 0);
    fails += run_wgrad("wg3_fused_ragged", 3, 40, 20, 3, 3, 18, -1, dw3, tr3, 1, false, 0, true);
    fails += run_wgrad("wg3_fused_128tiles", 16, 32, 32, 3, 3, 18, -1, dw3, tr3, 1, false, 0, true);
    fails += run_wgrad("wg3_fused_296tiles", 4, 96, 48, 3, 3, 18, -1, dw3, tr3, 1, false, 0, true);
    fails += run_wgrad("wg3_fused_cout256_ps", 2, 32, 16, 3, 3, 18, -1, dw3, tr3, 4, true, 0, true);
    fails += run_wgrad_batched("wgb_3layers_ragged", 3, 2, 40, 20, 0);
    fails += run_wgrad_batched("wgb_5layers", 5, 4, 96, 48, 0);
    fails += run_wgrad_batched("wgb_1layer_tiny", 1, 1, 9, 5, 0);
    if (iters > 0) fails += run_wgrad_batched("perf_wgb_trunk_33x16x96x96", 33, 16, 96, 96, iters / 10 > 0 ? iters / 10 : 1);
    const int dw1[1] = {0}, tr5[5] = {0, 2, 4, 6, 8};
    fails += run_wgrad("wg9_pairs", 2, 32, 16, 1, 5, 24, -3, dw1, tr5, 1, false, 0);
    if (iters > 0) {
      fails += run_wgrad("perf_wg_trunk_16x96x96", 16, 96, 96, 3, 3, 18, -1, dw3, tr3, 1, false, iters);
      fails += run_wgrad("perf_wg3_trunk_16x96x96", 16, 96, 96, 3, 3, 18, -1, dw3, tr3, 1, false, iters, true);
      fails += run_wgrad("perf_wg3_up3_16x192x192", 16, 192, 192, 3, 3, 18, -1, dw3, tr3, 4, true, iters, true);
      fails += run_wgrad("perf_wg_up3_16x192x192", 16, 192, 192, 3, 3, 18, -1, dw3, tr3, 4, true, iters);
    }
  }
  {  // 1x1 "plain GEMM" sanity: one strip, one tap
    Problem p = conv3x3("gemm1x1", 1, 16, 8, 64, false);
    p.n_strips = 1; p.n_taps = 1; p.strip_rows = 16; p.strip_dh = 0; p.strip_dw[0] = 0; p.tap_row[0] = 0;
    p.bias = false;
    fails += run(p, 0);
  }
  fails += run(conv3x3("c3x3_small", 2, 32, 24, 64, false), 0);
  fails += run(conv3x3("c3x3_ragged", 3, 40, 20, 64, false), 0);
  {
    Problem p = conv3x3("c3x3_lrelu_res", 2, 32, 16, 64, false);
    p.act = ACT_LRELU; p.residual = true;
    fails += run(p, 0);
    Problem m = conv3x3("c3x3_mask_ragged", 2, 24, 20, 64, false);
    m.mask = true;
    fails += run(m, 0);
  }
  {
    Problem p = conv3x3("c3x3_relu_ps", 2, 32, 16, 256, true);
    p.act = ACT_RELU;
    fails += run(p, 0);
  }
  {  // Cin = 256 through four strided pixel-shuffle views, weights streamed
    Problem p = conv3x3("c3x3_cin256_views", 2, 32, 16, 64, false);
    p.n_views = 4; p.strided_views = true;
    fails += run(p, 0);
  }
  {  // 9x9-as-5-row-pairs on a 64-channel unfolded buffer
    Problem p = conv3x3("c9_pairs", 2, 32, 16, 64, false);
    p.n_strips = 1; p.n_taps = 5; p.strip_rows = 16 + 8; p.strip_dh = -3; p.strip_dw[0] = 0;
    for (int r = 0; r < 5; ++r) p.tap_row[r] = 2 * r;
    p.act = ACT_LRELU;
    fails += run(p, 0);
  }
  {  // conv3: 9x9, Cout=3, horizontal taps folded into N=27(+5)
    Problem p = conv3x3("fold9", 2, 24, 56, 32, false);
    p.TH = 4; p.TW = 32;
    p.n_strips = 1; p.n_taps = 9; p.strip_rows = 4 + 8; p.strip_dh = -4; p.strip_dw[0] = 0;
    for (int r = 0; r < 9; ++r) p.tap_row[r] = r;
    p.block_n = 32; p.out_mode = OUT_FOLD9_NCHW;
    fails += run(p, 0);
  }
  {  // conv3 through conv9_rows (one image row per MMA, up to 8 output rows per MMA)
    const int geo[5][3] = {{2, 24, 56}, {3, 37, 130}, {1, 5, 7}, {2, 8, 120}, {1, 19, 245}};
    for (int g = 0; g < 5; ++g) {
      Problem p = conv3x3("c9rows", geo[g][0], geo[g][1], geo[g][2], 32, false);
      p.TH = 4; p.TW = 32;
      p.n_strips = 1; p.n_taps = 9; p.strip_rows = 4 + 8; p.strip_dh = -4; p.strip_dw[0] = 0;
      for (int r = 0; r < 9; ++r) p.tap_row[r] = r;
      p.block_n = 32; p.out_mode = OUT_FOLD9_NCHW; p.variant = 0;
      fails += run(p, 0);
    }
  }
  {  // row-interleaved 3x3 kernel (conv3_il)
    const int var = 0;
    printf("-- conv3_il\n");
    Problem p = conv3x3("il_small", 2, 32, 24, 64, false); p.variant = var; fails += run(p, 0);
    Problem r = conv3x3("il_ragged", 3, 40, 20, 64, false); r.variant = var; fails += run(r, 0);
    Problem o = conv3x3("il_odd_rows", 2, 37, 13, 64, false); o.variant = var; o.act = ACT_RELU; fails += run(o, 0);
    Problem q = conv3x3("il_ragged_res", 3, 37, 20, 64, false); q.variant = var; q.residual = true; q.act = ACT_LRELU; fails += run(q, 0);
    Problem m = conv3x3("il_mask_ragged", 2, 24, 20, 64, false); m.variant = var; m.mask = true; fails += run(m, 0);
    Problem u = conv3x3("il_relu_ps", 2, 30, 16, 256, true); u.variant = var; u.act = ACT_RELU; fails += run(u, 0);
    Problem t = conv3x3("il_many_tiles", 5, 96, 96, 64, false); t.variant = var; t.residual = true; fails += run(t, 0);
  }
  if (iters > 0) {
    {
      const int var = 0;
      printf("-- conv3_il\n");
      { Problem p = conv3x3("perf_il_trunk_16x96x96", 16, 96, 96, 64, false); p.variant = var; fails += run(p, iters); }
      { Problem p = conv3x3("perf_il_trunk_stats", 16, 96, 96, 64, false); p.variant = var; p.stats = true; fails += run(p, iters); }
      { Problem p = conv3x3("perf_il_trunk_mask", 16, 96, 96, 64, false); p.variant = var; p.mask = true; p.bias = false; fails += run(p, iters); }
      { Problem p = conv3x3("perf_il_trunk_residual", 16, 96, 96, 64, false); p.variant = var; p.residual = true; p.bias = false; fails += run(p, iters); }
      { Problem p = conv3x3("perf_il_up3_16x192x192", 16, 192, 192, 256, true); p.variant = var; p.act = ACT_RELU; fails += run(p, iters); }
    }
    fails += run(conv3x3("perf_trunk_16x96x96", 16, 96, 96, 64, false), iters);
    { Problem p = conv3x3("perf_trunk_stats", 16, 96, 96, 64, false); p.stats = true; fails += run(p, iters); }
    { Problem p = conv3x3("perf_trunk_mask", 16, 96, 96, 64, false); p.mask = true; p.bias = false; fails += run(p, iters); }
    { Problem p = conv3x3("perf_trunk_residual", 16, 96, 96, 64, false); p.residual = true; p.bias = false; fails += run(p, iters); }
    Problem p = conv3x3("perf_up3_16x192x192", 16, 192, 192, 256, true);
    p.act = ACT_RELU;
    fails += run(p, iters);
    {
      Problem f = conv3x3("perf_c9rows_16x384x384", 16, 384, 384, 32, false);
      f.TH = 4; f.TW = 32; f.n_strips = 1; f.n_taps = 9; f.strip_rows = 12; f.strip_dh = -4; f.strip_dw[0] = 0;
      for (int r = 0; r < 9; ++r) f.tap_row[r] = r;
      f.block_n = 32; f.out_mode = OUT_FOLD9_NCHW; f.variant = 0;
      fails += run(f, iters);
    }
    Problem f = conv3x3("perf_fold9_16x384x384", 16, 384, 384, 32, false);
    f.TH = 4; f.TW = 32; f.n_strips = 1; f.n_taps = 9; f.strip_rows = 12; f.strip_dh = -4; f.strip_dw[0] = 0;
    for (int r = 0; r < 9; ++r) f.tap_row[r] = r;
    f.block_n = 32; f.out_mode = OUT_FOLD9_NCHW;
    fails += run(f, iters);
  }
  printf("PROBE %s (%d failing cases)\n", fails == 0 ? "PASS" : "FAIL", fails);
  return fails == 0 ? 0 : 1;
}
