// Discriminator engine (reference: src/models.py:90-120).
//
// Strided convolutions run on the same tcgen05 strip implicit-GEMM kernel as the generator by re-expressing them as
// stride-1 convolutions over a space-to-depth operand:
//   * stage 0 (8x8, stride 2, pad 2, 3->64): the image is unfolded to U0[h'][w'][(v,a,b,c)] = x[c][2h'+a-2][2(w'+v)+b-2]
//     (48 of 64 channels used); the conv becomes 4 vertical taps u over U0 with K = 64 per tap, kh = 2u+a, kw = 2v+b.
//   * stages 1-3 (4x4, stride 2, pad 1, C->2C): the previous stage writes its activation directly in padded
//     space-to-depth layout XS[h'][w'][(a,b,c)] = z[2h'+a-1][2w'+b-1][c]; the conv becomes a dense 2x2 stride-1 conv over
//     4C channels (kh = 2u+a, kw = 2v+b), K = 16C.
// Conv outputs stay fp32 (the per-sample InstanceNorm over as few as 3 elements amplifies rounding); MaxPool(3,2),
// InstanceNorm (biased variance, eps 1e-5, no affine) and LeakyReLU(0.2)/Sigmoid are three HBM-bound passes:
// pool+statistics, finalize, apply(+space-to-depth store).  All reductions use fixed-order partials (deterministic).
#include "discriminator.cuh"

#include <cuda_bf16.h>
#include <stdio.h>
#include <string.h>

#include "conv_gemm.cuh"
#include "elementwise.cuh"

namespace srg {

namespace {

constexpr float kEps = 1e-5f;
constexpr float kSlope = 0.2f;
constexpr int kChunksMax = 128;   // pooled-pixel chunks per image in the statistics kernels

#define D_LAUNCH_CHECK(name)                                                      \
  do {                                                                            \
    cudaError_t e_ = cudaGetLastError();                                          \
    if (e_ != cudaSuccess) {                                                      \
      set_error("%s launch: %s", name, cudaGetErrorString(e_));                   \
      return int(e_);                                                             \
    }                                                                             \
    count_launch();                                                               \
  } while (0)
#define RC(x)                  \
  do {                         \
    int rc_ = (x);             \
    if (rc_ != 0) return rc_;  \
  } while (0)

__device__ __forceinline__ uint32_t bpack2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float blo2(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bhi2(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

int ew_grid(int64_t items) {
  int64_t b = (items + 255) / 256;
  if (b > 148 * 16) b = 148 * 16;
  if (b < 1) b = 1;
  return int(b);
}

// ------------------------------------------------------------------------------------------------ stage-0 unfold
// U0[n][h'][w'][ch], ch = ((v*2+a)*2+b)*3+c  <-  x[n][c][2h'+a-2][2(w'+v)+b-2]   (zero outside / ch >= 48)
// The 12 values of column pair j = w'+v, T[j] = {x[c][2h'+a-2][2j-2+b]}, are shared by four neighbouring pixels
// (pixel w' = [T[w'], T[w'+1], T[w'+2], T[w'+3], 16 zeros]).  One block per (n, h'): phase 1 builds T for the whole row in
// shared memory (coalesced reads along the image row, 24 bytes of bf16 per j), phase 2 writes the output row as
// consecutive 16-byte vectors copied from 96 contiguous shared-memory bytes per pixel.
__global__ void __launch_bounds__(256) d_unfold0_kernel(const float* __restrict__ x, int N, int H, int W, int Hs, int Ws,
                                                        uint4* __restrict__ dst) {
  extern __shared__ uint2 sT[];                 // [(Ws + 3)][3] uint2 = 12 bf16 per column pair
  const int hq = blockIdx.x % Hs, n = blockIdx.x / Hs;
  const int64_t plane = int64_t(H) * W;
  const float* xn = x + int64_t(n) * 3 * plane;
  for (int j = threadIdx.x; j < Ws + 3; j += blockDim.x) {
    float f[12];
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int yy = 2 * hq + a - 2;
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        const int xx = 2 * j - 2 + b;
        const bool ok = yy >= 0 && yy < H && xx >= 0 && xx < W;
#pragma unroll
        for (int c = 0; c < 3; ++c) f[a * 6 + b * 3 + c] = ok ? __ldg(xn + c * plane + int64_t(yy) * W + xx) : 0.f;
      }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) sT[j * 3 + k] = make_uint2(bpack2(f[4 * k], f[4 * k + 1]), bpack2(f[4 * k + 2], f[4 * k + 3]));
  }
  __syncthreads();
  uint4* row = dst + (int64_t(n) * Hs + hq) * Ws * 8;
  for (int u = threadIdx.x; u < Ws * 8; u += blockDim.x) {
    const int wq = u >> 3, k = u & 7;
    uint4 o = make_uint4(0u, 0u, 0u, 0u);
    if (k < 6) {
      const uint2 lo = sT[wq * 3 + 2 * k], hi = sT[wq * 3 + 2 * k + 1];     // bytes 24*wq + 16*k .. + 16
      o = make_uint4(lo.x, lo.y, hi.x, hi.y);
    }
    row[u] = o;
  }
}
// dx[n][c][y][x] = sum_v dU0[n][(y+2)>>1][((x+2)>>1) - v][ch(v, (y+2)&1, (x+2)&1, c)]
__global__ void __launch_bounds__(256) d_fold0_kernel(const __nv_bfloat16* __restrict__ dU, int N, int H, int W, int Hs, int Ws,
                                                      float* __restrict__ dx) {
  const int64_t total = int64_t(N) * 3 * H * W;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int xx = int(i % W);
    int64_t t = i / W;
    const int yy = int(t % H);
    t /= H;
    const int c = int(t % 3);
    const int n = int(t / 3);
    const int hq = (yy + 2) >> 1, a = (yy + 2) & 1, b = (xx + 2) & 1, wsum = (xx + 2) >> 1;
    float acc = 0.f;
    if (hq < Hs) {
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int wq = wsum - v;
        if (wq >= 0 && wq < Ws) {
          const int ch = ((v * 2 + a) * 2 + b) * 3 + c;
          acc += __bfloat162float(dU[((int64_t(n) * Hs + hq) * Ws + wq) * 64 + ch]);
        }
      }
    }
    dx[i] = acc;
  }
}

// ------------------------------------------------------------------------------------------------ pool + statistics
// Pooled value of window (0, 0) (y = &Y[n][0][0][c]), same scan as the pool in d_stats_kernel.  Out of line: inlined,
// it changes how the compiler schedules the pool loop's loads, and that loop runs a third slower.
__device__ __noinline__ float d_pool_first(const float* __restrict__ y, int Wo, int C) {
  float best = y[0];
#pragma unroll
  for (int k = 1; k < 9; ++k) {
    const float v = y[(int64_t(k / 3) * Wo + (k % 3)) * C];
    if (v > best) best = v;
  }
  return best;
}
// One block = one chunk of pooled pixels of one image.  Threads: channel-fastest.  partials[n][chunk][2][C].
// MODE 0 sums p - k and (p - k)^2 with k = p[n][0][0][c], one element of the map: a one-pass variance of shifted
// values keeps its rounding error proportional to the spread of p instead of to mean^2, which matters when an
// InstanceNorm map is nearly constant or has 2-4 elements (var << mean^2, at or below eps).  The shift must be an
// element of the map: the conv output at pixel (0, 0), for one, can sit far from a 3-element map's values.
template <int MODE>  // 0: max-pool Y -> P, idx ; sums p - k, (p - k)^2.   1: backward: g = dz * act'(xhat) ; sums g, g*xhat
__global__ void __launch_bounds__(256) d_stats_kernel(const float* __restrict__ Y, int Ho, int Wo, int Hp, int Wp, int C,
                                                      float* __restrict__ P, uint8_t* __restrict__ idx,
                                                      const float* __restrict__ stats, const void* __restrict__ dz_src,
                                                      int dz_mode, int Hs2, int Ws2, float* __restrict__ G,
                                                      int chunks, float* __restrict__ partials) {
  extern __shared__ float red[];      // [lanes][2][Ceff] with Ceff = min(C, 256)
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int npix = Hp * Wp;
  const int per = (npix + chunks - 1) / chunks;
  const int p0 = chunk * per, p1 = min(npix, p0 + per);
  const int Ceff = C < 256 ? C : 256;
  const int lanes = 256 / Ceff;
  const int lane = threadIdx.x / Ceff, cl = threadIdx.x % Ceff;
  for (int cbase = 0; cbase < C; cbase += 256) {
    const int c = cbase + cl;
    float s1 = 0.f, s2 = 0.f;
    float mean = 0.f, inv = 0.f, shift = 0.f;
    if (MODE == 0) shift = d_pool_first(Y + int64_t(n) * Ho * Wo * C + c, Wo, C);
    if (MODE == 1) { mean = stats[(int64_t(n) * C + c) * 2]; inv = stats[(int64_t(n) * C + c) * 2 + 1]; }
    for (int pp = p0 + lane; pp < p1; pp += lanes) {
      const int hp = pp / Wp, wp = pp - hp * Wp;
      const int64_t po = (int64_t(n) * npix + pp) * C + c;
      if (MODE == 0) {
        // MaxPool2d(3, 2): first maximum in (kh, kw) scan order wins (strict >), as in ATen
        const float* y = Y + ((int64_t(n) * Ho + 2 * hp) * Wo + 2 * wp) * C + c;
        float best = y[0];
        int bi = 0;
#pragma unroll
        for (int k = 1; k < 9; ++k) {
          const float v = y[(int64_t(k / 3) * Wo + (k % 3)) * C];
          if (v > best) { best = v; bi = k; }
        }
        P[po] = best;
        idx[po] = uint8_t(bi);
        const float q = best - shift;
        s1 += q;
        s2 += q * q;
      } else {
        const float xhat = (P[po] - mean) * inv;
        float dz, d;
        if (dz_mode == 0) {        // last stage: dOut is fp32 NCHW, activation = sigmoid
          dz = reinterpret_cast<const float*>(dz_src)[(int64_t(n) * C + c) * npix + pp];
          const float s = 1.f / (1.f + __expf(-xhat));
          d = s * (1.f - s);
        } else {                   // dz lives in the next stage's space-to-depth gradient tensor (bf16), LeakyReLU
          const int hq = (hp + 1) >> 1, wq = (wp + 1) >> 1;
          dz = 0.f;
          if (hq < Hs2 && wq < Ws2) {
            const int ab = ((hp + 1) & 1) * 2 + ((wp + 1) & 1);
            dz = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(dz_src)[((int64_t(n) * Hs2 + hq) * Ws2 + wq) * (4 * C) + ab * C + c]);
          }
          d = xhat > 0.f ? 1.f : kSlope;
        }
        const float g = dz * d;
        G[po] = g;
        s1 += g;
        s2 += g * xhat;
      }
    }
    red[(lane * 2 + 0) * Ceff + cl] = s1;
    red[(lane * 2 + 1) * Ceff + cl] = s2;
    __syncthreads();
    if (lane == 0) {
      float a = 0.f, b = 0.f;
      for (int l = 0; l < lanes; ++l) { a += red[(l * 2 + 0) * Ceff + cl]; b += red[(l * 2 + 1) * Ceff + cl]; }
      float* dst = partials + ((int64_t(n) * chunks + chunk) * 2) * C;
      dst[c] = a;
      dst[C + c] = b;
    }
    __syncthreads();
  }
}
// stats[n][c] = (mean, inv_std)  (MODE 0, P = pooled map holding the shift k at pixel 0)
//           or  (sum g / cnt, sum g*xhat / cnt)  (MODE 1, P unused)
template <int MODE>
__global__ void d_finalize_kernel(const float* __restrict__ partials, int chunks, int C, int NC, double count,
                                  const float* __restrict__ P, int64_t npix, float* __restrict__ stats) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NC) return;
  const int n = i / C, c = i - n * C;
  const float shift = MODE == 0 ? __ldg(P + int64_t(n) * npix * C + c) : 0.f;   // issued ahead of the partial sums
  double a = 0.0, b = 0.0;
  for (int k = 0; k < chunks; ++k) {
    const float* src = partials + ((int64_t(n) * chunks + k) * 2) * C;
    a += double(src[c]);
    b += double(src[C + c]);
  }
  if (MODE == 0) {
    const double m = a / count;                 // mean of p - k
    double var = b / count - m * m;
    if (var < 0.0) var = 0.0;
    const double mean = double(shift) + m;
    stats[2 * i] = float(mean);
    stats[2 * i + 1] = float(1.0 / sqrt(var + double(kEps)));
  } else {
    stats[2 * i] = float(a / count);
    stats[2 * i + 1] = float(b / count);
  }
}
// z = act((p - mean) * inv) written as the next conv's operand XS[n][h'][w'][(a,b,c)] = z[2h'+a-1][2w'+b-1][c] (bf16)
__global__ void __launch_bounds__(256) d_apply_s2d_kernel(const float* __restrict__ P, const float* __restrict__ stats, int Hp,
                                                          int Wp, int C, int N, int Hs, int Ws, uint4* __restrict__ XS) {
  const int C4 = 4 * C, groups = C4 / 8;
  const int64_t total = int64_t(N) * Hs * Ws * groups;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int gq = int(i % groups);
    int64_t t = i / groups;
    const int wq = int(t % Ws);
    t /= Ws;
    const int hq = int(t % Hs);
    const int n = int(t / Hs);
    const int ch0 = gq * 8, ab = ch0 / C, c0 = ch0 - ab * C;
    const int hp = 2 * hq + (ab >> 1) - 1, wp = 2 * wq + (ab & 1) - 1;
    float f[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] = 0.f;
    if (hp >= 0 && hp < Hp && wp >= 0 && wp < Wp) {
      const float* p = P + ((int64_t(n) * Hp + hp) * Wp + wp) * C + c0;
      const float* s = stats + (int64_t(n) * C + c0) * 2;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float xhat = (p[e] - s[2 * e]) * s[2 * e + 1];
        f[e] = xhat > 0.f ? xhat : kSlope * xhat;
      }
    }
    uint4 o;
    o.x = bpack2(f[0], f[1]); o.y = bpack2(f[2], f[3]); o.z = bpack2(f[4], f[5]); o.w = bpack2(f[6], f[7]);
    XS[i] = o;
  }
}
// last stage: out[n][c][hp][wp] = sigmoid((p - mean) * inv), fp32 NCHW
__global__ void d_apply_sigmoid_kernel(const float* __restrict__ P, const float* __restrict__ stats, int npix, int C, int N,
                                       float* __restrict__ out) {
  const int64_t total = int64_t(N) * C * npix;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int pp = int(i % npix);
    const int64_t nc = i / npix;
    const int n = int(nc / C), c = int(nc - int64_t(n) * C);
    const float xhat = (P[(int64_t(n) * npix + pp) * C + c] - stats[2 * nc]) * stats[2 * nc + 1];
    out[i] = 1.f / (1.f + __expf(-xhat));
  }
}
// dY[n][ho][wo][c] (bf16) = sum over pooled windows (hp, wp) containing (ho, wo) whose argmax is (ho, wo) of
//   inv * (g - c1 - xhat * c2)         (InstanceNorm backward + MaxPool backward, gather form: no atomics)
// One thread = a 2x2 block of outputs x 8 channels: the four pooling windows (hp in {i-1, i}, wp in {j-1, j}) that can
// route into it are read ONCE (9 window reads per block in the one-output-per-thread form), every argmax code is
// decoded to its target inside the block.
__global__ void __launch_bounds__(256) d_pool_bwd_kernel(const float* __restrict__ G, const float* __restrict__ P,
                                                         const uint8_t* __restrict__ idx, const float* __restrict__ stats,
                                                         const float* __restrict__ stats2, int Ho, int Wo, int Hp, int Wp,
                                                         int C, int N, uint4* __restrict__ dY) {
  const int groups = C / 8;
  const int Hb = (Ho + 1) / 2, Wb = (Wo + 1) / 2;
  const int64_t total = int64_t(N) * Hb * Wb * groups;
  for (int64_t t0 = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t0 < total; t0 += int64_t(gridDim.x) * blockDim.x) {
    const int gq = int(t0 % groups);
    int64_t t = t0 / groups;
    const int j = int(t % Wb);
    t /= Wb;
    const int i = int(t % Hb);
    const int n = int(t / Hb);
    const int c0 = gq * 8;
    float f[4][8];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int e = 0; e < 8; ++e) f[q][e] = 0.f;
    // per-(n, channel) statistics of this thread's 8 channels: {mean, inv} and {c1, c2} pairs, 128-bit loads
    const float4* s1 = reinterpret_cast<const float4*>(stats + (int64_t(n) * C + c0) * 2);
    const float4* s2 = reinterpret_cast<const float4*>(stats2 + (int64_t(n) * C + c0) * 2);
    float mean[8], inv[8], k1[8], k2[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 a = __ldg(s1 + q), b = __ldg(s2 + q);
      mean[2 * q] = a.x; inv[2 * q] = a.y; mean[2 * q + 1] = a.z; inv[2 * q + 1] = a.w;
      k1[2 * q] = b.x; k2[2 * q] = b.y; k1[2 * q + 1] = b.z; k2[2 * q + 1] = b.w;
    }
#pragma unroll
    for (int wi = 0; wi < 2; ++wi) {
      const int hp = i - 1 + wi;
      if (hp < 0 || hp >= Hp) continue;
#pragma unroll
      for (int wj = 0; wj < 2; ++wj) {
        const int wp = j - 1 + wj;
        if (wp < 0 || wp >= Wp) continue;
        const int64_t po = ((int64_t(n) * Hp + hp) * Wp + wp) * C + c0;
        const uint2 iv = *reinterpret_cast<const uint2*>(idx + po);           // 8 argmax codes r*3 + c (C % 8 == 0)
        // target inside the block: di = r - 2*(1 - wi), dj = c - 2*(1 - wj), both must be 0 or 1
        int tgt[8];
        bool any = false;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int code = int(((e < 4 ? iv.x : iv.y) >> (8 * (e & 3))) & 0xFFu);
          const int r = code / 3, c = code - 3 * r;
          const int di = r - 2 * (1 - wi), dj = c - 2 * (1 - wj);
          tgt[e] = (di >= 0 && di <= 1 && dj >= 0 && dj <= 1) ? di * 2 + dj : -1;
          any |= tgt[e] >= 0;
        }
        if (!any) continue;
        const float4 p0 = *reinterpret_cast<const float4*>(P + po), p1 = *reinterpret_cast<const float4*>(P + po + 4);
        const float4 g0 = *reinterpret_cast<const float4*>(G + po), g1 = *reinterpret_cast<const float4*>(G + po + 4);
        const float pv[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
        const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float xhat = (pv[e] - mean[e]) * inv[e];
          const float val = inv[e] * (gv[e] - k1[e] - xhat * k2[e]);
#pragma unroll
          for (int q = 0; q < 4; ++q) f[q][e] += (tgt[e] == q) ? val : 0.f;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int ho = 2 * i + (q >> 1), wo = 2 * j + (q & 1);
      if (ho < Ho && wo < Wo) {
        uint4 o;
        o.x = bpack2(f[q][0], f[q][1]); o.y = bpack2(f[q][2], f[q][3]); o.z = bpack2(f[q][4], f[q][5]); o.w = bpack2(f[q][6], f[q][7]);
        dY[((int64_t(n) * Ho + ho) * Wo + wo) * groups + gq] = o;
      }
    }
  }
}
// per-channel sums of a bf16 [pixels][C] tensor: partials[block][C], then out[c] = sum over blocks (fixed order)
__global__ void __launch_bounds__(256) d_chan_sum_kernel(const __nv_bfloat16* __restrict__ x, int64_t pixels, int C,
                                                         float* __restrict__ partials) {
  extern __shared__ float red[];
  const int Ceff = C < 256 ? C : 256;
  const int lanes = 256 / Ceff;
  const int lane = threadIdx.x / Ceff, cl = threadIdx.x % Ceff;
  for (int cbase = 0; cbase < C; cbase += 256) {
    const int c = cbase + cl;
    float s = 0.f;
    for (int64_t p = int64_t(blockIdx.x) * lanes + lane; p < pixels; p += int64_t(gridDim.x) * lanes)
      s += __bfloat162float(x[p * C + c]);
    red[lane * Ceff + cl] = s;
    __syncthreads();
    if (lane == 0) {
      float a = 0.f;
      for (int l = 0; l < lanes; ++l) a += red[l * Ceff + cl];
      partials[int64_t(blockIdx.x) * C + c] = a;
    }
    __syncthreads();
  }
}
__global__ void d_chan_sum_final_kernel(const float* __restrict__ partials, int blocks, int C, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double a = 0.0;
  for (int b = 0; b < blocks; ++b) a += double(partials[int64_t(b) * C + c]);
  out[c] = float(a);
}
// Sums the wgrad split-K partials of one launch (input-channel chunk `chunk`, output-channel group `grp`) straight into
// the OIHW gradient.  Partial layout (wgrad_gemm.cu): [split][nb][pair][128 = (t&1)*64 + row][64 = col], t = v*R + u.
__global__ void d_wgrad_reduce_kernel(const float* __restrict__ partials, int splits, size_t split_stride, int n_blocks,
                                      int n_pairs, int n_taps_total, int stage0, int Cin, int K, int chunk, int grp,
                                      float* __restrict__ dW) {
  const int total = n_blocks * n_taps_total * 64 * 64;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int col = e & 63, row = (e >> 6) & 63;
  const int t = (e >> 12) % n_taps_total, nb = (e >> 12) / n_taps_total;
  const float* p = partials + ((size_t(nb) * n_pairs + t / 2) * 128 + (t & 1) * 64 + row) * 64 + col;
  float acc = 0.f;
  for (int s = 0; s < splits; ++s) acc += p[size_t(s) * split_stride];
  const int co = (grp * n_blocks + nb) * 64 + col;
  int cin, kh, kw;
  if (stage0) {          // row = ((v*2+a)*2+b)*3+c, tap t = u
    if (row >= 48) return;
    const int v = row / 12, rem = row - v * 12, a = rem / 6, b = (rem % 6) / 3;
    cin = rem % 3; kh = 2 * t + a; kw = 2 * v + b;
  } else {               // ch' = chunk*64+row = (a*2+b)*Cin + cin, tap t = v*2+u
    const int ch = chunk * 64 + row, ab = ch / Cin;
    cin = ch - ab * Cin;
    const int v = t >> 1, u = t & 1;
    kh = 2 * u + (ab >> 1); kw = 2 * v + (ab & 1);
  }
  dW[((size_t(co) * Cin + cin) * K + kh) * K + kw] = acc;
}

struct Carver {
  size_t off = 0;
  size_t take(size_t bytes) { const size_t o = off; off += (bytes + 1023) & ~size_t(1023); return o; }
};

struct DLayout {
  size_t packed, partials, stats2, wg_partials;
  size_t X[4], Y[4], P[4], idx[4], stats[4];
  size_t G, dY[4], dX[4];
  size_t total;
};

struct DImpl : DiscriminatorEngine {
  DLayout L;
  std::vector<int> h_pack_idx;
  int64_t pk_f[4], pk_d[4];
};

int stat_chunks(const DiscStage& s) {
  int c = (s.Hp * s.Wp + 63) / 64;
  if (c > kChunksMax) c = kChunksMax;
  if (c < 1) c = 1;
  return c;
}

DLayout make_layout(const DImpl& e, bool training) {
  DLayout L;
  memset(&L, 0, sizeof(L));
  Carver c;
  L.packed = c.take(size_t(e.packed_elems) * 2);
  L.partials = c.take(size_t(e.N) * kChunksMax * 2 * 512 * 4 > size_t(2048) * 512 * 4 ? size_t(e.N) * kChunksMax * 2 * 512 * 4
                                                                                        : size_t(2048) * 512 * 4);
  L.stats2 = c.take(size_t(e.N) * 512 * 2 * 4);
  size_t gmax = 0;
  for (int l = 0; l < 4; ++l) {
    const DiscStage& s = e.st[l];
    L.X[l] = c.take(size_t(e.N) * s.Hs * s.Ws * s.Cs * 2);
    L.Y[l] = c.take(size_t(e.N) * s.Ho * s.Wo * s.Cout * 4);
    L.P[l] = c.take(size_t(e.N) * s.Hp * s.Wp * s.Cout * 4);
    L.idx[l] = c.take(size_t(e.N) * s.Hp * s.Wp * s.Cout);
    L.stats[l] = c.take(size_t(e.N) * s.Cout * 2 * 4);
    const size_t g = size_t(e.N) * s.Hp * s.Wp * s.Cout * 4;
    if (g > gmax) gmax = g;
  }
  if (training) {
    L.wg_partials = c.take(size_t(148) * 2 * 8192 * 4);
    L.G = c.take(gmax);
    for (int l = 0; l < 4; ++l) {
      const DiscStage& s = e.st[l];
      L.dY[l] = c.take(size_t(e.N) * s.Ho * s.Wo * s.Cout * 2);
      L.dX[l] = c.take(size_t(e.N) * s.Hs * s.Ws * s.Cs * 2);
    }
  }
  L.total = c.off;
  return L;
}

inline int widx(int64_t base, int Cin, int K, int co, int ci, int kh, int kw) {
  return int(base + ((int64_t(co) * Cin + ci) * K + kh) * K + kw);
}

InView view_of(const void* ptr, int H, int W, int Ctot, int c0, int channels) {
  InView v;
  v.ptr = reinterpret_cast<const uint16_t*>(ptr) + c0;
  v.stride_w = Ctot; v.stride_h = int64_t(W) * Ctot; v.stride_n = int64_t(H) * W * Ctot; v.channels = channels;
  return v;
}

}  // namespace

DiscriminatorEngine::~DiscriminatorEngine() { cudaFree(d_pack_idx); }

DiscriminatorEngine* discriminator_create(int N, int H, int W) {
  if (N < 1 || H < 1 || W < 1) { set_error("discriminator_create: bad geometry"); return nullptr; }
  DImpl* e = new DImpl();
  e->N = N; e->H = H; e->W = W;
  const int chans[5] = {3, 64, 128, 256, 512};
  int hin = H, win = W;
  for (int l = 0; l < 4; ++l) {
    DiscStage& s = e->st[l];
    s.Cin = chans[l]; s.Cout = chans[l + 1]; s.Hin = hin; s.Win = win;
    const int k = l == 0 ? 8 : 4, pad = l == 0 ? 2 : 1;
    s.Ho = (hin + 2 * pad - k) / 2 + 1;
    s.Wo = (win + 2 * pad - k) / 2 + 1;
    if (hin + 2 * pad < k || win + 2 * pad < k || s.Ho < 3 || s.Wo < 3) {
      // same condition the reference trips over inside MaxPool2d(3, 2) (SURVEY Appendix E)
      set_error("Discriminator input too small: stage %d conv output %dx%d cannot be max-pooled with a 3x3 window", l,
                s.Ho, s.Wo);
      delete e;
      return nullptr;
    }
    s.Hp = (s.Ho - 3) / 2 + 1;
    s.Wp = (s.Wo - 3) / 2 + 1;
    if (l == 0) { s.Hs = s.Ho + 3; s.Ws = s.Wo; s.Cs = 64; }
    else { s.Hs = s.Ho + 1; s.Ws = s.Wo + 1; s.Cs = 4 * s.Cin; }
    hin = s.Hp; win = s.Wp;
  }
  if (e->st[3].Hp * e->st[3].Wp <= 1) {
    set_error("Discriminator input too small: InstanceNorm expects more than 1 spatial element (got %dx%d)", e->st[3].Hp,
              e->st[3].Wp);
    delete e;
    return nullptr;
  }
  // parameters in registration order (src/models.py:93-114): model.0, model.4, model.8, model.12
  const int midx[4] = {0, 4, 8, 12};
  char nm[64];
  for (int l = 0; l < 4; ++l) {
    const int k = l == 0 ? 8 : 4;
    ParamInfo w;
    snprintf(nm, sizeof(nm), "model.%d.weight", midx[l]);
    w.name = nm; w.ndim = 4; w.shape[0] = chans[l + 1]; w.shape[1] = chans[l]; w.shape[2] = k; w.shape[3] = k;
    w.numel = int64_t(chans[l + 1]) * chans[l] * k * k; w.offset = e->param_elems;
    e->param_elems += (w.numel + 3) & ~int64_t(3);
    e->params.push_back(w);
    ParamInfo b;
    snprintf(nm, sizeof(nm), "model.%d.bias", midx[l]);
    b.name = nm; b.ndim = 1; b.shape[0] = chans[l + 1]; b.shape[1] = b.shape[2] = b.shape[3] = 1;
    b.numel = chans[l + 1]; b.offset = e->param_elems;
    e->param_elems += (b.numel + 3) & ~int64_t(3);
    e->params.push_back(b);
  }
  // ---- pack maps (bf16 GEMM operands, k-block order ((chunk*S + s)*R + r), rows = GEMM n, 64 k per row)
  std::vector<int>& idx = e->h_pack_idx;
  for (int l = 0; l < 4; ++l) {
    const int Cin = chans[l], Cout = chans[l + 1];
    const int64_t base = e->params[size_t(2 * l)].offset;
    e->pk_f[l] = int64_t(idx.size());
    if (l == 0) {
      for (int u = 0; u < 4; ++u)               // taps r = u (rows), one strip
        for (int co = 0; co < 64; ++co)
          for (int ch = 0; ch < 64; ++ch) {
            int val = -1;
            if (ch < 48) {
              const int v = ch / 12, rem = ch % 12, a = rem / 6, b = (rem % 6) / 3, c = rem % 3;
              val = widx(base, 3, 8, co, c, 2 * u + a, 2 * v + b);
            }
            idx.push_back(val);
          }
    } else {
      const int chunks = 4 * Cin / 64;
      for (int c = 0; c < chunks; ++c)
        for (int s = 0; s < 2; ++s)             // strip s = v (column shift +v)
          for (int r = 0; r < 2; ++r)           // tap r = u (row shift +u)
            for (int co = 0; co < Cout; ++co)
              for (int k = 0; k < 64; ++k) {
                const int ch = c * 64 + k, ab = ch / Cin, cin = ch % Cin;
                idx.push_back(widx(base, Cin, 4, co, cin, 2 * r + (ab >> 1), 2 * s + (ab & 1)));
              }
    }
    // data gradient: GEMM n = operand channel ch', k = output channel co
    e->pk_d[l] = int64_t(idx.size());
    if (l == 0) {
      for (int u = 0; u < 4; ++u)
        for (int ch = 0; ch < 64; ++ch)
          for (int co = 0; co < 64; ++co) {
            int val = -1;
            if (ch < 48) {
              const int v = ch / 12, rem = ch % 12, a = rem / 6, b = (rem % 6) / 3, c = rem % 3;
              val = widx(base, 3, 8, co, c, 2 * u + a, 2 * v + b);
            }
            idx.push_back(val);
          }
    } else {
      const int chunks = Cout / 64;
      for (int c = 0; c < chunks; ++c)
        for (int s = 0; s < 2; ++s)             // strip s: column shift -v, v = s
          for (int r = 0; r < 2; ++r)           // tap r: row shift -u, u = r
            for (int ch = 0; ch < 4 * Cin; ++ch)
              for (int k = 0; k < 64; ++k) {
                const int co = c * 64 + k, ab = ch / Cin, cin = ch % Cin;
                idx.push_back(widx(base, Cin, 4, co, cin, 2 * r + (ab >> 1), 2 * s + (ab & 1)));
              }
    }
  }
  e->packed_elems = int64_t(idx.size());
  e->workspace_bytes_train = make_layout(*e, true).total;
  e->workspace_bytes_eval = make_layout(*e, false).total;
  return e;
}

int discriminator_bind(DiscriminatorEngine* d, float* master, float* grads, void* ws, size_t ws_bytes, int training) {
  DImpl* e = static_cast<DImpl*>(d);
  const size_t need = training ? e->workspace_bytes_train : e->workspace_bytes_eval;
  if (ws_bytes < need) { set_error("discriminator_bind: workspace too small (%zu < %zu)", ws_bytes, need); return -20; }
  if ((reinterpret_cast<uintptr_t>(ws) & 1023) != 0) { set_error("discriminator_bind: workspace must be 1024-byte aligned"); return -21; }
  if (master == nullptr || (training && grads == nullptr)) { set_error("discriminator_bind: null buffer"); return -22; }
  if (e->d_pack_idx == nullptr) {
    if (cudaMalloc(&e->d_pack_idx, e->h_pack_idx.size() * sizeof(int)) != cudaSuccess ||
        cudaMemcpy(e->d_pack_idx, e->h_pack_idx.data(), e->h_pack_idx.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
      set_error("discriminator_bind: index map upload failed: %s", cudaGetErrorString(cudaGetLastError()));
      return -29;
    }
  }
  e->master = master; e->grads = grads;
  e->ws = reinterpret_cast<uint8_t*>(ws); e->ws_bytes = ws_bytes; e->ws_training = training != 0;
  e->L = make_layout(*e, training != 0);
  e->tensors.clear();
  auto reg = [&](const char* fmt, int l, size_t off, int n, int h, int w, int c, int dtype) {
    char nm[48];
    snprintf(nm, sizeof(nm), fmt, l);
    TensorInfo t; t.name = nm; t.byte_offset = int64_t(off); t.dims[0] = n; t.dims[1] = h; t.dims[2] = w; t.dims[3] = c; t.dtype = dtype;
    e->tensors.push_back(t);
  };
  for (int l = 0; l < 4; ++l) {
    const DiscStage& s = e->st[l];
    reg("x%d", l, e->L.X[l], e->N, s.Hs, s.Ws, s.Cs, 0);
    reg("y%d", l, e->L.Y[l], e->N, s.Ho, s.Wo, s.Cout, 1);
    reg("p%d", l, e->L.P[l], e->N, s.Hp, s.Wp, s.Cout, 1);
    if (training) {
      reg("dy%d", l, e->L.dY[l], e->N, s.Ho, s.Wo, s.Cout, 0);
      reg("dx%d", l, e->L.dX[l], e->N, s.Hs, s.Ws, s.Cs, 0);
    }
  }
  return 0;
}

int discriminator_pack(DiscriminatorEngine* d, cudaStream_t st) {
  DImpl* e = static_cast<DImpl*>(d);
  if (!e->ws) { set_error("discriminator_pack: not bound"); return -23; }
  return launch_pack_bf16(e->master, e->d_pack_idx, e->ws + e->L.packed, e->packed_elems, st);
}

static void set_tile(ConvGemmArgs& a) { a.TH = 16; a.TW = 8; }

int discriminator_forward(DiscriminatorEngine* d, const float* x, float* out, int keep, cudaStream_t st) {
  DImpl* e = static_cast<DImpl*>(d);
  (void)keep;
  if (!e->ws) { set_error("discriminator_forward: not bound"); return -23; }
  const DLayout& L = e->L;
  uint8_t* ws = e->ws;
  const uint16_t* packed = reinterpret_cast<const uint16_t*>(ws + L.packed);
  const int N = e->N;
  float* partials = reinterpret_cast<float*>(ws + L.partials);
  {
    const DiscStage& s = e->st[0];
    d_unfold0_kernel<<<N * s.Hs, 256, size_t(s.Ws + 3) * 24, st>>>(x, N, e->H, e->W, s.Hs, s.Ws, reinterpret_cast<uint4*>(ws + L.X[0]));
    D_LAUNCH_CHECK("d_unfold0");
  }
  for (int l = 0; l < 4; ++l) {
    const DiscStage& s = e->st[l];
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = s.Ho; a.W = s.Wo; set_tile(a);
    a.n_views = 1; a.views[0] = view_of(ws + L.X[l], s.Hs, s.Ws, s.Cs, 0, s.Cs); a.in_H = s.Hs; a.in_W = s.Ws;
    if (l == 0) {
      a.n_strips = 1; a.strip_dw[0] = 0; a.n_taps = 4; a.strip_dh = 0; a.strip_rows = a.TH + 3;
      for (int r = 0; r < 4; ++r) a.tap_row[r] = r;
    } else {
      a.n_strips = 2; a.strip_dw[0] = 0; a.strip_dw[1] = 1; a.n_taps = 2; a.strip_dh = 0; a.strip_rows = a.TH + 1;
      a.tap_row[0] = 0; a.tap_row[1] = 1;
    }
    a.weights = packed + e->pk_f[l]; a.cout_total = s.Cout; a.block_n = 64;
    a.bias = e->master + e->params[size_t(2 * l + 1)].offset; a.act = ACT_NONE;
    a.out = ws + L.Y[l]; a.out_mode = OUT_NHWC_F32;
    RC(launch_conv_gemm(a, st));
    const int chunks = stat_chunks(s);
    const int Ceff = s.Cout < 256 ? s.Cout : 256;
    const size_t sh = size_t(256 / Ceff) * 2 * Ceff * 4;
    float* stats = reinterpret_cast<float*>(ws + L.stats[l]);
    d_stats_kernel<0><<<dim3(chunks, N), 256, sh, st>>>(reinterpret_cast<const float*>(ws + L.Y[l]), s.Ho, s.Wo, s.Hp, s.Wp,
                                                       s.Cout, reinterpret_cast<float*>(ws + L.P[l]), ws + L.idx[l], nullptr,
                                                       nullptr, 0, 0, 0, nullptr, chunks, partials);
    D_LAUNCH_CHECK("d_pool_stats");
    d_finalize_kernel<0><<<(N * s.Cout + 127) / 128, 128, 0, st>>>(partials, chunks, s.Cout, N * s.Cout,
                                                                   double(s.Hp) * s.Wp,
                                                                   reinterpret_cast<const float*>(ws + L.P[l]),
                                                                   int64_t(s.Hp) * s.Wp, stats);
    D_LAUNCH_CHECK("d_in_finalize");
    if (l < 3) {
      const DiscStage& nx = e->st[l + 1];
      const int64_t total = int64_t(N) * nx.Hs * nx.Ws * (nx.Cs / 8);
      d_apply_s2d_kernel<<<ew_grid(total), 256, 0, st>>>(reinterpret_cast<const float*>(ws + L.P[l]), stats, s.Hp, s.Wp, s.Cout,
                                                        N, nx.Hs, nx.Ws, reinterpret_cast<uint4*>(ws + L.X[l + 1]));
      D_LAUNCH_CHECK("d_apply_s2d");
    } else {
      const int64_t total = int64_t(N) * s.Cout * s.Hp * s.Wp;
      d_apply_sigmoid_kernel<<<ew_grid(total), 256, 0, st>>>(reinterpret_cast<const float*>(ws + L.P[l]), stats, s.Hp * s.Wp,
                                                            s.Cout, N, out);
      D_LAUNCH_CHECK("d_apply_sigmoid");
    }
    e->launches += 4;
  }
  return 0;
}

int discriminator_backward(DiscriminatorEngine* d, const float* dout, int param_grads, float* dx, cudaStream_t st) {
  DImpl* e = static_cast<DImpl*>(d);
  if (!e->ws || !e->ws_training) { set_error("discriminator_backward: needs a training-sized bound workspace"); return -25; }
  const DLayout& L = e->L;
  uint8_t* ws = e->ws;
  const uint16_t* packed = reinterpret_cast<const uint16_t*>(ws + L.packed);
  const int N = e->N;
  float* partials = reinterpret_cast<float*>(ws + L.partials);
  float* stats2 = reinterpret_cast<float*>(ws + L.stats2);
  float* wgp = reinterpret_cast<float*>(ws + L.wg_partials);
  if (param_grads && cudaMemsetAsync(e->grads, 0, size_t(e->param_elems) * 4, st) != cudaSuccess) {
    set_error("memset grads failed");
    return -26;
  }
  for (int l = 3; l >= 0; --l) {
    const DiscStage& s = e->st[l];
    const int chunks = stat_chunks(s);
    const int Ceff = s.Cout < 256 ? s.Cout : 256;
    const size_t sh = size_t(256 / Ceff) * 2 * Ceff * 4;
    const float* stats = reinterpret_cast<const float*>(ws + L.stats[l]);
    float* G = reinterpret_cast<float*>(ws + L.G);
    // ---- activation + InstanceNorm backward statistics
    const void* dz_src = l == 3 ? static_cast<const void*>(dout) : static_cast<const void*>(ws + L.dX[l + 1]);
    const int Hs2 = l == 3 ? 0 : e->st[l + 1].Hs, Ws2 = l == 3 ? 0 : e->st[l + 1].Ws;
    d_stats_kernel<1><<<dim3(chunks, N), 256, sh, st>>>(nullptr, s.Ho, s.Wo, s.Hp, s.Wp, s.Cout,
                                                       reinterpret_cast<float*>(ws + L.P[l]), nullptr, stats, dz_src,
                                                       l == 3 ? 0 : 1, Hs2, Ws2, G, chunks, partials);
    D_LAUNCH_CHECK("d_in_bwd_stats");
    d_finalize_kernel<1><<<(N * s.Cout + 127) / 128, 128, 0, st>>>(partials, chunks, s.Cout, N * s.Cout,
                                                                   double(s.Hp) * s.Wp, nullptr, 0, stats2);
    D_LAUNCH_CHECK("d_in_bwd_finalize");
    // ---- InstanceNorm + MaxPool backward -> d(conv output), bf16
    {
      const int64_t total = int64_t(N) * ((s.Ho + 1) / 2) * ((s.Wo + 1) / 2) * (s.Cout / 8);
      d_pool_bwd_kernel<<<ew_grid(total), 256, 0, st>>>(G, reinterpret_cast<const float*>(ws + L.P[l]), ws + L.idx[l], stats,
                                                       stats2, s.Ho, s.Wo, s.Hp, s.Wp, s.Cout, N,
                                                       reinterpret_cast<uint4*>(ws + L.dY[l]));
      D_LAUNCH_CHECK("d_pool_bwd");
    }
    e->launches += 3;
    if (param_grads) {
      // bias gradient
      const int64_t pixels = int64_t(N) * s.Ho * s.Wo;
      int blocks = int((pixels + 63) / 64);
      if (blocks > 1024) blocks = 1024;
      const size_t shb = size_t(256 / Ceff) * Ceff * 4;
      d_chan_sum_kernel<<<blocks, 256, shb, st>>>(reinterpret_cast<const __nv_bfloat16*>(ws + L.dY[l]), pixels, s.Cout, partials);
      D_LAUNCH_CHECK("d_chan_sum");
      d_chan_sum_final_kernel<<<(s.Cout + 127) / 128, 128, 0, st>>>(partials, blocks, s.Cout,
                                                                    e->grads + e->params[size_t(2 * l + 1)].offset);
      D_LAUNCH_CHECK("d_chan_sum_final");
      // weight gradient: one launch per (64-channel operand chunk, group of <= 4 output-channel blocks)
      const int in_chunks = s.Cs / 64;
      const int out_blocks = s.Cout / 64;
      const int per_grp = out_blocks < 4 ? out_blocks : 4;
      const int groups = out_blocks / per_grp;
      for (int c = 0; c < in_chunks; ++c)
        for (int g = 0; g < groups; ++g) {
          WgradArgs a; memset(&a, 0, sizeof(a));
          a.N = N; a.H = s.Ho; a.W = s.Wo; a.TH = 16; a.TW = 8;
          a.x = view_of(ws + L.X[l], s.Hs, s.Ws, s.Cs, c * 64, 64); a.in_H = s.Hs; a.in_W = s.Ws;
          a.dy_views = 1; a.dy[0] = view_of(ws + L.dY[l], s.Ho, s.Wo, s.Cout, g * per_grp * 64, per_grp * 64);
          a.n_blocks = per_grp;
          if (l == 0) {
            a.n_strips = 1; a.strip_dw[0] = 0; a.n_taps = 4; a.strip_dh = 0; a.strip_rows = 16 + 3;
            for (int r = 0; r < 4; ++r) a.tap_row[r] = r;
          } else {
            a.n_strips = 2; a.strip_dw[0] = 0; a.strip_dw[1] = 1; a.n_taps = 2; a.strip_dh = 0; a.strip_rows = 16 + 1;
            a.tap_row[0] = 0; a.tap_row[1] = 1;
          }
          a.partials = wgp;
          int splits = 0;
          const int floats = wgrad_partials_floats(a, &splits);
          if (size_t(floats) * 4 > size_t(148) * 2 * 8192 * 4) { set_error("discriminator wgrad partials exceed workspace"); return -27; }
          RC(launch_wgrad_gemm(a, st));
          const int total = per_grp * 4 * 64 * 64;
          d_wgrad_reduce_kernel<<<(total + 255) / 256, 256, 0, st>>>(wgp, splits, size_t(per_grp) * 2 * 128 * 64, per_grp, 2, 4,
                                                                    l == 0 ? 1 : 0, s.Cin, l == 0 ? 8 : 4, c, g,
                                                                    e->grads + e->params[size_t(2 * l)].offset);
          D_LAUNCH_CHECK("d_wgrad_reduce");
          e->launches += 2;
        }
      e->launches += 2;
    }
    // ---- data gradient into the operand layout of this stage
    if (l > 0 || dx != nullptr) {
      ConvGemmArgs a; memset(&a, 0, sizeof(a));
      a.N = N; a.H = s.Hs; a.W = s.Ws; set_tile(a);
      a.n_views = 1; a.views[0] = view_of(ws + L.dY[l], s.Ho, s.Wo, s.Cout, 0, s.Cout); a.in_H = s.Ho; a.in_W = s.Wo;
      if (l == 0) {
        a.n_strips = 1; a.strip_dw[0] = 0; a.n_taps = 4; a.strip_dh = -3; a.strip_rows = a.TH + 3;
        for (int r = 0; r < 4; ++r) a.tap_row[r] = 3 - r;
      } else {
        a.n_strips = 2; a.strip_dw[0] = 0; a.strip_dw[1] = -1; a.n_taps = 2; a.strip_dh = -1; a.strip_rows = a.TH + 1;
        a.tap_row[0] = 1; a.tap_row[1] = 0;
      }
      a.weights = packed + e->pk_d[l]; a.cout_total = s.Cs; a.block_n = 64;
      a.bias = nullptr; a.act = ACT_NONE; a.out = ws + L.dX[l]; a.out_mode = OUT_NHWC;
      RC(launch_conv_gemm(a, st));
      e->launches += 1;
    }
  }
  if (dx != nullptr) {
    const DiscStage& s = e->st[0];
    const int64_t total = int64_t(N) * 3 * e->H * e->W;
    d_fold0_kernel<<<ew_grid(total), 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(ws + L.dX[0]), N, e->H, e->W, s.Hs,
                                                  s.Ws, dx);
    D_LAUNCH_CHECK("d_fold0");
  }
  return 0;
}

}  // namespace srg
