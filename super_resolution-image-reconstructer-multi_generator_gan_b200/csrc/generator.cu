// SRResNet generator engine (reference: src/models.py:10-25, :44-87).  Host-side orchestration only: every FLOP is in
// conv_gemm.cu / wgrad_gemm.cu (tcgen05) or elementwise.cu (HBM-bound passes).
//
// Data layout: activations NHWC bf16, 64 channels per pixel; images NCHW fp32; parameters in ONE flat fp32 buffer in
// the reference's parameters() order (state_dict keys of SURVEY Appendix A), gradients in a flat buffer of the same
// layout; packed bf16 GEMM operands are re-derived from the fp32 master after every optimizer step (generator_pack).
#include "generator.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "conv_gemm.cuh"
#include "elementwise.cuh"
#include "peer_sync.cuh"
#include "trunk_fused.cuh"

namespace srg {

namespace {

constexpr float kBnEps = 1e-5f;
constexpr float kBnMomentum = 0.1f;
constexpr float kSlope = 0.2f;

struct Carver {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t o = off;
    off += (bytes + 1023) & ~size_t(1023);
    return o;
  }
};

// ------------------------------------------------------------------ workspace layout
struct Layout {
  size_t packed, bias, bncoef, bwdcoef, partials, sums, trunk_err, wg_partials, ps_scratch, loss_scratch;
  size_t dyall = 0, slot = 0;             // per-layer output gradients of the trunk convs: slot l = 2*block + conv, last = conv2
  size_t wgb_partials = 0, wgb_floats = 0;  // partial sets of the batched trunk weight-gradient kernel
  size_t trunk_sync = 0, trunk_tab = 0;     // trunk_fused: flags / barrier words, the two TrunkLayer tables (fwd | bwd)
  size_t U1, out1, trunk;
  std::vector<size_t> y1, z1, y2, out;   // per residual block (eval: aliases of 4 rotating buffers)
  std::vector<size_t> up;                // per upsample stage
  size_t g[4];                           // P-sized gradient buffers
  std::vector<size_t> dup;               // gradient of each upsample stage output
  size_t Ud;                             // unfolded d(SR)
  size_t c1d = 0;                        // packed conv1 data-gradient filter (input-gradient backward only)
  size_t frozen_tab = 0;                 // int4 BatchNorm offset rows of the frozen (running-statistics) forward
  // debug (keep_grads): every inter-layer gradient in its own buffer instead of the 3 rotating ones
  std::vector<size_t> kd_y2, kd_p1, kd_y1, kd_in;
  size_t kd_last, kd_c1;
  size_t total;
};

size_t t64(int64_t pixels) { return size_t(pixels) * 128; }
constexpr int64_t kConv1DgradElems = 9 * 32 * 64;   // pack_conv1_dgrad: [9 row taps][32][64] bf16

int64_t wgrad_max_floats(int n_up) {
  // splits * n_blocks * n_pairs * 8192, with splits = SMs / n_blocks  => <= 148 * n_pairs * 8192
  (void)n_up;
  return int64_t(148) * 5 * 8192;
}

// upper bound of wgrad3_batched_partials_floats() for the trunk (148 SMs; the launcher re-checks against the device)
size_t wgrad_batched_floats(const GeneratorEngine& e) {
  const int64_t T = int64_t(e.N) * ((e.H + 15) / 16) * ((e.W + 7) / 8);
  const int64_t layers = 2 * e.n_res + 1;
  int64_t per = (T * layers + 147) / 148;
  if (per < 1) per = 1;
  const int64_t max_slots = (T + per - 1) / per + 1;
  return size_t(layers * max_slots) * 3 * 192 * 64;
}

Layout make_layout(const GeneratorEngine& e, bool training) {
  Layout L;
  Carver c;
  const int64_t P = int64_t(e.N) * e.H * e.W;
  L.packed = c.take(size_t(e.packed_elems) * 2);
  L.bias = c.take(size_t(e.bias_elems) * 4);
  L.bncoef = c.take(size_t(2 * e.n_res) * 256 * 4);
  L.bwdcoef = c.take(192 * 4);
  L.partials = c.take(size_t(kRedBlocksMax) * 128 * 4);
  L.sums = c.take(128 * 8);
  L.trunk_err = c.take(4);                 // the fused trunk kernel's error word (generator_trunk_error)
  L.trunk_sync = c.take(trunk_sync_bytes(e.N, e.H, e.W));
  L.trunk_tab = c.take(size_t(2) * (2 * e.n_res + 1) * sizeof(TrunkLayer));   // eval: 2*n_res int4 BatchNorm offset rows instead
  L.U1 = c.take(size_t(e.N) * (e.H + 1) * e.W * 128);
  L.out1 = c.take(t64(P));
  L.y1.resize(e.n_res); L.z1.resize(e.n_res); L.y2.resize(e.n_res); L.out.resize(e.n_res);
  if (training) {
    for (int b = 0; b < e.n_res; ++b) {
      L.y1[b] = c.take(t64(P)); L.z1[b] = c.take(t64(P)); L.y2[b] = c.take(t64(P)); L.out[b] = c.take(t64(P));
    }
  } else {
    const size_t y1 = c.take(t64(P)), z1 = c.take(t64(P)), y2 = c.take(t64(P)), oa = c.take(t64(P)), ob = c.take(t64(P));
    for (int b = 0; b < e.n_res; ++b) { L.y1[b] = y1; L.z1[b] = z1; L.y2[b] = y2; L.out[b] = (b & 1) ? ob : oa; }
  }
  L.trunk = c.take(t64(P));
  L.up.resize(e.n_up);
  for (int j = 0; j < e.n_up; ++j) L.up[j] = c.take(t64(P << (2 * (j + 1))));
  L.wg_partials = L.ps_scratch = L.loss_scratch = L.Ud = 0;
  for (int i = 0; i < 4; ++i) L.g[i] = 0;
  L.dup.assign(e.n_up, 0);
  if (training) {
    L.wg_partials = c.take(size_t(wgrad_max_floats(e.n_up)) * 4);
    L.ps_scratch = c.take(size_t(e.N) * (size_t(e.H) << e.n_up) * 128 * 4);
    L.loss_scratch = c.take(size_t(loss_scratch_doubles()) * 8);
    for (int i = 0; i < 3; ++i) L.g[i] = c.take(t64(P));
    // every trunk conv's output gradient stays alive until the batched weight-gradient kernel at the end of backward
    L.slot = (t64(P) + 1023) & ~size_t(1023);
    L.dyall = c.take(L.slot * size_t(2 * e.n_res + 1));
    L.g[3] = L.dyall + L.slot * size_t(2 * e.n_res);        // d(trunk) = output gradient of conv2
    // debug buffers directly behind dyall: g[0..2] | dyall | kd_* form ONE uniformly strided "gradient region" that the
    // fused trunk kernel addresses by buffer index
    L.kd_last = L.kd_c1 = 0;
    if (e.keep_grads) {
      L.kd_y2.resize(e.n_res); L.kd_p1.resize(e.n_res); L.kd_y1.resize(e.n_res); L.kd_in.resize(e.n_res);
      for (int b = 0; b < e.n_res; ++b) {
        L.kd_y2[b] = L.dyall + L.slot * size_t(2 * b + 1); L.kd_y1[b] = L.dyall + L.slot * size_t(2 * b);
        L.kd_p1[b] = c.take(t64(P)); L.kd_in[b] = c.take(t64(P));
      }
      L.kd_last = c.take(t64(P));
      L.kd_c1 = c.take(t64(P));
    }
    L.wgb_floats = wgrad_batched_floats(e);
    L.wgb_partials = c.take(L.wgb_floats * 4);
    for (int j = 0; j < e.n_up; ++j) L.dup[j] = c.take(t64(P << (2 * (j + 1))));
    const int64_t Hs = int64_t(e.H) << e.n_up, Ws = int64_t(e.W) << e.n_up;
    L.Ud = c.take(size_t(e.N) * (Hs + 1) * Ws * 128);
    L.c1d = c.take(size_t(kConv1DgradElems) * 2);
    L.frozen_tab = c.take(size_t(2 * e.n_res + 1) * 16);
  }
  L.total = c.off;
  return L;
}

// ------------------------------------------------------------------ parameter bookkeeping
int64_t add_param(GeneratorEngine& e, const std::string& name, std::initializer_list<int> shape) {
  ParamInfo p;
  p.name = name;
  p.ndim = int(shape.size());
  p.numel = 1;
  int i = 0;
  for (int s : shape) { p.shape[i++] = s; p.numel *= s; }
  for (; i < 4; ++i) p.shape[i] = 1;
  p.offset = e.param_elems;
  e.param_elems += (p.numel + 3) & ~int64_t(3);   // keep every tensor 16-byte aligned
  e.params.push_back(p);
  return p.offset;
}
int64_t poff(const GeneratorEngine& e, const std::string& name) {
  for (const auto& p : e.params)
    if (p.name == name) return p.offset;
  return -1;
}
int64_t boff(const GeneratorEngine& e, const std::string& name) {
  for (const auto& b : e.buffers)
    if (b.name == name) return b.offset;
  return -1;
}

// packed-weight offsets (bf16 elements)
struct PackOffsets {
  int64_t conv1_f;
  std::vector<int64_t> rb_f[2], rb_d[2];
  int64_t conv2_f, conv2_d;
  std::vector<int64_t> up_f, up_d;
  int64_t conv3_f, conv3_d;
  std::vector<int64_t> up_bias;  // fp32 elements in the packed-bias buffer
};

// W[co][ci][kh][kw] of an OIHW tensor at flat offset `base`
inline int widx(int64_t base, int Cin, int K, int co, int ci, int kh, int kw) {
  return int(base + ((int64_t(co) * Cin + ci) * K + kh) * K + kw);
}

void pack_c3x3_fwd(std::vector<int>& idx, int64_t base, int cout, bool pixel_shuffle) {
  // [kb = s*3 + r][n][ci]   s = kw, r = kh
  for (int s = 0; s < 3; ++s)
    for (int r = 0; r < 3; ++r)
      for (int n = 0; n < cout; ++n) {
        const int co = pixel_shuffle ? 4 * (n % 64) + n / 64 : n;
        for (int ci = 0; ci < 64; ++ci) idx.push_back(widx(base, 64, 3, co, ci, r, s));
      }
}
void pack_c3x3_dgrad(std::vector<int>& idx, int64_t base, int cout, bool pixel_shuffle) {
  // [(c*3 + s)*3 + r][n = ci][k]   co = pixel_shuffle ? 4k + c : k ; kh = 2-r, kw = 2-s
  const int chunks = cout / 64;
  for (int c = 0; c < chunks; ++c)
    for (int s = 0; s < 3; ++s)
      for (int r = 0; r < 3; ++r)
        for (int ci = 0; ci < 64; ++ci)
          for (int k = 0; k < 64; ++k) {
            const int co = pixel_shuffle ? 4 * k + c : c * 64 + k;
            idx.push_back(widx(base, 64, 3, co, ci, 2 - r, 2 - s));
          }
}
void pack_conv1_fwd(std::vector<int>& idx, int64_t base) {
  // [r][co][(dr, s, c)] = W1[co][c][2r+dr][s]
  for (int r = 0; r < 5; ++r)
    for (int co = 0; co < 64; ++co)
      for (int ch = 0; ch < 64; ++ch) {
        int v = -1;
        if (ch < 54) {
          const int dr = ch / 27, s = (ch % 27) / 3, c = ch % 3, kh = 2 * r + dr;
          if (kh <= 8) v = widx(base, 3, 9, co, c, kh, s);
        }
        idx.push_back(v);
      }
}
void pack_conv3_fwd(std::vector<int>& idx, int64_t base) {
  // fold9: [r = kh][n = s*3 + co (32)][ci] = W3[co][ci][kh][s]
  for (int r = 0; r < 9; ++r)
    for (int n = 0; n < 32; ++n)
      for (int ci = 0; ci < 64; ++ci) idx.push_back(n < 27 ? widx(base, 64, 9, n % 3, ci, r, n / 3) : -1);
}
void pack_conv1_dgrad(std::vector<int>& idx, int64_t base) {
  // fold9 form of conv1's data gradient (a 9x9 64 -> 3 conv over d(pre-LeakyReLU) with the transposed, flipped filter):
  // [r = kh'][n = s*3 + c (32)][co] = W1[co][c][8-r][8-s]
  for (int r = 0; r < 9; ++r)
    for (int n = 0; n < 32; ++n)
      for (int co = 0; co < 64; ++co) idx.push_back(n < 27 ? widx(base, 3, 9, co, n % 3, 8 - r, 8 - n / 3) : -1);
}
void pack_conv3_dgrad(std::vector<int>& idx, int64_t base) {
  // [r][ci][(dr, s, co)] = W3[co][ci][8-2r-dr][8-s]
  for (int r = 0; r < 5; ++r)
    for (int ci = 0; ci < 64; ++ci)
      for (int ch = 0; ch < 64; ++ch) {
        int v = -1;
        if (ch < 54) {
          const int dr = ch / 27, s = (ch % 27) / 3, co = ch % 3, kh = 8 - 2 * r - dr;
          if (kh >= 0) v = widx(base, 64, 9, co, ci, kh, 8 - s);
        }
        idx.push_back(v);
      }
}

// index of D_t[row][col] inside one split's partial block: ((nb*n_pairs + t/2)*128 + (t&1)*64 + row)*64 + col
inline int pidx(int nb, int n_pairs, int t, int row, int col) { return ((nb * n_pairs + t / 2) * 128 + (t & 1) * 64 + row) * 64 + col; }

int* upload(const std::vector<int>& v) {
  int* d = nullptr;
  if (cudaMalloc(&d, v.size() * sizeof(int)) != cudaSuccess) return nullptr;
  if (cudaMemcpy(d, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return nullptr; }
  return d;
}

// the engine object handed out by generator_create
struct EngineImpl : GeneratorEngine {
  PackOffsets po;
  Layout L;
  // host copies of the constant index maps; uploaded at the first bind (create() needs no device)
  std::vector<int> h_pack_idx, h_bias_idx, h_wg_c3x3, h_wg_up, h_wg_conv1, h_wg_conv3, h_conv1_dgrad;
  int* d_conv1_dgrad_idx = nullptr;
  bool last_frozen = false;     // the last forward on the training workspace used running BatchNorm statistics
  // srg_generator_forward_frozen_tiles: the windows and frame height / width of the last forward on the training workspace when
  // it was a frozen-tiles forward (tile_n == 0 otherwise); srg_generator_backward_tiles runs their backward
  int tile_n = 0, tile_H = 0, tile_W = 0;
  TileDesc tile_tab[kMaxTiles];
  ~EngineImpl() override { cudaFree(d_conv1_dgrad_idx); }
  // fused trunk (trunk_fused.cu): set at bind when the workspace layout is uniformly strided and the geometry fits
  bool trunk_ok = false;
  int trunk_act_buffers = 0, trunk_grad_buffers = 0;
  size_t trunk_act_slot = 0;
  int trunk_dout_idx = 0;       // gradient-region buffer that holds d(out1) of the block chain after the backward kernel
};

#define RC(x)                  \
  do {                         \
    int rc_ = (x);             \
    if (rc_ != 0) return rc_;  \
  } while (0)

InView plain_view(const void* ptr, int H, int W, int C = 64) {
  InView v;
  v.ptr = ptr; v.stride_w = C; v.stride_h = int64_t(W) * C; v.stride_n = int64_t(H) * W * C; v.channels = C;
  return v;
}
// view q = (i, j) of a pixel-shuffled tensor [N, 2H, 2W, 64] on the (H, W) grid
InView ps_view(const void* base, int H, int W, int q) {
  const int i = q >> 1, j = q & 1;
  InView v;
  v.ptr = reinterpret_cast<const uint16_t*>(base) + (size_t(i) * 2 * W + j) * 64;
  v.stride_w = 128; v.stride_h = int64_t(4) * W * 64; v.stride_n = int64_t(4) * H * W * 64; v.channels = 64;
  return v;
}

void set_taps_3x3(ConvGemmArgs& a) {
  a.TH = 16; a.TW = 8;
  a.n_strips = 3; a.n_taps = 3; a.strip_rows = 18; a.strip_dh = -1;
  for (int s = 0; s < 3; ++s) a.strip_dw[s] = s - 1;
  for (int r = 0; r < 3; ++r) a.tap_row[r] = r;
}
void set_taps_pairs(ConvGemmArgs& a) {
  a.TH = 16; a.TW = 8;
  a.n_strips = 1; a.n_taps = 5; a.strip_rows = 24; a.strip_dh = -3; a.strip_dw[0] = 0;
  for (int r = 0; r < 5; ++r) a.tap_row[r] = 2 * r;
}

}  // namespace

namespace {
struct ProfScope {
  GeneratorEngine* e; cudaStream_t st; bool on;
  ProfScope(GeneratorEngine* e_, cudaStream_t st_) : e(e_), st(st_), on(e_->prof_on) {
    if (!on) return;
    if (e->prof_used + 2 > e->prof_events.size()) {
      if (e->prof_events.size() >= 8192) { on = false; return; }
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) { on = false; return; }
      e->prof_events.push_back(a); e->prof_events.push_back(b);
    }
    cudaEventRecord(e->prof_events[e->prof_used], st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(e->prof_events[e->prof_used + 1], st);
    e->prof_used += 2;
  }
};
}  // namespace

// ---- fused trunk: per-layer tables for both directions (see TrunkLayer) and the uniform-stride checks they rely on
namespace {
bool build_trunk_tables(EngineImpl& e, std::vector<TrunkLayer>& fwd, std::vector<TrunkLayer>& bwd) {
  const Layout& L = e.L;
  const PackOffsets& po = e.po;
  const int R = e.n_res;
  if (R < 1 || trunk_grid(e.N, e.H, e.W) == 0) return false;
  // activation region: out1 | (y1 z1 y2 out) x R | trunk, one slot apart
  const size_t Sa = L.y1[0] - L.out1;
  if (Sa != L.slot) return false;
  for (int b = 0; b < R; ++b) {
    if (L.y1[b] != L.out1 + size_t(4 * b + 1) * Sa || L.z1[b] != L.out1 + size_t(4 * b + 2) * Sa ||
        L.y2[b] != L.out1 + size_t(4 * b + 3) * Sa || L.out[b] != L.out1 + size_t(4 * b + 4) * Sa) return false;
  }
  if (L.trunk != L.out1 + size_t(4 * R + 1) * Sa) return false;
  // gradient region: g0 g1 g2 | dyall (2R+1) | [keep: (kd_p1 kd_in) x R, kd_last, kd_c1]
  if (L.g[1] != L.g[0] + L.slot || L.g[2] != L.g[0] + 2 * L.slot || L.dyall != L.g[0] + 3 * L.slot) return false;
  const int kd0 = 3 + 2 * R + 1;
  if (e.keep_grads) {
    for (int b = 0; b < R; ++b)
      if (L.kd_p1[b] != L.g[0] + size_t(kd0 + 2 * b) * L.slot || L.kd_in[b] != L.g[0] + size_t(kd0 + 2 * b + 1) * L.slot) return false;
    if (L.kd_last != L.g[0] + size_t(kd0 + 2 * R) * L.slot) return false;
  }
  // packed filters: (fwd, dgrad) pairs of 576 rows each, layer order 2*block + conv, conv2 last
  const int64_t w0 = po.rb_f[0][0], set = 36864;
  for (int b = 0; b < R; ++b)
    for (int k = 0; k < 2; ++k)
      if (po.rb_f[k][b] != w0 + int64_t(2 * (2 * b + k)) * set || po.rb_d[k][b] != w0 + int64_t(2 * (2 * b + k) + 1) * set) return false;
  if (po.conv2_f != w0 + int64_t(4 * R) * set || po.conv2_d != w0 + int64_t(4 * R + 1) * set) return false;
  if (e.param_elems > (int64_t(1) << 30)) return false;

  char nm[96];
  auto P = [&](const char* fmt, int b, int k) { snprintf(nm, sizeof(nm), fmt, b, k); return int(poff(e, nm)); };
  auto clear = [](TrunkLayer& t) {
    memset(&t, 0, sizeof(t));
    t.st1_idx = t.st2_idx = t.aux1_idx = t.aux2_idx = t.y_idx = t.mask_bn = t.bn = t.bias_off = -1;
  };
  fwd.assign(size_t(2 * R + 1), TrunkLayer());
  for (int l = 0; l < 2 * R; ++l) {
    const int b = l / 2, k = l % 2;
    TrunkLayer& t = fwd[size_t(l)];
    clear(t);
    t.in_idx = 4 * b + 2 * k; t.st1_idx = 4 * b + 1 + 2 * k; t.st2_idx = 4 * b + 2 + 2 * k;
    t.aux2_idx = k ? 4 * b : -1; t.bn = l; t.relu = k ? 0 : 1; t.w_row = 2 * l * 576;
    t.bias_off = P("residual_blocks.%d.conv%d.bias", b, k + 1);
    t.gamma_off = P("residual_blocks.%d.bn%d.weight", b, k + 1);
    t.beta_off = P("residual_blocks.%d.bn%d.bias", b, k + 1);
    snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.running_mean", b, k + 1);
    t.rm_off = int(boff(e, nm));
  }
  {
    TrunkLayer& t = fwd[size_t(2 * R)];
    clear(t);
    t.in_idx = 4 * R; t.st1_idx = 4 * R + 1; t.aux1_idx = 0; t.w_row = 4 * R * 576; t.bias_off = int(poff(e, "conv2.bias"));
  }
  const bool keep = e.keep_grads;
  const int i_last = kd0 + 2 * R;
  auto i_p1 = [&](int b) { return kd0 + 2 * b; };
  auto i_in = [&](int b) { return kd0 + 2 * b + 1; };
  bwd.clear();
  {
    TrunkLayer t;
    clear(t);
    t.in_idx = 3 + 2 * R; t.st1_idx = keep ? i_last : 0; t.st2_idx = 3 + 2 * (R - 1) + 1;
    t.y_idx = 4 * (R - 1) + 3; t.bn = 2 * (R - 1) + 1; t.w_row = (4 * R + 1) * 576;
    t.gamma_off = P("residual_blocks.%d.bn%d.weight", R - 1, 2); t.beta_off = P("residual_blocks.%d.bn%d.bias", R - 1, 2);
    bwd.push_back(t);
  }
  for (int b = R - 1; b >= 0; --b) {
    TrunkLayer t;
    clear(t);                                   // conv2 of block b: d(z1) -> ReLU mask -> BatchNorm 1 backward
    t.in_idx = 3 + 2 * b + 1; t.st1_idx = keep ? i_p1(b) : 1; t.st2_idx = 3 + 2 * b;   // raw masked gradient: scratch g[1]
    t.y_idx = 4 * b + 1; t.mask_bn = 2 * b; t.bn = 2 * b; t.w_row = (2 * (2 * b + 1) + 1) * 576;
    t.gamma_off = P("residual_blocks.%d.bn%d.weight", b, 1); t.beta_off = P("residual_blocks.%d.bn%d.bias", b, 1);
    bwd.push_back(t);
    clear(t);                                   // conv1 of block b: + skip gradient -> BatchNorm 2 backward of block b-1
    t.in_idx = 3 + 2 * b;
    t.aux1_idx = keep ? (b == R - 1 ? i_last : i_in(b + 1)) : 0;
    t.st1_idx = keep ? i_in(b) : 0;
    t.w_row = (2 * (2 * b) + 1) * 576;
    if (b > 0) {
      t.y_idx = 4 * (b - 1) + 3; t.bn = 2 * (b - 1) + 1; t.st2_idx = 3 + 2 * (b - 1) + 1;
      t.gamma_off = P("residual_blocks.%d.bn%d.weight", b - 1, 2); t.beta_off = P("residual_blocks.%d.bn%d.bias", b - 1, 2);
    }
    bwd.push_back(t);
  }
  e.trunk_act_buffers = 4 * R + 2;
  e.trunk_grad_buffers = kd0 + (keep ? 2 * R + 2 : 0);
  e.trunk_act_slot = Sa;
  e.trunk_dout_idx = keep ? i_in(0) : 0;
  return true;
}

// the fused trunk applies to training passes on one GPU, or under data parallelism with the peer-memory SyncBatchNorm
// transport (the NCCL transport keeps the per-layer launches)
bool use_trunk_fused(const EngineImpl& e) {
  if (!e.trunk_ok || !trunk_fused_preferred(e.N, e.H, e.W)) return false;
  if (e.peer != nullptr) return true;
  return e.allreduce == nullptr && e.world == 1;
}

void fill_trunk_gen(EngineImpl* e, TrunkGen& t) {
  const Layout& L = e->L;
  uint8_t* ws = e->ws;
  t.act_base = ws + L.out1;
  t.grad_base = ws + L.g[0];
  t.weights = reinterpret_cast<const uint16_t*>(ws + L.packed) + e->po.rb_f[0][0];
  t.master = e->master; t.grads = e->grads; t.bn_buffers = e->bn_buffers;
  t.bncoef = reinterpret_cast<float*>(ws + L.bncoef);
  t.gpart = reinterpret_cast<float*>(ws + L.partials);
  t.sync = reinterpret_cast<unsigned int*>(ws + L.trunk_sync);
  t.err = reinterpret_cast<unsigned int*>(ws + L.trunk_err);
  t.peer = e->peer;
}

// one launch for the trunks of `n` engines of identical geometry / configuration (n = 1: the nn.Module path)
int run_trunk_multi(EngineImpl* const* es, int n, int bwd, int update_running, cudaStream_t st, bool param_grads = true) {
  EngineImpl* e = es[0];
  const Layout& L = e->L;
  const int64_t P = int64_t(e->N) * e->H * e->W;
  TrunkArgs a; memset(&a, 0, sizeof(a));
  a.bwd = bwd; a.N = e->N; a.H = e->H; a.W = e->W; a.n_layers = 2 * e->n_res + 1;
  a.layers = reinterpret_cast<const TrunkLayer*>(e->ws + L.trunk_tab) + (bwd ? a.n_layers : 0);
  a.act_slot = int64_t(e->trunk_act_slot); a.act_buffers = e->trunk_act_buffers;
  a.grad_slot = int64_t(L.slot); a.grad_buffers = e->trunk_grad_buffers;
  a.weight_rows = int64_t(4 * e->n_res + 2) * 576;
  a.count = double(P) * e->world; a.eps = kBnEps; a.momentum = kBnMomentum; a.update_running = update_running;
  a.param_grad_scale = 1.f / float(e->world);
  a.n_gen = n;
  for (int i = 0; i < n; ++i) {
    EngineImpl* o = es[i];
    if (!o->trunk_ok || o->N != e->N || o->H != e->H || o->W != e->W || o->n_res != e->n_res || o->keep_grads != e->keep_grads ||
        o->world != e->world || o->L.slot != L.slot || o->trunk_act_slot != e->trunk_act_slot) {
      set_error("trunk_fused: the engines of a joint launch must share geometry and configuration");
      return -65;
    }
    fill_trunk_gen(o, a.gen[i]);
    if (!param_grads) a.gen[i].grads = nullptr;
    o->prof_layers = a.n_layers;
  }
  e->launches += 1;
  ProfScope ps(e, st);
  return launch_trunk(a, st);
}
int run_trunk(EngineImpl* e, int bwd, int update_running, cudaStream_t st, bool param_grads = true) {
  return run_trunk_multi(&e, 1, bwd, update_running, st, param_grads);
}

// ------------------------------------------------------------------ grouped per-layer trunk
// Large geometries (several tiles per SM, where the fused trunk kernel loses to per-layer launches): the SAME trunk layer of
// n <= 3 generators runs as ONE grouped conv3_il launch (launch_conv_gemm_grouped: 49 CTAs per generator, 12 tiles per CTA
// at cfg2 instead of 4, so the launch ramp, the 72 KB filter load and the last tile's epilogue drain are paid once per 12
// tiles), and the BatchNorm passes between two layers run per generator on forked streams (they are HBM-bound and not
// SM-exclusive, so the n chains overlap) and join again ahead of the next grouped launch.  Arithmetic per generator is the
// per-layer path's (same kernels, same order).
// N: the items of the pass (the engine's N, or the window count of a tiled backward)
bool wgrad_layout_batched(const EngineImpl& e, int N) {
  const Layout& L = e.L;
  if (!e.wgrad_batched || e.n_res < 1) return false;
  for (int b = 0; b < e.n_res; ++b) {
    const size_t x1 = b > 0 ? L.out[b - 1] : L.out1;
    if (x1 != L.out1 + size_t(2 * b) * 2 * L.slot || L.z1[b] != L.out1 + size_t(2 * b + 1) * 2 * L.slot) return false;
  }
  if (L.out[e.n_res - 1] != L.out1 + size_t(2 * e.n_res) * 2 * L.slot) return false;
  WgradBatchArgs probe; memset(&probe, 0, sizeof(probe));
  probe.N = N; probe.H = e.H; probe.W = e.W; probe.n_layers = 2 * e.n_res + 1;
  // the partial-set workspace was sized for 148 SMs at create time: a device that splits the work differently keeps the
  // per-layer launches instead of overrunning it
  return wgrad3_batched_partials_floats(probe) <= L.wgb_floats;
}

bool use_trunk_grouped(const EngineImpl& e) {
  if (!e.ws || !e.ws_training || e.n_res < 1) return false;
  if (e.allreduce != nullptr && e.peer == nullptr) return false;      // NCCL SyncBatchNorm transport: per-generator branches
  return wgrad_layout_batched(e, e.N);
}

struct ForkJoin {
  cudaStream_t side[kIlMaxGroups] = {};
  cudaEvent_t fork = nullptr, join[kIlMaxGroups] = {};
  int device = -1;
};
// streams[0] = st, streams[1..n) = process-wide side streams; fork() makes them wait for st, join() the other way round
int fork_join_get(ForkJoin** out) {
  static ForkJoin fj;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { set_error("cudaGetDevice failed"); return -70; }
  if (fj.device != dev) {
    for (int i = 1; i < kIlMaxGroups; ++i) {
      if (cudaStreamCreateWithFlags(&fj.side[i], cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&fj.join[i], cudaEventDisableTiming) != cudaSuccess) {
        set_error("grouped trunk: side stream / event creation failed");
        return -71;
      }
    }
    if (cudaEventCreateWithFlags(&fj.fork, cudaEventDisableTiming) != cudaSuccess) { set_error("grouped trunk: event creation failed"); return -71; }
    fj.device = dev;
  }
  *out = &fj;
  return 0;
}
int fj_fork(ForkJoin* fj, int n, cudaStream_t st) {
  if (n < 2) return 0;
  if (cudaEventRecord(fj->fork, st) != cudaSuccess) { set_error("grouped trunk: event record failed"); return -72; }
  for (int i = 1; i < n; ++i)
    if (cudaStreamWaitEvent(fj->side[i], fj->fork, 0) != cudaSuccess) { set_error("grouped trunk: stream wait failed"); return -72; }
  return 0;
}
int fj_join(ForkJoin* fj, int n, cudaStream_t st) {
  for (int i = 1; i < n; ++i)
    if (cudaEventRecord(fj->join[i], fj->side[i]) != cudaSuccess || cudaStreamWaitEvent(st, fj->join[i], 0) != cudaSuccess) {
      set_error("grouped trunk: join failed");
      return -72;
    }
  return 0;
}

struct BnNames { int64_t gamma, beta, rm; };
BnNames bn_offsets(const EngineImpl& e, int b, int k) {
  char nm[96];
  BnNames o;
  snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.weight", b, k + 1); o.gamma = poff(e, nm);
  snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.bias", b, k + 1); o.beta = poff(e, nm);
  snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.running_mean", b, k + 1); o.rm = boff(e, nm);
  return o;
}

// one grouped 3x3 64 -> 64 launch: problem g reads in[g], writes out[g]
int grouped_conv3x3(EngineImpl* const* es, int n, const void* const* in, const int64_t* w_off, const float* const* bias,
                    const void* const* residual, const void* const* mask, void* const* out, bool stats, int* stats_rows,
                    cudaStream_t st) {
  ConvGemmArgs as[kIlMaxGroups];
  for (int g = 0; g < n; ++g) {
    EngineImpl* e = es[g];
    ConvGemmArgs& a = as[g];
    memset(&a, 0, sizeof(a));
    a.N = e->N; a.H = e->H; a.W = e->W; set_taps_3x3(a);
    a.n_views = 1; a.views[0] = plain_view(in[g], e->H, e->W); a.in_H = e->H; a.in_W = e->W;
    a.weights = reinterpret_cast<const uint16_t*>(e->ws + e->L.packed) + w_off[g]; a.cout_total = 64; a.block_n = 64;
    a.bias = bias ? bias[g] : nullptr; a.act = ACT_NONE;
    a.residual = residual ? residual[g] : nullptr; a.mask_src = mask ? mask[g] : nullptr;
    a.out = out[g]; a.out_mode = OUT_NHWC;
    if (stats) a.stats = reinterpret_cast<float*>(e->ws + e->L.partials);
  }
  if (stats) *stats_rows = n > 1 ? conv_gemm_grouped_rows(as[0], n) : conv_gemm_grid(as[0]);
  es[0]->launches += 1;
  es[0]->prof_layers = n;
  ProfScope ps(es[0], st);
  return launch_conv_gemm_grouped(as, n, st);
}

int grouped_check(EngineImpl* const* es, int n) {
  for (int g = 0; g < n; ++g) {
    const EngineImpl* o = es[g];
    if (!use_trunk_grouped(*o) || o->N != es[0]->N || o->H != es[0]->H || o->W != es[0]->W || o->n_res != es[0]->n_res ||
        o->world != es[0]->world) {
      set_error("grouped trunk: engine %d is not bound for training on the per-layer path or differs in geometry", g);
      return -67;
    }
  }
  return 0;
}

int trunk_layers_forward_multi(EngineImpl* const* es, int n, int update_running, cudaStream_t st) {
  RC(grouped_check(es, n));
  ForkJoin* fj = nullptr;
  RC(fork_join_get(&fj));
  const int R = es[0]->n_res;
  const int64_t P = int64_t(es[0]->N) * es[0]->H * es[0]->W;
  const void* x[kIlMaxGroups]; const void* in[kIlMaxGroups]; void* out[kIlMaxGroups];
  const float* bias[kIlMaxGroups]; const void* res[kIlMaxGroups]; int64_t woff[kIlMaxGroups];
  char nm[96];
  for (int g = 0; g < n; ++g) x[g] = es[g]->ws + es[g]->L.out1;
  // training-mode BatchNorm (+ReLU / +skip) of every generator behind a grouped conv, one forked stream per generator
  auto bn_stage = [&](int b, int k, int rows) -> int {
    RC(fj_fork(fj, n, st));
    for (int g = 0; g < n; ++g) {
      EngineImpl* e = es[g];
      const Layout& L = e->L;
      cudaStream_t sg = g == 0 ? st : fj->side[g];
      float* coef = reinterpret_cast<float*>(e->ws + L.bncoef) + size_t(2 * b + k) * 256;
      const BnNames o = bn_offsets(*e, b, k);
      ReduceFinalize f; memset(&f, 0, sizeof(f));
      f.mode = RF_BN_FWD; f.count = double(P) * e->world; f.eps = kBnEps; f.momentum = kBnMomentum;
      f.gamma = e->master + o.gamma; f.beta = e->master + o.beta;
      f.running_mean = update_running ? e->bn_buffers + o.rm : nullptr;
      f.running_var = update_running ? e->bn_buffers + o.rm + 64 : nullptr;
      f.out0 = coef; f.out1 = coef + 64; f.out2 = coef + 128; f.out3 = coef + 192;
      float* partials = reinterpret_cast<float*>(e->ws + L.partials);
      const void* y = e->ws + (k == 0 ? L.y1[b] : L.y2[b]);
      void* dst = e->ws + (k == 0 ? L.z1[b] : L.out[b]);
      if (e->peer) RC(launch_peer_finalize(e->peer, partials, rows, f, sg));
      else RC(launch_partials_finalize(partials, rows, f, sg));
      RC(launch_bn_apply(y, coef, coef + 64, k == 0 ? nullptr : x[g], k == 0 ? 1 : 0, dst, P, sg));
      e->launches += 2;
    }
    return fj_join(fj, n, st);
  };
  for (int b = 0; b < R; ++b) {
    int rows = 0;
    for (int k = 0; k < 2; ++k) {
      snprintf(nm, sizeof(nm), "residual_blocks.%d.conv%d.bias", b, k + 1);
      for (int g = 0; g < n; ++g) {
        const Layout& L = es[g]->L;
        in[g] = k == 0 ? x[g] : es[g]->ws + L.z1[b];
        out[g] = es[g]->ws + (k == 0 ? L.y1[b] : L.y2[b]);
        woff[g] = es[g]->po.rb_f[k][b];
        bias[g] = es[g]->master + poff(*es[g], nm);
      }
      RC(grouped_conv3x3(es, n, in, woff, bias, nullptr, nullptr, out, true, &rows, st));
      RC(bn_stage(b, k, rows));
    }
    for (int g = 0; g < n; ++g) x[g] = es[g]->ws + es[g]->L.out[b];
  }
  // conv2 + global skip (src/models.py:83-84)
  for (int g = 0; g < n; ++g) {
    in[g] = x[g]; out[g] = es[g]->ws + es[g]->L.trunk; res[g] = es[g]->ws + es[g]->L.out1;
    woff[g] = es[g]->po.conv2_f; bias[g] = es[g]->master + poff(*es[g], "conv2.bias");
  }
  return grouped_conv3x3(es, n, in, woff, bias, res, nullptr, out, false, nullptr, st);
}

// buffer that holds d(out1) of the block chain after the per-layer backward loop (the loop alternates g[0] / g[1])
void* layers_dout(const EngineImpl& e) {
  if (e.keep_grads) return e.ws + (e.n_res > 0 ? e.L.kd_in[0] : e.L.kd_last);
  return e.ws + e.L.g[e.n_res % 2 == 0 ? 0 : 1];
}

int trunk_layers_backward_multi(EngineImpl* const* es, int n, cudaStream_t st) {
  RC(grouped_check(es, n));
  ForkJoin* fj = nullptr;
  RC(fork_join_get(&fj));
  const int R = es[0]->n_res;
  const int64_t P = int64_t(es[0]->N) * es[0]->H * es[0]->W;
  const void* in[kIlMaxGroups]; void* out[kIlMaxGroups]; const void* res[kIlMaxGroups]; const void* mask[kIlMaxGroups];
  int64_t woff[kIlMaxGroups];
  void* dout[kIlMaxGroups]; void* dother[kIlMaxGroups];
  for (int g = 0; g < n; ++g) {
    const Layout& L = es[g]->L;
    dout[g] = es[g]->keep_grads ? es[g]->ws + L.kd_last : es[g]->ws + L.g[0];
    dother[g] = es[g]->ws + L.g[1];
    in[g] = es[g]->ws + L.g[3]; out[g] = dout[g]; woff[g] = es[g]->po.conv2_d;
  }
  RC(grouped_conv3x3(es, n, in, woff, nullptr, nullptr, nullptr, out, false, nullptr, st));
  // BatchNorm backward of every generator (sums of dz and dz*y, coefficients, apply) on forked streams
  auto bn_bwd_stage = [&](int b, int k, void* const* dz, void* const* dy) -> int {
    RC(fj_fork(fj, n, st));
    for (int g = 0; g < n; ++g) {
      EngineImpl* e = es[g];
      const Layout& L = e->L;
      cudaStream_t sg = g == 0 ? st : fj->side[g];
      const float* coef = reinterpret_cast<const float*>(e->ws + L.bncoef) + size_t(2 * b + k) * 256;
      float* bwd = reinterpret_cast<float*>(e->ws + L.bwdcoef);
      float* partials = reinterpret_cast<float*>(e->ws + L.partials);
      const BnNames o = bn_offsets(*e, b, k);
      const void* y = e->ws + (k == 0 ? L.y1[b] : L.y2[b]);
      RC(launch_chan_reduce(dz[g], y, P, partials, sg));
      const int r = reduce_blocks(P);
      e->launches += 1;
      ReduceFinalize f; memset(&f, 0, sizeof(f));
      f.mode = RF_BN_BWD; f.count = double(P) * e->world; f.gamma = e->master + o.gamma; f.save_mean = coef + 128; f.save_inv = coef + 192;
      f.dgamma = e->grads + o.gamma; f.dbeta = e->grads + o.beta; f.out0 = bwd; f.out1 = bwd + 64; f.out2 = bwd + 128;
      if (e->peer) RC(launch_peer_finalize(e->peer, partials, r, f, sg));
      else RC(launch_partials_finalize(partials, r, f, sg));
      RC(launch_bn_bwd_apply(dz[g], y, bwd, bwd + 64, bwd + 128, dy[g], P, sg));
      e->launches += 2;
    }
    return fj_join(fj, n, st);
  };
  void* d_y[kIlMaxGroups]; void* d_p1[kIlMaxGroups]; void* d_in[kIlMaxGroups];
  for (int b = R - 1; b >= 0; --b) {
    // out = bn2(y2) + x
    for (int g = 0; g < n; ++g) d_y[g] = es[g]->ws + es[g]->L.dyall + es[g]->L.slot * size_t(2 * b + 1);
    RC(bn_bwd_stage(b, 1, dout, d_y));
    for (int g = 0; g < n; ++g) {
      const Layout& L = es[g]->L;
      d_p1[g] = es[g]->keep_grads ? es[g]->ws + L.kd_p1[b] : dother[g];
      in[g] = d_y[g]; out[g] = d_p1[g]; mask[g] = es[g]->ws + L.z1[b]; woff[g] = es[g]->po.rb_d[1][b];   // ReLU backward via mask
    }
    RC(grouped_conv3x3(es, n, in, woff, nullptr, nullptr, mask, out, false, nullptr, st));
    // z1 = relu(bn1(y1))
    for (int g = 0; g < n; ++g) d_y[g] = es[g]->ws + es[g]->L.dyall + es[g]->L.slot * size_t(2 * b);
    RC(bn_bwd_stage(b, 0, d_p1, d_y));
    for (int g = 0; g < n; ++g) {
      const Layout& L = es[g]->L;
      d_in[g] = es[g]->keep_grads ? es[g]->ws + L.kd_in[b] : dother[g];
      in[g] = d_y[g]; out[g] = d_in[g]; res[g] = dout[g]; woff[g] = es[g]->po.rb_d[0][b];               // + skip gradient
    }
    RC(grouped_conv3x3(es, n, in, woff, nullptr, res, nullptr, out, false, nullptr, st));
    for (int g = 0; g < n; ++g) {
      if (es[g]->keep_grads) { dout[g] = d_in[g]; } else { void* t = dout[g]; dout[g] = dother[g]; dother[g] = t; }
    }
  }
  return 0;
}
}  // namespace

int generators_trunk(GeneratorEngine* const* gs, int n, int bwd, int update_running, cudaStream_t st) {
  if (n < 1 || n > kTrunkMaxGen) { set_error("generators_trunk: 1..%d engines", kTrunkMaxGen); return -62; }
  EngineImpl* es[kTrunkMaxGen];
  bool fused = true;
  for (int i = 0; i < n; ++i) {
    es[i] = static_cast<EngineImpl*>(gs[i]);
    if (!es[i]->ws || !es[i]->ws_training || !use_trunk_fused(*es[i]) || (bwd && !es[i]->wgrad_batched)) fused = false;
  }
  if (fused) return run_trunk_multi(es, n, bwd, update_running, st);
  for (int i = 0; i < n; ++i)
    if (!use_trunk_grouped(*es[i])) {
      set_error("generators_trunk: engine %d is not bound for training on the fused or the grouped per-layer trunk path", i);
      return -66;
    }
  // grouped per-layer launches, at most kIlMaxGroups generators per launch (4 generators: 2 + 2)
  const int chunks = (n + kIlMaxGroups - 1) / kIlMaxGroups;
  for (int c = 0, i0 = 0; c < chunks; ++c) {
    const int m = (n - i0 + (chunks - c) - 1) / (chunks - c);
    RC(bwd ? trunk_layers_backward_multi(es + i0, m, st) : trunk_layers_forward_multi(es + i0, m, update_running, st));
    i0 += m;
  }
  return 0;
}

int generator_trunk_error(GeneratorEngine* g) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  if (!e->ws) return 0;
  unsigned int v = 0;
  if (cudaMemcpy(&v, e->ws + e->L.trunk_err, 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return int(v);
}
int generator_prof_layers(const GeneratorEngine* g) { return g->prof_layers; }

int generator_set_keep_grads(GeneratorEngine* g, int keep) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  if (e->ws != nullptr) { set_error("set_keep_grads: call before bind"); return -30; }
  e->keep_grads = keep != 0;
  e->workspace_bytes_train = make_layout(*e, true).total;
  return 0;
}
int generator_profile_enable(GeneratorEngine* g, int on) { g->prof_on = on != 0; return 0; }
int generator_profile_read(GeneratorEngine* g, double* ms_sum, long long* count) {
  double total = 0.0;
  for (size_t i = 0; i + 1 < g->prof_used; i += 2) {
    cudaError_t e = cudaEventSynchronize(g->prof_events[i + 1]);
    if (e != cudaSuccess) { set_error("profile_read: %s", cudaGetErrorString(e)); return int(e); }
    float ms = 0.f;
    e = cudaEventElapsedTime(&ms, g->prof_events[i], g->prof_events[i + 1]);
    if (e != cudaSuccess) { set_error("profile_read: %s", cudaGetErrorString(e)); return int(e); }
    total += double(ms);
  }
  if (ms_sum) *ms_sum = total;
  if (count) *count = (long long)(g->prof_used / 2);
  g->prof_used = 0;
  return 0;
}

GeneratorEngine::~GeneratorEngine() {
  for (cudaEvent_t ev : prof_events) cudaEventDestroy(ev);
  cudaFree(d_pack_idx); cudaFree(d_bias_idx); cudaFree(d_wg_idx_c3x3); cudaFree(d_wg_idx_up);
  cudaFree(d_wg_idx_conv1); cudaFree(d_wg_idx_conv3); cudaFree(d_wgb_off);
}

GeneratorEngine* generator_create(int N, int H, int W, int n_res, int n_up) {
  if (N < 1 || H < 1 || W < 1 || n_res < 0 || n_up < 0 || n_up > 4) { set_error("generator_create: bad geometry"); return nullptr; }
  EngineImpl* e = new EngineImpl();
  e->N = N; e->H = H; e->W = W; e->n_res = n_res; e->n_up = n_up;
  {
    const char* ev = getenv("SRG_WGRAD_BATCHED");
    e->wgrad_batched = !(ev != nullptr && ev[0] == '0');
  }
  // ---- parameters in the reference's registration order (src/models.py:53-78)
  add_param(*e, "conv1.weight", {64, 3, 9, 9});
  add_param(*e, "conv1.bias", {64});
  char nm[96];
  for (int b = 0; b < n_res; ++b) {
    const char* sub[2][2] = {{"conv1", "bn1"}, {"conv2", "bn2"}};
    // registration order inside ResidualBlock: conv1, bn1, conv2, bn2 (src/models.py:15-19)
    for (int k = 0; k < 2; ++k) {
      snprintf(nm, sizeof(nm), "residual_blocks.%d.%s.weight", b, sub[k][0]); add_param(*e, nm, {64, 64, 3, 3});
      snprintf(nm, sizeof(nm), "residual_blocks.%d.%s.bias", b, sub[k][0]); add_param(*e, nm, {64});
      snprintf(nm, sizeof(nm), "residual_blocks.%d.%s.weight", b, sub[k][1]); add_param(*e, nm, {64});
      snprintf(nm, sizeof(nm), "residual_blocks.%d.%s.bias", b, sub[k][1]); add_param(*e, nm, {64});
      for (const char* stat : {"running_mean", "running_var"}) {
        BufferInfo bi;
        snprintf(nm, sizeof(nm), "residual_blocks.%d.%s.%s", b, sub[k][1], stat);
        bi.name = nm; bi.offset = e->buffer_elems; bi.numel = 64;
        e->buffer_elems += 64;
        e->buffers.push_back(bi);
      }
    }
  }
  add_param(*e, "conv2.weight", {64, 64, 3, 3});
  add_param(*e, "conv2.bias", {64});
  for (int j = 0; j < n_up; ++j) {
    snprintf(nm, sizeof(nm), "upsample.%d.weight", 3 * j); add_param(*e, nm, {256, 64, 3, 3});
    snprintf(nm, sizeof(nm), "upsample.%d.bias", 3 * j); add_param(*e, nm, {256});
  }
  add_param(*e, "conv3.weight", {3, 64, 9, 9});
  add_param(*e, "conv3.bias", {3});

  // ---- pack maps
  std::vector<int> idx;
  idx.reserve(size_t(e->param_elems) * 2 + 65536);
  PackOffsets& po = e->po;
  po.conv1_f = int64_t(idx.size()); pack_conv1_fwd(idx, poff(*e, "conv1.weight"));
  for (int k = 0; k < 2; ++k) { po.rb_f[k].resize(n_res); po.rb_d[k].resize(n_res); }
  for (int b = 0; b < n_res; ++b)
    for (int k = 0; k < 2; ++k) {
      snprintf(nm, sizeof(nm), "residual_blocks.%d.conv%d.weight", b, k + 1);
      const int64_t base = poff(*e, nm);
      po.rb_f[k][b] = int64_t(idx.size()); pack_c3x3_fwd(idx, base, 64, false);
      po.rb_d[k][b] = int64_t(idx.size()); pack_c3x3_dgrad(idx, base, 64, false);
    }
  po.conv2_f = int64_t(idx.size()); pack_c3x3_fwd(idx, poff(*e, "conv2.weight"), 64, false);
  po.conv2_d = int64_t(idx.size()); pack_c3x3_dgrad(idx, poff(*e, "conv2.weight"), 64, false);
  po.up_f.resize(n_up); po.up_d.resize(n_up); po.up_bias.resize(n_up);
  std::vector<int> bidx;
  for (int j = 0; j < n_up; ++j) {
    snprintf(nm, sizeof(nm), "upsample.%d.weight", 3 * j);
    const int64_t base = poff(*e, nm);
    po.up_f[j] = int64_t(idx.size()); pack_c3x3_fwd(idx, base, 256, true);
    po.up_d[j] = int64_t(idx.size()); pack_c3x3_dgrad(idx, base, 256, true);
    snprintf(nm, sizeof(nm), "upsample.%d.bias", 3 * j);
    const int64_t bb = poff(*e, nm);
    po.up_bias[j] = int64_t(bidx.size());
    for (int n = 0; n < 256; ++n) bidx.push_back(int(bb + 4 * (n % 64) + n / 64));
  }
  po.conv3_f = int64_t(idx.size()); pack_conv3_fwd(idx, poff(*e, "conv3.weight"));
  po.conv3_d = int64_t(idx.size()); pack_conv3_dgrad(idx, poff(*e, "conv3.weight"));
  e->packed_elems = int64_t(idx.size());
  if (bidx.empty()) bidx.push_back(-1);
  e->bias_elems = int64_t(bidx.size());

  // ---- wgrad scatter maps: out element -> index inside one split's partial block
  std::vector<int> m33(64 * 64 * 9), mup(256 * 64 * 9), mc1(64 * 3 * 81), mc3(3 * 64 * 81);
  for (int co = 0; co < 64; ++co)
    for (int ci = 0; ci < 64; ++ci)
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) m33[((co * 64 + ci) * 3 + kh) * 3 + kw] = pidx(0, 5, kw * 3 + kh, ci, co);
  for (int co = 0; co < 256; ++co)
    for (int ci = 0; ci < 64; ++ci)
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) mup[((co * 64 + ci) * 3 + kh) * 3 + kw] = pidx(co % 4, 5, kw * 3 + kh, ci, co / 4);
  for (int co = 0; co < 64; ++co)
    for (int c = 0; c < 3; ++c)
      for (int kh = 0; kh < 9; ++kh)
        for (int kw = 0; kw < 9; ++kw)
          mc1[((co * 3 + c) * 9 + kh) * 9 + kw] = pidx(0, 3, kh / 2, (kh % 2) * 27 + kw * 3 + c, co);
  for (int co = 0; co < 3; ++co)
    for (int ci = 0; ci < 64; ++ci)
      for (int kh = 0; kh < 9; ++kh)
        for (int kw = 0; kw < 9; ++kw) {
          const int dr = kh % 2, r = (8 - kh - dr) / 2, s = 8 - kw;
          mc3[((co * 64 + ci) * 9 + kh) * 9 + kw] = pidx(0, 3, r, dr * 27 + s * 3 + co, ci);
        }
  auto invert = [](const std::vector<int>& fwd, size_t n_part) {
    std::vector<int> inv(n_part, -1);
    for (size_t i = 0; i < fwd.size(); ++i)
      if (fwd[i] >= 0) inv[size_t(fwd[i])] = int(i);
    return inv;
  };
  // 3x3 layers use the fused wgrad kernel: partial index ((nb*3 + kw)*192 + (2-kh)*64 + co)*64 + ci
  for (int co = 0; co < 64; ++co)
    for (int ci = 0; ci < 64; ++ci)
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) m33[((co * 64 + ci) * 3 + kh) * 3 + kw] = ((0 * 3 + kw) * 192 + (2 - kh) * 64 + co) * 64 + ci;
  for (int co = 0; co < 256; ++co)
    for (int ci = 0; ci < 64; ++ci)
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw)
          mup[((co * 64 + ci) * 3 + kh) * 3 + kw] = (((co % 4) * 3 + kw) * 192 + (2 - kh) * 64 + co / 4) * 64 + ci;
  m33 = invert(m33, size_t(1) * 3 * 64 * 192);
  mup = invert(mup, size_t(4) * 3 * 64 * 192);
  mc1 = invert(mc1, size_t(1) * 3 * 8192);
  mc3 = invert(mc3, size_t(1) * 3 * 8192);
  e->h_pack_idx.swap(idx); e->h_bias_idx.swap(bidx);
  e->h_wg_c3x3.swap(m33); e->h_wg_up.swap(mup); e->h_wg_conv1.swap(mc1); e->h_wg_conv3.swap(mc3);
  pack_conv1_dgrad(e->h_conv1_dgrad, poff(*e, "conv1.weight"));
  e->workspace_bytes_train = make_layout(*e, true).total;
  e->workspace_bytes_eval = make_layout(*e, false).total;
  return e;
}

int generator_bind(GeneratorEngine* g, float* master, float* grads, float* bn_buffers, void* ws, size_t ws_bytes,
                   int training) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  const size_t need = training ? e->workspace_bytes_train : e->workspace_bytes_eval;
  if (ws_bytes < need) { set_error("generator_bind: workspace too small (%zu < %zu)", ws_bytes, need); return -20; }
  if ((reinterpret_cast<uintptr_t>(ws) & 1023) != 0) { set_error("generator_bind: workspace must be 1024-byte aligned"); return -21; }
  if (master == nullptr || bn_buffers == nullptr || (training && grads == nullptr)) { set_error("generator_bind: null buffer"); return -22; }
  if (e->d_pack_idx == nullptr) {
    e->d_pack_idx = upload(e->h_pack_idx);
    e->d_bias_idx = upload(e->h_bias_idx);
    e->d_wg_idx_c3x3 = upload(e->h_wg_c3x3);
    e->d_wg_idx_up = upload(e->h_wg_up);
    e->d_wg_idx_conv1 = upload(e->h_wg_conv1);
    e->d_wg_idx_conv3 = upload(e->h_wg_conv3);
    e->d_conv1_dgrad_idx = upload(e->h_conv1_dgrad);
    {
      std::vector<long long> off;
      char wn[96];
      for (int b = 0; b < e->n_res; ++b)
        for (int k = 0; k < 2; ++k) {
          snprintf(wn, sizeof(wn), "residual_blocks.%d.conv%d.weight", b, k + 1);
          off.push_back((long long)poff(*e, wn));
        }
      off.push_back((long long)poff(*e, "conv2.weight"));
      if (cudaMalloc(&e->d_wgb_off, off.size() * sizeof(long long)) != cudaSuccess ||
          cudaMemcpy(e->d_wgb_off, off.data(), off.size() * sizeof(long long), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("generator_bind: device allocation of the wgrad offset table failed");
        return -23;
      }
    }
    if (!e->d_pack_idx || !e->d_bias_idx || !e->d_wg_idx_c3x3 || !e->d_wg_idx_up || !e->d_wg_idx_conv1 || !e->d_wg_idx_conv3 ||
        !e->d_conv1_dgrad_idx) {
      set_error("generator_bind: device allocation of index maps failed: %s", cudaGetErrorString(cudaGetLastError()));
      return -29;
    }
  }
  e->master = master; e->grads = grads; e->bn_buffers = bn_buffers;
  e->ws = reinterpret_cast<uint8_t*>(ws); e->ws_bytes = ws_bytes; e->ws_training = training != 0;
  e->L = make_layout(*e, training != 0);
  if (cudaMemset(e->ws + e->L.trunk_err, 0, 4) != cudaSuccess) { set_error("generator_bind: memset failed"); return -29; }
  e->trunk_ok = false;
  e->last_frozen = false;
  e->tile_n = 0;
  if (e->n_res > 0) {
    // offsets of every BatchNorm's parameters / statistics / preceding conv bias: launch_bn_eval_coeffs_all (eval
    // workspace) or launch_bn_frozen_coeffs_all (training workspace)
    std::vector<int> tab;
    char nm[96];
    for (int b = 0; b < e->n_res; ++b)
      for (int k = 1; k <= 2; ++k) {
        snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.weight", b, k); tab.push_back(int(poff(*e, nm)));
        snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.bias", b, k); tab.push_back(int(poff(*e, nm)));
        snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.running_mean", b, k); tab.push_back(int(boff(*e, nm)));
        snprintf(nm, sizeof(nm), "residual_blocks.%d.conv%d.bias", b, k); tab.push_back(int(poff(*e, nm)));
      }
    const size_t tab_off = training ? e->L.frozen_tab : e->L.trunk_tab;
    if (cudaMemcpy(e->ws + tab_off, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) {
      set_error("generator_bind: upload of the BatchNorm offset table failed");
      return -29;
    }
  }
  if (training) {
    std::vector<TrunkLayer> tf, tb;
    if (build_trunk_tables(*e, tf, tb)) {
      tf.insert(tf.end(), tb.begin(), tb.end());
      if (cudaMemcpy(e->ws + e->L.trunk_tab, tf.data(), tf.size() * sizeof(TrunkLayer), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("generator_bind: upload of the trunk layer tables failed");
        return -29;
      }
      e->trunk_ok = true;
    }
  }
  // named tensors for parity tests
  e->tensors.clear();
  auto reg = [&](const std::string& name, size_t off, int n, int h, int w, int c, int dtype) {
    TensorInfo t; t.name = name; t.byte_offset = int64_t(off); t.dims[0] = n; t.dims[1] = h; t.dims[2] = w; t.dims[3] = c; t.dtype = dtype;
    e->tensors.push_back(t);
  };
  const Layout& L = e->L;
  reg("out1", L.out1, e->N, e->H, e->W, 64, 0);
  char nm[64];
  if (training)
    for (int b = 0; b < e->n_res; ++b) {
      snprintf(nm, sizeof(nm), "rb%d.y1", b); reg(nm, L.y1[b], e->N, e->H, e->W, 64, 0);
      snprintf(nm, sizeof(nm), "rb%d.z1", b); reg(nm, L.z1[b], e->N, e->H, e->W, 64, 0);
      snprintf(nm, sizeof(nm), "rb%d.y2", b); reg(nm, L.y2[b], e->N, e->H, e->W, 64, 0);
      snprintf(nm, sizeof(nm), "rb%d.out", b); reg(nm, L.out[b], e->N, e->H, e->W, 64, 0);
    }
  reg("trunk", L.trunk, e->N, e->H, e->W, 64, 0);
  for (int j = 0; j < e->n_up; ++j) {
    snprintf(nm, sizeof(nm), "up%d", j); reg(nm, L.up[j], e->N, e->H << (j + 1), e->W << (j + 1), 64, 0);
    if (training) { snprintf(nm, sizeof(nm), "d_up%d", j); reg(nm, L.dup[j], e->N, e->H << (j + 1), e->W << (j + 1), 64, 0); }
  }
  if (training) {
    reg("d_trunk", L.g[3], e->N, e->H, e->W, 64, 0);
    if (e->keep_grads) {
      for (int b = 0; b < e->n_res; ++b) {
        snprintf(nm, sizeof(nm), "rb%d.d_y2", b); reg(nm, L.kd_y2[b], e->N, e->H, e->W, 64, 0);
        snprintf(nm, sizeof(nm), "rb%d.d_pre1", b); reg(nm, L.kd_p1[b], e->N, e->H, e->W, 64, 0);
        snprintf(nm, sizeof(nm), "rb%d.d_y1", b); reg(nm, L.kd_y1[b], e->N, e->H, e->W, 64, 0);
        snprintf(nm, sizeof(nm), "rb%d.d_in", b); reg(nm, L.kd_in[b], e->N, e->H, e->W, 64, 0);
      }
      reg("d_last", L.kd_last, e->N, e->H, e->W, 64, 0);
      reg("d_pre_conv1", L.kd_c1, e->N, e->H, e->W, 64, 0);
    }
  }
  return 0;
}

int generator_pack(GeneratorEngine* g, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  if (!e->ws) { set_error("generator_pack: not bound"); return -23; }
  RC(launch_pack_bf16(e->master, e->d_pack_idx, e->ws + e->L.packed, e->packed_elems, st));
  RC(launch_gather_f32(e->master, e->d_bias_idx, reinterpret_cast<float*>(e->ws + e->L.bias), e->bias_elems, st));
  e->launches += 2;
  return 0;
}

// ------------------------------------------------------------------ forward
int generator_forward(GeneratorEngine* g, const float* lr, float* sr, int training, int update_running, cudaStream_t st) {
  return generator_forward_phases(g, lr, sr, training, update_running, kPhaseAll, st);
}

namespace {
// srg_generator_forward_tiles: n windows of larger frames in one eval pass (conv1's operand gathered from the frames,
// conv3's output scattered into them, cropped).  u8: the frames, in and out, are uint8 NHWC (srg_generator_forward_u8,
// whose dense batch of the engine's N frames has gather.n == 0 and scatter.n == 0, and _tiles_u8)
static_assert(kMaxWindows == kMaxTiles, "gather and scatter tables hold the same windows");
struct TileCall {
  const void* frames;
  bool u8;
  int n;
  WindowGather gather;
  FoldScatter scatter;
};

// frozen: eval-mode BatchNorm (running statistics, never updated or exchanged) on the training workspace, every
// activation the backward reads kept; per-layer trunk launches only
int forward_impl(EngineImpl* e, const float* lr, void* sr, int training, int update_running, int phases, bool frozen,
                 cudaStream_t st, const TileCall* tc = nullptr) {
  if (!e->ws) { set_error("generator_forward: not bound"); return -23; }
  if (training && !e->ws_training) { set_error("generator_forward: bound workspace is eval-sized"); return -24; }
  if (training) { e->last_frozen = frozen; e->tile_n = 0; }
  if (frozen) update_running = 0;
  const Layout& L = e->L;
  const PackOffsets& po = e->po;
  uint8_t* ws = e->ws;
  const uint16_t* packed = reinterpret_cast<const uint16_t*>(ws + L.packed);
  const float* pbias = reinterpret_cast<const float*>(ws + L.bias);
  const int N = tc ? tc->n : e->N, H = e->H, W = e->W;
  const int64_t P = int64_t(N) * H * W;
  char nm[96];

  if (phases != kPhaseAll && !(training && (use_trunk_fused(*e) || use_trunk_grouped(*e)))) {
    set_error("generator_forward_phases: split execution needs the fused or the grouped per-layer trunk path (training, supported configuration)");
    return -31;
  }
  // split execution on the per-layer path: the TRUNK phase belongs to generators_trunk() (grouped launches)
  const bool layers_here = phases == kPhaseAll;
  if (!training && e->n_res > 0) {
    // eval: every BatchNorm's folded coefficients in one launch, two kernels ahead of the first conv that reads them
    RC(launch_bn_eval_coeffs_all(e->master, e->bn_buffers, ws + L.trunk_tab, 2 * e->n_res, kBnEps,
                                 reinterpret_cast<float*>(ws + L.bncoef), st));
    e->launches += 1;
  }
  if (frozen && e->n_res > 0) {
    RC(launch_bn_frozen_coeffs_all(e->master, e->bn_buffers, ws + L.frozen_tab, 2 * e->n_res, kBnEps,
                                   reinterpret_cast<float*>(ws + L.bncoef), st));
    e->launches += 1;
  }
  // conv1: 9x9, 3->64, LeakyReLU(0.2)  (src/models.py:56-57,81)
  if (phases & kPhasePre) {
  if (tc && tc->u8 && tc->gather.n == 0) RC(launch_unfold9_u8(static_cast<const uint8_t*>(tc->frames), N, H, W, ws + L.U1, st));
  else if (tc && tc->u8) RC(launch_unfold9_windows_u8(static_cast<const uint8_t*>(tc->frames), tc->gather, H, W, ws + L.U1, st));
  else if (tc) RC(launch_unfold9_windows(static_cast<const float*>(tc->frames), tc->gather, H, W, ws + L.U1, st));
  else RC(launch_unfold9(lr, N, H, W, 1.f, ws + L.U1, st));
  {
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = H; a.W = W; set_taps_pairs(a);
    a.n_views = 1; a.views[0] = plain_view(ws + L.U1, H + 1, W); a.in_H = H + 1; a.in_W = W;
    a.weights = packed + po.conv1_f; a.cout_total = 64; a.block_n = 64;
    a.bias = e->master + poff(*e, "conv1.bias"); a.act = ACT_LRELU; a.slope = kSlope;
    a.out = ws + L.out1; a.out_mode = OUT_NHWC;
    RC(launch_conv_gemm(a, st));
  }
  e->launches += 2;
  }

  int stats_rows = 0;
  auto conv3x3 = [&](const void* in, int64_t w_off, const float* bias, const void* residual, void* out, bool stats,
                     const float* scale = nullptr, int act = ACT_NONE) -> int {
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = H; a.W = W; set_taps_3x3(a);
    a.n_views = 1; a.views[0] = plain_view(in, H, W); a.in_H = H; a.in_W = W;
    a.weights = packed + w_off; a.cout_total = 64; a.block_n = 64;
    a.bias = bias; a.scale = scale; a.act = act; a.residual = residual; a.out = out; a.out_mode = OUT_NHWC;
    a.exclusive = training ? 0 : 1;
    if (stats) { a.stats = reinterpret_cast<float*>(ws + L.partials); stats_rows = conv_gemm_grid(a); }
    e->launches += 1;
    ProfScope ps(e, st);
    return launch_conv_gemm(a, st);
  };
  auto bn_coeffs = [&](int b, int k, const void* y) -> int {
    // BatchNorm2d(64): batch statistics in training (biased var), running stats in eval (src/models.py:16,19)
    float* coef = reinterpret_cast<float*>(ws + L.bncoef) + size_t(2 * b + k) * 256;
    snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.weight", b, k + 1);
    const float* gamma = e->master + poff(*e, nm);
    snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.bias", b, k + 1);
    const float* beta = e->master + poff(*e, nm);
    snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.running_mean", b, k + 1);
    float* rm = e->bn_buffers + boff(*e, nm);
    float* rv = rm + 64;
    if (!training) {
      // eval: the coefficients are known before the conv runs, so BatchNorm (+ReLU / +skip) is folded into the conv
      // epilogue (out = act(acc * scale + shift') + skip); `y` carries the conv bias to absorb into the shift
      e->launches += 1;
      return launch_bn_eval_coeffs(gamma, beta, rm, rv, kBnEps, coef, coef + 64, st, reinterpret_cast<const float*>(y));
    }
    float* partials = reinterpret_cast<float*>(ws + L.partials);
    double* sums = reinterpret_cast<double*>(ws + L.sums);
    // batch statistics were accumulated by the producing conv's epilogue: [stats_rows][128] per-CTA partial sums
    (void)y;
    if (!e->allreduce || e->peer) {
      ReduceFinalize f; memset(&f, 0, sizeof(f));
      f.mode = RF_BN_FWD; f.count = double(P) * e->world; f.eps = kBnEps; f.momentum = kBnMomentum; f.gamma = gamma; f.beta = beta;
      f.running_mean = update_running ? rm : nullptr; f.running_var = update_running ? rv : nullptr;
      f.out0 = coef; f.out1 = coef + 64; f.out2 = coef + 128; f.out3 = coef + 192;
      e->launches += 1;
      if (e->peer) return launch_peer_finalize(e->peer, partials, stats_rows, f, st);
      return launch_partials_finalize(partials, stats_rows, f, st);
    }
    RC(launch_partials_sums(partials, stats_rows, sums, st));
    RC(e->allreduce(e->allreduce_ctx, sums, 128, st));
    e->launches += 2;
    return launch_bn_finalize(sums, double(P) * e->world, gamma, beta, kBnEps, kBnMomentum, update_running ? rm : nullptr,
                              update_running ? rv : nullptr, coef, coef + 64, coef + 128, coef + 192, st);
  };

  // training-mode BatchNorm (+ReLU / +skip) behind a conv whose epilogue left the per-CTA statistics in `partials`
  auto bn_train_apply = [&](int b, int k, const void* y, const void* skip, int relu, void* out) -> int {
    float* coef = reinterpret_cast<float*>(ws + L.bncoef) + size_t(2 * b + k) * 256;
    if (frozen) {
      e->launches += 1;
      return launch_bn_apply(y, coef, coef + 64, skip, relu, out, P, st);
    }
    RC(bn_coeffs(b, k, y));
    e->launches += 1;
    return launch_bn_apply(y, coef, coef + 64, skip, relu, out, P, st);
  };

  const void* x = ws + L.out1;
  const bool fused = training && !frozen && use_trunk_fused(*e);
  const bool stats = training && !frozen;       // batch statistics accumulated by the trunk convs' epilogues
  e->prof_layers = 1;
  if (fused && (phases & kPhaseTrunk)) RC(run_trunk(e, 0, update_running, st));
  for (int b = 0; b < e->n_res && !fused && layers_here; ++b) {
    const float* coef1 = reinterpret_cast<const float*>(ws + L.bncoef) + size_t(2 * b) * 256;
    const float* coef2 = coef1 + 256;
    if (!training) {
      // eval mode: 2 conv launches per block, BatchNorm folded into their epilogues (no y1 / y2 round trip through HBM)
      RC(conv3x3(x, po.rb_f[0][b], coef1 + 64, nullptr, ws + L.z1[b], false, coef1, ACT_RELU));
      RC(conv3x3(ws + L.z1[b], po.rb_f[1][b], coef2 + 64, x, ws + L.out[b], false, coef2, ACT_NONE));
      x = ws + L.out[b];
      continue;
    }
    snprintf(nm, sizeof(nm), "residual_blocks.%d.conv1.bias", b);
    RC(conv3x3(x, po.rb_f[0][b], e->master + poff(*e, nm), nullptr, ws + L.y1[b], stats));
    RC(bn_train_apply(b, 0, ws + L.y1[b], nullptr, 1, ws + L.z1[b]));
    snprintf(nm, sizeof(nm), "residual_blocks.%d.conv2.bias", b);
    RC(conv3x3(ws + L.z1[b], po.rb_f[1][b], e->master + poff(*e, nm), nullptr, ws + L.y2[b], stats));
    RC(bn_train_apply(b, 1, ws + L.y2[b], x, 0, ws + L.out[b]));
    x = ws + L.out[b];
  }
  // conv2 + global skip (src/models.py:83-84)
  if (!fused && layers_here) RC(conv3x3(x, po.conv2_f, e->master + poff(*e, "conv2.bias"), ws + L.out1, ws + L.trunk, false));
  if (!(phases & kPhasePost)) return 0;
  // upsample stages: conv 64->256, PixelShuffle(2), ReLU (src/models.py:69-75,85)
  const void* in = ws + L.trunk;
  for (int j = 0; j < e->n_up; ++j) {
    const int Hj = H << j, Wj = W << j;
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = Hj; a.W = Wj; set_taps_3x3(a);
    a.n_views = 1; a.views[0] = plain_view(in, Hj, Wj); a.in_H = Hj; a.in_W = Wj;
    a.weights = packed + po.up_f[j]; a.cout_total = 256; a.block_n = 64;
    a.bias = pbias + po.up_bias[j]; a.act = ACT_RELU; a.out = ws + L.up[j]; a.out_mode = OUT_PIXEL_SHUFFLE;
    a.exclusive = training ? 0 : 1;
    RC(launch_conv_gemm(a, st));
    e->launches += 1;
    in = ws + L.up[j];
  }
  // a frozen-tiles forward without an output recomputes the activations for its backward, which does not read SR
  if (tc && sr == nullptr) return 0;
  // conv3: 9x9, 64->3, no activation (src/models.py:78,86); fp32 NCHW output, or uint8 NHWC through tc->scatter
  {
    const int Hs = H << e->n_up, Ws = W << e->n_up;
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = Hs; a.W = Ws; a.TH = 4; a.TW = 32;
    a.n_strips = 1; a.n_taps = 9; a.strip_rows = 12; a.strip_dh = -4; a.strip_dw[0] = 0;
    for (int r = 0; r < 9; ++r) a.tap_row[r] = r;
    a.n_views = 1; a.views[0] = plain_view(in, Hs, Ws); a.in_H = Hs; a.in_W = Ws;
    a.weights = packed + po.conv3_f; a.cout_total = 32; a.block_n = 32;
    a.bias = e->master + poff(*e, "conv3.bias"); a.act = ACT_NONE; a.out = sr; a.out_mode = OUT_FOLD9_NCHW;
    if (tc) a.scatter = &tc->scatter;
    RC(launch_conv_gemm(a, st));
    e->launches += 1;
  }
  return 0;
}
}  // namespace

int generator_tile_halo(int n_res, int n_up) {
  if (n_res < 0 || n_up < 0 || n_up > 8) { set_error("tile_halo: num_residuals >= 0 and 0 <= num_upsample_stages <= 8"); return -1; }
  // rows of the input an output row at LR row 0 depends on, walked from conv3 (9x9 at 2^n_up) back to conv1
  int lo = -4, hi = (1 << n_up) + 3;
  for (int j = 0; j < n_up; ++j) {
    lo = (lo >> 1) - 1;               // PixelShuffle (floor division), then the up-conv's 3x3 taps
    hi = (hi >> 1) + 1;
  }
  const int r = lo < -hi ? -lo : hi;
  return r + (2 * n_res + 1) + 4;      // the trunk's 3x3 convs (2 per block + conv2), conv1's 9x9
}

namespace {
// argument checks shared by the eval and the frozen tiled forwards (no CUDA call) and the call's gather / scatter tables.
// Frames are fp32 NCHW, or uint8 NHWC (u8): element strides per frame, channel, row and pixel.
int make_tile_call(const EngineImpl* e, const char* who, const void* frames, bool u8, int F, int H, int W,
                   const TileDesc* tiles, int n, void* sr, bool sr_optional, TileCall* tc) {
  if (frames == nullptr) { set_error("%s: null pointer (frames)", who); return -22; }
  if (tiles == nullptr) { set_error("%s: null pointer (tiles)", who); return -22; }
  if (sr == nullptr && !sr_optional) { set_error("%s: null pointer (output)", who); return -22; }
  if (F < 1 || H < 1 || W < 1) { set_error("%s: F, H and W must be >= 1 (got %d, %d, %d)", who, F, H, W); return -26; }
  const int n_max = e->N < kMaxTiles ? e->N : kMaxTiles;
  if (n < 1 || n > n_max) { set_error("%s: tile count %d outside 1..%d (engine N and SRG_MAX_TILES)", who, n, n_max); return -27; }
  for (int i = 0; i < n; ++i) {
    const TileDesc& t = tiles[i];
    if (t.frame < 0 || t.frame >= F) { set_error("%s: tile %d frame index %d outside 0..%d", who, i, t.frame, F - 1); return -28; }
    if (t.y0 < 0 || t.x0 < 0 || int64_t(t.y0) + e->H > H || int64_t(t.x0) + e->W > W) {
      set_error("%s: tile %d window (%d, %d) + %d x %d is not inside the %d x %d frame", who, i, t.y0, t.x0, e->H, e->W, H, W);
      return -29;
    }
    if (t.crop_h < 1 || t.crop_w < 1) { set_error("%s: tile %d crop is empty", who, i); return -30; }
    if (t.crop_y0 < 0 || t.crop_x0 < 0 || int64_t(t.crop_y0) + t.crop_h > e->H || int64_t(t.crop_x0) + t.crop_w > e->W) {
      set_error("%s: tile %d crop is not inside its window", who, i);
      return -31;
    }
  }
  const int s = e->n_up;
  const int64_t plane = int64_t(H) * W, Ws = int64_t(W) << s, plane_o = (int64_t(H) << s) * Ws;
  memset(tc, 0, sizeof(*tc));
  tc->frames = frames;
  tc->u8 = u8;
  tc->n = n;
  const int64_t px = u8 ? 3 : 1;
  tc->gather.n = n; tc->gather.plane = u8 ? 1 : plane; tc->gather.pitch = px * W;
  tc->scatter.n = n; tc->scatter.u8 = u8; tc->scatter.plane = u8 ? 1 : plane_o; tc->scatter.pitch = px * Ws;
  tc->scatter.px = px;
  for (int i = 0; i < n; ++i) {
    const TileDesc& t = tiles[i];
    tc->gather.base[i] = int64_t(t.frame) * 3 * plane + (int64_t(t.y0) * W + t.x0) * px;
    FoldTile& o = tc->scatter.t[i];
    o.base = int64_t(t.frame) * 3 * plane_o + ((int64_t(t.y0) << s) * Ws + (int64_t(t.x0) << s)) * px;
    o.h_lo = t.crop_y0 << s; o.h_hi = (t.crop_y0 + t.crop_h) << s;
    o.w_lo = t.crop_x0 << s; o.w_hi = (t.crop_x0 + t.crop_w) << s;
  }
  return 0;
}
}  // namespace

int generator_forward_tiles(GeneratorEngine* g, const float* frames, int F, int H, int W, const TileDesc* tiles, int n,
                            float* sr, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  TileCall tc;
  RC(make_tile_call(e, "srg_generator_forward_tiles", frames, false, F, H, W, tiles, n, sr, false, &tc));
  if (!e->ws) { set_error("srg_generator_forward_tiles: no workspace bound"); return -23; }
  if (e->ws_training) { set_error("srg_generator_forward_tiles: needs an eval-sized workspace (this one is bound for training)"); return -24; }
  return forward_impl(e, nullptr, sr, 0, 0, kPhaseAll, false, st, &tc);
}

int generator_forward_tiles_u8(GeneratorEngine* g, const uint8_t* frames, int F, int H, int W, const TileDesc* tiles, int n,
                               uint8_t* sr, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  TileCall tc;
  RC(make_tile_call(e, "srg_generator_forward_tiles_u8", frames, true, F, H, W, tiles, n, sr, false, &tc));
  if (!e->ws) { set_error("srg_generator_forward_tiles_u8: no workspace bound"); return -23; }
  if (e->ws_training) { set_error("srg_generator_forward_tiles_u8: needs an eval-sized workspace (this one is bound for training)"); return -24; }
  return forward_impl(e, nullptr, sr, 0, 0, kPhaseAll, false, st, &tc);
}

int generator_forward_u8(GeneratorEngine* g, const uint8_t* lr, uint8_t* sr, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  if (lr == nullptr) { set_error("srg_generator_forward_u8: null pointer (input frames)"); return -22; }
  if (sr == nullptr) { set_error("srg_generator_forward_u8: null pointer (output)"); return -22; }
  if (!e->ws) { set_error("srg_generator_forward_u8: no workspace bound"); return -23; }
  TileCall tc;
  memset(&tc, 0, sizeof(tc));
  tc.frames = lr;
  tc.u8 = true;
  tc.n = e->N;
  const int64_t Ws = int64_t(e->W) << e->n_up, Hs = int64_t(e->H) << e->n_up;
  tc.scatter.u8 = 1;
  tc.scatter.item = 3 * Hs * Ws; tc.scatter.plane = 1; tc.scatter.pitch = 3 * Ws; tc.scatter.px = 3;
  return forward_impl(e, nullptr, sr, 0, 0, kPhaseAll, false, st, &tc);
}

int generator_forward_frozen_tiles(GeneratorEngine* g, const float* frames, int F, int H, int W, const TileDesc* tiles, int n,
                                   float* sr, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  TileCall tc;
  RC(make_tile_call(e, "srg_generator_forward_frozen_tiles", frames, false, F, H, W, tiles, n, sr, true, &tc));
  if (!e->ws) { set_error("srg_generator_forward_frozen_tiles: no workspace bound"); return -23; }
  if (!e->ws_training) { set_error("srg_generator_forward_frozen_tiles: needs a training-sized workspace (this one is bound for eval)"); return -24; }
  RC(forward_impl(e, nullptr, sr, 1, 0, kPhaseAll, true, st, &tc));
  e->tile_n = n; e->tile_H = H; e->tile_W = W;
  memcpy(e->tile_tab, tiles, sizeof(TileDesc) * size_t(n));
  return 0;
}

int generator_forward_phases(GeneratorEngine* g, const float* lr, float* sr, int training, int update_running, int phases,
                             cudaStream_t st) {
  return forward_impl(static_cast<EngineImpl*>(g), lr, sr, training, update_running, phases, false, st);
}

int generator_forward_frozen(GeneratorEngine* g, const float* lr, float* sr, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  if (lr == nullptr || sr == nullptr) { set_error("generator_forward_frozen: null image pointer"); return -22; }
  if (!e->ws || !e->ws_training) { set_error("generator_forward_frozen: needs a training-sized bound workspace"); return -25; }
  return forward_impl(e, lr, sr, 1, 0, kPhaseAll, true, st);
}

// ------------------------------------------------------------------ backward
namespace {
// param_grads == false: only the data-gradient chain runs (no gradient memset, weight gradients, bias sums or BatchNorm
// parameter gradients; the flat gradient buffer is not touched).  dlr != null: conv1's data gradient, fp32 NCHW.
// n_win > 0: the backward of a frozen-tiles forward over its n_win windows (the first n_win items of the workspace)
int backward_impl(EngineImpl* e, const float* dsr, int phases, bool param_grads, float* dlr, cudaStream_t st, int n_win = 0) {
  if (!e->ws || !e->ws_training) { set_error("generator_backward: needs a training-sized bound workspace"); return -25; }
  if (e->tile_n > 0 && n_win == 0) {
    set_error("generator_backward: the last forward was srg_generator_forward_frozen_tiles; its backward is srg_generator_backward_tiles");
    return -32;
  }
  const bool frozen = e->last_frozen;
  if (frozen && phases != kPhaseAll) {
    set_error("generator_backward_phases: the last forward used running BatchNorm statistics; split execution needs a training forward");
    return -31;
  }
  const bool pg = param_grads;
  const Layout& L = e->L;
  const PackOffsets& po = e->po;
  uint8_t* ws = e->ws;
  const uint16_t* packed = reinterpret_cast<const uint16_t*>(ws + L.packed);
  const int N = n_win > 0 ? n_win : e->N, H = e->H, W = e->W, S = e->n_up;
  const int64_t P = int64_t(N) * H * W;
  const int Hs = H << S, Ws = W << S;
  float* partials = reinterpret_cast<float*>(ws + L.partials);
  double* sums = reinterpret_cast<double*>(ws + L.sums);
  float* wgp = reinterpret_cast<float*>(ws + L.wg_partials);
  char nm[96];

  const bool pre = (phases & kPhasePre) != 0, mid = (phases & kPhaseTrunk) != 0, post = (phases & kPhasePost) != 0;
  if (dlr != nullptr) {
    // conv1's data-gradient filter, gathered from the fp32 master only when an input gradient is requested (the conv that
    // reads it runs at the end of this pass, far behind this launch)
    RC(launch_pack_bf16(e->master, e->d_conv1_dgrad_idx, ws + L.c1d, kConv1DgradElems, st));
    e->launches += 1;
  }
  if (pre && pg && cudaMemsetAsync(e->grads, 0, size_t(e->param_elems) * 4, st) != cudaSuccess) { set_error("memset grads failed"); return -26; }

  auto wgrad = [&](InView xv, int in_H, int in_W, bool pairs, int gh, int gw, const void* dy_base, int n_blocks,
                   bool dy_ps, const int* idx, const std::string& wname) -> int {
    WgradArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = gh; a.W = gw; a.TH = 16; a.TW = 8;
    a.x = xv; a.in_H = in_H; a.in_W = in_W;
    a.n_blocks = n_blocks;
    if (dy_ps) {
      a.dy_views = 4;
      for (int q = 0; q < 4; ++q) a.dy[q] = ps_view(dy_base, gh, gw, q);
    } else {
      a.dy_views = 1; a.dy[0] = plain_view(dy_base, gh, gw, 64 * n_blocks);
    }
    if (pairs) {
      a.n_strips = 1; a.n_taps = 5; a.strip_rows = 24; a.strip_dh = -3; a.strip_dw[0] = 0;
      for (int r = 0; r < 5; ++r) a.tap_row[r] = 2 * r;
    } else {
      a.n_strips = 3; a.n_taps = 3; a.strip_rows = 18; a.strip_dh = -1;
      for (int s = 0; s < 3; ++s) a.strip_dw[s] = s - 1;
      for (int r = 0; r < 3; ++r) a.tap_row[r] = r;
    }
    a.partials = wgp;
    int splits = 0;
    const ParamInfo* pi = nullptr;
    for (const auto& p : e->params) if (p.name == wname) pi = &p;
    if (!pi) { set_error("wgrad: unknown parameter %s", wname.c_str()); return -28; }
    e->launches += 2;
    if (!pairs) {
      // 3x3: taps fused along M (two column shifts) and N (three row shifts)
      const int floats = wgrad3x3_partials_floats(a, &splits);
      if (int64_t(floats) > wgrad_max_floats(S)) { set_error("wgrad partials exceed workspace"); return -27; }
      RC(launch_wgrad3x3(a, st));
      const size_t per_split = size_t(n_blocks) * 3 * 64 * 192;
      return launch_wgrad_reduce_inv(wgp, idx, e->grads + pi->offset, int(per_split), splits, per_split, st);
    }
    const int floats = wgrad_partials_floats(a, &splits);
    if (int64_t(floats) > wgrad_max_floats(S)) { set_error("wgrad partials exceed workspace"); return -27; }
    RC(launch_wgrad_gemm(a, st));
    const int n_pairs = (a.n_strips * a.n_taps + 1) / 2;
    const size_t per_split = size_t(n_blocks) * n_pairs * 128 * 64;
    return launch_wgrad_reduce_inv(wgp, idx, e->grads + pi->offset, int(per_split), splits, per_split, st);
  };
  auto bias_grad = [&](const void* dy, int64_t pixels, const std::string& bname) -> int {
    ReduceFinalize f; memset(&f, 0, sizeof(f));
    f.mode = RF_SUM; f.count = double(pixels); f.out0 = e->grads + poff(*e, bname);
    RC(launch_chan_reduce(dy, nullptr, pixels, partials, st));
    e->launches += 2;
    return launch_partials_finalize(partials, reduce_blocks(pixels), f, st);
  };
  // dgrad of a 3x3 conv whose output gradient has `chunks`*64 channels (4 pixel-shuffle views when chunks == 4)
  auto dgrad3x3 = [&](const void* dy_base, int gh, int gw, bool dy_ps, int64_t w_off, const void* residual, const void* mask,
                      void* out) -> int {
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = gh; a.W = gw; set_taps_3x3(a);
    if (dy_ps) {
      a.n_views = 4;
      for (int q = 0; q < 4; ++q) a.views[q] = ps_view(dy_base, gh, gw, q);
    } else {
      a.n_views = 1; a.views[0] = plain_view(dy_base, gh, gw);
    }
    a.in_H = gh; a.in_W = gw;
    a.weights = packed + w_off; a.cout_total = 64; a.block_n = 64;
    a.bias = nullptr; a.act = ACT_NONE; a.residual = residual; a.mask_src = mask; a.out = out; a.out_mode = OUT_NHWC;
    e->launches += 1;
    if (dy_ps) return launch_conv_gemm(a, st);
    ProfScope ps(e, st);
    return launch_conv_gemm(a, st);
  };

  const void* conv3_in = S > 0 ? ws + L.up[S - 1] : ws + L.trunk;
  void* d_trunk = ws + L.g[3];
  if (pre) {
  // ---- conv3 (9x9, 64->3): unfold d(SR) once; it feeds the bias sum, wgrad and dgrad
  RC(launch_unfold9(dsr, N, Hs, Ws, 1.f, ws + L.Ud, st));
  e->launches += 1;
  if (pg) {
    RC(launch_nchw_chan_sum(dsr, N, 3, int64_t(Hs) * Ws, reinterpret_cast<double*>(ws + L.loss_scratch),
                            e->grads + poff(*e, "conv3.bias"), 1.f, st));
    e->launches += 2;
    InView uv = plain_view(ws + L.Ud, Hs + 1, Ws);
    RC(wgrad(uv, Hs + 1, Ws, true, Hs, Ws, conv3_in, 1, false, e->d_wg_idx_conv3, "conv3.weight"));
  }
  {
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = Hs; a.W = Ws; set_taps_pairs(a);
    a.n_views = 1; a.views[0] = plain_view(ws + L.Ud, Hs + 1, Ws); a.in_H = Hs + 1; a.in_W = Ws;
    a.weights = packed + po.conv3_d; a.cout_total = 64; a.block_n = 64;
    a.act = ACT_NONE; a.out_mode = OUT_NHWC;
    a.mask_src = S > 0 ? conv3_in : nullptr;      // ReLU after the last PixelShuffle (src/models.py:73)
    a.out = S > 0 ? ws + L.dup[S - 1] : d_trunk;
    RC(launch_conv_gemm(a, st));
    e->launches += 1;
  }
  // ---- upsample stages, last to first
  for (int j = S - 1; j >= 0; --j) {
    const int Hj = H << j, Wj = W << j;
    const void* in_j = j > 0 ? ws + L.up[j - 1] : ws + L.trunk;
    if (pg) {
      snprintf(nm, sizeof(nm), "upsample.%d.bias", 3 * j);
      RC(launch_ps_bias_grad(ws + L.dup[j], N, Hj * 2, Wj * 2, reinterpret_cast<float*>(ws + L.ps_scratch),
                             e->grads + poff(*e, nm), st));
      e->launches += 2;
      snprintf(nm, sizeof(nm), "upsample.%d.weight", 3 * j);
      RC(wgrad(plain_view(in_j, Hj, Wj), Hj, Wj, false, Hj, Wj, ws + L.dup[j], 4, true, e->d_wg_idx_up, nm));
    }
    RC(dgrad3x3(ws + L.dup[j], Hj, Wj, true, po.up_d[j], nullptr, j > 0 ? in_j : nullptr, j > 0 ? ws + L.dup[j - 1] : d_trunk));
  }
  }
  // ---- conv2 (trunk = conv2(x_last) + out1)
  const void* x_last = e->n_res > 0 ? ws + L.out[e->n_res - 1] : ws + L.out1;
  if (pre && pg) RC(bias_grad(d_trunk, P, "conv2.bias"));
  // The 2*n_res + 1 trunk weight gradients run as ONE batched launch at the end of backward (wgrad3_batched_kernel):
  // x of layer l = 2*block + conv sits at out1 + l * 2 * slot (out[b-1] | z1[b] are two slots apart, conv2 reads out[last]),
  // dy of layer l at dyall + l * slot.  SRG_WGRAD_BATCHED=0 (or a non-uniform layout) keeps one launch per layer.
  const bool batched = wgrad_layout_batched(*e, N);
  if (!batched && pre && pg) RC(wgrad(plain_view(x_last, H, W), H, W, false, H, W, d_trunk, 1, false, e->d_wg_idx_c3x3, "conv2.weight"));
  const bool keep = e->keep_grads;
  void* dout = keep ? ws + L.kd_last : ws + L.g[0];
  void* dother = ws + L.g[1];
  void* dmid = ws + L.g[2];
  // the whole dgrad chain of the trunk (conv2, then every block's BatchNorm / ReLU / conv backward) in one launch
  const bool fused = batched && !frozen && use_trunk_fused(*e);
  const bool layers_here = !fused && phases == kPhaseAll;
  if (phases != kPhaseAll && !fused && !(batched && use_trunk_grouped(*e))) {
    set_error("generator_backward_phases: split execution needs the fused or the grouped per-layer trunk path");
    return -31;
  }
  if (fused) {
    if (mid) RC(run_trunk(e, 1, 0, st, pg));
    dout = ws + L.g[0] + L.slot * size_t(e->trunk_dout_idx);
  } else if (!layers_here) {
    // split execution on the per-layer path: generators_trunk() ran (or will run) the dgrad chain as grouped launches
    dout = layers_dout(*e);
  } else {
    RC(dgrad3x3(d_trunk, H, W, false, po.conv2_d, nullptr, nullptr, dout));
  }
  // ---- residual blocks, last to first (src/models.py:21-25)
  float* bwd = reinterpret_cast<float*>(ws + L.bwdcoef);
  auto bn_backward = [&](int b, int k, const void* dz, const void* y, void* dy) -> int {
    const float* coef = reinterpret_cast<const float*>(ws + L.bncoef) + size_t(2 * b + k) * 256;
    snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.weight", b, k + 1);
    const int64_t go = poff(*e, nm);
    snprintf(nm, sizeof(nm), "residual_blocks.%d.bn%d.bias", b, k + 1);
    const int64_t bo = poff(*e, nm);
    // sum dz and sum dz*y
    RC(launch_chan_reduce(dz, y, P, partials, st));
    const int rows = reduce_blocks(P);
    e->launches += 1;
    if (frozen) {
      // running statistics: no cross-rank exchange, dy = gamma * inv * dz, and the preceding conv's bias gets A * sum(dz)
      ReduceFinalize f; memset(&f, 0, sizeof(f));
      f.mode = RF_BN_BWD_FROZEN; f.count = double(P); f.gamma = e->master + go; f.save_mean = coef + 128; f.save_inv = coef + 192;
      if (pg) {
        snprintf(nm, sizeof(nm), "residual_blocks.%d.conv%d.bias", b, k + 1);
        f.dgamma = e->grads + go; f.dbeta = e->grads + bo; f.dbias = e->grads + poff(*e, nm);
      }
      f.out0 = bwd; f.out1 = bwd + 64; f.out2 = bwd + 128;
      RC(launch_partials_finalize(partials, rows, f, st));
      e->launches += 2;
      return launch_bn_bwd_apply(dz, y, bwd, bwd + 64, bwd + 128, dy, P, st);
    }
    float* dgamma = pg ? e->grads + go : nullptr;
    float* dbeta = pg ? e->grads + bo : nullptr;
    if (!e->allreduce || e->peer) {
      ReduceFinalize f; memset(&f, 0, sizeof(f));
      f.mode = RF_BN_BWD; f.count = double(P) * e->world; f.gamma = e->master + go; f.save_mean = coef + 128; f.save_inv = coef + 192;
      f.dgamma = dgamma; f.dbeta = dbeta; f.out0 = bwd; f.out1 = bwd + 64; f.out2 = bwd + 128;
      if (e->peer) RC(launch_peer_finalize(e->peer, partials, rows, f, st));
      else RC(launch_partials_finalize(partials, rows, f, st));
      e->launches += 2;
    } else {
      RC(launch_partials_sums(partials, rows, sums, st));
      RC(e->allreduce(e->allreduce_ctx, sums, 128, st));
      RC(launch_bn_bwd_finalize(sums, double(P) * e->world, e->master + go, coef + 128, coef + 192, dgamma, dbeta,
                                bwd, bwd + 64, bwd + 128, 1.f / float(e->world), st));
      e->launches += 4;
    }
    return launch_bn_bwd_apply(dz, y, bwd, bwd + 64, bwd + 128, dy, P, st);
  };
  for (int b = e->n_res - 1; b >= 0 && layers_here; --b) {
    const void* x_in = b > 0 ? ws + L.out[b - 1] : ws + L.out1;
    void* d_y2 = ws + L.dyall + L.slot * size_t(2 * b + 1);
    void* d_p1 = keep ? ws + L.kd_p1[b] : dother;
    void* d_y1 = ws + L.dyall + L.slot * size_t(2 * b);
    void* d_in = keep ? ws + L.kd_in[b] : dother;
    // out = bn2(y2) + x
    RC(bn_backward(b, 1, dout, ws + L.y2[b], d_y2));
    snprintf(nm, sizeof(nm), "residual_blocks.%d.conv2.weight", b);
    if (!batched && pg) RC(wgrad(plain_view(ws + L.z1[b], H, W), H, W, false, H, W, d_y2, 1, false, e->d_wg_idx_c3x3, nm));
    RC(dgrad3x3(d_y2, H, W, false, po.rb_d[1][b], nullptr, ws + L.z1[b], d_p1));   // ReLU backward via mask
    // z1 = relu(bn1(y1))
    RC(bn_backward(b, 0, d_p1, ws + L.y1[b], d_y1));
    snprintf(nm, sizeof(nm), "residual_blocks.%d.conv1.weight", b);
    if (!batched && pg) RC(wgrad(plain_view(x_in, H, W), H, W, false, H, W, d_y1, 1, false, e->d_wg_idx_c3x3, nm));
    RC(dgrad3x3(d_y1, H, W, false, po.rb_d[0][b], dout, nullptr, d_in));   // + skip gradient
    if (keep) { dout = d_in; } else { void* t = dout; dout = dother; dother = t; }
  }
  if (!post) return 0;
  // ---- conv1: out1 = lrelu(conv1(x)); d(out1) = block-chain gradient + trunk skip gradient
  if (keep) dmid = ws + L.kd_c1;
  RC(launch_lrelu_bwd_add2(dout, d_trunk, ws + L.out1, kSlope, dmid, P, st));
  e->launches += 1;
  if (dlr != nullptr) {
    // d(lr): 9x9 64 -> 3 conv of d(pre-LeakyReLU) with the flipped filter, through the fold9 path of conv3's forward
    ConvGemmArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = H; a.W = W; a.TH = 4; a.TW = 32;
    a.n_strips = 1; a.n_taps = 9; a.strip_rows = 12; a.strip_dh = -4; a.strip_dw[0] = 0;
    for (int r = 0; r < 9; ++r) a.tap_row[r] = r;
    a.n_views = 1; a.views[0] = plain_view(dmid, H, W); a.in_H = H; a.in_W = W;
    a.weights = reinterpret_cast<const uint16_t*>(ws + L.c1d); a.cout_total = 32; a.block_n = 32;
    a.bias = nullptr; a.act = ACT_NONE; a.out = dlr; a.out_mode = OUT_FOLD9_NCHW;
    RC(launch_conv_gemm(a, st));
    e->launches += 1;
  }
  if (!pg) return 0;
  RC(bias_grad(dmid, P, "conv1.bias"));
  RC(wgrad(plain_view(ws + L.U1, H + 1, W), H + 1, W, true, H, W, dmid, 1, false, e->d_wg_idx_conv1, "conv1.weight"));
  if (batched) {
    WgradBatchArgs a; memset(&a, 0, sizeof(a));
    a.N = N; a.H = H; a.W = W; a.n_layers = 2 * e->n_res + 1;
    a.x_base = ws + L.out1; a.x_layer_stride_bytes = int64_t(2 * L.slot);
    a.dy_base = ws + L.dyall; a.dy_layer_stride_bytes = int64_t(L.slot);
    a.partials = reinterpret_cast<float*>(ws + L.wgb_partials);
    a.inv = e->d_wg_idx_c3x3; a.grads = e->grads; a.out_off = e->d_wgb_off;
    if (wgrad3_batched_partials_floats(a) > L.wgb_floats) { set_error("batched wgrad partials exceed workspace"); return -27; }
    RC(launch_wgrad3x3_batched(a, st));
    e->launches += 2;
  }
  return 0;
}
}  // namespace

int generator_backward(GeneratorEngine* g, const float* dsr, cudaStream_t st) {
  return generator_backward_phases(g, dsr, kPhaseAll, st);
}

int generator_backward_phases(GeneratorEngine* g, const float* dsr, int phases, cudaStream_t st) {
  return backward_impl(static_cast<EngineImpl*>(g), dsr, phases, true, nullptr, st);
}

int generator_backward_ex(GeneratorEngine* g, const float* dsr, int param_grads, float* dlr, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  if (dsr == nullptr) { set_error("generator_backward_ex: null d(sr)"); return -22; }
  if (param_grads == 0 && dlr == nullptr) { set_error("generator_backward_ex: nothing to compute (param_grads == 0 and dlr == NULL)"); return -22; }
  if (!e->ws || !e->ws_training) { set_error("generator_backward_ex: needs a training-sized bound workspace"); return -25; }
  return backward_impl(e, dsr, kPhaseAll, param_grads != 0, dlr, st);
}

// Staging buffers of srg_generator_backward_tiles, in workspace regions that are dead while they are live:
//  - the window-shaped, crop-masked d(SR) (n x 3 x Hs x Ws fp32, 12 B per HR pixel) sits in dup[S-1] (128 B per HR
//    pixel), or in g[3] = d(trunk) (one 128 B-per-pixel slot) when S = 0.  backward_impl reads it only in its first two
//    launches (unfold9 into Ud, the conv3.bias sum); the first write to dup[S-1] / g[3] is conv3's data gradient, which
//    reads Ud.  debug_keep_grads changes neither buffer (its kd_* buffers are separate; g[3] stays the conv2 slot).
//  - conv1's window-shaped data gradient (n x 3 x H x W fp32) goes to Ud (128 B per HR pixel), which only conv3's
//    bias sum, weight gradient and data gradient read, all of them enqueued before conv1's data gradient.
int generator_backward_tiles(GeneratorEngine* g, const float* dsr, int param_grads, float* dlr, cudaStream_t st) {
  EngineImpl* e = static_cast<EngineImpl*>(g);
  if (dsr == nullptr) { set_error("srg_generator_backward_tiles: null d(sr)"); return -22; }
  if (param_grads == 0 && dlr == nullptr) { set_error("srg_generator_backward_tiles: nothing to compute (param_grads == 0 and dlr == NULL)"); return -22; }
  if (!e->ws || !e->ws_training) { set_error("srg_generator_backward_tiles: needs a training-sized bound workspace"); return -25; }
  if (e->tile_n < 1) { set_error("srg_generator_backward_tiles: no preceding srg_generator_forward_frozen_tiles"); return -32; }
  const int S = e->n_up, n = e->tile_n;
  WindowTable hr, lr;
  memset(&hr, 0, sizeof(hr));
  hr.n = n; hr.fh = e->tile_H << S; hr.fw = e->tile_W << S;
  for (int i = 0; i < n; ++i) {
    const TileDesc& t = e->tile_tab[i];
    hr.frame[i] = t.frame; hr.y0[i] = t.y0 << S; hr.x0[i] = t.x0 << S;
    hr.h_lo[i] = t.crop_y0 << S; hr.h_hi[i] = (t.crop_y0 + t.crop_h) << S;
    hr.w_lo[i] = t.crop_x0 << S; hr.w_hi[i] = (t.crop_x0 + t.crop_w) << S;
  }
  lr = hr;
  lr.fh = e->tile_H; lr.fw = e->tile_W;
  for (int i = 0; i < n; ++i) {
    const TileDesc& t = e->tile_tab[i];
    lr.y0[i] = t.y0; lr.x0[i] = t.x0;
    lr.h_lo[i] = t.crop_y0; lr.h_hi[i] = t.crop_y0 + t.crop_h; lr.w_lo[i] = t.crop_x0; lr.w_hi[i] = t.crop_x0 + t.crop_w;
  }
  float* dsr_win = reinterpret_cast<float*>(e->ws + (S > 0 ? e->L.dup[S - 1] : e->L.g[3]));
  float* dlr_win = reinterpret_cast<float*>(e->ws + e->L.Ud);
  RC(launch_crop_masked_gather(dsr, hr, e->H << S, e->W << S, dsr_win, st));
  e->launches += 1;
  RC(backward_impl(e, dsr_win, kPhaseAll, param_grads != 0, dlr ? dlr_win : nullptr, st, n));
  if (dlr == nullptr) return 0;
  e->launches += 1;
  return launch_window_scatter_add(dlr_win, lr, e->H, e->W, dlr, st);
}

}  // namespace srg
