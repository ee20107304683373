// C ABI of libsrgan_b200.so (declared in include/srgan_b200.h): thin wrappers over the internal launchers.
#include "../../include/srgan_b200.h"

#include <dlfcn.h>
#include <stdio.h>
#include <string.h>

#include "conv_gemm.cuh"
#include "conv_ops.cuh"
#include "elementwise.cuh"
#include "discriminator.cuh"
#include "generator.cuh"
#include "metrics.cuh"
#include "peer_sync.cuh"
#include "resample.cuh"
#include "trunk_fused.cuh"
#include "vgg_ops.cuh"

using namespace srg;

namespace {
inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline GeneratorEngine* G(srg_generator_t* g) { return reinterpret_cast<GeneratorEngine*>(g); }
inline const GeneratorEngine* G(const srg_generator_t* g) { return reinterpret_cast<const GeneratorEngine*>(g); }
void copy_name(const std::string& s, char* dst, int cap) {
  if (dst == nullptr || cap <= 0) return;
  snprintf(dst, size_t(cap), "%s", s.c_str());
}

// ---- NCCL through dlopen (the library torch bundles is already mapped in a training process) -------------------
struct NcclId { char internal[128]; };
typedef void* NcclComm;
typedef int (*GetUniqueIdFn)(NcclId*);
typedef int (*CommInitRankFn)(NcclComm*, int, NcclId, int);
typedef int (*AllReduceFn)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t);
typedef int (*CommDestroyFn)(NcclComm);
typedef const char* (*GetErrorStringFn)(int);
struct NcclApi {
  void* handle = nullptr;
  GetUniqueIdFn get_unique_id = nullptr;
  CommInitRankFn comm_init_rank = nullptr;
  AllReduceFn all_reduce = nullptr;
  CommDestroyFn comm_destroy = nullptr;
  GetErrorStringFn error_string = nullptr;
} g_nccl;
constexpr int kNcclFloat32 = 7, kNcclFloat64 = 8, kNcclSum = 0, kNcclAvg = 4;

int nccl_load() {
  if (g_nccl.handle) return 0;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.handle) break;
  }
  if (!g_nccl.handle) { set_error("dlopen(libnccl.so.2) failed: %s", dlerror()); return -40; }
  g_nccl.get_unique_id = reinterpret_cast<GetUniqueIdFn>(dlsym(g_nccl.handle, "ncclGetUniqueId"));
  g_nccl.comm_init_rank = reinterpret_cast<CommInitRankFn>(dlsym(g_nccl.handle, "ncclCommInitRank"));
  g_nccl.all_reduce = reinterpret_cast<AllReduceFn>(dlsym(g_nccl.handle, "ncclAllReduce"));
  g_nccl.comm_destroy = reinterpret_cast<CommDestroyFn>(dlsym(g_nccl.handle, "ncclCommDestroy"));
  g_nccl.error_string = reinterpret_cast<GetErrorStringFn>(dlsym(g_nccl.handle, "ncclGetErrorString"));
  if (!g_nccl.get_unique_id || !g_nccl.comm_init_rank || !g_nccl.all_reduce || !g_nccl.comm_destroy) {
    set_error("libnccl is missing a required symbol");
    return -41;
  }
  return 0;
}
int nccl_check(int rc, const char* what) {
  if (rc == 0) return 0;
  set_error("%s: NCCL error %d (%s)", what, rc, g_nccl.error_string ? g_nccl.error_string(rc) : "?");
  return -42;
}
}  // namespace

extern "C" {

int srg_abi_version(void) { return SRG_ABI_VERSION; }
const char* srg_last_error(void) { return last_error(); }

int srg_generator_create(srg_generator_t** out, int N, int H, int W, int num_residuals, int num_upsample_stages) {
  if (out == nullptr) { set_error("srg_generator_create: null out"); return -1; }
  GeneratorEngine* g = generator_create(N, H, W, num_residuals, num_upsample_stages);
  if (g == nullptr) return -2;
  *out = reinterpret_cast<srg_generator_t*>(g);
  return 0;
}
void srg_generator_destroy(srg_generator_t* g) { delete G(g); }

int srg_generator_num_params(const srg_generator_t* g) { return int(G(g)->params.size()); }
int64_t srg_generator_param_elems(const srg_generator_t* g) { return G(g)->param_elems; }
int srg_generator_param_info(const srg_generator_t* g, int i, char* name, int name_cap, int64_t* offset, int64_t* numel,
                             int* ndim, int* shape4) {
  const GeneratorEngine* e = G(g);
  if (i < 0 || i >= int(e->params.size())) { set_error("param index out of range"); return -3; }
  const ParamInfo& p = e->params[size_t(i)];
  copy_name(p.name, name, name_cap);
  if (offset) *offset = p.offset;
  if (numel) *numel = p.numel;
  if (ndim) *ndim = p.ndim;
  if (shape4) for (int k = 0; k < 4; ++k) shape4[k] = p.shape[k];
  return 0;
}
int srg_generator_num_buffers(const srg_generator_t* g) { return int(G(g)->buffers.size()); }
int64_t srg_generator_buffer_elems(const srg_generator_t* g) { return G(g)->buffer_elems; }
int srg_generator_buffer_info(const srg_generator_t* g, int i, char* name, int name_cap, int64_t* offset, int64_t* numel) {
  const GeneratorEngine* e = G(g);
  if (i < 0 || i >= int(e->buffers.size())) { set_error("buffer index out of range"); return -3; }
  const BufferInfo& b = e->buffers[size_t(i)];
  copy_name(b.name, name, name_cap);
  if (offset) *offset = b.offset;
  if (numel) *numel = b.numel;
  return 0;
}
size_t srg_generator_workspace_bytes(const srg_generator_t* g, int training) {
  return training ? G(g)->workspace_bytes_train : G(g)->workspace_bytes_eval;
}
int srg_generator_bind(srg_generator_t* g, float* params, float* grads, float* bn_buffers, void* workspace,
                       size_t workspace_bytes, int training) {
  return generator_bind(G(g), params, grads, bn_buffers, workspace, workspace_bytes, training);
}
int srg_generator_set_grads(srg_generator_t* g, float* grads) {
  if (grads == nullptr) { set_error("srg_generator_set_grads: null buffer"); return -22; }
  G(g)->grads = grads;
  return 0;
}
int srg_generator_pack(srg_generator_t* g, void* stream) { return generator_pack(G(g), S(stream)); }
int srg_generator_forward(srg_generator_t* g, const float* lr_nchw, float* sr_nchw, int training, int update_running,
                          void* stream) {
  return generator_forward(G(g), lr_nchw, sr_nchw, training, update_running, S(stream));
}
int srg_generator_backward(srg_generator_t* g, const float* dsr_nchw, void* stream) {
  return generator_backward(G(g), dsr_nchw, S(stream));
}
int srg_generator_forward_frozen(srg_generator_t* g, const float* lr_nchw, float* sr_nchw, void* stream) {
  if (g == nullptr) { set_error("srg_generator_forward_frozen: null engine"); return -1; }
  return generator_forward_frozen(G(g), lr_nchw, sr_nchw, S(stream));
}
static_assert(sizeof(srg_tile_t) == sizeof(TileDesc) && SRG_MAX_TILES == kMaxTiles, "srg_tile_t mirrors srg::TileDesc");
int srg_generator_tile_halo(int num_residuals, int num_upsample_stages) {
  return generator_tile_halo(num_residuals, num_upsample_stages);
}
int srg_generator_forward_tiles(srg_generator_t* g, const float* frames_nchw, int F, int H, int W, const srg_tile_t* tiles,
                                int n, float* sr_nchw, void* stream) {
  if (g == nullptr) { set_error("srg_generator_forward_tiles: null engine"); return -1; }
  return generator_forward_tiles(G(g), frames_nchw, F, H, W, reinterpret_cast<const TileDesc*>(tiles), n, sr_nchw, S(stream));
}
int srg_generator_forward_u8(srg_generator_t* g, const uint8_t* lr_nhwc, uint8_t* sr_nhwc, void* stream) {
  if (g == nullptr) { set_error("srg_generator_forward_u8: null engine"); return -1; }
  return generator_forward_u8(G(g), lr_nhwc, sr_nhwc, S(stream));
}
int srg_generator_forward_tiles_u8(srg_generator_t* g, const uint8_t* frames_nhwc, int F, int H, int W,
                                   const srg_tile_t* tiles, int n, uint8_t* sr_nhwc, void* stream) {
  if (g == nullptr) { set_error("srg_generator_forward_tiles_u8: null engine"); return -1; }
  return generator_forward_tiles_u8(G(g), frames_nhwc, F, H, W, reinterpret_cast<const TileDesc*>(tiles), n, sr_nhwc,
                                    S(stream));
}
int srg_generator_forward_frozen_tiles(srg_generator_t* g, const float* frames_nchw, int F, int H, int W,
                                       const srg_tile_t* tiles, int n, float* sr_nchw, void* stream) {
  if (g == nullptr) { set_error("srg_generator_forward_frozen_tiles: null engine"); return -1; }
  return generator_forward_frozen_tiles(G(g), frames_nchw, F, H, W, reinterpret_cast<const TileDesc*>(tiles), n, sr_nchw,
                                        S(stream));
}
int srg_generator_backward_tiles(srg_generator_t* g, const float* dsr_nchw, int param_grads, float* dlr_nchw, void* stream) {
  if (g == nullptr) { set_error("srg_generator_backward_tiles: null engine"); return -1; }
  return generator_backward_tiles(G(g), dsr_nchw, param_grads, dlr_nchw, S(stream));
}
int srg_generator_backward_ex(srg_generator_t* g, const float* dsr_nchw, int param_grads, float* dlr_nchw, void* stream) {
  if (g == nullptr) { set_error("srg_generator_backward_ex: null engine"); return -1; }
  return generator_backward_ex(G(g), dsr_nchw, param_grads, dlr_nchw, S(stream));
}
int srg_generator_num_tensors(const srg_generator_t* g) { return int(G(g)->tensors.size()); }
int srg_generator_tensor_info(const srg_generator_t* g, int i, char* name, int name_cap, int64_t* byte_offset, int* dims4,
                              int* dtype) {
  const GeneratorEngine* e = G(g);
  if (i < 0 || i >= int(e->tensors.size())) { set_error("tensor index out of range"); return -3; }
  const TensorInfo& t = e->tensors[size_t(i)];
  copy_name(t.name, name, name_cap);
  if (byte_offset) *byte_offset = t.byte_offset;
  if (dims4) for (int k = 0; k < 4; ++k) dims4[k] = t.dims[k];
  if (dtype) *dtype = t.dtype;
  return 0;
}
long long srg_generator_launch_count(const srg_generator_t* g) { return G(g)->launches; }
long long srg_total_launches(void) { return total_launches(); }
int srg_set_conv_variant(int variant) { return set_conv_variant(variant); }
int srg_conv9_rows_window(int ri, int* jlo, int* jhi, int* slot_lo, int* fresh) {
  if (ri < 0 || ri > 15) { set_error("conv9_rows_window: ri must be 0..15"); return -1; }
  const C9Window w = c9_window(ri);
  if (jlo) *jlo = w.jlo;
  if (jhi) *jhi = w.jhi;
  if (slot_lo) *slot_lo = w.slot_lo;
  if (fresh) *fresh = w.fresh;
  return 0;
}
int srg_wgrad_batched_plan(int N, int H, int W, int layers, int* tiles_per_layer, int* grid, int* per_cta, int* max_slots) {
  WgradBatchArgs a;
  memset(&a, 0, sizeof(a));
  a.N = N; a.H = H; a.W = W; a.n_layers = layers;
  int t = 0, g = 0, p = 0, m = 0;
  wgrad3_batched_plan(a, &t, &g, &p, &m);
  if (tiles_per_layer) *tiles_per_layer = t;
  if (grid) *grid = g;
  if (per_cta) *per_cta = p;
  if (max_slots) *max_slots = m;
  return 0;
}
int srg_generator_set_keep_grads(srg_generator_t* g, int keep) { return generator_set_keep_grads(G(g), keep); }
int srg_generator_profile_enable(srg_generator_t* g, int on) { return generator_profile_enable(G(g), on); }
int srg_generator_profile_read(srg_generator_t* g, double* ms_sum, long long* count) {
  return generator_profile_read(G(g), ms_sum, count);
}

int srg_generator_forward_phases(srg_generator_t* g, const float* lr, float* sr, int training, int update_running, int phases,
                                 void* stream) {
  return generator_forward_phases(G(g), lr, sr, training, update_running, phases, S(stream));
}
int srg_generator_backward_phases(srg_generator_t* g, const float* dsr, int phases, void* stream) {
  return generator_backward_phases(G(g), dsr, phases, S(stream));
}
int srg_generators_trunk(srg_generator_t* const* gs, int n, int backward, int update_running, void* stream) {
  GeneratorEngine* es[8];
  if (n < 1 || n > 8) { set_error("srg_generators_trunk: bad engine count"); return -62; }
  for (int i = 0; i < n; ++i) es[i] = G(gs[i]);
  return generators_trunk(es, n, backward, update_running, S(stream));
}
// ---- per-operator BatchNorm entry points
int srg_bn_stats_rows(int64_t pixels) { return reduce_blocks(pixels); }
int srg_bn_stats(const void* a, const void* b, int64_t pixels, float* partials, void* stream) {
  if (a == nullptr || partials == nullptr || pixels < 1) { set_error("srg_bn_stats: bad arguments"); return -70; }
  return launch_chan_reduce(a, b, pixels, partials, S(stream));
}
int srg_bn_finalize(const float* partials, int rows, double count, const float* gamma, const float* beta, float eps,
                    float momentum, float* running_mean, float* running_var, float* scale, float* shift, float* save_mean,
                    float* save_inv, void* stream) {
  if (!partials || rows < 1 || !gamma || !beta || !scale || !shift || !save_mean || !save_inv) { set_error("srg_bn_finalize: bad arguments"); return -70; }
  ReduceFinalize f; memset(&f, 0, sizeof(f));
  f.mode = RF_BN_FWD; f.count = count; f.eps = eps; f.momentum = momentum; f.gamma = gamma; f.beta = beta;
  f.running_mean = running_mean; f.running_var = running_var;
  f.out0 = scale; f.out1 = shift; f.out2 = save_mean; f.out3 = save_inv;
  return launch_partials_finalize(partials, rows, f, S(stream));
}
int srg_bn_apply(const void* y, const float* scale, const float* shift, const void* skip, int relu, void* out, int64_t pixels,
                 void* stream) {
  if (!y || !scale || !shift || !out || pixels < 1) { set_error("srg_bn_apply: bad arguments"); return -70; }
  return launch_bn_apply(y, scale, shift, skip, relu, out, pixels, S(stream));
}
int srg_bn_backward_finalize(const float* partials, int rows, double count, const float* gamma, const float* save_mean,
                             const float* save_inv, float* dgamma, float* dbeta, float* coef_a, float* coef_b, float* coef_c,
                             void* stream) {
  if (!partials || rows < 1 || !gamma || !save_mean || !save_inv || !coef_a || !coef_b || !coef_c) { set_error("srg_bn_backward_finalize: bad arguments"); return -70; }
  ReduceFinalize f; memset(&f, 0, sizeof(f));
  f.mode = RF_BN_BWD; f.count = count; f.gamma = gamma; f.save_mean = save_mean; f.save_inv = save_inv;
  f.dgamma = dgamma; f.dbeta = dbeta; f.out0 = coef_a; f.out1 = coef_b; f.out2 = coef_c;
  return launch_partials_finalize(partials, rows, f, S(stream));
}
int srg_bn_backward_apply(const void* dout, const void* y, const float* coef_a, const float* coef_b, const float* coef_c,
                          void* dy, int64_t pixels, void* stream) {
  if (!dout || !y || !coef_a || !coef_b || !coef_c || !dy || pixels < 1) { set_error("srg_bn_backward_apply: bad arguments"); return -70; }
  return launch_bn_bwd_apply(dout, y, coef_a, coef_b, coef_c, dy, pixels, S(stream));
}

int srg_set_trunk_fused(int on) { return set_trunk_fused(on); }
int srg_debug_trunk_prof(long long* host, int n) { return trunk_prof_read(host, n); }
int srg_generator_trunk_layers(const srg_generator_t* g) { return generator_prof_layers(G(g)); }
int srg_generator_trunk_error(srg_generator_t* g) { return generator_trunk_error(G(g)); }

int srg_generator_set_allreduce(srg_generator_t* g, srg_allreduce_f64_fn fn, void* ctx, int world) {
  if (world < 1) { set_error("set_allreduce: world < 1"); return -4; }
  GeneratorEngine* e = G(g);
  e->allreduce = reinterpret_cast<AllreduceF64Fn>(fn);
  e->allreduce_ctx = ctx;
  e->world = world;
  return 0;
}

int srg_nccl_unique_id(void* out128) {
  int rc = nccl_load();
  if (rc) return rc;
  NcclId id;
  rc = nccl_check(g_nccl.get_unique_id(&id), "ncclGetUniqueId");
  if (rc) return rc;
  memcpy(out128, &id, 128);
  return 0;
}
int srg_nccl_comm_create(const void* unique_id128, int world, int rank, void** comm_out) {
  int rc = nccl_load();
  if (rc) return rc;
  if (comm_out == nullptr || unique_id128 == nullptr || world < 1 || rank < 0 || rank >= world) {
    set_error("srg_nccl_comm_create: bad arguments");
    return -43;
  }
  NcclId id;
  memcpy(&id, unique_id128, 128);
  NcclComm comm = nullptr;
  rc = nccl_check(g_nccl.comm_init_rank(&comm, world, id, rank), "ncclCommInitRank");
  if (rc) return rc;
  *comm_out = comm;
  return 0;
}
void srg_nccl_comm_destroy(void* comm) {
  if (comm != nullptr && g_nccl.comm_destroy) g_nccl.comm_destroy(comm);
}
int srg_nccl_allreduce_f64(void* comm, double* buf, int n, void* stream) {
  if (comm == nullptr) { set_error("NCCL communicator is null"); return -44; }
  return nccl_check(g_nccl.all_reduce(buf, buf, size_t(n), kNcclFloat64, kNcclSum, comm, S(stream)), "ncclAllReduce");
}
int srg_nccl_allreduce_f32(void* comm, float* buf, int64_t n, void* stream) {
  if (comm == nullptr) { set_error("NCCL communicator is null"); return -44; }
  return nccl_check(g_nccl.all_reduce(buf, buf, size_t(n), kNcclFloat32, kNcclSum, comm, S(stream)), "ncclAllReduce");
}
int srg_nccl_allreduce_mean_f32(void* comm, float* buf, int64_t n, void* stream) {
  if (comm == nullptr) { set_error("NCCL communicator is null"); return -44; }
  return nccl_check(g_nccl.all_reduce(buf, buf, size_t(n), kNcclFloat32, kNcclAvg, comm, S(stream)), "ncclAllReduce(avg)");
}
int srg_generator_use_nccl(srg_generator_t* g, void* comm, int world) {
  if (comm == nullptr) { set_error("NCCL communicator is null"); return -44; }
  return srg_generator_set_allreduce(g, srg_nccl_allreduce_f64, comm, world);
}

// ---- NVLink peer-memory SyncBatchNorm exchange ----------------------------------------------------------------------
int srg_peer_sync_create(srg_peer_sync_t** out, int world, int rank) {
  if (out == nullptr) { set_error("srg_peer_sync_create: null out"); return -1; }
  PeerSync* ps = peer_sync_create(world, rank);
  if (ps == nullptr) return -2;
  *out = reinterpret_cast<srg_peer_sync_t*>(ps);
  return 0;
}
int srg_peer_sync_handle(srg_peer_sync_t* ps, void* out64) { return peer_sync_handle(reinterpret_cast<PeerSync*>(ps), out64); }
int srg_peer_sync_connect(srg_peer_sync_t* ps, const void* handles) {
  return peer_sync_connect(reinterpret_cast<PeerSync*>(ps), handles);
}
void srg_peer_sync_destroy(srg_peer_sync_t* ps) { peer_sync_destroy(reinterpret_cast<PeerSync*>(ps)); }
int srg_peer_sync_error(srg_peer_sync_t* ps) { return peer_sync_error(reinterpret_cast<PeerSync*>(ps)); }
int srg_generator_use_peer_sync(srg_generator_t* g, srg_peer_sync_t* ps) {
  if (ps == nullptr) { set_error("srg_generator_use_peer_sync: null"); return -45; }
  GeneratorEngine* e = G(g);
  e->peer = reinterpret_cast<PeerSync*>(ps);
  e->world = peer_sync_world(e->peer);
  return 0;
}

// ---- discriminator ------------------------------------------------------------------------------------------------
static inline DiscriminatorEngine* D(srg_discriminator_t* d) { return reinterpret_cast<DiscriminatorEngine*>(d); }
static inline const DiscriminatorEngine* DC(const srg_discriminator_t* d) { return reinterpret_cast<const DiscriminatorEngine*>(d); }
int srg_discriminator_create(srg_discriminator_t** out, int N, int H, int W) {
  if (out == nullptr) { set_error("srg_discriminator_create: null out"); return -1; }
  DiscriminatorEngine* d = discriminator_create(N, H, W);
  if (d == nullptr) return -2;
  *out = reinterpret_cast<srg_discriminator_t*>(d);
  return 0;
}
void srg_discriminator_destroy(srg_discriminator_t* d) { delete D(d); }
int srg_discriminator_output_hw(const srg_discriminator_t* d, int* h, int* w) {
  if (h) *h = DC(d)->st[3].Hp;
  if (w) *w = DC(d)->st[3].Wp;
  return 0;
}
int srg_discriminator_num_params(const srg_discriminator_t* d) { return int(DC(d)->params.size()); }
int64_t srg_discriminator_param_elems(const srg_discriminator_t* d) { return DC(d)->param_elems; }
int srg_discriminator_param_info(const srg_discriminator_t* d, int i, char* name, int name_cap, int64_t* offset,
                                 int64_t* numel, int* ndim, int* shape4) {
  const DiscriminatorEngine* e = DC(d);
  if (i < 0 || i >= int(e->params.size())) { set_error("param index out of range"); return -3; }
  const ParamInfo& p = e->params[size_t(i)];
  copy_name(p.name, name, name_cap);
  if (offset) *offset = p.offset;
  if (numel) *numel = p.numel;
  if (ndim) *ndim = p.ndim;
  if (shape4) for (int k = 0; k < 4; ++k) shape4[k] = p.shape[k];
  return 0;
}
size_t srg_discriminator_workspace_bytes(const srg_discriminator_t* d, int training) {
  return training ? DC(d)->workspace_bytes_train : DC(d)->workspace_bytes_eval;
}
int srg_discriminator_bind(srg_discriminator_t* d, float* params, float* grads, void* workspace, size_t workspace_bytes,
                           int training) {
  return discriminator_bind(D(d), params, grads, workspace, workspace_bytes, training);
}
int srg_discriminator_set_grads(srg_discriminator_t* d, float* grads) {
  if (grads == nullptr) { set_error("srg_discriminator_set_grads: null buffer"); return -22; }
  D(d)->grads = grads;
  return 0;
}
int srg_discriminator_pack(srg_discriminator_t* d, void* stream) { return discriminator_pack(D(d), S(stream)); }
int srg_discriminator_forward(srg_discriminator_t* d, const float* x_nchw, float* out_nchw, void* stream) {
  return discriminator_forward(D(d), x_nchw, out_nchw, 1, S(stream));
}
int srg_discriminator_backward(srg_discriminator_t* d, const float* dout_nchw, int param_grads, float* dx_nchw,
                               void* stream) {
  return discriminator_backward(D(d), dout_nchw, param_grads, dx_nchw, S(stream));
}
int srg_discriminator_num_tensors(const srg_discriminator_t* d) { return int(DC(d)->tensors.size()); }
int srg_discriminator_tensor_info(const srg_discriminator_t* d, int i, char* name, int name_cap, int64_t* byte_offset,
                                  int* dims4, int* dtype) {
  const DiscriminatorEngine* e = DC(d);
  if (i < 0 || i >= int(e->tensors.size())) { set_error("tensor index out of range"); return -3; }
  const TensorInfo& t = e->tensors[size_t(i)];
  copy_name(t.name, name, name_cap);
  if (byte_offset) *byte_offset = t.byte_offset;
  if (dims4) for (int k = 0; k < 4; ++k) dims4[k] = t.dims[k];
  if (dtype) *dtype = t.dtype;
  return 0;
}

size_t srg_recon_loss_scratch_bytes(void) { return size_t(loss_scratch_doubles()) * 8; }
int srg_recon_loss_forward(const float* hr_nchw, const float* sr_nchw, int N, int C, int H, int W, void* scratch,
                           size_t scratch_bytes, float* e_buf, float* g_buf, float* losses2, void* stream) {
  if (scratch_bytes < srg_recon_loss_scratch_bytes()) { set_error("recon_loss: scratch too small"); return -5; }
  if (!hr_nchw || !sr_nchw || !scratch || !e_buf || !g_buf || !losses2) { set_error("recon_loss: null pointer"); return -6; }
  return launch_recon_loss_forward(hr_nchw, sr_nchw, N, C, H, W, reinterpret_cast<double*>(scratch), e_buf, g_buf, losses2,
                                   S(stream));
}
int srg_recon_loss_backward(const float* hr_nchw, const float* sr_nchw, int N, int C, int H, int W, const void* scratch,
                            const float* e_buf, const float* g_buf, const float* w_edge, const float* w_tv, float* grad_sr,
                            float grad_scale, void* stream) {
  if (!hr_nchw || !sr_nchw || !scratch || !e_buf || !g_buf || !grad_sr) { set_error("recon_loss_backward: null pointer"); return -6; }
  return launch_recon_loss_backward(hr_nchw, sr_nchw, N, C, H, W, reinterpret_cast<const double*>(scratch), e_buf, g_buf,
                                    w_edge, w_tv, grad_sr, grad_scale, S(stream));
}
int srg_tanh_mean(const float* a, const float* b, int64_t n, float sign, void* scratch, size_t scratch_bytes, float* out1,
                  float* da, float* db, float grad_scale, void* stream) {
  if (scratch_bytes < srg_recon_loss_scratch_bytes()) { set_error("tanh_mean: scratch too small"); return -5; }
  return launch_tanh_mean(a, b, n, sign, reinterpret_cast<double*>(scratch), out1, da, db, grad_scale, S(stream));
}
int srg_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, int step, float grad_scale, void* stream) {
  if (step < 1) { set_error("adam: step must be >= 1"); return -7; }
  return launch_adam(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, step, grad_scale, S(stream));
}

int srg_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, const float* lr_dev,
                      float beta1, float beta2, float eps, int* step_dev, float grad_scale, void* stream) {
  if (lr_dev == nullptr || step_dev == nullptr) { set_error("adam_dev: null device scalar"); return -7; }
  return launch_adam_dev(params, grads, exp_avg, exp_avg_sq, n, lr_dev, beta1, beta2, eps, step_dev, grad_scale, S(stream));
}

int srg_point_loss(int kind, const float* a, const float* b, int64_t n, void* scratch, size_t scratch_bytes, float* out1,
                   float* grad_a, float grad_scale, void* stream) {
  if (scratch_bytes < srg_recon_loss_scratch_bytes()) { set_error("point_loss: scratch too small"); return -5; }
  if (!a || !b || !out1) { set_error("point_loss: null pointer"); return -6; }
  return launch_point_loss(kind, a, b, n, reinterpret_cast<double*>(scratch), out1, grad_a, grad_scale, S(stream));
}
int srg_image_enhance(const float* x_nchw, int N, int C, int H, int W, float factor, float* out_nchw, void* stream) {
  if (!x_nchw || !out_nchw) { set_error("image_enhance: null pointer"); return -6; }
  return launch_image_enhance(x_nchw, N, C, H, W, factor, out_nchw, S(stream));
}
int srg_mse(const float* a, const float* b, int64_t n, void* scratch, size_t scratch_bytes, double* out1, void* stream) {
  if (scratch_bytes < srg_recon_loss_scratch_bytes()) { set_error("mse: scratch too small"); return -5; }
  if (!a || !b || !out1) { set_error("mse: null pointer"); return -6; }
  return launch_mse(a, b, n, reinterpret_cast<double*>(scratch), out1, S(stream));
}
size_t srg_image_metrics_scratch_bytes(int N, int H, int W) { return image_metrics_scratch_bytes(N, H, W); }
int srg_image_metrics(const float* sr, const float* hr, int N, int C, int H, int W, void* scratch, size_t scratch_bytes,
                      double* psnr_out, double* ssim_out, void* stream) {
  if (N < 1 || C != 3 || H < 3 || W < 3) {
    set_error("image_metrics: need N >= 1 images of 3 x H x W with H, W >= 3 (got N=%d C=%d H=%d W=%d)", N, C, H, W);
    return -100;
  }
  if (!sr || !hr || !scratch || !psnr_out || !ssim_out) { set_error("image_metrics: null pointer"); return -6; }
  if (scratch_bytes < image_metrics_scratch_bytes(N, H, W)) {
    set_error("image_metrics: scratch too small (%zu < %zu bytes)", scratch_bytes, image_metrics_scratch_bytes(N, H, W));
    return -5;
  }
  return launch_image_metrics(sr, hr, N, H, W, reinterpret_cast<double*>(scratch), psnr_out, ssim_out, S(stream));
}

}  // extern "C"

// ---- per-operator convolution (SURVEY 8b) -----------------------------------------------------------------------
extern "C" size_t srg_conv2d_packed_weight_bytes(int cout, int cin, int ksize) { return conv2d_packed_elems(cout, cin, ksize) * 2; }
extern "C" int srg_conv2d_pack_weights(const float* w_oihw, int cout, int cin, int ksize, int for_dgrad, void* packed, void* stream) {
  return launch_conv2d_pack(w_oihw, cout, cin, ksize, for_dgrad, packed, S(stream));
}
extern "C" int srg_conv2d_fprop(const void* x, int N, int H, int W, int cin, const void* w_packed, int cout, int ksize,
                                const float* bias, int act, float slope, const void* residual, void* out, void* stream) {
  return launch_conv2d(x, N, H, W, cin, w_packed, cout, ksize, bias, act, slope, residual, nullptr, out, S(stream));
}
extern "C" int srg_conv2d_dgrad(const void* dy, int N, int H, int W, int cout, const void* w_packed_dgrad, int cin, int ksize,
                                const void* relu_mask_src, const void* residual, void* dx, void* stream) {
  if (relu_mask_src != nullptr && residual != nullptr) { set_error("srg_conv2d_dgrad: mask and residual are exclusive"); return -74; }
  return launch_conv2d(dy, N, H, W, cout, w_packed_dgrad, cin, ksize, nullptr, ACT_NONE, 0.f, residual, relu_mask_src, dx, S(stream));
}
extern "C" size_t srg_conv2d_wgrad_workspace_bytes(int N, int H, int W, int cin, int cout) {
  return conv2d_wgrad_workspace_bytes(N, H, W, cin, cout);
}
extern "C" int srg_conv2d_wgrad(const void* x, const void* dy, int N, int H, int W, int cin, int cout, void* workspace,
                                size_t workspace_bytes, float* dw_oihw, float* dbias, void* stream) {
  return launch_conv2d_wgrad(x, dy, N, H, W, cin, cout, workspace, workspace_bytes, dw_oihw, dbias, S(stream));
}

// ---- VGG19 perceptual loss helpers (src/models.py:123-151, src/utils.py:154-166) ------------------------------------
extern "C" int srg_unfold3x3_rgb(const float* x_nchw, int N, int H, int W, void* out, void* stream) {
  return launch_unfold3(x_nchw, N, H, W, out, S(stream));
}
extern "C" int srg_fold3x3_rgb(const void* d_unfolded, int N, int H, int W, float scale, float* dx_nchw, void* stream) {
  return launch_fold3(d_unfolded, N, H, W, scale, dx_nchw, S(stream));
}
extern "C" int srg_maxpool2x2_forward(const void* x, int N, int H, int W, int C, void* out, void* stream) {
  return launch_maxpool2_forward(x, N, H, W, C, out, S(stream));
}
extern "C" int srg_maxpool2x2_backward(const void* x, const void* dy, const void* add, int N, int H, int W, int C, void* dx,
                                       void* stream) {
  return launch_maxpool2_backward(x, dy, add, N, H, W, C, dx, S(stream));
}
extern "C" size_t srg_l1_bf16_scratch_bytes(void) { return l1_feat_scratch_bytes(); }
extern "C" int srg_l1_bf16(const void* a, const void* b, int64_t n, float weight, int accumulate, float grad_scale, int relu_mask,
                           void* grad_a, void* scratch, size_t scratch_bytes, float* out1, void* stream) {
  if (scratch_bytes < l1_feat_scratch_bytes()) { set_error("srg_l1_bf16: scratch too small"); return -83; }
  return launch_l1_feat(a, b, n, weight, accumulate, grad_scale, relu_mask, grad_a, scratch, out1, S(stream));
}

// ---- image-size transforms either side of the path (src/transformers.py:73-82) -------------------------------------
extern "C" int srg_resize_plan_ksize(int in_size, int out_size, int filter) { return resize_plan_ksize(in_size, out_size, filter); }
extern "C" int srg_resize_plan(int in_size, int out_size, int filter, int32_t* bounds_host, int32_t* coeffs_host) {
  return resize_plan(in_size, out_size, filter, bounds_host, coeffs_host);
}
extern "C" int srg_resize_u8(const uint8_t* src_nhwc, int N, int H, int W, int out_h, int out_w, const int32_t* bounds_w,
                             const int32_t* coeffs_w, int ksize_w, const int32_t* bounds_h, const int32_t* coeffs_h, int ksize_h,
                             uint8_t* tmp, uint8_t* out_u8_nhwc, float* out_f32_nchw, const float* noise_nchw,
                             const float* sigma_per_image, void* stream) {
  return launch_resize_u8(src_nhwc, N, H, W, out_h, out_w, bounds_w, coeffs_w, ksize_w, bounds_h, coeffs_h, ksize_h, tmp,
                          out_u8_nhwc, out_f32_nchw, noise_nchw, sigma_per_image, S(stream));
}
