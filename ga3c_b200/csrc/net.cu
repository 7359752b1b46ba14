// C-ABI host layer: handle, flat arenas, workspace, and the launch sequences of the hot path.
// See include/ga3c_b200.h for the contract and the reference call sites each entry replaces.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ga3c_b200.h"
#include "common.cuh"
#include "kernels.h"
#include "handle.h"
#include "mlp.cuh"
#include "dp_exchange.cuh"

using namespace ga3c;

static thread_local std::string g_err;

struct ga3c_net : Handle<ga3c_config> {
  int64_t small_floats = 0;        // prefix holding every tensor except dense1/w (grads zeroed per step)
  // the arena slab holds [params | grads | ms | mom | bf16 shadow of dense1/w | LL receive buffers | comm flags]: a single CUDA
  // IPC handle exposes everything a data-parallel peer needs (ga3c_dp_*)
  uint16_t* w1_shadow = nullptr;   // bf16 [3872,256]
  // data parallel over peer memory (single node, <= 8 ranks)
  int dp_rank = 0, dp_world = 1;
  uint8_t* dp_peer[DP_MAX_WORLD] = {};   // slab base of every rank as mapped in this process (own slab at dp_rank)
  bool dp_ipc[DP_MAX_WORLD] = {};        // mapped with cudaIpcOpenMemHandle (to be closed on detach)
  uint64_t dp_step = 0;
  int64_t xbuf_off = 0, comm_off = 0;    // byte offsets in the slab: LL receive buffers [2][8][small prefix * 8 B], comm block
  cudaStream_t dp_stream = nullptr;      // the dense1/w exchange runs here, next to the conv kernels
  bool dp_big_pending = false;           // an exchange was launched since the ranks attached: dense_fwd waits for its flags (dp_gate)
  cudaEvent_t dp_grad_ready = nullptr;   // recorded behind dense_bwd: the side stream waits for it
  // workspace
  uint16_t *n2 = nullptr, *dd1 = nullptr, *dn1 = nullptr;
  // training-only activations, stored in the UMMA operand layouts the conv backward consumes (common.cuh); their zero borders /
  // slack rows are never written, so they are cleared once, at allocation
  uint8_t *n1 = nullptr, *dn2 = nullptr, *xblk = nullptr;
  float* d1 = nullptr;
  float* d1_part = nullptr;        // [splits][B,256] raw split-K partials of dense1 (dense_tc.cu)
  // gradient partials: one slab per CTA of the heads / conv backward kernels, laid out like the small-tensor prefix
  // of the gradient arena followed by the 4 loss sums; summed by grad_reduce at the end of ga3c_fb_tail
  float* gpart = nullptr;
  int64_t gp_stride = 0;
  int gp_heads_grid = 0;           // slabs the heads kernel of the current step wrote
  float* loss_out = nullptr;       // caller's loss buffer of the current step (may be null)
  bool keep_dn1 = false;           // tests: also store dn1 (which otherwise never leaves the SM) to the workspace
  std::mutex mtx;                  // ga3c_lock / ga3c_unlock
  unsigned long long* evt = nullptr;       // pipeline event log of CTA 0 (ga3c_evt_*), device memory
  unsigned long long* trace = nullptr;     // [K_COUNT][TRACE_SLOTS] globaltimer stamps (ga3c_trace_*), device memory
  // input geometry: 84x84x4 runs the specialised trunk (conv_fwd.cu, conv_bwd_fused.cu), every other one the generic trunk
  // (conv_gen.cu) on the row-major buffers in gen (gen.n2 / gen.dn2 alias n2 / dn2 above)
  GenGeom geo{};
  bool generic = false;
  GenBufs gen{};
  int conv_slabs = 0;              // gradient-partial slabs the conv backward of the current step wrote

  int64_t off(int i) const { return params[i].offset; }
  int64_t w1_count() const { return (int64_t)geo.kdim * FC; }
};


static const char* const kKernelNames[K_COUNT] = {"conv_fwd", "dense_fwd", "heads", "dense_wgrad", "dense_bwd",
                                                  "conv_bwd", "conv11_wgrad", "rmsprop", "grad_reduce",
                                                  "mlp_fused", "mlp_wgrad", "mlp_reduce", "dp_big", "mlp_tc",
                                                  "histograms", "gen_wprep", "gen_im2col11", "gen_conv11",
                                                  "gen_im2col12", "gen_conv12", "gen_conv12_dgrad", "gen_col2im",
                                                  "gen_conv12_wgrad", "gen_conv11_wgrad"};

enum { P_C11W = 0, P_C11B, P_C12W, P_C12B, P_D1W, P_D1B, P_VW, P_VB, P_PW, P_PB, P_COUNT };

static int alloc_workspace(ga3c_net* n, int max_batch);
static int trace_attach_all(unsigned long long* buf);
static int dp_attach_finish(ga3c_net* n, int32_t rank, int32_t world);

namespace ga3c {
int set_error(const std::string& m) { g_err = m; return -1; }     // for the other host files (mlp_net.cu)
const char* kernel_name(int kid) { return (kid >= 0 && kid < K_COUNT) ? kKernelNames[kid] : nullptr; }
}
extern "C" const char* ga3c_last_error(void) { return g_err.c_str(); }
extern "C" int ga3c_abi_version(void) { return 10; }

extern "C" int ga3c_create(const ga3c_config* cfg, ga3c_net** out) {
  if (!cfg || !out) return set_error("ga3c_create: null argument");
  *out = nullptr;
  if (cfg->num_actions < 1 || cfg->num_actions > MAX_ACTIONS) return set_error("ga3c_create: num_actions must be 1..18");
  if (cfg->max_batch < 1) return set_error("ga3c_create: max_batch must be >= 1");
  const int ih = cfg->image_height ? cfg->image_height : IMG, iw = cfg->image_width ? cfg->image_width : IMG;
  const int ic = cfg->stacked_frames ? cfg->stacked_frames : IMG_C;
  if (ih < 1 || ih > 256) return set_error("ga3c_create: image_height (Config.IMAGE_HEIGHT) must be 1..256");
  if (iw < 1 || iw > 256) return set_error("ga3c_create: image_width (Config.IMAGE_WIDTH) must be 1..256");
  if (ic < 1 || ic > 8) return set_error("ga3c_create: stacked_frames (Config.STACKED_FRAMES) must be 1..8");
  int num_sms = 0;
  if (int r = open_device(cfg->device, "ga3c_create", &num_sms)) return r;
  ga3c_net* n = new ga3c_net();
  n->cfg = *cfg;
  n->cfg.image_height = ih; n->cfg.image_width = iw; n->cfg.stacked_frames = ic;
  n->geo = gen_geom(ih, iw, ic);
  n->generic = !(ih == IMG && iw == IMG && ic == IMG_C);
  n->num_sms = num_sms;
  const int A = cfg->num_actions;
  // TF creation order (NetworkVP.py:284-285 would list them so); offsets pack the small tensors first
  struct { const char* name; int nd; int64_t s[4]; } spec[P_COUNT] = {
      {"conv11/w:0", 4, {8, 8, ic, 16}}, {"conv11/b:0", 1, {16, 0, 0, 0}},
      {"conv12/w:0", 4, {4, 4, 16, 32}}, {"conv12/b:0", 1, {32, 0, 0, 0}},
      {"dense1/w:0", 2, {n->geo.kdim, FC, 0, 0}}, {"dense1/b:0", 1, {FC, 0, 0, 0}},
      {"logits_v/w:0", 2, {FC, 1, 0, 0}}, {"logits_v/b:0", 1, {1, 0, 0, 0}},
      {"logits_p/w:0", 2, {FC, A, 0, 0}}, {"logits_p/b:0", 1, {A, 0, 0, 0}}};
  n->params.resize(P_COUNT);
  for (int i = 0; i < P_COUNT; ++i) {
    Param& d = n->params[i];
    d.name = spec[i].name;
    d.ndim = spec[i].nd;
    d.live = 1;
    d.count = 1;
    for (int k = 0; k < 4; ++k) { d.shape[k] = spec[i].s[k]; if (k < d.ndim) d.count *= d.shape[k]; }
  }
  int64_t cur = 0;
  const int order[P_COUNT] = {P_C11W, P_C11B, P_C12W, P_C12B, P_D1B, P_VW, P_VB, P_PW, P_PB, P_D1W};
  for (int k = 0; k < P_COUNT; ++k) {
    if (order[k] == P_D1W) n->small_floats = cur;
    n->params[order[k]].offset = cur;
    cur = align_up(cur + n->params[order[k]].count);
  }
  n->arena_floats = cur;
  const int skip[4] = {P_VW, P_VB, P_PW, P_PB};          // cost_p does not reach logits_v (stop_gradient), cost_v not logits_p
  for (int i = 0; i < 4; ++i) { n->skip_lo[i] = n->off(skip[i]); n->skip_hi[i] = n->off(skip[i]) + n->params[skip[i]].count; }
  // opt.minimize(..., global_step=self.global_step) once per optimizer (NetworkVP_discrate.py:130; DUAL_RMSPROP: both minimize
  // calls, :125-126); clipped, apply_gradients is called without global_step (:107-117, :121) and the step counter stays put
  n->step_advance = cfg->use_grad_clip ? 0 : cfg->dual_rmsprop ? 2 : 1;

  const size_t ab = (size_t)n->arena_floats * sizeof(float);
  const size_t shadow_bytes = (size_t)n->w1_count() * 2;
  n->xbuf_off = (int64_t)(4 * ab + shadow_bytes);
  n->comm_off = n->xbuf_off + 2 * (int64_t)DP_MAX_WORLD * n->small_floats * 8;
  if (int r = alloc_arenas(n, (size_t)n->comm_off + DP_COMM_BYTES - 4 * ab)) { ga3c_destroy(n); return r; }
  n->w1_shadow = reinterpret_cast<uint16_t*>(n->slab + 4 * ab);
  n->gp_stride = n->small_floats + 64;
  cudaError_t e = cudaMalloc((void**)&n->gpart, (size_t)2 * n->num_sms * n->gp_stride * sizeof(float));
  if (e != cudaSuccess) { ga3c_destroy(n); return fail_cuda("cudaMalloc", e); }
  cudaMemset(n->gpart, 0, (size_t)2 * n->num_sms * n->gp_stride * sizeof(float));
  if (int r = alloc_workspace(n, cfg->max_batch)) { ga3c_destroy(n); return r; }
  int r;
  if ((r = configure_conv_fwd()) || (r = configure_conv_bwd_fused()) || (r = configure_dense_tc()) || (r = configure_conv_gen())) {
    ga3c_destroy(n);
    return fail_cuda("cudaFuncSetAttribute", (cudaError_t)r);
  }
  e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { ga3c_destroy(n); return fail_cuda("ga3c_create sync", e); }
  *out = n;
  return 0;
}

static void free_workspace(ga3c_net* n) {
  cudaFree(n->n1); cudaFree(n->n2); cudaFree(n->d1); cudaFree(n->dd1); cudaFree(n->dn2); cudaFree(n->dn1); cudaFree(n->xblk);
  cudaFree(n->d1_part);
  cudaFree(n->gen.x1); cudaFree(n->gen.n1); cudaFree(n->gen.x2); cudaFree(n->gen.dx2); cudaFree(n->gen.dn1); cudaFree(n->gen.w11t);
  n->n2 = n->dd1 = n->dn1 = nullptr; n->n1 = n->dn2 = n->xblk = nullptr; n->d1 = n->d1_part = nullptr;
  n->gen = GenBufs{};
}

// the generic trunk's buffers (DESIGN.md, "The generic conv trunk": X1 and dx2 dominate)
static int alloc_workspace_generic(ga3c_net* n, size_t mb) {
  const GenGeom& g = n->geo;
  const size_t p1 = mb * g.h1 * g.w1, p2 = mb * g.h2 * g.w2;
  GenBufs& b = n->gen;
  CK(cudaMalloc((void**)&b.x1, p1 * g.ld1 * 2)); CK(cudaMalloc((void**)&b.n1, p1 * 16 * 2));
  CK(cudaMalloc((void**)&b.x2, p2 * GEN_LD2 * 2)); CK(cudaMalloc((void**)&b.dx2, p2 * 256 * 4));
  CK(cudaMalloc((void**)&b.dn1, p1 * 16 * 2));
  CK(cudaMalloc((void**)&b.w11t, ((size_t)16 * g.k1 + 2 * 32 * 256) * 2));
  b.w12t = b.w11t + (size_t)16 * g.k1; b.w12 = b.w12t + 32 * 256;
  CK(cudaMalloc((void**)&n->n2, mb * g.kdim * 2)); CK(cudaMalloc((void**)&n->dn2, mb * g.kdim * 2));
  b.n2 = n->n2; b.dn2 = reinterpret_cast<uint16_t*>(n->dn2);
  return 0;
}

static int alloc_workspace(ga3c_net* n, int max_batch) {
  const size_t mb = (size_t)max_batch;
  if (n->generic) {
    if (int r = alloc_workspace_generic(n, mb)) return r;
  } else {
    CK(cudaMalloc((void**)&n->n1, mb * B2_BYTES)); CK(cudaMalloc((void**)&n->n2, mb * FLAT * 2));
    CK(cudaMalloc((void**)&n->dn2, mb * G_BYTES)); CK(cudaMalloc((void**)&n->dn1, mb * N1_POS * C1_OUT * 2));
    CK(cudaMalloc((void**)&n->xblk, mb * XB_FRAME_BYTES));
    CK(cudaMemset(n->n1, 0, mb * B2_BYTES)); CK(cudaMemset(n->dn2, 0, mb * G_BYTES)); CK(cudaMemset(n->xblk, 0, mb * XB_FRAME_BYTES));
  }
  CK(cudaMalloc((void**)&n->d1, mb * FC * 4)); CK(cudaMalloc((void**)&n->dd1, mb * FC * 2));
  // splits * batch <= max(batch, 64 * num_sms) rows for every batch (dense_fwd_splits)
  const size_t part_rows = mb > (size_t)64 * n->num_sms ? mb : (size_t)64 * n->num_sms;
  CK(cudaMalloc((void**)&n->d1_part, part_rows * FC * 4));
  n->cfg.max_batch = max_batch;
  return 0;
}

extern "C" int ga3c_reserve(ga3c_net* n, int32_t max_batch) {
  if (!n) return set_error("ga3c_reserve: null handle");
  if (max_batch <= n->cfg.max_batch) return 0;
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  free_workspace(n);
  if (int r = alloc_workspace(n, max_batch)) { free_workspace(n); cudaGetLastError(); n->cfg.max_batch = 0; return r; }
  return 0;
}

extern "C" int ga3c_destroy(ga3c_net* n) {
  if (!n) return 0;
  ga3c_dp_detach(n);
  free_arenas(n);
  cudaFree(n->gpart);
  if (n->trace) { trace_attach_all(nullptr); cudaFree(n->trace); }
  free_workspace(n);
  delete n;
  return 0;
}

extern "C" int ga3c_lock(ga3c_net* n) {
  if (!n) return set_error("ga3c_lock: null handle");
  n->mtx.lock();
  return 0;
}
extern "C" int ga3c_unlock(ga3c_net* n) {
  if (!n) return set_error("ga3c_unlock: null handle");
  n->mtx.unlock();
  return 0;
}

extern "C" int ga3c_param_count(const ga3c_net* n) { return n ? (int)n->params.size() : 0; }

extern "C" int ga3c_param_info(const ga3c_net* n, int i, const char** name, int64_t* offset, int32_t* ndim,
                               int64_t shape[4]) {
  return param_info(n, i, name, offset, ndim, shape, nullptr, "ga3c_param_info");
}

extern "C" int64_t ga3c_arena_floats(const ga3c_net* n) { return n ? n->arena_floats : 0; }

extern "C" int ga3c_arena_ptrs(ga3c_net* n, float** p, float** g, float** ms, float** mom) {
  if (!n) return set_error("ga3c_arena_ptrs: null handle");
  if (p) *p = n->w;
  if (g) *g = n->g;
  if (ms) *ms = n->ms;
  if (mom) *mom = n->mom;
  return 0;
}

extern "C" int ga3c_arena_ptr(ga3c_net* n, int which, float** ptr_dev) {
  if (!n || !ptr_dev) return set_error("ga3c_arena_ptr: null argument");
  *ptr_dev = arena_of(n, which);
  if (!*ptr_dev) return set_error("ga3c_arena_ptr: bad arena id");
  return 0;
}

extern "C" int ga3c_arena_upload(ga3c_net* n, int which, const float* host, int64_t nf) {
  if (int r = arena_upload(n, which, host, nf, "ga3c_arena_upload")) return r;
  if (which == 0) {
    CKL(launch_f32_to_bf16(n->w + n->off(P_D1W), n->w1_shadow, n->w1_count(), 0));
    n->log.launches++;
    CK(cudaDeviceSynchronize());
  }
  return 0;
}

extern "C" int ga3c_arena_download(ga3c_net* n, int which, float* host, int64_t nf) {
  if (int r = arena_download(n, which, host, nf, "ga3c_arena_download")) return r;
  if (n->dp_world > 1 && (which == 0 || which == 2 || which == 3)) {
    // peer-memory exchange: the fp32 master copy and the RMSProp slots of a dense1/w slice live on its owner (only the bf16
    // shadow travels).  A peer's slice is stable here: it changes only inside a step this rank takes part in.
    const int64_t n4 = n->w1_count() / 4, per = (n4 + n->dp_world - 1) / n->dp_world;
    for (int q = 0; q < n->dp_world; ++q) {
      if (q == n->dp_rank) continue;
      const int64_t lo = per * q, hi = lo + per < n4 ? lo + per : n4;
      if (hi <= lo) continue;
      const int64_t off = n->off(P_D1W) + lo * 4;
      CK(cudaMemcpy(host + off, n->dp_peer[q] + (size_t)which * nf * 4 + (size_t)off * 4, (size_t)(hi - lo) * 16,
                    cudaMemcpyDeviceToHost));
    }
  }
  return 0;
}

extern "C" int64_t ga3c_global_step(const ga3c_net* n) { return n ? n->global_step : -1; }
extern "C" int ga3c_set_global_step(ga3c_net* n, int64_t s) { if (!n) return -1; n->global_step = s; return 0; }

static HeadsArgs heads_args(ga3c_net* n, int batch, int splits, float beta = 0.f, int part = 0) {
  HeadsArgs h{};
  h.d1 = n->d1; h.d1_part = n->d1_part; h.n_split = splits; h.b1 = n->w + n->off(P_D1B);
  h.wp = n->w + n->off(P_PW); h.bp = n->w + n->off(P_PB);
  h.wv = n->w + n->off(P_VW); h.bv = n->w + n->off(P_VB);
  h.batch = batch; h.num_actions = n->cfg.num_actions;
  h.la = LossArgs{beta, n->cfg.log_epsilon, n->cfg.min_policy, n->cfg.use_log_softmax != 0, part};
  h.preload = batch >= n->num_sms;
  return h;
}

// data parallel: the bf16 shadow of dense1/w is complete when dense_fwd's TMA producer has seen every rank's "slice landed
// everywhere" flag of the last exchanged step in this rank's comm block (DpGate, dense_tc.cu): no stream operation between
// conv_fwd and dense_fwd, so the launch chain stays programmatic.  (dp_big_pending is cleared by ga3c_dp_detach, so it implies
// dp_world > 1.)
static DpGate dp_gate(const ga3c_net* n) {
  DpGate g{};
  if (n->dp_big_pending) {
    uint8_t* comm = n->dp_peer[n->dp_rank] + n->comm_off;
    g.flags = comm + DPC_BIGDONE; g.err = comm + DPC_ERR; g.step = n->dp_step; g.world = n->dp_world;
  }
  return g;
}

// the generic trunk's forward: n1 and n2 (and X1, X2 for the backward) from the frames
static int gen_forward(ga3c_net* n, const void* x, bool x_u8, int batch, cudaStream_t st) {
  const GenGeom& g = n->geo;
  const float* w = n->w;
  LAUNCH(n, K_GEN_WPREP, st, launch_gen_wprep(g, n->gen, w + n->off(P_C11W), w + n->off(P_C12W), st));
  LAUNCH(n, K_GEN_IM2COL1, st, launch_gen_im2col1(g, n->gen, x, x_u8, batch, st));
  LAUNCH(n, K_GEN_CONV11, st, launch_gen_conv11(g, n->gen, w + n->off(P_C11B), batch, st));
  LAUNCH(n, K_GEN_IM2COL2, st, launch_gen_im2col2(g, n->gen, batch, st));
  LAUNCH(n, K_GEN_CONV12, st, launch_gen_conv12(g, n->gen, w + n->off(P_C12B), batch, st));
  return 0;
}

static int predict_impl(ga3c_net* n, const void* x, bool x_u8, int32_t batch, float* p_out, float* v_out, void* stream) {
  if (int r = check_batch(n, batch, "ga3c_predict")) return r;
  if (!x || !p_out || !v_out) return set_error("ga3c_predict: null buffer");
  CK(cudaSetDevice(n->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const float* w = n->w;
  if (n->generic) {
    if (int r = gen_forward(n, x, x_u8, batch, st)) return r;
  } else {
    LAUNCH(n, K_CONV_FWD, st, launch_conv_fwd(x, x_u8, w + n->off(P_C11W), w + n->off(P_C11B), w + n->off(P_C12W),
                                              w + n->off(P_C12B), nullptr, nullptr, n->n2, batch, n->num_sms, st));
  }
  const DpGate gate = dp_gate(n);
  const int splits = dense_fwd_splits(batch, n->num_sms, n->geo.kdim);
  HeadsArgs h = heads_args(n, batch, splits);
  h.p_out = p_out; h.v_out = v_out; h.train = 0;
  LAUNCH(n, K_DENSE_FWD, st, launch_dense_fwd_tc(n->n2, n->w1_shadow, n->d1_part, batch, n->geo.kdim, splits, st, &gate));
  LAUNCH(n, K_HEADS, st, launch_heads(h, n->num_sms, st));
  n->last_batch = batch;
  return 0;
}

extern "C" int ga3c_predict(ga3c_net* n, const float* x, int32_t batch, float* p_out, float* v_out, void* stream) {
  return predict_impl(n, x, false, batch, p_out, v_out, stream);
}
extern "C" int ga3c_predict_u8(ga3c_net* n, const uint8_t* x, int32_t batch, float* p_out, float* v_out, void* stream) {
  return predict_impl(n, x, true, batch, p_out, v_out, stream);
}

// forward, fused loss forward/backward, and the dense1 weight gradient: on return (in stream order) the
// gradients of dense1/w, dense1/b, logits_v/*, logits_p/* are final, so their allreduce can start while
// ga3c_fb_tail computes the conv gradients.
static int fb_head_impl(ga3c_net* n, const void* x, bool x_u8, const float* yr, const float* a, int32_t batch, float beta,
                        float* loss, void* stream, bool with_wgrad, int part = 0, bool skip_forward = false) {
  if (int r = check_batch(n, batch, "ga3c_fb_head")) return r;
  if (!x || !yr || !a) return set_error("ga3c_fb_head: null buffer");
  CK(cudaSetDevice(n->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const float* w = n->w;
  float* g = n->g;
  float* gp = n->gpart;       // small-tensor gradients: per-CTA partial slabs, summed at the end of ga3c_fb_tail
  const int splits = dense_fwd_splits(batch, n->num_sms, n->geo.kdim);
  if (!skip_forward) {        // the second DUAL_RMSPROP pass reuses n1 / n2 / the dense1 partials of the first
    if (n->generic) {
      if (int r = gen_forward(n, x, x_u8, batch, st)) return r;
    } else {
      LAUNCH(n, K_CONV_FWD, st, launch_conv_fwd(x, x_u8, w + n->off(P_C11W), w + n->off(P_C11B), w + n->off(P_C12W),
                                                w + n->off(P_C12B), n->n1, n->xblk, n->n2, batch, n->num_sms, st));
    }
    const DpGate gate = dp_gate(n);
    LAUNCH(n, K_DENSE_FWD, st, launch_dense_fwd_tc(n->n2, n->w1_shadow, n->d1_part, batch, n->geo.kdim, splits, st, &gate));
  }
  HeadsArgs h = heads_args(n, batch, splits, beta, part);
  h.yr = yr; h.a = a; h.train = 1; h.dd1 = n->dd1;
  h.g_wp = gp + n->off(P_PW); h.g_bp = gp + n->off(P_PB); h.g_wv = gp + n->off(P_VW); h.g_bv = gp + n->off(P_VB);
  h.g_b1 = gp + n->off(P_D1B); h.loss = gp + n->small_floats; h.gp_stride = n->gp_stride;
  n->gp_heads_grid = heads_grid(batch, n->num_sms);
  n->loss_out = loss;
  LAUNCH(n, K_HEADS, st, launch_heads(h, n->num_sms, st));
  (void)g;
  if (with_wgrad) LAUNCH(n, K_DENSE_WGRAD, st, launch_dense_wgrad_tc(n->n2, n->dd1, n->g + n->off(P_D1W), batch, n->geo.kdim, st));
  n->last_batch = batch;
  return 0;
}

extern "C" int ga3c_fb_head(ga3c_net* n, const float* x, const float* yr, const float* a, int32_t batch, float beta,
                            float* loss, void* stream) {
  return fb_head_impl(n, x, false, yr, a, batch, beta, loss, stream, true);
}

// sum of the per-CTA slabs: conv tensors (the first four of the arena) over the conv grids, head tensors and the loss
// sums over the heads grid
static GradReduceArgs reduce_args(ga3c_net* n, int batch, float* g_dst = nullptr) {
  GradReduceArgs r{};
  r.part = n->gpart; r.stride = n->gp_stride; r.out = g_dst ? g_dst : n->g; r.out_tail = n->loss_out;
  r.out_floats = (int)n->small_floats; r.n_floats = (int)n->small_floats + 4;
  for (int s = 0; s < GR_MAX_SEG; ++s) { r.seg_end[s] = r.n_floats; r.seg_count[s] = n->gp_heads_grid; }
  r.seg_end[0] = (int)n->off(P_D1B); r.seg_count[0] = n->generic ? n->conv_slabs : conv_bwd_grid(batch, n->num_sms);
  return r;
}

// the dense1/w exchange on the side stream, behind everything enqueued on `st` so far (dense1/w's gradient is final there)
static int enqueue_dp_big(ga3c_net* n, const DpBigArgs& b, cudaStream_t st) {
  CK(cudaEventRecord(n->dp_grad_ready, st));
  CK(cudaStreamWaitEvent(n->dp_stream, n->dp_grad_ready, 0));
  CKL(launch_dp_big_side(b, n->num_sms, n->dp_stream));
  n->log.launches++;
  n->dp_big_pending = true;
  return 0;
}

// dense1 data gradient and the two conv backward kernels; with `reduce` the slabs are summed into the gradient arena
// (conv11/*, conv12/*, dense1/b, heads, loss sums), otherwise the caller does it (fused with RMSProp).  With `dp` the dense1/w
// exchange of the data-parallel step is launched on the side stream as soon as dense1/w's gradient is final.
static int fb_tail_impl(ga3c_net* n, const void* x, bool x_u8, int32_t batch, void* stream, bool with_wgrad, bool reduce,
                        const DpBigArgs* dp = nullptr, float* g_dst = nullptr) {
  if (int r = check_batch(n, batch, "ga3c_fb_tail")) return r;
  if (!x) return set_error("ga3c_fb_tail: null buffer");
  if (batch != n->last_batch) return set_error("ga3c_fb_tail: batch differs from the preceding ga3c_fb_head");
  CK(cudaSetDevice(n->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const float* w = n->w;
  float* gp = n->gpart;
  float* const g_w1 = (g_dst ? g_dst : n->g) + n->off(P_D1W);
  if (n->generic) {
    const GenGeom& ge = n->geo;
    if (with_wgrad)
      LAUNCH(n, K_DENSE_DGRAD, st, launch_dense_bwd_rows_tc(n->dd1, n->w1_shadow, n->n2, n->gen.dn2, g_w1, batch, ge.kdim, st));
    else
      LAUNCH(n, K_DENSE_DGRAD, st, launch_dense_dgrad_rows_tc(n->dd1, n->w1_shadow, n->n2, n->gen.dn2, batch, ge.kdim, st));
    n->conv_slabs = gen_wgrad_slabs(ge, batch, n->num_sms);
    LAUNCH(n, K_GEN_CONV12_DGRAD, st, launch_gen_conv12_dgrad(ge, n->gen, batch, st));
    LAUNCH(n, K_GEN_COL2IM, st, launch_gen_col2im(ge, n->gen, batch, st));
    LAUNCH(n, K_GEN_CONV12_WGRAD, st, launch_gen_conv12_wgrad(ge, n->gen, gp + n->off(P_C12W), gp + n->off(P_C12B), n->gp_stride,
                                                              n->conv_slabs, batch, st));
    LAUNCH(n, K_GEN_CONV11_WGRAD, st, launch_gen_conv11_wgrad(ge, n->gen, gp + n->off(P_C11W), gp + n->off(P_C11B), n->gp_stride,
                                                              n->conv_slabs, batch, st));
  } else {
    if (with_wgrad)   // dgrad + wgrad tiles of dense1 in one grid
      LAUNCH(n, K_DENSE_DGRAD, st, launch_dense_bwd_tc(n->dd1, n->w1_shadow, n->n2, n->dn2, g_w1, batch, st));
    else
      LAUNCH(n, K_DENSE_DGRAD, st, launch_dense_dgrad_tc(n->dd1, n->w1_shadow, n->n2, n->dn2, batch, st));
    if (dp != nullptr)
      if (int r = enqueue_dp_big(n, *dp, st)) return r;
    LAUNCH(n, K_CONV12_BWD, st, launch_conv_bwd(n->xblk, n->n1, n->dn2, w + n->off(P_C12W), n->keep_dn1 ? n->dn1 : nullptr,
                                                gp + n->off(P_C11W), gp + n->off(P_C11B), gp + n->off(P_C12W),
                                                gp + n->off(P_C12B), n->gp_stride, batch, n->num_sms, x_u8, st));
  }
  if (reduce) LAUNCH(n, K_GRAD_REDUCE, st, launch_grad_reduce(reduce_args(n, batch, g_dst), st));
  return 0;
}

extern "C" int ga3c_fb_tail(ga3c_net* n, const float* x, int32_t batch, void* stream) {
  return fb_tail_impl(n, x, false, batch, stream, false, true);
}

static int forward_backward_impl(ga3c_net* n, const void* x, bool x_u8, const float* yr, const float* a, int32_t batch,
                                 float beta, float* loss, void* stream) {
  if (int r = fb_head_impl(n, x, x_u8, yr, a, batch, beta, loss, stream, false)) return r;
  return fb_tail_impl(n, x, x_u8, batch, stream, true, true);
}
extern "C" int ga3c_forward_backward(ga3c_net* n, const float* x, const float* yr, const float* a, int32_t batch,
                                     float beta, float* loss, void* stream) {
  return forward_backward_impl(n, x, false, yr, a, batch, beta, loss, stream);
}
extern "C" int ga3c_forward_backward_u8(ga3c_net* n, const uint8_t* x, const float* yr, const float* a, int32_t batch,
                                        float beta, float* loss, void* stream) {
  return forward_backward_impl(n, x, true, yr, a, batch, beta, loss, stream);
}
extern "C" int ga3c_fb_head_u8(ga3c_net* n, const uint8_t* x, const float* yr, const float* a, int32_t batch, float beta,
                               float* loss, void* stream) {
  return fb_head_impl(n, x, true, yr, a, batch, beta, loss, stream, true);
}
extern "C" int ga3c_fb_tail_u8(ga3c_net* n, const uint8_t* x, int32_t batch, void* stream) {
  return fb_tail_impl(n, x, true, batch, stream, false, true);
}

static RmsPropArgs rmsprop_args(ga3c_net* n, float lr) {
  RmsPropArgs a = rmsprop_base(n, lr, n->arena_floats);
  a.w1_shadow = n->w1_shadow; a.w1_offset = n->off(P_D1W); a.w1_count = n->w1_count();
  return a;
}

static int apply_rmsprop_impl(ga3c_net* n, float lr, void* stream) {
  if (!n) return set_error("ga3c_apply_rmsprop: null handle");
  CK(cudaSetDevice(n->cfg.device));
  if (n->cfg.dual_rmsprop) return set_error("ga3c_apply_rmsprop: with DUAL_RMSPROP use ga3c_train_step (two backward passes)");
  // clip_by_average_norm needs the whole (reduced) gradient of a variable: local arena only (single GPU, or after the
  // host's NCCL allreduce in dp_mode 'nccl')
  if (n->cfg.use_grad_clip && n->dp_world > 1)
    return set_error("ga3c_apply_rmsprop: USE_GRAD_CLIP is not available with the peer-memory exchange");
  // the peer-memory exchange is part of the train step (its dense1/w half starts behind dense_bwd, on a side stream)
  if (n->dp_world > 1) return set_error("ga3c_apply_rmsprop: not available on a peer-memory data-parallel handle; use ga3c_train_step");
  return launch_optimizer(n, rmsprop_args(n, lr), (cudaStream_t)stream);
}

extern "C" int ga3c_apply_rmsprop(ga3c_net* n, float lr, void* stream) { return apply_rmsprop_impl(n, lr, stream); }

// ---- data parallel over CUDA IPC peer memory ---------------------------------------------------------
extern "C" int ga3c_dp_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

extern "C" int ga3c_dp_export(ga3c_net* n, void* handle_out) {
  if (!n || !handle_out) return set_error("ga3c_dp_export: null argument");
  CK(cudaSetDevice(n->cfg.device));
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, n->slab));
  memcpy(handle_out, &h, sizeof(h));
  return 0;
}

extern "C" int ga3c_dp_detach(ga3c_net* n) {
  if (!n) return 0;
  if (n->dp_stream) {
    cudaStreamSynchronize(n->dp_stream);
    cudaStreamDestroy(n->dp_stream);
    cudaEventDestroy(n->dp_grad_ready);
    n->dp_stream = nullptr; n->dp_big_pending = false;
  }
  for (int r = 0; r < DP_MAX_WORLD; ++r)
    if (n->dp_peer[r] && n->dp_ipc[r]) cudaIpcCloseMemHandle(n->dp_peer[r]);
  for (int r = 0; r < DP_MAX_WORLD; ++r) { n->dp_peer[r] = nullptr; n->dp_ipc[r] = false; }
  n->dp_world = 1; n->dp_rank = 0;
  return 0;
}

extern "C" int ga3c_dp_attach(ga3c_net* n, int32_t rank, int32_t world, const void* handles) {
  if (!n || !handles) return set_error("ga3c_dp_attach: null argument");
  if (n->generic) return set_error("ga3c_dp_attach: the peer-memory exchange needs the 84x84x4 geometry (use dp_mode 'nccl')");
  if (world < 1 || world > DP_MAX_WORLD || rank < 0 || rank >= world)
    return set_error("ga3c_dp_attach: world must be 1.." + std::to_string(DP_MAX_WORLD) + " and 0 <= rank < world");
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  ga3c_dp_detach(n);
  const cudaIpcMemHandle_t* hs = static_cast<const cudaIpcMemHandle_t*>(handles);
  for (int r = 0; r < world; ++r) {
    if (r == rank) { n->dp_peer[r] = n->slab; continue; }
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, hs[r], cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      ga3c_dp_detach(n);
      return fail_cuda("cudaIpcOpenMemHandle (peer-to-peer access between the ranks' GPUs is required)", e);
    }
    n->dp_peer[r] = static_cast<uint8_t*>(p);
    n->dp_ipc[r] = true;
  }
  return dp_attach_finish(n, rank, world);
}

// ranks that live in ONE process (tests; a host that drives several GPUs from one process): the peers' slabs are ordinary
// device pointers, no IPC handles involved.  peers[r] is rank r's handle (peers[rank] == net).
extern "C" int ga3c_dp_attach_local(ga3c_net* n, int32_t rank, int32_t world, ga3c_net* const* peers) {
  if (!n || !peers) return set_error("ga3c_dp_attach_local: null argument");
  if (n->generic) return set_error("ga3c_dp_attach_local: the peer-memory exchange needs the 84x84x4 geometry (use dp_mode 'nccl')");
  if (world < 1 || world > DP_MAX_WORLD || rank < 0 || rank >= world || peers[rank] != n)
    return set_error("ga3c_dp_attach_local: need 0 <= rank < world <= 8 and peers[rank] == net");
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  ga3c_dp_detach(n);
  for (int r = 0; r < world; ++r) {
    if (!peers[r] || peers[r]->arena_floats != n->arena_floats) { ga3c_dp_detach(n); return set_error("ga3c_dp_attach_local: peers must be handles of the same network"); }
    if (peers[r]->cfg.device != n->cfg.device) {
      int can = 0;
      cudaDeviceCanAccessPeer(&can, n->cfg.device, peers[r]->cfg.device);
      if (!can) { ga3c_dp_detach(n); return set_error("ga3c_dp_attach_local: no peer access between the devices"); }
      cudaError_t e = cudaDeviceEnablePeerAccess(peers[r]->cfg.device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { ga3c_dp_detach(n); return fail_cuda("cudaDeviceEnablePeerAccess", e); }
      cudaGetLastError();
    }
    n->dp_peer[r] = peers[r]->slab;
  }
  return dp_attach_finish(n, rank, world);
}

static int dp_attach_finish(ga3c_net* n, int32_t rank, int32_t world) {
  n->dp_rank = rank; n->dp_world = world; n->dp_step = 0;
  CK(cudaMemset(n->slab + n->xbuf_off, 0, n->slab_bytes - (size_t)n->xbuf_off));
  CKL(configure_dp());
  if (!n->dp_stream) {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    CK(cudaStreamCreateWithPriority(&n->dp_stream, cudaStreamNonBlocking, hi));
    CK(cudaEventCreateWithFlags(&n->dp_grad_ready, cudaEventDisableTiming));
  }
  n->dp_big_pending = false;
  return 0;
}

// 0: every cross-rank wait of the exchange kernels completed; 1: one gave up (a rank died, or the ranks' train calls fell out
// of step) and the weights can no longer be trusted.  Synchronises the device.
extern "C" int ga3c_dp_error(ga3c_net* n, int32_t* error_out) {
  if (!n || !error_out) return set_error("ga3c_dp_error: null argument");
  *error_out = 0;
  if (n->dp_world <= 1) return 0;
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  unsigned int e = 0;
  CK(cudaMemcpy(&e, n->slab + n->comm_off + DPC_ERR, 4, cudaMemcpyDeviceToHost));
  *error_out = (int32_t)e;
  return 0;
}

// Config.DUAL_RMSPROP: one forward, two backward passes (cost_p into g, cost_v into g2) ...
static int dual_forward_backward_impl(ga3c_net* n, const void* x, bool x_u8, const float* yr, const float* a, int32_t batch,
                                      float beta, float* loss, void* stream) {
  if (!n || !n->cfg.dual_rmsprop) return set_error("ga3c_dual_forward_backward: the handle was not created with dual_rmsprop");
  if (int r = fb_head_impl(n, x, x_u8, yr, a, batch, beta, loss, stream, false, 1)) return r;
  if (int r = fb_tail_impl(n, x, x_u8, batch, stream, true, true)) return r;
  if (int r = fb_head_impl(n, x, x_u8, yr, a, batch, beta, nullptr, stream, false, 2, true)) return r;
  return fb_tail_impl(n, x, x_u8, batch, stream, true, true, nullptr, n->g2);
}
// ... and one update that subtracts both optimizers' steps, each taken at the weights the call started with
static int dual_apply_impl(ga3c_net* n, float lr, void* stream) {
  if (!n || !n->cfg.dual_rmsprop) return set_error("ga3c_dual_apply: the handle was not created with dual_rmsprop");
  CK(cudaSetDevice(n->cfg.device));
  return launch_optimizer(n, rmsprop_args(n, lr), (cudaStream_t)stream);
}
extern "C" int ga3c_dual_forward_backward(ga3c_net* n, const float* x, const float* yr, const float* a, int32_t batch, float beta,
                                          float* loss, void* stream) {
  return dual_forward_backward_impl(n, x, false, yr, a, batch, beta, loss, stream);
}
extern "C" int ga3c_dual_forward_backward_u8(ga3c_net* n, const uint8_t* x, const float* yr, const float* a, int32_t batch,
                                             float beta, float* loss, void* stream) {
  return dual_forward_backward_impl(n, x, true, yr, a, batch, beta, loss, stream);
}
extern "C" int ga3c_dual_apply(ga3c_net* n, float lr, void* stream) { return dual_apply_impl(n, lr, stream); }

static DpBigArgs dp_big_args(ga3c_net* n, float lr) {
  DpBigArgs b{};
  for (int r = 0; r < n->dp_world; ++r) b.peer[r] = n->dp_peer[r];
  b.rank = n->dp_rank; b.world = n->dp_world; b.step = ++n->dp_step;
  b.arena_bytes = (int64_t)n->arena_floats * 4; b.shadow_off = 4 * b.arena_bytes; b.comm_offset = n->comm_off;
  b.w1_offset = n->off(P_D1W); b.w1_count = n->w1_count();
  b.lr = lr; b.decay = n->cfg.rmsprop_decay; b.momentum = n->cfg.rmsprop_momentum; b.eps = n->cfg.rmsprop_epsilon;
  return b;
}
static RmsPropDpArgs dp_small_args(ga3c_net* n, float lr, int batch, const DpBigArgs& b) {
  RmsPropDpArgs d{};
  d.base = rmsprop_args(n, lr);
  d.base.preload = batch >= n->num_sms;         // the preload rule (elementwise.cu)
  for (int q = 0; q < n->dp_world; ++q) d.peer[q] = n->dp_peer[q];
  d.rank = n->dp_rank; d.world = n->dp_world; d.step = b.step;
  d.arena_bytes = b.arena_bytes; d.comm_offset = n->comm_off;
  d.red = reduce_args(n, batch);
  return d;
}

// A rank of a data-parallel job that has no experiences this round still takes part in the exchange (every rank must enter
// every step: the asynchronous trainer loop of the reference, ThreadTrainer.py:42-62, gives no such guarantee, so the host
// ticks all ranks in lock step and idle ranks contribute a zero gradient).  No forward / backward kernels run.
static int train_step_empty(ga3c_net* n, float lr, float* loss, void* stream) {
  CK(cudaSetDevice(n->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (n->cfg.dual_rmsprop || n->cfg.use_grad_clip)
    return set_error("ga3c_train_step: batch 0 is only defined for the peer-memory data-parallel step");
  n->gp_heads_grid = 0;
  n->loss_out = loss;
  n->last_batch = 0;
  // the exchange publishes "gradient final" itself; dp_small sums zero slabs
  CK(cudaMemsetAsync(n->g + n->off(P_D1W), 0, (size_t)n->w1_count() * 4, st));
  const DpBigArgs b = dp_big_args(n, lr);
  if (int r = enqueue_dp_big(n, b, st)) return r;                  // behind the zeroed gradient
  LAUNCH(n, K_RMSPROP, st, launch_dp_small(dp_small_args(n, lr, 0, b), n->xbuf_off, st));
  n->global_step += n->step_advance;
  return 0;
}

static int train_step_impl(ga3c_net* n, const void* x, bool x_u8, const float* yr, const float* a, int32_t batch, float lr,
                           float beta, float* loss, void* stream) {
  if (n && batch == 0 && n->dp_world > 1) return train_step_empty(n, lr, loss, stream);
  if (n->cfg.dual_rmsprop) {
    if (n->dp_world > 1) return set_error("ga3c_train_step: DUAL_RMSPROP is not available with the peer-memory exchange (dp_mode 'nccl' is)");
    if (int r = dual_forward_backward_impl(n, x, x_u8, yr, a, batch, beta, loss, stream)) return r;
    return dual_apply_impl(n, lr, stream);
  }
  if (int r = fb_head_impl(n, x, x_u8, yr, a, batch, beta, loss, stream, false)) return r;
  if (n->cfg.use_grad_clip) {
    if (int r = fb_tail_impl(n, x, x_u8, batch, stream, true, true)) return r;
    return apply_rmsprop_impl(n, lr, stream);
  }
  if (n->dp_world > 1) {
    // the conv backward keeps every SM; the exchange of dense1/w is launched behind dense_bwd on the side stream and runs next
    // to it (and next to the conv forward of the following step); dp_small follows the conv backward on this stream with the
    // small tensors.  dense_fwd of the next call waits for the exchange's flags (dp_gate).
    // (launched behind an event after dense_bwd, NOT on a flag the conv backward would publish: at batch >= 148 a spinning side
    //  grid that got its blocks resident first kept conv_bwd CTA 0 -- the publisher -- off its SM, and the step timed out)
    const DpBigArgs b = dp_big_args(n, lr);
    if (int r = fb_tail_impl(n, x, x_u8, batch, stream, true, false, &b)) return r;
    LAUNCH(n, K_RMSPROP, (cudaStream_t)stream, launch_dp_small(dp_small_args(n, lr, batch, b), n->xbuf_off, (cudaStream_t)stream));
    n->global_step += n->step_advance;
    return 0;
  }
  // single GPU: the slab reduction rides in the optimizer launch
  if (int r = fb_tail_impl(n, x, x_u8, batch, stream, true, false)) return r;
  RmsPropArgs ra = rmsprop_args(n, lr);
  ra.preload = batch >= n->num_sms;               // the preload rule (elementwise.cu)
  LAUNCH(n, K_RMSPROP, (cudaStream_t)stream, launch_rmsprop_reduce(ra, reduce_args(n, batch), (cudaStream_t)stream));
  n->global_step += n->step_advance;
  return 0;
}
extern "C" int ga3c_train_step(ga3c_net* n, const float* x, const float* yr, const float* a, int32_t batch, float lr,
                               float beta, float* loss, void* stream) {
  return train_step_impl(n, x, false, yr, a, batch, lr, beta, loss, stream);
}
extern "C" int ga3c_train_step_u8(ga3c_net* n, const uint8_t* x, const float* yr, const float* a, int32_t batch, float lr,
                                  float beta, float* loss, void* stream) {
  return train_step_impl(n, x, true, yr, a, batch, lr, beta, loss, stream);
}

extern "C" int ga3c_returns(const double* rewards, const int64_t* seg, int32_t n_segments, const double* terminal,
                            double discount, int32_t flags, double rmin, double rmax, double* out, void* stream) {
  if (n_segments < 0) return set_error("ga3c_returns: negative segment count");
  if (n_segments == 0) return 0;
  if (!rewards || !seg || !terminal || !out) return set_error("ga3c_returns: null buffer");
  CKL(launch_returns(rewards, seg, n_segments, terminal, discount, flags, rmin, rmax, out, (cudaStream_t)stream));
  return 0;
}

extern "C" int ga3c_select_actions(const float* p, const double* u, int32_t batch, int32_t na, int32_t* action,
                                   void* stream) {
  if (batch < 0) return set_error("ga3c_select_actions: negative batch");
  if (batch == 0) return 0;
  if (!p || !u || !action) return set_error("ga3c_select_actions: null buffer");
  if (na < 1 || na > MAX_ACTIONS) return set_error("ga3c_select_actions: num_actions must be 1..18");
  CKL(launch_select_actions(p, u, batch, na, action, (cudaStream_t)stream));
  return 0;
}

extern "C" int ga3c_workspace_ptr(ga3c_net* n, int which, void** ptr, int64_t* bytes) {
  if (!n || !ptr) return set_error("ga3c_workspace_ptr: null argument");
  const int64_t b = n->last_batch;
  if (n->generic) {          // row-major: n1 / dn1 [B,H1,W1,16], n2 / dn2 [B,K] bf16, 7 = X1 [B*H1*W1][64C + 8] bf16
    const GenGeom& g = n->geo;
    const int64_t p1 = b * g.h1 * g.w1;
    switch (which) {
      case 0: *ptr = n->gen.n1; if (bytes) *bytes = p1 * 32; return 0;
      case 1: *ptr = n->n2; if (bytes) *bytes = b * g.kdim * 2; return 0;
      case 4: *ptr = n->dn2; if (bytes) *bytes = b * g.kdim * 2; return 0;
      case 5: *ptr = n->gen.dn1; if (bytes) *bytes = p1 * 32; return 0;
      case 6: *ptr = n->w1_shadow; if (bytes) *bytes = n->w1_count() * 2; return 0;
      case 7: *ptr = n->gen.x1; if (bytes) *bytes = p1 * g.ld1 * 2; return 0;
    }
  }
  switch (which) {
    case 0: *ptr = n->n1; if (bytes) *bytes = b * B2_BYTES; break;
    case 1: *ptr = n->n2; if (bytes) *bytes = b * FLAT * 2; break;
    case 2: *ptr = n->d1; if (bytes) *bytes = b * FC * 4; break;
    case 3: *ptr = n->dd1; if (bytes) *bytes = b * FC * 2; break;
    case 4: *ptr = n->dn2; if (bytes) *bytes = b * G_BYTES; break;
    case 5: *ptr = n->dn1; if (bytes) *bytes = b * N1_POS * C1_OUT * 2; break;
    case 6: *ptr = n->w1_shadow; if (bytes) *bytes = (int64_t)FLAT * FC * 2; break;
    case 7: *ptr = n->xblk; if (bytes) *bytes = b * XB_FRAME_BYTES; break;
    default: return set_error("ga3c_workspace_ptr: bad id");
  }
  return 0;
}

extern "C" int ga3c_histograms(ga3c_net* n, int32_t batch, const float* p, const float* v, double* out, int32_t* bad,
                               void* stream) {
  if (int r = check_batch(n, batch, "ga3c_histograms")) return r;
  if (!p || !v || !out || !bad) return set_error("ga3c_histograms: null buffer");
  if (batch != n->last_batch) return set_error("ga3c_histograms: batch differs from the last forward on this handle");
  if (n->dp_world > 1) return set_error("ga3c_histograms: not available on a peer-memory data-parallel handle");
  CK(cudaSetDevice(n->cfg.device));
  static_assert(GA3C_HISTO_SOURCES == P_COUNT + 5, "sources: the variables, n1, n2, d1, v, p");
  HistoArgs a{};
  for (int i = 0; i < P_COUNT; ++i) a.src[i] = HistoSrc{n->w + n->off(i), n->params[i].count, 0, 0};
  const long long b = batch;
  if (n->generic) {
    a.src[P_COUNT + 0] = HistoSrc{n->gen.n1, b * n->geo.h1 * n->geo.w1 * C1_OUT, 1, 0};
    a.src[P_COUNT + 1] = HistoSrc{n->n2, b * n->geo.kdim, 1, 0};
  } else {
    a.src[P_COUNT + 0] = HistoSrc{n->n1, b * B2_BYTES / 2, 1, 1};
    a.src[P_COUNT + 1] = HistoSrc{n->n2, b * FLAT, 1, 0};
  }
  a.src[P_COUNT + 2] = HistoSrc{n->d1, b * FC, 0, 0};
  a.src[P_COUNT + 3] = HistoSrc{v, b, 0, 0};
  a.src[P_COUNT + 4] = HistoSrc{p, b * n->cfg.num_actions, 0, 0};
  a.n_src = GA3C_HISTO_SOURCES;
  a.out = out;
  a.bad = bad;
  return launch_histograms(n, a, (cudaStream_t)stream);
}

extern "C" int ga3c_keep_dn1(ga3c_net* n, int32_t on) {
  if (!n) return set_error("ga3c_keep_dn1: null handle");
  n->keep_dn1 = on != 0;
  return 0;
}

extern "C" int64_t ga3c_launch_count(const ga3c_net* n) { return n ? n->log.launches : 0; }

extern "C" int ga3c_kernel_count(void) { return K_COUNT; }
extern "C" const char* ga3c_kernel_name(int kid) { return (kid >= 0 && kid < K_COUNT) ? kKernelNames[kid] : nullptr; }

// ---- step timeline trace --------------------------------------------------------------------------
static int trace_attach_all(unsigned long long* buf) {
  int r;
  if ((r = trace_attach_conv_fwd(buf)) || (r = trace_attach_conv_bwd_fused(buf)) || (r = trace_attach_dense_tc(buf)) ||
      (r = trace_attach_heads(buf)) || (r = trace_attach_elementwise(buf)) || (r = trace_attach_conv_gen(buf)) || (r = trace_attach_mlp(buf)) || (r = trace_attach_mlp_tc(buf)) || (r = trace_attach_mlp_stream(buf)))
    return r;
  return 0;
}

extern "C" int ga3c_trace_begin(ga3c_net* n, void* stream) {
  if (!n) return set_error("ga3c_trace_begin: null handle");
  CK(cudaSetDevice(n->cfg.device));
  const size_t words = (size_t)K_COUNT * TRACE_SLOTS;
  if (!n->trace) CK(cudaMalloc((void**)&n->trace, words * 8));
  std::vector<unsigned long long> init(words);
  for (size_t i = 0; i < words; ++i) init[i] = (i & 1) ? 0ull : ~0ull;      // even slots take a min, odd slots a max
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  CK(cudaMemcpy(n->trace, init.data(), words * 8, cudaMemcpyHostToDevice));
  CKL(trace_attach_all(n->trace));
  return 0;
}

extern "C" int ga3c_trace_end(ga3c_net* n, uint64_t* stamps, int32_t n_kernels) {
  if (!n || !stamps || n_kernels < K_COUNT) return set_error("ga3c_trace_end: bad argument");
  if (!n->trace) return set_error("ga3c_trace_end: no trace in progress");
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  CKL(trace_attach_all(nullptr));
  CK(cudaMemcpy(stamps, n->trace, (size_t)K_COUNT * TRACE_SLOTS * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// ---- pipeline event log (debug) ----------------------------------------------------------------------
extern "C" int ga3c_evt_begin(ga3c_net* n) {
  if (!n) return set_error("ga3c_evt_begin: null handle");
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  if (!n->evt) CK(cudaMalloc((void**)&n->evt, (size_t)2 * 16384 * 8));
  CK(cudaMemset(n->evt, 0, (size_t)2 * 16384 * 8));
  // the kernels share the 16 warp regions of one buffer: GA3C_EVT_DENSE=1 (tools/evt_dense.py, a -DGA3C_DENSE_EVT build) leaves them
  // to the dense1 GEMMs
  if (getenv("GA3C_EVT_DENSE") == nullptr) {
    CKL(evt_attach_conv_fwd(n->evt));
    CKL(evt_attach_conv_bwd(n->evt));
    CKL(evt_attach_elementwise(n->evt));
  } else {
    CKL(evt_attach_dense_tc(n->evt));
  }
  return 0;
}

extern "C" int ga3c_evt_end(ga3c_net* n, uint64_t* records, int32_t cap, int32_t* count) {
  if (!n || !records || !count || !n->evt || cap < 16384) return set_error("ga3c_evt_end: bad argument");
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  CKL(evt_attach_conv_fwd(nullptr));
  CKL(evt_attach_conv_bwd(nullptr));
  CKL(evt_attach_elementwise(nullptr));
  CKL(evt_attach_dense_tc(nullptr));
  std::vector<uint64_t> all((size_t)2 * 16384);
  CK(cudaMemcpy(all.data(), n->evt, all.size() * 8, cudaMemcpyDeviceToHost));
  int32_t c = 0;
  for (int i = 0; i < 16384; ++i)
    if (all[2 * i] != 0) { records[2 * c] = all[2 * i]; records[2 * c + 1] = all[2 * i + 1]; ++c; }
  *count = c;
  return 0;
}

extern "C" int ga3c_timing_enable(ga3c_net* n, int32_t max_records) {
  return timing_enable(n, max_records, "ga3c_timing_enable");
}

extern "C" int ga3c_timing_collect(ga3c_net* n, double* total_ms, int64_t* counts, int32_t n_kernels) {
  return timing_collect(n, total_ms, counts, n_kernels, "ga3c_timing_collect");
}
