// C-ABI host layer of the low-dimensional MLP networks (ga3c_mlp_*, include/ga3c_b200.h): handle, arenas, workspace and
// the launch sequences.  Kernels: mlp.cu (+ the arena RMSProp of elementwise.cu).
#include <string>
#include <algorithm>
#include <vector>

#include "handle.h"
#include "mlp.cuh"

using namespace ga3c;

struct ga3c_mlp : Handle<ga3c_mlp_config> {
  MlpNet net{};
  int64_t live_floats = 0;               // live tensors are packed first; [live_floats, arena_floats) is never updated
  float* part = nullptr;                 // [MLP_MAX_SPLITS][live_floats] weight-gradient partial arenas
  // workspace for max_batch rows; last_batch: rows of act[] written by the last forward (0: none since it was allocated)
  float* act[MLP_MAX_LAYERS] = {};
  float* dz[MLP_MAX_LAYERS] = {};
  float* dlogits = nullptr;
  float* loss_part = nullptr;
  // tensor-core mode (mlp_tc.cu): the run of wide layers [tc_lo, tc_hi) as 3xTF32 GEMMs for training batches >= tc_min_batch
  int tc_lo = 0, tc_hi = 0, tc_min_batch = 4096;
  bool stream_ok = false;                // ... with the narrow ends as streaming passes (mlp_stream.cu)
};

static void free_workspace(ga3c_mlp* n) {
  for (int l = 0; l < MLP_MAX_LAYERS; ++l) { cudaFree(n->act[l]); cudaFree(n->dz[l]); n->act[l] = n->dz[l] = nullptr; }
  cudaFree(n->dlogits); cudaFree(n->loss_part);
  n->dlogits = n->loss_part = nullptr;
}

static int alloc_workspace(ga3c_mlp* n, int max_batch) {
  const size_t mb = (size_t)max_batch;
  for (int l = 0; l < n->net.n_layers; ++l) {
    CK(cudaMalloc((void**)&n->act[l], mb * n->net.L[l].n * 4));
    CK(cudaMalloc((void**)&n->dz[l], mb * n->net.L[l].n * 4));
  }
  CK(cudaMalloc((void**)&n->dlogits, mb * n->net.n_out_ld * 4));
  // one row per batch tile (tiles of >= 16 rows), or one per block of the streaming heads kernel (mlp_heads_loss_rows <= 8 per SM)
  const size_t loss_rows = std::max((mb + 15) / 16, (size_t)n->num_sms * 64);
  CK(cudaMalloc((void**)&n->loss_part, loss_rows * 4 * 4));
  n->cfg.max_batch = max_batch;
  return 0;
}

extern "C" int ga3c_mlp_destroy(ga3c_mlp* n) {
  if (!n) return 0;
  free_arenas(n);
  cudaFree(n->part);
  free_workspace(n);
  delete n;
  return 0;
}

extern "C" int ga3c_mlp_create(const ga3c_mlp_config* cfg, ga3c_mlp** out) {
  if (!cfg || !out) return set_error("ga3c_mlp_create: null argument");
  *out = nullptr;
  if (cfg->kind != GA3C_MLP_FORK_VP && cfg->kind != GA3C_MLP_DISCRATE) return set_error("ga3c_mlp_create: unknown kind");
  if (cfg->num_actions < 1 || cfg->num_actions > MAX_ACTIONS) return set_error("ga3c_mlp_create: num_actions must be 1..18");
  if (cfg->state_dim < 1 || cfg->state_dim > MLP_MAX_WIDTH) return set_error("ga3c_mlp_create: state_dim must be 1..256");
  if (cfg->max_batch < 1) return set_error("ga3c_mlp_create: max_batch must be >= 1");
  if (cfg->kind == GA3C_MLP_DISCRATE) {
    if (cfg->n_dense < 1 || cfg->n_dense > MLP_MAX_LAYERS) return set_error("ga3c_mlp_create: n_dense must be 1..8");
    for (int i = 0; i < cfg->n_dense; ++i)
      if (cfg->dense_width[i] < 1 || cfg->dense_width[i] > MLP_MAX_WIDTH)
        return set_error("ga3c_mlp_create: dense widths must be 1..256");
    if (cfg->dense_width[cfg->n_dense - 1] > MLP_MAX_HID) return set_error("ga3c_mlp_create: the last dense width must be <= 128");
  }
  int num_sms = 0;
  if (int r = open_device(cfg->device, "ga3c_mlp_create", &num_sms)) return r;

  ga3c_mlp* n = new ga3c_mlp();
  n->cfg = *cfg;
  n->num_sms = num_sms;
  const int S = cfg->state_dim, A = cfg->num_actions;
  MlpNet& net = n->net;
  net.kind = cfg->kind; net.state_dim = S; net.num_actions = A;

  auto add = [&](const std::string& scope, int k, int width, int live) {    // dense_layer: 'w' [k, width] then 'b' [width]
    Param w{scope + "/w:0", 0, (int64_t)k * width, 2, {k, width, 0, 0}, live};
    Param b{scope + "/b:0", 0, (int64_t)width, 1, {width, 0, 0, 0}, live};
    n->params.push_back(w); n->params.push_back(b);
    return (int)n->params.size() - 2;
  };
  std::vector<int> layer_param;          // index of each live hidden layer's 'w' in params
  if (cfg->kind == GA3C_MLP_FORK_VP) {   // NetworkVP.py:79-85
    const char* names[5] = {"dense11_p", "dense12_p", "dense13_p", "dense14_p", "dense1"};
    const int widths[5] = {4, 256, 256, 100, 64};
    const int acts[5] = {MLP_ACT_LINEAR, MLP_ACT_LINEAR, MLP_ACT_LINEAR, MLP_ACT_SIGMOID, MLP_ACT_SIGMOID};
    int fan = S;
    net.n_layers = 5;
    for (int l = 0; l < 5; ++l) {
      layer_param.push_back(add(names[l], fan, widths[l], 1));
      net.L[l].k = fan; net.L[l].n = widths[l]; net.L[l].act = acts[l];
      fan = widths[l];
    }
  } else {                               // NetworkVP_discrate.py:52-56: every layer reads x; the last one is self.denselayer
    for (int i = 0; i < cfg->n_dense; ++i) {
      const int live = i == cfg->n_dense - 1;
      const int idx = add("dense1_" + std::to_string(i + 1) + "_p", S, cfg->dense_width[i], live);
      if (live) layer_param.push_back(idx);
    }
    net.n_layers = 1;
    net.L[0].k = S; net.L[0].n = cfg->dense_width[cfg->n_dense - 1]; net.L[0].act = MLP_ACT_SIGMOID;
  }
  net.hid = net.L[net.n_layers - 1].n;
  {  // the first run of consecutive layers wide enough for 128 x BN tensor-core tiles (fork NetworkVP: 256 -> 256 -> 100 -> 64)
    int lo = 0;
    while (lo < net.n_layers && !mlp_tc_layer_ok(net.L[lo])) ++lo;
    int hi = lo;
    while (hi < net.n_layers && mlp_tc_layer_ok(net.L[hi])) ++hi;
    if (lo >= 1 && hi > lo) { n->tc_lo = lo; n->tc_hi = hi; }       // (layer 0 reads x: never wide here)
    if (const char* e = getenv("GA3C_MLP_TC")) {                     // 0: never; N > 0: from training batches of N rows
      const int v = atoi(e);
      if (v <= 0) n->tc_lo = n->tc_hi = 0; else n->tc_min_batch = v;
    }
  }
  const int pv = add("logits_v", net.hid, 1, 1);
  int px, py = -1;
  if (cfg->kind == GA3C_MLP_FORK_VP) {
    px = add("logits_p/out_x", net.hid, A, 1);
    py = add("logits_p/out_y", net.hid, A, 1);
    net.n_out = 1 + 2 * A;
  } else {
    px = add("logits_p", net.hid, A, 1);
    net.n_out = 1 + A;
  }
  net.n_out_ld = (net.n_out + 3) & ~3;
  int64_t cur = 0;
  for (int pass = 1; pass >= 0; --pass) {          // live tensors first, then the gradient-less ones
    for (Param& p : n->params)
      if (p.live == pass) { p.offset = cur; cur = align_up(cur + p.count); }
    if (pass == 1) n->live_floats = cur;
  }
  n->arena_floats = cur;
  for (int l = 0; l < net.n_layers; ++l) {
    net.L[l].w_off = (int)n->params[layer_param[l]].offset;
    net.L[l].b_off = (int)n->params[layer_param[l] + 1].offset;
  }
  net.wv_off = (int)n->params[pv].offset; net.bv_off = (int)n->params[pv + 1].offset;
  net.wp_off = (int)n->params[px].offset; net.bp_off = (int)n->params[px + 1].offset;
  if (py >= 0) { net.wy_off = (int)n->params[py].offset; net.by_off = (int)n->params[py + 1].offset; }
  // DUAL_RMSPROP (NetworkVP.py:107-118): cost_p does not reach logits_v/*, cost_v not the policy head, whose variables are
  // consecutive in the arena
  n->skip_lo[0] = n->params[pv].offset; n->skip_hi[0] = n->params[pv + 1].offset + n->params[pv + 1].count;
  const int plast = py >= 0 ? py + 1 : px + 1;
  n->skip_lo[2] = n->params[px].offset; n->skip_hi[2] = n->params[plast].offset + n->params[plast].count;
  // opt.minimize(..., global_step=self.global_step) once per optimizer; clipped, the fork's NetworkVP still hands global_step to
  // apply_gradients (NetworkVP.py:127-141) and NetworkVP_discrate does not (NetworkVP_discrate.py:107-121)
  n->step_advance = cfg->use_grad_clip && cfg->kind != GA3C_MLP_FORK_VP ? 0 : cfg->dual_rmsprop ? 2 : 1;
  n->stream_ok = n->tc_hi > n->tc_lo && mlp_stream_ok(net, n->tc_lo, n->tc_hi);

  if (cfg->use_grad_clip) {
    for (const Param& p : n->params)
      if (!p.live && !cfg->dual_rmsprop) {     // opt.compute_gradients yields (None, var) and tf.clip_by_average_norm(None, ..) raises;
                                               // the DUAL_RMSPROP branch filters `if not g is None` (NetworkVP_discrate.py:110,:115)
        ga3c_mlp_destroy(n);
        return set_error("ga3c_mlp_create: USE_GRAD_CLIP with gradient-less variables (NetworkVP_discrate.py:55 builds every "
                         "DENSE_LAYERS entry from x): the reference graph cannot be built either");
      }
    if ((int)n->params.size() > CLIP_MAX_TENSORS) { ga3c_mlp_destroy(n); return set_error("ga3c_mlp_create: too many variables for USE_GRAD_CLIP"); }
  }
  if (int r = alloc_arenas(n, 0)) { ga3c_mlp_destroy(n); return r; }
  cudaError_t e = cudaMalloc((void**)&n->part, (size_t)MLP_MAX_SPLITS * n->live_floats * 4);
  if (e != cudaSuccess) { ga3c_mlp_destroy(n); return fail_cuda("cudaMalloc", e); }
  cudaMemset(n->part, 0, (size_t)MLP_MAX_SPLITS * n->live_floats * 4);
  if (int r = alloc_workspace(n, cfg->max_batch)) { ga3c_mlp_destroy(n); return r; }
  if (int r = configure_mlp()) { ga3c_mlp_destroy(n); return fail_cuda("cudaFuncSetAttribute", (cudaError_t)r); }
  e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { ga3c_mlp_destroy(n); return fail_cuda("ga3c_mlp_create sync", e); }
  *out = n;
  return 0;
}

extern "C" int ga3c_mlp_reserve(ga3c_mlp* n, int32_t max_batch) {
  if (!n) return set_error("ga3c_mlp_reserve: null handle");
  if (max_batch <= n->cfg.max_batch) return 0;
  CK(cudaSetDevice(n->cfg.device));
  CK(cudaDeviceSynchronize());
  free_workspace(n);
  n->last_batch = 0;
  if (int r = alloc_workspace(n, max_batch)) { n->cfg.max_batch = 0; return r; }
  return 0;
}

extern "C" int ga3c_mlp_param_count(const ga3c_mlp* n) { return n ? (int)n->params.size() : 0; }

extern "C" int ga3c_mlp_param_info(const ga3c_mlp* n, int i, const char** name, int64_t* offset, int32_t* ndim,
                                   int64_t shape[4], int32_t* live) {
  return param_info(n, i, name, offset, ndim, shape, live, "ga3c_mlp_param_info");
}

extern "C" int64_t ga3c_mlp_arena_floats(const ga3c_mlp* n) { return n ? n->arena_floats : 0; }

extern "C" int ga3c_mlp_arena_upload(ga3c_mlp* n, int which, const float* host, int64_t nf) {
  return arena_upload(n, which, host, nf, "ga3c_mlp_arena_upload");
}

extern "C" int ga3c_mlp_arena_download(ga3c_mlp* n, int which, float* host, int64_t nf) {
  return arena_download(n, which, host, nf, "ga3c_mlp_arena_download");
}

extern "C" int64_t ga3c_mlp_global_step(const ga3c_mlp* n) { return n ? n->global_step : -1; }
extern "C" int ga3c_mlp_set_global_step(ga3c_mlp* n, int64_t s) { if (!n) return -1; n->global_step = s; return 0; }
extern "C" int64_t ga3c_mlp_launch_count(const ga3c_mlp* n) { return n ? n->log.launches : 0; }

// kernel-level test entry for the 3xTF32 tensor-core GEMMs of mlp_tc.cu (all pointers device, fp32 row-major):
//   mode 0  out [m, n] = act(a [m, k] x b [k, n] + aux [n])                       (forward)
//   mode 1  out [m, k] = (a [m, n] x b [k, n]^T) * act'(aux [m, k])               (data gradient)
//   mode 2  out [splits][k, n] = a [m, k]^T x b [m, n] per batch split of rows_per_split rows (weight gradient)
extern "C" int ga3c_debug_tf32x3_gemm(int32_t mode, const float* a, const float* b, const float* aux, float* out, int32_t m,
                                      int32_t k, int32_t nn, int32_t act, int32_t splits, int32_t rows_per_split, void* stream) {
  if (!a || !b || !out || m < 1 || k < 4 || nn < 4 || k > 256 || nn > 256 || (k & 3) || (nn & 3))
    return set_error("ga3c_debug_tf32x3_gemm: bad argument (k, n multiples of 4 up to 256)");
  cudaStream_t st = (cudaStream_t)stream;
  int r = 0;
  if (mode == 0) r = launch_mlp_tc_fwd(b, aux, k, nn, act, a, out, m, st);
  else if (mode == 1) r = launch_mlp_tc_dgrad(b, k, nn, a, aux, act, out, m, st);
  else if (mode == 2) {
    if (splits < 1 || rows_per_split < 32 || rows_per_split % 32) return set_error("ga3c_debug_tf32x3_gemm: rows_per_split must be a multiple of 32");
    r = launch_mlp_tc_wgrad(k, nn, a, b, m, splits, rows_per_split, out, nullptr, (int64_t)k * nn, st);
  } else return set_error("ga3c_debug_tf32x3_gemm: mode must be 0, 1 or 2");
  if (r) return fail_cuda("ga3c_debug_tf32x3_gemm", (cudaError_t)r);
  return 0;
}
extern "C" int ga3c_mlp_workspace_ptr(ga3c_mlp* n, int32_t which, int32_t layer, void** ptr, int32_t* width) {
  if (!n || !ptr || !width) return set_error("ga3c_mlp_workspace_ptr: null argument");
  if (which < 0 || which > 1 || layer < 0 || layer >= n->net.n_layers) return set_error("ga3c_mlp_workspace_ptr: bad matrix id");
  *ptr = which == 0 ? n->act[layer] : n->dz[layer];
  *width = n->net.L[layer].n;
  return 0;
}

extern "C" int ga3c_mlp_histogram_count(const ga3c_mlp* n) {
  return n ? (int)n->params.size() + n->net.n_layers + 2 : 0;
}

extern "C" int ga3c_mlp_histograms(ga3c_mlp* n, int32_t batch, const float* p, const float* v, double* out, int32_t* bad,
                                   void* stream) {
  if (int r = check_batch(n, batch, "ga3c_mlp_histograms")) return r;
  if (!p || !v || !out || !bad) return set_error("ga3c_mlp_histograms: null buffer");
  if (batch != n->last_batch) return set_error("ga3c_mlp_histograms: batch differs from the last forward on this handle");
  const int n_src = ga3c_mlp_histogram_count(n);
  if (n_src > HISTO_MAX_SRC) return set_error("ga3c_mlp_histograms: more than " + std::to_string(HISTO_MAX_SRC) + " sources");
  CK(cudaSetDevice(n->cfg.device));
  // the variables (gradient-less ones included: they are trainable variables of the graph), act[] of every live hidden layer,
  // v, p.  Arena offsets are multiples of ALIGN_FLOATS and each act[l] is its own allocation: every source is 16-byte aligned.
  HistoArgs a{};
  int s = 0;
  for (const Param& q : n->params) a.src[s++] = HistoSrc{n->w + q.offset, q.count, 0, 0};
  const long long b = batch;
  for (int l = 0; l < n->net.n_layers; ++l) a.src[s++] = HistoSrc{n->act[l], b * n->net.L[l].n, 0, 0};
  a.src[s++] = HistoSrc{v, b, 0, 0};
  a.src[s++] = HistoSrc{p, b * n->cfg.num_actions, 0, 0};
  a.n_src = n_src;
  a.out = out;
  a.bad = bad;
  return launch_histograms(n, a, (cudaStream_t)stream);
}

// the first optimizer over the live prefix; no bf16 shadow
static RmsPropArgs rmsprop_args(ga3c_mlp* n, float lr) {
  RmsPropArgs a = rmsprop_base(n, lr, n->live_floats);
  a.w1_offset = n->live_floats;
  return a;
}

static MlpStepArgs step_args(ga3c_mlp* n, const float* x, int batch, float beta = 0.f, int part = 0) {
  MlpStepArgs s{};
  s.w = n->w; s.x = x; s.batch = batch;
  s.la = LossArgs{beta, n->cfg.log_epsilon, n->cfg.min_policy, n->cfg.use_log_softmax != 0, part};
  for (int l = 0; l < n->net.n_layers; ++l) { s.act[l] = n->act[l]; s.dz[l] = n->dz[l]; }
  s.dlogits = n->dlogits; s.loss_part = n->loss_part;
  return s;
}

extern "C" int ga3c_mlp_predict(ga3c_mlp* n, const float* x, int32_t batch, float* p_out, float* v_out, void* stream) {
  if (int r = check_batch(n, batch, "ga3c_mlp_predict")) return r;
  if (!x || !p_out || !v_out) return set_error("ga3c_mlp_predict: null buffer");
  CK(cudaSetDevice(n->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  MlpStepArgs s = step_args(n, x, batch);
  s.p_out = p_out; s.v_out = v_out; s.train = 0;
  if (n->stream_ok && batch >= n->tc_min_batch) {
    // large batches: front as a streaming pass, the wide layers as 3xTF32 GEMMs, heads as a streaming pass (the layer outputs go
    // through the training workspace; the handle mutex of the host layer serialises predict and train)
    const MlpNet& net = n->net;
    LAUNCH(n, K_MLP_FUSED, st, launch_mlp_front_fwd(net, s, n->num_sms, st));
    for (int l = n->tc_lo; l < n->tc_hi; ++l)
      LAUNCH(n, K_MLP_TC, st, launch_mlp_tc_fwd(n->w + net.L[l].w_off, n->w + net.L[l].b_off, net.L[l].k, net.L[l].n, net.L[l].act,
                                                n->act[l - 1], n->act[l], batch, st));
    LAUNCH(n, K_MLP_FUSED, st, launch_mlp_heads(net, s, n->num_sms, st));
    n->last_batch = batch;
    return 0;
  }
  LAUNCH(n, K_MLP_FUSED, st, launch_mlp_fused(n->net, s, n->num_sms, st));     // writes no act[]: last_batch stays
  return 0;
}

static int mlp_fb_impl(ga3c_mlp* n, const float* x, const float* yr, const float* a, int32_t batch, float beta, float* loss,
                       void* stream, int part, float* g_dst) {
  if (int r = check_batch(n, batch, "ga3c_mlp_forward_backward")) return r;
  if (!x || !yr || !a) return set_error("ga3c_mlp_forward_backward: null buffer");
  CK(cudaSetDevice(n->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  MlpStepArgs s = step_args(n, x, batch, beta, part);
  s.yr = yr; s.a = a; s.train = 1;
  n->last_batch = batch;
  const int tm = mlp_tile_rows(batch, n->num_sms);
  if (n->tc_hi > n->tc_lo && batch >= n->tc_min_batch) {
    // the wide layers as 3xTF32 tensor-core GEMMs over the activations the fused kernel keeps in HBM anyway
    const MlpNet& net = n->net;
    const int lo = n->tc_lo, hi = n->tc_hi;
    s.tc_lo = lo; s.tc_hi = hi;
    const bool streamed = n->stream_ok;       // narrow ends as streaming passes (mlp_stream.cu), else as fused-kernel phases
    s.phase = 1;
    if (streamed) LAUNCH(n, K_MLP_FUSED, st, launch_mlp_front_fwd(net, s, n->num_sms, st));
    else LAUNCH(n, K_MLP_FUSED, st, launch_mlp_fused(net, s, n->num_sms, st));
    for (int l = lo; l < hi; ++l)
      LAUNCH(n, K_MLP_TC, st, launch_mlp_tc_fwd(n->w + net.L[l].w_off, n->w + net.L[l].b_off, net.L[l].k, net.L[l].n, net.L[l].act,
                                                n->act[l - 1], n->act[l], batch, st));
    s.phase = 2;
    if (streamed) LAUNCH(n, K_MLP_FUSED, st, launch_mlp_heads(net, s, n->num_sms, st));
    else LAUNCH(n, K_MLP_FUSED, st, launch_mlp_fused(net, s, n->num_sms, st));
    for (int l = hi - 1; l >= lo; --l)
      LAUNCH(n, K_MLP_TC, st, launch_mlp_tc_dgrad(n->w + net.L[l].w_off, net.L[l].k, net.L[l].n, n->dz[l], n->act[l - 1],
                                                  net.L[l - 1].act, n->dz[l - 1], batch, st));
    if (lo >= 2) {
      s.phase = 3;
      if (streamed) LAUNCH(n, K_MLP_FUSED, st, launch_mlp_front_bwd(net, s, n->num_sms, st));
      else LAUNCH(n, K_MLP_FUSED, st, launch_mlp_fused(net, s, n->num_sms, st));
    }
    const int splits = MLP_MAX_SPLITS;
    int rows = (batch + splits - 1) / splits;
    rows = (rows + 31) / 32 * 32;
    // weight gradients: tensor-core layers by GEMM (+ a streaming pass for the bias), fan-in <= 4 layers by the streaming kernel
    // alone, whatever is left (the head matrix) by the tile kernel
    for (int l = 0; l < net.n_layers; ++l)
      if ((l >= lo && l < hi) || net.L[l].k <= 4) s.wgrad_skip |= 1u << l;
    if (mlp_heads_wgrad_ok(net)) {
      s.wgrad_skip |= 1u << net.n_layers;
      LAUNCH(n, K_MLP_WGRAD, st, launch_mlp_heads_wgrad(net, s, n->part, n->live_floats, splits, rows, st));
    }
    if (s.wgrad_skip != (2u << net.n_layers) - 1u)
      LAUNCH(n, K_MLP_WGRAD, st, launch_mlp_wgrad(net, s, n->part, n->live_floats, splits, st, rows));
    for (int l = 0; l < net.n_layers; ++l) {
      if (!((s.wgrad_skip >> l) & 1u)) continue;
      const bool tc = l >= lo && l < hi;
      const float* in = l == 0 ? x : n->act[l - 1];
      if (tc)
        LAUNCH(n, K_MLP_TC, st, launch_mlp_tc_wgrad(net.L[l].k, net.L[l].n, in, n->dz[l], batch, splits, rows,
                                                    n->part + net.L[l].w_off, n->part + net.L[l].b_off, n->live_floats, st));
      LAUNCH(n, K_MLP_WGRAD, st, launch_mlp_skinny_wgrad(tc ? 0 : net.L[l].k, net.L[l].n, in, n->dz[l], batch, splits, rows,
                                                         n->part + net.L[l].w_off, n->part + net.L[l].b_off, n->live_floats, st));
    }
    LAUNCH(n, K_MLP_REDUCE, st, launch_mlp_reduce(n->part, n->live_floats, splits, g_dst, (int)n->live_floats, n->loss_part,
                                                  streamed ? mlp_heads_loss_rows(batch, n->num_sms) : (batch + tm - 1) / tm, loss, st));
    return 0;
  }
  LAUNCH(n, K_MLP_FUSED, st, launch_mlp_fused(n->net, s, n->num_sms, st));
  const int splits = mlp_wgrad_splits(n->net, batch, n->num_sms);
  LAUNCH(n, K_MLP_WGRAD, st, launch_mlp_wgrad(n->net, s, n->part, n->live_floats, splits, st));
  LAUNCH(n, K_MLP_REDUCE, st, launch_mlp_reduce(n->part, n->live_floats, splits, g_dst, (int)n->live_floats, n->loss_part,
                                                (batch + tm - 1) / tm, loss, st));
  return 0;
}

extern "C" int ga3c_mlp_forward_backward(ga3c_mlp* n, const float* x, const float* yr, const float* a, int32_t batch,
                                         float beta, float* loss, void* stream) {
  if (!n) return set_error("ga3c_mlp_forward_backward: null handle");
  return mlp_fb_impl(n, x, yr, a, batch, beta, loss, stream, 0, n->g);
}

extern "C" int ga3c_mlp_apply_rmsprop(ga3c_mlp* n, float lr, void* stream) {
  if (!n) return set_error("ga3c_mlp_apply_rmsprop: null handle");
  CK(cudaSetDevice(n->cfg.device));
  if (n->cfg.dual_rmsprop) return set_error("ga3c_mlp_apply_rmsprop: with DUAL_RMSPROP use ga3c_mlp_train_step (two backward passes)");
  // USE_GRAD_CLIP: tf.clip_by_average_norm per variable (NetworkVP.py:138-141, NetworkVP_discrate.py:118-121); every variable
  // is live then (checked at create)
  return launch_optimizer(n, rmsprop_args(n, lr), (cudaStream_t)stream);
}

extern "C" int ga3c_mlp_train_step(ga3c_mlp* n, const float* x, const float* yr, const float* a, int32_t batch, float lr,
                                   float beta, float* loss, void* stream) {
  if (n && n->cfg.dual_rmsprop) {
    // Config.DUAL_RMSPROP (NetworkVP.py:107-118, :143-147): cost_p into g, cost_v into g2, both steps from the same weights
    if (int r = mlp_fb_impl(n, x, yr, a, batch, beta, loss, stream, 1, n->g)) return r;
    if (int r = mlp_fb_impl(n, x, yr, a, batch, beta, nullptr, stream, 2, n->g2)) return r;
    return launch_optimizer(n, rmsprop_args(n, lr), (cudaStream_t)stream);
  }
  if (int r = ga3c_mlp_forward_backward(n, x, yr, a, batch, beta, loss, stream)) return r;
  return ga3c_mlp_apply_rmsprop(n, lr, stream);
}

extern "C" int ga3c_mlp_timing_enable(ga3c_mlp* n, int32_t max_records) {
  return timing_enable(n, max_records, "ga3c_mlp_timing_enable");
}

extern "C" int ga3c_mlp_timing_collect(ga3c_mlp* n, double* total_ms, int64_t* counts, int32_t n_kernels) {
  return timing_collect(n, total_ms, counts, n_kernels, "ga3c_mlp_timing_collect");
}
