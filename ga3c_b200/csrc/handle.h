// The state and host logic the conv handle (ga3c_net, net.cu) and the MLP handle (ga3c_mlp, mlp_net.cu) share: the variable
// table, the flat arenas and the optimizer state in them, batch and step bookkeeping, the histogram launches and the
// per-kernel timing.  Each handle derives from Handle<its config struct>; the config fields read here have the same names in
// ga3c_config and ga3c_mlp_config.  Entry points pass their own name (`who`) for the error messages.
#pragma once
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/ga3c_b200.h"
#include "common.cuh"
#include "kernels.h"
#include "host_util.h"

namespace ga3c {

// one variable of the arenas; live = 0: no cost reaches it (NetworkVP_discrate builds every DENSE_LAYERS entry from x, only
// the last one feeds the heads), so it has no gradient and no optimizer touches it
struct Param {
  std::string name;
  int64_t offset, count;
  int32_t ndim;
  int64_t shape[4];
  int32_t live;
};

constexpr int64_t ALIGN_FLOATS = 64;
inline int64_t align_up(int64_t v) { return (v + ALIGN_FLOATS - 1) / ALIGN_FLOATS * ALIGN_FLOATS; }

template <class Config>
struct Handle {
  Config cfg;
  int num_sms = 148;
  std::vector<Param> params;       // TF creation order
  int64_t arena_floats = 0;
  // one allocation [w | g | ms | mom | the handle's extra bytes]
  uint8_t* slab = nullptr;
  size_t slab_bytes = 0;
  float *w = nullptr, *g = nullptr, *ms = nullptr, *mom = nullptr;
  float *g2 = nullptr, *ms2 = nullptr, *mom2 = nullptr;   // Config.DUAL_RMSPROP: gradient of cost_v and the second optimizer's slots
  float *clip_ss = nullptr, *clip_scale = nullptr;        // Config.USE_GRAD_CLIP scratch: chunk sums of squares, per-tensor scale
  float *clip_ss2 = nullptr, *clip_scale2 = nullptr;      // ... of the second optimizer's gradient (DUAL_RMSPROP + USE_GRAD_CLIP)
  double* histo_part = nullptr;    // histograms: fp64 partial moments per block
  size_t histo_part_bytes = 0;
  int64_t skip_lo[4] = {}, skip_hi[4] = {};     // Config.DUAL_RMSPROP: what each optimizer leaves alone (RmsPropDualArgs)
  int last_batch = 0;              // rows of the activation workspace written by the last forward
  int64_t global_step = 0;
  int step_advance = 1;            // global_step per optimizer update, set at create from the reference's rules
  LaunchLog log;                   // launch counter + per-kernel CUDA-event timing
};

// selects the device of a new handle; the number of its SMs
inline int open_device(int device, const char* who, int* num_sms) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return set_error(std::string(who) + ": no CUDA device (there is no CPU fallback)");
  if (device < 0 || device >= ndev) return set_error(std::string(who) + ": device ordinal out of range");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return set_error(std::string(who) + ": kernels are built for sm_100a only; device is sm_" + std::to_string(prop.major) +
                     std::to_string(prop.minor));
  *num_sms = prop.multiProcessorCount;
  return 0;
}

// once the table is laid out: the four arenas in one zeroed allocation with extra_bytes behind them, the second optimizer's
// arenas and the clip scratch as the config asks.  The caller destroys the handle on failure.
template <class C>
int alloc_arenas(Handle<C>* h, size_t extra_bytes) {
  const size_t ab = (size_t)h->arena_floats * sizeof(float);
  h->slab_bytes = 4 * ab + extra_bytes;
  CK(cudaMalloc((void**)&h->slab, h->slab_bytes));
  CK(cudaMemset(h->slab, 0, h->slab_bytes));
  h->w = reinterpret_cast<float*>(h->slab);
  h->g = h->w + h->arena_floats; h->ms = h->g + h->arena_floats; h->mom = h->ms + h->arena_floats;
  if (h->cfg.dual_rmsprop) {
    CK(cudaMalloc((void**)&h->g2, 3 * ab));
    CK(cudaMemset(h->g2, 0, 3 * ab));
    h->ms2 = h->g2 + h->arena_floats; h->mom2 = h->ms2 + h->arena_floats;
  }
  const std::vector<float> ones((size_t)h->arena_floats, 1.0f);    // ms slots start at 1.0 [TF-SEMANTICS]
  float* const ms_slots[2] = {h->ms, h->ms2};
  for (float* ms : ms_slots)
    if (ms) CK(cudaMemcpy(ms, ones.data(), ab, cudaMemcpyHostToDevice));
  if (h->cfg.use_grad_clip) {
    int64_t mx = 0;
    for (const Param& p : h->params) mx = std::max(mx, p.count);
    const size_t ss = h->params.size() * clip_chunks(mx) * sizeof(float), sc = h->params.size() * sizeof(float);
    CK(cudaMalloc((void**)&h->clip_ss, ss));
    CK(cudaMalloc((void**)&h->clip_scale, sc));
    if (h->cfg.dual_rmsprop) {
      CK(cudaMalloc((void**)&h->clip_ss2, ss));
      CK(cudaMalloc((void**)&h->clip_scale2, sc));
    }
  }
  return 0;
}

template <class C>
void free_arenas(Handle<C>* h) {
  cudaFree(h->slab);
  cudaFree(h->g2);
  cudaFree(h->clip_ss); cudaFree(h->clip_scale); cudaFree(h->clip_ss2); cudaFree(h->clip_scale2);
  cudaFree(h->histo_part);
  h->log.clear();
}

// arena ids of the C ABI
template <class C>
float* arena_of(Handle<C>* h, int which) {
  switch (which) {
    case 0: return h->w; case 1: return h->g; case 2: return h->ms; case 3: return h->mom;
    case 4: return h->g2; case 5: return h->ms2; case 6: return h->mom2;      // null unless dual_rmsprop
  }
  return nullptr;
}

// whole-arena copies, behind the work queued on the device
template <class C>
int arena_upload(Handle<C>* h, int which, const float* host, int64_t nf, const char* who) {
  if (!h || !host) return set_error(std::string(who) + ": null argument");
  float* dst = arena_of(h, which);
  if (!dst || nf != h->arena_floats) return set_error(std::string(who) + ": bad arena id or size");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(dst, host, (size_t)nf * 4, cudaMemcpyHostToDevice));
  return 0;
}

template <class C>
int arena_download(Handle<C>* h, int which, float* host, int64_t nf, const char* who) {
  if (!h || !host) return set_error(std::string(who) + ": null argument");
  float* src = arena_of(h, which);
  if (!src || nf != h->arena_floats) return set_error(std::string(who) + ": bad arena id or size");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(host, src, (size_t)nf * 4, cudaMemcpyDeviceToHost));
  return 0;
}

template <class C>
int param_info(const Handle<C>* h, int i, const char** name, int64_t* offset, int32_t* ndim, int64_t shape[4], int32_t* live,
               const char* who) {
  if (!h || i < 0 || i >= (int)h->params.size()) return set_error(std::string(who) + ": bad index");
  const Param& d = h->params[i];
  if (name) *name = d.name.c_str();
  if (offset) *offset = d.offset;
  if (ndim) *ndim = d.ndim;
  if (shape) for (int k = 0; k < 4; ++k) shape[k] = d.shape[k];
  if (live) *live = d.live;
  return 0;
}

template <class C>
int check_batch(const Handle<C>* h, int batch, const char* who) {
  if (!h) return set_error(std::string(who) + ": null handle");
  if (batch < 1 || batch > h->cfg.max_batch)
    return set_error(std::string(who) + ": batch " + std::to_string(batch) + " outside 1.." + std::to_string(h->cfg.max_batch));
  return 0;
}

// the histograms of the sources in `a` (out / bad filled in by the caller) into a.out, a.bad on stream st
template <class C>
int launch_histograms(Handle<C>* h, HistoArgs& a, cudaStream_t st) {
  if (int r = histo_plan(a)) return r;
  const size_t part_bytes = sizeof(double) * 4 * histo_blocks(a);
  if (part_bytes > h->histo_part_bytes) {
    CK(cudaFree(h->histo_part));
    h->histo_part = nullptr;
    h->histo_part_bytes = 0;
    CK(cudaMalloc((void**)&h->histo_part, part_bytes));
    h->histo_part_bytes = part_bytes;
  }
  a.part = h->histo_part;
  if (int r = histo_zero(a, st)) return r;
  LAUNCH(h, K_HISTO, st, launch_histo(a, st));
  LAUNCH(h, K_HISTO, st, launch_histo_merge(a, st));
  return 0;
}

template <class C>
int timing_enable(Handle<C>* h, int32_t max_records, const char* who) {
  if (!h || max_records < 0) return set_error(std::string(who) + ": bad argument");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  return h->log.enable(max_records);
}

template <class C>
int timing_collect(Handle<C>* h, double* total_ms, int64_t* counts, int32_t n_kernels, const char* who) {
  if (!h || !total_ms || !counts || n_kernels < K_COUNT) return set_error(std::string(who) + ": bad argument");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  return h->log.collect(total_ms, reinterpret_cast<long long*>(counts), n_kernels);
}

// the fields of the first optimizer's RMSPropArgs both handles set; it updates the arena's first n_floats
template <class C>
RmsPropArgs rmsprop_base(const Handle<C>* h, float lr, int64_t n_floats) {
  RmsPropArgs a{};
  a.w = h->w; a.ms = h->ms; a.mom = h->mom; a.g = h->g;
  a.n_floats = n_floats;
  a.lr = lr; a.decay = h->cfg.rmsprop_decay; a.momentum = h->cfg.rmsprop_momentum; a.eps = h->cfg.rmsprop_epsilon;
  return a;
}

// Config.USE_GRAD_CLIP over the live variables: which = 0 the (first) optimizer's gradient, 1 the second one's
template <class C>
ClipArgs clip_args(const Handle<C>* h, int which) {
  ClipArgs c{};
  c.g = which ? h->g2 : h->g;
  int64_t mx = 0;
  for (const Param& p : h->params) {
    if (!p.live) continue;
    c.offset[c.n_tensors] = p.offset; c.count[c.n_tensors] = p.count; ++c.n_tensors;
    mx = std::max(mx, p.count);
  }
  c.max_chunks = clip_chunks(mx);
  c.clip = h->cfg.grad_clip_norm;
  c.chunk_ss = which ? h->clip_ss2 : h->clip_ss; c.scale = which ? h->clip_scale2 : h->clip_scale;
  return c;
}

// The optimizer update of the arena the config selects -- RMSProp, with Config.USE_GRAD_CLIP, with Config.DUAL_RMSPROP, or
// with both -- over the handle's first optimizer arguments `a`.  One timing record under K_RMSPROP, every kernel counted.
template <class C>
int launch_optimizer(Handle<C>* h, const RmsPropArgs& a, cudaStream_t st) {
  const bool clip = h->cfg.use_grad_clip;
  int kernels = 0;
  ClipArgs c1{}, c2{};
  if (h->cfg.dual_rmsprop) {
    RmsPropDualArgs d{};
    d.a = a;
    d.g2 = h->g2; d.ms2 = h->ms2; d.mom2 = h->mom2;
    for (int i = 0; i < 4; ++i) { d.skip_lo[i] = h->skip_lo[i]; d.skip_hi[i] = h->skip_hi[i]; }
    // tf.clip_by_norm per variable and optimizer (NetworkVP.py:127-137, NetworkVP_discrate.py:107-117); the gradient-less
    // variables' gradient is None there, which the reference filters and clip_args leaves out
    if (clip) { c1 = clip_args(h, 0); c2 = clip_args(h, 1); c1.by_norm = c2.by_norm = 1; }
    LAUNCH(h, K_RMSPROP, st, launch_rmsprop_dual(d, clip ? &c1 : nullptr, clip ? &c2 : nullptr, st, &kernels));
  } else {
    if (clip) c1 = clip_args(h, 0);
    LAUNCH(h, K_RMSPROP, st, launch_rmsprop(a, clip ? &c1 : nullptr, st, &kernels));
  }
  h->log.launches += kernels - 1;        // LAUNCH counted one
  h->global_step += h->step_advance;
  return 0;
}

}  // namespace ga3c
