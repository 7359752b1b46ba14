// HBM-bound elementwise kernels: RMSProp over the flat arena, bf16 shadow refresh, discounted
// returns, action sampling.
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "kernels.h"
#include "dp_exchange.cuh"

namespace ga3c {

// ---- gradient-partial reduction ---------------------------------------------------------------------
// The heads / conv12_bwd / conv11_wgrad kernels leave one slab of partial sums per CTA (a mirror of the small-tensor
// prefix of the gradient arena + the loss sums).  512 threads = 16 slab lanes x 32 float4 columns: lane l adds slabs
// l, l + 16, ... (independent 16-byte loads of L2-resident data), then the 16 lane sums are added in lane order.
// The order is a function of the launch geometry only, so the gradients are bit-reproducible.  Every kernel that sums the
// slabs (grad_reduce_kernel, the slab blocks of rmsprop_reduce_kernel, dp_small_kernel) does it in slab_column_sum, so the
// sum is the same whichever of them runs: ga3c_fb_tail leaves the gradient ga3c_train_step applies, and every data-parallel
// rank computes its share of the small tensors alike.
constexpr int GR_LANES = 16, GR_COLS = 32, GR_UNROLL = 10;     // 160 slabs (one per SM) in a single batch of loads

// Floats j .. j + 3, j = (blockIdx.x * GR_COLS + col) * 4, summed over their slabs by the whole block (lane sl = threadIdx.x /
// GR_COLS), after the dependency wait.  Lane 0 gets the sum (the other lanes a partial one); it stores the loss sums
// (j >= out_floats) itself and leaves the gradient prefix to the caller.
__device__ __forceinline__ float4 slab_column_sum(const GradReduceArgs& r, int col, int sl) {
  __shared__ float4 part[GR_LANES][GR_COLS];
  const int j = (blockIdx.x * GR_COLS + col) * 4;
  int count = 0;
  if (j < r.n_floats) {
#pragma unroll
    for (int s = GR_MAX_SEG - 1; s >= 0; --s)
      if (j < r.seg_end[s]) count = r.seg_count[s];
  }
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const float* src = r.part + j;
  for (int i0 = sl; i0 < count; i0 += GR_UNROLL * GR_LANES) {
    float4 q[GR_UNROLL];
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u) {
      const int i = i0 + u * GR_LANES;
      q[u] = i < count ? __ldcg(reinterpret_cast<const float4*>(src + (int64_t)i * r.stride)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u) { acc.x += q[u].x; acc.y += q[u].y; acc.z += q[u].z; acc.w += q[u].w; }
  }
  part[sl][col] = acc;
  __syncthreads();
  if (sl == 0 && j < r.n_floats) {
#pragma unroll
    for (int l = 1; l < GR_LANES; ++l) {
      const float4 q = part[l][col];
      acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
    }
    if (j >= r.out_floats && r.out_tail != nullptr) {          // caller's buffer: no alignment assumed
      float* t = r.out_tail + (j - r.out_floats);
      t[0] = acc.x; t[1] = acc.y; t[2] = acc.z; t[3] = acc.w;
    }
  }
  return acc;
}

__global__ void __launch_bounds__(GR_LANES * GR_COLS) grad_reduce_kernel(GradReduceArgs a) {
  const int col = threadIdx.x & (GR_COLS - 1), sl = threadIdx.x / GR_COLS;
  const int j = (blockIdx.x * GR_COLS + col) * 4;
  griddep_launch();
  griddep_wait(K_GRAD_REDUCE);  // the slabs come from the kernels that precede this one
  const float4 acc = slab_column_sum(a, col, sl);
  if (sl == 0 && j < a.out_floats) *reinterpret_cast<float4*>(a.out + j) = acc;
  trace_mark(K_GRAD_REDUCE, 2);
}

GA3C_TRACE_ATTACH(trace_attach_elementwise)

int launch_grad_reduce(const GradReduceArgs& a, cudaStream_t stream) {
  const int grid = (a.n_floats / 4 + GR_COLS - 1) / GR_COLS;
  return launch_pdl(grad_reduce_kernel, dim3(grid), dim3(GR_LANES * GR_COLS), 0, stream, a);
}

// ---- optimizer state ---------------------------------------------------------------------------------------
// w, ms and mom of one float4 of an arena.  With mu == 0 (Config.RMSPROP_MOMENTUM, HAS_MOM = false) the mom slot is dead: it
// reads as zero and is never written.
// Preload rule.  w / ms (and mom) do not depend on the kernels that precede an optimizer launch, so the optimizer kernels of
// the train step (rmsprop_reduce_kernel, dp_small_kernel) load them BEFORE the dependency wait and their latency hides under the
// tail of the backward -- but only when a.preload says that this is safe: w / ms were last written by the optimizer launch of
// the PREVIOUS step, and a prologue is ordered after that launch only if some kernel in between cannot become resident next to
// it.  With batch >= num_sms the conv kernels of this step occupy every SM with a CTA that takes the SM's whole shared memory,
// so every CTA of the previous optimizer launch has exited before this kernel can be launched; with smaller batches the whole
// chain of a step can sit in its prologues while the previous optimizer is still running (back-to-back asynchronous calls),
// and the loads move behind the wait.
// e: the arena element of the float4, a multiple of 4
template <bool HAS_MOM>
__device__ __forceinline__ void load_slots(const float* ms, const float* mom, int64_t e, float4& ms_v, float4& mo_v) {
  ms_v = *reinterpret_cast<const float4*>(ms + e);
  mo_v = HAS_MOM ? *reinterpret_cast<const float4*>(mom + e) : make_float4(0.f, 0.f, 0.f, 0.f);
}
template <bool HAS_MOM>
__device__ __forceinline__ void store_slots(float* ms, float* mom, int64_t e, const float4& ms_v, const float4& mo_v) {
  *reinterpret_cast<float4*>(ms + e) = ms_v;
  if (HAS_MOM) *reinterpret_cast<float4*>(mom + e) = mo_v;
}
template <bool HAS_MOM>
__device__ __forceinline__ void load_state(const RmsPropArgs& a, int64_t e, float4& w, float4& ms, float4& mo) {
  w = *reinterpret_cast<const float4*>(a.w + e);
  load_slots<HAS_MOM>(a.ms, a.mom, e, ms, mo);
}
template <bool HAS_MOM>
__device__ __forceinline__ void store_state(const RmsPropArgs& a, int64_t e, const float4& w, const float4& ms, const float4& mo) {
  *reinterpret_cast<float4*>(a.w + e) = w;
  store_slots<HAS_MOM>(a.ms, a.mom, e, ms, mo);
}
// the bf16 shadow of dense1/w, if the float4 lies in [w1_offset, w1_offset + w1_count) (one unsigned compare)
__device__ __forceinline__ void store_shadow(const RmsPropArgs& a, int64_t e, const float4& w) {
  if ((uint64_t)(e - a.w1_offset) < (uint64_t)a.w1_count)
    reinterpret_cast<uint2*>(a.w1_shadow)[(e - a.w1_offset) >> 2] = make_uint2(pack_bf16(w.x, w.y), pack_bf16(w.z, w.w));
}

// grid of the grid-stride arena kernels: 256-thread blocks, at most 8 per SM of a 148-SM B200
static int arena_grid(int64_t n4) { return (int)std::min<int64_t>((n4 + 255) / 256, 148 * 8); }

// launch(std::true_type) when the optimizer has momentum (a live mom slot), launch(std::false_type) when it has none
template <class F>
static int by_momentum(float momentum, F&& launch) {
  return momentum != 0.f ? launch(std::true_type{}) : launch(std::false_type{});
}

// ---- Config.USE_GRAD_CLIP: tf.clip_by_average_norm per variable (NetworkVP_discrate.py:118-121) --------------
//   g' = g * clip / max(||g||_2 / n, clip),  n = number of elements of the variable        [TF-SEMANTICS]
// Three launches over the finished gradient arena: per-chunk sums of squares (one block per 4096 elements of one tensor,
// fixed-order block reduction), one warp per tensor turning the chunk sums into a scale, RMSProp with the scale of the
// tensor an element belongs to.  Fixed summation order: bit-reproducible.
constexpr int CLIP_CHUNK = 4096;
__global__ void __launch_bounds__(256) grad_sqnorm_kernel(ClipArgs c) {
  __shared__ float wsum[8];
  griddep_launch();
  griddep_wait(K_RMSPROP);
  const int t = blockIdx.y;
  const int64_t lo = (int64_t)blockIdx.x * CLIP_CHUNK;
  if (lo >= c.count[t]) return;
  const int64_t hi = lo + CLIP_CHUNK < c.count[t] ? lo + CLIP_CHUNK : c.count[t];
  const float* g = c.g + c.offset[t];
  float s = 0.f;
  for (int64_t i = lo + threadIdx.x; i < hi; i += 256) s = fmaf(g[i], g[i], s);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += wsum[w];
    c.chunk_ss[(int64_t)t * c.max_chunks + blockIdx.x] = tot;
  }
}

__global__ void __launch_bounds__(32 * CLIP_MAX_TENSORS) clip_scale_kernel(ClipArgs c) {
  griddep_launch();
  griddep_wait(K_RMSPROP);
  const int t = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (t >= c.n_tensors) return;
  const int nch = (int)((c.count[t] + CLIP_CHUNK - 1) / CLIP_CHUNK);
  float s = 0.f;
  for (int i = lane; i < nch; i += 32) s += c.chunk_ss[(int64_t)t * c.max_chunks + i];
  s = warp_sum(s);
  if (lane == 0) c.scale[t] = c.clip / fmaxf(c.by_norm ? sqrtf(s) : sqrtf(s) / (float)c.count[t], c.clip);
}

// the entry of `scale` (one per tensor of c) for arena element e, 0 in the alignment gaps between tensors (they hold zeros).
// One scale per float4 is exact: tensors start 4-aligned, and when a count is not a multiple of 4 the rest of its last float4
// lies in the gap.
__device__ __forceinline__ float clip_scale_at(const ClipArgs& c, const float* scale, int64_t e) {
  float sc = 0.f;
#pragma unroll
  for (int t = 0; t < CLIP_MAX_TENSORS; ++t)
    if (t < c.n_tensors && e >= c.offset[t] && e < c.offset[t] + c.count[t]) sc = scale[t];
  return sc;
}

int clip_chunks(int64_t max_count) { return (int)((max_count + CLIP_CHUNK - 1) / CLIP_CHUNK); }

// c.scale of every tensor of c: 2 launches
static int launch_clip_scales(const ClipArgs& c, cudaStream_t stream) {
  if (int r = launch_pdl(grad_sqnorm_kernel, dim3(c.max_chunks, c.n_tensors), dim3(256), 0, stream, c)) return r;
  return launch_pdl(clip_scale_kernel, dim3(1), dim3(32 * CLIP_MAX_TENSORS), 0, stream, c);
}

// ---- RMSProp over the arena ---------------------------------------------------------------------------------
// One float4 per thread per iteration over the whole arena (all 10 variables in one launch instead of TF's 10 ApplyRMSProp
// launches).  Without momentum: 20 B/param of traffic (read w,g,ms; write w,ms) + 2 B/param for the bf16 shadow of dense1/w.
// CLIP: each gradient scaled by its tensor's clip scale (c.scale) first.
template <bool HAS_MOM, bool CLIP>
__global__ void __launch_bounds__(256) rmsprop_kernel(RmsPropArgs a, ClipArgs c) {
  griddep_launch();
  griddep_wait(K_RMSPROP);      // the gradients come from the kernels that precede this one
  const int64_t n4 = a.n_floats >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const int64_t e = i << 2;
    float4 g = reinterpret_cast<const float4*>(a.g)[i];
    if (CLIP) {
      const float sc = clip_scale_at(c, c.scale, e);
      g.x *= sc; g.y *= sc; g.z *= sc; g.w *= sc;
    }
    float4 w, ms, mo;
    load_state<HAS_MOM>(a, e, w, ms, mo);
    rms_update(g, w, ms, mo, a.lr, a.decay, a.momentum, a.eps);
    store_state<HAS_MOM>(a, e, w, ms, mo);
    store_shadow(a, e, w);
  }
  trace_mark(K_RMSPROP, 2);
}

int launch_rmsprop(const RmsPropArgs& a, const ClipArgs* c, cudaStream_t stream, int* kernels) {
  *kernels = c != nullptr ? 3 : 1;
  if (c != nullptr)
    if (int r = launch_clip_scales(*c, stream)) return r;
  const int grid = arena_grid(a.n_floats >> 2);
  return by_momentum(a.momentum, [&](auto mom) {
    return c != nullptr ? launch_pdl(rmsprop_kernel<mom, true>, dim3(grid), dim3(256), 0, stream, a, *c)
                        : launch_pdl(rmsprop_kernel<mom, false>, dim3(grid), dim3(256), 0, stream, a, ClipArgs{});
  });
}

// ---- Config.DUAL_RMSPROP (NetworkVP_discrate.py:87-98, :124-128) ---------------------------------------------
template <bool HAS_MOM>
__global__ void __launch_bounds__(256) rmsprop_dual_kernel(RmsPropDualArgs d, ClipArgs c) {
  const RmsPropArgs& a = d.a;
  griddep_launch();
  griddep_wait(K_RMSPROP);
  const int64_t n4 = a.n_floats >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const int64_t e = i << 2;
    const bool skip1 = (e >= d.skip_lo[0] && e < d.skip_hi[0]) || (e >= d.skip_lo[1] && e < d.skip_hi[1]);
    const bool skip2 = (e >= d.skip_lo[2] && e < d.skip_hi[2]) || (e >= d.skip_lo[3] && e < d.skip_hi[3]);
    const float4 w0 = reinterpret_cast<float4*>(a.w)[i];
    float4 w = w0;
    float s1 = 1.f, s2 = 1.f;
    if (d.scale1 != nullptr) { s1 = clip_scale_at(c, d.scale1, e); s2 = clip_scale_at(c, d.scale2, e); }
    // one optimizer's step, taken at w0 and subtracted from w
    auto step = [&](const float* g_arena, float* ms_arena, float* mom_arena, float s) {
      float4 g = reinterpret_cast<const float4*>(g_arena)[i];
      g.x *= s; g.y *= s; g.z *= s; g.w *= s;
      float4 ms, mo;
      load_slots<HAS_MOM>(ms_arena, mom_arena, e, ms, mo);
      float4 wk = w0;
      rms_update(g, wk, ms, mo, a.lr, a.decay, a.momentum, a.eps);
      w.x -= w0.x - wk.x; w.y -= w0.y - wk.y; w.z -= w0.z - wk.z; w.w -= w0.w - wk.w;
      store_slots<HAS_MOM>(ms_arena, mom_arena, e, ms, mo);
    };
    if (!skip1) step(a.g, a.ms, a.mom, s1);
    if (!skip2) step(d.g2, d.ms2, d.mom2, s2);
    reinterpret_cast<float4*>(a.w)[i] = w;
    store_shadow(a, e, w);
  }
  trace_mark(K_RMSPROP, 2);
}

int launch_rmsprop_dual(RmsPropDualArgs d, const ClipArgs* c1, const ClipArgs* c2, cudaStream_t stream, int* kernels) {
  *kernels = c1 != nullptr ? 5 : 1;
  if (c1 != nullptr) {
    int r;
    if ((r = launch_clip_scales(*c1, stream)) || (r = launch_clip_scales(*c2, stream))) return r;
    d.scale1 = c1->scale; d.scale2 = c2->scale;
  }
  const ClipArgs table = c1 != nullptr ? *c1 : ClipArgs{};
  const int grid = arena_grid(d.a.n_floats >> 2);
  return by_momentum(d.a.momentum, [&](auto mom) {
    return launch_pdl(rmsprop_dual_kernel<mom>, dim3(grid), dim3(256), 0, stream, d, table);
  });
}

// ---- single-GPU step tail: grad_reduce + RMSProp in one launch -------------------------------------------
// Blocks [0, n_red) sum the gradient-partial slabs of 32 float4 columns (slab_column_sum), store the reduced gradient and
// apply RMSProp to those columns; the remaining blocks update dense1/w, one float4 per thread.  Both load w / ms (and mom)
// before the dependency wait when a.preload allows it (the preload rule above load_slots).
constexpr int RR_U = 3;      // float4 per thread in the dense1/w blocks of rmsprop_reduce_kernel
template <bool HAS_MOM>
__global__ void __launch_bounds__(GR_LANES * GR_COLS, 2) rmsprop_reduce_kernel(RmsPropArgs a, GradReduceArgs r, int n_red) {
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  if ((int)blockIdx.x < n_red) {
    const int col = threadIdx.x & (GR_COLS - 1), sl = threadIdx.x / GR_COLS;
    const int j = (blockIdx.x * GR_COLS + col) * 4;
    const bool owner = sl == 0 && j < r.out_floats;
    float4 w = zero, ms = zero, mo = zero;
    if (owner && a.preload) load_state<HAS_MOM>(a, j, w, ms, mo);
    griddep_launch();
    griddep_wait(K_RMSPROP);      // the slabs come from the kernels that precede this one
    if (owner && !a.preload) load_state<HAS_MOM>(a, j, w, ms, mo);
    const float4 g = slab_column_sum(r, col, sl);
    if (owner) {
      *reinterpret_cast<float4*>(r.out + j) = g;                 // the reduced gradient (introspection, checkpoints)
      rms_update(g, w, ms, mo, a.lr, a.decay, a.momentum, a.eps);
      store_state<HAS_MOM>(a, j, w, ms, mo);
    }
  } else {
    // RR_U float4 per thread, a block apart (coalesced).  RR_U = 3 keeps the whole grid -- 113 slab blocks + 162 of these at
    // B = 1024 -- inside ONE wave of 2 blocks per SM (52 registers x 512 threads); with two per thread the grid was 357 blocks
    // against 296 slots, and the 61 stragglers of the second wave cost the step ~3 us (profiles/r3c_step_trace_n1.md)
    const int64_t i0 = (r.out_floats >> 2) + (int64_t)(blockIdx.x - n_red) * (RR_U * blockDim.x) + threadIdx.x;
    const int64_t n4 = a.n_floats >> 2;
    float4 w[RR_U], ms[RR_U], mo[RR_U];
#pragma unroll
    for (int u = 0; u < RR_U; ++u) {
      const int64_t i = i0 + u * blockDim.x;
      w[u] = ms[u] = mo[u] = zero;
      if (i < n4 && a.preload) load_state<HAS_MOM>(a, i << 2, w[u], ms[u], mo[u]);
    }
    griddep_launch();
    griddep_wait(K_RMSPROP);      // dense1/w's gradient comes from the wgrad GEMM
    if (!a.preload) {
#pragma unroll
      for (int u = 0; u < RR_U; ++u) {
        const int64_t i = i0 + u * blockDim.x;
        if (i < n4) load_state<HAS_MOM>(a, i << 2, w[u], ms[u], mo[u]);
      }
    }
    float4 g[RR_U];
#pragma unroll
    for (int u = 0; u < RR_U; ++u) {
      const int64_t i = i0 + u * blockDim.x;
      g[u] = i < n4 ? reinterpret_cast<const float4*>(a.g)[i] : zero;
    }
#pragma unroll
    for (int u = 0; u < RR_U; ++u) {
      const int64_t i = i0 + u * blockDim.x;
      if (i < n4) {
        rms_update(g[u], w[u], ms[u], mo[u], a.lr, a.decay, a.momentum, a.eps);
        store_state<HAS_MOM>(a, i << 2, w[u], ms[u], mo[u]);
        store_shadow(a, i << 2, w[u]);
      }
    }
  }
  trace_mark(K_RMSPROP, 2);
}

int launch_rmsprop_reduce(const RmsPropArgs& a, const GradReduceArgs& r, cudaStream_t stream) {
  constexpr int T = GR_LANES * GR_COLS;
  const int n_red = (r.n_floats / 4 + GR_COLS - 1) / GR_COLS;
  const int64_t rest4 = (a.n_floats - r.out_floats) >> 2;
  const int grid = n_red + (int)((rest4 + RR_U * T - 1) / (RR_U * T));
  return by_momentum(a.momentum, [&](auto mom) {
    return launch_pdl(rmsprop_reduce_kernel<mom>, dim3(grid), dim3(T), 0, stream, a, r, n_red);
  });
}

GA3C_EVT_ATTACH(evt_attach_elementwise)

// ---- data-parallel exchange, small tensors (dp_exchange.cuh) ---------------------------------------------
// One block per 32-float4 column block of the small-tensor prefix (+ the loss sums).  Block cb sums this rank's per-CTA
// slabs for its columns (slab_column_sum); its 32 owner threads push the sums into every peer's
// receive buffer in the LL wire format, collect the peers' contributions from this rank's own receive buffer, add them in
// rank order (every rank computes the identical sum) and apply RMSProp to the local copy.  Receive buffers alternate with
// the step parity: a peer pushes step s + 2 only after it has seen this rank's step s + 1, i.e. after this rank's step-s
// launch has ended.
template <bool HAS_MOM>
__global__ void __launch_bounds__(GR_LANES * GR_COLS) dp_small_kernel(RmsPropDpArgs d, int64_t recv_offset) {
  EvtLog evt_i = evt_open();
  const RmsPropArgs& a = d.base;
  const GradReduceArgs& r = d.red;
  const int col = threadIdx.x & (GR_COLS - 1), sl = threadIdx.x / GR_COLS;
  const int j = (blockIdx.x * GR_COLS + col) * 4;
  const bool owner = sl == 0 && j < r.out_floats;
  float4 w = make_float4(0.f, 0.f, 0.f, 0.f), ms = w, mo = w;
  // w / ms of the small prefix were last written by this kernel one step ago: the preload rule above load_slots
  if (owner && a.preload) load_state<HAS_MOM>(a, j, w, ms, mo);
  griddep_launch();
  evt_mark(evt_i, 60, 0);
  griddep_wait(K_RMSPROP);        // the slabs come from the conv backward launch that precedes this one
  evt_mark(evt_i, 61, 0);
  if (owner && !a.preload) load_state<HAS_MOM>(a, j, w, ms, mo);
  const float4 acc = slab_column_sum(r, col, sl);
  evt_mark(evt_i, 62, 0);
  if (owner) {
    // receive buffers: [parity][source rank][small prefix in LL format: 8 bytes per float]
    uint8_t* my_comm = d.peer[d.rank] + d.comm_offset;
    const uint32_t flag = (uint32_t)d.step;
    const int64_t slot = recv_offset + ((int64_t)(d.step & 1) * DP_WORLD_MAX + d.rank) * r.out_floats * 8 + (int64_t)j * 8;
#pragma unroll
    for (int q = 0; q < DP_WORLD_MAX; ++q)
      if (q < d.world && q != d.rank) dp_ll_store(d.peer[q] + slot, acc, flag);
    *reinterpret_cast<float4*>(r.out + j) = acc;                     // this rank's own gradient (introspection)
    evt_mark(evt_i, 66, 0);
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int q = 0; q < DP_WORLD_MAX; ++q)
      if (q < d.world) {
        const float4 v = q == d.rank ? acc
                                     : dp_ll_load(d.peer[d.rank] + recv_offset +
                                                      ((int64_t)(d.step & 1) * DP_WORLD_MAX + q) * r.out_floats * 8 + (int64_t)j * 8,
                                                  flag, my_comm + DPC_ERR);
        g.x += v.x; g.y += v.y; g.z += v.z; g.w += v.w;
      }
    evt_mark(evt_i, 63, 0);
    rms_update(g, w, ms, mo, a.lr, a.decay, a.momentum, a.eps);
    store_state<HAS_MOM>(a, j, w, ms, mo);
  }
  evt_mark(evt_i, 64, 0);
  trace_mark(K_RMSPROP, 2);
}

// ---- data-parallel exchange, dense1/w: a kernel of its own on a side stream -----------------------------------------------
// 128-thread blocks without shared memory: small enough to be resident NEXT TO the conv backward CTAs of this step and the conv
// forward CTAs of the next one (both leave ~12 K registers and 1,500 thread slots per SM), so the whole chain of NVLink latencies
// -- wait for every rank's "dense_bwd done" flag, pull the slices, RMSProp, push the bf16 shadow, fence, "slice landed" flags, wait
// for every rank's -- runs under kernels that do not depend on it.  The next launch that reads the shadow (dense_fwd) waits for
// every rank's "slice landed" flag (DpGate, dense_tc.cu); block 0 ends only when every rank's slice has landed in THIS rank's slab.
// It is launched behind an event recorded after dense_bwd (its own gradient is final by stream order) and publishes
// that to the peers itself: it then only ever waits for OTHER GPUs, never for a kernel of its own GPU that might not find room
// on an SM next to it (a spinning kernel that waits for a kernel it keeps from being resident is a deadlock).
__global__ void __launch_bounds__(128, 6) dp_big_side_kernel(DpBigArgs big) {      // <= 85 registers: 11 K per block
  trace_mark(K_DP_BIG, 0);
  int dp_last = 0;      // thread 0's only.  NO shared memory: next to a conv CTA an SM has room for the reserved 1 KB of a block and no more
  dp_big_group(big, (int)threadIdx.x, 128, (int)blockIdx.x, (int)gridDim.x, 1, &dp_last);
  __syncthreads();
  trace_mark(K_DP_BIG, 1);             // (trace row of this kernel: first/last block started, own slice done, all slices landed)
  uint8_t* my_comm = big.peer[big.rank] + big.comm_offset;
  if (blockIdx.x == 0 && (int)threadIdx.x < big.world)
    dp_wait_flag_acquire(my_comm + DPC_BIGDONE + 64 * threadIdx.x, big.step, my_comm + DPC_ERR, 16u);
  if (blockIdx.x == 0) {
    __syncthreads();
    trace_mark(K_DP_BIG, 2);
  }
}
int launch_dp_big_side(const DpBigArgs& big, int num_sms, cudaStream_t side_stream) {
  int grid = num_sms;
  if (const char* e = getenv("GA3C_DP_SIDE_CTAS")) {     // tests with several ranks on one GPU leave room for the other ranks' kernels
    const int g = atoi(e);
    if (g >= 1 && g <= grid) grid = g;
  }
  dp_big_side_kernel<<<grid, 128, 0, side_stream>>>(big);
  return (int)cudaGetLastError();
}

// CUDA loads a kernel lazily at its first launch, and that load can wait for running kernels to finish.  A rank whose
// exchange CTAs are already spinning on a peer would then block the very launch the peer needs (ranks that share a
// process), so every kernel of the exchange is loaded when the ranks attach.
int configure_dp() {
  cudaFuncAttributes a;
  int r;
  if ((r = (int)cudaFuncGetAttributes(&a, dp_small_kernel<false>))) return r;
  if ((r = (int)cudaFuncGetAttributes(&a, dp_small_kernel<true>))) return r;
  return (int)cudaFuncGetAttributes(&a, dp_big_side_kernel);
}

int launch_dp_small(const RmsPropDpArgs& d, int64_t recv_offset, cudaStream_t stream) {
  const int n_cb = (d.red.n_floats / 4 + GR_COLS - 1) / GR_COLS;
  if (n_cb > DP_MAX_CB) return (int)cudaErrorInvalidValue;
  return by_momentum(d.base.momentum, [&](auto mom) {
    return launch_pdl(dp_small_kernel<mom>, dim3(n_cb), dim3(GR_LANES * GR_COLS), 0, stream, d, recv_offset);
  });
}

__global__ void __launch_bounds__(256) f32_to_bf16_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, int64_t n4) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    reinterpret_cast<uint2*>(dst)[i] = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
  }
}

int launch_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, cudaStream_t stream) {
  const int64_t n4 = n >> 2;
  f32_to_bf16_kernel<<<arena_grid(n4), 256, 0, stream>>>(src, dst, n4);
  return (int)cudaGetLastError();
}

// ---- discounted returns (ProcessAgent.py:70-84) -------------------------------------------------
// One thread per segment, sequential over time in fp64 with the reference's exact operation order
// (explicit __dmul_rn / __dadd_rn: no FMA contraction), so the result is bit-identical to the Python
// loop.  Parallel across agents; a parallel scan over time would reassociate and lose bit-exactness.
__global__ void __launch_bounds__(128)
returns_kernel(const double* __restrict__ rewards, const int64_t* __restrict__ seg, int n_segments,
               const double* __restrict__ terminal, double discount, int flags, double rmin, double rmax,
               double* __restrict__ out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_segments) return;
  const int64_t lo = seg[s], hi = seg[s + 1];
  if (hi <= lo) return;
  const bool discounting = flags & 1, intermediate = flags & 2, clipping = flags & 4, nstep = flags & 8;
  double run = terminal[s];
  if (nstep) {
    out[hi - 1] = run;
    for (int64_t t = hi - 2; t >= lo; --t) {
      double r = rewards[t];
      if (clipping) r = fmin(fmax(r, rmin), rmax);
      run = __dadd_rn(__dmul_rn(discount, run), r);
      out[t] = run;
    }
    return;
  }
  out[hi - 1] = rewards[hi - 1];
  for (int64_t t = hi - 2; t >= lo; --t) {
    double r = rewards[t];
    if (clipping) r = fmin(fmax(r, rmin), rmax);
    double o = rewards[t];
    if (discounting) {
      run = __dmul_rn(discount, run);
      if (intermediate) run = __dadd_rn(__dmul_rn(discount, run), r);
      else o = run;
    }
    out[t] = o;
  }
}

int launch_returns(const double* rewards, const int64_t* seg_offsets, int n_segments, const double* terminal,
                   double discount, int flags, double rmin, double rmax, double* out, cudaStream_t stream) {
  if (n_segments <= 0) return 0;
  returns_kernel<<<(n_segments + 127) / 128, 128, 0, stream>>>(rewards, seg_offsets, n_segments, terminal, discount,
                                                                 flags, rmin, rmax, out);
  return (int)cudaGetLastError();
}

// ---- action sampling (ProcessAgent.py:110-115) ---------------------------------------------------
// np.random.choice(actions, p=p) == searchsorted(cumsum(float64(p)) / cumsum[-1], u, side='right')
__global__ void __launch_bounds__(128)
select_actions_kernel(const float* __restrict__ p, const double* __restrict__ u, int batch, int na, int32_t* __restrict__ action) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch) return;
  double cdf[MAX_ACTIONS];
  double run = 0.0;
  for (int k = 0; k < na; ++k) { run = __dadd_rn(run, (double)p[(size_t)i * na + k]); cdf[k] = run; }
  const double tot = cdf[na - 1], ui = u[i];
  int idx = 0;
  for (int k = 0; k < na; ++k) idx += (__ddiv_rn(cdf[k], tot) <= ui) ? 1 : 0;   // side='right': count of cdf <= u
  action[i] = idx;
}

int launch_select_actions(const float* p, const double* u, int batch, int num_actions, int32_t* action,
                          cudaStream_t stream) {
  if (batch <= 0) return 0;
  if (num_actions < 1 || num_actions > MAX_ACTIONS) return (int)cudaErrorInvalidValue;
  select_actions_kernel<<<(batch + 127) / 128, 128, 0, stream>>>(p, u, batch, num_actions, action);
  return (int)cudaGetLastError();
}

}  // namespace ga3c
