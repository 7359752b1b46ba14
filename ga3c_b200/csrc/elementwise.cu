// HBM-bound elementwise kernels: RMSProp over the flat arena, bf16 shadow refresh, discounted
// returns, action sampling.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "dp_exchange.cuh"

namespace ga3c {

// ---- gradient-partial reduction ---------------------------------------------------------------------
// The heads / conv12_bwd / conv11_wgrad kernels leave one slab of partial sums per CTA (a mirror of the small-tensor
// prefix of the gradient arena + the loss sums).  512 threads = 16 slab lanes x 32 float4 columns: lane l adds slabs
// l, l + 16, ... (independent 16-byte loads of L2-resident data), then the 16 lane sums are added in lane order.
// The order is a function of the launch geometry only, so the gradients are bit-reproducible.
constexpr int GR_LANES = 16, GR_COLS = 32, GR_UNROLL = 10;     // 160 slabs (one per SM) in a single batch of loads
__global__ void __launch_bounds__(GR_LANES * GR_COLS) grad_reduce_kernel(GradReduceArgs a) {
  __shared__ float4 part[GR_LANES][GR_COLS];
  const int col = threadIdx.x & (GR_COLS - 1), sl = threadIdx.x / GR_COLS;
  const int j = (blockIdx.x * GR_COLS + col) * 4;
  int count = 0;
  if (j < a.n_floats) {
#pragma unroll
    for (int s = GR_MAX_SEG - 1; s >= 0; --s)
      if (j < a.seg_end[s]) count = a.seg_count[s];
  }
  griddep_launch();
  griddep_wait(K_GRAD_REDUCE);  // the slabs come from the kernels that precede this one
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const float* src = a.part + j;
  for (int i0 = sl; i0 < count; i0 += GR_UNROLL * GR_LANES) {
    float4 q[GR_UNROLL];
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u) {
      const int i = i0 + u * GR_LANES;
      q[u] = i < count ? __ldcg(reinterpret_cast<const float4*>(src + (int64_t)i * a.stride)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u) { acc.x += q[u].x; acc.y += q[u].y; acc.z += q[u].z; acc.w += q[u].w; }
  }
  part[sl][col] = acc;
  __syncthreads();
  if (sl == 0 && j < a.n_floats) {
#pragma unroll
    for (int l = 1; l < GR_LANES; ++l) {
      const float4 q = part[l][col];
      acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
    }
    if (j < a.out_floats) *reinterpret_cast<float4*>(a.out + j) = acc;
    else if (a.out_tail != nullptr) {          // caller's buffer: no alignment assumed
      float* t = a.out_tail + (j - a.out_floats);
      t[0] = acc.x; t[1] = acc.y; t[2] = acc.z; t[3] = acc.w;
    }
  }
  trace_mark(K_GRAD_REDUCE, 2);
}

GA3C_TRACE_ATTACH(trace_attach_elementwise)

int launch_grad_reduce(const GradReduceArgs& a, cudaStream_t stream) {
  const int grid = (a.n_floats / 4 + GR_COLS - 1) / GR_COLS;
  return launch_pdl(grad_reduce_kernel, dim3(grid), dim3(GR_LANES * GR_COLS), 0, stream, a);
}

// ---- RMSProp, TensorFlow semantics (tf.train.RMSPropOptimizer, NetworkVP_discrate.py:101-105) ----
//   ms  <- rho*ms + (1-rho)*g^2 ; mom <- mu*mom + lr*g/sqrt(ms + eps) ; w <- w - mom       [TF-SEMANTICS]
// One float4 per thread per iteration over the whole arena (all 10 variables in one launch instead
// of TF's 10 ApplyRMSProp launches).  With mu == 0 (Config.RMSPROP_MOMENTUM) the mom slot is dead:
// 20 B/param of traffic (read w,g,ms; write w,ms) + 2 B/param for the bf16 shadow of dense1/w.
template <bool HAS_MOM>
__device__ __forceinline__ void rms_update(const RmsPropArgs& a, const float4& g, float4& w, float4& ms, float4& mo) {
  const float one_m_rho = 1.f - a.decay;
#define GA3C_RMS(c)                                                          \
  ms.c = a.decay * ms.c + one_m_rho * g.c * g.c;                             \
  mo.c = a.momentum * mo.c + a.lr * g.c / sqrtf(ms.c + a.eps);              \
  w.c -= mo.c;
  GA3C_RMS(x) GA3C_RMS(y) GA3C_RMS(z) GA3C_RMS(w)
#undef GA3C_RMS
}

template <bool HAS_MOM>
__global__ void __launch_bounds__(256) rmsprop_kernel(RmsPropArgs a) {
  griddep_launch();
  griddep_wait(K_RMSPROP);      // the gradients come from the backward kernels that precede this one
  const int64_t n4 = a.n_floats >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 g = reinterpret_cast<const float4*>(a.g)[i];
    float4 w = reinterpret_cast<float4*>(a.w)[i];
    float4 ms = reinterpret_cast<float4*>(a.ms)[i];
    float4 mo = HAS_MOM ? reinterpret_cast<float4*>(a.mom)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    rms_update<HAS_MOM>(a, g, w, ms, mo);
    reinterpret_cast<float4*>(a.w)[i] = w;
    reinterpret_cast<float4*>(a.ms)[i] = ms;
    if (HAS_MOM) reinterpret_cast<float4*>(a.mom)[i] = mo;
    const int64_t e = i << 2;
    if (e >= a.w1_offset && e < a.w1_offset + a.w1_count)
      reinterpret_cast<uint2*>(a.w1_shadow)[(e - a.w1_offset) >> 2] = make_uint2(pack_bf16(w.x, w.y), pack_bf16(w.z, w.w));
  }
  trace_mark(K_RMSPROP, 2);
}

int launch_rmsprop(const RmsPropArgs& a, cudaStream_t stream) {
  const int64_t n4 = a.n_floats >> 2;
  const int grid = (int)((n4 + 255) / 256 < 148 * 8 ? (n4 + 255) / 256 : 148 * 8);
  if (a.momentum != 0.f) return launch_pdl(rmsprop_kernel<true>, dim3(grid), dim3(256), 0, stream, a);
  return launch_pdl(rmsprop_kernel<false>, dim3(grid), dim3(256), 0, stream, a);
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

template <bool HAS_MOM>
__global__ void __launch_bounds__(256) rmsprop_clip_kernel(RmsPropArgs a, ClipArgs c) {
  griddep_launch();
  griddep_wait(K_RMSPROP);
  const int64_t n4 = a.n_floats >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const int64_t e = i << 2;
    float sc = 0.f;                       // alignment gaps between tensors hold zeros
#pragma unroll
    for (int t = 0; t < CLIP_MAX_TENSORS; ++t)
      if (t < c.n_tensors && e >= c.offset[t] && e < c.offset[t] + c.count[t]) sc = c.scale[t];
    float4 g = reinterpret_cast<const float4*>(a.g)[i];
    // a float4 never straddles two tensors' live elements with different scales unless a count is not a multiple of 4: then
    // the tail elements belong to the gap (zeros), so one scale per float4 is exact
    g.x *= sc; g.y *= sc; g.z *= sc; g.w *= sc;
    float4 w = reinterpret_cast<float4*>(a.w)[i];
    float4 ms = reinterpret_cast<float4*>(a.ms)[i];
    float4 mo = HAS_MOM ? reinterpret_cast<float4*>(a.mom)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    rms_update<HAS_MOM>(a, g, w, ms, mo);
    reinterpret_cast<float4*>(a.w)[i] = w;
    reinterpret_cast<float4*>(a.ms)[i] = ms;
    if (HAS_MOM) reinterpret_cast<float4*>(a.mom)[i] = mo;
    if (a.w1_count > 0 && e >= a.w1_offset && e < a.w1_offset + a.w1_count)
      reinterpret_cast<uint2*>(a.w1_shadow)[(e - a.w1_offset) >> 2] = make_uint2(pack_bf16(w.x, w.y), pack_bf16(w.z, w.w));
  }
  trace_mark(K_RMSPROP, 2);
}

int clip_chunks(int64_t max_count) { return (int)((max_count + CLIP_CHUNK - 1) / CLIP_CHUNK); }

int launch_rmsprop_clipped(const RmsPropArgs& a, const ClipArgs& c, cudaStream_t stream) {
  int r;
  if ((r = launch_pdl(grad_sqnorm_kernel, dim3(c.max_chunks, c.n_tensors), dim3(256), 0, stream, c))) return r;
  if ((r = launch_pdl(clip_scale_kernel, dim3(1), dim3(32 * CLIP_MAX_TENSORS), 0, stream, c))) return r;
  const int64_t n4 = a.n_floats >> 2;
  const int grid = (int)((n4 + 255) / 256 < 148 * 8 ? (n4 + 255) / 256 : 148 * 8);
  if (a.momentum != 0.f) return launch_pdl(rmsprop_clip_kernel<true>, dim3(grid), dim3(256), 0, stream, a, c);
  return launch_pdl(rmsprop_clip_kernel<false>, dim3(grid), dim3(256), 0, stream, a, c);
}

// ---- Config.DUAL_RMSPROP (NetworkVP_discrate.py:87-98, :124-128) ---------------------------------------------
template <bool HAS_MOM>
__global__ void __launch_bounds__(256) rmsprop_dual_kernel(RmsPropDualArgs d) {
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
    if (d.scale1 != nullptr) {           // one scale per float4 is exact: tensors start 4-aligned, gaps hold zeros
      s1 = s2 = 0.f;
#pragma unroll
      for (int t = 0; t < CLIP_MAX_TENSORS; ++t)
        if (t < d.n_tensors && e >= d.t_offset[t] && e < d.t_offset[t] + d.t_count[t]) { s1 = d.scale1[t]; s2 = d.scale2[t]; }
    }
    if (!skip1) {
      float4 g = reinterpret_cast<const float4*>(a.g)[i];
      g.x *= s1; g.y *= s1; g.z *= s1; g.w *= s1;
      float4 ms = reinterpret_cast<float4*>(a.ms)[i];
      float4 mo = HAS_MOM ? reinterpret_cast<float4*>(a.mom)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 w1 = w0;
      rms_update<HAS_MOM>(a, g, w1, ms, mo);
      w.x -= w0.x - w1.x; w.y -= w0.y - w1.y; w.z -= w0.z - w1.z; w.w -= w0.w - w1.w;
      reinterpret_cast<float4*>(a.ms)[i] = ms;
      if (HAS_MOM) reinterpret_cast<float4*>(a.mom)[i] = mo;
    }
    if (!skip2) {
      float4 g = reinterpret_cast<const float4*>(d.g2)[i];
      g.x *= s2; g.y *= s2; g.z *= s2; g.w *= s2;
      float4 ms = reinterpret_cast<float4*>(d.ms2)[i];
      float4 mo = HAS_MOM ? reinterpret_cast<float4*>(d.mom2)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 w2 = w0;
      rms_update<HAS_MOM>(a, g, w2, ms, mo);
      w.x -= w0.x - w2.x; w.y -= w0.y - w2.y; w.z -= w0.z - w2.z; w.w -= w0.w - w2.w;
      reinterpret_cast<float4*>(d.ms2)[i] = ms;
      if (HAS_MOM) reinterpret_cast<float4*>(d.mom2)[i] = mo;
    }
    reinterpret_cast<float4*>(a.w)[i] = w;
    if (a.w1_count > 0 && e >= a.w1_offset && e < a.w1_offset + a.w1_count)
      reinterpret_cast<uint2*>(a.w1_shadow)[(e - a.w1_offset) >> 2] = make_uint2(pack_bf16(w.x, w.y), pack_bf16(w.z, w.w));
  }
  trace_mark(K_RMSPROP, 2);
}

int launch_rmsprop_dual(const RmsPropDualArgs& d, cudaStream_t stream) {
  const int64_t n4 = d.a.n_floats >> 2;
  const int grid = (int)((n4 + 255) / 256 < 148 * 8 ? (n4 + 255) / 256 : 148 * 8);
  if (d.a.momentum != 0.f) return launch_pdl(rmsprop_dual_kernel<true>, dim3(grid), dim3(256), 0, stream, d);
  return launch_pdl(rmsprop_dual_kernel<false>, dim3(grid), dim3(256), 0, stream, d);
}

int launch_rmsprop_dual_clipped(RmsPropDualArgs d, const ClipArgs& c1, const ClipArgs& c2, cudaStream_t stream) {
  int r;
  for (const ClipArgs* c : {&c1, &c2}) {
    if ((r = launch_pdl(grad_sqnorm_kernel, dim3(c->max_chunks, c->n_tensors), dim3(256), 0, stream, *c))) return r;
    if ((r = launch_pdl(clip_scale_kernel, dim3(1), dim3(32 * CLIP_MAX_TENSORS), 0, stream, *c))) return r;
  }
  d.scale1 = c1.scale; d.scale2 = c2.scale; d.n_tensors = c1.n_tensors;
  for (int t = 0; t < c1.n_tensors; ++t) { d.t_offset[t] = c1.offset[t]; d.t_count[t] = c1.count[t]; }
  return launch_rmsprop_dual(d, stream);
}

// ---- single-GPU step tail: grad_reduce + RMSProp in one launch -------------------------------------------
// Blocks [0, n_red) sum the gradient-partial slabs of 32 float4 columns exactly like grad_reduce_kernel (same order,
// same bits), store the reduced gradient and apply RMSProp to those columns; the remaining blocks update dense1/w,
// one float4 per thread.  w / ms (and mom) do not depend on the preceding kernels, so they are loaded BEFORE the
// dependency wait and their latency hides under the tail of the backward -- but only when a.preload says that this is safe:
// w / ms were last written by the optimizer launch of the PREVIOUS step, and a prologue is ordered after that launch only if
// some kernel in between cannot become resident next to it.  With batch >= num_sms the conv kernels of this step occupy every
// SM with a CTA that takes the SM's whole shared memory, so every CTA of the previous optimizer launch has exited before this
// kernel can be launched; with smaller batches the whole chain of a step can sit in its prologues while the previous
// optimizer is still running (back-to-back asynchronous calls), and the loads move behind the wait.
constexpr int RR_U = 3;      // float4 per thread in the dense1/w blocks of rmsprop_reduce_kernel
template <bool HAS_MOM>
__global__ void __launch_bounds__(GR_LANES * GR_COLS, 2) rmsprop_reduce_kernel(RmsPropArgs a, GradReduceArgs r, int n_red) {
  __shared__ float4 part[GR_LANES][GR_COLS];
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  if ((int)blockIdx.x < n_red) {
    const int col = threadIdx.x & (GR_COLS - 1), sl = threadIdx.x / GR_COLS;
    const int j = (blockIdx.x * GR_COLS + col) * 4;
    int count = 0;
    if (j < r.n_floats) {
#pragma unroll
      for (int s = GR_MAX_SEG - 1; s >= 0; --s)
        if (j < r.seg_end[s]) count = r.seg_count[s];
    }
    const bool owner = sl == 0 && j < r.out_floats;
    float4 w = zero, ms = zero, mo = zero;
    if (owner && a.preload) {
      w = *reinterpret_cast<const float4*>(a.w + j);
      ms = *reinterpret_cast<const float4*>(a.ms + j);
      if (HAS_MOM) mo = *reinterpret_cast<const float4*>(a.mom + j);
    }
    griddep_launch();
    griddep_wait(K_RMSPROP);      // the slabs come from the kernels that precede this one
    if (owner && !a.preload) {
      w = *reinterpret_cast<const float4*>(a.w + j);
      ms = *reinterpret_cast<const float4*>(a.ms + j);
      if (HAS_MOM) mo = *reinterpret_cast<const float4*>(a.mom + j);
    }
    float4 acc = zero;
    const float* src = r.part + j;
    for (int i0 = sl; i0 < count; i0 += GR_UNROLL * GR_LANES) {
      float4 q[GR_UNROLL];
#pragma unroll
      for (int u = 0; u < GR_UNROLL; ++u) {
        const int i = i0 + u * GR_LANES;
        q[u] = i < count ? __ldcg(reinterpret_cast<const float4*>(src + (int64_t)i * r.stride)) : zero;
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
      if (owner) {
        *reinterpret_cast<float4*>(r.out + j) = acc;                 // the reduced gradient (introspection, checkpoints)
        rms_update<HAS_MOM>(a, acc, w, ms, mo);
        *reinterpret_cast<float4*>(a.w + j) = w;
        *reinterpret_cast<float4*>(a.ms + j) = ms;
        if (HAS_MOM) *reinterpret_cast<float4*>(a.mom + j) = mo;
      } else if (r.out_tail != nullptr) {
        float* t = r.out_tail + (j - r.out_floats);
        t[0] = acc.x; t[1] = acc.y; t[2] = acc.z; t[3] = acc.w;
      }
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
      if (i < n4 && a.preload) {
        w[u] = reinterpret_cast<const float4*>(a.w)[i];
        ms[u] = reinterpret_cast<const float4*>(a.ms)[i];
        if (HAS_MOM) mo[u] = reinterpret_cast<const float4*>(a.mom)[i];
      }
    }
    griddep_launch();
    griddep_wait(K_RMSPROP);      // dense1/w's gradient comes from the wgrad GEMM
    if (!a.preload) {
#pragma unroll
      for (int u = 0; u < RR_U; ++u) {
        const int64_t i = i0 + u * blockDim.x;
        if (i < n4) {
          w[u] = reinterpret_cast<const float4*>(a.w)[i];
          ms[u] = reinterpret_cast<const float4*>(a.ms)[i];
          if (HAS_MOM) mo[u] = reinterpret_cast<const float4*>(a.mom)[i];
        }
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
        rms_update<HAS_MOM>(a, g[u], w[u], ms[u], mo[u]);
        reinterpret_cast<float4*>(a.w)[i] = w[u];
        reinterpret_cast<float4*>(a.ms)[i] = ms[u];
        if (HAS_MOM) reinterpret_cast<float4*>(a.mom)[i] = mo[u];
        const int64_t e = i << 2;
        if (e >= a.w1_offset && e < a.w1_offset + a.w1_count)
          reinterpret_cast<uint2*>(a.w1_shadow)[(e - a.w1_offset) >> 2] = make_uint2(pack_bf16(w[u].x, w[u].y), pack_bf16(w[u].z, w[u].w));
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
  if (a.momentum != 0.f) return launch_pdl(rmsprop_reduce_kernel<true>, dim3(grid), dim3(T), 0, stream, a, r, n_red);
  return launch_pdl(rmsprop_reduce_kernel<false>, dim3(grid), dim3(T), 0, stream, a, r, n_red);
}

GA3C_EVT_ATTACH(evt_attach_elementwise)

// ---- data-parallel exchange, small tensors (dp_exchange.cuh) ---------------------------------------------
// One block per 32-float4 column block of the small-tensor prefix (+ the loss sums).  Block cb sums this rank's per-CTA
// slabs for its columns (same order and bits as grad_reduce_kernel); its 32 owner threads push the sums into every peer's
// receive buffer in the LL wire format, collect the peers' contributions from this rank's own receive buffer, add them in
// rank order (every rank computes the identical sum) and apply RMSProp to the local copy.  Receive buffers alternate with
// the step parity: a peer pushes step s + 2 only after it has seen this rank's step s + 1, i.e. after this rank's step-s
// launch has ended.
template <bool HAS_MOM>
__global__ void __launch_bounds__(GR_LANES * GR_COLS) dp_small_kernel(RmsPropDpArgs d, int64_t recv_offset) {
  __shared__ float4 part[GR_LANES][GR_COLS];
  EvtLog evt_i = evt_open();
  const RmsPropArgs& a = d.base;
  const GradReduceArgs& r = d.red;
  const int col = threadIdx.x & (GR_COLS - 1), sl = threadIdx.x / GR_COLS;
  const int j = (blockIdx.x * GR_COLS + col) * 4;
  const bool owner = sl == 0 && j < r.out_floats;
  int count = 0;
  if (j < r.n_floats) {
#pragma unroll
    for (int s = GR_MAX_SEG - 1; s >= 0; --s)
      if (j < r.seg_end[s]) count = r.seg_count[s];
  }
  float4 w = make_float4(0.f, 0.f, 0.f, 0.f), ms = w, mo = w;
  auto load_state = [&]() {
    w = *reinterpret_cast<const float4*>(a.w + j);
    ms = *reinterpret_cast<const float4*>(a.ms + j);
    if (HAS_MOM) mo = *reinterpret_cast<const float4*>(a.mom + j);
  };
  // w / ms of the small prefix were last written by this kernel one step ago; see rmsprop_reduce_kernel for when the early
  // loads are safe
  if (owner && a.preload) load_state();
  griddep_launch();
  evt_mark(evt_i, 60, 0);
  griddep_wait(K_RMSPROP);        // the slabs come from the conv backward launch that precedes this one
  evt_mark(evt_i, 61, 0);
  if (owner && !a.preload) load_state();
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
    if (j >= r.out_floats && r.out_tail != nullptr) {
      float* t = r.out_tail + (j - r.out_floats);
      t[0] = acc.x; t[1] = acc.y; t[2] = acc.z; t[3] = acc.w;
    }
  }
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
    rms_update<HAS_MOM>(a, g, w, ms, mo);
    *reinterpret_cast<float4*>(a.w + j) = w;
    *reinterpret_cast<float4*>(a.ms + j) = ms;
    if (HAS_MOM) *reinterpret_cast<float4*>(a.mom + j) = mo;
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
  if (d.base.momentum != 0.f)
    return launch_pdl(dp_small_kernel<true>, dim3(n_cb), dim3(GR_LANES * GR_COLS), 0, stream, d, recv_offset);
  return launch_pdl(dp_small_kernel<false>, dim3(n_cb), dim3(GR_LANES * GR_COLS), 0, stream, d, recv_offset);
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
  const int grid = (int)((n4 + 255) / 256 < 148 * 8 ? (n4 + 255) / 256 : 148 * 8);
  f32_to_bf16_kernel<<<grid, 256, 0, stream>>>(src, dst, n4);
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
