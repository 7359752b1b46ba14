// Data-parallel exchange over CUDA-IPC peer memory (one process per GPU, NVLink / NVSwitch loads and stores).
//
// The step's gradients become final in two instalments, and so does the exchange:
//   dense1/w (98.6 % of the bytes) is final after dense_bwd.  dp_big_side_kernel (elementwise.cu), launched on a side stream
//       behind dense_bwd, reduce-scatters it, applies RMSProp to the owned slice and all-gathers the bf16 shadow into every
//       rank's slab WHILE the conv backward of this step and the conv forward of the next run on the main stream.  Only the
//       bf16 shadow (what dense_fwd / dense_bwd read) travels: the fp32 master copy and the ms slot of a slice live on its
//       owner, and ga3c_arena_download collects the owners' slices when the host asks for the weights.  dense_fwd of the next
//       step waits for every rank's "slice landed" flag before it reads the shadow (DpGate, dense_tc.cu).
//   the small tensors (conv11 / conv12 / dense1 bias / heads, 58 KB) are final after the conv backward.  dp_small_kernel
//       (elementwise.cu) sums this rank's per-CTA slabs and PUSHES the sums into every rank's receive buffer with the
//       step number packed into every 8 bytes ({value, flag} pairs, the "LL" wire format: an 8-byte store lands whole,
//       so data that carries the expected flag is valid -- no fence, no separate flag, one NVLink one-way trip).  Every
//       rank adds the contributions in rank order and applies the identical update locally; nothing is written back.
// Flags are monotonically increasing step numbers PUSHED into every rank's comm block; a waiter only polls its own HBM.
#pragma once
#include "common.cuh"

namespace ga3c {

constexpr int DP_WORLD_MAX = 8;
// comm block layout (bytes from comm_offset)
constexpr int DPC_CTR_BIG = 1032;     // u32 block counter of this rank's own dense1/w exchange grid
constexpr int DPC_ERR = 1040;         // u32: set when a wait gave up (a rank died or fell out of step): ga3c_dp_error
constexpr int DPC_BIGREADY = 2048;    // [8] x 64 B   dense_bwd of the step complete on rank r
constexpr int DPC_BIGDONE = 2560;     // [8] x 64 B   rank r's dense1/w slice stored everywhere
constexpr int DP_COMM_BYTES = DPC_BIGDONE + DP_WORLD_MAX * 64;
constexpr int DP_MAX_CB = 256;        // column blocks of the small tensors (blocks of dp_small_kernel)

__device__ __forceinline__ uint64_t dp_ld_flag(const void* p) {
  uint64_t v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void dp_st_flag(void* p, uint64_t v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;\n" ::"l"(p), "l"(v) : "memory");
}
// Every cross-rank wait is bounded (2^25 polls of local HBM, some tens of seconds: far beyond any legitimate skew between ranks
// that train in lock step, short enough for a job to fail instead of hanging): a rank that died or was called a different
// number of times must not hold the others' GPUs for ever.  On expiry the waiter raises the error word of its own comm block and carries on;
// the host sees it through ga3c_dp_error (results of that step are garbage).
constexpr unsigned int DP_SPIN_LIMIT = 1u << 25;
// error bits: 4 dense_bwd-done flags of the dense1/w exchange, 8 small-tensor LL data, 16 dense1/w slices landed
__device__ __forceinline__ void dp_wait_flag(const void* p, unsigned long long want, void* err, unsigned int bit) {
  for (unsigned int i = 0; dp_ld_flag(p) < want; ++i)
    if (i > DP_SPIN_LIMIT) { atomicOr(static_cast<unsigned int*>(err), bit); break; }
}
// the same wait, ending in an ACQUIRE load: what the waiter reads afterwards (the peer's gradients) is ordered behind the flag
// without a fence.sys -- which would also wait for every remote store this thread block has in flight (~2.7 us measured)
__device__ __forceinline__ void dp_wait_flag_acquire(const void* p, unsigned long long want, void* err, unsigned int bit) {
  dp_wait_flag(p, want, err, bit);
  uint64_t v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
  (void)v;
}
// LL wire format: a float4 travels as two 16-byte stores {x, flag, y, flag} {z, flag, w, flag}
__device__ __forceinline__ void dp_ll_store(void* dst, const float4& v, uint32_t flag) {
  asm volatile("st.relaxed.sys.global.v4.b32 [%0], {%1,%2,%3,%4};\n" ::"l"(dst), "r"(__float_as_uint(v.x)), "r"(flag),
               "r"(__float_as_uint(v.y)), "r"(flag) : "memory");
  asm volatile("st.relaxed.sys.global.v4.b32 [%0], {%1,%2,%3,%4};\n" ::"l"(static_cast<uint8_t*>(dst) + 16),
               "r"(__float_as_uint(v.z)), "r"(flag), "r"(__float_as_uint(v.w)), "r"(flag) : "memory");
}
__device__ __forceinline__ float4 dp_ll_load(const void* src, uint32_t flag, void* err) {   // spins until all four flags match
  uint32_t a0, f0, a1, f1, a2, f2, a3, f3;
  unsigned int spins = 0;
  do {
    if (++spins > DP_SPIN_LIMIT) { atomicOr(static_cast<unsigned int*>(err), 8u); break; }
    asm volatile("ld.relaxed.sys.global.v4.b32 {%0,%1,%2,%3}, [%4];\n" : "=r"(a0), "=r"(f0), "=r"(a1), "=r"(f1) : "l"(src) : "memory");
    asm volatile("ld.relaxed.sys.global.v4.b32 {%0,%1,%2,%3}, [%4];\n" : "=r"(a2), "=r"(f2), "=r"(a3), "=r"(f3)
                 : "l"(static_cast<const uint8_t*>(src) + 16) : "memory");
  } while (f0 != flag || f1 != flag || f2 != flag || f3 != flag);
  return make_float4(__uint_as_float(a0), __uint_as_float(a1), __uint_as_float(a2), __uint_as_float(a3));
}
__device__ __forceinline__ float4 dp_ld_f4(const float4* p) {      // L2 (the owner's) is the coherence point: skip L1
  float4 r;
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];\n" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
  return r;
}

// ---- RMSProp, TensorFlow semantics (tf.train.RMSPropOptimizer, NetworkVP_discrate.py:101-105) ----
//   ms  <- rho*ms + (1-rho)*g^2 ; mom <- mu*mom + lr*g/sqrt(ms + eps) ; w <- w - mom       [TF-SEMANTICS]
// The one element update of every optimizer kernel (elementwise.cu) and of the dense1/w exchange (dp_big_loop).  With mu == 0
// (Config.RMSPROP_MOMENTUM) mom enters as zero and leaves as the step.
__device__ __forceinline__ void rms_update(const float4& g, float4& w, float4& ms, float4& mo, float lr, float decay, float momentum,
                                           float eps) {
  const float one_m_rho = 1.f - decay;
  auto one = [&](float gc, float& wc, float& msc, float& moc) {
    msc = decay * msc + one_m_rho * gc * gc;
    moc = momentum * moc + lr * gc / sqrtf(msc + eps);
    wc -= moc;
  };
  one(g.x, w.x, ms.x, mo.x); one(g.y, w.y, ms.y, mo.y); one(g.z, w.z, ms.z, mo.z); one(g.w, w.w, ms.w, mo.w);
}

struct DpBigArgs {
  uint8_t* peer[DP_WORLD_MAX];      // slab bases: [params | grads | ms | mom | shadow | LL receive buffers | comm]
  int rank, world;
  unsigned long long step;
  long long arena_bytes, shadow_off, comm_offset;
  long long w1_offset, w1_count;    // dense1/w inside the arena, in floats (multiples of 4)
  float lr, decay, momentum, eps;
};

// reduce-scatter + RMSProp + all-gather over float4 indices [lo, hi) of dense1/w, strided over the exchange CTAs.  The loop is
// bound by NVLink round trips, so what matters is loads in flight: W * U remote / local gradient loads per thread and trip
// (W = world size as a compile-time constant, 0 = any world size with predicated loads).
template <int W, int U>
__device__ __forceinline__ void dp_big_loop(const DpBigArgs& d, long long lo, long long hi, long long first, long long stride) {
  const long long base4 = d.w1_offset >> 2;
  const float lr = d.lr, decay = d.decay, momentum = d.momentum, eps = d.eps;     // read ahead of the loop: 4 B less spill
  float4* w_own = reinterpret_cast<float4*>(d.peer[d.rank]) + base4;
  float4* g_own = reinterpret_cast<float4*>(d.peer[d.rank] + d.arena_bytes) + base4;
  float4* ms_own = reinterpret_cast<float4*>(d.peer[d.rank] + 2 * d.arena_bytes) + base4;
  float4* mom_own = reinterpret_cast<float4*>(d.peer[d.rank] + 3 * d.arena_bytes) + base4;
  const bool has_mom = d.momentum != 0.f;
  constexpr int NW = W > 0 ? W : DP_WORLD_MAX;
  for (long long i0 = lo + first; i0 < hi; i0 += U * stride) {
    float4 q[U][NW], w[U], ms[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
#pragma unroll
      for (int r = 0; r < NW; ++r)
        q[u][r] = (i < hi && (W > 0 || r < d.world))
                      ? dp_ld_f4(reinterpret_cast<const float4*>(d.peer[r] + d.arena_bytes) + base4 + i)
                      : make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < hi) { w[u] = w_own[i]; ms[u] = ms_own[i]; }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
      if (i >= hi) continue;
      float4 g = q[u][0];
#pragma unroll
      for (int r = 1; r < NW; ++r) { g.x += q[u][r].x; g.y += q[u][r].y; g.z += q[u][r].z; g.w += q[u][r].w; }   // rank order
      float4 mo = has_mom ? mom_own[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      rms_update(g, w[u], ms[u], mo, lr, decay, momentum, eps);
      ms_own[i] = ms[u];
      if (has_mom) mom_own[i] = mo;
      g_own[i] = g;                    // the reduced gradient of the owned slice (introspection); only this rank reads the slice
      const uint2 sh = make_uint2(pack_bf16(w[u].x, w[u].y), pack_bf16(w[u].z, w[u].w));
      w_own[i] = w[u];                 // fp32 master: owner only (collected by ga3c_arena_download)
#pragma unroll
      for (int r = 0; r < NW; ++r)
        if (W > 0 || r < d.world) reinterpret_cast<uint2*>(d.peer[r] + d.shadow_off)[i] = sh;
    }
  }
}

// The whole exchange on a GROUP of `nthreads` threads (thread t of the group, named barrier `bar_id`).  `cta` / `n_cta`: index and
// number of the groups that share the work; last_smem: one int that only thread 0 uses.  Group 0 publishes "dense_bwd done on
// this rank" (the dense1/w gradient is final by stream order), every group waits for every rank's, takes its share of the loop,
// and the last group to finish pushes the rank's "slice landed everywhere" flag.  Waits with acquire loads, no fence between the
// two flag hops.
__device__ __forceinline__ void dp_big_group(const DpBigArgs& d, int t, int nthreads, int cta, int n_cta, int bar_id, int* last_smem) {
  uint8_t* my_comm = d.peer[d.rank] + d.comm_offset;
  const long long n4 = d.w1_count >> 2;
  const long long per = (n4 + d.world - 1) / d.world;
  const long long lo = per * d.rank, hi = lo + per < n4 ? lo + per : n4;
  const long long stride = (long long)n_cta * nthreads, first = (long long)cta * nthreads + t;
  if (cta == 0 && t < d.world) {
    __threadfence_system();
    dp_st_flag(d.peer[t] + d.comm_offset + DPC_BIGREADY + 64 * d.rank, d.step);
  }
  if (t < d.world) dp_wait_flag_acquire(my_comm + DPC_BIGREADY + 64 * t, d.step, my_comm + DPC_ERR, 4u);
  asm volatile("bar.sync %0, %1;\n" ::"r"(bar_id), "r"(nthreads) : "memory");
  if (d.world == 2) dp_big_loop<2, 4>(d, lo, hi, first, stride);
  else if (d.world == 4) dp_big_loop<4, 2>(d, lo, hi, first, stride);
  else if (d.world == 8) dp_big_loop<8, 1>(d, lo, hi, first, stride);
  else dp_big_loop<0, 1>(d, lo, hi, first, stride);
  asm volatile("bar.sync %0, %1;\n" ::"r"(bar_id), "r"(nthreads) : "memory");
  if (t == 0) {
    __threadfence_system();            // cumulative over the group's peer stores (observed through the barrier)
    unsigned int* ctr = reinterpret_cast<unsigned int*>(my_comm + DPC_CTR_BIG);
    *last_smem = atomicAdd(ctr, 1u) == (unsigned int)n_cta - 1;
    if (*last_smem) {
      *ctr = 0;
      __threadfence_system();
      for (int r = 0; r < d.world; ++r) dp_st_flag(d.peer[r] + d.comm_offset + DPC_BIGDONE + 64 * d.rank, d.step);
    }
  }
}

}  // namespace ga3c
