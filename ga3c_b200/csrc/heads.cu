// Value / policy heads, softmax, A3C loss and its backward, fused.  All fp32.
//
// Reference graph (NetworkVP_discrate.py:60-85, :100; SURVEY Appendix A.3/A.4):
//   v = d1.Wv + bv ; z = d1.Wp + bp ; s = softmax(z) ; p = (s + MIN_POLICY) / (1 + MIN_POLICY*A)
//   cost_p_1 = log(max(sum(p*a), eps)) * (R - stop_gradient(v)) ; cost_p_2 = -beta * sum(log(max(p, eps)) * p)
//   cost_v = 0.5 * (R - v)^2 ; every batch reduction is a SUM.
// The kernel is also the tail of dense1 (NetworkDNav.py:90): it sums the split-K partial tiles the
// tcgen05 GEMM left in d1_part (fixed order => deterministic), adds the bias and applies the ReLU.
// Phase 1: one warp per sample, warp-shuffle reductions for the A+1 dot products, then the whole
//          softmax / loss / dlogits chain in registers; writes d1, p, v, dd1 (bf16) and stages (dz, dv).
// Phase 2: one thread per dense1 feature accumulates dWp[j,:], dWv[j], db1[j] over the chunk.
// Gradient / loss accumulators live in registers across chunks; each CTA stores its partial sums into its own slab
// of the gradient-partial workspace (summed in a fixed order by grad_reduce: no atomics, bit-reproducible).
#include "common.cuh"
#include "kernels.h"
#include "heads_core.cuh"

namespace ga3c {

template <int A>
__global__ void __launch_bounds__(HD_THREADS) heads_kernel(HeadsArgs p) {
  __shared__ HeadsSmem<A> hs;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // The head weights are written by the optimizer launch of the previous step.  A prologue may run while a kernel two or more
  // launches back is still executing (only code after the wait is ordered transitively, common.cuh), so reading them before
  // the dependency wait is safe only when something in between cannot be resident next to that optimizer launch: p.preload
  // (batch >= num_sms: the conv forward in front of this kernel fills every SM, see the preload rule in elementwise.cu).  Otherwise
  // they are read after the wait.
  if (p.preload) heads_load_weights<A>(p, hs, tid, HD_THREADS);
  griddep_launch();
  griddep_wait(K_HEADS);               // d1_part comes from the dense1 GEMM that precedes this kernel
  if (!p.preload) heads_load_weights<A>(p, hs, tid, HD_THREADS);
  __syncthreads();

  HeadsAcc<A> ac;
  ac.clear();
  const float inv_mix = 1.f / (1.f + p.min_policy * (float)A);

  const int n_chunks = (p.batch + HD_CHUNK - 1) / HD_CHUNK;
  for (int c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    // ---------------- phase 1: warp per sample ----------------
    {
      const int sl = warp;
      const int b = c * HD_CHUNK + sl;
      if (b < p.batch) {
        // dense1 tail: sum the split-K partials in split order, + bias, ReLU
        float4 fa = *reinterpret_cast<const float4*>(&hs.b1s[4 * lane]);
        float4 fb = *reinterpret_cast<const float4*>(&hs.b1s[128 + 4 * lane]);
        {
          float4 sa = make_float4(0.f, 0.f, 0.f, 0.f), sb = sa;
          // the partial tiles sit in L2; every load of a pass is in flight before the first add (the training batch's 9 splits
          // in one pass: one L2 round trip instead of three), the adds stay in split order
#pragma unroll 9
          for (int sp = 0; sp < p.n_split; ++sp) {
            const float* src = p.d1_part + ((size_t)sp * p.batch + b) * FC;
            const float4 qa = *reinterpret_cast<const float4*>(src + 4 * lane);
            const float4 qb = *reinterpret_cast<const float4*>(src + 128 + 4 * lane);
            sa.x += qa.x; sa.y += qa.y; sa.z += qa.z; sa.w += qa.w;
            sb.x += qb.x; sb.y += qb.y; sb.z += qb.z; sb.w += qb.w;
          }
          fa.x = fmaxf(fa.x + sa.x, 0.f); fa.y = fmaxf(fa.y + sa.y, 0.f); fa.z = fmaxf(fa.z + sa.z, 0.f); fa.w = fmaxf(fa.w + sa.w, 0.f);
          fb.x = fmaxf(fb.x + sb.x, 0.f); fb.y = fmaxf(fb.y + sb.y, 0.f); fb.z = fmaxf(fb.z + sb.z, 0.f); fb.w = fmaxf(fb.w + sb.w, 0.f);
        }
        heads_sample<A>(p, hs, ac, b, sl, lane, fa, fb, inv_mix);
      } else if (p.train) {
        heads_pad_sample<A>(hs, sl, lane);
      }
    }
    if (!p.train) continue;
    __syncthreads();
    // ---------------- phase 2: thread per feature ----------------
    heads_accumulate<A>(p, hs, ac, c * HD_CHUNK, tid);
    __syncthreads();
  }

  if (!p.train) { trace_mark(K_HEADS, 2); return; }
  heads_store_slab<A>(p, hs, ac, blockIdx.x, tid, warp, lane);
  trace_mark(K_HEADS, 2);
}

GA3C_TRACE_ATTACH(trace_attach_heads)

template <int A>
static int launch_heads_t(const HeadsArgs& args, int grid, cudaStream_t stream) {
  return launch_pdl(heads_kernel<A>, dim3(grid), dim3(HD_THREADS), 0, stream, args);
}

int heads_grid(int batch, int num_sms) { return min((batch + HD_CHUNK - 1) / HD_CHUNK, 2 * num_sms); }

int launch_heads(const HeadsArgs& args, int num_sms, cudaStream_t stream) {
  const int grid = heads_grid(args.batch, num_sms);
  switch (args.num_actions) {
#define GA3C_CASE(N) case N: return launch_heads_t<N>(args, grid, stream);
    GA3C_CASE(1) GA3C_CASE(2) GA3C_CASE(3) GA3C_CASE(4) GA3C_CASE(5) GA3C_CASE(6) GA3C_CASE(7) GA3C_CASE(8)
    GA3C_CASE(9) GA3C_CASE(10) GA3C_CASE(11) GA3C_CASE(12) GA3C_CASE(13) GA3C_CASE(14) GA3C_CASE(15)
    GA3C_CASE(16) GA3C_CASE(17) GA3C_CASE(18)
#undef GA3C_CASE
    default: return (int)cudaErrorInvalidValue;
  }
}

}  // namespace ga3c
