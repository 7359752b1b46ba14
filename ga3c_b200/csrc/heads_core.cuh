// The fused value / policy heads of the conv net, with the A3C loss and its backward of a3c_loss.cuh, as device functions, run by
// heads_kernel (heads.cu: behind the split-K dense1 GEMM, summing its partial tiles from L2).  All fp32.
#pragma once
#include "common.cuh"
#include "kernels.h"
#include "a3c_loss.cuh"

namespace ga3c {

constexpr int HD_THREADS = 256, HD_CHUNK = 8;

template <int A>
struct HeadsSmem {
  alignas(16) float wt[A + 1][FC];                 // wt[k][j]: k < A -> Wp[j][k]; k == A -> Wv[j]
  float dzs[HD_CHUNK][A + 1];                      // (dz_0..dz_{A-1}, dv) per sample of the chunk
  alignas(16) uint16_t dd1s[HD_CHUNK][FC];
  alignas(16) float d1s[HD_CHUNK][FC];             // dense1 output of the chunk (post bias + ReLU)
  alignas(16) float b1s[FC];
  float bias_s[A + 1];
  float loss_s[HD_THREADS / 32][3];
};

// per-thread accumulators that live across the chunks of a CTA
template <int A>
struct HeadsAcc {
  float acc[A + 1];        // thread j: dWp[j][0..A-1], dWv[j]
  float acc_b1, acc_bh;    // thread j: db1[j]; thread k <= A: dbp[k] / dbv
  A3cSums loss;            // lane 0 of each warp: loss partial sums
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int k = 0; k <= A; ++k) acc[k] = 0.f;
    acc_b1 = acc_bh = 0.f;
    loss = A3cSums{};
  }
};

template <int A>
__device__ __forceinline__ void heads_load_weights(const HeadsArgs& p, HeadsSmem<A>& hs, int tid, int nthreads) {
  constexpr int A1 = A + 1;
  for (int i = tid; i < A1 * FC; i += nthreads) {
    const int k = i / FC, jx = i - k * FC;
    hs.wt[k][jx] = (k < A) ? p.wp[jx * A + k] : p.wv[jx];
  }
  if (tid < A1) hs.bias_s[tid] = (tid < A) ? p.bp[tid] : p.bv[0];
  for (int i = tid; i < FC; i += nthreads) hs.b1s[i] = p.b1[i];
}

// One warp, one sample b (slot sl of the chunk): fa / fb are this lane's 8 dense1 outputs (features 4 lane .. and 128 + 4 lane ..,
// bias added, ReLU applied).  Writes d1, p, v; when training also dd1 (global + chunk copy), the chunk's (dz, dv) and d1 rows,
// and adds the sample's loss terms to lane 0's sums.
template <int A>
__device__ __forceinline__ void heads_sample(const HeadsArgs& p, HeadsSmem<A>& hs, HeadsAcc<A>& ac, int b, int sl, int lane,
                                             const float4& fa, const float4& fb, float inv_mix) {
  constexpr int A1 = A + 1;
  *reinterpret_cast<float4*>(p.d1 + (size_t)b * FC + 4 * lane) = fa;
  *reinterpret_cast<float4*>(p.d1 + (size_t)b * FC + 128 + 4 * lane) = fb;
  if (p.train) {
    *reinterpret_cast<float4*>(&hs.d1s[sl][4 * lane]) = fa;
    *reinterpret_cast<float4*>(&hs.d1s[sl][128 + 4 * lane]) = fb;
  }
  float z[A1];
#pragma unroll
  for (int k = 0; k < A1; ++k) {
    const float4 wa = *reinterpret_cast<const float4*>(&hs.wt[k][4 * lane]);
    const float4 wb = *reinterpret_cast<const float4*>(&hs.wt[k][128 + 4 * lane]);
    float s = fa.x * wa.x;
    s = fmaf(fa.y, wa.y, s); s = fmaf(fa.z, wa.z, s); s = fmaf(fa.w, wa.w, s);
    s = fmaf(fb.x, wb.x, s); s = fmaf(fb.y, wb.y, s); s = fmaf(fb.z, wb.z, s); s = fmaf(fb.w, wb.w, s);
    z[k] = warp_sum(s) + hs.bias_s[k];
  }
  const float v = z[A];
  const LossArgs la = p.la;
  float dz[A];
  const float* arow = p.a + (size_t)b * A;
  if (p.p_out != nullptr && lane == 0) p.v_out[b] = v;
  const float yr = p.train ? p.yr[b] : 0.f;
  const A3cTerms t = softmax_policy_row(
      z, A, v, yr, la, inv_mix, p.train, [&](int k) { return arow[k]; },
      [&](int k, float pk) { if (p.p_out != nullptr && lane == k) p.p_out[(size_t)b * A + k] = pk; },
      [&](int k, float dzk) { dz[k] = dzk; });
  if (p.train) {
    const float dv = t.dv;
    if (lane == 0) {
      t.add_to(p.la.beta, ac.loss);
#pragma unroll
      for (int k = 0; k < A; ++k) hs.dzs[sl][k] = dz[k];
      hs.dzs[sl][A] = dv;
    }
    // dd1[j] = relu'(d1[j]) * (sum_k dz_k Wp[j][k] + dv Wv[j]) for this lane's 8 features
    float da[4], db[4];
    {
      const float4 wa = *reinterpret_cast<const float4*>(&hs.wt[A][4 * lane]);
      const float4 wb = *reinterpret_cast<const float4*>(&hs.wt[A][128 + 4 * lane]);
      da[0] = dv * wa.x; da[1] = dv * wa.y; da[2] = dv * wa.z; da[3] = dv * wa.w;
      db[0] = dv * wb.x; db[1] = dv * wb.y; db[2] = dv * wb.z; db[3] = dv * wb.w;
    }
#pragma unroll
    for (int k = 0; k < A; ++k) {
      const float4 wa = *reinterpret_cast<const float4*>(&hs.wt[k][4 * lane]);
      const float4 wb = *reinterpret_cast<const float4*>(&hs.wt[k][128 + 4 * lane]);
      da[0] = fmaf(dz[k], wa.x, da[0]); da[1] = fmaf(dz[k], wa.y, da[1]);
      da[2] = fmaf(dz[k], wa.z, da[2]); da[3] = fmaf(dz[k], wa.w, da[3]);
      db[0] = fmaf(dz[k], wb.x, db[0]); db[1] = fmaf(dz[k], wb.y, db[1]);
      db[2] = fmaf(dz[k], wb.z, db[2]); db[3] = fmaf(dz[k], wb.w, db[3]);
    }
    const uint2 qa = make_uint2(pack_bf16(fa.x > 0.f ? da[0] : 0.f, fa.y > 0.f ? da[1] : 0.f),
                                pack_bf16(fa.z > 0.f ? da[2] : 0.f, fa.w > 0.f ? da[3] : 0.f));
    const uint2 qb = make_uint2(pack_bf16(fb.x > 0.f ? db[0] : 0.f, fb.y > 0.f ? db[1] : 0.f),
                                pack_bf16(fb.z > 0.f ? db[2] : 0.f, fb.w > 0.f ? db[3] : 0.f));
    *reinterpret_cast<uint2*>(&hs.dd1s[sl][4 * lane]) = qa;
    *reinterpret_cast<uint2*>(&hs.dd1s[sl][128 + 4 * lane]) = qb;
    *reinterpret_cast<uint2*>(p.dd1 + (size_t)b * FC + 4 * lane) = qa;
    *reinterpret_cast<uint2*>(p.dd1 + (size_t)b * FC + 128 + 4 * lane) = qb;
  }

}

// a slot of the chunk beyond the batch: contributes nothing to phase 2
template <int A>
__device__ __forceinline__ void heads_pad_sample(HeadsSmem<A>& hs, int sl, int lane) {
  if (lane < A + 1) hs.dzs[sl][lane] = 0.f;
  *reinterpret_cast<uint2*>(&hs.dd1s[sl][4 * lane]) = make_uint2(0, 0);
  *reinterpret_cast<uint2*>(&hs.dd1s[sl][128 + 4 * lane]) = make_uint2(0, 0);
}

// phase 2 (after a block barrier): thread jx (< 256) accumulates dWp[jx][:], dWv[jx], db1[jx] over the chunk that starts at row b0
template <int A>
__device__ __forceinline__ void heads_accumulate(const HeadsArgs& p, HeadsSmem<A>& hs, HeadsAcc<A>& ac, int b0, int jx) {
  constexpr int A1 = A + 1;
#pragma unroll 4
  for (int sl = 0; sl < HD_CHUNK; ++sl) {
    const float dval = (b0 + sl < p.batch) ? hs.d1s[sl][jx] : 0.f;
#pragma unroll
    for (int k = 0; k < A1; ++k) ac.acc[k] = fmaf(dval, hs.dzs[sl][k], ac.acc[k]);
    ac.acc_b1 += __uint_as_float((uint32_t)hs.dd1s[sl][jx] << 16);
  }
  if (jx < A1) {
#pragma unroll 4
    for (int sl = 0; sl < HD_CHUNK; ++sl) ac.acc_bh += hs.dzs[sl][jx];
  }
}

// end of the CTA: partial sums into slab `slab_index` of the gradient-partial workspace (thread jx < 256; contains block barriers)
template <int A>
__device__ __forceinline__ void heads_store_slab(const HeadsArgs& p, HeadsSmem<A>& hs, const HeadsAcc<A>& ac, int slab_index, int jx,
                                                 int warp, int lane) {
  const int64_t slab = (int64_t)slab_index * p.gp_stride;
#pragma unroll
  for (int k = 0; k < A; ++k) p.g_wp[slab + jx * A + k] = ac.acc[k];
  p.g_wv[slab + jx] = ac.acc[A];
  p.g_b1[slab + jx] = ac.acc_b1;
  if (jx < A) p.g_bp[slab + jx] = ac.acc_bh;
  if (jx == A) p.g_bv[slab] = ac.acc_bh;
  if (lane == 0) { hs.loss_s[warp][0] = ac.loss.l1; hs.loss_s[warp][1] = ac.loss.l2; hs.loss_s[warp][2] = ac.loss.lv; }
  __syncthreads();
  if (jx < 4) {
    float t = 0.f;
    if (jx < 3)
#pragma unroll
      for (int w = 0; w < HD_THREADS / 32; ++w) t += hs.loss_s[w][jx];
    p.loss[slab + jx] = t;
  }
}

}  // namespace ga3c
