// The A3C policy / value loss of one batch row and its gradient w.r.t. the head logits, for every kernel that computes it: the conv
// heads (heads_core.cuh), the MLP tile kernel (mlp.cu) and the MLP streaming heads (mlp_stream.cu).  Register-only: the callers
// load the logits, hand in the action row and R, and store p, the logit gradients and the loss sums.  All fp32.
//
// Reference graphs (every batch reduction is a SUM):
//   value head (all networks):  cost_v = 0.5 (R - v)^2
//   softmax head (NetworkVP_discrate.py:60-85, :100; SURVEY A.3 / A.4):
//     s = softmax(z);  p = (s + MIN_POLICY) / (1 + MIN_POLICY A)
//     cost_p_1 = log(max(sum(p a), eps)) (R - stop_gradient(v));  cost_p_2 = -beta sum(log(max(p, eps)) p)
//     Config.USE_LOG_SOFTMAX (NetworkVP_discrate.py:64-71): p = s, lsm = z - max - log(sum exp(z - max));
//     cost_p_1 = sum(lsm a) (R - stop_gradient(v));  cost_p_2 = -beta sum(lsm s)
//   fork NetworkVP angle head (NetworkVP.py:175-192, :95-101), per action:
//     p = atan2(sigmoid(out_y) - 0.5, sigmoid(out_x) - 0.5) / pi;  softmax_p = log_softmax_p = p
//     cost_p_1 = sum(p a) (R - stop_gradient(v));  cost_p_2 = -beta sum(p^2)
//   Config.DUAL_RMSPROP (LossArgs::part): pass 1 takes the gradient of cost_p alone, which does not reach the value head; pass 2
//   of cost_v alone, which does not reach the policy head.
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace ga3c {

constexpr float PI_F = 3.14159265358979323846f;

// running sums of (cost_p_1, cost_p_2, cost_v) over the rows a thread owns
struct A3cSums {
  float l1 = 0.f, l2 = 0.f, lv = 0.f;
};

// The loss terms of one row.  add_to() forms the costs where the caller adds them to its sums, so that a product and its sum
// compile to one fused multiply-add whatever branch the caller adds in.
struct A3cTerms {
  float dv;                   // d cost_all / dv (DUAL_RMSPROP mask applied)
  float p1, p1_adv;           // cost_p_1 = p1 p1_adv (softmax head: cost_p_1, rounded in its own branch, and 1)
  float ent;                  // cost_p_2 = -beta ent
  float yr, v;                // cost_v = 0.5 (R - v)^2
  __device__ __forceinline__ void add_to(float beta, A3cSums& s) const {
    s.l1 += p1 * p1_adv;
    s.l2 += -beta * ent;
    s.lv += 0.5f * (yr - v) * (yr - v);
  }
};

__device__ __forceinline__ float policy_inv_mix(const LossArgs& la, int A) { return 1.f / (1.f + la.min_policy * (float)A); }

// dv = d cost_all / dv: zero in DUAL_RMSPROP pass 1
__device__ __forceinline__ float value_grad(float v, float yr, const LossArgs& la) { return la.part == 1 ? 0.f : v - yr; }

// Softmax head of one row (NetworkVP_discrate.py:60-85): the A policy logits z[0..A-1], the value v and, when `train`, R = yr
// and the action row a(k).  Hands p_k to put_p(k, p_k) and, when training, d cost_all / dz_k (DUAL_RMSPROP mask applied) to
// put_dz(k, dz_k), and returns the row's terms (meaningful when training).  put_dz(k, .) may overwrite z[k]: the last sweep reads
// only z[k] before it.  s_k = softmax(z)_k and the terms built on it are recomputed where they are used instead of held in arrays:
// a compile-time A unrolls every loop and the compiler merges the copies; a runtime A keeps the loops rolled and needs no local
// arrays.  inv_mix = policy_inv_mix(la, A).
template <class Act, class PutP, class PutDz>
__device__ __forceinline__ A3cTerms softmax_policy_row(const float* z, int A, float v, float yr, const LossArgs& la, float inv_mix,
                                                       bool train, Act a, PutP put_p, PutDz put_dz) {
  float mx = z[0];
#pragma unroll
  for (int k = 1; k < A; ++k) mx = fmaxf(mx, z[k]);
  float den = 0.f;
#pragma unroll
  for (int k = 0; k < A; ++k) den += expf(z[k] - mx);
  const float inv_den = 1.f / den;
#pragma unroll
  for (int k = 0; k < A; ++k) {
    const float sm = expf(z[k] - mx) * inv_den;
    put_p(k, la.log_softmax ? sm : (sm + la.min_policy) * inv_mix);
  }
  if (!train) return A3cTerms{};
  float sel = 0.f;
#pragma unroll
  for (int k = 0; k < A; ++k) {
    const float sm = expf(z[k] - mx) * inv_den;
    sel = fmaf(la.log_softmax ? sm : (sm + la.min_policy) * inv_mix, a(k), sel);
  }
  const float adv = yr - v;                         // stop_gradient(v) inside cost_p_1
  float ent = 0.f, c1;
  if (la.log_softmax) {
    // p = s, lsm_k = z_k - max - log(den);  dz_k = -adv (a_k - s_k sum(a)) + beta s_k (lsm_k - sum(lsm s))
    const float lden = logf(den);
    float sa = 0.f, sla = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) {
      const float lsm = (z[k] - mx) - lden, ak = a(k);
      ent = fmaf(lsm, expf(z[k] - mx) * inv_den, ent);
      sa += ak;
      sla = fmaf(lsm, ak, sla);
    }
#pragma unroll
    for (int k = 0; k < A; ++k) {
      const float sm = expf(z[k] - mx) * inv_den, lsm = (z[k] - mx) - lden;
      put_dz(k, la.part == 2 ? 0.f : -adv * (a(k) - sm * sa) + la.beta * sm * (lsm - ent));
    }
    c1 = sla * adv;
  } else {
    // through the MIN_POLICY mix and the eps floors: g_k = d cost_all / dp_k, h_k = g_k / (1 + MIN_POLICY A),
    // dz_k = s_k (h_k - sum(s h)); two sweeps, sum(s h) first
    const float coef = (sel >= la.log_eps) ? __fdiv_rn(adv, sel) : 0.f;   // IEEE round-to-nearest, as `/` compiles
    float sh = 0.f;
#pragma unroll
    for (int k = 0; k < A; ++k) {
      const float sm = expf(z[k] - mx) * inv_den, p = (sm + la.min_policy) * inv_mix;
      const float lg = logf(fmaxf(p, la.log_eps));
      ent = fmaf(lg, p, ent);
      const float gk = -a(k) * coef + la.beta * (lg + (p >= la.log_eps ? 1.f : 0.f));
      sh = fmaf(sm, gk * inv_mix, sh);
    }
#pragma unroll
    for (int k = 0; k < A; ++k) {
      const float sm = expf(z[k] - mx) * inv_den, p = (sm + la.min_policy) * inv_mix;
      const float lg = logf(fmaxf(p, la.log_eps));
      const float gk = -a(k) * coef + la.beta * (lg + (p >= la.log_eps ? 1.f : 0.f));
      put_dz(k, la.part == 2 ? 0.f : sm * fmaf(gk, inv_mix, -sh));  // h_k - sum(s h) with one rounding
    }
    c1 = logf(fmaxf(sel, la.log_eps)) * adv;
  }
  return A3cTerms{value_grad(v, yr, la), c1, 1.f, ent, yr, v};
}

// Fork angle head, one action: the logits zx (out_x) and zy (out_y) of the action, its entry a of the action row.  Returns p and
// the two logit gradients, and adds p a to sel and p^2 to sq (fork_policy_terms turns them into cost_p_1 / cost_p_2).
struct ForkAction {
  float p, dzx, dzy;
};
__device__ __forceinline__ ForkAction fork_policy(float zx, float zy, float a, float v, float yr, const LossArgs& la, float& sel,
                                                  float& sq) {
  const float ox = sigmoid(zx), oy = sigmoid(zy);
  const float X = ox - 0.5f, Y = oy - 0.5f;
  ForkAction f;
  f.p = atan2f(Y, X) / PI_F;
  sel = fmaf(f.p, a, sel);
  sq = fmaf(f.p, f.p, sq);
  const float adv = yr - v;                         // stop_gradient(v) inside cost_p_1
  const float dp = -a * adv + 2.f * la.beta * f.p;
  const float inv = 1.f / (PI_F * (X * X + Y * Y));
  f.dzx = la.part == 2 ? 0.f : dp * (-Y * inv) * ox * (1.f - ox);
  f.dzy = la.part == 2 ? 0.f : dp * (X * inv) * oy * (1.f - oy);
  return f;
}
__device__ __forceinline__ A3cTerms fork_policy_terms(float sel, float sq, float v, float yr, const LossArgs& la) {
  return A3cTerms{value_grad(v, yr, la), sel, yr - v, sq, yr, v};
}

}  // namespace ga3c
