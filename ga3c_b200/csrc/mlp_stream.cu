// Streaming kernels for the narrow ends of the fork's low-dimensional NetworkVP in tensor-core mode (mlp_tc.cu; BASELINE configs[3]):
//   x[S <= 4] -> 4 -> 256 | 256 -> 256 -> 100 -> 64 on tcgen05 | heads (v, out_x, out_y), atan2, loss      (NetworkVP.py:79-105, :175-210)
// Between the GEMM launches the step used to call the fused tile kernel (mlp.cu) three times -- for a 3 -> 4 -> 256 front (a
// reduction of depth 4), a 64 x 3 head matrix and a 256 -> 4 data gradient.  Its 64-row tiles, weight-chunk ring and block barriers
// are built for 256-deep reductions: those three launches took 75 + 73 + 50 us of a 690 us step at B = 65,536 for work that is
// ~30 us of HBM time (profiles/r3e_mlp_launches_before.md).  Here each of them is a plain streaming pass: rows are independent,
// weights live in registers / shared memory, every HBM byte is touched once and coalesced.
//   mlp_front_fwd   act[0] = f0(x W0 + b0), act[1] = f1(act[0] W1 + b1)             thread = 4 columns of one row
//   mlp_heads       logits = h Wh + bh -> v, p = atan2(..)/pi, loss terms, dlogits, dz[last] = (dlogits Wh^T) f'(h)   warp = four rows
//   mlp_front_bwd   dz[0] = (dz[1] W1^T) f0'(act[0])                                warp = one row
// Loss terms: every warp adds the terms of its rows in row order, every block its warps in warp order into one row of loss_part;
// mlp_reduce adds the rows in a fixed order (bit-reproducible, as the tile kernel's per-tile sums are).
#include "common.cuh"
#include "kernels.h"
#include "mlp.cuh"
#include "a3c_loss.cuh"

namespace ga3c {

namespace {

constexpr int ST_THREADS = 256, ST_WARPS = ST_THREADS / 32;
__device__ __forceinline__ float act_(float z, int act) { return act == MLP_ACT_SIGMOID ? sigmoid(z) : z; }

// ---- front, forward ---------------------------------------------------------------------------------------------------------------
// 64 threads per row (N1 = 256: four columns each), 4 rows per block and iteration.  W1's four columns (x N0 <= 4 rows) and the
// biases stay in registers; W0 / b0 (<= 16 + 4 floats) in shared memory (every thread of a row reads the same words).
__global__ void __launch_bounds__(ST_THREADS) mlp_front_fwd_kernel(const MlpNet net, const float* __restrict__ w,
                                                                   const float* __restrict__ x, int batch, float* __restrict__ act0,
                                                                   float* __restrict__ act1) {
  __shared__ float w0s[4][4], b0s[4];
  const MlpLayerDesc L0 = net.L[0], L1 = net.L[1];
  const int S = L0.k, N0 = L0.n, N1 = L1.n;
  const int tpr = N1 >> 2;                                   // threads per row
  const int rpb = ST_THREADS / tpr;                          // rows per block and iteration
  const int tid = threadIdx.x, rl = tid / tpr, c0 = (tid - rl * tpr) * 4;
  griddep_launch();
  griddep_wait(K_MLP_FUSED);                                 // the weights come from the optimizer launch of the previous step
  if (tid < 16) w0s[tid >> 2][tid & 3] = ((tid >> 2) < S && (tid & 3) < N0) ? __ldg(w + L0.w_off + (tid >> 2) * N0 + (tid & 3)) : 0.f;
  if (tid < 4) b0s[tid] = tid < N0 ? __ldg(w + L0.b_off + tid) : 0.f;
  float w1[4][4], b1[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float4 v = (k < N0 && rl < rpb) ? __ldg(reinterpret_cast<const float4*>(w + L1.w_off + k * N1 + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
    w1[k][0] = v.x; w1[k][1] = v.y; w1[k][2] = v.z; w1[k][3] = v.w;
  }
  {
    const float4 v = rl < rpb ? __ldg(reinterpret_cast<const float4*>(w + L1.b_off + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
    b1[0] = v.x; b1[1] = v.y; b1[2] = v.z; b1[3] = v.w;
  }
  __syncthreads();
  if (rl >= rpb) return;
  for (int r = blockIdx.x * rpb + rl; r < batch; r += gridDim.x * rpb) {
    float xv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) xv[k] = k < S ? __ldg(x + (size_t)r * S + k) : 0.f;
    // every aligned quad of lanes belongs to one row (threads per row is a multiple of 4): lane q of the quad computes h0[q]
    // -- one sigmoid instead of four -- and the quad exchanges the four values
    float h0[4];
    {
      const int nq = tid & 3;
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) acc = fmaf(xv[k], w0s[k][nq], acc);
      const float mine = nq < N0 ? act_(acc + b0s[nq], L0.act) : 0.f;
#pragma unroll
      for (int n = 0; n < 4; ++n) h0[n] = __shfl_sync(0xffffffffu, mine, (tid & 28) + n);
    }
    if (c0 == 0) {
      if (N0 == 4) *reinterpret_cast<float4*>(act0 + (size_t)r * 4) = make_float4(h0[0], h0[1], h0[2], h0[3]);
      else
        for (int n = 0; n < N0; ++n) act0[(size_t)r * N0 + n] = h0[n];
    }
    float o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) acc = fmaf(h0[k], w1[k][e], acc);
      o[e] = act_(acc + b1[e], L1.act);
    }
    __stcs(reinterpret_cast<float4*>(act1 + (size_t)r * N1 + c0), make_float4(o[0], o[1], o[2], o[3]));
  }
  trace_mark(K_MLP_FUSED, 2);
}

// ---- heads, loss, dlogits, gradient w.r.t. the last hidden pre-activation ---------------------------------------------------------------
// One warp per group of HU = 4 rows.  hid <= 128: lane l holds h[l], h[l + 32], ... of each row; the three logits of a row are warp
// sums (every lane gets them).  The scalar head arithmetic of NetworkVP.py:175-192 (two sigmoids, atan2, the loss terms, dlogits:
// ~100 instructions) then runs ONCE per row -- lane l works on row l & 3 -- and the three dlogits of each row are handed to the
// whole warp by shuffles for the lanes' own columns of dz.  (Every lane doing every row's scalar part made the kernel
// instruction-bound: 60 % issue-active, 35 us at B = 65,536.)  A = 1 (n_out = 3).
template <bool TRAIN>
__global__ void __launch_bounds__(ST_THREADS) mlp_heads_kernel(const MlpNet net, const MlpStepArgs s, const float* __restrict__ h,
                                                                float* __restrict__ dz_out) {
  constexpr int HU = 4, KMAX = MLP_MAX_HID / 32;
  const int lane = threadIdx.x & 31, warp = blockIdx.x * ST_WARPS + (threadIdx.x >> 5), nwarps = gridDim.x * ST_WARPS;
  const int hid = net.hid, B = s.batch;
  const int last_act = net.L[net.n_layers - 1].act;
  griddep_launch();
  griddep_wait(K_MLP_FUSED);
  float wh[KMAX][3], bh[3];
#pragma unroll
  for (int i = 0; i < KMAX; ++i) {
    const int k = lane + 32 * i;
    wh[i][0] = k < hid ? __ldg(s.w + net.wv_off + k) : 0.f;
    wh[i][1] = k < hid ? __ldg(s.w + net.wp_off + k) : 0.f;
    wh[i][2] = k < hid ? __ldg(s.w + net.wy_off + k) : 0.f;
  }
  bh[0] = __ldg(s.w + net.bv_off); bh[1] = __ldg(s.w + net.bp_off); bh[2] = __ldg(s.w + net.by_off);
  const int my = lane & (HU - 1);                                  // the row of the group whose scalar part this lane computes
  A3cSums sums;                                                   // loss terms of the rows this lane owns (lanes 0 .. HU-1 count)
  for (int r0 = warp * HU; r0 < B; r0 += nwarps * HU) {
    float hv[HU][KMAX];
#pragma unroll
    for (int u = 0; u < HU; ++u)
#pragma unroll
      for (int i = 0; i < KMAX; ++i) {
        const int k = lane + 32 * i;
        hv[u][i] = (r0 + u < B && k < hid) ? __ldcs(h + (size_t)(r0 + u) * hid + k) : 0.f;
      }
    const int r = r0 + my;
    const bool valid = r < B;
    float yr = 0.f, av = 0.f;
    if (TRAIN && valid) { yr = __ldg(s.yr + r); av = __ldg(s.a + r); }
    float z0 = 0.f, z1 = 0.f, z2 = 0.f;                            // logits of row `my`
#pragma unroll
    for (int u = 0; u < HU; ++u) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
      for (int i = 0; i < KMAX; ++i) {
        a0 = fmaf(hv[u][i], wh[i][0], a0); a1 = fmaf(hv[u][i], wh[i][1], a1); a2 = fmaf(hv[u][i], wh[i][2], a2);
      }
      a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2);
      if (u == my) { z0 = a0 + bh[0]; z1 = a1 + bh[1]; z2 = a2 + bh[2]; }
    }
    const float v = z0;
    float sel = 0.f, sq = 0.f;
    const ForkAction f = fork_policy(z1, z2, av, v, yr, s.la, sel, sq);
    if (lane < HU && valid) {
      if (s.v_out != nullptr) s.v_out[r] = v;
      if (s.p_out != nullptr) s.p_out[r] = f.p;
    }
    if (TRAIN) {
      const A3cTerms t = fork_policy_terms(sel, sq, v, yr, s.la);
      const float d0 = t.dv, d1 = f.dzx, d2 = f.dzy;
      if (lane < HU && valid) {
        t.add_to(s.la.beta, sums);
        *reinterpret_cast<float4*>(s.dlogits + (size_t)r * net.n_out_ld) = make_float4(d0, d1, d2, 0.f);
      }
#pragma unroll
      for (int u = 0; u < HU; ++u) {
        const float e0 = __shfl_sync(0xffffffffu, d0, u), e1 = __shfl_sync(0xffffffffu, d1, u), e2 = __shfl_sync(0xffffffffu, d2, u);
        if (r0 + u < B) {
#pragma unroll
          for (int i = 0; i < KMAX; ++i) {
            const int k = lane + 32 * i;
            if (k < hid) {
              float d = fmaf(e0, wh[i][0], 0.f);
              d = fmaf(e1, wh[i][1], d);
              d = fmaf(e2, wh[i][2], d);
              if (last_act == MLP_ACT_SIGMOID) d *= hv[u][i] * (1.f - hv[u][i]);
              dz_out[(size_t)(r0 + u) * hid + k] = d;
            }
          }
        }
      }
    }
  }
  if (TRAIN) {                                                  // one row of loss_part per block: lanes 0 .. HU-1 of a warp in lane
    __shared__ float red[ST_WARPS][3];                          // order, then the warps in warp order
    float t1 = sums.l1, t2 = sums.l2, tv = sums.lv;
#pragma unroll
    for (int u = 1; u < HU; ++u) {
      t1 += __shfl_sync(0xffffffffu, sums.l1, u); t2 += __shfl_sync(0xffffffffu, sums.l2, u); tv += __shfl_sync(0xffffffffu, sums.lv, u);
    }
    if (lane == 0) { red[threadIdx.x >> 5][0] = t1; red[threadIdx.x >> 5][1] = t2; red[threadIdx.x >> 5][2] = tv; }
    __syncthreads();
    if (threadIdx.x < 4) {
      float t = 0.f;
      if (threadIdx.x < 3)
#pragma unroll
        for (int wq = 0; wq < ST_WARPS; ++wq) t += red[wq][threadIdx.x];
      s.loss_part[(size_t)blockIdx.x * 4 + threadIdx.x] = t;
    }
  }
  trace_mark(K_MLP_FUSED, 2);
}

// ---- front, data gradient ------------------------------------------------------------------------------------------------------------
// dz[0][r][k] = (sum_c dz[1][r][c] W1[k][c]) f0'(act[0][r][k]): one warp per row, lane l holds columns 4l .. 4l+3 and 128 + 4l .. of
// dz[1] (N1 <= 256) and the matching 4 x 8 weights; BU rows in flight per warp.
__global__ void __launch_bounds__(ST_THREADS) mlp_front_bwd_kernel(const MlpNet net, const float* __restrict__ w,
                                                                   const float* __restrict__ dz1, const float* __restrict__ act0,
                                                                   int batch, float* __restrict__ dz0) {
  constexpr int BU = 4;
  const MlpLayerDesc L0 = net.L[0], L1 = net.L[1];
  const int N0 = L0.n, N1 = L1.n;
  const int lane = threadIdx.x & 31, warp = blockIdx.x * ST_WARPS + (threadIdx.x >> 5), nwarps = gridDim.x * ST_WARPS;
  griddep_launch();
  griddep_wait(K_MLP_FUSED);
  float w1[4][8];
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int c = 128 * hh + 4 * lane;
      const float4 v = (k < N0 && c < N1) ? __ldg(reinterpret_cast<const float4*>(w + L1.w_off + k * N1 + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
      w1[k][4 * hh] = v.x; w1[k][4 * hh + 1] = v.y; w1[k][4 * hh + 2] = v.z; w1[k][4 * hh + 3] = v.w;
    }
  for (int r0 = warp * BU; r0 < batch; r0 += nwarps * BU) {
    float4 d[BU][2];
#pragma unroll
    for (int u = 0; u < BU; ++u)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int c = 128 * hh + 4 * lane;
        d[u][hh] = (r0 + u < batch && c < N1) ? __ldcs(reinterpret_cast<const float4*>(dz1 + (size_t)(r0 + u) * N1 + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
    for (int u = 0; u < BU; ++u) {
      const int r = r0 + u;
      if (r >= batch) break;                                     // warp-uniform
      float t[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float a = 0.f;
        a = fmaf(d[u][0].x, w1[k][0], a); a = fmaf(d[u][0].y, w1[k][1], a); a = fmaf(d[u][0].z, w1[k][2], a); a = fmaf(d[u][0].w, w1[k][3], a);
        a = fmaf(d[u][1].x, w1[k][4], a); a = fmaf(d[u][1].y, w1[k][5], a); a = fmaf(d[u][1].z, w1[k][6], a); a = fmaf(d[u][1].w, w1[k][7], a);
        t[k] = warp_sum(a);
      }
      if (lane < N0) {
        float g = lane == 0 ? t[0] : lane == 1 ? t[1] : lane == 2 ? t[2] : t[3];
        if (L0.act == MLP_ACT_SIGMOID) { const float o = __ldg(act0 + (size_t)r * N0 + lane); g *= o * (1.f - o); }
        dz0[(size_t)r * N0 + lane] = g;
      }
    }
  }
  trace_mark(K_MLP_FUSED, 2);
}

}  // namespace

GA3C_TRACE_ATTACH(trace_attach_mlp_stream)

// the pattern these kernels cover: the fork NetworkVP (one action) with the GEMM run starting at layer 2 and reaching the heads
bool mlp_stream_ok(const MlpNet& net, int tc_lo, int tc_hi) {
  if (net.kind != MLP_KIND_FORK_VP || net.num_actions != 1 || net.n_out != 3 || net.n_out_ld != 4) return false;
  if (tc_lo != 2 || tc_hi != net.n_layers || net.hid > MLP_MAX_HID) return false;
  const MlpLayerDesc &L0 = net.L[0], &L1 = net.L[1];
  // L1.n a multiple of 128: a warp of mlp_front_fwd never spans two rows (its quad shuffles run in warp-uniform code)
  return L0.k <= 4 && L0.n <= 4 && L1.k == L0.n && L1.n <= 256 && L1.n % 128 == 0 && ST_THREADS % (L1.n / 4) == 0 &&
         (L0.w_off & 3) == 0 && (L1.w_off & 3) == 0 && (L1.b_off & 3) == 0;
}

static int stream_grid(int batch, int rows_per_block, int num_sms) {
  const int want = (batch + rows_per_block - 1) / rows_per_block, cap = num_sms * 8;     // 8 blocks of 256 threads per SM
  return want < cap ? (want < 1 ? 1 : want) : cap;
}

int launch_mlp_front_fwd(const MlpNet& net, const MlpStepArgs& s, int num_sms, cudaStream_t stream) {
  const int rpb = ST_THREADS / (net.L[1].n / 4);
  return launch_pdl(mlp_front_fwd_kernel, dim3(stream_grid(s.batch, rpb * 4, num_sms)), dim3(ST_THREADS), 0, stream, net, s.w, s.x,
                    s.batch, s.act[0], s.act[1]);
}

// rows of loss_part the heads kernel writes (one per block); the grid depends on the batch alone
int mlp_heads_loss_rows(int batch, int num_sms) { return stream_grid(batch, ST_WARPS * 4 * 2, num_sms); }

int launch_mlp_heads(const MlpNet& net, const MlpStepArgs& s, int num_sms, cudaStream_t stream) {
  const int grid = stream_grid(s.batch, ST_WARPS * 4 * 2, num_sms);
  const float* h = s.act[net.n_layers - 1];
  if (s.train) return launch_pdl(mlp_heads_kernel<true>, dim3(grid), dim3(ST_THREADS), 0, stream, net, s, h, s.dz[net.n_layers - 1]);
  return launch_pdl(mlp_heads_kernel<false>, dim3(grid), dim3(ST_THREADS), 0, stream, net, s, h, (float*)nullptr);
}

int launch_mlp_front_bwd(const MlpNet& net, const MlpStepArgs& s, int num_sms, cudaStream_t stream) {
  return launch_pdl(mlp_front_bwd_kernel, dim3(stream_grid(s.batch, ST_WARPS * 4 * 2, num_sms)), dim3(ST_THREADS), 0, stream, net, s.w,
                    (const float*)s.dz[1], (const float*)s.act[0], s.batch, s.dz[0]);
}

}  // namespace ga3c
