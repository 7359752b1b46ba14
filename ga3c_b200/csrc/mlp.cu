// Low-dimensional MLP policy/value networks of the fork (BASELINE config 4; SURVEY 8a rows A6 / A7), fp32 throughout:
//   fork NetworkVP          NetworkVP.py:79-105, :175-210   x -> 4 -> 256 -> 256 (linear) -> 100 -> 64 (sigmoid); atan2 angle head
//   NetworkVP_discrate      NetworkVP_discrate.py:52-85     x -> last DENSE_LAYERS entry (sigmoid); softmax head, A3C loss
//
// Three kernels per training step (one per prediction):
//   mlp_fused   one persistent CTA (16 warps) per SM walks 64-row batch tiles.  A tile's activations stay in shared memory through
//               all layers, the heads, the loss and the whole data-gradient chain; HBM sees x once, p / v, and (training
//               only) the layer outputs and pre-activation gradients that the weight-gradient pass needs.
//   mlp_wgrad   every dW = in^T dz and db = sum dz of the step as 64x64 output tiles, the batch split over CTAs; split s
//               writes its own partial arena -- no atomics, fixed summation order, bit-reproducible.
//   mlp_reduce  sums the partial arenas into the gradient arena and the per-tile loss sums into loss[4].
// RMSProp is the arena kernel of elementwise.cu.  The weights (0.4 MB) stay L2-resident; they are staged through shared
// memory in 16-row chunks, transposed on the fly for the data gradients (no transposed shadow copy to keep in sync).
#include "common.cuh"
#include "kernels.h"
#include "mlp.cuh"
#include "a3c_loss.cuh"

namespace ga3c {

namespace {

constexpr int LD = 260;              // row pitch (floats) of the activation tiles and of the weight chunk: 16-B aligned rows
constexpr int RC = 16;               // reduction chunk
constexpr int WS = 3;                // stages of the weight-chunk ring (cp.async)
constexpr int HLD = 49;              // row pitch of the head matrix / logits tile (odd: conflict-free column walks)
constexpr int NT = 256;              // threads of the weight-gradient / reduce kernels
constexpr int FT = 512;              // threads of the fused kernel: 16 warps x 4 rows = one 64-row tile
constexpr int HW = 48;               // head matrix columns held in shared memory (>= MLP_MAX_OUT, zero padded)

constexpr size_t FUSED_SMEM =
    (size_t)(2 * MLP_TM * LD + WS * RC * LD + MLP_MAX_HID * HLD + MLP_TM * HLD + 48 + 32) * sizeof(float);
static_assert(FUSED_SMEM <= 232448, "shared memory budget of one CTA per SM");

__device__ __forceinline__ int round_up16(int v) { return (v + 15) & ~15; }

// element (k, j) of the head matrix [hid][n_out]: column 0 = logits_v, then logits_p (discrate) or out_x | out_y (fork_vp)
__device__ __forceinline__ int head_w_index(const MlpNet& net, int k, int j) {
  const int A = net.num_actions;
  if (j == 0) return net.wv_off + k;
  if (j <= A) return net.wp_off + k * A + (j - 1);
  return net.wy_off + k * A + (j - 1 - A);
}
__device__ __forceinline__ int head_b_index(const MlpNet& net, int j) {
  const int A = net.num_actions;
  if (j == 0) return net.bv_off;
  if (j <= A) return net.bp_off + (j - 1);
  return net.by_off + (j - 1 - A);
}

// One 64-row x (128 * JH)-column product through the CTA:  out[r][c] = sum_q in_s[r][q] * Wq[q][c], q < kred, with
//   TRANS = false:  Wq[q][c] = Wg[q * ldw + c]        (forward:        W is [k][n], q = k, c = n)
//   TRANS = true :  Wq[q][c] = Wg[c * ldw + q]        (data gradient:  W is [k][n], q = n, c = k)
// Thread (ty = warp, tx = lane) owns rows ty*RT .. ty*RT+RT-1 (RT = 4: 64-row tiles; RT = 1: 16-row tiles for small
// batches, where 64-row tiles would leave most SMs idle) and columns tx*4 .. tx*4+3 (+128 with JH = 2): 16 warps, four per
// scheduler (two 8-row warps per scheduler left the FMA pipe idle 45 % of the time: nothing to switch to on a shared-memory
// wait).
// epi(r, c0, v[4]) receives the finished sums of 4 consecutive columns, turns them into what the next pass reads and
// stores whatever goes to HBM; the result lands in out_s.  in_s must be zero (finite) up to round_up16(kred).
template <bool TRANS, int JH, int RT, class Epi>
__device__ __forceinline__ void tile_pass(const float* in_s, float* out_s, float* Wc, int kred, const float* __restrict__ Wg,
                                          int ldw, int nout, Epi epi) {
  const int tid = threadIdx.x, ty = tid >> 5, tx = tid & 31;
  float acc[RT][4 * JH];
#pragma unroll
  for (int i = 0; i < RT; ++i)
#pragma unroll
    for (int j = 0; j < 4 * JH; ++j) acc[i][j] = 0.f;

  // weight chunks travel global -> shared with cp.async through a ring of WS stages: chunk ci + WS - 1 is in flight while
  // chunk ci is consumed (one block barrier per chunk).  16-byte copies along contiguous rows in the forward layout when the
  // row pitch allows it, 4-byte copies otherwise and for the transposed (data-gradient) layout; out-of-range elements are
  // zero-filled by the copy itself (src-size 0).
  const bool vec = !TRANS && (ldw & 3) == 0 && (nout & 3) == 0;
  auto issue = [&](int q0, int stage) {
    float* dst = Wc + stage * (RC * LD);
    if (!TRANS) {
      if (vec) {
#pragma unroll
        for (int i = 0; i < RC * 64 / FT; ++i) {           // 16 rows x 64 float4
          const int idx = tid + FT * i, rr = idx >> 6, c = (idx & 63) * 4;
          const bool ok = q0 + rr < kred && c < nout;
          cp_async16(smem_u32(dst + rr * LD + c), Wg + (size_t)(ok ? q0 + rr : 0) * ldw + (ok ? c : 0), ok ? 16 : 0);
        }
      } else {
        const int c = tid & 255, rh = tid >> 8;            // column c, chunk rows rh, rh + 2, ...
#pragma unroll
        for (int i = 0; i < RC * 256 / FT; ++i) {
          const int rr = rh + 2 * i;
          const bool ok = q0 + rr < kred && c < nout;
          cp_async4(smem_u32(dst + rr * LD + c), Wg + (size_t)(ok ? q0 + rr : 0) * ldw + (ok ? c : 0), ok ? 4 : 0);
        }
      }
    } else {
      const int rr = tid & 15, cb = tid >> 4;              // 16 consecutive n of W row c: 64-byte segments
#pragma unroll
      for (int i = 0; i < RC * 256 / FT; ++i) {
        const int c = cb + 32 * i;
        const bool ok = q0 + rr < kred && c < nout;
        cp_async4(smem_u32(dst + rr * LD + c), Wg + (size_t)(ok ? c : 0) * ldw + (ok ? q0 + rr : 0), ok ? 4 : 0);
      }
    }
  };

  const int nchunks = (kred + RC - 1) / RC;
  __syncthreads();                   // in_s is complete and nobody still reads the ring (previous pass)
#pragma unroll
  for (int st = 0; st < WS - 1; ++st) {
    if (st < nchunks) issue(st * RC, st);
    cp_async_commit();
  }
  for (int ci = 0; ci < nchunks; ++ci) {
    const int q0 = ci * RC;
    cp_async_wait<WS - 2>();         // this thread's copies of chunk ci have landed ...
    __syncthreads();                 // ... and everybody's; everybody is also done with chunk ci - 1, whose stage is refilled now
    if (ci + WS - 1 < nchunks) issue((ci + WS - 1) * RC, (ci + WS - 1) % WS);
    cp_async_commit();
    const float* Wst = Wc + (ci % WS) * (RC * LD);
#pragma unroll
    for (int q4 = 0; q4 < RC / 4; ++q4) {
      float4 a[RT];
#pragma unroll
      for (int i = 0; i < RT; ++i) a[i] = *reinterpret_cast<const float4*>(in_s + (ty * RT + i) * LD + q0 + q4 * 4);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float4 w[JH];
#pragma unroll
        for (int h = 0; h < JH; ++h) w[h] = *reinterpret_cast<const float4*>(Wst + (q4 * 4 + e) * LD + tx * 4 + 128 * h);
#pragma unroll
        for (int i = 0; i < RT; ++i) {
          const float av = e == 0 ? a[i].x : e == 1 ? a[i].y : e == 2 ? a[i].z : a[i].w;
#pragma unroll
          for (int h = 0; h < JH; ++h) {
            acc[i][4 * h + 0] = fmaf(av, w[h].x, acc[i][4 * h + 0]);
            acc[i][4 * h + 1] = fmaf(av, w[h].y, acc[i][4 * h + 1]);
            acc[i][4 * h + 2] = fmaf(av, w[h].z, acc[i][4 * h + 2]);
            acc[i][4 * h + 3] = fmaf(av, w[h].w, acc[i][4 * h + 3]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < RT; ++i)
#pragma unroll
    for (int h = 0; h < JH; ++h) {
      float v[4] = {acc[i][4 * h], acc[i][4 * h + 1], acc[i][4 * h + 2], acc[i][4 * h + 3]};
      const int r = ty * RT + i, c0 = tx * 4 + 128 * h;
      epi(r, c0, v);
      *reinterpret_cast<float4*>(out_s + r * LD + c0) = make_float4(v[0], v[1], v[2], v[3]);
    }
}

// Data gradient into a NARROW layer (nout <= 8 columns; fork NetworkVP: 256 -> 4): tile_pass would compute 128 columns for them.
// The nout x kred weights are staged in shared memory (the chunk ring is idle here; straight from global every term of the
// dot products waited out an L2 latency: 133 us for this pass at B = 65,536, measured).  TPR threads share a row: each sums every
// TPR-th term of the dot products, a shuffle tree adds them, lane 0 of the group finishes the row.
//   out[r][c] = sum_q in_s[r][q] * Wg[c * ldw + q], q < kred   (the transposed weight layout of tile_pass<true>)
template <int RT, class Epi>
__device__ __forceinline__ void narrow_dgrad_pass(const float* in_s, float* out_s, float* Wc, int kred, const float* __restrict__ Wg,
                                                  int ldw, int nout, Epi epi) {
  constexpr int TM = (FT / 32) * RT, TPR = FT / TM;        // 8 threads per row (64-row tiles) or 32 (16-row tiles)
  const int tid = threadIdx.x, row = tid / TPR, part = tid % TPR;
  __syncthreads();                   // in_s is complete, nobody reads the ring any more
  for (int idx = tid; idx < 8 * kred; idx += FT) {
    const int c = idx / kred, q = idx - c * kred;
    Wc[c * LD + q] = c < nout ? __ldg(Wg + (size_t)c * ldw + q) : 0.f;
  }
  __syncthreads();
  float acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.f;
  if (nout <= 4) {
#pragma unroll 4
    for (int q = part; q < kred; q += TPR) {
      const float a = in_s[row * LD + q];
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[c] = fmaf(a, Wc[c * LD + q], acc[c]);
    }
  } else {
#pragma unroll 4
    for (int q = part; q < kred; q += TPR) {
      const float a = in_s[row * LD + q];
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[c] = fmaf(a, Wc[c * LD + q], acc[c]);
    }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int o = TPR / 2; o >= 1; o >>= 1) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], o);
  if (part == 0) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (4 * h >= nout) break;
      float v[4] = {acc[4 * h], acc[4 * h + 1], acc[4 * h + 2], acc[4 * h + 3]};
      epi(row, 4 * h, v);
      *reinterpret_cast<float4*>(out_s + row * LD + 4 * h) = make_float4(v[0], v[1], v[2], v[3]);
    }
    for (int c = (nout + 3) & ~3; c < 16; c += 4) *reinterpret_cast<float4*>(out_s + row * LD + c) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// store 4 consecutive columns c0.. of row `row` of a [B][n] matrix (n need not be a multiple of 4)
__device__ __forceinline__ void store_row4(float* base, int64_t row, int n, int c0, const float (&v)[4]) {
  float* dst = base + row * n + c0;
  if ((n & 3) == 0) {
    if (c0 < n) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (c0 + e < n) dst[e] = v[e];
  }
}

template <bool TRAIN, int RT>
__global__ void __launch_bounds__(FT, 1) mlp_fused_kernel(const MlpNet net, const MlpStepArgs s) {
  constexpr int TM = (FT / 32) * RT;       // rows per tile (64 or 16)
  constexpr int TPR = FT / TM;             // threads per row in the head stages (8 or 32)
  constexpr int NJ = (HW + TPR - 1) / TPR; // head columns per thread
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = buf0 + MLP_TM * LD;
  float* Wc = buf1 + MLP_TM * LD;
  float* Wh = Wc + WS * RC * LD;           // [hid][HLD] head matrix, columns >= n_out zero
  float* lg = Wh + MLP_MAX_HID * HLD;      // [64][HLD] logits, then dlogits
  float* hb = lg + MLP_TM * HLD;           // [48] head biases
  float* red = hb + 48;                    // [8 warps][4] loss sums
  const int tid = threadIdx.x;
  const int B = s.batch, S = net.state_dim, A = net.num_actions, NL = net.n_layers, hid = net.hid, n_out = net.n_out;

  griddep_launch();
  griddep_wait(K_MLP_FUSED);               // the weights come from the optimizer launch of the previous step

  for (int idx = tid; idx < hid * HW; idx += FT) {
    const int k = idx / HW, j = idx - k * HW;
    Wh[k * HLD + j] = j < n_out ? __ldg(s.w + head_w_index(net, k, j)) : 0.f;
  }
  if (tid < 48) hb[tid] = tid < n_out ? __ldg(s.w + head_b_index(net, tid)) : 0.f;

  const int ntiles = (B + TM - 1) / TM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    __syncthreads();                       // the previous tile is fully consumed (and Wh / hb are staged)
    {
      // the tile's input: x, or (tensor-core mode, MlpStepArgs::phase) what the GEMM launches before this one left in HBM
      const float* src = s.phase == 2 ? s.act[s.tc_hi - 1] : s.phase == 3 ? s.dz[s.tc_lo - 1] : s.x;
      const int W = s.phase == 2 ? net.L[s.tc_hi - 1].n : s.phase == 3 ? net.L[s.tc_lo - 1].n : S;
      const int Sp = round_up16(W);
      if ((W & 3) == 0 && s.phase != 0) {
        // wide HBM matrices: 16-byte loads, all of a thread's loads in flight (scalar loads in a rolled loop cost one memory
        // latency per 512 floats of the tile: 112 us of a 242 us launch, measured)
        const int S4 = Sp >> 2, n4 = TM * S4;
#pragma unroll 8
        for (int idx = tid; idx < n4; idx += FT) {
          const int r = idx / S4, c = (idx - r * S4) * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row0 + r < B && c < W) v = __ldcs(reinterpret_cast<const float4*>(src + (size_t)(row0 + r) * W + c));
          *reinterpret_cast<float4*>(buf0 + r * LD + c) = v;
        }
      } else {
        for (int idx = tid; idx < TM * Sp; idx += FT) {
          const int r = idx / Sp, c = idx - r * Sp;
          buf0[r * LD + c] = (row0 + r < B && c < W) ? src[(size_t)(row0 + r) * W + c] : 0.f;
        }
      }
    }
    float* cur = buf0;
    float* nxt = buf1;
    const int l_first = s.phase == 2 ? s.tc_hi : 0;                 // forward layers [l_first, l_end)
    const int l_end = s.phase == 1 ? s.tc_lo : s.phase == 3 ? 0 : NL;

    // ---- forward: out_l = act(in_l W_l + b_l)  (NetworkVP.py:194-210) ----
    for (int l = l_first; l < l_end; ++l) {
      const MlpLayerDesc L = net.L[l];
      const float* bias = s.w + L.b_off;
      float* out_g = TRAIN ? s.act[l] : nullptr;
      auto epi = [&](int r, int c0, float (&v)[4]) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int c = c0 + e;
          float z = 0.f;
          if (c < L.n) {
            z = v[e] + __ldg(bias + c);
            if (L.act == MLP_ACT_SIGMOID) z = sigmoid(z);
          }
          v[e] = z;
        }
        if (TRAIN && row0 + r < B) store_row4(out_g, row0 + r, L.n, c0, v);
      };
      if (L.n > 128) tile_pass<false, 2, RT>(cur, nxt, Wc, L.k, s.w + L.w_off, L.n, L.n, epi);
      else tile_pass<false, 1, RT>(cur, nxt, Wc, L.k, s.w + L.w_off, L.n, L.n, epi);
      float* t = cur; cur = nxt; nxt = t;
    }
    if (s.phase == 1) continue;            // the wide layers follow as GEMM launches
    if (s.phase != 3) {
    __syncthreads();                       // h = cur[64][hid] is complete

    // ---- head logits: thread (row, jq) sums columns jq, jq + TPR, ... of h Wh ----
    {
      const int row = tid / TPR, jq = tid % TPR;
      float z[NJ];
#pragma unroll
      for (int jj = 0; jj < NJ; ++jj) z[jj] = 0.f;
      for (int k = 0; k < hid; ++k) {
        const float h = cur[row * LD + k];
#pragma unroll
        for (int jj = 0; jj < NJ; ++jj)
          if (jq + TPR * jj < HW) z[jj] = fmaf(h, Wh[k * HLD + jq + TPR * jj], z[jj]);
      }
#pragma unroll
      for (int jj = 0; jj < NJ; ++jj) {
        const int j = jq + TPR * jj;
        if (j < n_out) lg[row * HLD + j] = z[jj] + hb[j];
      }
    }
    __syncthreads();

    // ---- per row: p, v, loss terms, dlogits (a3c_loss.cuh) ----
    A3cSums sums;
    if (tid < TM) {
      const int r = tid;
      const bool valid = row0 + r < B;
      float* z = lg + r * HLD;
      const float v = z[0];
      const float yr = TRAIN && valid ? s.yr[row0 + r] : 0.f;
      if (valid && s.v_out != nullptr) s.v_out[row0 + r] = v;
      A3cTerms t{};
      if (net.kind == MLP_KIND_FORK_VP) {
        float sel = 0.f, sq = 0.f;
        for (int j = 0; j < A; ++j) {
          const float av = TRAIN && valid ? s.a[(size_t)(row0 + r) * A + j] : 0.f;
          const ForkAction f = fork_policy(z[1 + j], z[1 + A + j], av, v, yr, s.la, sel, sq);
          if (valid && s.p_out != nullptr) s.p_out[(size_t)(row0 + r) * A + j] = f.p;
          if (TRAIN) {
            z[1 + j] = valid ? f.dzx : 0.f;
            z[1 + A + j] = valid ? f.dzy : 0.f;
          }
        }
        t = fork_policy_terms(sel, sq, v, yr, s.la);
      } else {
        // a row beyond the batch takes zero actions; its p is not stored and its gradients are zero
        const float* arow = s.a + (size_t)(row0 + r) * A;
        float* prow = s.p_out + (size_t)(row0 + r) * A;
        t = softmax_policy_row(
            z + 1, A, v, yr, s.la, policy_inv_mix(s.la, A), TRAIN, [&](int j) { return valid ? arow[j] : 0.f; },
            [&](int j, float pj) { if (valid && s.p_out != nullptr) prow[j] = pj; },
            [&](int j, float dzj) { z[1 + j] = valid ? dzj : 0.f; });
      }
      if (TRAIN) {
        z[0] = valid ? t.dv : 0.f;
        if (valid) {
          t.add_to(s.la.beta, sums);
          float* dl = s.dlogits + (size_t)(row0 + r) * net.n_out_ld;
          for (int j = 0; j < n_out; ++j) dl[j] = z[j];
        }
      }
    }
    if (!TRAIN) continue;

    // loss sums of the tile, fixed order: warp tree, then warp 0 + warp 1
    constexpr int RW = (TM + 31) / 32;     // warps that hold rows (threads beyond TM contribute zeros)
    if (tid < 32 * RW) {
      const float l1 = warp_sum(sums.l1), l2 = warp_sum(sums.l2), lv = warp_sum(sums.lv);
      if ((tid & 31) == 0) { red[(tid >> 5) * 4 + 0] = l1; red[(tid >> 5) * 4 + 1] = l2; red[(tid >> 5) * 4 + 2] = lv; }
    }
    __syncthreads();                       // dlogits tile + loss partials visible
    if (tid < 4) {
      float t = 0.f;
      if (tid < 3)
#pragma unroll
        for (int w = 0; w < RW; ++w) t += red[w * 4 + tid];
      s.loss_part[(size_t)tile * 4 + tid] = t;
    }

    // ---- gradient w.r.t. the last hidden pre-activation: dz = (dlogits Wh^T) * act'(h) ----
    {
      const MlpLayerDesc L = net.L[NL - 1];
      const int row = tid / TPR, kq = tid % TPR;
      const int hp = round_up16(hid);
      float* dz_g = s.dz[NL - 1];
      for (int k = kq; k < hp; k += TPR) {
        float d = 0.f;
        if (k < hid) {
          for (int j = 0; j < n_out; ++j) d = fmaf(lg[row * HLD + j], Wh[k * HLD + j], d);
          if (L.act == MLP_ACT_SIGMOID) { const float h = cur[row * LD + k]; d *= h * (1.f - h); }
          if (row0 + row < B) dz_g[(size_t)(row0 + row) * hid + k] = d;
        }
        nxt[row * LD + k] = d;
      }
    }
    { float* t = cur; cur = nxt; nxt = t; }
    }   // phase != 3

    // ---- data-gradient chain: dz_{l-1} = (dz_l W_l^T) * act'(out_{l-1}) ----
    const int l_top = s.phase == 3 ? s.tc_lo - 1 : NL - 1;          // the chain starts from dz[l_top] (in `cur`) ...
    const int l_stop = s.phase == 2 ? (s.tc_hi > 1 ? s.tc_hi : 1) : 1;   // ... and ends with dz[l_stop - 1]
    for (int l = l_top; l >= l_stop; --l) {
      const MlpLayerDesc L = net.L[l];
      const MlpLayerDesc Lp = net.L[l - 1];
      const float* out_prev = s.act[l - 1];
      float* dz_g = s.dz[l - 1];
      auto epi = [&](int r, int c0, float (&v)[4]) {
        const bool valid = row0 + r < B;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int c = c0 + e;
          float d = 0.f;
          if (c < Lp.n && valid) {
            d = v[e];
            if (Lp.act == MLP_ACT_SIGMOID) { const float o = out_prev[(size_t)(row0 + r) * Lp.n + c]; d *= o * (1.f - o); }
          }
          v[e] = d;
        }
        if (valid) store_row4(dz_g, row0 + r, Lp.n, c0, v);
      };
      if (Lp.n > 128) tile_pass<true, 2, RT>(cur, nxt, Wc, L.n, s.w + L.w_off, L.n, Lp.n, epi);
      else if (Lp.n <= 8) narrow_dgrad_pass<RT>(cur, nxt, Wc, L.n, s.w + L.w_off, L.n, Lp.n, epi);
      else tile_pass<true, 1, RT>(cur, nxt, Wc, L.n, s.w + L.w_off, L.n, Lp.n, epi);
      float* t = cur; cur = nxt; nxt = t;
    }
  }
  trace_mark(K_MLP_FUSED, 2);
}

// ---- weight gradients ---------------------------------------------------------------------------------------
// blockIdx.x walks the 64x64 output tiles of every dW (hidden layers in order, then the head matrix), blockIdx.y the
// batch splits.  256 threads = 16 (k quads) x 16 (n quads), 4x4 sums each, rows staged 16 at a time.
constexpr int WT = 64, WLD = 68;
__global__ void __launch_bounds__(NT) mlp_wgrad_kernel(const MlpNet net, const MlpStepArgs s, float* part, int64_t part_stride,
                                                       int rows_per_split) {
  __shared__ __align__(16) float inC[RC][WLD];
  __shared__ __align__(16) float dzC[RC][WLD];
  const int tid = threadIdx.x, NL = net.n_layers;
  // which tile
  int t = blockIdx.x, l = 0, K = 0, N = 0, tn = 1;
  for (; l <= NL; ++l) {
    K = l < NL ? net.L[l].k : net.hid;
    N = l < NL ? net.L[l].n : net.n_out;
    const int tk = (K + WT - 1) / WT;
    tn = (N + WT - 1) / WT;
    if (t < tk * tn) break;
    t -= tk * tn;
  }
  if (l > NL) return;
  if ((s.wgrad_skip >> l) & 1u) return;              // tensor-core mode: this matrix's dW / db come from the kernels of mlp_tc.cu
  const int k0 = (t / tn) * WT, n0 = (t % tn) * WT;
  const float* in = l == 0 ? s.x : s.act[l - 1];
  const int ld_in = K;
  const float* dz = l < NL ? s.dz[l] : s.dlogits;
  const int ld_dz = l < NL ? N : net.n_out_ld;
  const int r_begin = blockIdx.y * rows_per_split;
  const int r_end = min(s.batch, r_begin + rows_per_split);

  griddep_launch();
  griddep_wait(K_MLP_WGRAD);

  const int cc = tid & 63, rq = tid >> 6;           // staging: column cc, rows rq, rq + 4, rq + 8, rq + 12
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4], bs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float pa[4], pb[4];
  auto fetch = [&](int r0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = r0 + rq + 4 * i;
      pa[i] = (r < r_end && k0 + cc < K) ? in[(size_t)r * ld_in + k0 + cc] : 0.f;
      pb[i] = (r < r_end && n0 + cc < N) ? dz[(size_t)r * ld_dz + n0 + cc] : 0.f;
    }
  };
  if (r_begin < r_end) fetch(r_begin);
  for (int r0 = r_begin; r0 < r_end; r0 += RC) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) { inC[rq + 4 * i][cc] = pa[i]; dzC[rq + 4 * i][cc] = pb[i]; }
    __syncthreads();
    if (r0 + RC < r_end) fetch(r0 + RC);
#pragma unroll
    for (int rr = 0; rr < RC; ++rr) {
      const float4 a = *reinterpret_cast<const float4*>(&inC[rr][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&dzC[rr][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
#pragma unroll
      for (int j = 0; j < 4; ++j) bs[j] += bv[j];
    }
  }
  float* out = part + (size_t)blockIdx.y * part_stride;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = n0 + tx * 4 + j;
    if (n >= N) continue;
    // column n of this layer's dz -> (tensor, column) of the arena
    int w_off, b_off, width, col;
    if (l < NL) { w_off = net.L[l].w_off; b_off = net.L[l].b_off; width = N; col = n; }
    else {
      const int A = net.num_actions;
      if (n == 0) { w_off = net.wv_off; b_off = net.bv_off; width = 1; col = 0; }
      else if (n <= A) { w_off = net.wp_off; b_off = net.bp_off; width = A; col = n - 1; }
      else { w_off = net.wy_off; b_off = net.by_off; width = A; col = n - 1 - A; }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = k0 + ty * 4 + i;
      if (k < K) out[w_off + (size_t)k * width + col] = acc[i][j];
    }
    if (k0 == 0 && ty == 0) out[b_off + col] = bs[j];
  }
  trace_mark(K_MLP_WGRAD, 2);
}

// Head matrices (logits_v | logits_p [| out_y]: n_out <= 4 columns) for large batches: dW[k][j] = sum_r h[r][k] dlogits[r][j],
// db[j] = sum_r dlogits[r][j] per batch split, streaming h once: 1024 threads = 16 row groups x 64 columns of h, the row groups
// added in a fixed order.  (The 64 x 64 tile kernel above spends 157 us on this 64 x 3 product at B = 65,536.)
__global__ void __launch_bounds__(1024) mlp_heads_wgrad_kernel(const MlpNet net, const float* __restrict__ h,
                                                                const float* __restrict__ dl, int batch, int rows_per_split,
                                                                float* part, int64_t part_stride) {
  __shared__ float red[16][8][64];
  griddep_launch();
  griddep_wait(K_MLP_WGRAD);
  const int rg = threadIdx.x >> 6, c = threadIdx.x & 63, k = blockIdx.y * 64 + c;
  const int hid = net.hid, J = net.n_out, ld = net.n_out_ld;
  const int r0 = blockIdx.x * rows_per_split, r1 = min(batch, r0 + rows_per_split);
  float acc[4] = {0.f, 0.f, 0.f, 0.f}, bs[4] = {0.f, 0.f, 0.f, 0.f};
  if (k < hid) {
    constexpr int U = 4;
    int r = r0 + rg;
    for (; r + 16 * (U - 1) < r1; r += 16 * U) {
      float4 d[U];
      float hv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        d[u] = __ldg(reinterpret_cast<const float4*>(dl + (size_t)(r + 16 * u) * ld));
        hv[u] = __ldcs(h + (size_t)(r + 16 * u) * hid + k);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        acc[0] = fmaf(d[u].x, hv[u], acc[0]); acc[1] = fmaf(d[u].y, hv[u], acc[1]);
        acc[2] = fmaf(d[u].z, hv[u], acc[2]); acc[3] = fmaf(d[u].w, hv[u], acc[3]);
        bs[0] += d[u].x; bs[1] += d[u].y; bs[2] += d[u].z; bs[3] += d[u].w;
      }
    }
    for (; r < r1; r += 16) {
      const float4 d = __ldg(reinterpret_cast<const float4*>(dl + (size_t)r * ld));
      const float hv = h[(size_t)r * hid + k];
      acc[0] = fmaf(d.x, hv, acc[0]); acc[1] = fmaf(d.y, hv, acc[1]); acc[2] = fmaf(d.z, hv, acc[2]); acc[3] = fmaf(d.w, hv, acc[3]);
      bs[0] += d.x; bs[1] += d.y; bs[2] += d.z; bs[3] += d.w;
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) { red[rg][j][c] = acc[j]; red[rg][4 + j][c] = bs[j]; }
  __syncthreads();
  if (rg == 0 && k < hid) {
    float* out = part + (size_t)blockIdx.x * part_stride;
    for (int j = 0; j < J; ++j) {
      float t = 0.f, b = 0.f;
#pragma unroll
      for (int g = 0; g < 16; ++g) { t += red[g][j][c]; b += red[g][4 + j][c]; }
      out[head_w_index(net, k, j)] = t;
      if (k == 0) out[head_b_index(net, j)] = b;
    }
  }
}

// ---- partial arenas -> gradient arena; per-tile loss sums -> loss[4] -----------------------------------------
__global__ void __launch_bounds__(NT) mlp_reduce_kernel(const float* part, int64_t part_stride, int splits, float* g, int n4,
                                                        const float* loss_part, int tiles, float* loss_out) {
  griddep_launch();
  griddep_wait(K_MLP_REDUCE);
  // four adjacent lanes share one float4 of the arena: lane q adds its quarter of the splits in split order (RU loads in flight),
  // then (q0 + q1) + (q2 + q3) by two shuffles -- a fixed order.  (One thread per float4 walking all 74 splits with one load per
  // memory latency made this kernel 27 us at B = 65,536.)
  constexpr int RU = 8;
  const int i = (blockIdx.x * NT + threadIdx.x) >> 2, q4 = threadIdx.x & 3;
  const int per = (splits + 3) >> 2, s_lo = q4 * per, s_hi = min(splits, s_lo + per);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < n4) {
    for (int sp0 = s_lo; sp0 < s_hi; sp0 += RU) {
      float4 q[RU];
#pragma unroll
      for (int u = 0; u < RU; ++u)
        q[u] = sp0 + u < s_hi ? __ldcg(reinterpret_cast<const float4*>(part + (size_t)(sp0 + u) * part_stride) + i)
                              : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < RU; ++u) { acc.x += q[u].x; acc.y += q[u].y; acc.z += q[u].z; acc.w += q[u].w; }
    }
  }
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1) {
    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
    acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
  }
  if (i < n4 && q4 == 0) reinterpret_cast<float4*>(g)[i] = acc;
  if (blockIdx.x == 0 && threadIdx.x < 128 && loss_out != nullptr) {
    // warp c sums component c: lane adds tiles lane, lane + 32, ... in order, then the fixed shuffle tree
    const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float v = 0.f;
    for (int t0 = lane; t0 < tiles; t0 += 32 * RU) {           // same order as a plain loop, RU loads in flight
      float q[RU];
#pragma unroll
      for (int u = 0; u < RU; ++u) q[u] = t0 + 32 * u < tiles ? __ldcg(loss_part + (size_t)(t0 + 32 * u) * 4 + c) : 0.f;
#pragma unroll
      for (int u = 0; u < RU; ++u) v += q[u];
    }
    v = warp_sum(v);
    if (lane == 0) loss_out[c] = v;
  }
  trace_mark(K_MLP_REDUCE, 2);
}

int total_wgrad_tiles(const MlpNet& net) {
  int t = 0;
  for (int l = 0; l <= net.n_layers; ++l) {
    const int K = l < net.n_layers ? net.L[l].k : net.hid, N = l < net.n_layers ? net.L[l].n : net.n_out;
    t += ((K + WT - 1) / WT) * ((N + WT - 1) / WT);
  }
  return t;
}

}  // namespace

GA3C_TRACE_ATTACH(trace_attach_mlp)

int configure_mlp() {
  int r;
  if ((r = (int)cudaFuncSetAttribute(mlp_fused_kernel<true, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FUSED_SMEM))) return r;
  if ((r = (int)cudaFuncSetAttribute(mlp_fused_kernel<false, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FUSED_SMEM))) return r;
  if ((r = (int)cudaFuncSetAttribute(mlp_fused_kernel<true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FUSED_SMEM))) return r;
  return (int)cudaFuncSetAttribute(mlp_fused_kernel<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FUSED_SMEM);
}

// rows per tile: 64, or 16 when 64-row tiles would occupy less than half of the SMs
int mlp_tile_rows(int batch, int num_sms) { return (batch + MLP_TM - 1) / MLP_TM * 2 < num_sms ? 16 : MLP_TM; }

int mlp_fused_grid(int batch, int num_sms) {
  const int tm = mlp_tile_rows(batch, num_sms);
  const int tiles = (batch + tm - 1) / tm;
  return tiles < num_sms ? tiles : num_sms;
}

int launch_mlp_fused(const MlpNet& net, const MlpStepArgs& args, int num_sms, cudaStream_t stream) {
  const dim3 grid(mlp_fused_grid(args.batch, num_sms));
  if (mlp_tile_rows(args.batch, num_sms) == 16) {
    if (args.train) return launch_pdl(mlp_fused_kernel<true, 1>, grid, dim3(FT), FUSED_SMEM, stream, net, args);
    return launch_pdl(mlp_fused_kernel<false, 1>, grid, dim3(FT), FUSED_SMEM, stream, net, args);
  }
  if (args.train) return launch_pdl(mlp_fused_kernel<true, 4>, grid, dim3(FT), FUSED_SMEM, stream, net, args);
  return launch_pdl(mlp_fused_kernel<false, 4>, grid, dim3(FT), FUSED_SMEM, stream, net, args);
}

int mlp_wgrad_splits(const MlpNet& net, int batch, int num_sms) {
  const int tiles = total_wgrad_tiles(net);
  int splits = (4 * num_sms + tiles - 1) / tiles;
  const int by_rows = (batch + 127) / 128;            // at least 128 rows per split
  if (splits > by_rows) splits = by_rows;
  if (splits > MLP_MAX_SPLITS) splits = MLP_MAX_SPLITS;
  return splits < 1 ? 1 : splits;
}

int launch_mlp_wgrad(const MlpNet& net, const MlpStepArgs& args, float* part, int64_t part_stride, int splits,
                     cudaStream_t stream, int rows_per_split) {
  int rows = rows_per_split > 0 ? rows_per_split : (args.batch + splits - 1) / splits;
  rows = (rows + RC - 1) / RC * RC;
  const dim3 grid(total_wgrad_tiles(net), splits);
  return launch_pdl(mlp_wgrad_kernel, grid, dim3(NT), 0, stream, net, args, part, part_stride, rows);
}

bool mlp_heads_wgrad_ok(const MlpNet& net) { return net.n_out <= 4 && net.n_out_ld == 4; }
int launch_mlp_heads_wgrad(const MlpNet& net, const MlpStepArgs& args, float* part, int64_t part_stride, int splits,
                           int rows_per_split, cudaStream_t stream) {
  const dim3 grid(splits, (net.hid + 63) / 64);
  return launch_pdl(mlp_heads_wgrad_kernel, grid, dim3(1024), 0, stream, net, (const float*)args.act[net.n_layers - 1],
                    (const float*)args.dlogits, args.batch, rows_per_split, part, part_stride);
}

int launch_mlp_reduce(const float* part, int64_t part_stride, int splits, float* g, int live_floats, const float* loss_part,
                      int tiles, float* loss_out, cudaStream_t stream) {
  const int n4 = live_floats / 4;
  const int grid = (4 * n4 + NT - 1) / NT;          // four lanes per float4
  return launch_pdl(mlp_reduce_kernel, dim3(grid < 1 ? 1 : grid), dim3(NT), 0, stream, part, part_stride, splits, g, n4,
                    loss_part, tiles, loss_out);
}

}  // namespace ga3c
