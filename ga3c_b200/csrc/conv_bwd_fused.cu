// Backward of both convolutions in ONE persistent, warp-specialised kernel on the 5th-generation tensor cores
// (the autodiff half of opt.minimize, NetworkVP_discrate.py:130, for the layers at NetworkVP.py:212-228 wired as
// NetworkDNav.py:81-82):
//     dn1  = conv12 data-gradient of dn2, masked by relu'(n1)          (never leaves the SM)
//     g_w12 = patches(n1)^T dn2 , g_b12 = colsum(dn2)
//     g_w11 = patches(x)^T dn1  , g_b11 = colsum(dn1)                  (conv11 has no data-gradient: x is the input)
// bf16 operands, fp32 accumulation in TMEM; the weight-gradient accumulators stay in TMEM for all frames of the CTA and are
// stored once into the CTA's slab of the gradient-partial workspace (rmsprop_reduce / dp_small add the slabs in a fixed order).
//
// Every input arrives in HBM already in the no-swizzle UMMA operand layout it is consumed in (common.cuh): xblk (the bf16
// block matrix of the frame, written by conv_fwd next to n1), n1 as Blk2, dn2 as G (written by the dense1 data-gradient
// epilogue).  The kernel therefore has no conversion or re-layout stage at all: two warps issue cp.async.bulk copies, one warp
// issues UMMAs, the rest run the data-gradient epilogue.  Per frame it reads 64 KB + 20 KB + 11 KB (+ 11 KB again, an L2 hit)
// and writes nothing.  (The first version of this kernel re-read the fp32 frame through a TMA ring and converted it with six
// warps; it was bound by its 110 small UMMAs per frame.  experiments/conv_bwd_v1_fp32_ring_110_umma.cu.txt.)
//
// All three products are GEMMs over space-to-depth block matrices with every row contiguous, so that a spatial shift is a
// different descriptor start address, and a shift that must be part of ONE operand is a second copy stored next to the first:
// conv12 data gradient.  Output pixel (2Yh+py, 2Xh+px) of the padded image gets taps kh = py + 2a, kw = px + 2b from
//   dn2[Yh - a, Xh - b].  With m = Yh*13 + Xh:   D[m, (py, px, ci)] = sum_{a,b} G[m + 14 - 13a - b, :] . Wd_ab
//   where Wd_ab[co, (py, px, ci)] = w12[py + 2a, px + 2b, ci, co]: four row-shifted GEMMs, M = 156 (two 128-row tiles, the
//   second one starting at row 28), N = 64, K = 32 each -> 16 UMMAs.  Row m of D is the whole 2x2 block (Yh, Xh) of dn1.
// conv12 weight gradient.  kh = 2a + dy, kw = 2b + dx: quadrant (a, b) is  dW_ab[(dy, dx, ci), co] = sum_r Blk2[r]^T
//   G[r + 14 - 13a - b]  over the block rows r.  A = Blk2 read MN-major (M = 64), B = G read MN-major with N = 64 = (b, co): the
//   b = 1 half is a second copy of G moved down by one row (a second bulk copy of the same bytes, 16 B further on), the a shift
//   is the start row -> 2 x 9 UMMAs (M = 64, N = 64).
// conv11 weight gradient.  Quadrant (a, b) is dW_ab = sum_r Blk[r]^T dn1[r - 22a - b] over ALL block rows r (dn1 on the 21 x 22
//   position grid, zero elsewhere).  A = Blk read MN-major (M = 64), B = dn1 in EIGHT planes (a, b, half): the data-gradient
//   epilogue writes every dn1 pixel four times, at rows p, p + 1, p + 22, p + 23, so ONE UMMA per k-step with N = 64 =
//   (a, b, cout) covers all four quadrants: 31 UMMAs (M = 64, N = 64).
// 65 UMMAs per frame in all.  Every small UMMA occupies the tensor pipe for ~80 cycles whatever its M / N <= 128
// (profiles/r1h_umma_issue_cost_microbench.txt), so a frame costs ~2.7 us of pipe time against ~2.5 us of HBM time at 1/148 of
// the measured bandwidth.  G / Blk2 are double-buffered: a single buffer put the load latency of the next frame (1.9 us) between
// the conv12 UMMAs of consecutive frames (profiles/r2d_evt_conv_bwd_single_buffer.txt).
//
//   warp  0      Blk quarters of the next frame -> ring of 4 slots (one 16 KB cp.async.bulk each)
//   warp  1      issues every UMMA: conv12 of frame k+2 after the conv11 gradient of frame k
//   warp  2      G (two copies) / Blk2 of frame k+2 into the buffer frame k has left
//   warps 4-7    data-gradient epilogue: TMEM -> relu' mask (n1 from Blk2) -> bf16 -> the eight dn1 planes, bias gradient of
//                conv11; final store of the TMEM weight-gradient accumulators
//   warp  11     the 28 live rows of the second data-gradient tile (it shares TMEM lane quarter 3 with warp 7)
//   warps 3,8-10 bias gradient of conv12 (column sums of G: warp = chunk plane, lane = row phase)
//   warps 12-15  no work: they go straight to the final block barrier
#include "common.cuh"
#include "kernels.h"
#include "tcgen05.cuh"
#include "conv_blk.cuh"

namespace ga3c {

constexpr int FB_THREADS = 512, FB_LOAD_WARP = 0, FB_ISSUE_WARP = 1, FB_C12_WARP = 2, FB_EPI_WARP0 = 4, FB_T1_WARP = 11,
              FB_IDLE_WARP0 = 12;
static_assert(FB_EPI_WARP0 % 4 == 0 && FB_T1_WARP % 4 == 3, "an epilogue warp may only read TMEM lane quarter warp % 4");
constexpr int FB_RING = 4;                                        // Blk quarter slots: one frame
constexpr int W11_KSTEPS = 31;                                    // 496 >= 484 block rows
constexpr int DN1_ROWS = 16 * W11_KSTEPS, DN1_PLANE = DN1_ROWS * 16, DN1_BYTES = 8 * DN1_PLANE;        // 63,488
constexpr int DG_TILE1 = 28;                                      // first row of the second data-gradient tile
constexpr int DG_ROWS = 12 * G_W;                                 // 156 rows of D (12 x 12 blocks + dead column)
constexpr int W12_KSTEPS = 9;                                     // 144 > 140, the last non-zero row of Blk2
constexpr int W12D_BYTES = 4 * 4 * 64 * 16;                       // 4 taps x [4 k-chunks (8 co)][64 rows (py, px, ci)][16 B]
static_assert(4 * XB_QROWS >= DN1_ROWS && DN1_ROWS >= XB_LIVE_ROWS, "the k-steps must cover every block row");
static_assert(16 * (W12_KSTEPS - 1) + G_W + 1 + 15 < G_ROWS && DG_TILE1 + G_W + 1 + 127 < G_ROWS, "G rows read by the UMMAs");
// one conv12 input buffer: G, G moved down by one row, Blk2
constexpr int C12_G1 = G_BYTES, C12_B2 = 2 * G_BYTES, C12_BYTES = 2 * G_BYTES + B2_BYTES;              // 42,496

constexpr int FB_OFF_RING = 0;
constexpr int FB_OFF_DN1 = FB_OFF_RING + FB_RING * XB_QBYTES;     //  65,536
constexpr int FB_OFF_C12 = FB_OFF_DN1 + DN1_BYTES;                // 129,024: two buffers
constexpr int FB_OFF_W12D = FB_OFF_C12 + 2 * C12_BYTES;           // 214,016
constexpr int FB_OFF_RED = FB_OFF_W12D + W12D_BYTES;              // 230,400: [5][16] conv11 bias partials
constexpr int FB_OFF_BAR = FB_OFF_RED + 5 * C1_OUT * 4;
constexpr int FB_QFULL = 0;       // [4] Blk quarter landed in ring slot i (TMA bytes)
constexpr int FB_QFREE = 4;       // [4] the conv11 UMMAs that read slot i retired (tcgen05.commit)       (-> loader)
constexpr int FB_C12RDY = 8;      // [2] G / Blk2 of a frame landed in buffer p (TMA bytes)                (-> issuer, bias warps)
constexpr int FB_EPI12 = 10;      // [2] D drained, Blk2 mask reads and G column sums of the frame in buffer p done, 9 arrivals
                                  //                                                                       (-> loader: buffer free; issuer: D free)
constexpr int FB_MMA12 = 12;      //     conv12 UMMAs of the frame retired (tcgen05.commit)                (-> epilogue)
constexpr int FB_DN1RDY = 13;     //     dn1 operand written, 5 arrivals                                   (epilogue -> issuer)
constexpr int FB_DN1FREE = 14;    //     every conv11 UMMA of the frame retired                            (-> epilogue: operand free)
constexpr int FB_DONE = 15;       //     every UMMA of the kernel retired                                  (-> final store)
constexpr int FB_W12DRDY = 16;    //     data-gradient weights laid out, 9 arrivals                        (-> issuer)
constexpr int FB_NBAR = 17;
constexpr int FB_OFF_TSLOT = FB_OFF_BAR + FB_NBAR * 8;
constexpr int FB_SMEM = FB_OFF_TSLOT + 16 + 128;                  // incl. slack to align the base to 128 B
static_assert(FB_SMEM <= 232448, "shared memory budget of one CTA per SM");
constexpr int FB_TMEM_COLS = 512, TM_W11 = 0, TM_W12 = 64, TM_D12 = 192;   // 64 | 2x64 | 2x64 columns

// EVT: the instantiation with the pipeline event log of CTA 0 (ga3c_evt_*, tools/evt_timeline.py); the production
// instantiation carries none of it.
template <bool EVT>
__global__ void __launch_bounds__(FB_THREADS, 1)
conv_bwd_kernel(const uint8_t* __restrict__ xblk, const uint8_t* __restrict__ n1b2, const uint8_t* __restrict__ dn2g,
                const float* __restrict__ w12, uint16_t* __restrict__ dn1_out, float* __restrict__ g_w11,
                float* __restrict__ g_b11, float* __restrict__ g_w12, float* __restrict__ g_b12, int64_t gp_stride, int batch,
                int hints) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
  uint8_t* const smem = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t ring = sbase + FB_OFF_RING, dn1s = sbase + FB_OFF_DN1, c12 = sbase + FB_OFF_C12, w12d = sbase + FB_OFF_W12D,
                 bars = sbase + FB_OFF_BAR, tslot = sbase + FB_OFF_TSLOT;
  float* red = reinterpret_cast<float*>(smem + FB_OFF_RED);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  EvtLog evt_i = EVT ? evt_open() : EvtLog{nullptr, 0};
  auto mark = [&](int id, int arg) { if (EVT) evt_mark(evt_i, id, arg); };
  const int stride = (int)gridDim.x;
  const int n_frames = ((int)blockIdx.x < batch) ? (batch - 1 - (int)blockIdx.x) / stride + 1 : 0;
  auto frame_of = [&](int k) { return (size_t)(blockIdx.x + k * stride); };
  auto bar = [&](int i) { return bars + i * 8; };
  const uint64_t pol_last_use = (hints & 4) ? l2_policy_evict_first() : l2_policy_normal();    // every input is dead once it has been read

  // ---------------- prologue: everything that does not depend on the preceding kernels ----------------
  if (tid == 0) {
    for (int i = 0; i < FB_RING; ++i) { mbar_init(bar(FB_QFULL + i), 1); mbar_init(bar(FB_QFREE + i), 1); }
    for (int p = 0; p < 2; ++p) { mbar_init(bar(FB_C12RDY + p), 1); mbar_init(bar(FB_EPI12 + p), 9); }
    mbar_init(bar(FB_MMA12), 1);
    mbar_init(bar(FB_DN1RDY), 5);
    mbar_init(bar(FB_DN1FREE), 1);
    mbar_init(bar(FB_DONE), 1);
    mbar_init(bar(FB_W12DRDY), 9);
    fence_mbar_init();
  }
  if (warp == FB_EPI_WARP0) tmem_alloc<FB_TMEM_COLS>(tslot);
  // zero once: rows of the dn1 planes that no pixel is ever written to (dead column, slack); row 0 of the moved copy of G
  for (int i = tid; i < DN1_BYTES / 16; i += FB_THREADS) sts128(dn1s + i * 16, make_uint4(0, 0, 0, 0));
  if (tid < 2) sts128(c12 + tid * C12_BYTES + C12_G1, make_uint4(0, 0, 0, 0));
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(tmem_base) : "r"(tslot));
  // data-gradient weights as the UMMA B operand (K-major, no swizzle): tap (a, b), k-chunk j (8 co), row n = (py, px, ci).
  // Warps 3..11 (the loaders and the issuer are already at work); the issuer waits for FB_W12DRDY before its first UMMA.
  auto build_w12d = [&]() {
    constexpr int NT = 9 * 32, ITEMS = 4 * 4 * 64, PER = (ITEMS + NT - 1) / NT, UNR = 5;
    static_assert(PER % UNR == 0 || PER < UNR * 4, "unroll chunks");
    const int t = tid - 3 * 32;
#pragma unroll 1
    for (int i0 = 0; i0 < PER; i0 += UNR) {
      float4 lo[UNR], hi[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int i = t + (i0 + u) * NT;
        if (i < ITEMS && i0 + u < PER) {
          const int tap = i >> 8, j = (i >> 6) & 3, n = i & 63, a = tap >> 1, b = tap & 1, py = n >> 5, px = (n >> 4) & 1, ci = n & 15;
          const float4* w = reinterpret_cast<const float4*>(w12 + (((py + 2 * a) * 4 + px + 2 * b) * C1_OUT + ci) * C2_OUT + 8 * j);
          lo[u] = w[0]; hi[u] = w[1];
        }
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int i = t + (i0 + u) * NT;
        if (i < ITEMS && i0 + u < PER) {
          const int tap = i >> 8, j = (i >> 6) & 3, n = i & 63;
          sts128(w12d + tap * 4096 + j * 1024 + n * 16,
                 make_uint4(pack_bf16(lo[u].x, lo[u].y), pack_bf16(lo[u].z, lo[u].w), pack_bf16(hi[u].x, hi[u].y), pack_bf16(hi[u].z, hi[u].w)));
        }
      }
    }
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(FB_W12DRDY));
    mark(51, 0);
  };
  // With batch >= the number of SMs the weights can be laid out BEFORE the dependency wait (3 us that used to sit between the wait
  // and the first UMMA, profiles/r2e_evt_*): a CTA of this launch exists only once every CTA of dense_bwd has started, hence of
  // heads, dense_fwd and conv_fwd of this step; the 148 conv_fwd CTAs take a whole SM each, so by then no block of the previous
  // optimizer launch -- the last writer of conv12/w -- is left anywhere (the same argument as RmsPropArgs::preload).
  const bool w12d_early = (hints & 8) != 0;
  if (w12d_early && warp >= 3 && warp <= 11) build_w12d();
  griddep_launch();
  mark(50, 0);
  griddep_wait(K_CONV12_BWD);   // every input comes from the kernels that precede this one
  mark(53, 0);

  // Data-gradient epilogue of one 128-row tile for TMEM lane quarter `qt`: rows of the first tile go to warps 4-7, the 28
  // live rows of the second tile (lanes 100..127) to warp 11.
  auto dgrad_epilogue = [&](int k, int t, int qt, float (&bacc)[C1_OUT]) {
    const uint32_t tlane = tmem_base + ((uint32_t)(qt * 32) << 16);
    const uint32_t b2 = c12 + (k & 1) * C12_BYTES + C12_B2;
    mbar_wait(bar(FB_MMA12), k & 1);
    mark(40, k);
    tc_fence_after();
    uint16_t* dn1_dst = dn1_out ? dn1_out + frame_of(k) * (N1_POS * C1_OUT) : nullptr;
    // Phase 1: TMEM -> relu' mask -> packed bf16 in registers (one 2x2 block of dn1 per row).  Nothing is written yet: the
    // conv11 UMMAs of frame k-1 may still be reading the dn1 operand.
    uint32_t o[4][8];
    int p22[4];
    const int m = (t ? DG_TILE1 : 0) + 32 * qt + lane;
    const int Yh = m / G_W, Xh = m - Yh * G_W;
    const bool row_ok = (t == 0 || m >= 128) && m < DG_ROWS && Xh < 12;
#pragma unroll
    for (int cls = 0; cls < 4; ++cls) {
      uint32_t r[16];
      tc_ld16(tlane + TM_D12 + 64 * t + 16 * cls, r);
      const int y = 2 * Yh + (cls >> 1) - 1, xx = 2 * Xh + (cls & 1) - 1;
      p22[cls] = -1;
      if (row_ok && y >= 0 && y < H1 && xx >= 0 && xx < H1) {
        uint32_t mk[8];                                            // n1 of this pixel: relu'(n1) = (n1 > 0); post-ReLU values are >= 0
        lds128(*reinterpret_cast<uint32_t(*)[4]>(&mk[0]), b2 + (2 * cls) * B2_LBO + m * 16);
        lds128(*reinterpret_cast<uint32_t(*)[4]>(&mk[4]), b2 + (2 * cls + 1) * B2_LBO + m * 16);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const float lo = (mk[jj] & 0x7FFFu) ? __uint_as_float(r[2 * jj]) : 0.f;
          const float hi = (mk[jj] & 0x7FFF0000u) ? __uint_as_float(r[2 * jj + 1]) : 0.f;
          o[cls][jj] = pack_bf16(lo, hi);
          bacc[2 * jj] += bf16_lo(o[cls][jj]);
          bacc[2 * jj + 1] += bf16_hi(o[cls][jj]);
        }
        p22[cls] = y * BLK_W + xx;
        if (dn1_dst) {
          uint4* d = reinterpret_cast<uint4*>(dn1_dst + (y * H1 + xx) * C1_OUT);
          d[0] = make_uint4(o[cls][0], o[cls][1], o[cls][2], o[cls][3]);
          d[1] = make_uint4(o[cls][4], o[cls][5], o[cls][6], o[cls][7]);
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(FB_EPI12 + (k & 1)));           // D is drained and Blk2 has been read
    mark(43, k);
    // Phase 2: the operand buffer is free once every conv11 UMMA of frame k-1 has retired
    if (k > 0) mbar_wait(bar(FB_DN1FREE), (k - 1) & 1);
    mark(41, k);
#pragma unroll
    for (int cls = 0; cls < 4; ++cls) {
      if (p22[cls] >= 0) {
        const uint4 lo4 = make_uint4(o[cls][0], o[cls][1], o[cls][2], o[cls][3]), hi4 = make_uint4(o[cls][4], o[cls][5], o[cls][6], o[cls][7]);
        const uint32_t dst = dn1s + p22[cls] * 16;
#pragma unroll
        for (int ab = 0; ab < 4; ++ab) {                           // planes (a, b, half): the pixel's row moved down by 22a + b
          const uint32_t d = dst + (2 * ab) * DN1_PLANE + (BLK_W * (ab >> 1) + (ab & 1)) * 16;
          sts128(d, lo4);
          sts128(d + DN1_PLANE, hi4);
        }
      }
    }
    fence_proxy_async();                                           // the dn1 operand is read by the tensor core
    __syncwarp();
    if (lane == 0) mbar_arrive(bar(FB_DN1RDY));
    mark(42, k);
  };
  auto b11_partial = [&](int slot, const float (&bacc)[C1_OUT]) {   // warp-reduce the 16 channel sums of this warp
#pragma unroll
    for (int c = 0; c < C1_OUT; ++c) {
      float v = bacc[c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[slot * C1_OUT + c] = v;
    }
  };

  if (warp == FB_LOAD_WARP) {
    // =========================== Blk quarters -> ring ===========================
    const int n_q = n_frames * XB_QUARTERS;
    for (int qg = 0; qg < n_q; ++qg) {
      const int slot = qg % FB_RING, use = qg / FB_RING;
      mark(1, qg);
      if (use > 0) mbar_wait(bar(FB_QFREE + slot), (use - 1) & 1);
      mark(2, qg);
      if (elect_one()) {
        const int k = qg >> 2, q = qg & 3;
        mbar_expect_tx(bar(FB_QFULL + slot), XB_QBYTES);
        bulk_load_hint(ring + slot * XB_QBYTES, xblk + frame_of(k) * XB_FRAME_BYTES + q * XB_QBYTES, XB_QBYTES, bar(FB_QFULL + slot),
                       pol_last_use);
      }
      __syncwarp();
    }
  } else if (warp == FB_C12_WARP) {
    // =========================== G (two copies) / Blk2 of frame k into buffer k & 1 ===========================
    for (int k = 0; k < n_frames; ++k) {
      const int p = k & 1;
      mark(20, k);
      if (k >= 2) mbar_wait(bar(FB_EPI12 + p), ((k >> 1) - 1) & 1);   // UMMAs, mask reads and column sums of frame k-2 are done
      mark(21, k);
      if (elect_one()) {
        const uint32_t buf = c12 + p * C12_BYTES;
        mbar_expect_tx(bar(FB_C12RDY + p), 2 * G_BYTES - 16 + B2_BYTES);
        bulk_load(buf, dn2g + frame_of(k) * G_BYTES, G_BYTES, bar(FB_C12RDY + p));
        bulk_load_hint(buf + C12_G1 + 16, dn2g + frame_of(k) * G_BYTES, G_BYTES - 16, bar(FB_C12RDY + p), pol_last_use);   // the same, one row down
        bulk_load_hint(buf + C12_B2, n1b2 + frame_of(k) * B2_BYTES, B2_BYTES, bar(FB_C12RDY + p), pol_last_use);
      }
      __syncwarp();
    }
  } else if (warp == FB_ISSUE_WARP) {
    // =========================== MMA issuer ===========================
    // warp-uniform: all 32 lanes run the loops and wait on the barriers, elect_one() issues
    constexpr uint32_t idesc_dg = make_idesc_m(128, 64, false, false), idesc_w12 = make_idesc_m(64, 2 * C2_OUT, true, true),
                       idesc_w11 = make_idesc_m(64, 4 * C1_OUT, true, true);
    // descriptor low words of row 0 / k-chunk 0 of every operand; a shift of r rows is + r, a k-chunk plane is + LBO/16
    const uint32_t wd_k = desc_ns_lo(w12d, 1024);                                              // K-major: LBO = plane, SBO = 128
    const uint32_t ring_mn = desc_ns_lo(ring, 128), dn1_mn = desc_ns_lo(dn1s, 128);            // MN-major: LBO = 128, SBO = plane
    constexpr uint32_t hi_k = desc_ns_hi(128), hi_g = desc_ns_hi(G_LBO), hi_b2 = desc_ns_hi(B2_LBO), hi_ring = desc_ns_hi(XB_PLANE_BYTES),
                       hi_dn1 = desc_ns_hi(DN1_PLANE);
    mbar_wait(bar(FB_W12DRDY), 0);
    auto conv12_mmas = [&](int k) {
      const int p = k & 1;
      const uint32_t buf = c12 + p * C12_BYTES;
      const uint32_t g_k = desc_ns_lo(buf, G_LBO), g_mn = desc_ns_lo(buf, 128), b2_mn = desc_ns_lo(buf + C12_B2, 128);
      mark(10, k);
      mbar_wait(bar(FB_C12RDY + p), (k >> 1) & 1);                 // G / Blk2 of frame k have landed
      if (k > 0) mbar_wait(bar(FB_EPI12 + (p ^ 1)), ((k - 1) >> 1) & 1);   // D of frame k-1 has been drained
      mark(11, k);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int tap = 0; tap < 4; ++tap)
#pragma unroll
            for (int kk = 0; kk < 2; ++kk)
              tc_mma_bf16_w(tmem_base + TM_D12 + 64 * t,
                            g_k + ((t ? DG_TILE1 : 0) + G_W + 1 - G_W * (tap >> 1) - (tap & 1)) + 2 * kk * (G_LBO / 16), hi_k,
                            wd_k + (tap * 4096 + 2 * kk * 1024) / 16, hi_k, idesc_dg, (tap | kk) ? 1u : 0u);
        const uint32_t acc = k ? 1u : 0u;
#pragma unroll
        for (int s = 0; s < W12_KSTEPS; ++s)
#pragma unroll
          for (int a = 0; a < 2; ++a)
            // A: Blk2 rows 16 s .. (8 planes), B: G rows 16 s + 14 - 13 a .. in 8 planes (b, co chunk): G, then G moved down a row
            tc_mma_bf16_w(tmem_base + TM_W12 + 64 * a, b2_mn + 16 * s, hi_b2, g_mn + 16 * s + G_W + 1 - G_W * a, hi_g,
                          idesc_w12, s ? 1u : acc);
        tc_commit(bar(FB_MMA12));
      }
      __syncwarp();
      mark(12, k);
    };
    auto conv11_mmas = [&](int k) {
      mark(13, k);
      mbar_wait(bar(FB_DN1RDY), k & 1);
      mark(14, k);
#pragma unroll 1
      for (int q = 0; q < XB_QUARTERS; ++q) {
        const int qg = k * XB_QUARTERS + q, slot = qg % FB_RING;
        mbar_wait(bar(FB_QFULL + slot), (qg / FB_RING) & 1);
        mark(15, qg);
        tc_fence_after();
        if (elect_one()) {
          const int n_kk = q == 3 ? W11_KSTEPS - 24 : 8;
          for (int kk = 0; kk < n_kk; ++kk) {
            const int s = 8 * q + kk;
            // A: block rows 16 s .. of the quarter slot (8 planes), B: dn1 rows 16 s .. in the eight (a, b, half) planes
            tc_mma_bf16_w(tmem_base + TM_W11, ring_mn + slot * (XB_QBYTES / 16) + kk * 16, hi_ring, dn1_mn + 16 * s, hi_dn1,
                          idesc_w11, (k | s) ? 1u : 0u);
          }
          tc_commit(bar(FB_QFREE + slot));
          if (q == 3) tc_commit(bar(FB_DN1FREE));
        }
        __syncwarp();
        mark(16, qg);
      }
    };
    if (n_frames > 0) conv12_mmas(0);
    if (n_frames > 1) conv12_mmas(1);
    for (int k = 0; k < n_frames; ++k) {
      conv11_mmas(k);
      if (k + 2 < n_frames) conv12_mmas(k + 2);                    // two frames ahead: its epilogue runs under the next conv11 gradient
    }
    if (elect_one()) tc_commit(bar(FB_DONE));
    __syncwarp();
  } else if (warp >= FB_IDLE_WARP0) {
    // no role: straight to the final barrier (kept out of the "warp >= 8" bias branch below)
  } else if (warp == FB_T1_WARP) {
    // =========================== second data-gradient tile ===========================
    if (!w12d_early) build_w12d();
    float bacc11[C1_OUT];
#pragma unroll
    for (int c = 0; c < C1_OUT; ++c) bacc11[c] = 0.f;
    for (int k = 0; k < n_frames; ++k) dgrad_epilogue(k, 1, 3, bacc11);
    b11_partial(4, bacc11);
  } else if (warp == 3 || warp >= 8) {
    // =========================== conv12 bias gradient: column sums of G ===========================
    // warp -> chunk plane j (8 channels), lane -> row phase: 16-byte rows, conflict-free; border rows are zero
    if (!w12d_early) build_w12d();
    const int j = warp == 3 ? 3 : warp - 8;
    float acc8[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc8[e] = 0.f;
    for (int k = 0; k < n_frames; ++k) {
      const int p = k & 1;
      mbar_wait(bar(FB_C12RDY + p), (k >> 1) & 1);
      mark(30, k);
      const uint32_t plane = c12 + p * C12_BYTES + j * G_LBO;
      for (int row = lane; row < G_ROWS; row += 32) {
        uint32_t v[4];
        lds128(v, plane + row * 16);
#pragma unroll
        for (int e = 0; e < 4; ++e) { acc8[2 * e] += bf16_lo(v[e]); acc8[2 * e + 1] += bf16_hi(v[e]); }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(FB_EPI12 + p));
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v = acc8[e];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) g_b12[(int64_t)blockIdx.x * gp_stride + 8 * j + e] = v;
    }
  } else {
    // =========================== data-gradient epilogue; final store ===========================
    if (!w12d_early) build_w12d();
    const int ew = warp - FB_EPI_WARP0;                            // TMEM lane quarter
    const uint32_t tlane = tmem_base + ((uint32_t)(ew * 32) << 16);
    float bacc[C1_OUT];                                            // db11 partials of this thread's pixels
#pragma unroll
    for (int c = 0; c < C1_OUT; ++c) bacc[c] = 0.f;
    for (int k = 0; k < n_frames; ++k) dgrad_epilogue(k, 0, ew, bacc);
    b11_partial(ew, bacc);                                         // summed with warp 11's after the final block barrier
    if (n_frames > 0) {
      mbar_wait(bar(FB_DONE), 0);
      mark(54, 0);
      tc_fence_after();
      float* const s11 = g_w11 + (int64_t)blockIdx.x * gp_stride;
      float* const s12 = g_w12 + (int64_t)blockIdx.x * gp_stride;
      // the accumulators have M = 64: rows sit on TMEM lanes 32 w + (0..15) (rows 16 w ..); row = chunk plane j * 8 + e
      const int row = 16 * ew + lane, j = row >> 3, e = row & 7;
#pragma unroll 1
      for (int q = 0; q < 4; ++q) {                                // conv11: columns 16 q .. of quadrant q = a*2 + b
        uint32_t r[16];
        tc_ld16(tlane + TM_W11 + 16 * q, r);
        if (lane < 16) {
          // conv11 block element: j = dy*2 + (dx>>1), e = (dx&1)*4 + c
          const int kh = 4 * (q >> 1) + (j >> 1), kw = 4 * (q & 1) + (j & 1) * 2 + (e >> 2), c = e & 3;
          float4* o = reinterpret_cast<float4*>(s11 + ((kh * 8 + kw) * 4 + c) * C1_OUT);
#pragma unroll
          for (int n = 0; n < C1_OUT / 4; ++n)
            o[n] = make_float4(__uint_as_float(r[4 * n]), __uint_as_float(r[4 * n + 1]), __uint_as_float(r[4 * n + 2]),
                               __uint_as_float(r[4 * n + 3]));
        }
      }
#pragma unroll 1
      for (int q = 0; q < 4; ++q)                                  // conv12: accumulator a = q >> 1, columns 32 b .. (b = q & 1)
#pragma unroll 1
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t r[16];
          tc_ld16(tlane + TM_W12 + 64 * (q >> 1) + 32 * (q & 1) + 16 * hh, r);
          if (lane < 16) {
            // conv12 block element: j = (dy*2 + dx)*2 + (ci>>3), e = ci & 7
            const int kh = 2 * (q >> 1) + (j >> 2), kw = 2 * (q & 1) + ((j >> 1) & 1), ci = (j & 1) * 8 + e;
            float4* o = reinterpret_cast<float4*>(s12 + ((kh * 4 + kw) * C1_OUT + ci) * C2_OUT + 16 * hh);
#pragma unroll
            for (int n = 0; n < 4; ++n)
              o[n] = make_float4(__uint_as_float(r[4 * n]), __uint_as_float(r[4 * n + 1]), __uint_as_float(r[4 * n + 2]),
                                 __uint_as_float(r[4 * n + 3]));
          }
        }
    }
  }

  mark(52, 0);
  tc_fence_before();
  __syncthreads();
  if (tid < C1_OUT)                                                // conv11 bias gradient: the five warp partials in a fixed order
    g_b11[(int64_t)blockIdx.x * gp_stride + tid] =
        red[tid] + red[C1_OUT + tid] + red[2 * C1_OUT + tid] + red[3 * C1_OUT + tid] + red[4 * C1_OUT + tid];
  trace_mark(K_CONV12_BWD, 2);
  if (warp == FB_EPI_WARP0) {
    tc_fence_after();
    tmem_dealloc<FB_TMEM_COLS>(tmem_base);
  }
}

GA3C_TRACE_ATTACH(trace_attach_conv_bwd_fused)
static bool g_evt_attached = false;     // host side: the event-log instantiation is launched only while a log is attached
int evt_attach_conv_bwd(unsigned long long* buf) {
  g_evt_attached = buf != nullptr;
  return (int)cudaMemcpyToSymbol(g_evt, &buf, sizeof(buf));
}

int conv_bwd_grid(int batch, int num_sms) { return min(batch, num_sms); }

int configure_conv_bwd_fused() {
  cudaError_t e = cudaFuncSetAttribute(conv_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FB_SMEM);
  if (e != cudaSuccess) return (int)e;
  return (int)cudaFuncSetAttribute(conv_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FB_SMEM);
}

int launch_conv_bwd(const uint8_t* xblk, const uint8_t* n1b2, const uint8_t* dn2g, const float* w12, uint16_t* dn1_out,
                    float* g_w11, float* g_b11, float* g_w12, float* g_b12, int64_t gp_stride, int batch, int num_sms, bool x_u8,
                    cudaStream_t stream) {
  const dim3 grid(conv_bwd_grid(batch, num_sms));
  if (grid.x == 0) return 0;
  auto kernel = g_evt_attached ? conv_bwd_kernel<true> : conv_bwd_kernel<false>;
  return launch_pdl(kernel, grid, dim3(FB_THREADS), FB_SMEM, stream, xblk, n1b2, dn2g, w12, dn1_out, g_w11, g_b11, g_w12, g_b12,
                    gp_stride, batch, l2_hints(true, x_u8) | (batch >= num_sms ? 8 : 0));
}

}  // namespace ga3c
