// dense1 GEMMs on the 5th-generation tensor cores: tcgen05.mma with TMEM accumulators, operands
// staged in shared memory by TMA (cp.async.bulk.tensor, SWIZZLE_128B), mbarrier pipeline, warp roles.
//
// Reference ops: dense1 = relu(flat @ w + b) (NetworkDNav.py:90, dense_layer :256-269) and the two
// matmul gradients TF autodiff derives from it (opt.minimize, NetworkVP_discrate.py:130).
//
//   fwd  : part[s][B,256]  = n2[B,3872]    x w1[3872,256]           (A K-major,  B MN-major)  split-K
//   dgrad: dn2[B,3872]     = dd1[B,256]    x w1[3872,256]^T  ⊙ n2>0 (A K-major,  B K-major)
//   wgrad: g_w1[3872,256]  = n2[B,3872]^T  x dd1[B,256]             (A MN-major, B MN-major)
//
// The GEMM core (warp roles, pipeline, tensor maps) is gemm_tc.cuh.  The 84x84x4 trunk passes K = FLAT = 3872; the generic
// trunk (conv_gen.cu) passes its own K = H2 * W2 * 32 and takes dn2 row-major (EpiReluMaskBf16Row) instead of in G.
#include <cstdio>
#include <cstdlib>

#include "gemm_tc.cuh"

namespace ga3c {

struct EpiReluMaskBf16Tc {  // dn2 = acc where n2 > 0 else 0, bf16, stored in the G operand layout the conv backward consumes (common.cuh)
  uint8_t* out; const uint16_t* act; int ldc;
  struct Pre { uint4 a[4]; };     // this thread's 32 activations: fetched while the MMAs are still running
  __device__ __forceinline__ void prefetch(Pre& p, int m, int n, bool ok) const {
    const uint4* a = reinterpret_cast<const uint4*>(act + (size_t)m * ldc + n);
#pragma unroll
    for (int i = 0; i < 4; ++i) p.a[i] = ok ? a[i] : make_uint4(0, 0, 0, 0);
  }
  __device__ __forceinline__ void operator()(const Pre& p, int, int m, int n, const uint32_t (&r)[32]) const {
    // the 32 columns are the 32 channels of ONE conv12 output position: four 16-byte chunks, one per chunk plane of frame m's G
    const int pos = n >> 5, oy = pos / H2, ox = pos - oy * H2;
    uint8_t* dst0 = out + (size_t)m * G_BYTES + g_pos_offset(oy, ox, 0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint4 av = p.a[i];
      const uint32_t aw[4] = {av.x, av.y, av.z, av.w};
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        // post-ReLU activations are never negative: "> 0" == any magnitude bit set
        const float lo = (aw[j] & 0x7FFFu) ? __uint_as_float(r[8 * i + 2 * j]) : 0.f;
        const float hi = (aw[j] & 0x7FFF0000u) ? __uint_as_float(r[8 * i + 2 * j + 1]) : 0.f;
        o[j] = pack_bf16(lo, hi);
      }
      *reinterpret_cast<uint4*>(dst0 + i * G_LBO) = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
};


struct EpiReluMaskBf16Row { // generic trunk: dn2 = acc where n2 > 0 else 0, bf16, row-major [B][K] like n2
  uint16_t* out; const uint16_t* act; int ldc;
  struct Pre { uint4 a[4]; };
  __device__ __forceinline__ void prefetch(Pre& p, int m, int n, bool ok) const {
    const uint4* a = reinterpret_cast<const uint4*>(act + (size_t)m * ldc + n);
#pragma unroll
    for (int i = 0; i < 4; ++i) p.a[i] = ok ? a[i] : make_uint4(0, 0, 0, 0);
  }
  __device__ __forceinline__ void operator()(const Pre& p, int, int m, int n, const uint32_t (&r)[32]) const {
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)m * ldc + n);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t aw[4] = {p.a[i].x, p.a[i].y, p.a[i].z, p.a[i].w};
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float lo = (aw[j] & 0x7FFFu) ? __uint_as_float(r[8 * i + 2 * j]) : 0.f;
        const float hi = (aw[j] & 0x7FFF0000u) ? __uint_as_float(r[8 * i + 2 * j + 1]) : 0.f;
        o[j] = pack_bf16(lo, hi);
      }
      dst[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
};

// dense1 backward in ONE launch: both GEMMs only need dd1, so their tiles share a grid.  Blocks [0, n_dg) are the
// data-gradient tiles (first: conv12_bwd waits for dn2), the rest the weight-gradient tiles (needed at the step's end).
constexpr int DG_BN = 128, DG_ST = 2;       // dgrad: M = B,   N = K (3872), K = 256
constexpr int WG_BN = 64, WG_ST = 4;        // wgrad: M = K (3872), N = 256, K = B
constexpr int WGM_ST = 3;                   // wgrad inside the merged launch: 3 stages -> 3 CTAs per SM, one wave
template <class EpiDg>
struct DenseBwdArgs {
  int batch, kdim, dg_mtiles, n_dg, wg_mtiles, wg_kblocks;
  EpiDg epi_dg;
  EpiPartialF32 epi_wg;
};
template <class EpiDg>
__global__ void __launch_bounds__(TC_THREADS, 3)     // <= 96 registers: 18 warps fit the four 16K register files
dense_bwd_kernel(const __grid_constant__ CUtensorMap dg_a, const __grid_constant__ CUtensorMap dg_b,
                 const __grid_constant__ CUtensorMap wg_a, const __grid_constant__ CUtensorMap wg_b, const DenseBwdArgs<EpiDg> p) {
  const int b = blockIdx.x;
  if (b < p.n_dg) {
    gemm_tc_body<DG_BN, DG_ST, false, false, EpiDg>(dg_a, dg_b, p.batch, p.kdim, FC / TC_BK, FC / TC_BK,
                                                    p.epi_dg, b % p.dg_mtiles, b / p.dg_mtiles, 0);
  } else {
    const int t = b - p.n_dg;
    gemm_tc_body<WG_BN, WGM_ST, true, true, EpiPartialF32>(wg_a, wg_b, p.kdim, (int)FC, p.wg_kblocks, p.wg_kblocks,
                                                           p.epi_wg, t % p.wg_mtiles, t / p.wg_mtiles, 0);
  }
}

GA3C_TRACE_ATTACH(trace_attach_dense_tc)
GA3C_EVT_ATTACH(evt_attach_dense_tc)


constexpr int FWD_BN = 128, FWD_ST = 4;     // fwd : M = B,    N = 256,  K = 3872  (split-K)
constexpr int DBW_SMEM = tc_smem<DG_BN, DG_ST>() > tc_smem<WG_BN, WGM_ST>() ? tc_smem<DG_BN, DG_ST>() : tc_smem<WG_BN, WGM_ST>();

template <class EpiDg>
static int configure_dense_bwd() {
  cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<DG_BN, DG_ST, false, false, EpiDg>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<DG_BN, DG_ST>());
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(dense_bwd_kernel<EpiDg>, cudaFuncAttributeMaxDynamicSharedMemorySize, DBW_SMEM);
  if (e != cudaSuccess) return (int)e;
  // 3 CTAs per SM (all dgrad + wgrad tiles in one wave) need the full shared-memory carveout
  return (int)cudaFuncSetAttribute(dense_bwd_kernel<EpiDg>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                   cudaSharedmemCarveoutMaxShared);
}

int configure_dense_tc() {
  cudaError_t e;
  e = cudaFuncSetAttribute(gemm_tc_kernel<FWD_BN, FWD_ST, false, true, EpiPartialF32>,
                           cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<FWD_BN, FWD_ST>());
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(gemm_tc_kernel<WG_BN, WG_ST, true, true, EpiPartialF32>,
                           cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<WG_BN, WG_ST>());
  if (e != cudaSuccess) return (int)e;
  if (int r = configure_dense_bwd<EpiReluMaskBf16Tc>()) return r;
  if (int r = configure_dense_bwd<EpiReluMaskBf16Row>()) return r;
  if (getenv("GA3C_DEBUG_OCC")) {
    auto* const kern = dense_bwd_kernel<EpiReluMaskBf16Tc>;
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, TC_THREADS, DBW_SMEM);
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, kern);
    int smem_sm = 0, regs_sm = 0, dev = 0, resv = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&resv, cudaDevAttrReservedSharedMemoryPerBlock, dev);
    fprintf(stderr, "[ga3c] dense_bwd_kernel: %d CTAs/SM at %d B dynamic smem; regs %d static smem %zu maxdyn %d carveout %d; SM smem %d regs %d reserved/block %d\n",
            nb, DBW_SMEM, fa.numRegs, fa.sharedSizeBytes, fa.maxDynamicSharedSizeBytes, fa.preferredShmemCarveout, smem_sm, regs_sm, resv);
    for (int sm = 16384; sm <= 114688; sm += 16384) {
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, TC_THREADS, sm);
      fprintf(stderr, "[ga3c]   dyn smem %d -> %d CTAs/SM\n", sm, nb);
    }
  }
  return 0;
}

int dense_fwd_splits(int batch, int num_sms, int kdim) {
  const int tiles = ((batch + TC_BM - 1) / TC_BM) * (FC / FWD_BN);
  const int kblocks = (kdim + TC_BK - 1) / TC_BK;                 // 61 at 84x84x4
  int s = num_sms / tiles;
  if (s < 1) s = 1;
  if (s > 16) s = 16;
  const int per = (kblocks + s - 1) / s;
  return (kblocks + per - 1) / per;                               // no empty splits
}

int launch_dense_fwd_tc(const uint16_t* n2, const uint16_t* w1bf, float* d1_part, int batch, int kdim, int splits,
                        cudaStream_t stream, const DpGate* gate) {
  CUtensorMap ta, tb;
  if (make_tmap(&ta, n2, batch, kdim, kdim, TC_BM)) return (int)cudaErrorInvalidValue;        // A: [B][K], K inner
  if (make_tmap(&tb, w1bf, kdim, FC, FC, 64)) return (int)cudaErrorInvalidValue;              // B: [K][256], N inner
  const int kblocks = (kdim + TC_BK - 1) / TC_BK;
  const int per = (kblocks + splits - 1) / splits;
  dim3 grid((batch + TC_BM - 1) / TC_BM, FC / FWD_BN, splits);
  return launch_pdl(gemm_tc_kernel<FWD_BN, FWD_ST, false, true, EpiPartialF32>, grid, dim3(TC_THREADS),
                    tc_smem<FWD_BN, FWD_ST>(), stream, ta, tb, batch, (int)FC, kblocks, per,
                    EpiPartialF32{d1_part, FC, (int64_t)batch * FC}, gate ? *gate : DpGate{});
}

template <class EpiDg, class Out>
static int dense_dgrad(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, Out* dn2, int batch, int kdim,
                       cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (make_tmap(&ta, dd1, batch, FC, FC, TC_BM)) return (int)cudaErrorInvalidValue;           // A: [B][256], K inner
  if (make_tmap(&tb, w1bf, kdim, FC, FC, DG_BN)) return (int)cudaErrorInvalidValue;           // B: [K][256] = [N][K]
  dim3 grid((batch + TC_BM - 1) / TC_BM, (kdim + DG_BN - 1) / DG_BN, 1);
  return launch_pdl(gemm_tc_kernel<DG_BN, DG_ST, false, false, EpiDg>, grid, dim3(TC_THREADS),
                    tc_smem<DG_BN, DG_ST>(), stream, ta, tb, batch, kdim, FC / TC_BK, FC / TC_BK,
                    EpiDg{dn2, n2, kdim}, DpGate{});
}
int launch_dense_dgrad_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint8_t* dn2, int batch,
                          cudaStream_t stream) {
  return dense_dgrad<EpiReluMaskBf16Tc>(dd1, w1bf, n2, dn2, batch, (int)FLAT, stream);
}
int launch_dense_dgrad_rows_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint16_t* dn2, int batch,
                               int kdim, cudaStream_t stream) {
  return dense_dgrad<EpiReluMaskBf16Row>(dd1, w1bf, n2, dn2, batch, kdim, stream);
}

int launch_dense_wgrad_tc(const uint16_t* n2, const uint16_t* dd1, float* g_w1, int batch, int kdim, cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (make_tmap(&ta, n2, batch, kdim, kdim, 64)) return (int)cudaErrorInvalidValue;           // A: [K=B][M=K], M inner
  if (make_tmap(&tb, dd1, batch, FC, FC, 64)) return (int)cudaErrorInvalidValue;              // B: [K=B][N=256],  N inner
  const int kblocks = (batch + TC_BK - 1) / TC_BK;
  dim3 grid((kdim + TC_BM - 1) / TC_BM, FC / WG_BN, 1);
  return launch_pdl(gemm_tc_kernel<WG_BN, WG_ST, true, true, EpiPartialF32>, grid, dim3(TC_THREADS),
                    tc_smem<WG_BN, WG_ST>(), stream, ta, tb, kdim, (int)FC, kblocks, kblocks,
                    EpiPartialF32{g_w1, FC, 0}, DpGate{});
}

template <class EpiDg, class Out>
static int dense_bwd(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, Out* dn2, float* g_w1, int batch, int kdim,
                     cudaStream_t stream) {
  CUtensorMap da, db, wa, wb;
  if (make_tmap(&da, dd1, batch, FC, FC, TC_BM)) return (int)cudaErrorInvalidValue;           // dgrad A: [B][256], K inner
  if (make_tmap(&db, w1bf, kdim, FC, FC, DG_BN)) return (int)cudaErrorInvalidValue;           // dgrad B: [K][256] = [N][K]
  if (make_tmap(&wa, n2, batch, kdim, kdim, 64)) return (int)cudaErrorInvalidValue;           // wgrad A: [K=B][M=K], M inner
  if (make_tmap(&wb, dd1, batch, FC, FC, 64)) return (int)cudaErrorInvalidValue;              // wgrad B: [K=B][N=256],  N inner
  DenseBwdArgs<EpiDg> p{};
  p.batch = batch;
  p.kdim = kdim;
  p.dg_mtiles = (batch + TC_BM - 1) / TC_BM;
  p.n_dg = p.dg_mtiles * ((kdim + DG_BN - 1) / DG_BN);
  p.wg_mtiles = (kdim + TC_BM - 1) / TC_BM;
  p.wg_kblocks = (batch + TC_BK - 1) / TC_BK;
  p.epi_dg = EpiDg{dn2, n2, kdim};
  p.epi_wg = EpiPartialF32{g_w1, FC, 0};
  const int grid = p.n_dg + p.wg_mtiles * (FC / WG_BN);
  return launch_pdl(dense_bwd_kernel<EpiDg>, dim3(grid), dim3(TC_THREADS), DBW_SMEM, stream, da, db, wa, wb, p);
}
int launch_dense_bwd_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint8_t* dn2, float* g_w1, int batch,
                        cudaStream_t stream) {
  return dense_bwd<EpiReluMaskBf16Tc>(dd1, w1bf, n2, dn2, g_w1, batch, (int)FLAT, stream);
}
int launch_dense_bwd_rows_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint16_t* dn2, float* g_w1,
                             int batch, int kdim, cudaStream_t stream) {
  return dense_bwd<EpiReluMaskBf16Row>(dd1, w1bf, n2, dn2, g_w1, batch, kdim, stream);
}

}  // namespace ga3c
