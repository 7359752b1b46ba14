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
// One output tile (128 x BN, fp32 in BN TMEM columns) per CTA.  192 threads:
//   warp 0   TMA producer (one elected lane)
//   warp 1   TMEM allocator + MMA issuer (one elected lane issues tcgen05.mma.cta_group::1.kind::f16)
//   warp 2-5 epilogue: tcgen05.ld 32 lanes x 32 columns -> registers -> fused epilogue -> global
// K is consumed in blocks of 64 (one 128-byte swizzle row); a k-block is 4 MMAs of K = 16.
#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "tcgen05.cuh"
#include "dp_exchange.cuh"

namespace ga3c {

constexpr int TC_BK = 64, TC_THREADS = 192;
constexpr int TC_A_STAGE = TC_BM * TC_BK * 2;                       // 16 KB

// Debug build only (GA3C_NVCC_EXTRA=-DGA3C_DENSE_EVT, tools/evt_dense.py): lane 0 of every warp of the first tile of each GEMM
// logs {globaltimer, event, k-block} into the event buffer of ga3c_evt_* -- regions 0-5 forward, 6-11 data gradient, 12-15
// weight gradient (warps 0-3).  The production build carries none of it.
#ifdef GA3C_DENSE_EVT
#define DEVT(id, arg) evt_mark_region(ev, ev_region, id, arg)
__device__ __forceinline__ void evt_mark_region(EvtLog& l, int region, int id, int arg) {
  if (l.base != nullptr && l.i < EVT_PER_WARP) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(now));
    const unsigned int slot = region * EVT_PER_WARP + l.i++;
    l.base[2 * slot] = now;
    l.base[2 * slot + 1] = ((unsigned long long)region << 32) | ((unsigned long long)id << 16) | (unsigned long long)(arg & 0xFFFF);
  }
}
#else
#define DEVT(id, arg) do { } while (0)
#endif

// ---- PTX wrappers -------------------------------------------------------------------------------
// ---- epilogues: one thread owns one output row and 32 consecutive columns ------------------------
struct EpiPartialF32 {      // raw fp32 tile into part[split][M][N]  (bias + relu are applied by the consumer)
  float* out; int ldc; int64_t split_stride;
  struct Pre {};
  __device__ __forceinline__ void prefetch(Pre&, int, int, bool) const {}
  __device__ __forceinline__ void operator()(const Pre&, int split, int m, int n, const uint32_t (&r)[32]) const {
    float4* dst = reinterpret_cast<float4*>(out + split * split_stride + (size_t)m * ldc + n);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      dst[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]),
                           __uint_as_float(r[4 * i + 3]));
  }
};
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

// gate (dense1 forward, data parallel with the side-stream exchange): the B operand is the bf16 shadow of dense1/w, whose slices
// the ranks' exchange kernels of the PREVIOUS step store into this rank's slab.  Instead of a stream-level event wait in front
// of this launch (which takes the launch out of the programmatic-dependent-launch chain: +3.6 us per step, measured) the TMA
// producer warp looks at the "slice of rank r landed everywhere" flags in this rank's own comm block -- pushed there long ago in
// the normal case -- before its first load.  The exchange grid it might wait for only ever waits for other GPUs and has been
// resident since the previous step's conv backward, so the wait cannot keep it off an SM.
template <int BN, int STAGES, bool A_MN, bool B_MN, class Epi>
__device__ __forceinline__ void gemm_tc_body(const CUtensorMap& tm_a, const CUtensorMap& tm_b, int M, int N, int k_blocks,
                                             int k_blocks_per_split, const Epi& epi, int bx, int by, int bz,
                                             const DpGate* gate = nullptr) {
  constexpr int B_STAGE = BN * TC_BK * 2;
  constexpr int STAGE = TC_A_STAGE + B_STAGE;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B atoms need 1024-byte alignment
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = sbase + STAGES * STAGE;            // full[STAGES], empty[STAGES], tmem_full : 8 B each
  const uint32_t tmem_slot = bars + (2 * STAGES + 1) * 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = bx * TC_BM, n0 = by * BN, split = bz;
  const int kb0 = split * k_blocks_per_split;
  const int kb1 = min(kb0 + k_blocks_per_split, k_blocks);
#ifdef GA3C_DENSE_EVT
  const int ev_region = (A_MN ? 12 : (B_MN ? 0 : 6)) + warp;
  EvtLog ev;
  ev.base = ((bx | by | bz) == 0 && lane == 0 && (!A_MN || warp < 4)) ? g_evt : nullptr;
  ev.i = 0;
#endif

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tm_a));
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tm_b));
    for (int s = 0; s < STAGES; ++s) { mbar_init(bars + s * 8, 1); mbar_init(bars + (STAGES + s) * 8, 1); }
    mbar_init(bars + 2 * STAGES * 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tmem_slot), "n"(BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  griddep_launch();             // every CTA of this grid holds its TMEM columns and shared memory
  constexpr int kid = A_MN ? K_DENSE_WGRAD : (B_MN ? K_DENSE_FWD : K_DENSE_DGRAD);
  griddep_wait(kid);            // operands are produced by the preceding kernels
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(tmem_base) : "r"(tmem_slot));
  DEVT(0, 0);

  // producer and issuer run warp-uniform (all lanes loop and wait, elect_one() issues): descriptors and TMA coordinates
  // stay in uniform registers instead of going through R2UR inside an ELECT retry loop
  if (warp == 0) {
    if (gate != nullptr && gate->flags != nullptr) {
      if (lane < gate->world)
        dp_wait_flag_acquire(gate->flags + 64 * lane, gate->step, gate->err, 16u);
      __syncwarp();
      asm volatile("fence.proxy.async;\n" ::: "memory");      // the shadow was written through the generic proxy, TMA reads it
    }
    for (int kb = kb0; kb < kb1; ++kb) {
      const int it = kb - kb0, s = it % STAGES;
      mbar_wait(bars + (STAGES + s) * 8, ((it / STAGES) & 1) ^ 1);          // slot free
      DEVT(1, kb);
      if (elect_one()) {
        const uint32_t full = bars + s * 8, sa = sbase + s * STAGE, sb = sa + TC_A_STAGE;
        mbar_expect_tx(full, STAGE);
        if (A_MN) {
          tma_load_2d(sa, &tm_a, m0, kb * TC_BK, full);
          tma_load_2d(sa + 8192, &tm_a, m0 + 64, kb * TC_BK, full);
        } else {
          tma_load_2d(sa, &tm_a, kb * TC_BK, m0, full);
        }
        if (B_MN) {
#pragma unroll
          for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, &tm_b, n0 + 64 * j, kb * TC_BK, full);
        } else {
          tma_load_2d(sb, &tm_b, kb * TC_BK, n0, full);
        }
      }
      __syncwarp();
      DEVT(2, kb);
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(BN, A_MN, B_MN);
    for (int kb = kb0; kb < kb1; ++kb) {
      const int it = kb - kb0, s = it % STAGES;
      mbar_wait(bars + s * 8, (it / STAGES) & 1);                           // TMA bytes landed
      DEVT(3, kb);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t sa = sbase + s * STAGE, sb = sa + TC_A_STAGE;
        const uint64_t da = make_desc(sa, A_MN), db = make_desc(sb, B_MN);
#pragma unroll
        for (int k = 0; k < TC_BK / 16; ++k) {
          // advance K by 16: +32 B inside the 128-B swizzle row (K-major), +2 k-atoms = 2048 B (MN-major)
          const uint64_t ka = (uint64_t)((A_MN ? 2048u : 32u) * k >> 4), kbv = (uint64_t)((B_MN ? 2048u : 32u) * k >> 4);
          tc_mma_bf16(tmem_base, da + ka, db + kbv, idesc, (it > 0 || k > 0) ? 1u : 0u);
        }
        tc_commit(bars + (STAGES + s) * 8);                                  // frees the slot when the MMAs retire
      }
      __syncwarp();
      DEVT(4, kb);
    }
    if (elect_one()) tc_commit(bars + 2 * STAGES * 8);                       // accumulator complete
    __syncwarp();
  } else {
    const int q = warp & 3;                       // TMEM lane quarter this warp may read
    const int m = m0 + q * 32 + lane;
    typename Epi::Pre pre[BN / 32];               // epilogue inputs from global memory, loaded under the MMAs
#pragma unroll
    for (int c = 0; c < BN / 32; ++c) epi.prefetch(pre[c], m, n0 + c * 32, m < M && n0 + c * 32 < N);
    DEVT(5, 0);
    mbar_wait(bars + 2 * STAGES * 8, 0);
    DEVT(6, 0);
    tc_fence_after();
#pragma unroll
    for (int c = 0; c < BN / 32; ++c) {
      uint32_t r[32];
      tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + c * 32, r);
      const int n = n0 + c * 32;
      if (m < M && n < N) epi(pre[c], split, m, n, r);
      DEVT(7, c);
    }
  }
  tc_fence_before();
  __syncthreads();
  DEVT(8, 0);
  trace_mark(kid, 2);
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(BN) : "memory");
  }
}

template <int BN, int STAGES, bool A_MN, bool B_MN, class Epi>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, int M, int N,
               int k_blocks, int k_blocks_per_split, Epi epi, const DpGate gate) {
  gemm_tc_body<BN, STAGES, A_MN, B_MN, Epi>(tm_a, tm_b, M, N, k_blocks, k_blocks_per_split, epi, blockIdx.x, blockIdx.y,
                                            blockIdx.z, &gate);
}

// dense1 backward in ONE launch: both GEMMs only need dd1, so their tiles share a grid.  Blocks [0, n_dg) are the
// data-gradient tiles (first: conv12_bwd waits for dn2), the rest the weight-gradient tiles (needed at the step's end).
constexpr int DG_BN = 128, DG_ST = 2;       // dgrad: M = B,   N = 3872, K = 256
constexpr int WG_BN = 64, WG_ST = 4;        // wgrad: M = 3872, N = 256, K = B
constexpr int WGM_ST = 3;                   // wgrad inside the merged launch: 3 stages -> 3 CTAs per SM, one wave
struct DenseBwdArgs {
  int batch, dg_mtiles, n_dg, wg_mtiles, wg_kblocks;
  EpiReluMaskBf16Tc epi_dg;
  EpiPartialF32 epi_wg;
};
__global__ void __launch_bounds__(TC_THREADS, 3)     // <= 96 registers: 18 warps fit the four 16K register files
dense_bwd_kernel(const __grid_constant__ CUtensorMap dg_a, const __grid_constant__ CUtensorMap dg_b,
                 const __grid_constant__ CUtensorMap wg_a, const __grid_constant__ CUtensorMap wg_b, const DenseBwdArgs p) {
  const int b = blockIdx.x;
  if (b < p.n_dg) {
    gemm_tc_body<DG_BN, DG_ST, false, false, EpiReluMaskBf16Tc>(dg_a, dg_b, p.batch, (int)FLAT, FC / TC_BK, FC / TC_BK,
                                                                p.epi_dg, b % p.dg_mtiles, b / p.dg_mtiles, 0);
  } else {
    const int t = b - p.n_dg;
    gemm_tc_body<WG_BN, WGM_ST, true, true, EpiPartialF32>(wg_a, wg_b, (int)FLAT, (int)FC, p.wg_kblocks, p.wg_kblocks,
                                                           p.epi_wg, t % p.wg_mtiles, t / p.wg_mtiles, 0);
  }
}

GA3C_TRACE_ATTACH(trace_attach_dense_tc)
GA3C_EVT_ATTACH(evt_attach_dense_tc)

// ---- host side ----------------------------------------------------------------------------------
// 2-D bf16 row-major matrix [rows][cols] (ld elements between rows), box = 64 inner x box_rows, 128-B swizzle,
// out-of-bounds elements read as zero (ragged M / N / K tails need no special casing in the kernel).
// cuTensorMapEncodeTiled is resolved through the runtime (cudaGetDriverEntryPoint) so the library has no
// link-time dependency on libcuda.so.1 and still loads on a box without a driver (symbol-export test).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

static int make_tmap(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  EncodeTiledFn cuTensorMapEncodeTiled = encode_tiled_fn();
  if (!cuTensorMapEncodeTiled) return (int)cudaErrorNotSupported;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = cuTensorMapEncodeTiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                                      estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

template <int BN, int STAGES>
constexpr int tc_smem() { return STAGES * (TC_A_STAGE + BN * TC_BK * 2) + (2 * STAGES + 1) * 8 + 16 + 1024; }

constexpr int FWD_BN = 128, FWD_ST = 4;     // fwd : M = B,    N = 256,  K = 3872  (split-K)
constexpr int DBW_SMEM = tc_smem<DG_BN, DG_ST>() > tc_smem<WG_BN, WGM_ST>() ? tc_smem<DG_BN, DG_ST>() : tc_smem<WG_BN, WGM_ST>();

using FwdKernel = decltype(&gemm_tc_kernel<FWD_BN, FWD_ST, false, true, EpiPartialF32>);

int configure_dense_tc() {
  cudaError_t e;
  e = cudaFuncSetAttribute(gemm_tc_kernel<FWD_BN, FWD_ST, false, true, EpiPartialF32>,
                           cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<FWD_BN, FWD_ST>());
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(gemm_tc_kernel<DG_BN, DG_ST, false, false, EpiReluMaskBf16Tc>,
                           cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<DG_BN, DG_ST>());
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(gemm_tc_kernel<WG_BN, WG_ST, true, true, EpiPartialF32>,
                           cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<WG_BN, WG_ST>());
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(dense_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DBW_SMEM);
  if (e != cudaSuccess) return (int)e;
  // 3 CTAs per SM (all dgrad + wgrad tiles in one wave) need the full shared-memory carveout
  e = cudaFuncSetAttribute(dense_bwd_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return (int)e;
  if (getenv("GA3C_DEBUG_OCC")) {
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, dense_bwd_kernel, TC_THREADS, DBW_SMEM);
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, dense_bwd_kernel);
    int smem_sm = 0, regs_sm = 0, dev = 0, resv = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&resv, cudaDevAttrReservedSharedMemoryPerBlock, dev);
    fprintf(stderr, "[ga3c] dense_bwd_kernel: %d CTAs/SM at %d B dynamic smem; regs %d static smem %zu maxdyn %d carveout %d; SM smem %d regs %d reserved/block %d\n",
            nb, DBW_SMEM, fa.numRegs, fa.sharedSizeBytes, fa.maxDynamicSharedSizeBytes, fa.preferredShmemCarveout, smem_sm, regs_sm, resv);
    for (int sm = 16384; sm <= 114688; sm += 16384) {
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, dense_bwd_kernel, TC_THREADS, sm);
      fprintf(stderr, "[ga3c]   dyn smem %d -> %d CTAs/SM\n", sm, nb);
    }
  }
  return (int)e;
}

int dense_fwd_splits(int batch, int num_sms) {
  const int tiles = ((batch + TC_BM - 1) / TC_BM) * (FC / FWD_BN);
  const int kblocks = (FLAT + TC_BK - 1) / TC_BK;                 // 61
  int s = num_sms / tiles;
  if (s < 1) s = 1;
  if (s > 16) s = 16;
  const int per = (kblocks + s - 1) / s;
  return (kblocks + per - 1) / per;                               // no empty splits
}

int launch_dense_fwd_tc(const uint16_t* n2, const uint16_t* w1bf, float* d1_part, int batch, int splits, cudaStream_t stream,
                        const DpGate* gate) {
  CUtensorMap ta, tb;
  if (make_tmap(&ta, n2, batch, FLAT, FLAT, TC_BM)) return (int)cudaErrorInvalidValue;        // A: [B][3872], K inner
  if (make_tmap(&tb, w1bf, FLAT, FC, FC, 64)) return (int)cudaErrorInvalidValue;              // B: [3872][256], N inner
  const int kblocks = (FLAT + TC_BK - 1) / TC_BK;
  const int per = (kblocks + splits - 1) / splits;
  dim3 grid((batch + TC_BM - 1) / TC_BM, FC / FWD_BN, splits);
  return launch_pdl(gemm_tc_kernel<FWD_BN, FWD_ST, false, true, EpiPartialF32>, grid, dim3(TC_THREADS),
                    tc_smem<FWD_BN, FWD_ST>(), stream, ta, tb, batch, (int)FC, kblocks, per,
                    EpiPartialF32{d1_part, FC, (int64_t)batch * FC}, gate ? *gate : DpGate{});
}

int launch_dense_dgrad_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint8_t* dn2, int batch,
                          cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (make_tmap(&ta, dd1, batch, FC, FC, TC_BM)) return (int)cudaErrorInvalidValue;           // A: [B][256], K inner
  if (make_tmap(&tb, w1bf, FLAT, FC, FC, DG_BN)) return (int)cudaErrorInvalidValue;           // B: [3872][256] = [N][K]
  dim3 grid((batch + TC_BM - 1) / TC_BM, (FLAT + DG_BN - 1) / DG_BN, 1);
  return launch_pdl(gemm_tc_kernel<DG_BN, DG_ST, false, false, EpiReluMaskBf16Tc>, grid, dim3(TC_THREADS),
                    tc_smem<DG_BN, DG_ST>(), stream, ta, tb, batch, (int)FLAT, FC / TC_BK, FC / TC_BK,
                    EpiReluMaskBf16Tc{dn2, n2, FLAT}, DpGate{});
}

int launch_dense_wgrad_tc(const uint16_t* n2, const uint16_t* dd1, float* g_w1, int batch, cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (make_tmap(&ta, n2, batch, FLAT, FLAT, 64)) return (int)cudaErrorInvalidValue;           // A: [K=B][M=3872], M inner
  if (make_tmap(&tb, dd1, batch, FC, FC, 64)) return (int)cudaErrorInvalidValue;              // B: [K=B][N=256],  N inner
  const int kblocks = (batch + TC_BK - 1) / TC_BK;
  dim3 grid((FLAT + TC_BM - 1) / TC_BM, FC / WG_BN, 1);
  return launch_pdl(gemm_tc_kernel<WG_BN, WG_ST, true, true, EpiPartialF32>, grid, dim3(TC_THREADS),
                    tc_smem<WG_BN, WG_ST>(), stream, ta, tb, (int)FLAT, (int)FC, kblocks, kblocks,
                    EpiPartialF32{g_w1, FC, 0}, DpGate{});
}

int launch_dense_bwd_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint8_t* dn2, float* g_w1, int batch,
                        cudaStream_t stream) {
  CUtensorMap da, db, wa, wb;
  if (make_tmap(&da, dd1, batch, FC, FC, TC_BM)) return (int)cudaErrorInvalidValue;           // dgrad A: [B][256], K inner
  if (make_tmap(&db, w1bf, FLAT, FC, FC, DG_BN)) return (int)cudaErrorInvalidValue;           // dgrad B: [3872][256] = [N][K]
  if (make_tmap(&wa, n2, batch, FLAT, FLAT, 64)) return (int)cudaErrorInvalidValue;           // wgrad A: [K=B][M=3872], M inner
  if (make_tmap(&wb, dd1, batch, FC, FC, 64)) return (int)cudaErrorInvalidValue;              // wgrad B: [K=B][N=256],  N inner
  DenseBwdArgs p{};
  p.batch = batch;
  p.dg_mtiles = (batch + TC_BM - 1) / TC_BM;
  p.n_dg = p.dg_mtiles * ((FLAT + DG_BN - 1) / DG_BN);
  p.wg_mtiles = (FLAT + TC_BM - 1) / TC_BM;
  p.wg_kblocks = (batch + TC_BK - 1) / TC_BK;
  p.epi_dg = EpiReluMaskBf16Tc{dn2, n2, FLAT};
  p.epi_wg = EpiPartialF32{g_w1, FC, 0};
  const int grid = p.n_dg + p.wg_mtiles * (FC / WG_BN);
  return launch_pdl(dense_bwd_kernel, dim3(grid), dim3(TC_THREADS), DBW_SMEM, stream, da, db, wa, wb, p);
}

}  // namespace ga3c
