// The tcgen05 GEMM core shared by the dense1 GEMMs (dense_tc.cu) and the generic conv trunk (conv_gen.cu): one 128 x BN
// output tile per CTA, operands staged in shared memory by TMA (cp.async.bulk.tensor, SWIZZLE_128B), an mbarrier pipeline of
// STAGES k-blocks, the fp32 accumulator in TMEM, and an epilogue functor that turns the accumulator into the caller's output.
// M, N and the k-blocks are runtime values; tensor-map reads past a matrix's edge return zeros, so ragged tiles need no code.
//
// 192 threads:
//   warp 0   TMA producer (one elected lane)
//   warp 1   TMEM allocator + MMA issuer (one elected lane issues tcgen05.mma.cta_group::1.kind::f16)
//   warp 2-5 epilogue: tcgen05.ld 32 lanes x 32 columns -> registers -> fused epilogue -> global
// K is consumed in blocks of 64 (one 128-byte swizzle row); a k-block is 4 MMAs of K = 16.
#pragma once
#include <cuda.h>

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

// gate (dense1 forward, data parallel with the side-stream exchange): the B operand is the bf16 shadow of dense1/w, whose slices
// the ranks' exchange kernels of the PREVIOUS step store into this rank's slab.  Instead of a stream-level event wait in front
// of this launch (which takes the launch out of the programmatic-dependent-launch chain: +3.6 us per step, measured) the TMA
// producer warp looks at the "slice of rank r landed everywhere" flags in this rank's own comm block -- pushed there long ago in
// the normal case -- before its first load.  The exchange grid it might wait for only ever waits for other GPUs and has been
// resident since the previous step's conv backward, so the wait cannot keep it off an SM.
// KID: the kernel id of the trace stamps (-1: the dense1 id the operand majors imply).  BN = 16 (the generic conv11 GEMM, N = 16)
// runs an N = 16 UMMA into the smallest TMEM allocation (32 columns) and reads it back with the half-width tcgen05.ld.
template <int BN, int STAGES, bool A_MN, bool B_MN, class Epi, int KID = -1>
__device__ __forceinline__ void gemm_tc_body(const CUtensorMap& tm_a, const CUtensorMap& tm_b, int M, int N, int k_blocks,
                                             int k_blocks_per_split, const Epi& epi, int bx, int by, int bz,
                                             const DpGate* gate = nullptr) {
  constexpr int B_STAGE = BN * TC_BK * 2;
  constexpr int STAGE = TC_A_STAGE + B_STAGE;
  constexpr int TMEM_COLS = BN < 32 ? 32 : BN;
  constexpr int EC = BN < 32 ? BN : 32;                    // accumulator columns per epilogue call
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
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tmem_slot), "n"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  griddep_launch();             // every CTA of this grid holds its TMEM columns and shared memory
  constexpr int kid = KID >= 0 ? KID : A_MN ? K_DENSE_WGRAD : (B_MN ? K_DENSE_FWD : K_DENSE_DGRAD);
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
    typename Epi::Pre pre[BN / EC];               // epilogue inputs from global memory, loaded under the MMAs
#pragma unroll
    for (int c = 0; c < BN / EC; ++c) epi.prefetch(pre[c], m, n0 + c * EC, m < M && n0 + c * EC < N);
    DEVT(5, 0);
    mbar_wait(bars + 2 * STAGES * 8, 0);
    DEVT(6, 0);
    tc_fence_after();
#pragma unroll
    for (int c = 0; c < BN / EC; ++c) {
      uint32_t r[32];
      if constexpr (EC == 32) tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + c * 32, r);
      else tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + c * EC, *reinterpret_cast<uint32_t(*)[16]>(r));
      const int n = n0 + c * EC;
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
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
  }
}

template <int BN, int STAGES, bool A_MN, bool B_MN, class Epi, int KID = -1>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, int M, int N,
               int k_blocks, int k_blocks_per_split, Epi epi, const DpGate gate) {
  gemm_tc_body<BN, STAGES, A_MN, B_MN, Epi, KID>(tm_a, tm_b, M, N, k_blocks, k_blocks_per_split, epi, blockIdx.x, blockIdx.y,
                                            blockIdx.z, &gate);
}

// ---- host side ----------------------------------------------------------------------------------
// 2-D bf16 row-major matrix [rows][cols] (ld elements between rows), box = 64 inner x box_rows, 128-B swizzle,
// out-of-bounds elements read as zero (ragged M / N / K tails need no special casing in the kernel).
// cuTensorMapEncodeTiled is resolved through the runtime (cudaGetDriverEntryPoint) so the library has no
// link-time dependency on libcuda.so.1 and still loads on a box without a driver (symbol-export test).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static inline EncodeTiledFn encode_tiled_fn() {
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

static inline int make_tmap(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
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

}  // namespace ga3c
