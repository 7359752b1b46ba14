// The wide layers of the low-dimensional MLP networks (BASELINE configs[3]; fork NetworkVP.py:79-105: 256 -> 256 and 256 -> 100 hold
// 92 % of the flops) on the 5th-generation tensor cores, in fp32-equivalent precision: tcgen05.mma.kind::tf32 with the 3xTF32
// operand split.  Every fp32 operand x is split into  hi = tf32(x)  (round to nearest, 10 mantissa bits)  and  lo = x - hi  (exact
// in fp32; the tensor core reads its leading 11 bits), and  a.b ~ hi_a.hi_b + hi_a.lo_b + lo_a.hi_b  accumulates in fp32 in TMEM:
// the dropped terms are 2^-22 relative, the error of the products is that of an fp32 FMA chain (experiments/tf32_mlp_error_study.py).
//
//   fwd  : out_l [B, n]   = act(in_l [B, k] x W_l [k, n] + b_l)           (A K-major,  B MN-major)
//   dgrad: dz_{l-1} [B,k] = (dz_l [B, n] x W_l [k, n]^T) . act'(out_{l-1})  (A K-major,  B K-major)
//   wgrad: dW_l [k, n]    = in_l [B, k]^T x dz_l [B, n]                    (A MN-major, B MN-major), split over the batch into
//                                                                           the partial arenas mlp_reduce sums in a fixed order
// Operands are the fp32 row-major matrices the fused kernel (mlp.cu) already keeps in HBM for training; nothing is transposed
// or converted in HBM.  One 128 x BN output tile per CTA, 448 threads:
//   warp 0     TMA producer: fp32 boxes of 32 floats (one 128-byte swizzle row) x rows, SWIZZLE_128B
//   warp 1     TMEM allocator + UMMA issuer: per 32-float k-block 4 k-steps (K = 8) x 3 products
//   warps 2-5  epilogue: tcgen05.ld 32 lanes x 32 columns -> bias / activation / act' -> global
//   warps 6-13 splitters: rewrite a landed stage in place as hi and write lo into the stage's twin buffer (the operand layout
//              is whatever TMA produced: the split is element-wise), fence.proxy.async, arrive on the stage's "split" barrier
#include "common.cuh"
#include "kernels.h"
#include "mlp.cuh"
#include "tcgen05.cuh"

namespace ga3c {

namespace {

// A stage is 16 floats of K (two UMMA k-steps): fine-grained on purpose.  The chain TMA -> split -> UMMA of one stage is ~2 us
// long against ~0.5 us of tensor time, and what hides it is stages in flight per SM: 96 KB of stages per CTA, TWO CTAs per SM
// (2 x 256 TMEM columns), which also lets one CTA's epilogue run under the other's main loop.  (32-float stages, one CTA per
// SM: 3 us per 32 floats of K, tensor pipe 25 % busy -- profiles/r3h.)
constexpr int T3_BK = 16;                          // floats of K per stage: one 64-byte swizzle row (K-major operands)
constexpr int T3_THREADS = 448, T3_SPLIT_WARP0 = 6, T3_SPLIT_WARPS = 8;
constexpr int T3_A_BYTES = TC_BM * T3_BK * 4;      // 8 KB
constexpr int T3_MN_BOX = 32 * T3_BK * 4;          // one MN-major TMA box: 32 floats of M / N x 16 k-rows = 2 KB

template <int BN>
constexpr int t3_half() { return T3_A_BYTES + BN * T3_BK * 4; }      // hi (or lo) operands of one stage
// DEEP = false: 96 KB of stages, two CTAs per SM (forward / data gradient: hundreds of tiles); DEEP = true: 192 KB, one CTA per SM
// (weight gradient: at most one CTA per SM anyway, each streaming a long K = batch range -- stages in flight is all it has)
template <int BN, bool DEEP>
constexpr int t3_stages() { return (BN >= 256 ? 2 : 3) * (DEEP ? 2 : 1); }
template <int BN, bool DEEP>
constexpr int t3_smem() { return t3_stages<BN, DEEP>() * 2 * t3_half<BN>() + (3 * t3_stages<BN, DEEP>() + 1) * 8 + 16 + 1024; }

// instruction descriptor, kind::tf32: D = f32, A = B = tf32
__host__ __device__ constexpr uint32_t make_idesc_tf32(int m, int n, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}
// Shared-memory descriptor of an fp32 operand.  K-major: SWIZZLE_64B (layout type 4), rows of 64 B (16 floats of K), 8-row atoms:
// SBO = 512.  MN-major: 32-bit operands can only be transposed from the SWIZZLE_128B_BASE32B layout (layout type 1: 32-byte
// chunks swizzled within 128 B, pattern period 4 rows; TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): atom = 4 k-rows x 128 B (32
// floats of M / N), SBO = 512 between k-atoms, LBO = 2048 between the 32-wide atoms (one TMA box of 16 k-rows each).
__device__ __forceinline__ uint64_t make_desc_f32(uint32_t saddr, bool mn_major) {
  const uint64_t lbo = mn_major ? (uint64_t)(T3_MN_BOX >> 4) : 1u, sbo = 512u >> 4, type = mn_major ? 1ull : 4ull;
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (lbo << 16) | (sbo << 32) | (1ull << 46) | (type << 61);
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(acc)
      : "memory");
}

// ---- epilogues -------------------------------------------------------------------------------------------------------------------
// A warp drains 32 rows x 32 columns of the accumulator (tcgen05.ld: one row per lane), turns the chunk around through a swizzled
// 4 KB staging tile in shared memory, and finishes it in the COALESCED domain: 8 lanes per row, one float4 each, so every global
// access of the warp is four whole 128-byte lines.  (One row per lane straight to global -- 32 lines touched by every store
// instruction -- made the epilogue 40 % of the forward GEMM and 60 % of the data-gradient GEMM, measured.)  The functors below see
// (row m, column n .. n + 3, the accumulator float4); n, N are multiples of 4.  load() fetches what the chunk's 8 float4 need from
// global memory BEFORE any of them is stored (loads issued between stores would each wait out a memory latency).
struct Epi3Fwd {         // out = act(acc + b)
  const float* bias; float* out; int N, act;
  __device__ __forceinline__ float4 load(int, int n) const { return __ldg(reinterpret_cast<const float4*>(bias + n)); }
  __device__ __forceinline__ void operator()(int, int m, int n, float4 v, const float4 b) const {
    v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
    if (act == MLP_ACT_SIGMOID) {
      v.x = sigmoid(v.x); v.y = sigmoid(v.y); v.z = sigmoid(v.z); v.w = sigmoid(v.w);
    }
    *reinterpret_cast<float4*>(out + (size_t)m * N + n) = v;
  }
};
struct Epi3Dgrad {       // dz_prev = acc * act'(out_prev)
  const float* out_prev; float* dz; int N, act;
  __device__ __forceinline__ float4 load(int m, int n) const {
    return act == MLP_ACT_SIGMOID ? __ldcs(reinterpret_cast<const float4*>(out_prev + (size_t)m * N + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __device__ __forceinline__ void operator()(int, int m, int n, float4 v, const float4 o) const {
    if (act == MLP_ACT_SIGMOID) {
      v.x *= o.x * (1.f - o.x); v.y *= o.y * (1.f - o.y); v.z *= o.z * (1.f - o.z); v.w *= o.w * (1.f - o.w);
    }
    *reinterpret_cast<float4*>(dz + (size_t)m * N + n) = v;
  }
};
struct Epi3Wgrad {       // raw tile into partial arena `split` (part points at the layer's weights in arena 0)
  float* part; int64_t part_stride; int N;
  __device__ __forceinline__ float4 load(int, int) const { return make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ void operator()(int split, int m, int n, float4 v, const float4) const {
    *reinterpret_cast<float4*>(part + (size_t)split * part_stride + (size_t)m * N + n) = v;
  }
};

template <int BN, bool A_MN, bool B_MN, bool DEEP, class Epi>
__global__ void __launch_bounds__(T3_THREADS, 2)
gemm3_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, int M, int N, int k_blocks,
             int k_blocks_per_split, const Epi epi, int dbg) {
  constexpr int STAGES = t3_stages<BN, DEEP>(), HALF = t3_half<BN>(), STAGE = 2 * HALF;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;     // SWIZZLE_128B atoms need 1024-byte alignment
  uint8_t* const smem = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bars = sbase + STAGES * STAGE;     // full[STAGES] | split[STAGES] | empty[STAGES] | tmem_full
  const uint32_t tmem_slot = bars + (3 * STAGES + 1) * 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * TC_BM, n0 = blockIdx.y * BN, split = blockIdx.z;
  const int kb0 = split * k_blocks_per_split;
  const int kb1 = min(kb0 + k_blocks_per_split, k_blocks);
  auto bar_full = [&](int s) { return bars + s * 8; };
  auto bar_split = [&](int s) { return bars + (STAGES + s) * 8; };
  auto bar_empty = [&](int s) { return bars + (2 * STAGES + s) * 8; };
  const uint32_t bar_done = bars + 3 * STAGES * 8;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tm_a));
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tm_b));
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_split(s), T3_SPLIT_WARPS); mbar_init(bar_empty(s), 1); }
    mbar_init(bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) tmem_alloc<BN>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  griddep_launch();
  griddep_wait(K_MLP_TC);           // operands are produced by the preceding kernels
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    for (int kb = kb0; kb < kb1; ++kb) {
      const int it = kb - kb0, s = it % STAGES;
      mbar_wait(bar_empty(s), ((it / STAGES) & 1) ^ 1);
      if (elect_one()) {
        const uint32_t sa = sbase + s * STAGE, sb = sa + T3_A_BYTES;
        mbar_expect_tx(bar_full(s), HALF);
        if (A_MN) {
#pragma unroll
          for (int j = 0; j < TC_BM / 32; ++j) tma_load_2d(sa + j * T3_MN_BOX, &tm_a, m0 + 32 * j, kb * T3_BK, bar_full(s));
        } else {
          tma_load_2d(sa, &tm_a, kb * T3_BK, m0, bar_full(s));
        }
        if (B_MN) {
#pragma unroll
          for (int j = 0; j < BN / 32; ++j) tma_load_2d(sb + j * T3_MN_BOX, &tm_b, n0 + 32 * j, kb * T3_BK, bar_full(s));
        } else {
          tma_load_2d(sb, &tm_b, kb * T3_BK, n0, bar_full(s));
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_tf32(TC_BM, BN, A_MN, B_MN);
    for (int kb = kb0; kb < kb1; ++kb) {
      const int it = kb - kb0, s = it % STAGES;
      mbar_wait(bar_split(s), (it / STAGES) & 1);          // hi / lo of the stage written (and visible to the async proxy)
      tc_fence_after();
      if (elect_one()) {
        const uint32_t sa = sbase + s * STAGE, sb = sa + T3_A_BYTES;
        const uint64_t a_hi = make_desc_f32(sa, A_MN), b_hi = make_desc_f32(sb, B_MN);
        const uint64_t a_lo = make_desc_f32(sa + HALF, A_MN), b_lo = make_desc_f32(sb + HALF, B_MN);
#pragma unroll
        for (int k = 0; k < T3_BK / 8; ++k) {
          // advance K by 8: +32 B inside the 64-B swizzle row (K-major), +2 k-atoms = 1024 B (MN-major)
          const uint64_t ka = (uint64_t)((A_MN ? 1024u : 32u) * k >> 4), kbv = (uint64_t)((B_MN ? 1024u : 32u) * k >> 4);
          if (dbg & 2) continue;
          tc_mma_tf32(tmem_base, a_lo + ka, b_hi + kbv, idesc, (it > 0 || k > 0) ? 1u : 0u);      // small terms first
          tc_mma_tf32(tmem_base, a_hi + ka, b_lo + kbv, idesc, 1u);
          tc_mma_tf32(tmem_base, a_hi + ka, b_hi + kbv, idesc, 1u);
        }
        tc_commit(bar_empty(s));
      }
      __syncwarp();
    }
    if (elect_one()) tc_commit(bar_done);
    __syncwarp();
  } else if (warp < T3_SPLIT_WARP0) {
    const int q = warp & 3;                       // TMEM lane quarter this warp may read
    const bool zero = kb1 <= kb0;                 // an empty split still writes its (zero) tile
    if (!zero) {
      mbar_wait(bar_done, 0);                     // every UMMA has retired: the accumulator is final and the stages are free
      tc_fence_after();
    }
    const uint32_t stg = sbase + (uint32_t)(warp - 2) * 4096u;      // staging tile of this warp, in stage 0
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      const int n = n0 + c * 32;
      if (n >= N) break;
      uint32_t r[32];
      if (!zero) tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + c * 32, r);
#pragma unroll
      for (int j = 0; j < 8; ++j) {               // own row, 16-byte chunk j at chunk position j ^ (row & 7): conflict-free both ways
        const uint32_t dst = stg + lane * 128 + ((j ^ (lane & 7)) << 4);
        if (zero) asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};\n" ::"r"(dst), "r"(0u) : "memory");
        else asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(dst), "r"(r[4 * j]), "r"(r[4 * j + 1]), "r"(r[4 * j + 2]),
                          "r"(r[4 * j + 3]) : "memory");
      }
      __syncwarp();
      if (!(dbg & 4)) {
        const int ch = lane & 7, nn = n + ch * 4, mrow0 = m0 + q * 32 + (lane >> 3);
#pragma unroll
        for (int h = 0; h < 2; ++h) {             // two rounds of 4 rows per lane (register budget of two CTAs per SM)
          float4 aux[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int m = mrow0 + 4 * (4 * h + i);
            aux[i] = (m < M && nn < N) ? epi.load(m, nn) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = 4 * (4 * h + i) + (lane >> 3), m = mrow0 + 4 * (4 * h + i);
            float4 v;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                         : "r"(stg + row * 128 + ((ch ^ (row & 7)) << 4)) : "memory");
            if (m < M && nn < N) epi(split, m, nn, v, aux[i]);
          }
        }
      }
      __syncwarp();
    }
  } else {
    const int t = threadIdx.x - 32 * T3_SPLIT_WARP0;      // 0 .. 255
    for (int kb = kb0; kb < kb1; ++kb) {
      const int it = kb - kb0, s = it % STAGES;
      mbar_wait(bar_full(s), (it / STAGES) & 1);           // TMA bytes landed
      float4* hi = reinterpret_cast<float4*>(smem + s * STAGE);
      float4* lo = reinterpret_cast<float4*>(smem + s * STAGE + HALF);
      if (!(dbg & 1))
#pragma unroll
      for (int i = 0; i < HALF / 16 / (32 * T3_SPLIT_WARPS); ++i) {
        const int idx = t + 32 * T3_SPLIT_WARPS * i;
        const float4 x = hi[idx];
        float4 h;
        h.x = __uint_as_float((__float_as_uint(x.x) + 0x1000u) & 0xFFFFE000u);
        h.y = __uint_as_float((__float_as_uint(x.y) + 0x1000u) & 0xFFFFE000u);
        h.z = __uint_as_float((__float_as_uint(x.z) + 0x1000u) & 0xFFFFE000u);
        h.w = __uint_as_float((__float_as_uint(x.w) + 0x1000u) & 0xFFFFE000u);
        hi[idx] = h;
        lo[idx] = make_float4(x.x - h.x, x.y - h.y, x.z - h.z, x.w - h.w);
      }
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_split(s));
    }
  }
  tc_fence_before();
  __syncthreads();
  trace_mark(K_MLP_TC, 2);
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<BN>(tmem_base);
  }
}
static_assert(2 * (t3_smem<256, false>() + 1024) <= 233472 && 2 * (t3_smem<128, false>() + 1024) <= 233472, "two CTAs per SM");
static_assert(t3_smem<256, true>() <= 232448 && t3_smem<128, true>() <= 232448, "shared memory budget of one CTA");
static_assert(t3_half<256>() % (16 * 32 * T3_SPLIT_WARPS) == 0 && t3_half<128>() % (16 * 32 * T3_SPLIT_WARPS) == 0,
              "the splitters cover a stage in whole rounds");

// Weight gradient of a layer with fan-in K <= 4 (the state and the 4-wide first layer of the fork NetworkVP; K = 0: none) and the
// bias gradient of any layer, per batch split: dW[k][n] = sum_r in[r][k] dz[r][n], db[n] = sum_r dz[r][n].  Pure streaming --
// dz is read once, coalesced -- where a 64 x 64 tile kernel would spend its time on zero padding.  1024 threads = 16 row groups
// x 64 columns (the loop is bound by memory latency: rows in flight are what counts); the row groups are added in a fixed order.
constexpr int SK_RG = 16;
template <int K>
__global__ void __launch_bounds__(64 * SK_RG) mlp_skinny_wgrad_kernel(const float* __restrict__ in, const float* __restrict__ dz,
                                                                      int batch, int N, int rows_per_split, float* part_w,
                                                                      float* part_b, int64_t part_stride) {
  __shared__ float red[SK_RG][K + 1][64];
  griddep_launch();
  griddep_wait(K_MLP_TC);
  const int rg = threadIdx.x >> 6, c = threadIdx.x & 63, n = blockIdx.y * 64 + c;
  const int r0 = blockIdx.x * rows_per_split, r1 = min(batch, r0 + rows_per_split);
  float acc[K + 1];
#pragma unroll
  for (int k = 0; k <= K; ++k) acc[k] = 0.f;
  if (n < N) {
    constexpr int U = 4;
    int r = r0 + rg;
    for (; r + SK_RG * (U - 1) < r1; r += SK_RG * U) {
      float d[U], x[U][K > 0 ? K : 1];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        d[u] = __ldcs(dz + (size_t)(r + SK_RG * u) * N + n);
#pragma unroll
        for (int k = 0; k < K; ++k) x[u][k] = __ldg(in + (size_t)(r + SK_RG * u) * K + k);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = fmaf(x[u][k], d[u], acc[k]);
        acc[K] += d[u];
      }
    }
    for (; r < r1; r += SK_RG) {
      const float d = dz[(size_t)r * N + n];
#pragma unroll
      for (int k = 0; k < K; ++k) acc[k] = fmaf(__ldg(in + (size_t)r * K + k), d, acc[k]);
      acc[K] += d;
    }
  }
#pragma unroll
  for (int k = 0; k <= K; ++k) red[rg][k][c] = acc[k];
  __syncthreads();
  if (rg == 0 && n < N) {
    float* pw = part_w + (size_t)blockIdx.x * part_stride;
#pragma unroll
    for (int k = 0; k <= K; ++k) {
      float t = 0.f;
#pragma unroll
      for (int g = 0; g < SK_RG; ++g) t += red[g][k][c];
      if (k < K) pw[(size_t)k * N + n] = t;
      else part_b[(size_t)blockIdx.x * part_stride + n] = t;
    }
  }
}

// 2-D fp32 row-major matrix [rows][cols] (ld floats between rows).  K-major operand: box = 16 inner x box_rows, 64-B swizzle;
// MN-major operand: box = 32 inner x 16 rows, 128-B swizzle of 32-byte chunks.  Out-of-bounds
// elements read as zero, so ragged M / N / K tails need no special casing in the kernel
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
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
int make_tmap_f32(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, bool mn_major) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return (int)cudaErrorNotSupported;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 4};
  cuuint32_t box[2] = {mn_major ? 32u : (cuuint32_t)T3_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

static int t3_debug() { static const int v = [] { const char* e = getenv("GA3C_T3_DEBUG"); return e ? atoi(e) : 0; }(); return v; }

template <int BN, bool A_MN, bool B_MN, bool DEEP = false, class Epi>
int launch_gemm3(const CUtensorMap& ta, const CUtensorMap& tb, int M, int N, int k_blocks, int per, int splits, const Epi& epi,
                 cudaStream_t stream) {
  static const int configured = [] {
    int r = (int)cudaFuncSetAttribute(gemm3_kernel<BN, A_MN, B_MN, DEEP, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      t3_smem<BN, DEEP>());
    if (r) return r;       // two CTAs per SM need the full shared-memory carveout
    return (int)cudaFuncSetAttribute(gemm3_kernel<BN, A_MN, B_MN, DEEP, Epi>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                     (int)cudaSharedmemCarveoutMaxShared);
  }();
  if (configured) return configured;
  const dim3 grid((M + TC_BM - 1) / TC_BM, (N + BN - 1) / BN, splits);
  return launch_pdl(gemm3_kernel<BN, A_MN, B_MN, DEEP, Epi>, grid, dim3(T3_THREADS), (size_t)t3_smem<BN, DEEP>(), stream, ta, tb, M, N,
                    k_blocks, per, epi, t3_debug());
}

}  // namespace

GA3C_TRACE_ATTACH(trace_attach_mlp_tc)

bool mlp_tc_layer_ok(const MlpLayerDesc& L) { return L.k >= 64 && L.n >= 64 && L.k % 4 == 0 && L.n % 4 == 0 && L.n <= 256 && L.k <= 256; }

// out = act(in [B, k] x W [k, n] + bias)
int launch_mlp_tc_fwd(const float* W, const float* bias, int k, int n, int act, const float* in, float* out, int batch,
                      cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (make_tmap_f32(&ta, in, batch, k, k, TC_BM, false)) return (int)cudaErrorInvalidValue;            // A: [B][k], K inner
  if (make_tmap_f32(&tb, W, k, n, n, T3_BK, true)) return (int)cudaErrorInvalidValue;                 // B: [k][n], N inner
  const int kblocks = (k + T3_BK - 1) / T3_BK;
  const Epi3Fwd epi{bias, out, n, act};
  if (n > 128) return launch_gemm3<256, false, true>(ta, tb, batch, n, kblocks, kblocks, 1, epi, stream);
  return launch_gemm3<128, false, true>(ta, tb, batch, n, kblocks, kblocks, 1, epi, stream);
}

// dz_prev [B, k] = (dz [B, n] x W [k, n]^T) * act'(out_prev);  prev_act: activation of the layer that produced out_prev
int launch_mlp_tc_dgrad(const float* W, int k, int n, const float* dz, const float* out_prev, int prev_act, float* dz_prev,
                        int batch, cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (make_tmap_f32(&ta, dz, batch, n, n, TC_BM, false)) return (int)cudaErrorInvalidValue;            // A: [B][n], reduction n inner
  const int bn = k > 128 ? 256 : 128;
  if (make_tmap_f32(&tb, W, k, n, n, bn, false)) return (int)cudaErrorInvalidValue;                    // B: [k][n] = [N_out][K_red]
  const int kblocks = (n + T3_BK - 1) / T3_BK;
  const Epi3Dgrad epi{out_prev, dz_prev, k, prev_act};
  if (bn == 256) return launch_gemm3<256, false, false>(ta, tb, batch, k, kblocks, kblocks, 1, epi, stream);
  return launch_gemm3<128, false, false>(ta, tb, batch, k, kblocks, kblocks, 1, epi, stream);
}

// dW [k, n] = in [B, k]^T x dz [B, n]: batch split s into part_w + s * part_stride (every split writes its whole tile, zeros
// if it has no rows); the bias gradient comes from launch_mlp_skinny_wgrad with k = 0
int launch_mlp_tc_wgrad(int k, int n, const float* in, const float* dz, int batch, int splits, int rows_per_split, float* part_w,
                        float* part_b, int64_t part_stride, cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (make_tmap_f32(&ta, in, batch, k, k, T3_BK, true)) return (int)cudaErrorInvalidValue;            // A: [K=B][M=k], M inner
  if (make_tmap_f32(&tb, dz, batch, n, n, T3_BK, true)) return (int)cudaErrorInvalidValue;            // B: [K=B][N=n], N inner
  const int kblocks = (batch + T3_BK - 1) / T3_BK;
  const int per = rows_per_split / T3_BK;
  const Epi3Wgrad epi{part_w, part_stride, n};
  int r;
  if (n > 128) r = launch_gemm3<256, true, true, true>(ta, tb, k, n, kblocks, per, splits, epi, stream);
  else r = launch_gemm3<128, true, true, true>(ta, tb, k, n, kblocks, per, splits, epi, stream);
  (void)part_b;
  return r;
}

int launch_mlp_skinny_wgrad(int k, int n, const float* in, const float* dz, int batch, int splits, int rows_per_split,
                            float* part_w, float* part_b, int64_t part_stride, cudaStream_t stream) {
  const dim3 grid(splits, (n + 63) / 64), block(64 * SK_RG);
  switch (k) {
    case 0: return launch_pdl(mlp_skinny_wgrad_kernel<0>, grid, block, 0, stream, in, dz, batch, n, rows_per_split, part_w, part_b, part_stride);
    case 1: return launch_pdl(mlp_skinny_wgrad_kernel<1>, grid, block, 0, stream, in, dz, batch, n, rows_per_split, part_w, part_b, part_stride);
    case 2: return launch_pdl(mlp_skinny_wgrad_kernel<2>, grid, block, 0, stream, in, dz, batch, n, rows_per_split, part_w, part_b, part_stride);
    case 3: return launch_pdl(mlp_skinny_wgrad_kernel<3>, grid, block, 0, stream, in, dz, batch, n, rows_per_split, part_w, part_b, part_stride);
    case 4: return launch_pdl(mlp_skinny_wgrad_kernel<4>, grid, block, 0, stream, in, dz, batch, n, rows_per_split, part_w, part_b, part_stride);
  }
  return (int)cudaErrorInvalidValue;
}

}  // namespace ga3c
