// Shared device helpers for the sm_100a kernels of the GA3C hot path.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace ga3c {

// ---- geometry of the conv NetworkVP (NetworkDNav.py:81-90; SAME padding, SURVEY A.1) ----
constexpr int IMG = 84, IMG_C = 4, STATE_DIM = IMG * IMG * IMG_C;      // 28224
constexpr int C1_OUT = 16, H1 = 21, N1_POS = H1 * H1;                  // conv11: 8x8 s4 pad (2,2) -> 21x21x16
constexpr int C2_OUT = 32, H2 = 11, N2_POS = H2 * H2;                  // conv12: 4x4 s2 pad (1,2) -> 11x11x32
constexpr int FLAT = N2_POS * C2_OUT;                                  // 3872
constexpr int FC = 256;
constexpr int MAX_ACTIONS = 18;

// padded bf16 image in shared memory: 88x88 pixels x 4 channels (8 B / pixel), zero border of 2
constexpr int XS_W = 88, XS_ROW_BYTES = XS_W * 8, XS_BYTES = XS_W * XS_ROW_BYTES;   // 61952
// padded conv11 output in shared memory: 24x24 pixels x 16 channels (32 B / pixel), pad (1 before, 2 after)
constexpr int N1P_W = 24, N1P_BYTES = N1P_W * N1P_W * 32;                            // 18432

// ---- HBM layouts of the training-only activations ---------------------------------------------------------------------
// The conv backward kernel (conv_bwd_fused.cu) consumes its three inputs as tcgen05 operands exactly as they lie in HBM: the
// kernels that PRODUCE them write the no-swizzle UMMA layouts (16-byte chunk j of row r at j*LBO + r*16, all rows of a plane
// contiguous, so a spatial shift is a different descriptor start address), and the consumer only issues bulk copies.
//   xblk  bf16 copy of the frame as conv_fwd's space-to-depth block matrix Blk (conv_blk.cuh): 22x22 blocks of 4x4 pixels of the
//         zero-padded 88x88x4 image, row Y*22 + X, 64 elements (dy, dx, c) in 8 chunk planes.  Stored in 4 quarters of 128 rows,
//         [frame][quarter][plane][128 rows][16 B]; rows >= 484 stay zero (never written)
//   n1    Blk2: n1 SAME-padded (1 before, 2 after) to 24x24 and cut into 12x12 blocks of 2x2 pixels, row Yb*13 + Xb (column 12
//         dead), 64 elements (dy, dx, ci) in 8 chunk planes of 160 rows; [frame][plane][160 rows][16 B], borders stay zero
//   dn2   G: dn2 on a zero-bordered 13x13 grid, row (oy+1)*13 + (ox+1), 32 co in 4 chunk planes of 176 rows;
//         [frame][plane][172 rows][16 B], borders stay zero
constexpr int XB_QROWS = 128, XB_QUARTERS = 4, XB_PLANE_BYTES = XB_QROWS * 16, XB_QBYTES = 8 * XB_PLANE_BYTES,
              XB_FRAME_BYTES = XB_QUARTERS * XB_QBYTES, XB_LIVE_ROWS = 484;                                        // 65,536 B / frame
constexpr int G_W = 13, G_ROWS = 172, G_LBO = G_ROWS * 16, G_BYTES = 4 * G_LBO;                                 // 11,008 B / frame
constexpr int B2_ROWS = 160, B2_LBO = B2_ROWS * 16, B2_BYTES = 8 * B2_LBO;                                      // 20,480 B / frame
// byte offset of channels [8h, 8h+8) of conv11 output pixel (y, x) inside a frame's Blk2 image
__host__ __device__ constexpr int b2_pixel_offset(int y, int x, int h) {
  return ((((y + 1) & 1) * 2 + ((x + 1) & 1)) * 2 + h) * B2_LBO + (((y + 1) >> 1) * G_W + ((x + 1) >> 1)) * 16;
}
// byte offset of channels [8j, 8j+8) of conv12 output position (oy, ox) inside a frame's G image
__host__ __device__ constexpr int g_pos_offset(int oy, int ox, int j) { return j * G_LBO + ((oy + 1) * G_W + ox + 1) * 16; }

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);   // .x = lo (low 16 bits), .y = hi
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

// D(16x8,f32) += A(16x16,bf16,row) * B(16x8,bf16,col)
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void lds64(uint32_t& a, uint32_t& b, uint32_t addr) {
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];\n" : "=r"(a), "=r"(b) : "r"(addr));
}
__device__ __forceinline__ void lds128(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;\n" ::"r"(addr), "r"(v));
}
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.u32 [%0], {%1,%2};\n" ::"r"(addr), "r"(a), "r"(b));
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};\n" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}

// 16-byte async copy global -> shared; src_bytes in {0,16}: 0 zero-fills the destination
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(src), "r"(src_bytes));
}
// 4-byte variant (src_bytes in {0,4}); .ca: weights are re-read by every tile of the CTA
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(dst), "l"(src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// streaming 128-bit global load that does not pollute L1 (frames are read exactly once)
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];\n"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

// ---- mbarrier + bulk async copy (TMA engine) ---------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared through the TMA engine; bytes % 16 == 0, both addresses 16-B aligned.
// Completion is signalled on `bar` as `bytes` of transaction count.
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// ---- L2 residency hints --------------------------------------------------------------------------------------------------
// The step's transient activations (xblk, n1, n2, dn2: ~100 MB at B = 1024) are written by one kernel and read once or twice by
// a later one; the fp32 frames (115 MB) are streamed exactly once.  Frames are loaded evict_first and the transients stored
// evict_last, so that the 126 MB L2 keeps what will be read again instead of what will not; the consumers load with evict_first
// (after that read the data is dead).  The policy is a runtime operand: hints = 0 (GA3C_L2_HINTS=0) passes evict_normal everywhere.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_normal() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;\n" : "=l"(p));
  return p;
}
__device__ __forceinline__ void bulk_load_hint(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;\n" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void bulk_store_hint(void* dst, uint32_t src, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;\n" ::"l"(dst), "r"(src), "r"(bytes),
               "l"(policy)
               : "memory");
}
__device__ __forceinline__ void stg128_hint(void* dst, uint4 v, uint64_t policy) {
  asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1,%2,%3,%4}, %5;\n" ::"l"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(policy)
               : "memory");
}
// 1-D bulk copy shared -> global through the TMA engine (bulk async-group completion)
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }

// ---- fp32 frame staging ring (conv_fwd, conv11_wgrad) ---------------------------------------------
// A frame (112,896 B, dense NHWC fp32) is streamed by the TMA engine into a shared-memory staging buffer in
// NCH chunks, each signalled on its own mbarrier.  The consumer converts chunk c and, as soon as every thread
// is done with it, re-arms that chunk with the NEXT frame's bytes: with NCH > 1 close to a full frame is always
// in flight per SM (a 1/148 share of HBM bandwidth moves 112,896 B in ~2.6 us), at the price of NCH - 1 extra
// block barriers per frame.  conv_fwd (compute-bound per frame) uses 1 chunk, conv11_wgrad 2.
constexpr int FRAME_BYTES = STATE_DIM * 4;                         // 112,896
template <int NCH>
__device__ __forceinline__ void stg_issue_chunk(uint32_t stg, const float* frame, int c, uint32_t bars) {
  constexpr int CB = FRAME_BYTES / NCH, PARTS = 4 / NCH > 0 ? 4 / NCH : 1, PB = CB / PARTS;   // <= 28,224 B per bulk copy
  static_assert(CB * NCH == FRAME_BYTES && PB * PARTS == CB && PB % 16 == 0, "chunking must be exact and 16-B granular");
  mbar_expect_tx(bars + 8 * c, CB);
#pragma unroll
  for (int k = 0; k < PARTS; ++k)
    bulk_load(stg + c * CB + k * PB, reinterpret_cast<const uint8_t*>(frame) + c * CB + k * PB, PB, bars + 8 * c);
}

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------
// Every kernel of the step is launched with programmatic stream serialization: it may start (and run its
// prologue: shared-memory setup, TMEM allocation, barrier init, weight fragments, input prefetch) while its
// predecessor in the stream is still draining.  griddep_wait() blocks until the predecessor grid has
// completed and its memory is visible; EVERY kernel calls it, which makes the ordering transitive.
// griddep_launch() lets the successor begin launching; kernels call it once all their CTAs hold the
// resources they need (so an early successor can never starve a not-yet-started CTA of this grid).
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }

// ---- step timeline trace (ga3c_trace_*) ---------------------------------------------------------------
// When a trace buffer is attached, thread 0 of every CTA stamps %globaltimer (ns) at three points of its kernel:
// launched (reached the dependency wait), started (dependency satisfied), ended.  Per kernel id the buffer keeps
// {min, max} of each: 6 uint64.  This is the only way to see the pipelined step as it runs (per-kernel events
// serialise the PDL chain, ncu serialises and flushes the caches).  One pointer per translation unit, set by
// trace_attach_<file>(); detached (the default) it costs one predicated load per CTA.
enum KernelId { K_CONV_FWD = 0, K_DENSE_FWD, K_HEADS, K_DENSE_WGRAD, K_DENSE_DGRAD, K_CONV12_BWD, K_CONV11_WGRAD, K_RMSPROP,
                K_GRAD_REDUCE, K_MLP_FUSED, K_MLP_WGRAD, K_MLP_REDUCE, K_DP_BIG, K_MLP_TC, K_HISTO,
                // the generic conv trunk (conv_gen.cu)
                K_GEN_WPREP, K_GEN_IM2COL1, K_GEN_CONV11, K_GEN_IM2COL2, K_GEN_CONV12, K_GEN_CONV12_DGRAD, K_GEN_COL2IM,
                K_GEN_CONV12_WGRAD, K_GEN_CONV11_WGRAD,
                K_COUNT };
constexpr int TRACE_SLOTS = 6;
static __device__ unsigned long long* g_trace = nullptr;
__device__ __forceinline__ void trace_mark(int kid, int what) {      // what: 0 launched, 1 started, 2 ended
  if (threadIdx.x == 0) {
    unsigned long long* t = g_trace;
    if (t != nullptr) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(now));
      atomicMin(t + kid * TRACE_SLOTS + 2 * what, now);
      atomicMax(t + kid * TRACE_SLOTS + 2 * what + 1, now);
    }
  }
}
// the same stamp by whichever single thread the caller names (kernels whose thread 0 does not wait for the dependency)
__device__ __forceinline__ void trace_mark_by(int kid, int what, bool me) {
  if (me) {
    unsigned long long* t = g_trace;
    if (t != nullptr) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(now));
      atomicMin(t + kid * TRACE_SLOTS + 2 * what, now);
      atomicMax(t + kid * TRACE_SLOTS + 2 * what + 1, now);
    }
  }
}
__device__ __forceinline__ void griddep_wait(int kid) {
  trace_mark(kid, 0);
  asm volatile("griddepcontrol.wait;\n" ::: "memory");
  trace_mark(kid, 1);
}
// fine-grained event log of CTA 0 (debug view of a kernel's pipeline): lane 0 of every warp appends {globaltimer, id, arg}
// to the warp's own region of the buffer with plain stores (index in a register: no atomics, nothing to wait for)
static __device__ unsigned long long* g_evt = nullptr;
constexpr unsigned int EVT_PER_WARP = 1024, EVT_WARPS = 16;
struct EvtLog {                      // per-thread cursor; `base` is read ONCE (a load per mark would sit on CTA 0's critical path)
  unsigned long long* base;
  unsigned int i;
};
__device__ __forceinline__ EvtLog evt_open() {
  EvtLog l;
  l.base = (blockIdx.x == 0 && (threadIdx.x & 31) == 0) ? g_evt : nullptr;
  l.i = 0;
  return l;
}
__device__ __forceinline__ void evt_mark(EvtLog& l, int id, int arg) {
  if (l.base != nullptr && l.i < EVT_PER_WARP) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(now));
    const unsigned int slot = (threadIdx.x >> 5) * EVT_PER_WARP + l.i++;
    l.base[2 * slot] = now;
    l.base[2 * slot + 1] = ((unsigned long long)(threadIdx.x >> 5) << 32) | ((unsigned long long)id << 16) | (unsigned long long)(arg & 0xFFFF);
  }
}
#define GA3C_EVT_ATTACH(fn) \
  int fn(unsigned long long* buf) { return (int)cudaMemcpyToSymbol(g_evt, &buf, sizeof(buf)); }
#define GA3C_TRACE_ATTACH(fn)                                                                   \
  int fn(unsigned long long* buf) { return (int)cudaMemcpyToSymbol(g_trace, &buf, sizeof(buf)); }

template <class... KArgs, class... Args>
inline int launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return (int)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float sigmoid(float z) { return 1.f / (1.f + expf(-z)); }

// ---- swizzles shared by producer and consumer kernels -----------------------------------------
// padded conv11 output (n1p): pixel (py, px) in 24x24, 32 B per pixel, two 16-B chunks.
//   slot(px): rotate the low 3 bits of px right by one, so px, px+2, px+4, px+6 land in four
//   different 32-B bank groups; the 16-B chunk is XORed with bit 3 of px so 8 stride-2 pixels
//   reading one chunk each are conflict-free under ldmatrix.
__device__ __forceinline__ int n1p_slot(int px) { return (px & ~7) | ((px >> 1) & 3) | ((px & 1) << 2); }
__device__ __forceinline__ int n1p_off(int py, int px, int chunk) {
  return ((py * N1P_W + n1p_slot(px)) << 5) + (((chunk ^ (px >> 3)) & 1) << 4);
}

// stage one fp32 frame (28224 floats, NHWC) into the padded bf16 smem image; NT threads cooperate
template <int NT>
__device__ __forceinline__ void stage_frame_bf16(const float* __restrict__ x, uint32_t xs_base, int tid) {
  const float4* src = reinterpret_cast<const float4*>(x);
  constexpr int NPIX = IMG * IMG;          // 7056 pixels, one float4 each
  constexpr int UNROLL = 7;
  for (int base = 0; base < NPIX; base += NT * UNROLL) {
    float4 v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      int i = base + u * NT + tid;
      if (i < NPIX) v[u] = ldg_stream(src + i);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      int i = base + u * NT + tid;
      if (i < NPIX) {
        int y = i / IMG, xx = i - y * IMG;
        sts64(xs_base + (y + 2) * XS_ROW_BYTES + (xx + 2) * 8, pack_bf16(v[u].x, v[u].y), pack_bf16(v[u].z, v[u].w));
      }
    }
  }
}

}  // namespace ga3c
