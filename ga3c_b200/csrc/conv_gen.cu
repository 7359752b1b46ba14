// The conv trunk for any input geometry (Config.IMAGE_HEIGHT, IMAGE_WIDTH, STACKED_FRAMES) other than 84x84x4, which keeps
// its specialised kernels (conv_fwd.cu, conv_bwd_fused.cu).  Same layers (NetworkDNav.py:81-90): conv11 8x8 stride 4 -> 16,
// conv12 4x4 stride 2 -> 32, TF SAME padding (low side smaller), ReLU.  Each conv is an im2col gather and a GEMM on the
// tcgen05 core of gemm_tc.cuh; the GEMMs' epilogues apply bias + ReLU (forward) or write the weight-gradient slabs (backward).
//
//   forward   X1 [P1][64C | 1]  = im2col(x)             P1 = B*H1*W1, columns (kh, kw, c), then a column of ones
//             n1 [P1][16]       = relu(X1 W11 + b11)     bf16; GEMM N = 16: an N = 16 UMMA, half-width tcgen05.ld
//             X2 [P2][256 | 1]  = im2col(n1)            P2 = B*H2*W2, columns (kh, kw, ci)
//             n2 [P2][32]       = relu(X2 W12 + b12)     = [B][H2*W2*32], the (h, w, c) flatten dense1 reads
//   backward  dx2 [P2][256]     = dn2 W12^T              fp32
//             dn1 [P1][16]      = col2im(dx2) * (n1 > 0) gather form: every output sums its (at most 4) taps in a fixed order
//             [gW12^T | gb12]   = dn2^T [X2 | 1]         over P2, split into k-block ranges -> one gradient-partial slab each
//             [gW11^T | gb11]   = dn1^T [X1 | 1]         likewise over P1
// The bias gradients are the column sums of dn2 / dn1: the ones column of X2 / X1 makes them the last column of the
// weight-gradient GEMM.  bf16 rounding points as on the 84x84x4 path: frames, n1, n2, dn2, dn1, the conv weights as GEMM
// operands; fp32 accumulation.
#include <cstdio>

#include "gemm_tc.cuh"

namespace ga3c {

GenGeom gen_geom(int h, int w, int c) {
  GenGeom g{};
  g.h = h; g.w = w; g.c = c;
  auto same = [](int n, int k, int s, int* out, int* before) {
    *out = (n + s - 1) / s;
    const int total = (*out - 1) * s + k - n;
    *before = total > 0 ? total / 2 : 0;
  };
  same(h, 8, 4, &g.h1, &g.pt1); same(w, 8, 4, &g.w1, &g.pl1);
  same(g.h1, 4, 2, &g.h2, &g.pt2); same(g.w1, 4, 2, &g.w2, &g.pl2);
  g.k1 = 64 * c; g.ld1 = g.k1 + 8;
  g.kdim = g.h2 * g.w2 * C2_OUT;
  return g;
}

// ---- epilogues -------------------------------------------------------------------------------------------------------------
template <int NC>           // NC (16 or 32) accumulator columns -> relu(acc + bias) as bf16, row-major
struct EpiBiasReluBf16 {
  uint16_t* out; const float* bias; int ldc;
  struct Pre {};
  __device__ __forceinline__ void prefetch(Pre&, int, int, bool) const {}
  __device__ __forceinline__ void operator()(const Pre&, int, int m, int n, const uint32_t (&r)[32]) const {
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)m * ldc + n);
#pragma unroll
    for (int i = 0; i < NC / 8; ++i) {
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = 8 * i + 2 * j;
        o[j] = pack_bf16(fmaxf(__uint_as_float(r[k]) + __ldg(bias + n + k), 0.f),
                         fmaxf(__uint_as_float(r[k + 1]) + __ldg(bias + n + k + 1), 0.f));
      }
      dst[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
};

// weight-gradient GEMM (transposed: row m = output channel, column n = tap of the im2col row, column kdim = the ones column)
// -> slab `split` of the gradient partials: w[tap * co + m], b[m].  A split whose k-block range is empty writes zeros, so every
// slab the reduction reads is written.
struct EpiConvWgrad {
  float *gw, *gb; int co, kdim; int64_t stride; int kb_total, kb_per;
  struct Pre {};
  __device__ __forceinline__ void prefetch(Pre&, int, int, bool) const {}
  __device__ __forceinline__ void operator()(const Pre&, int split, int m, int n, const uint32_t (&r)[32]) const {
    const bool empty = split * kb_per >= kb_total;
    float* w = gw + split * stride;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int k = n + j;
      const float v = empty ? 0.f : __uint_as_float(r[j]);
      if (k < kdim) w[(size_t)k * co + m] = v;
      else if (k == kdim) gb[split * stride + m] = v;
    }
  }
};

// ---- gathers ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void gen_begin(int kid) { griddep_wait(kid); griddep_launch(); }

// conv11/w [64C][16], conv12/w [256][32] (TF HWIO, fp32) -> bf16 W11^T [16][64C], W12^T [32][256], W12 [256][32]
__global__ void gen_wprep_kernel(const float* __restrict__ w11, const float* __restrict__ w12, uint16_t* w11t, uint16_t* w12t,
                                 uint16_t* w12bf, int k1) {
  gen_begin(K_GEN_WPREP);
  const int n11 = 16 * k1, n12 = 32 * 256;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n11 + 2 * n12; i += gridDim.x * blockDim.x) {
    float v;
    uint16_t* dst;
    if (i < n11) {
      const int co = i / k1, k = i - co * k1;
      v = w11[k * 16 + co]; dst = w11t + i;
    } else if (i < n11 + n12) {
      const int j = i - n11, co = j >> 8, k = j & 255;
      v = w12[k * 32 + co]; dst = w12t + j;
    } else {
      const int j = i - n11 - n12;
      v = w12[j]; dst = w12bf + j;
    }
    *dst = __bfloat16_as_ushort(__float2bfloat16_rn(v));
  }
  trace_mark(K_GEN_WPREP, 2);
}

// X1: one thread per 16-byte chunk (8 columns) of a row; chunk 8C is {1, 0, ..., 0}.  Columns (kh, kw, c): the C chunks of
// one kh are 8 consecutive pixels of one frame row, each pixel bounds-checked (SAME zero padding).
template <bool U8>
__global__ void gen_im2col1_kernel(const void* __restrict__ xv, uint16_t* __restrict__ x1, GenGeom g, int64_t chunks) {
  gen_begin(K_GEN_IM2COL1);
  const int per_row = 8 * g.c + 1;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < chunks; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = t / per_row;
    const int ch = (int)(t - row * per_row);
    uint32_t o[4] = {0, 0, 0, 0};
    if (ch == 8 * g.c) {
      o[0] = 0x3F80u;                                    // bf16 1.0 in the low half
    } else {
      const int npos = g.h1 * g.w1;
      const int b = (int)(row / npos), pos = (int)(row - (int64_t)b * npos);
      const int oy = pos / g.w1, ox = pos - oy * g.w1;
      const int kh = ch / g.c, e0 = (ch - kh * g.c) * 8;      // first element of (kw, c) inside the kh row
      const int iy = oy * 4 - g.pt1 + kh;
      if (iy >= 0 && iy < g.h) {
        const int64_t rowbase = ((int64_t)b * g.h + iy) * g.w;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int e = e0 + j, kw = e / g.c, cc = e - kw * g.c, ix = ox * 4 - g.pl1 + kw;
          v[j] = 0.f;
          if (ix >= 0 && ix < g.w) {
            const int64_t idx = (rowbase + ix) * g.c + cc;
            v[j] = U8 ? (float)static_cast<const uint8_t*>(xv)[idx] * (1.f / 128.f) - 1.f     // Environment.py:60, exact
                      : __ldg(static_cast<const float*>(xv) + idx);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = pack_bf16(v[2 * j], v[2 * j + 1]);
      }
    }
    *reinterpret_cast<uint4*>(x1 + row * g.ld1 + ch * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
  trace_mark(K_GEN_IM2COL1, 2);
}

// X2: one thread per 16-byte chunk: chunk 2 * tap + half = channels [8 half, 8 half + 8) of n1 at tap (kh, kw); chunk 32 = ones
__global__ void gen_im2col2_kernel(const uint16_t* __restrict__ n1, uint16_t* __restrict__ x2, GenGeom g, int64_t chunks) {
  gen_begin(K_GEN_IM2COL2);
  constexpr int per_row = GEN_LD2 / 8;                     // 33
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < chunks; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = t / per_row;
    const int ch = (int)(t - row * per_row);
    uint4 o = make_uint4(0, 0, 0, 0);
    if (ch == 32) {
      o.x = 0x3F80u;
    } else {
      const int npos = g.h2 * g.w2;
      const int b = (int)(row / npos), pos = (int)(row - (int64_t)b * npos);
      const int oy = pos / g.w2, ox = pos - oy * g.w2;
      const int tap = ch >> 1, kh = tap >> 2, kw = tap & 3;
      const int iy = oy * 2 - g.pt2 + kh, ix = ox * 2 - g.pl2 + kw;
      if (iy >= 0 && iy < g.h1 && ix >= 0 && ix < g.w1)
        o = __ldg(reinterpret_cast<const uint4*>(n1 + ((((int64_t)b * g.h1 + iy) * g.w1 + ix) * 16 + (ch & 1) * 8)));
    }
    *reinterpret_cast<uint4*>(x2 + row * GEN_LD2 + ch * 8) = o;
  }
  trace_mark(K_GEN_IM2COL2, 2);
}

// dn1: one thread per 8 channels of one conv11 output pixel: the sum of the dx2 entries of the conv12 taps that read it
// (kh, kw ascending), masked by n1 > 0, rounded to bf16
__global__ void gen_col2im_kernel(const float* __restrict__ dx2, const uint16_t* __restrict__ n1, uint16_t* __restrict__ dn1,
                                  GenGeom g, int64_t items) {
  gen_begin(K_GEN_COL2IM);
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < items; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t px = t >> 1;
    const int half = (int)(t & 1);
    const int npos = g.h1 * g.w1;
    const int b = (int)(px / npos), pos = (int)(px - (int64_t)b * npos);
    const int y = pos / g.w1, x = pos - y * g.w1;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int kh = 0; kh < 4; ++kh) {
      const int ty = y + g.pt2 - kh;
      if (ty < 0 || (ty & 1) || (ty >> 1) >= g.h2) continue;
      for (int kw = 0; kw < 4; ++kw) {
        const int tx = x + g.pl2 - kw;
        if (tx < 0 || (tx & 1) || (tx >> 1) >= g.w2) continue;
        const float4* s = reinterpret_cast<const float4*>(
            dx2 + (((int64_t)b * g.h2 + (ty >> 1)) * g.w2 + (tx >> 1)) * 256 + (kh * 4 + kw) * 16 + half * 8);
        const float4 a0 = __ldg(s), a1 = __ldg(s + 1);
        acc[0] += a0.x; acc[1] += a0.y; acc[2] += a0.z; acc[3] += a0.w;
        acc[4] += a1.x; acc[5] += a1.y; acc[6] += a1.z; acc[7] += a1.w;
      }
    }
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(n1 + px * 16 + half * 8));
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      o[j] = pack_bf16((aw[j] & 0x7FFFu) ? acc[2 * j] : 0.f, (aw[j] & 0x7FFF0000u) ? acc[2 * j + 1] : 0.f);
    *reinterpret_cast<uint4*>(dn1 + px * 16 + half * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
  trace_mark(K_GEN_COL2IM, 2);
}

GA3C_TRACE_ATTACH(trace_attach_conv_gen)

// ---- host side --------------------------------------------------------------------------------------------------------------
constexpr int C11_BN = 16, C11_ST = 4;      // conv11 fwd: M = P1, N = 16,  K = 64C
constexpr int C12_BN = 32, C12_ST = 4;      // conv12 fwd: M = P2, N = 32,  K = 256
constexpr int CDG_BN = 128, CDG_ST = 2;     // conv12 data gradient: M = P2, N = 256, K = 32
constexpr int CWG_BN = 64, CWG_ST = 4;      // weight gradients: M = 16 / 32, N = 64C + 1 / 257, K = P1 / P2 (split)

#define GEN_C11 gemm_tc_kernel<C11_BN, C11_ST, false, false, EpiBiasReluBf16<16>, K_GEN_CONV11>
#define GEN_C12 gemm_tc_kernel<C12_BN, C12_ST, false, false, EpiBiasReluBf16<32>, K_GEN_CONV12>
#define GEN_CDG gemm_tc_kernel<CDG_BN, CDG_ST, false, false, EpiPartialF32, K_GEN_CONV12_DGRAD>
#define GEN_W12 gemm_tc_kernel<CWG_BN, CWG_ST, true, true, EpiConvWgrad, K_GEN_CONV12_WGRAD>
#define GEN_W11 gemm_tc_kernel<CWG_BN, CWG_ST, true, true, EpiConvWgrad, K_GEN_CONV11_WGRAD>

int configure_conv_gen() {
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(GEN_C11, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<C11_BN, C11_ST>())) ||
      (e = cudaFuncSetAttribute(GEN_C12, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<C12_BN, C12_ST>())) ||
      (e = cudaFuncSetAttribute(GEN_CDG, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<CDG_BN, CDG_ST>())) ||
      (e = cudaFuncSetAttribute(GEN_W12, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<CWG_BN, CWG_ST>())) ||
      (e = cudaFuncSetAttribute(GEN_W11, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem<CWG_BN, CWG_ST>())))
    return (int)e;
  return 0;
}

static int grid_for(int64_t items, int threads) {
  const int64_t b = (items + threads - 1) / threads;
  return (int)(b < 1 ? 1 : b > (1 << 20) ? (1 << 20) : b);
}

int launch_gen_wprep(const GenGeom& g, const GenBufs& b, const float* w11, const float* w12, cudaStream_t st) {
  const int n = 16 * g.k1 + 2 * 32 * 256;
  return launch_pdl(gen_wprep_kernel, dim3(grid_for(n, 256)), dim3(256), 0, st, w11, w12, b.w11t, b.w12t, b.w12, g.k1);
}

int launch_gen_im2col1(const GenGeom& g, const GenBufs& b, const void* x, bool x_u8, int batch, cudaStream_t st) {
  const int64_t chunks = (int64_t)batch * g.h1 * g.w1 * (8 * g.c + 1);
  if (x_u8) return launch_pdl(gen_im2col1_kernel<true>, dim3(grid_for(chunks, 256)), dim3(256), 0, st, x, b.x1, g, chunks);
  return launch_pdl(gen_im2col1_kernel<false>, dim3(grid_for(chunks, 256)), dim3(256), 0, st, x, b.x1, g, chunks);
}

int launch_gen_conv11(const GenGeom& g, const GenBufs& b, const float* b11, int batch, cudaStream_t st) {
  const int64_t p1 = (int64_t)batch * g.h1 * g.w1;
  CUtensorMap ta, tb;
  if (make_tmap(&ta, b.x1, p1, g.k1, g.ld1, TC_BM)) return (int)cudaErrorInvalidValue;        // A: X1 [P1][64C], K inner
  if (make_tmap(&tb, b.w11t, 16, g.k1, g.k1, C11_BN)) return (int)cudaErrorInvalidValue;      // B: W11^T [16][64C] = [N][K]
  const int kb = (g.k1 + TC_BK - 1) / TC_BK;
  return launch_pdl(GEN_C11, dim3((unsigned)((p1 + TC_BM - 1) / TC_BM), 1, 1), dim3(TC_THREADS), tc_smem<C11_BN, C11_ST>(), st,
                    ta, tb, (int)p1, 16, kb, kb, EpiBiasReluBf16<16>{b.n1, b11, 16}, DpGate{});
}

int launch_gen_im2col2(const GenGeom& g, const GenBufs& b, int batch, cudaStream_t st) {
  const int64_t chunks = (int64_t)batch * g.h2 * g.w2 * (GEN_LD2 / 8);
  return launch_pdl(gen_im2col2_kernel, dim3(grid_for(chunks, 256)), dim3(256), 0, st, (const uint16_t*)b.n1, b.x2, g, chunks);
}

int launch_gen_conv12(const GenGeom& g, const GenBufs& b, const float* b12, int batch, cudaStream_t st) {
  const int64_t p2 = (int64_t)batch * g.h2 * g.w2;
  CUtensorMap ta, tb;
  if (make_tmap(&ta, b.x2, p2, 256, GEN_LD2, TC_BM)) return (int)cudaErrorInvalidValue;       // A: X2 [P2][256], K inner
  if (make_tmap(&tb, b.w12t, 32, 256, 256, C12_BN)) return (int)cudaErrorInvalidValue;        // B: W12^T [32][256] = [N][K]
  return launch_pdl(GEN_C12, dim3((unsigned)((p2 + TC_BM - 1) / TC_BM), 1, 1), dim3(TC_THREADS), tc_smem<C12_BN, C12_ST>(), st,
                    ta, tb, (int)p2, 32, 256 / TC_BK, 256 / TC_BK, EpiBiasReluBf16<32>{b.n2, b12, 32}, DpGate{});
}

int gen_wgrad_slabs(const GenGeom& g, int batch, int num_sms) {
  const int64_t kb2 = ((int64_t)batch * g.h2 * g.w2 + TC_BK - 1) / TC_BK;
  return (int)(kb2 < num_sms ? kb2 : num_sms);
}

int launch_gen_conv12_dgrad(const GenGeom& g, const GenBufs& b, int batch, cudaStream_t st) {
  const int64_t p2 = (int64_t)batch * g.h2 * g.w2;
  CUtensorMap ta, tb;
  if (make_tmap(&ta, b.dn2, p2, 32, 32, TC_BM)) return (int)cudaErrorInvalidValue;            // A: dn2 [P2][32], K inner
  if (make_tmap(&tb, b.w12, 256, 32, 32, CDG_BN)) return (int)cudaErrorInvalidValue;          // B: W12 [256][32] = [N][K]
  return launch_pdl(GEN_CDG, dim3((unsigned)((p2 + TC_BM - 1) / TC_BM), 256 / CDG_BN, 1), dim3(TC_THREADS),
                    tc_smem<CDG_BN, CDG_ST>(), st, ta, tb, (int)p2, 256, 1, 1, EpiPartialF32{b.dx2, 256, 0}, DpGate{});
}

int launch_gen_col2im(const GenGeom& g, const GenBufs& b, int batch, cudaStream_t st) {
  const int64_t items = (int64_t)batch * g.h1 * g.w1 * 2;
  return launch_pdl(gen_col2im_kernel, dim3(grid_for(items, 256)), dim3(256), 0, st, (const float*)b.dx2, (const uint16_t*)b.n1,
                    b.dn1, g, items);
}

// dact^T [co][P] x [X | 1] [P][kdim + 1] over `slabs` k-block ranges of P
template <class Kern>
static int conv_wgrad(Kern kern, const uint16_t* dact, int co, const uint16_t* x, int kdim, int ld, int64_t rows, float* gw,
                      float* gb, int64_t gp_stride, int slabs, cudaStream_t st) {
  CUtensorMap ta, tb;
  if (make_tmap(&ta, dact, rows, co, co, 64)) return (int)cudaErrorInvalidValue;              // A: [K=P][M=co], M inner
  if (make_tmap(&tb, x, rows, kdim + 1, ld, 64)) return (int)cudaErrorInvalidValue;           // B: [K=P][N=kdim+1], N inner
  const int kb = (int)((rows + TC_BK - 1) / TC_BK), per = (kb + slabs - 1) / slabs;
  return launch_pdl(kern, dim3(1, (kdim + 1 + CWG_BN - 1) / CWG_BN, slabs), dim3(TC_THREADS), tc_smem<CWG_BN, CWG_ST>(), st,
                    ta, tb, co, kdim + 1, kb, per, EpiConvWgrad{gw, gb, co, kdim, gp_stride, kb, per}, DpGate{});
}

int launch_gen_conv12_wgrad(const GenGeom& g, const GenBufs& b, float* g_w12, float* g_b12, int64_t gp_stride, int slabs,
                            int batch, cudaStream_t st) {
  return conv_wgrad(GEN_W12, b.dn2, 32, b.x2, 256, GEN_LD2, (int64_t)batch * g.h2 * g.w2, g_w12, g_b12, gp_stride, slabs, st);
}

int launch_gen_conv11_wgrad(const GenGeom& g, const GenBufs& b, float* g_w11, float* g_b11, int64_t gp_stride, int slabs,
                            int batch, cudaStream_t st) {
  return conv_wgrad(GEN_W11, b.dn1, 16, b.x1, g.k1, g.ld1, (int64_t)batch * g.h1 * g.w1, g_w11, g_b11, gp_stride, slabs, st);
}

}  // namespace ga3c
