// Histograms of the TensorBoard summaries Network.log writes (NetworkVP.py:152-173, :259-265): TensorFlow's
// histogram::Histogram (min, max, num, sum, sum_squares and 1551 exponential buckets) of every variable and activation, on the
// device.  At B = 1024 that is ~12.4 M values in ~27 MB of HBM; only the 15 x 1556 doubles of the result go back to the host.
//
// One pass (histo_kernel): every block takes a range of 16-byte chunks of ONE source (4 fp32 or 8 bf16 values), counts its values
// into a shared-memory histogram and adds the non-empty buckets to the source's 64-bit integer counters in the output (integer
// atomics: the counts do not depend on the order blocks finish in).  Its fp64 partial moments go to a scratch row per block, which
// histo_merge_kernel sums in block order: the output is bit-identical from call to call.
//
// Bucket of x (TF: std::upper_bound over the limits) = the number of limits <= double(x).  With P = the 775 positive limits
// (1e-12 * 1.1^k by repeated fp64 multiplication while < 1e20, then DBL_MAX) the limits are -P reversed, 0.0, P, so
//   x > 0: 776 + #{P <= x}        x < 0: 775 - #{P < |x|}        x == 0 (either sign): 776.
// The count is guessed from log2|x| and corrected against the fp64 table in shared memory: exact for every input.
// Post-ReLU sources are mostly exact zeros, all in bucket 776: each thread counts them in a register and every warp adds its
// total once, so they never contend for the shared counter.
#include <cfloat>
#include <cmath>
#include <mutex>
#include <vector>

#include "../../include/ga3c_b200.h"
#include "common.cuh"
#include "kernels.h"
#include "host_util.h"

namespace ga3c {
namespace {

constexpr int HB = GA3C_HISTO_BUCKETS;     // 1551
constexpr int NPOS = 775;                  // positive limits, DBL_MAX included
constexpr int ZERO_BUCKET = 776;           // upper_bound of 0.0: the 775 negative limits and 0.0 itself are <= 0
constexpr int HT = 256;                    // threads per block
constexpr int CPB = 4096;                  // 16-byte chunks per block (64 KB of input)
constexpr int UNROLL = 4;                  // chunk loads a thread keeps in flight
constexpr int ROW = 5 + HB;                // output doubles per source

__device__ double g_pos_limits[NPOS];

// chunk cc of an n1 image in the Blk2 layout ([frame][8 planes][160 rows][8 bf16], common.cuh) holds channels 8h.. of pixel
// (Y - 1, X - 1) of the zero-padded 24 x 24 image; only 1 <= Y, X <= 21 are live, everything else is border or slack
__device__ __forceinline__ bool blk2_live(unsigned cc) {
  const int c = (int)(cc % (unsigned)(B2_BYTES / 16));
  const int plane = c / B2_ROWS, r = c - plane * B2_ROWS;
  const int yb = r / G_W, xb = r - yb * G_W;
  const int y = 2 * yb + ((plane >> 2) & 1), x = 2 * xb + ((plane >> 1) & 1);
  return y >= 1 && y <= H1 && x >= 1 && x <= H1;
}

// f finite and non-zero
__device__ __forceinline__ int bucket_of(float f, const double* P) {
  const double a = fabs((double)f);
  int k = 0;
  if (a >= P[0]) {
    // log2(1e-12) = -39.863..., 1 / log2(1.1) = 7.2725...: the guess is within one or two of the answer
    const int g = (int)((__log2f(fabsf(f)) + 39.863137f) * 7.2725409f) + 1;
    k = min(max(g, 1), NPOS - 1);
    if (f > 0.f) {                         // P[k-1] <= a < P[k]; P[0] <= a and P[NPOS-1] = DBL_MAX > a bound both loops
      while (P[k] <= a) ++k;
      while (P[k - 1] > a) --k;
    } else {                               // P[k-1] < a <= P[k]
      while (P[k] < a) ++k;
      while (k > 0 && P[k - 1] >= a) --k;
    }
  }
  return f > 0.f ? ZERO_BUCKET + k : ZERO_BUCKET - 1 - k;
}

struct Acc {
  float mn = INFINITY, mx = -INFINITY;
  double sum = 0.0, sumsq = 0.0;
  unsigned zeros = 0;
  bool bad = false;

  __device__ __forceinline__ void add(float f, unsigned* cnt, const double* P) {
    if (!isfinite(f)) { bad = true; return; }
    mn = fminf(mn, f);
    mx = fmaxf(mx, f);
    if (f == 0.f) { ++zeros; return; }
    const double d = f;
    sum += d;
    sumsq += d * d;                        // exact: a product of two floats fits a double
    atomicAdd(cnt + bucket_of(f, P), 1u);
  }
};

// KIND 0: fp32, 1: bf16, 2: bf16 in the Blk2 layout (border chunks are not even loaded).  Chunk indices of a source fit 32 bits
// (histo_plan).  The UNROLL loads are issued together; the values are then consumed from v[0] with the registers shifted down,
// so that the bucket search is instantiated once per kind instead of UNROLL times.
template <int KIND>
__device__ __forceinline__ void run_chunks(const uint4* p, unsigned c0, unsigned c1, Acc& acc, unsigned* cnt, const double* P) {
  for (unsigned c = c0 + threadIdx.x; c < c1; c += UNROLL * HT) {
    uint4 v[UNROLL];
    bool ok[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const unsigned cc = c + u * HT;
      ok[u] = cc < c1 && (KIND != 2 || blk2_live(cc));
      if (ok[u]) v[u] = __ldcs(p + cc);
    }
#pragma unroll 1
    for (int u = 0; u < UNROLL; ++u) {
      if (ok[0]) {
        const uint32_t w[4] = {v[0].x, v[0].y, v[0].z, v[0].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (KIND == 0) {
            acc.add(__uint_as_float(w[j]), cnt, P);
          } else {
            acc.add(bf16_lo(w[j]), cnt, P);
            acc.add(bf16_hi(w[j]), cnt, P);
          }
        }
      }
#pragma unroll
      for (int k = 0; k + 1 < UNROLL; ++k) { v[k] = v[k + 1]; ok[k] = ok[k + 1]; }
    }
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ int source_of(const HistoArgs& a, int blk) {
  int s = 0;
  while (blk >= a.blk_end[s]) ++s;
  return s;
}

__global__ void __launch_bounds__(HT) histo_kernel(const HistoArgs a) {
  __shared__ double s_pos[NPOS];
  __shared__ unsigned s_cnt[HB];
  __shared__ double s_sum[HT / 32], s_sq[HT / 32];
  __shared__ float s_mn[HT / 32], s_mx[HT / 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int s = source_of(a, blockIdx.x);
  const void* const src_p = a.src[s].p;       // field by field: a copy of the struct would go through local memory
  const long long src_n = a.src[s].n;
  const int src_bf16 = a.src[s].bf16, src_blk2 = a.src[s].blk2;
  for (int i = tid; i < NPOS; i += HT) s_pos[i] = g_pos_limits[i];
  for (int i = tid; i < HB; i += HT) s_cnt[i] = 0u;
  __syncthreads();

  Acc acc;
  const int width = src_bf16 ? 8 : 4;
  const long long nch = src_n / width;
  const unsigned c0 = (unsigned)(blockIdx.x - (s ? a.blk_end[s - 1] : 0)) * CPB;
  const unsigned c1 = c0 + CPB < nch ? c0 + CPB : (unsigned)nch;
  const uint4* p = static_cast<const uint4*>(src_p);
  if (!src_bf16) run_chunks<0>(p, c0, c1, acc, s_cnt, s_pos);
  else if (src_blk2) run_chunks<2>(p, c0, c1, acc, s_cnt, s_pos);
  else run_chunks<1>(p, c0, c1, acc, s_cnt, s_pos);
  if (c1 == nch) {                         // the last block of the source also takes the < width values after the last chunk
    const long long e = nch * width + tid;
    if (e < src_n) {
      const float f = src_bf16 ? __uint_as_float((uint32_t)static_cast<const uint16_t*>(src_p)[e] << 16)
                               : static_cast<const float*>(src_p)[e];
      acc.add(f, s_cnt, s_pos);
    }
  }

  const unsigned z = __reduce_add_sync(0xffffffffu, acc.zeros);
  const double sum = warp_sum(acc.sum), sq = warp_sum(acc.sumsq);
  const float mn = warp_min(acc.mn), mx = warp_max(acc.mx);
  if (lane == 0) {
    if (z) atomicAdd(s_cnt + ZERO_BUCKET, z);
    s_sum[warp] = sum; s_sq[warp] = sq; s_mn[warp] = mn; s_mx[warp] = mx;
  }
  const int bad = __syncthreads_or(acc.bad);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(a.out + (size_t)s * ROW + 5);
  for (int i = tid; i < HB; i += HT)
    if (s_cnt[i]) atomicAdd(counts + i, (unsigned long long)s_cnt[i]);
  if (tid == 0) {
    double t_sum = 0.0, t_sq = 0.0;
    float t_mn = INFINITY, t_mx = -INFINITY;
    for (int w = 0; w < HT / 32; ++w) {
      t_sum += s_sum[w]; t_sq += s_sq[w]; t_mn = fminf(t_mn, s_mn[w]); t_mx = fmaxf(t_mx, s_mx[w]);
    }
    double* part = a.part + 4 * (size_t)blockIdx.x;
    part[0] = t_mn; part[1] = t_mx; part[2] = t_sum; part[3] = t_sq;
    if (bad) a.bad[s] = 1;
  }
}

// one block per source: the blocks' partial moments in block order, the integer counts turned into doubles in place, num
__global__ void __launch_bounds__(HT) histo_merge_kernel(const HistoArgs a) {
  __shared__ double s_sum[HT / 32], s_sq[HT / 32];
  __shared__ float s_mn[HT / 32], s_mx[HT / 32];
  __shared__ unsigned long long s_num[HT / 32];
  const int s = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b0 = s ? a.blk_end[s - 1] : 0, b1 = a.blk_end[s];
  double sum = 0.0, sq = 0.0;
  float mn = INFINITY, mx = -INFINITY;
  for (int b = b0 + tid; b < b1; b += HT) {
    const double* part = a.part + 4 * (size_t)b;
    mn = fminf(mn, (float)part[0]); mx = fmaxf(mx, (float)part[1]); sum += part[2]; sq += part[3];
  }
  double* row = a.out + (size_t)s * ROW;
  unsigned long long num = 0;
  for (int i = tid; i < HB; i += HT) {
    unsigned long long* slot = reinterpret_cast<unsigned long long*>(row + 5 + i);
    const unsigned long long c = *slot;
    num += c;
    row[5 + i] = (double)c;
  }
  num = __reduce_add_sync(0xffffffffu, (unsigned)num);     // a source holds < 2^32 values (histo_plan)
  sum = warp_sum(sum); sq = warp_sum(sq); mn = warp_min(mn); mx = warp_max(mx);
  if (lane == 0) { s_sum[warp] = sum; s_sq[warp] = sq; s_mn[warp] = mn; s_mx[warp] = mx; s_num[warp] = num; }
  __syncthreads();
  if (tid == 0) {
    double t_sum = 0.0, t_sq = 0.0;
    float t_mn = INFINITY, t_mx = -INFINITY;
    unsigned long long t_num = 0;
    for (int w = 0; w < HT / 32; ++w) {
      t_sum += s_sum[w]; t_sq += s_sq[w]; t_mn = fminf(t_mn, s_mn[w]); t_mx = fmaxf(t_mx, s_mx[w]); t_num += s_num[w];
    }
    row[0] = t_mn == INFINITY ? DBL_MAX : (double)t_mn;          // TF starts min / max at +-DBL_MAX
    row[1] = t_mx == -INFINITY ? -DBL_MAX : (double)t_mx;
    row[2] = (double)t_num;
    row[3] = t_sum;
    row[4] = t_sq;
  }
}

// the positive limits, built exactly as TF builds them (fp64, repeated multiplication), copied once per device
int upload_limits() {
  static std::mutex mtx;
  static std::vector<int> done;
  int dev = 0;
  CK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mtx);
  if ((int)done.size() <= dev) done.resize(dev + 1, 0);
  if (done[dev]) return 0;
  std::vector<double> pos;
  for (double v = 1e-12; v < 1e20; v *= 1.1) pos.push_back(v);
  pos.push_back(DBL_MAX);
  if ((int)pos.size() != NPOS) return set_error("histograms: unexpected bucket-limit count");
  CK(cudaMemcpyToSymbol(g_pos_limits, pos.data(), sizeof(double) * NPOS));
  done[dev] = 1;
  return 0;
}

}  // namespace

int histo_plan(HistoArgs& a) {
  if (a.n_src < 1 || a.n_src > HISTO_MAX_SRC) return set_error("histograms: 1.." + std::to_string(HISTO_MAX_SRC) + " sources");
  long long blocks = 0;
  for (int s = 0; s < a.n_src; ++s) {
    const HistoSrc& src = a.src[s];
    if (!src.p || src.n < 1 || src.n > 0xffffffffll) return set_error("histograms: each source holds 1..2^32-1 values");
    if (reinterpret_cast<uintptr_t>(src.p) % 16) return set_error("histograms: source buffers must be 16-byte aligned");
    const long long nch = src.n / (src.bf16 ? 8 : 4);
    blocks += nch > 0 ? (nch + CPB - 1) / CPB : 1;
    if (blocks > 0x7fffffffll) return set_error("histograms: too many values");
    a.blk_end[s] = (int)blocks;
  }
  return 0;
}

int histo_blocks(const HistoArgs& a) { return a.blk_end[a.n_src - 1]; }

int histo_zero(const HistoArgs& a, cudaStream_t st) {
  if (int r = upload_limits()) return r;
  CK(cudaMemsetAsync(a.out, 0, sizeof(double) * ROW * a.n_src, st));
  CK(cudaMemsetAsync(a.bad, 0, sizeof(int32_t) * a.n_src, st));
  return 0;
}

int launch_histo(const HistoArgs& a, cudaStream_t st) {
  histo_kernel<<<histo_blocks(a), HT, 0, st>>>(a);
  CK(cudaGetLastError());
  return 0;
}

int launch_histo_merge(const HistoArgs& a, cudaStream_t st) {
  histo_merge_kernel<<<a.n_src, HT, 0, st>>>(a);
  CK(cudaGetLastError());
  return 0;
}

}  // namespace ga3c

extern "C" int ga3c_debug_histogram(const void* x, int32_t dtype, int64_t n, double* out, int32_t* bad, void* stream) {
  using namespace ga3c;
  if (!x || !out || !bad || (dtype != 0 && dtype != 1)) return set_error("ga3c_debug_histogram: bad argument");
  HistoArgs a{};
  a.n_src = 1;
  a.src[0] = HistoSrc{x, (long long)n, dtype, 0};
  a.out = out;
  a.bad = bad;
  if (int r = histo_plan(a)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMallocAsync((void**)&a.part, sizeof(double) * 4 * histo_blocks(a), st));
  int r = histo_zero(a, st);
  if (!r && (r = launch_histo(a, st)) == 0) r = launch_histo_merge(a, st);
  cudaFreeAsync(a.part, st);
  return r;
}
