// Internal launch interface between the C-ABI host layer (net.cu) and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

namespace ga3c {

// step timeline trace: attach (or detach with nullptr) the [K_COUNT][TRACE_SLOTS] uint64 buffer, one call per kernel file
int trace_attach_conv_fwd(unsigned long long* buf);
int trace_attach_conv_bwd_fused(unsigned long long* buf);
int trace_attach_dense_tc(unsigned long long* buf);
int trace_attach_heads(unsigned long long* buf);
int trace_attach_elementwise(unsigned long long* buf);
int trace_attach_conv_gen(unsigned long long* buf);

// pipeline event log of CTA 0 (debug): attach a zeroed [16 warps][1024][2] uint64 buffer (or nullptr)
int evt_attach_conv_fwd(unsigned long long* buf);
int evt_attach_conv_bwd(unsigned long long* buf);
int evt_attach_elementwise(unsigned long long* buf);
int evt_attach_dense_tc(unsigned long long* buf);      // records only in a -DGA3C_DENSE_EVT build

// L2 residency hints on the conv kernels' loads and stores (common.cuh); GA3C_L2_HINTS=0 switches them off (evict_normal)
// bit 0: frames loaded evict_first, bit 1: activations stored evict_last, bit 2: the conv backward loads evict_first.
// Measured at B = 1024 / 4096 (profiles/r2g_l2_hint_sweep.txt): predict gains 3 % from bit 0; the fp32 train step is fastest
// with none of them (the L2 already keeps what fits), the uint8 train step with all three (-2.5 %).  GA3C_L2_HINTS overrides.
inline int l2_hints(bool train, bool x_u8) {
  static const int env = [] { const char* e = getenv("GA3C_L2_HINTS"); return e ? atoi(e) : -1; }();
  if (env >= 0) return env;
  return train ? (x_u8 ? 7 : 0) : 1;
}

// one-time per-process function-attribute setup (dynamic smem opt-in); returns cudaError_t as int
int configure_conv_fwd();
int configure_conv_bwd_fused();
int configure_dense_tc();
int configure_conv_gen();

// conv_fwd.cu -- x fp32 (or uint8, x_u8: k/128 - 1 applied on the fly) [B,28224] -> n2 bf16 [B,3872]; when training also n1 (bf16, in
// the Blk2 operand layout) and xblk (the bf16 block matrix of the frame): both are read back by the conv backward (common.cuh)
int launch_conv_fwd(const void* x, bool x_u8, const float* w11, const float* b11, const float* w12, const float* b12,
                    uint8_t* n1_out, uint8_t* xblk_out, uint16_t* n2_out, int batch, int num_sms, cudaStream_t stream);

// dense_tc.cu -- the three dense1 GEMMs (NetworkDNav.py:90 and its autodiff) on tcgen05 / TMEM / TMA.  fwd leaves `splits` raw fp32 partial tiles
// in d1_part[splits][B][256]; the heads kernel sums them, adds the bias and applies the ReLU.  kdim: dense1's K (FLAT = 3872 at
// 84x84x4, H2 * W2 * 32 on the generic trunk).
int dense_fwd_splits(int batch, int num_sms, int kdim);
// data parallel, side-stream exchange: flags = this rank's comm block + DPC_BIGDONE ([world] x 64 B, u64 step numbers), see
// gemm_tc_body (dense_tc.cu).  flags == nullptr: no gate.
struct DpGate {
  const uint8_t* flags;
  void* err;                        // this rank's error word (bit 16 on a wait that gave up)
  unsigned long long step;          // every flag must have reached this step
  int world;
};
int launch_dense_fwd_tc(const uint16_t* n2, const uint16_t* w1bf, float* d1_part, int batch, int kdim, int splits,
                        cudaStream_t stream, const DpGate* gate = nullptr);
int launch_dense_dgrad_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint8_t* dn2, int batch,
                          cudaStream_t stream);       // dn2 in the G operand layout (common.cuh), borders untouched
int launch_dense_wgrad_tc(const uint16_t* n2, const uint16_t* dd1, float* g_w1, int batch, int kdim, cudaStream_t stream);
// dgrad + wgrad tiles in one grid (both only need dd1): the train step uses this one
int launch_dense_bwd_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint8_t* dn2, float* g_w1, int batch,
                        cudaStream_t stream);
// the generic trunk's forms of the two: dn2 row-major [B][kdim], like n2
int launch_dense_dgrad_rows_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint16_t* dn2, int batch,
                               int kdim, cudaStream_t stream);
int launch_dense_bwd_rows_tc(const uint16_t* dd1, const uint16_t* w1bf, const uint16_t* n2, uint16_t* dn2, float* g_w1,
                             int batch, int kdim, cudaStream_t stream);

// conv_gen.cu -- the conv trunk for any input geometry (H, W, C) other than 84x84x4: im2col gathers and GEMMs on the tcgen05
// core of dense_tc.cu.  All activations are row-major: X1 [B*H1*W1][ld1 = 64C + 8] (the im2col of the frames, column 64C = 1,
// the rest of the pad 0), n1 [B*H1*W1][16], X2 [B*H2*W2][GEN_LD2] (the im2col of n1, column 256 = 1), n2 = [B*H2*W2][32].
constexpr int GEN_LD2 = 264;
struct GenGeom {
  int h, w, c;                 // input
  int h1, w1, pt1, pl1;        // conv11 output size and SAME padding before (top, left)
  int h2, w2, pt2, pl2;        // conv12
  int k1, ld1;                 // conv11 K = 64C and X1's row length
  int kdim;                    // dense1 K = h2 * w2 * 32
};
GenGeom gen_geom(int h, int w, int c);
struct GenBufs {
  uint16_t *x1, *n1, *x2, *n2, *dn2, *dn1;
  float* dx2;                  // [B*H2*W2][256] fp32: conv12's data gradient before col2im
  uint16_t *w11t, *w12t, *w12; // bf16 GEMM operands: conv11/w^T [16][64C], conv12/w^T [32][256], conv12/w [256][32]
};
// forward, one launch each: weights -> bf16 operands, im2col of the frames, conv11 GEMM (bias + ReLU) -> n1, im2col of n1,
// conv12 GEMM (bias + ReLU) -> n2
int launch_gen_wprep(const GenGeom& g, const GenBufs& b, const float* w11, const float* w12, cudaStream_t st);
int launch_gen_im2col1(const GenGeom& g, const GenBufs& b, const void* x, bool x_u8, int batch, cudaStream_t st);
int launch_gen_conv11(const GenGeom& g, const GenBufs& b, const float* b11, int batch, cudaStream_t st);
int launch_gen_im2col2(const GenGeom& g, const GenBufs& b, int batch, cudaStream_t st);
int launch_gen_conv12(const GenGeom& g, const GenBufs& b, const float* b12, int batch, cudaStream_t st);
// backward from dn2: conv12 data gradient -> dx2, col2im + the n1 > 0 mask -> dn1, and the weight / bias gradients of conv12
// and conv11 as `slabs` partial sums (slab s = k-block range s of the GEMM over positions) into the gradient-partial slabs,
// gp_stride floats apart, that launch_grad_reduce sums in a fixed order
int gen_wgrad_slabs(const GenGeom& g, int batch, int num_sms);
int launch_gen_conv12_dgrad(const GenGeom& g, const GenBufs& b, int batch, cudaStream_t st);
int launch_gen_col2im(const GenGeom& g, const GenBufs& b, int batch, cudaStream_t st);
int launch_gen_conv12_wgrad(const GenGeom& g, const GenBufs& b, float* g_w12, float* g_b12, int64_t gp_stride, int slabs,
                            int batch, cudaStream_t st);
int launch_gen_conv11_wgrad(const GenGeom& g, const GenBufs& b, float* g_w11, float* g_b11, int64_t gp_stride, int slabs,
                            int batch, cudaStream_t st);

// heads.cu -- value / policy heads, softmax, A3C loss and its backward (NetworkVP_discrate.py:60-85)
struct HeadsArgs {
  const float* d1_part; // [n_split][B,256] raw split-K partial sums of dense1 (no bias, no ReLU)
  int n_split;
  const float* b1;      // dense1 bias
  float* d1;            // [B,256] out: relu(sum of partials + b1)
  const float *wp, *bp, *wv, *bv;
  const float *yr, *a;  // train only
  int batch, num_actions;
  float beta, log_eps, min_policy;
  float *p_out, *v_out;        // may be null in train mode
  uint16_t* dd1;               // [B,256] bf16, train only
  // train only: this CTA's partial sums go to slab blockIdx.x of the gradient-partial workspace (pointers are
  // into slab 0, consecutive slabs gp_stride floats apart); launch_grad_reduce sums the slabs
  float *g_wp, *g_bp, *g_wv, *g_bv, *g_b1;
  float* loss;                 // [4] (cost_p_1, cost_p_2, cost_v, 0) partial sums, same slab scheme
  int64_t gp_stride;
  int train;
  int log_softmax;             // Config.USE_LOG_SOFTMAX
  int part;                    // Config.DUAL_RMSPROP passes: 0 gradient of cost_all, 1 of cost_p alone, 2 of cost_v alone
  int preload;                 // the head weights may be read before the dependency wait (heads.cu)
};
int heads_grid(int batch, int num_sms);          // CTAs (= slabs written) of a training launch
int launch_heads(const HeadsArgs& args, int num_sms, cudaStream_t stream);

// conv_bwd_fused.cu
// Weight / bias gradients are per-CTA partial sums: CTA i stores into slab i (g_* point into slab 0, slabs are
// gp_stride floats apart) and launch_grad_reduce adds the slabs in a fixed order.  No contended atomics, and the
// step is bit-reproducible.
int conv_bwd_grid(int batch, int num_sms);       // conv CTAs (= slabs written)
// conv_bwd_fused.cu -- conv12 data gradient (dn1, kept on chip; dn1_out: optional copy for tests), conv12 and conv11
// weight / bias gradients in one kernel on tcgen05
int launch_conv_bwd(const uint8_t* xblk, const uint8_t* n1b2, const uint8_t* dn2g, const float* w12, uint16_t* dn1_out,
                    float* g_w11, float* g_b11, float* g_w12, float* g_b12, int64_t gp_stride, int batch, int num_sms, bool x_u8,
                    cudaStream_t stream);

// elementwise.cu
// out[j] = sum over slabs i < count(j) of part[i * stride + j], j in [0, n_floats): the per-CTA gradient partials of
// the heads / conv12_bwd / conv11_wgrad kernels -> the small-tensor prefix of the gradient arena (+ the loss sums).
constexpr int GR_MAX_SEG = 4;
struct GradReduceArgs {
  const float* part;
  int64_t stride;
  float* out;                       // floats [0, out_floats) go here ...
  float* out_tail;                  // ... and floats [out_floats, n_floats) here (the loss sums; may be null)
  int out_floats, n_floats;         // multiples of 4
  int seg_end[GR_MAX_SEG];          // segment s covers [seg_end[s-1], seg_end[s]) and sums seg_count[s] slabs
  int seg_count[GR_MAX_SEG];
};
int launch_grad_reduce(const GradReduceArgs& a, cudaStream_t stream);
struct RmsPropArgs {
  float *w, *ms, *mom;
  const float* g;
  uint16_t* w1_shadow;     // bf16 shadow of dense1/w
  int64_t n_floats;        // arena size (multiple of 4)
  int64_t w1_offset, w1_count;
  float lr, decay, momentum, eps;
  int preload;             // the optimizer kernels may load w / ms / mom before their dependency wait (elementwise.cu, preload rule)
};
// Config.USE_GRAD_CLIP: tf.clip_by_average_norm per variable before RMSProp.  offset / count: the variables' element ranges in
// the arena; chunk_ss: [n_tensors][max_chunks] scratch, max_chunks = clip_chunks(largest count); scale: [n_tensors] scratch.
constexpr int CLIP_MAX_TENSORS = 24;
struct ClipArgs {
  const float* g;
  int n_tensors, max_chunks;
  int64_t offset[CLIP_MAX_TENSORS], count[CLIP_MAX_TENSORS];
  float clip;
  float *chunk_ss, *scale;
  int by_norm;                      // 0: tf.clip_by_average_norm (||g|| / n against clip), 1: tf.clip_by_norm (||g|| against clip)
};
int clip_chunks(int64_t max_count);
// RMSProp over the arena, its gradient clipped first unless c is null.  *kernels: the launches it enqueued (clipped: chunk sums
// of squares, per-tensor scale, update).
int launch_rmsprop(const RmsPropArgs& a, const ClipArgs* c, cudaStream_t stream, int* kernels);
// Config.DUAL_RMSPROP: two optimizers with their own slots, both steps taken from the weights the call started with:
// w <- w - step(g, ms, mom) - step(g2, ms2, mom2).  Elements inside [skip_lo[i], skip_hi[i]) are left alone by optimizer i / 2
// (i = 0, 1: first optimizer; 2, 3: second): the variables its cost does not reach.
struct RmsPropDualArgs {
  RmsPropArgs a;                   // w, g, ms, mom + scalars (+ bf16 shadow range)
  const float* g2;
  float *ms2, *mom2;
  int64_t skip_lo[4], skip_hi[4];
  const float *scale1, *scale2;    // set by launch_rmsprop_dual when it clips
};
// DUAL_RMSPROP + USE_GRAD_CLIP (NetworkVP_discrate.py:107-117) unless c1 is null: c1 describes g (d.a.g), c2 describes g2, both
// by_norm.  *kernels: 1, or 5 when clipped.
int launch_rmsprop_dual(RmsPropDualArgs d, const ClipArgs* c1, const ClipArgs* c2, cudaStream_t stream, int* kernels);
// grad_reduce + RMSProp in one launch (single-GPU step; r.out must be a.g, r.out_floats the small-tensor prefix)
int launch_rmsprop_reduce(const RmsPropArgs& a, const GradReduceArgs& r, cudaStream_t stream);
// data-parallel exchange over peer memory (dp_exchange.cuh), in two instalments.
constexpr int DP_MAX_WORLD = 8;
struct DpBigArgs;
// dense1/w on a side stream, resident next to the conv kernels (elementwise.cu dp_big_side_kernel): rank r owns slice r, sums that
// slice of every rank's gradient (fixed rank order), applies RMSProp and stores the bf16 shadow into every rank's slab
int launch_dp_big_side(const DpBigArgs& big, int num_sms, cudaStream_t side_stream);
// the small tensors behind the conv backward: slab reduction, LL push into every rank's receive buffer, identical RMSProp on
// every rank.  recv_offset: byte offset in the slab of the receive buffers [2][DP_MAX_WORLD][small prefix * 8 B].
struct RmsPropDpArgs {
  RmsPropArgs base;                 // this rank's own arenas
  uint8_t* peer[DP_MAX_WORLD];      // slab bases: [params | grads | ms | mom | shadow | LL receive buffers | comm]
  int rank, world;
  uint64_t step;                    // 1, 2, ... : the flag value of this step
  int64_t arena_bytes, comm_offset;
  GradReduceArgs red;               // this rank's gradient-partial slabs
};
int launch_dp_small(const RmsPropDpArgs& a, int64_t recv_offset, cudaStream_t stream);
int configure_dp();     // load the exchange kernels now (not lazily at their first launch)
int launch_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, cudaStream_t stream);
int launch_returns(const double* rewards, const int64_t* seg_offsets, int n_segments, const double* terminal,
                   double discount, int flags, double rmin, double rmax, double* out, cudaStream_t stream);
int launch_select_actions(const float* p, const double* u, int batch, int num_actions, int32_t* action,
                          cudaStream_t stream);

// histo.cu -- TF's histogram::Histogram of each source (the TensorBoard summaries of Network.log): output row s of `out` is
// {min, max, num, sum, sum_squares, 1551 bucket counts} in fp64, bad[s] != 0 if source s holds a NaN / Inf.  histo_zero clears
// out / bad, launch_histo counts (integer atomics into the count slots) and leaves fp64 partial moments in part[block][4],
// launch_histo_merge sums them in block order: bit-identical output from call to call.
constexpr int HISTO_MAX_SRC = 23;     // conv net 15; MLP nets: variables + live hidden layers + 2, at most 23
struct HistoSrc {
  const void* p;                  // 16-byte aligned
  long long n;                    // values in storage (Blk2: frames x B2_BYTES / 2, borders included)
  int bf16;                       // 0 fp32, 1 bf16
  int blk2;                       // bf16 n1 in the Blk2 layout (common.cuh): only the live 441 x 16 values of a frame count
};
struct HistoArgs {
  HistoSrc src[HISTO_MAX_SRC];
  int blk_end[HISTO_MAX_SRC];     // histo_plan: prefix sums of the blocks per source
  int n_src;
  double* out;                    // [n_src][5 + 1551]
  int32_t* bad;                   // [n_src]
  double* part;                   // [histo_blocks()][4] scratch
};
int histo_plan(HistoArgs& a);     // validates the sources and fills blk_end
int histo_blocks(const HistoArgs& a);
int histo_zero(const HistoArgs& a, cudaStream_t stream);
int launch_histo(const HistoArgs& a, cudaStream_t stream);
int launch_histo_merge(const HistoArgs& a, cudaStream_t stream);

}  // namespace ga3c
