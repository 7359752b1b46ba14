// Launch interface of the low-dimensional MLP networks (BASELINE config 4; SURVEY 8a rows A6 / A7).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.h"

namespace ga3c {

constexpr int MLP_MAX_LAYERS = 8;     // live hidden layers
constexpr int MLP_MAX_WIDTH = 256;    // of any layer and of the state
constexpr int MLP_MAX_HID = 128;      // width of the last hidden layer (the one the heads read)
constexpr int MLP_MAX_OUT = 1 + 2 * 18;
constexpr int MLP_TM = 64;            // batch rows per tile
constexpr int MLP_MAX_SPLITS = 74;    // batch splits of the weight-gradient pass (partial arenas); 2 x 74 GEMM CTAs = one per SM
constexpr int MLP_ACT_LINEAR = 0, MLP_ACT_SIGMOID = 1;
constexpr int MLP_KIND_FORK_VP = 0, MLP_KIND_DISCRATE = 1;

struct MlpLayerDesc {
  int k, n, act;        // fan-in, width, activation
  int w_off, b_off;     // float offsets into the parameter arena ([k][n] row-major, [n])
};

// everything the kernels need to know about the network; built once by ga3c_mlp_create
struct MlpNet {
  int n_layers;
  MlpLayerDesc L[MLP_MAX_LAYERS];
  int kind, state_dim, num_actions;
  int hid;              // L[n_layers - 1].n
  int n_out;            // columns of the head matrix: v | p (discrate)  or  v | out_x | out_y (fork_vp)
  int n_out_ld;         // row pitch of dlogits in HBM (n_out rounded up to 4)
  int wv_off, bv_off;   // logits_v
  int wp_off, bp_off;   // logits_p   (fork_vp: logits_p/out_x)
  int wy_off, by_off;   // fork_vp: logits_p/out_y
};

struct MlpStepArgs {
  const float* w;                       // parameter arena
  const float* x;                       // [B, state_dim]
  const float *yr, *a;                  // train: [B], [B, A]
  int batch, train;
  LossArgs la;                          // log_softmax, min_policy: DISCRATE only
  float *p_out, *v_out;                 // may be null in train mode
  float* act[MLP_MAX_LAYERS];           // train: layer outputs [B, n_l]
  float* dz[MLP_MAX_LAYERS];            // train: gradients w.r.t. the pre-activations [B, n_l]
  float* dlogits;                       // train: [B, n_out_ld]
  float* loss_part;                     // train: [tiles][4] (cost_p_1, cost_p_2, cost_v, 0) per batch tile (mlp_tile_rows)
  // Tensor-core mode (mlp_tc.cu): the wide layers [tc_lo, tc_hi) run as 3xTF32 GEMM launches between three launches of the fused
  // kernel.  phase 0: everything (tc_lo = tc_hi = 0).  phase 1: x -> layers [0, tc_lo).  phase 2: act[tc_hi - 1] -> layers
  // [tc_hi, n_layers), heads, loss, data gradients down to dz[tc_hi - 1].  phase 3: dz[tc_lo - 1] -> data gradients down to dz[0].
  int phase, tc_lo, tc_hi;
  unsigned wgrad_skip;                  // bit l: mlp_wgrad leaves layer l's dW / db to launch_mlp_tc_wgrad / launch_mlp_skinny_wgrad
};

int configure_mlp();
int mlp_fused_grid(int batch, int num_sms);
int mlp_tile_rows(int batch, int num_sms);       // 64, or 16 for small batches; loss_part has one row per tile
// forward (+ heads, loss, and the whole data-gradient chain when args.train) in one persistent kernel
int launch_mlp_fused(const MlpNet& net, const MlpStepArgs& args, int num_sms, cudaStream_t stream);

// all weight / bias gradients in one grid: split s of tile t writes part[s][arena layout]
int mlp_wgrad_splits(const MlpNet& net, int batch, int num_sms);
// rows_per_split: 0 = derive from splits; tensor-core mode passes its own (a multiple of 32) and skips layers [tc_lo, tc_hi)
int launch_mlp_wgrad(const MlpNet& net, const MlpStepArgs& args, float* part, int64_t part_stride, int splits,
                     cudaStream_t stream, int rows_per_split = 0);
// the head matrices' dW / db by a streaming kernel (n_out <= 4; large batches: bit n_layers of MlpStepArgs::wgrad_skip)
bool mlp_heads_wgrad_ok(const MlpNet& net);
int launch_mlp_heads_wgrad(const MlpNet& net, const MlpStepArgs& args, float* part, int64_t part_stride, int splits,
                           int rows_per_split, cudaStream_t stream);
// g[i] = sum_s part[s][i] (fixed order) over the live prefix; loss[0..3] = sum over tiles (fixed order)
int launch_mlp_reduce(const float* part, int64_t part_stride, int splits, float* g, int live_floats, const float* loss_part,
                      int tiles, float* loss_out, cudaStream_t stream);

int trace_attach_mlp(unsigned long long* buf);

// ---- mlp_tc.cu: wide layers on tcgen05 (kind::tf32, 3xTF32 split: fp32-equivalent) ----------------------------------------------
bool mlp_tc_layer_ok(const MlpLayerDesc& L);
// (k, n multiples of 4; fp32 row-major matrices, W = [k][n])
int launch_mlp_tc_fwd(const float* W, const float* bias, int k, int n, int act, const float* in, float* out, int batch,
                      cudaStream_t stream);                                        // out = act(in x W + bias)
int launch_mlp_tc_dgrad(const float* W, int k, int n, const float* dz, const float* out_prev, int prev_act, float* dz_prev,
                        int batch, cudaStream_t stream);                           // dz_prev = (dz x W^T) * act'(out_prev)
int launch_mlp_tc_wgrad(int k, int n, const float* in, const float* dz, int batch, int splits, int rows_per_split, float* part_w,
                        float* part_b, int64_t part_stride, cudaStream_t stream);  // split s: in^T x dz, colsum(dz) of its rows
// dW = in^T x dz for a layer with fan-in k <= 4 (k = 0: none) and db = colsum(dz), per batch split: streaming kernel, no tiles
int launch_mlp_skinny_wgrad(int k, int n, const float* in, const float* dz, int batch, int splits, int rows_per_split,
                            float* part_w, float* part_b, int64_t part_stride, cudaStream_t stream);
int trace_attach_mlp_tc(unsigned long long* buf);

// ---- mlp_stream.cu: the narrow ends of the fork NetworkVP in tensor-core mode as streaming passes (instead of phases 1 / 2 / 3 of
// the fused tile kernel) ----
bool mlp_stream_ok(const MlpNet& net, int tc_lo, int tc_hi);
int launch_mlp_front_fwd(const MlpNet& net, const MlpStepArgs& args, int num_sms, cudaStream_t stream);   // x -> act[0], act[1]
// act[last] -> v, p (when the pointers are set); args.train: loss_part rows (one per block: mlp_heads_loss_rows), dlogits, dz[last]
int launch_mlp_heads(const MlpNet& net, const MlpStepArgs& args, int num_sms, cudaStream_t stream);
int mlp_heads_loss_rows(int batch, int num_sms);
int launch_mlp_front_bwd(const MlpNet& net, const MlpStepArgs& args, int num_sms, cudaStream_t stream);   // dz[1] -> dz[0]
int trace_attach_mlp_stream(unsigned long long* buf);

}  // namespace ga3c
