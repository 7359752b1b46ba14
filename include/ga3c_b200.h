/* ga3c_b200.h -- C ABI of the B200-native GA3C predict/train hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Every entry point replaces one
 * `tf.Session.run` call site of the reference `Network` class (paths into /root/reference/ga3c):
 *
 *   ga3c_create / ga3c_destroy      NetworkVP.py:37-64    (graph + session + variable init)
 *   ga3c_param_*                    NetworkVP.py:284-288  (get_variables_names / get_variable_value)
 *   ga3c_predict                    NetworkVP.py:248-252  (predict_p_and_v: sess.run([softmax_p, logits_v]))
 *   ga3c_forward_backward           NetworkVP_discrate.py:60-85,:100 + the autodiff half of opt.minimize (:130)
 *   ga3c_apply_rmsprop              NetworkVP_discrate.py:101-105 (ApplyRMSProp on every variable) + global_step++
 *   ga3c_train_step                 NetworkVP.py:254-257  (train: sess.run(train_op))
 *   ga3c_returns                    ProcessAgent.py:70-84 (_accumulate_rewards), on device, fp64, bit-exact
 *   ga3c_select_actions             ProcessAgent.py:110-115 (np.random.choice given its uniform draw), bit-exact
 *
 * Conventions
 *   - plain C, no torch / C++ types.  Every function returns 0 on success, non-zero on error;
 *     ga3c_last_error() returns a thread-local message for the last failure on this thread.
 *   - pointers named *_dev are DEVICE pointers owned by the caller; `stream` is a cudaStream_t
 *     passed as void* (NULL = legacy default stream).  Calls are asynchronous on `stream`.
 *   - the handle owns the parameter / gradient / RMSProp-slot arenas and the activation workspace.
 *   - there is no CPU fallback: ga3c_create fails if no sm_100 device is present.
 *   - a handle is NOT re-entrant: the caller serialises predict/train on one handle (the Python
 *     `Network` holds a lock; the reference gives no ordering guarantee between its predictor and
 *     trainer threads, Server.py:123-134, so serialising them changes nothing observable).
 */
#ifndef GA3C_B200_H
#define GA3C_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ga3c_net ga3c_net;

/* Config.py knobs the path reads (SURVEY.md section 5). */
typedef struct ga3c_config {
  int32_t device;            /* CUDA ordinal; Config.DEVICE 'gpu:N' -> N                      */
  int32_t num_actions;       /* A, 1..18                                                      */
  int32_t max_batch;         /* rows of activation workspace (predict and train)              */
  float   rmsprop_decay;     /* Config.RMSPROP_DECAY    (0.99)                                */
  float   rmsprop_momentum;  /* Config.RMSPROP_MOMENTUM (0.0)                                 */
  float   rmsprop_epsilon;   /* Config.RMSPROP_EPSILON  (0.1)  -- inside the sqrt             */
  float   log_epsilon;       /* Config.LOG_EPSILON      (1e-6)                                */
  float   min_policy;        /* Config.MIN_POLICY       (0.0)                                 */
  int32_t use_log_softmax;   /* Config.USE_LOG_SOFTMAX  (False): NetworkVP_discrate.py:64-71  */
  int32_t use_grad_clip;     /* Config.USE_GRAD_CLIP    (False): tf.clip_by_average_norm per variable before RMSProp
                              * (NetworkVP_discrate.py:118-121).  As in that file, global_step is then NOT advanced
                              * (its apply_gradients call has no global_step argument).  Not available with the
                              * peer-memory exchange (ga3c_dp_attach): the norm needs the whole reduced gradient.   */
  float   grad_clip_norm;    /* Config.GRAD_CLIP_NORM   (40.0)                                */
  int32_t dual_rmsprop;      /* Config.DUAL_RMSPROP     (False): cost_p and cost_v minimised by two RMSProp optimizers with
                              * their own slots (NetworkVP_discrate.py:87-98, :124-128).  TensorFlow runs the two train ops in
                              * no defined order; here both gradients are taken at the weights the call started with and
                              * both steps are subtracted; global_step advances by 2.  With USE_GRAD_CLIP each optimizer's
                              * gradients go through tf.clip_by_norm per variable and global_step stays put
                              * (NetworkVP_discrate.py:107-117).  Data parallel: dp_mode 'nccl' only (two allreduces).       */
  /* Input geometry (ABI 10), appended so that a caller that zero-fills the struct keeps 84 x 84 x 4.  0 = the default.
   * Frames are NHWC [B, H, W, C] flattened, H * W * C floats (or bytes, _u8) per row.  84 x 84 x 4 runs the specialised
   * trunk; every other geometry a generic one (im2col + tcgen05 GEMMs, same layers, same bf16 rounding points), whose
   * activations lie row-major in the workspace (ga3c_workspace_ptr).  Derived sizes (TF SAME): H1 = ceil(H/4), W1 = ceil(W/4),
   * H2 = ceil(H1/2), W2 = ceil(W1/2); dense1/w is [K = H2 * W2 * 32, 256] and conv11/w [8, 8, C, 16] (ga3c_param_info).
   * Generic handles cannot attach the peer-memory exchange (ga3c_dp_attach fails; dp_mode 'nccl' works). */
  int32_t image_height;      /* Config.IMAGE_HEIGHT     (84): 1..256                          */
  int32_t image_width;       /* Config.IMAGE_WIDTH      (84): 1..256                          */
  int32_t stacked_frames;    /* Config.STACKED_FRAMES   (4):  1..8                            */
} ga3c_config;

const char* ga3c_last_error(void);
/* 10: ga3c_config gained image_height, image_width, stacked_frames (input geometry) */
int ga3c_abi_version(void);

int ga3c_create(const ga3c_config* cfg, ga3c_net** out);
int ga3c_destroy(ga3c_net* net);
/* grow the activation workspace to hold `max_batch` rows (no-op if already large enough).  The
 * reference's train batch is unbounded (ThreadTrainer.py:48-59 concatenates agent batches). */
int ga3c_reserve(ga3c_net* net, int32_t max_batch);

/* ---- parameter arena -------------------------------------------------------------------
 * One flat fp32 arena holds all 10 variables; grads / ms / mom arenas have the same layout.
 * Tensors are listed in TF creation order (conv11/w:0, conv11/b:0, conv12/w:0, ... logits_p/b:0);
 * offsets are in floats and are NOT in that order (small tensors are packed first). */
int     ga3c_param_count(const ga3c_net* net);
int     ga3c_param_info(const ga3c_net* net, int index, const char** name, int64_t* offset,
                        int32_t* ndim, int64_t shape[4]);
int64_t ga3c_arena_floats(const ga3c_net* net);
/* device base pointers of the four arenas (any may be NULL to skip) */
int ga3c_arena_ptrs(ga3c_net* net, float** params_dev, float** grads_dev, float** ms_dev, float** mom_dev);
/* one arena by id (the ids of ga3c_arena_upload below) */
int ga3c_arena_ptr(ga3c_net* net, int which, float** ptr_dev);
/* host <-> device copies of a whole arena; which: 0 params, 1 grads, 2 ms, 3 mom; with dual_rmsprop also 4 / 5 / 6: gradient,
 * ms, mom of the second optimizer (the one minimising cost_v; 1 / 2 / 3 then belong to cost_p).  Synchronous.
 * Writing params also refreshes the bf16 shadow of dense1/w. */
int ga3c_arena_upload(ga3c_net* net, int which, const float* host, int64_t n_floats);
int ga3c_arena_download(ga3c_net* net, int which, float* host, int64_t n_floats);
int64_t ga3c_global_step(const ga3c_net* net);
int ga3c_set_global_step(ga3c_net* net, int64_t step);

/* ---- hot path -----------------------------------------------------------------------------
 * x_dev   fp32 [B, 28224]  NHWC frames flattened (84*84*4), exactly what ThreadPredictor stacks
 * p_dev   fp32 [B, A]      softmax policy (fp32 so np.random.choice accepts it, SURVEY A.6)
 * v_dev   fp32 [B]
 * yr_dev  fp32 [B]         discounted returns; a_dev fp32 [B, A] one-hot actions
 * loss_dev fp32 [4] or NULL: {cost_p_1_agg, cost_p_2_agg, cost_v, 0} (sums over the batch);
 *          cost_p = -(loss[0]+loss[1]), cost_all = cost_p + loss[2]  (NetworkVP_discrate.py:83-85,:100)
 */
int ga3c_predict(ga3c_net* net, const float* x_dev, int32_t batch, float* p_dev, float* v_dev, void* stream);
int ga3c_forward_backward(ga3c_net* net, const float* x_dev, const float* yr_dev, const float* a_dev,
                          int32_t batch, float beta, float* loss_dev, void* stream);
/* ga3c_forward_backward in two halves, so that a data-parallel host can overlap the gradient allreduce with
 * the conv backward: after ga3c_fb_head (in stream order) the gradients of dense1/w (98.8 % of the arena, the
 * last tensor: floats [offset(dense1/w:0), arena_floats)), dense1/b and both heads are final; ga3c_fb_tail
 * (same batch, same x) then completes the conv11 and conv12 gradients. */
int ga3c_fb_head(ga3c_net* net, const float* x_dev, const float* yr_dev, const float* a_dev, int32_t batch, float beta,
                 float* loss_dev, void* stream);
int ga3c_fb_tail(ga3c_net* net, const float* x_dev, int32_t batch, void* stream);
int ga3c_apply_rmsprop(ga3c_net* net, float learning_rate, void* stream);
int ga3c_train_step(ga3c_net* net, const float* x_dev, const float* yr_dev, const float* a_dev,
                    int32_t batch, float learning_rate, float beta, float* loss_dev, void* stream);
/* Config.DUAL_RMSPROP in two halves (handles created with dual_rmsprop): both gradients (cost_p -> arena 1, cost_v -> arena 4),
 * then the update with both optimizers' steps.  ga3c_train_step is the two back to back; a data-parallel host allreduces
 * arenas 1 and 4 in between (dp_mode 'nccl'). */
int ga3c_dual_forward_backward(ga3c_net* net, const float* x_dev, const float* yr_dev, const float* a_dev, int32_t batch,
                               float beta, float* loss_dev, void* stream);
int ga3c_dual_apply(ga3c_net* net, float learning_rate, void* stream);

/* ---- uint8 frame ingestion (SURVEY 8f F2) ---------------------------------------------------------
 * Same calls with x8_dev = uint8 [B, 28224]: the raw 0..255 pixels BEFORE the reference's
 * `image.astype(np.float32) / 128.0 - 1.0` (Environment.py:60).  The kernels apply x = k/128 - 1 while converting to
 * bf16 (exact), so every output is bit-identical to the fp32 call on the normalised frames, with 4x fewer host->device
 * and HBM input bytes.  An extension of the reference contract (its queues carry float32 states): see INTEGRATION.md. */
int ga3c_predict_u8(ga3c_net* net, const uint8_t* x8_dev, int32_t batch, float* p_dev, float* v_dev, void* stream);
int ga3c_forward_backward_u8(ga3c_net* net, const uint8_t* x8_dev, const float* yr_dev, const float* a_dev,
                             int32_t batch, float beta, float* loss_dev, void* stream);
int ga3c_fb_head_u8(ga3c_net* net, const uint8_t* x8_dev, const float* yr_dev, const float* a_dev, int32_t batch, float beta,
                    float* loss_dev, void* stream);
int ga3c_fb_tail_u8(ga3c_net* net, const uint8_t* x8_dev, int32_t batch, void* stream);
int ga3c_train_step_u8(ga3c_net* net, const uint8_t* x8_dev, const float* yr_dev, const float* a_dev,
                       int32_t batch, float learning_rate, float beta, float* loss_dev, void* stream);
int ga3c_dual_forward_backward_u8(ga3c_net* net, const uint8_t* x8_dev, const float* yr_dev, const float* a_dev, int32_t batch,
                                  float beta, float* loss_dev, void* stream);

/* ---- data parallel over peer memory (one process per GPU, one node, <= 8 ranks) ---------------------
 * Every rank exports a CUDA IPC handle of its state slab (ga3c_dp_export), the host exchanges the handles
 * (torch.distributed all_gather in ga3c_b200.Network) and attaches them in rank order (ga3c_dp_attach).  From
 * then on ga3c_train_step exchanges the gradients and updates the weights inside the step, in two instalments
 * (dp_exchange.cuh).  dense1/w: as soon as its gradient is final, a kernel on a side stream of the handle sums this
 * rank's slice of every rank's gradient over NVLink, applies RMSProp to the slice and stores its bf16 copy into every
 * rank's slab, while the conv backward runs; the fp32 weights and slots of a slice stay on the rank that owns it
 * (ga3c_arena_download collects them).  The other variables: after the conv backward every rank pushes its gradient
 * to every rank, and every rank applies the identical update to its own copy.  Sums in fixed rank order, so the
 * replicas stay bit-identical; the next forward waits until every rank's dense1/w slice has landed.  SUM, no averaging:
 * every loss term is a reduce_sum (NetworkVP_discrate.py:61,:83-85).  ga3c_apply_rmsprop refuses an attached handle
 * (use ga3c_train_step), and ga3c_train_step refuses one created with use_grad_clip or dual_rmsprop.  All ranks must call
 * train the same number
 * of times; a rank with nothing to train on calls ga3c_train_step with batch = 0 (buffers may be NULL): it contributes a
 * zero gradient and applies the same update as everybody else (the host-side lock step that makes the reference's
 * asynchronous trainer loop, ThreadTrainer.py:42-62, fit this rule is ga3c_b200.threads.LockstepTrainer). */
int ga3c_dp_handle_bytes(void);
int ga3c_dp_export(ga3c_net* net, void* handle_out);
int ga3c_dp_attach(ga3c_net* net, int32_t rank, int32_t world, const void* handles);
int ga3c_dp_detach(ga3c_net* net);
/* ranks living in one process (one host process driving several GPUs, or tests with two handles on one GPU): peers[r] is
 * rank r's handle, peers[rank] == net; the slabs are addressed directly, no IPC handles. */
int ga3c_dp_attach_local(ga3c_net* net, int32_t rank, int32_t world, ga3c_net* const* peers);
/* Every cross-rank wait inside the exchange kernels is bounded (some tens of seconds).  *error_out != 0 (a mask of the wait sites, dp_exchange.cuh) if one of them gave up since
 * the last attach: a rank died or the ranks' train calls fell out of step; the weights can no longer be trusted.  Synchronises. */
int ga3c_dp_error(ga3c_net* net, int32_t* error_out);

/* ---- returns (ProcessAgent.py:70-84) --------------------------------------------------------
 * Segments (one per agent rollout) are packed back to back; seg_offsets_dev has n_segments+1
 * entries.  fp64 throughout, same operation order as the reference loop => bit-exact.
 * flags: bit0 DISCOUNTING, bit1 USE_INTERMEDIATE_REWARD, bit2 REWARD_CLIPPING  (Config.py:73-83)
 *        bit3 NSTEP: upstream semantics R_t = clip(r_t) + gamma*R_{t+1} seeded with terminal[s]
 *             (the commented ProcessAgent.py:83,:146); out[n-1] is set to the seed.              */
#define GA3C_RET_DISCOUNTING 1
#define GA3C_RET_INTERMEDIATE 2
#define GA3C_RET_CLIPPING 4
#define GA3C_RET_NSTEP 8
int ga3c_returns(const double* rewards_dev, const int64_t* seg_offsets_dev, int32_t n_segments,
                 const double* terminal_dev, double discount, int32_t flags, double reward_min,
                 double reward_max, double* out_dev, void* stream);

/* ---- sampling (ProcessAgent.py:110-115) ------------------------------------------------------
 * action[i] = searchsorted(cumsum(float64(p[i])) / sum, u[i], side='right'): np.random.choice given
 * the uniform it drew.  Bit-exact.  */
int ga3c_select_actions(const float* p_dev, const double* u_dev, int32_t batch, int32_t num_actions,
                        int32_t* action_dev, void* stream);

/* ---- low-dimensional MLP networks (BASELINE config 4; SURVEY 8a rows A6 / A7) --------------------------
 * The fork's two non-conv `Network` plugins behind the same call shapes, fp32 throughout:
 *   GA3C_MLP_FORK_VP   NetworkVP.py:79-105 (+ :175-210): x[S] -> dense 4 -> 256 -> 256 (all linear) -> 100 (sigmoid) ->
 *                      'dense1' 64 (sigmoid); v = dense 1; p = atan2(sigmoid(out_y) - 0.5, sigmoid(out_x) - 0.5) / pi;
 *                      softmax_p = log_softmax_p = p (:95-96); cost_p_1 = sum_a(p a) (R - sg(v)); cost_p_2 = -beta sum p^2.
 *                      `a` is whatever ProcessAgent hands over ([B, A] float32; the continuous action for Pendulum).
 *   GA3C_MLP_DISCRATE  NetworkVP_discrate.py:52-85 AS WRITTEN: every Config.DENSE_LAYERS entry is built from x (:55), so
 *                      only the LAST one (sigmoid, the default func of dense_layer, NetworkVP.py:194) feeds the heads; the
 *                      earlier ones are variables without a gradient: listed by ga3c_mlp_param_info with live = 0, never
 *                      touched by the optimizer (tf's minimize skips variables whose gradient is None).  Heads / loss as
 *                      the conv net: softmax + MIN_POLICY mix, log(max(., eps)) terms (:66-85).
 * All variables start U(-0.3, 0.3) in the reference (NetworkVP.py:199-202): the host uploads them (ga3c_mlp_arena_upload).
 * ga3c_mlp_predict       replaces sess.run([softmax_p, logits_v])  (NetworkVP.py:248-252)
 * ga3c_mlp_train_step    replaces sess.run(train_op)               (NetworkVP.py:254-257)
 * loss_dev as for the conv net: {cost_p_1_agg, cost_p_2_agg, cost_v, 0}.                                             */
typedef struct ga3c_mlp ga3c_mlp;
#define GA3C_MLP_FORK_VP 0
#define GA3C_MLP_DISCRATE 1
typedef struct ga3c_mlp_config {
  int32_t device;
  int32_t kind;              /* GA3C_MLP_*                                                             */
  int32_t state_dim;         /* S, 1..256                                                              */
  int32_t num_actions;       /* A, 1..18                                                               */
  int32_t max_batch;
  int32_t n_dense;           /* DISCRATE: len(Config.DENSE_LAYERS), 1..8; FORK_VP: ignored             */
  int32_t dense_width[8];    /* DISCRATE: Config.DENSE_LAYERS (each 1..256, the last <= 128)           */
  float   rmsprop_decay, rmsprop_momentum, rmsprop_epsilon, log_epsilon, min_policy;
  int32_t use_log_softmax;   /* DISCRATE only (the fork's NetworkVP has no softmax at all)                          */
  int32_t use_grad_clip;     /* Config.USE_GRAD_CLIP: FORK_VP advances global_step (NetworkVP.py:141), DISCRATE does
                              * not (NetworkVP_discrate.py:121); DISCRATE with gradient-less variables is refused, as
                              * the reference graph cannot be built (clip_by_average_norm(None))                    */
  float   grad_clip_norm;
  int32_t dual_rmsprop;      /* Config.DUAL_RMSPROP, as for the conv net                                            */
} ga3c_mlp_config;
int ga3c_mlp_create(const ga3c_mlp_config* cfg, ga3c_mlp** out);
int ga3c_mlp_destroy(ga3c_mlp* net);
int ga3c_mlp_reserve(ga3c_mlp* net, int32_t max_batch);
/* variables in TF creation order; live = 0 for the gradient-less variables of DISCRATE */
int     ga3c_mlp_param_count(const ga3c_mlp* net);
int     ga3c_mlp_param_info(const ga3c_mlp* net, int index, const char** name, int64_t* offset, int32_t* ndim,
                            int64_t shape[4], int32_t* live);
int64_t ga3c_mlp_arena_floats(const ga3c_mlp* net);
int ga3c_mlp_arena_upload(ga3c_mlp* net, int which, const float* host, int64_t n_floats);   /* which: 0 params, 1 grads, 2 ms, 3 mom */
int ga3c_mlp_arena_download(ga3c_mlp* net, int which, float* host, int64_t n_floats);
int64_t ga3c_mlp_global_step(const ga3c_mlp* net);
int ga3c_mlp_set_global_step(ga3c_mlp* net, int64_t step);
int ga3c_mlp_predict(ga3c_mlp* net, const float* x_dev, int32_t batch, float* p_dev, float* v_dev, void* stream);
int ga3c_mlp_forward_backward(ga3c_mlp* net, const float* x_dev, const float* yr_dev, const float* a_dev, int32_t batch,
                              float beta, float* loss_dev, void* stream);
int ga3c_mlp_apply_rmsprop(ga3c_mlp* net, float learning_rate, void* stream);
int ga3c_mlp_train_step(ga3c_mlp* net, const float* x_dev, const float* yr_dev, const float* a_dev, int32_t batch,
                        float learning_rate, float beta, float* loss_dev, void* stream);
int64_t ga3c_mlp_launch_count(const ga3c_mlp* net);
/* parity tests: device pointer to a training-workspace matrix of the last forward/backward, fp32 row-major [batch][*width].
 * which: 0 output of live hidden layer `layer`, 1 gradient w.r.t. that layer's pre-activation. */
int ga3c_mlp_workspace_ptr(ga3c_mlp* net, int32_t which, int32_t layer, void** ptr, int32_t* width);
/* kernel-level test entry for the 3xTF32 tensor-core GEMMs behind the wide MLP layers (device pointers, fp32 row-major;
 * k, n multiples of 4 up to 256):
 *   mode 0  out [m, n] = act(a [m, k] x b [k, n] + aux [n])                    act: 0 linear, 1 sigmoid
 *   mode 1  out [m, k] = (a [m, n] x b [k, n]^T) * act'(aux [m, k])
 *   mode 2  out [splits][k, n] = a [m, k]^T x b [m, n] over each batch split of rows_per_split (multiple of 32) rows */
int ga3c_debug_tf32x3_gemm(int32_t mode, const float* a, const float* b, const float* aux, float* out, int32_t m, int32_t k,
                           int32_t n, int32_t act, int32_t splits, int32_t rows_per_split, void* stream);
/* per-kernel event timing, as ga3c_timing_* (kernel ids are shared: ga3c_kernel_name) */
int ga3c_mlp_timing_enable(ga3c_mlp* net, int32_t max_records);
int ga3c_mlp_timing_collect(ga3c_mlp* net, double* total_ms, int64_t* counts, int32_t n_kernels);
/* TensorBoard histograms of an MLP handle (Network.log; the histogram itself is described with ga3c_histograms below).
 * ga3c_mlp_histogram_count: the number of sources, variables + live hidden layers + 2 (at most 23: fork NetworkVP 16 + 5 + 2,
 * DISCRATE with 8 DENSE_LAYERS 20 + 1 + 2).  ga3c_mlp_histograms sources, in this order: every variable in ga3c_mlp_param_info
 * order (the gradient-less DISCRATE ones included), the output of every live hidden layer in forward order as the last forward
 * on this handle left it (ga3c_mlp_forward_backward / ga3c_mlp_train_step, or a ga3c_mlp_predict of a tensor-core batch,
 * which writes the same workspace; `batch` must be that forward's batch), then v_dev [B] and p_dev [B, A] (fp32, 16-byte
 * aligned: what ga3c_mlp_predict wrote for the same rows).  out_dev: ga3c_mlp_histogram_count(net) x (5 + GA3C_HISTO_BUCKETS)
 * doubles, bad_dev: as many int32.  Launches two kernels, both under kernel id "histograms". */
int ga3c_mlp_histogram_count(const ga3c_mlp* net);
int ga3c_mlp_histograms(ga3c_mlp* net, int32_t batch, const float* p_dev, const float* v_dev, double* out_dev,
                        int32_t* bad_dev, void* stream);

/* ---- serialisation ---------------------------------------------------------------------------------
 * A handle is not re-entrant (one activation workspace).  Whoever drives it from several threads -- the reference calls
 * predict_p_and_v and train from PREDICTORS + TRAINERS threads without locks (Server.py:123-134) -- takes this mutex around
 * [enqueue ... stream synchronise]: the Python Network does, and so does the native batcher below. */
int ga3c_lock(ga3c_net* net);
int ga3c_unlock(ga3c_net* net);

/* ---- native predictor batcher (SURVEY 8f F1) ----------------------------------------------------------
 * ThreadPredictor.run (ThreadPredictor.py:45-66) as a thread inside the library, over the shared-memory slab of
 * ga3c_b200.transport.SlabPredictionQueue: wait for a request (work_sem), take every pending row (at most max_batch, round
 * robin), copy those rows from the page-locked, device-mapped state slab into the batch with ONE kernel (no host gather, no
 * staging copy), ga3c_predict[_u8], write (p, v) into the agents' reply rows and post their semaphores -- the `wait_q.put` of
 * ThreadPredictor.py:63.  The interpreter is never entered.  All pointers are HOST pointers into memory shared with the
 * agent processes; semaphores are POSIX sem_t* (what multiprocessing.Semaphore wraps: SemLock.handle).
 * state_bytes: bytes per state row (28224 for uint8 frames, 112896 for float32), a multiple of 16. */
typedef struct ga3c_batcher ga3c_batcher;
typedef struct ga3c_batcher_config {
  int32_t device, num_agents, state_bytes, x_u8, max_batch, num_actions;
  void*    states;      /* [num_agents][state_bytes]; registered with cudaHostRegister for the batcher's lifetime */
  uint8_t* pending;     /* [num_agents]: 1 = a request is posted in that agent's row                              */
  float*   reply_p;     /* [num_agents][num_actions]                                                              */
  float*   reply_v;     /* [num_agents]                                                                           */
  void*    work_sem;    /* sem_t*: one permit per posted request (a wake-up hint; the pending bytes are the truth) */
  void**   wake_sems;   /* sem_t* [num_agents]: posted when the agent's reply row is filled                       */
} ga3c_batcher_config;
int ga3c_batcher_create(ga3c_net* net, const ga3c_batcher_config* cfg, ga3c_batcher** out);
int ga3c_batcher_start(ga3c_batcher* b);
int ga3c_batcher_stop(ga3c_batcher* b);
/* batches / rows served since creation; *error != 0 (and a non-zero return with ga3c_last_error) if the thread gave up */
int ga3c_batcher_stats(ga3c_batcher* b, int64_t* batches, int64_t* rows, int32_t* error);
int ga3c_batcher_destroy(ga3c_batcher* b);

/* ---- host staging of pageable caller arrays ------------------------------------------------------------
 * ThreadTrainer hands Network.train ordinary numpy arrays (np.concatenate output, ThreadTrainer.py:54-58); a cudaMemcpyAsync
 * from pageable memory runs at a fraction of the PCIe rate.  ga3c_stage_h2d copies `bytes` from `src` (any host memory) into the
 * page-locked `staging` buffer with `threads` worker threads of the library (non-temporal stores, 512 KB pieces claimed in
 * address order; threads <= 1: the calling thread alone) and enqueues cudaMemcpyAsync(dst_dev + off, staging + off) on `stream`
 * for every chunk of `chunk_bytes` (0: 8 MB) as soon as the chunk is in place, so the DMA of chunk k runs under the host copy of
 * chunk k + 1.  Returns once the host copy is complete and every DMA is enqueued; `staging` must stay untouched until the
 * stream has passed them.  dst_dev == NULL: host copy only (no CUDA call is made).  One job at a time per process: concurrent
 * callers queue.  Needs no handle. */
int ga3c_stage_h2d(void* dst_dev, void* staging, const void* src, int64_t bytes, int64_t chunk_bytes, int32_t threads,
                   void* stream);

/* ---- introspection for tests / profiling ---------------------------------------------------- */
/* device pointers to the activation workspace of the last call (bf16 stored as uint16):
 * which: 0 n1 bf16 in the Blk2 operand layout [B][8 planes][160 rows][8] (channels 8h.. of pixel (y, x) in plane
 *          (((y+1)&1)*2 + ((x+1)&1))*2 + h, row ((y+1)>>1)*13 + ((x+1)>>1); zero borders), 1 n2 [B,3872] bf16, 2 d1 [B,256] fp32,
 *        3 dd1 [B,256] bf16, 4 dn2 bf16 in the G operand layout [B][4 planes][172 rows][8] (channels 8j.. of position (oy, ox) in
 *          plane j, row (oy+1)*13 + ox+1; zero borders), 5 dn1 [B,441,16] bf16 (only with ga3c_keep_dn1), 7 xblk: the bf16
 *          block matrix of the frames [B][4 quarters][8 planes][128 rows][8] that the conv backward reads instead of x, 6 the bf16 shadow of dense1/w [3872,256] (what the dense1 GEMMs read; in a
 *        data-parallel job the copy every rank holds, so comparing it across ranks checks the exchange).
 * A handle of any other geometry than 84x84x4 (the generic trunk) keeps its activations row-major: 0 n1 [B,H1,W1,16] bf16,
 * 1 n2 [B,K] bf16, 4 dn2 [B,K] bf16, 5 dn1 [B,H1,W1,16] bf16 (always stored), 7 X1 [B*H1*W1][64C + 8] bf16, the im2col
 * matrix of the frames (columns (kh, kw, c), then a column of ones and 7 zero columns), which the backward reads instead of x;
 * 2, 3 and 6 as above with K = H2*W2*32 for 3872. */
int ga3c_workspace_ptr(ga3c_net* net, int which, void** ptr_dev, int64_t* bytes);
/* dn1 (the conv12 data gradient) normally never leaves the SM: the fused conv backward kernel consumes it from shared
 * memory.  on != 0 makes that kernel also store it to the workspace (id 5 above) so that tests can compare it. */
int ga3c_keep_dn1(ga3c_net* net, int32_t on);
/* number of kernels this library has launched on this handle since creation */
int64_t ga3c_launch_count(const ga3c_net* net);


/* ---- TensorBoard histograms (NetworkVP.py:152-173, written by Network.log every TENSORBOARD_UPDATE_FREQUENCY steps) ----
 * TensorFlow's histogram::Histogram of each source, computed on the device: {min, max, num, sum, sum_squares} in fp64 and the
 * counts of its 1551 default buckets (bucket i holds limit[i-1] <= x < limit[i]; limits: +-1e-12 * 1.1^k up to 1e20, +-DBL_MAX
 * and 0.0).  Deterministic: the same inputs give bit-identical output.  Non-finite values are left out of the statistics and
 * flagged (TF's HistogramSummary refuses them).  The MLP networks' entry is ga3c_mlp_histograms (above).
 * ga3c_histograms sources, in this order: the 10 variables (TF creation order), then n1, n2, d1 of the last
 * ga3c_forward_backward[_u8] on this handle (`batch` must be its batch; n1 and n2 as stored, bf16), then v_dev [B] and
 * p_dev [B, A] (fp32, 16-byte aligned: what ga3c_predict wrote for the same frames).  Not available once ga3c_dp_attach* has
 * run: dense1/w slices then live on their owners.  Launches two kernels, both under kernel id "histograms".
 * out_dev: GA3C_HISTO_SOURCES x (5 + GA3C_HISTO_BUCKETS) doubles {min, max, num, sum, sum_squares, counts...}
 * bad_dev: GA3C_HISTO_SOURCES int32, non-zero if that source holds a NaN / Inf */
#define GA3C_HISTO_BUCKETS 1551
#define GA3C_HISTO_SOURCES 15
int ga3c_histograms(ga3c_net* net, int32_t batch, const float* p_dev, const float* v_dev, double* out_dev, int32_t* bad_dev,
                    void* stream);
/* kernel-level test entry: one flat, 16-byte aligned array of n >= 1 fp32 (dtype 0) or bf16 (dtype 1) values; out_dev holds
 * 5 + GA3C_HISTO_BUCKETS doubles, bad_dev one int32 */
int ga3c_debug_histogram(const void* x_dev, int32_t dtype, int64_t n, double* out_dev, int32_t* bad_dev, void* stream);

/* ---- per-kernel device timing (bench.py's roofline leg)-------------------------------------
 * ga3c_timing_enable(net, R) pre-creates events for R kernel records (R = 0 switches timing off).
 * While enabled, every kernel the hot path launches is bracketed by cudaEventRecord on the launch
 * stream -- no synchronisation is added.  ga3c_timing_collect synchronises the device, sums the
 * durations per kernel id (ga3c_kernel_name(id), id < ga3c_kernel_count()) and rewinds the record
 * cursor; launches beyond R records are simply not timed. */
int         ga3c_kernel_count(void);
const char* ga3c_kernel_name(int kernel_id);
int ga3c_timing_enable(ga3c_net* net, int32_t max_records);
int ga3c_timing_collect(ga3c_net* net, double* total_ms, int64_t* counts, int32_t n_kernels);

/* ---- step timeline trace (profiles/: where the pipelined step spends its time) ----------------
 * Between ga3c_trace_begin and ga3c_trace_end thread 0 of every CTA of every hot-path kernel stamps
 * %globaltimer (ns) when it is launched (reaches its dependency wait), started (dependency satisfied)
 * and ended.  stamps[k*6 + {0,1}] = first/last CTA launched, {2,3} = first/last started, {4,5} =
 * first/last ended, for kernel id k < ga3c_kernel_count(); kernels that did not run keep
 * {UINT64_MAX, 0}.  The trace is process-wide (one handle at a time).  Unlike the event timing above it
 * does not serialise the programmatic-dependent-launch chain.  ga3c_trace_begin synchronises `stream`;
 * ga3c_trace_end synchronises the device. */
int ga3c_trace_begin(ga3c_net* net, void* stream);
int ga3c_trace_end(ga3c_net* net, uint64_t* stamps, int32_t n_kernels);

/* ---- pipeline event log (debug) ----------------------------------------------------------------
 * CTA 0 of the conv backward kernel appends {globaltimer ns, warp << 32 | event id << 16 | arg} records (two uint64
 * each, at most 16384) between ga3c_evt_begin and ga3c_evt_end; tools/evt_timeline.py prints them per warp role. */
int ga3c_evt_begin(ga3c_net* net);
int ga3c_evt_end(ga3c_net* net, uint64_t* records, int32_t cap, int32_t* count);

#ifdef __cplusplus
}
#endif
#endif /* GA3C_B200_H */
