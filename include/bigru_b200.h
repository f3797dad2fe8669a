/* bigru_b200.h - C ABI of libbigru_b200.so: the B200 (sm_100a) biGRU hot path.
 *
 * The reference (radoslawkrolikowski/financial-market-data-analysis) has no FFI layer of its
 * own: its hot path is the Python class surface of biGRU_model.py / sql_pytorch_dataloader.py,
 * with the arithmetic inside torch.nn.GRU.  Each entry point below names the reference
 * interface (file:line under /root/reference) whose work it replaces.  The Python mirror in
 * financial_market_data_analysis_b200/ binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *  - plain C types only; every pointer named d_* is a DEVICE pointer owned by the caller; the
 *    library never frees caller memory and keeps no reference to it after the call returns;
 *  - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on that stream and
 *    never synchronise; a plan may be used from one stream at a time;
 *  - every function returns 0 on success, <0 on error (BIGRU_ERR_*); bigru_last_error() returns
 *    a thread-local message.  There is no CPU fallback anywhere: without a CUDA device of
 *    compute capability 10.x every compute call fails with BIGRU_ERR_DEVICE.
 *
 * Flat parameter vector ("params", "grads", Adam moments): float32, order
 *     for l in [0,L): for d in [0,D):  w_ih[3H,I_l]  w_hh[3H,H]  b_ih[3H]  b_hh[3H]
 *     lin_w[C,3H]  lin_b[C]                       with I_0 = F, I_l = D*H, gate rows r|z|n
 * i.e. torch.nn.GRU's own per-layer order (state_dict keys gru.weight_ih_l{l}[_reverse] ...,
 * biGRU_model.py:54-60), so the Python side exposes each block as an ordinary nn.Parameter view.
 */
#ifndef BIGRU_B200_H
#define BIGRU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BIGRU_OK               0
#define BIGRU_ERR_ARG         -1   /* bad shape / null pointer / unsupported combination */
#define BIGRU_ERR_CUDA        -2   /* a CUDA runtime call failed (message has the reason) */
#define BIGRU_ERR_DEVICE      -3   /* no sm_100-class device */
#define BIGRU_ERR_UNSUPPORTED -4   /* shape not supported by the requested precision path */

#define BIGRU_PREC_FP32 0          /* fp32 FFMA path: exact, any shape (<=1e-4 rel on logits) */
#define BIGRU_PREC_BF16 1          /* bf16 operands on tcgen05 tensor cores, fp32 accumulate/state.
                                      hidden_size 128 or 256 with batch % 16 == 0, hidden_size 512 with batch % 32 == 0
                                      (BASELINE.json configs[4]); d_h0 / d_dh0 are supported (W_hh h0 is formed in fp32,
                                      h0 enters the gate math of the first step and dW_hh in fp32) */
#define BIGRU_PREC_BF16X3 2        /* fp32-class on tensor cores: (hi, lo) bf16 operand pairs, 3-4 products per term,
                                      fp32 accumulate / gate math / stash; meets the 1e-4 logit tolerance at tensor-core speed.
                                      hidden_size 128 or 256, batch % 32 == 0.
                                      Both tensor-core paths take any n_features (the layer-0 operands are stored with the
                                      feature extent zero-padded to a multiple of 8 inside the plan's workspaces).  Other
                                      batch sizes: append zero rows to x (and zero rows to d_logits) up to the next multiple -
                                      batch rows are independent; the Python mirror does exactly that.  Smaller hidden sizes:
                                      zero-pad the parameters to the next supported hidden size (padded units stay at state 0 and
                                      feed zero weights; BiGRU.plan_hidden / _pad_map of the mirror).  Anything else returns
                                      BIGRU_ERR_UNSUPPORTED. */

#define BIGRU_LOSS_CE   0          /* torch.nn.CrossEntropyLoss (BASELINE.json configs) */
#define BIGRU_LOSS_BCE  1          /* torch.nn.BCEWithLogitsLoss(weight,pos_weight) notebook raw :1192 */
#define BIGRU_LOSS_MLSM 2          /* torch.nn.MultiLabelSoftMarginLoss  predict.py:94 */

typedef struct bigru_plan bigru_plan;

const char* bigru_last_error(void);
int  bigru_version(void);
/* 0 when device `dev` exists and is compute capability 10.x */
int  bigru_device_check(int dev);

/* --- plan: shapes, offsets, workspace sizes.  Replaces BiGRU.__init__ bookkeeping
 *     (biGRU_model.py:32-60).  Immutable after creation. */
int  bigru_plan_create(int B, int T, int F, int H, int L, int C, int bidirectional, int precision,
                       bigru_plan** out);
int  bigru_plan_destroy(bigru_plan* plan);
int64_t bigru_param_count(const bigru_plan* plan);
/* which: 0 w_ih, 1 w_hh, 2 b_ih, 3 b_hh for layer<L; layer==L: 0 lin_w, 2 lin_b */
int  bigru_param_offset(const bigru_plan* plan, int layer, int dir, int which,
                        int64_t* offset, int64_t* rows, int64_t* cols);
/* stash: activations kept from forward for backward; scratch: reusable temporary space */
int  bigru_workspace_bytes(const bigru_plan* plan, size_t* stash_bytes, size_t* scratch_bytes);

/* byte offset, inside the stash written by the last forward, of argmax_t of the max-pooled output (int32 [B][H],
 * biGRU_model.py:125).  The max-pool's gradient routing is discontinuous where two time steps tie to within rounding;
 * parity tests read the routing that was actually taken (tests/test_gpu_parity.py). */
int  bigru_stash_argmax_offset(const bigru_plan* plan, size_t* byte_offset);

/* --- BiGRU.forward (biGRU_model.py:63-138): dropout :87-94, nn.GRU :102, head :111-137.
 *  d_x[B,T,F]; d_h0 nullable [L*D,B,H] (the `hidden` argument); d_logits[B,C];
 *  d_hn nullable [L*D,B,H]; training!=0 applies dropout p (spatial!=0: per (b,f) channel over T,
 *  :87-92; inter-layer dropout when L>1, :55) with a counter-based generator keyed by `seed`. */
int  bigru_forward(const bigru_plan* plan, const float* d_params, const float* d_x, const float* d_h0,
                   float dropout_p, int spatial, int training, uint64_t seed,
                   void* d_stash, void* d_scratch, float* d_logits, float* d_hn, void* stream);

/* --- loss.backward() through the model (biGRU_model.py:204): every parameter gradient into
 *  d_grads (flat, overwritten), optional d_dx[B,T,F] and d_dh0[L*D,B,H].  d_x may be NULL after
 *  bigru_forward_windows (the input is then taken from the stash).  Must follow
 *  bigru_forward on the same plan/stash with the same dropout arguments. */
int  bigru_backward(const bigru_plan* plan, const float* d_params, const float* d_x, const float* d_h0,
                    float dropout_p, int spatial, int training, uint64_t seed,
                    const void* d_stash, void* d_scratch, const float* d_dlogits,
                    float* d_grads, float* d_dx, float* d_dh0, void* stream);

/* The same backward pass in two (or more) calls, layers layer_from .. layer_to downwards (tensor-core precisions only): the call
 * that starts at the top layer also zeroes d_grads and forms the head's gradients.  After bigru_backward_layers(.., L-1, 1, ..) the
 * gradients of layers >= 1 and of the head are final, so a data-parallel caller can start their all-reduce while
 * bigru_backward_layers(.., 0, 0, ..) still runs (BiGRU.train_step with enable_data_parallel does exactly that; no reference
 * counterpart: /root/reference has no distributed code). */
int  bigru_backward_layers(const bigru_plan* plan, const float* d_params, const float* d_x, const float* d_h0,
                           float dropout_p, int spatial, int training, uint64_t seed,
                           const void* d_stash, void* d_scratch, const float* d_dlogits,
                           float* d_grads, float* d_dx, float* d_dh0, int layer_from, int layer_to, void* stream);

/* --- losses (biGRU_model.py:202 `self.loss_fn(pred, target)`), fused value + d(loss)/d(logits).
 *  kind CE: d_target int64[B]; BCE/MLSM: d_target float[B,C]; d_weight/d_pos_weight nullable [C]
 *  (BCE only).  Mean reduction over `denom` elements (B for CE, B*C otherwise; pass the GLOBAL
 *  count under data parallelism).  d_loss: one float, overwritten. */
int  bigru_loss(int kind, const float* d_logits, const void* d_target, const float* d_weight,
                const float* d_pos_weight, int B, int C, double denom, float* d_loss,
                float* d_dlogits, void* stream);

/* --- nn.utils.clip_grad_norm_ + optimizer.step() (biGRU_model.py:208-210, Adam, notebook raw :1194)
 *  bigru_sqnorm accumulates sum(g^2) into *d_out (caller zeroes it first);
 *  bigru_clip_adam_step: g *= grad_scale; coef = min(1, clip/(sqrt(*d_sqnorm)*grad_scale+1e-6));
 *  g *= coef; Adam(lr,b1,b2,eps) with bias correction for `step` (1-based). */
int  bigru_sqnorm(const float* d_g, int64_t n, float* d_out, void* stream);
int  bigru_clip_adam_step(float* d_params, float* d_grads, float* d_m, float* d_v, int64_t n,
                          const float* d_sqnorm, float clip, float lr, float b1, float b2, float eps,
                          int step, float grad_scale, void* stream);

/* Device-resident step counter variant of the same update, for CUDA-graph capture of the train step (SURVEY.md 8(f) N5):
 *  bigru_adam_tick: *d_step += 1, *d_sqnorm = 0 (one tiny launch, before bigru_sqnorm);
 *  bigru_clip_adam_step_dev: as bigru_clip_adam_step with the bias corrections formed on the device from *d_step. */
int  bigru_adam_tick(int* d_step, float* d_sqnorm, void* stream);
int  bigru_clip_adam_step_dev(float* d_params, float* d_grads, float* d_m, float* d_v, int64_t n,
                              const float* d_sqnorm, float clip, float lr, float b1, float b2, float eps,
                              const int* d_step, float grad_scale, void* stream);

/* --- MySQLBatchLoader collation (sql_pytorch_dataloader.py:239-245 + default_collate):
 *  out[b,t,f] = (src[start+b+t, f] - xmin[f]) / (xmax[f] - xmin[f]);  src is [N,F], start+B+T-1 <= N.
 *  xmin/xmax nullable (then a plain gather).  targets: out[b,0,c] = y[start+b+T-1, c]. */
int  bigru_window_gather_norm(const float* d_src, const float* d_xmin, const float* d_xmax,
                              int64_t start, int64_t N, int B, int T, int F, float* d_out, void* stream);
int  bigru_window_targets(const float* d_y, int64_t start, int64_t N, int B, int T, int C,
                          float* d_out, void* stream);

/* --- SURVEY.md 8(f) N1, zero-copy windows: forward straight from the HBM-resident chunk src[N,F] - the batch
 *  x[b,t,:] = (src[start+b+t,:] - xmin) / (xmax - xmin) is formed inside the first kernel of the path and never
 *  materialised as fp32 [B,T,F] by the caller (sql_pytorch_dataloader.py:239-245 + biGRU_model.py:63).  Pair it with
 *  bigru_backward(..., d_x = NULL, ...): the backward then takes the layer-0 input from the stash. */
int  bigru_forward_windows(const bigru_plan* plan, const float* d_params, const float* d_src, const float* d_xmin,
                           const float* d_xmax, int64_t start, int64_t N, float dropout_p, int spatial, int training,
                           uint64_t seed, void* d_stash, void* d_scratch, float* d_logits, float* d_hn, void* stream);

/* --- SURVEY.md 8(f) N3, chunk statistics on the GPU: per-feature MIN / MAX over rows [row_lo, row_hi) of a
 *  table[N,F] (NaN = SQL NULL, ignored), i.e. the two aggregate queries of MySQLChunkLoader
 *  (sql_pytorch_dataloader.py:96-105).  The min==max guard and order-book sharing stay on the host. */
int  bigru_chunk_minmax(const float* d_table, int64_t N, int F, int64_t row_lo, int64_t row_hi, float* d_min,
                        float* d_max, void* stream);

/* --- SURVEY.md 8(f) N4, the SQL window-function features of the reference (create_database.py:76-190) over the joined
 *  table's columns (device pointers, n rows, time order): per row, in the order of the reference's join statement
 *  (create_database.py:239-240): [upper_BB_dist, lower_BB_dist] (bb_period > 0; STD is the population std), vol_MA{p},
 *  price_MA{p}, delta_MA{p} (AVG over ROWS BETWEEN p-1 PRECEDING AND CURRENT ROW, shorter at the head of the table),
 *  [stoch] (15-row MIN / MAX of close; NaN = SQL NULL when max == min), ATR (15-row AVG(high - low)), price_change
 *  (close - LAG(close, 1); NaN on the first row) -> d_out[n][n_out]; and the four targets up1, up2, down1, down2
 *  (create_database.py:163-185: LEAD(close, 8 / 15) against close +- n1 / n2 * ATR, 0 where the lead is NULL)
 *  -> d_targets[n][4] (nullable).  At most 8 periods per list.  Returns n_out through *n_out (pass d_out = NULL to query). */
int  bigru_window_features(const float* d_close, const float* d_high, const float* d_low, const float* d_volume,
                           const float* d_delta, int64_t n, const int* vol_periods, int n_vol, const int* price_periods,
                           int n_price, const int* delta_periods, int n_delta, int bb_period, float bb_std,
                           int stochastic, float n1, float n2, float* d_out, float* d_targets, int* n_out, void* stream);

/* --- SURVEY.md 8(f) N5, the live predictor's forward pass in one launch (predict.py:165-181): normalise the raw
 *  window(s) d_x[B,T,F] with d_xmin/d_xmax[F] (nullable: already normalised), eval-mode forward of the flat parameters
 *  (order above), d_logits[B,C] and d_probs[B,C] = sigmoid(logits) (nullable).  One CTA per window, activations in shared
 *  memory, fp32 exact math; for small live windows only: D*H <= 1024 and T*(max(F,D*H)+D*H)*4 bytes of shared memory
 *  (BIGRU_ERR_UNSUPPORTED beyond) - batches belong to bigru_forward. */
int  bigru_infer_window(const float* d_params, const float* d_x, const float* d_xmin, const float* d_xmax, int B, int T,
                        int F, int H, int L, int C, int bidirectional, float* d_logits, float* d_probs, void* stream);

/* --- The live predictor's forward for full-size models (any T, F, L; H <= 512): same inputs, outputs and fp32 exact math
 *  as bigru_infer_window, for a few windows at a time (B of 1 to ~16 is the intended use; any B works).  Per layer one
 *  SGEMM forms the input projection of all T steps, then one thread-block cluster per (direction, group of up to 4
 *  windows) walks the recurrence with its W_hh slices resident in shared memory, exchanging h through distributed shared
 *  memory each step; a last kernel applies the pooling head, Linear and sigmoid.  2L+1 launches (2L+2 with d_xmin).
 *  Hidden sizes above 256 need a 16-CTA (non-portable) cluster; where the device does not grant one, and for H > 512,
 *  the call returns BIGRU_ERR_UNSUPPORTED with a message.  d_work: caller-owned device buffer, 16-byte aligned, of
 *  bigru_infer_cluster_workspace_bytes() bytes for the same (B, T, F, H, L, bidirectional); the library never
 *  allocates.  The workspace query needs no device. */
int  bigru_infer_cluster_workspace_bytes(int B, int T, int F, int H, int L, int bidirectional, size_t* bytes);
int  bigru_infer_cluster(const float* d_params, const float* d_x, const float* d_xmin, const float* d_xmax, int B, int T, int F,
                         int H, int L, int C, int bidirectional, void* d_work, float* d_logits, float* d_probs, void* stream);
/* The launch geometry bigru_infer_cluster picks on the current device for B windows of hidden size H: CTAs per cluster,
 *  hidden units per CTA, windows per cluster, and cudaOccupancyMaxActiveClusters of that launch.  Needs the device. */
int  bigru_infer_cluster_geometry(int B, int H, int bidirectional, int* cluster_ctas, int* units_per_cta, int* windows_per_cluster,
                                  int* max_active_clusters);

/* --- train_model/evaluate_model metrics (biGRU_model.py:213-221): pred = sigmoid(logit) > 0.5;
 *  d_counts[0] += #rows with all labels right; [1] += #label mismatches;
 *  [2+3c], [3+3c], [4+3c] += tp, fp, fn of class c.  int64 accumulators, caller zeroes. */
int  bigru_multilabel_counts(const float* d_logits, const float* d_target, int B, int C,
                             long long* d_counts, void* stream);

/* --- measurement hooks used by bench.py (no reference counterpart).
 *  bigru_launch_count: kernels launched by this library since load (gpu_launches).
 *  bigru_prof_enable(1): every subsequent launch is bracketed by CUDA events on its own stream;
 *  bigru_prof_report(cls): summed device time, launch count, algorithmic flops and bytes of one
 *  kernel class (names via bigru_prof_class_name) since the last enable.  Timing adds event records
 *  to the stream, so bench.py enables it only for a separate, untimed-for-throughput pass. */
long long   bigru_launch_count(void);
void        bigru_launch_count_add(long long n);   /* launches replayed from a captured CUDA graph (not seen by the macros) */
int         bigru_prof_enable(int on);
int         bigru_prof_classes(void);
const char* bigru_prof_class_name(int cls);
int         bigru_prof_report(int cls, double* ms, long long* launches, double* flops, double* bytes);

#ifdef __cplusplus
}
#endif
#endif
