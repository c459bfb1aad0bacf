/*
 * deeptables_b200 -- C ABI of the B200-native feature-interaction engine.
 *
 * The reference (DataCanvasIO/DeepTables) has no native boundary at all: every op below is, in
 * the reference, a chain of TensorFlow/Keras ops inside a Keras layer (file:line cited per
 * entry point, relative to /root/reference).  This header is therefore the boundary a
 * maintainer would bind (ctypes stub shown in INTEGRATION.md) to replace those layers' `call`
 * bodies.  Conventions:
 *
 *  - every pointer is a DEVICE pointer unless the name ends in `_host`; the caller owns every
 *    buffer (outputs and workspaces alike); the library never allocates device memory and links no GEMM library;
 *  - `stream` is a `cudaStream_t` passed as `void*`; all work is enqueued asynchronously on it;
 *  - return value: 0 = OK, negative = error (DTB_ERR_*); `dtb_last_error()` gives the text;
 *    no C++ exception crosses this boundary;
 *  - categorical ids: `idx` is int32 [B, F] row-major; the F tables live in ONE buffer
 *    `table` [sum_f V_f, D] (row-major, uniform D) with `row_offsets` int64 [F+1] the prefix sum
 *    of the vocabulary sizes (device memory).  Row r of field f is table[(row_offsets[f]+r)*D].
 *    An id outside [0, V_f) sets bit f&31 of *status (if status != NULL) and reads as zeros
 *    (TF-GPU behaviour; TF-CPU raises -- the host checks `status`, layers.py:893-898);
 *  - embedding gradients are scatter-ADDED into `grad_table` (same shape as `table`), which the
 *    caller keeps zeroed between steps (the row-wise Adam kernel re-zeroes rows it consumes);
 *  - fp32 everywhere unless stated; "rows" are batch rows.
 */
#ifndef DEEPTABLES_B200_H_
#define DEEPTABLES_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTB_OK 0
#define DTB_ERR_INVALID_ARG (-1)
#define DTB_ERR_UNSUPPORTED (-2)
#define DTB_ERR_CUDA (-3)

/* activation codes (keras Activation names the hot path uses) */
#define DTB_ACT_NONE 0
#define DTB_ACT_RELU 1
#define DTB_ACT_TANH 2 /* Dense layers and the FGCNN convolution (layers.py:211,219) */

/* ---- library ---------------------------------------------------------------------------- */
int dtb_version(void);
const char* dtb_last_error(void);
int dtb_device_sm_count(int* out_host);
/* debug aid: 0 = `stream` is not capturing, 1 = capturing, 2 = its capture has been invalidated, < 0 = -cudaError */
int dtb_capture_status(void* stream);
/* number of kernels this library has launched so far (every kernel on the path is hand-written) */
long long dtb_launch_count(void);
/* kernels launched by replaying a CUDA graph captured through this library (counted once at capture): added per replay */
void dtb_launch_count_add(long long n);

/* ---- MultiColumnEmbedding (layers.py:889-904) ------------------------------------------- */
/* out[B,F,D] = table rows; the materialising form used by custom nets / tests. */
int dtb_embedding_gather(const int32_t* idx, const float* table, const int64_t* row_offsets,
                         float* out, int B, int F, int D, int* status, void* stream);
/* grad_table[row] += d_out[b,f,:]  (gradient of embedding_lookup). */
int dtb_embedding_scatter_add(const int32_t* idx, const int64_t* row_offsets, const float* d_out,
                              float* grad_table, int B, int F, int D, void* stream);

/* ---- linear (deepnets.py:43-66) + FM (layers.py:53-62), gather fused -------------------- */
/* out_lin[b] = sum_f w_lin[f]*sum_d e[b,f,d] + sum_c w_lin[F+c]*dense[b,c]   (NULL: skipped)
 * out_fm[b]  = 0.5*sum_d[(sum_f e)^2 - sum_f e^2]                             (NULL: skipped)
 * dense may be NULL iff C == 0; idx/table may be NULL iff F == 0. */
int dtb_fm_linear_fwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                      const float* dense, const float* w_lin, float* out_lin, float* out_fm,
                      int B, int F, int D, int C, int* status, void* stream);
/* g_lin/g_fm: dLoss/d out_lin, dLoss/d out_fm [B] (NULL: that branch absent).
 * grad_table += dE ; grad_wlin[F+C] += dW (both accumulate). */
int dtb_fm_linear_bwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                      const float* dense, const float* w_lin, const float* g_lin, const float* g_fm,
                      float* grad_table, float* grad_wlin, int B, int F, int D, int C, void* stream);

/* ---- flatten_embeddings + concat_embedding_dense (deepmodel.py:269-278,348-357) --------- */
/* X[b, :] = [e[b,0,:], ..., e[b,F-1,:], dense[b,:]]   width W = F*D + C. */
int dtb_concat_emb_dense_fwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                             const float* dense, float* X, int B, int F, int D, int C, int* status,
                             void* stream);
/* grad_table += dX[:, :F*D] scattered by idx (the dense columns are inputs: no gradient). */
int dtb_concat_emb_dense_bwd(const int32_t* idx, const int64_t* row_offsets, const float* dX,
                             float* grad_table, int B, int F, int D, int C, void* stream);

/* ---- BatchNormalization(axis=-1) (deepmodel.py:359; layers.py:152; deepnets.py:422) ------ */
/* Training forward over X[rows, cols]: batch mean / biased variance (two-pass, fp64 accumulate),
 * Y = gamma*(X-mean)*rsqrt(var+eps)+beta, save_mean/save_var [cols] written for backward, and
 * moving = moving*momentum + batch*(1-momentum).  Y may alias X. */
int dtb_batchnorm_train_fwd(const float* X, float* Y, const float* gamma, const float* beta,
                            float* moving_mean, float* moving_var, float* save_mean, float* save_var,
                            double* workspace /* [2*cols] */, int rows, int cols, float eps,
                            float momentum, void* stream);
/* Inference forward with the moving statistics. */
int dtb_batchnorm_infer_fwd(const float* X, float* Y, const float* gamma, const float* beta,
                            const float* moving_mean, const float* moving_var, int rows, int cols,
                            float eps, void* stream);
/* Backward of the training forward.  dX may alias dY.  dgamma/dbeta [cols] accumulate. */
int dtb_batchnorm_bwd(const float* X, const float* dY, float* dX, const float* gamma,
                      const float* save_mean, const float* save_var, float* dgamma, float* dbeta,
                      double* workspace /* [2*cols] */, int rows, int cols, float eps, void* stream);

/* ---- Dense (keras Dense used by deepnets.dnn 415-424, stacking 292, task_output 455; the four
 * projections of MultiheadAttention, layers.py:106-127) ----------------------------------------- */
/* Layers wider than 8 outputs run as hand-written tcgen05 GEMMs (csrc/dense_tc.cu: operands split on the fly into
 * bf16 hi + lo, three tensor passes, fp32 accumulation in TMEM => fp32-grade results; bias / activation fused into the
 * accumulator read-out); out_dim <= 8 (logit layers) as row-dot kernels.  The GEMM path packs the weights into
 * `workspace` (dtb_dense_workspace_bytes(in_dim, out_dim), 16-byte aligned; 0 for the narrow kernels). */
size_t dtb_dense_workspace_bytes(int in_dim, int out_dim);
/* Y[rows,out] = act(X[rows,in] @ W[in,out] + bias).  bias may be NULL. */
int dtb_dense_fwd(const float* X, const float* W, const float* bias, float* Y, void* workspace,
                  size_t workspace_bytes, int rows, int in_dim, int out_dim, int act, void* stream);
/* dY holds dLoss/dY on entry and is overwritten with dLoss/d(pre-activation).  dX may be NULL.
 * dW[in,out] and dbias[out] accumulate (dbias may be NULL). */
int dtb_dense_bwd(const float* X, const float* W, const float* Y, float* dY, float* dX, float* dW,
                  float* dbias, void* workspace, size_t workspace_bytes, int rows, int in_dim, int out_dim,
                  int act, void* stream);

/* ---- Dropout (keras Dropout, deepmodel.py:430, deepnets.py:426; SpatialDropout1D on the (B,1,D)
 * field embeddings, layers.py:878-901, is element-wise too) -------------------------------------- */
/* Y[i] = keep(seed, i) ? X[i]/(1-rate) : 0 with a counter-based mask: calling it again on dLoss/dY with
 * the same seed IS the backward.  Y may alias X. */
int dtb_dropout(const float* X, float* Y, int64_t n, float rate, unsigned long long seed, void* stream);

/* ---- losses on the task_output pre-activation (deepmodel.py:319-346, 436-457) ------------ */
/* task: 0 binary/multilabel (sigmoid + BCE, probabilities clipped to [1e-7,1-1e-7] as keras),
 *       1 regression (identity + MSE), 2 multiclass (softmax + CCE, y one-hot).
 * prob[rows,cols] always written; if dz != NULL: dz = dLoss/dz with Loss = mean over rows (and
 * over cols for task 0/1) of the per-sample loss times sample_weight (NULL = 1).
 * loss_sum (double, device, may be NULL) += sum of per-row losses (un-normalised). */
int dtb_loss_fwd_bwd(const float* z, const float* y_true, const float* sample_weight, float* prob,
                     float* dz, double* loss_sum, int rows, int cols, int task, void* stream);

/* Focal losses (layers.py:983-1083) passed as ModelConfig.loss: task 0 BinaryFocalLoss (sigmoid; the
 * loss is the mean over all rows x cols elements), task 2 CategoricalFocalLoss (softmax; mean over
 * rows of the per-sample sums).  Same outputs as dtb_loss_fwd_bwd; no sample weights. */
int dtb_focal_loss_fwd_bwd(const float* z, const float* y_true, float* prob, float* dz,
                           double* loss_sum, int rows, int cols, int task, float gamma, float alpha,
                           void* stream);

/* ---- keras Adam (deepmodel.py:321-322), dense semantics ---------------------------------- */
/* m += (g-m)(1-b1); v += (g^2-v)(1-b2); p -= m*alpha/(sqrt(v)+eps), alpha computed by caller
 * as lr*sqrt(1-b2^t)/(1-b1^t).  If zero_grad != 0, g is zeroed after use. */
int dtb_adam_dense(float* p, float* m, float* v, float* g, int64_t n, float alpha, double beta1,
                   double beta2, float eps, int zero_grad, void* stream);

/* Exact-lazy row-wise Adam for embedding tables (same arithmetic as dtb_adam_dense applied to
 * every row every step, but rows whose gradient is zero are caught up only when next touched).
 * last_step[row] = last optimiser step already applied to that row.  alpha_table[s] (device,
 * s = 1..) = alpha of step s.
 *   catchup: for every (b,f): apply the zero-gradient steps last_step+1 .. upto to that row once.
 *   apply  : for every (b,f): apply step `step` with the accumulated grad_table row once, zero
 *            the grad row, set last_step = step. */
int dtb_adam_rows_catchup(const int32_t* idx, const int64_t* row_offsets, float* table, float* m,
                          float* v, int32_t* last_step, const float* alpha_table, int upto,
                          double beta1, double beta2, float eps, int B, int F, int D, void* stream);
int dtb_adam_rows_apply(const int32_t* idx, const int64_t* row_offsets, float* table, float* m,
                        float* v, float* grad_table, int32_t* last_step, const float* alpha_table,
                        int step, double beta1, double beta2, float eps, int B, int F, int D,
                        void* stream);
/* Bring every row of the table up to date (before save / export / dense evaluation). */
int dtb_adam_rows_flush(float* table, float* m, float* v, int32_t* last_step,
                        const float* alpha_table, int upto, double beta1, double beta2, float eps,
                        int64_t n_rows, int D, void* stream);
/* CUDA-graph forms: the optimiser step counter lives in DEVICE memory (*step_dev = steps completed so far), so a
 * captured train step replays with the right bias correction: dense = step *step_dev + 1 with alpha_table[*step_dev + 1];
 * rows catch-up to *step_dev; rows apply = step *step_dev + 1; dtb_step_increment bumps the counter at the end. */
int dtb_adam_dense_dev(float* p, float* m, float* v, float* g, int64_t n, const float* alpha_table,
                       const int32_t* step_dev, double beta1, double beta2, float eps, int zero_grad, void* stream);
int dtb_adam_rows_catchup_dev(const int32_t* idx, const int64_t* row_offsets, float* table, float* m, float* v,
                              int32_t* last_step, const float* alpha_table, const int32_t* step_dev, double beta1,
                              double beta2, float eps, int B, int F, int D, void* stream);
int dtb_adam_rows_apply_dev(const int32_t* idx, const int64_t* row_offsets, float* table, float* m, float* v,
                            float* grad_table, int32_t* last_step, const float* alpha_table, const int32_t* step_dev,
                            double beta1, double beta2, float eps, int B, int F, int D, void* stream);
int dtb_step_increment(int32_t* step_dev, void* stream);

/* Data-parallel exchange of the embedding gradient by rows (deepmodel.py:88-103: MirroredStrategy
 * exchanges embedding gradients as IndexedSlices too).  pack: every (b,f) reference claims its row once
 * per step (claim[row] = step); the owner MOVES the accumulated gradient row into packed[b,f,:] and zeroes
 * the table row, other references of that row write zeros.  unpack: adds one rank's packed rows into the
 * local gradient table; at most one reference per row carries data, so no atomics are needed and
 * calling it for rank 0..W-1 in order yields identical bits on every replica. */
int dtb_grad_rows_pack(const int32_t* idx, const int64_t* row_offsets, float* grad_table, int32_t* claim,
                       float* packed /* [B,F,D] */, int step, int B, int F, int D, void* stream);
int dtb_grad_rows_unpack(const int32_t* idx, const int64_t* row_offsets, const float* packed,
                         float* grad_table, int B, int F, int D, void* stream);

/* ---- CIN (layers.py:638-734), gather fused ------------------------------------------------ */
/* Shapes: F0 = F fields, D, n_layers layer sizes L[k] (host array), direct flag; H[0]=F,
 * H[k+1] = direct ? L[k] : L[k]/2 (all L[k]); K[k] = F*H[k].
 * weights: concatenation of the n_layers filters, filter k is [K[k], L[k]] row-major (the
 * reference's f_k[0]); bias: concatenation of [L[k]] or NULL.  act in {NONE, RELU}.
 * pooled[B, P] with P = direct ? sum L : sum_{k<last} L[k]/2 + L[last]  (layers.py:725-726; the
 * final Dense(1) / residual MLP is a dtb_dense_* call).
 * saved (training only, may be NULL for inference): workspace of dtb_cin_saved_bytes() holding
 * the activations backward needs. */
size_t dtb_cin_saved_bytes(int B, int F, int D, const int* layer_sizes_host, int n_layers, int direct);
size_t dtb_cin_workspace_bytes(int B, int F, int D, const int* layer_sizes_host, int n_layers,
                               int direct, int training);
int dtb_cin_fwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                const float* weights, const float* bias, float* pooled, void* saved,
                void* workspace, size_t workspace_bytes, int B, int F, int D,
                const int* layer_sizes_host, int n_layers, int direct, int act, int precision,
                int* status, void* stream);
/* d_pooled[B,P] -> grad_table += dE, d_weights/d_bias accumulate. */
int dtb_cin_bwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                const float* weights, const float* d_pooled, const void* saved, float* grad_table,
                float* d_weights, float* d_bias, void* workspace, size_t workspace_bytes, int B, int F,
                int D, const int* layer_sizes_host, int n_layers, int direct, int act, int precision,
                void* stream);
/* The same backward in two launches: phase 1 = everything that contributes to grad_table (after it the
 * embedding gradient of this op is final), phase 2 = d_weights / d_bias.  The host starts the data-parallel
 * exchange of the table gradient between the two so that it overlaps the weight-gradient kernels. */
int dtb_cin_bwd_phase(const int32_t* idx, const float* table, const int64_t* row_offsets,
                      const float* weights, const float* d_pooled, const void* saved, float* grad_table,
                      float* d_weights, float* d_bias, void* workspace, size_t workspace_bytes, int B, int F,
                      int D, const int* layer_sizes_host, int n_layers, int direct, int act, int precision,
                      int phase, void* stream);
/* precision:
 *   0 = auto: ONE tensor pass on fp16 operands scaled by exact powers of two (per GEMM row / per layer; csrc/cin_tc2.cu:
 *       forward, data gradient and weight gradient, embedding dim 16 or 32, layer sizes multiples of 32, <= 64 hidden
 *       fields) -- error ~2e-4 of the output scale, inside the 1e-3 parity bar; shapes outside it fall to 2, then to 1;
 *   1 = the any-shape materialising formulation (outer product in HBM chunks + the bf16x3 GEMMs of csrc/dense_tc.cu);
 *   2 = tensor-core bf16x3 split (hi*hi + lo*hi + hi*lo, ~2^-16 per product: fp32-grade); 3 = one bf16 pass (4e-3: tests only);
 *   4 = force the single fp16 pass (DTB_ERR_UNSUPPORTED from forward and backward when the shape is outside it). */
#define DTB_CIN_AUTO 0
#define DTB_CIN_FP32 1
#define DTB_CIN_TC_BF16X3 2
#define DTB_CIN_TC_BF16X1 3
#define DTB_CIN_TC_F16X1 4
int dtb_cin_tc_supported(int F, int D, const int* layer_sizes_host, int n_layers, int direct);
/* which of the codes 1 / 2 / 4 a forward + backward with `precision` runs for this shape (0 = auto is resolved) */
int dtb_cin_resolved_precision(int F, int D, const int* layer_sizes_host, int n_layers, int direct, int precision);
/* Test hooks for the tensor-core path.  set_variant: process-wide flags read by later CIN calls; bit 0 is
 * accepted and ignored, bit 16 runs the exact-fp32 backward after a tensor-core forward, bit 17 keeps the full
 * (fp32 T_k) saved-activation format.  Any other bit returns DTB_ERR_INVALID_ARG and leaves the flags unchanged.
 * selftest: C[128,N] = bf16(A[128,K]) @ bf16(Bmat[K,N]) with one M=128 UMMA tile (N <= 128, K <= 64, multiples
 * of 16), the A operand through TMEM (a_operand_in_tmem = 1) or shared memory (0); workspace >= 4*N*K bytes. */
int dtb_cin_tc_set_variant(int flags);
int dtb_tc_selftest(const float* A, const float* Bmat, float* C, void* workspace, int N, int K,
                    int a_operand_in_tmem, void* stream);

/* ---- Cross (layers.py:417-436) on a dense [B,W] input ------------------------------------- */
/* x_{l+1} = x0*(x_l . w_l) + x_l + b_l ; kernels/biases [n_layers, W]; Y [B,W].
 * xw_saved [B, n_layers] keeps the per-layer scalars x_l.w_l for backward. */
int dtb_cross_fwd(const float* X, const float* kernels, const float* biases, float* Y,
                  float* xw_saved, int B, int W, int n_layers, void* stream);
size_t dtb_cross_bwd_workspace_bytes(int B, int W, int n_layers);
int dtb_cross_bwd(const float* X, const float* kernels, const float* biases, const float* xw_saved,
                  const float* dY, float* dX, float* d_kernels, float* d_biases, void* workspace,
                  size_t workspace_bytes, int B, int W, int n_layers, void* stream);

/* ---- InnerProduct / OuterProduct (layers.py:473-487, 541-581), gather fused --------------- */
/* ip[B,P] (NULL: skipped), op[B,P] (NULL: skipped); P = F(F-1)/2 pairs (i<j) row-major.
 * kernel_type 0 mat [D,P,D], 1 vec [P,D], 2 num [P,1]. */
int dtb_pnn_fwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                const float* op_kernel, float* ip, float* op, int B, int F, int D, int kernel_type,
                int* status, void* stream);
int dtb_pnn_bwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                const float* op_kernel, const float* d_ip, const float* d_op, float* grad_table,
                float* d_op_kernel, int B, int F, int D, int kernel_type, void* stream);

/* ---- AFM (layers.py:742-812; afm_nets deepnets.py:99-107), gather fused ---------------------- */
/* pooled[B,D] = sum_p softmax_p(act((e_i*e_j) att_kernel + att_bias) . projection_h) (e_i*e_j) over
 * the F(F-1)/2 field pairs in itertools.combinations order (what AFM.call hands to its Dropout and
 * Dense(1, use_bias=False)).  att_kernel [D,H] row-major, att_bias [H], projection_h [H];
 * act = DTB_ACT_NONE | DTB_ACT_RELU.  D in {4,8,16,32}, H <= 32, else DTB_ERR_UNSUPPORTED.
 * Backward: adds into grad_table (same layout as the table) and into d_att_kernel / d_att_bias /
 * d_projection_h (caller zero-fills); workspace of dtb_afm_workspace_bytes(B,F,D,H) bytes. */
size_t dtb_afm_workspace_bytes(int B, int F, int D, int H);
int dtb_afm_fwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                const float* att_kernel, const float* att_bias, const float* projection_h,
                float* pooled, int B, int F, int D, int H, int act, int* status, void* stream);
int dtb_afm_bwd(const int32_t* idx, const float* table, const int64_t* row_offsets,
                const float* att_kernel, const float* att_bias, const float* projection_h,
                const float* d_pooled, float* grad_table, float* d_att_kernel, float* d_att_bias,
                float* d_projection_h, void* workspace, size_t workspace_bytes, int B, int F, int D,
                int H, int act, void* stream);

/* ---- FiBiNet: SENET + BilinearInteraction (layers.py:245-382; fibi_nets deepnets.py:344-371) -- */
/* On a dense block X [B,F,D] (the concatenated embeddings or their SENET re-weighting).
 * Bilinear: out[b,p,:] = (x_i W_s) * x_j over the F(F-1)/2 pairs in itertools.combinations order;
 * W [n_w,D,D] row-major, bilinear_type 0 field_all (n_w = 1, s = 0) | 1 field_each (n_w = F-1, s = i)
 * | 2 field_interaction (n_w = pairs, s = p).  Backward: dX [B,F,D] overwritten (may be NULL), dW
 * accumulated (caller zero-fills).  D in {4,8,16,32}, else DTB_ERR_UNSUPPORTED.
 * SENET: Z[b,f] = mean (pooling_op 0) or max (1) over d; V = X * A[:,:,None]; the two Dense layers
 * between Z and A are dtb_dense_* calls.  Max-pool gradient: ties share it (tf.reduce_max). */
int dtb_bilinear_fwd(const float* X, const float* W, float* out, int B, int F, int D,
                     int bilinear_type, void* stream);
int dtb_bilinear_bwd(const float* X, const float* W, const float* d_out, float* dX, float* dW, int B,
                     int F, int D, int bilinear_type, void* stream);
int dtb_senet_pool_fwd(const float* X, float* Z, int B, int F, int D, int pooling_op, void* stream);
int dtb_senet_pool_bwd(const float* X, const float* Z, const float* dZ, float* dX, int B, int F,
                       int D, int pooling_op, void* stream);
int dtb_senet_scale_fwd(const float* X, const float* A, float* V, int B, int F, int D, void* stream);
int dtb_senet_scale_bwd(const float* X, const float* A, const float* dV, float* dX, float* dA, int B,
                        int F, int D, void* stream);

/* ---- FGCNN (layers.py:161-242; fg_nets deepnets.py:227-261) -------------------------------- */
/* Channels-last block X [B,H,W,Cin] (H = fields, W = embedding width).  Convolution along H only:
 * Y[b,h,w,co] = act(bias[co] + sum_{t,ci} X[b,h+t-pad,w,ci] kernel[t,ci,co]), kernel [kh,1,Cin,Cout]
 * as Keras stores it, TensorFlow 'same' padding (pad = (kh-1)/2 in front), act = NONE | RELU | TANH.
 * Cin, Cout <= 32, kh <= 8, else DTB_ERR_UNSUPPORTED.  Backward: dX overwritten (may be NULL),
 * d_kernel / d_bias accumulated (caller zero-fills; d_bias may be NULL).
 * Max pooling along H: windows of `pool` rows, stride `pool`, 'same' padding; Y [B,ceil(H/pool),WC];
 * the gradient goes to the first maximum of a window; dX [B,H,WC] overwritten.
 * The recombination layer is dtb_dense_fwd/bwd with DTB_ACT_TANH. */
int dtb_conv_fields_fwd(const float* X, const float* kernel, const float* bias, float* Y, int B,
                        int H, int W, int Cin, int Cout, int kh, int act, void* stream);
int dtb_conv_fields_bwd(const float* X, const float* kernel, const float* Y, const float* dY,
                        float* dX, float* d_kernel, float* d_bias, int B, int H, int W, int Cin,
                        int Cout, int kh, int act, void* stream);
int dtb_maxpool_fields_fwd(const float* X, float* Y, int B, int H, int WC, int pool, void* stream);
int dtb_maxpool_fields_bwd(const float* X, const float* dY, float* dX, int B, int H, int WC, int pool,
                           void* stream);

/* ---- MultiheadAttention core (layers.py:129-150), between the projections and the BN ------- */
/* qkvr [B, F, 4*D]: the four relu(Dense) projections of each field row, concatenated [Q|K|V|R]
 * (one dtb_dense_fwd with the four kernels side by side).  Y[B,F,D] = relu(concat_h softmax(Q_h
 * K_h^T / sqrt(D/heads)) V_h + R).  Backward: d_qkvr [B,F,4*D] (overwritten); with mask_relu_inputs
 * the result is zeroed where qkvr is zero, i.e. it is the gradient of the PRE-relu projections (the
 * caller then runs dtb_dense_bwd with act = linear and skips the activation-gradient pass). */
int dtb_attention_core_fwd(const float* qkvr, float* Y, int B, int F, int D, int heads,
                           int use_residual, void* stream);
int dtb_attention_core_bwd(const float* qkvr, const float* Y, const float* dY, float* d_qkvr, int B,
                           int F, int D, int heads, int use_residual, int mask_relu_inputs,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DEEPTABLES_B200_H_ */
