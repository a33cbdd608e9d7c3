/* lcrec_b200 - C ABI of the B200-native LC-Rec item-indexing hot path.
 *
 * The reference (jiaozihao18/LC-Rec, index/) is pure Python on torch; it has no FFI of its own.
 * This header is the boundary a maintainer binds with ctypes (see INTEGRATION.md): every entry
 * point names the reference code it replaces.  All pointers are BORROWED.  `stream` is a
 * cudaStream_t passed as void* (NULL = legacy default stream).  Device pointers unless a name
 * ends in `_host`.  Return value: 0 = LCREC_OK, otherwise an LCREC_ERR_* code; the text of the
 * last error on the calling thread is available from lcrec_last_error().  There is no CPU
 * fallback anywhere: on a machine without an sm_100 device every compute call fails with
 * LCREC_ERR_CUDA / LCREC_ERR_UNSUPPORTED.
 */
#ifndef LCREC_B200_H
#define LCREC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCREC_OK 0
#define LCREC_ERR_ARG 1          /* bad argument (NULL, size, alignment)            */
#define LCREC_ERR_CUDA 2         /* CUDA runtime / driver error                      */
#define LCREC_ERR_UNSUPPORTED 3  /* shape or device outside what the kernels cover   */
#define LCREC_ERR_NOMEM 4        /* workspace too small / allocation failure         */
#define LCREC_ERR_NUMERIC 5      /* reference `assert amplitude > 0` (vq.py:59) etc. */

#define LCREC_MAX_LEVELS 8

/* ---- library ------------------------------------------------------------------------- */
int lcrec_version(void);
const char* lcrec_strerror(int code);
const char* lcrec_last_error(void);
/* LCREC_OK iff the current CUDA device is compute capability 10.x (B200). */
int lcrec_device_check(void);

/* ---- a2: MLPLayers.forward (index/models/layers.py:18-43) ------------------------------
 * y = relu(x W^T + b) per layer, last layer without ReLU unless relu_last.  Eval-mode
 * BatchNorm1d is folded into (W, b) by the caller.  fp32-accurate: every product is
 * evaluated as 3 tcgen05 MMAs (hi*hi + lo*hi + hi*lo) on a two-term operand split (fp16 pairs
 * with power-of-two scales by default, tf32 pairs with engine 0) with chunked fp32 accumulation.
 * `weights[i]` is (dims[i+1], dims[i]) row-major like nn.Linear.weight.  The handle owns
 * split copies of the weights; call lcrec_mlp_update() after the caller changes them.
 */
typedef struct lcrec_mlp lcrec_mlp_t;
int lcrec_mlp_create(int n_layers, const int32_t* dims, const float* const* weights,
                     const float* const* biases, int relu_last, void* stream, lcrec_mlp_t** out);
int lcrec_mlp_update(lcrec_mlp_t* mlp, const float* const* weights, const float* const* biases,
                     void* stream);
int lcrec_mlp_destroy(lcrec_mlp_t* mlp);
int64_t lcrec_mlp_workspace_bytes(const lcrec_mlp_t* mlp, int64_t n_rows);
/* acts (nullable): n_layers device pointers receiving the fp32 output of every layer
 * (acts[n_layers-1] may alias y).  Used by the training path to keep activations. */
int lcrec_mlp_forward(lcrec_mlp_t* mlp, const float* x, int64_t n_rows, float* y,
                      float* const* acts, void* workspace, int64_t workspace_bytes, void* stream);
/* The same with x of element type `dtype`: 0 = fp32, 1 = fp16, 2 = bf16 (the codes of lcrec_masked_mean_pool).  Half
 * inputs are read as they are (no fp32 copy) and converted to fp32 in the layer-1 operand split; the result is
 * bit-identical to lcrec_mlp_forward on the input upcast to fp32.  x: (n_rows, dims[0]) contiguous; any alignment
 * (a misaligned base falls back to scalar loads).  dtype outside {0, 1, 2}: LCREC_ERR_ARG, before anything touches the
 * device.  Half input with engine 0 (tf32 x3): LCREC_ERR_UNSUPPORTED.  lcrec_mlp_forward(...) is
 * lcrec_mlp_forward_ex(mlp, x, 0, ...). */
int lcrec_mlp_forward_ex(lcrec_mlp_t* mlp, const void* x, int dtype, int64_t n_rows, float* y,
                         float* const* acts, void* workspace, int64_t workspace_bytes, void* stream);
/* accumulation chunk: number of K elements accumulated inside TMEM before the partial sum is
 * folded into fp32 registers with round-to-nearest (0 = whole K in TMEM). */
int lcrec_mlp_set_acc_chunk(lcrec_mlp_t* mlp, int k_elems);
/* kernel selection / measurement switches (bit mask): 1 = alternative stage shape of the single-CTA kernel,
 * 4 = no TMA loads after the first ring fill, 8 = no MMAs (4 and 8: timing experiments, results are garbage),
 * 16 = never use the CTA-pair kernel, 32 = CTA-pair kernel with 6 x 32 KB stages instead of 3 x 64 KB. */
int lcrec_mlp_set_variant(lcrec_mlp_t* mlp, int variant);
/* persistent grid of the CTA-pair GEMM limited to `cap` CTA pairs (0 = all 74): leaves SMs to kernels that run
 * concurrently on other streams (the pair GEMM is power-bound, memory-bound stages are not) */
int lcrec_pair_set_cluster_cap(int cap);
/* measurement only: device buffer of 6 x 512 x 4 int64 that receives clock64 stamps of the pipeline roles of
 * one CTA of the layer-0 pair kernel (producer / MMA k-blocks / MMA chunks / fold), or NULL to switch off. */
int lcrec_mlp_set_trace(lcrec_mlp_t* mlp, void* trace);
/* operand encoding of the GEMMs: 0 = tf32 x3 (fp32 operands split into two tf32 numbers), 1 = f16 x3 (per-row
 * power-of-two scale, two fp16 numbers; same 22-bit operand precision, twice the tensor rate). */
int lcrec_mlp_set_engine(lcrec_mlp_t* mlp, int engine);
int lcrec_mlp_in_dim(const lcrec_mlp_t* mlp);
int lcrec_mlp_out_dim(const lcrec_mlp_t* mlp);
/* One nn.Linear (+ReLU) on raw fp32 operands (layers.py:23): splits x and w on the fly into ws.
 * variant: bit 0 = alternative tile for wide N, bit 1 = f16 x3 engine. */
int64_t lcrec_linear_workspace_bytes(int64_t n_rows, int k_in, int n_out);
int lcrec_linear_forward(const float* x, int64_t n_rows, int k_in, const float* w, const float* b,
                         int n_out, int relu, float* y, int acc_chunk, int variant, void* ws,
                         int64_t ws_bytes, void* stream);

/* Backward of one nn.Linear (+ fused ReLU) for the training step (trainer.py:114-118): with g = gy * (y_relu > 0)
 * (y_relu = the layer's ReLU output, NULL when the forward did not fuse a ReLU): gb = column sums of g,
 * gx = g W, gw = g^T x - both on the fp32-accurate split-operand tensor-core GEMMs (operands are transposed by a
 * tiled copy so that the contraction dimension is contiguous).  Any of gx / gw / gb may be NULL.  k_in, n_out
 * multiples of 4. */
int64_t lcrec_linear_backward_workspace_bytes(int64_t n_rows, int k_in, int n_out);
int lcrec_linear_backward(const float* x, const float* w, const float* y_relu, const float* gy, int64_t n_rows,
                          int k_in, int n_out, float* gx, float* gw, float* gb, void* ws, int64_t ws_bytes,
                          void* stream);
/* Backward of a whole MLPLayers stack in one call: acts[l] = output of layer l as returned by lcrec_mlp_forward(acts),
 * gy = gradient w.r.t. the stack's output; gw[l] (dims[l+1] x dims[l]) and gb[l] receive the parameter gradients,
 * gx (nullable) the input gradient.  weights[l]: the fp32 weights the forward used. */
int64_t lcrec_mlp_backward_workspace_bytes(const lcrec_mlp_t* mlp, int64_t n_rows);
int lcrec_mlp_backward(lcrec_mlp_t* mlp, const float* const* weights, const float* x, const float* const* acts,
                       const float* gy, int64_t n_rows, float* gx, float* const* gw, float* const* gb, void* ws,
                       int64_t ws_bytes, void* stream);

/* ---- a3/a4/a7/a9: ResidualVectorQuantizer.forward, argmin branch ------------------------
 * (index/models/rq.py:39-56, vq.py:63-75,87-99).  One fused pass over all L levels:
 * d = (|r|^2 + |c|^2) - 2 r.c in fp32, lowest-index argmin, x_res = r + (q - r), r -= x_res.
 * codebooks: L device pointers to (n_codes[l], e_dim) fp32.  Nullable outputs:
 *   codes       (n, L) int64      xq  (n, e_dim) fp32 sum of x_res
 *   resid_last  (n, e_dim) fp32   residual ENTERING level `resid_level` (for the Sinkhorn pass)
 *   sq_err      (L) fp64          sum over rows and dims of (q - r)^2 per level (losses)
 * n_levels_run <= L lets the caller stop before a Sinkhorn level.
 */
int lcrec_rq_quantize(const float* z, int64_t n, int e_dim, int n_levels, const float* const* codebooks,
                      const int32_t* n_codes, int n_levels_run, int resid_level, int64_t* codes,
                      float* xq, float* resid_last, double* sq_err, void* stream);
/* Kernel choice of lcrec_rq_quantize: 0 = never the tensor-core distance path, 1 (default) = tensor cores (CTA-pair
 * tcgen05 GEMM with a distance + argmin epilogue, fp32-accurate split operands) for large codebooks (>= 4096 codes or
 * e_dim >= 128) and, from 4096 rows on, for e_dim 16 / 32 / 64 (code counts multiples of 256 in all cases; other shapes
 * and smaller batches: SIMT kernels), 2 = whenever the shape allows it (cross-checks). */
int lcrec_rq_set_tc_mode(int mode);

/* ---- a9/a11: training-side residual quantiser for GIVEN codes (rq.py:39-56 over vq.py:87-99) -------------------------
 * forward: xq (n, D) = sum of x_res over the levels, diffs (L, n, D) = q_l - r_l per level, codes_t (L, n) = transposed
 * codes, sq_err (L) fp64 = sum |q_l - r_l|^2 (loss_l = (1 + beta) * sq_err_l / (n D)); values identical to the per-level
 * torch ops of the reference.  backward: analytic gradients of (x_q, mean of the level losses) - the straight-through
 * estimator leaves d x_q / d z = I and only level 0's commitment term reaches z:
 *   g_z = g_xq - g_loss / L * beta0 * 2 / (n D) * diffs[0];  g_codebooks[l][k] = g_loss / L * 2 / (n D) * sum of diffs[l]
 * over the rows with code k, added in item order (deterministic).  g_xq (nullable = 0) (n, D); g_loss: ONE fp32 on the
 * device (nullable = 0); g_z / g_codebooks nullable. */
int lcrec_rq_train_forward(const float* z, const int64_t* codes, int64_t n, int e_dim, int n_levels,
                           const float* const* codebooks, float* xq, float* diffs, int64_t* codes_t, double* sq_err,
                           void* stream);
int lcrec_rq_train_backward(const float* diffs, const int64_t* codes_t, int64_t n, int e_dim, int n_levels,
                            const int32_t* n_codes, const float* g_xq, const float* g_loss, double beta0, float* g_z,
                            float* const* g_codebooks, void* stream);

/* ---- a11: clip_grad_norm_(parameters, max_norm) + optimizer.step() for Adam / AdamW (index/trainer.py:49-81, :117-119) -
 * All tensors in two launches.  Pass 1: sum of squares of every gradient (per-CTA partials, fixed order).  Pass 2: every CTA
 * derives coef = min(1, max_norm / (||g|| + 1e-6)) from the partials, then per element (torch.optim semantics, fp32):
 * g *= coef;  AdamW (decoupled = 1): p *= 1 - lr wd;  Adam (0): g += wd p;  m += (g - m)(1 - beta1);
 * v = v beta2 + (1 - beta2) g^2;  p -= lr / (1 - beta1^step) * m / (sqrt(v) / sqrt(1 - beta2^step) + eps).
 * params / grads / exp_avg / exp_avg_sq: HOST arrays of n_tensors device pointers (fp32, contiguous), numel: host array;
 * step >= 1 is the value AFTER this call's increment; max_norm <= 0 skips clipping; write_clipped_grads stores the clipped
 * gradients back (what clip_grad_norm_ leaves in .grad); total_norm_out (nullable, 1 fp32 on the device) = ||g||. */
int64_t lcrec_adam_workspace_bytes(int n_tensors, const int64_t* numel);
int lcrec_adam_clip_step(int n_tensors, float* const* params, float* const* grads, float* const* exp_avg,
                         float* const* exp_avg_sq, const int64_t* numel, double lr, double beta1, double beta2, double eps,
                         double weight_decay, int decoupled, int64_t step, double max_norm, int write_clipped_grads,
                         float* total_norm_out, void* workspace, int64_t workspace_bytes, void* stream);

/* The same update with its three per-step scalars {1 - lr wd, lr / (1 - beta1^t), sqrt(1 - beta2^t)} (lcrec_adam_hyper writes
 * them to HOST memory) read from DEVICE memory: the launches of a training step can be captured ONCE in a CUDA graph and
 * replayed while the schedule of index/trainer.py:83-92,120 advances; the caller refreshes hyper_dev before each replay. */
int lcrec_adam_hyper(double lr, double beta1, double beta2, double weight_decay, int64_t step, float* out3_host);
int lcrec_adam_clip_step_dev(int n_tensors, float* const* params, float* const* grads, float* const* exp_avg,
                             float* const* exp_avg_sq, const int64_t* numel, const float* hyper_dev, double beta1, double beta2,
                             double eps, double weight_decay, int decoupled, double max_norm, int write_clipped_grads,
                             float* total_norm_out, void* workspace, int64_t workspace_bytes, void* stream);

/* SGD / Adagrad / RMSprop of index/trainer.py:62-75 (torch.optim defaults: no momentum, lr_decay 0, alpha 0.99, not centred) with
 * the same fused clipping: kind 1 = SGD (state NULL), 2 = Adagrad (state = `sum`), 3 = RMSprop (state = `square_avg`).
 * g *= coef; g += wd p; SGD: p -= lr g; Adagrad: sum += g^2, p -= lr g / (sqrt(sum) + eps); RMSprop: sq = alpha sq + (1 - alpha) g^2,
 * p -= lr g / (sqrt(sq) + eps).  Workspace: lcrec_adam_workspace_bytes. */
int lcrec_simple_opt_clip_step(int kind, int n_tensors, float* const* params, float* const* grads, float* const* state,
                               const int64_t* numel, double lr, double weight_decay, double alpha, double eps, double max_norm,
                               int write_clipped_grads, float* total_norm_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- a2 (training): BatchNorm1d in training mode + the ReLU behind it (index/models/layers.py:25-29; `run.sh --bn False`
 * parses to bn=True, index/main.py:31) -----------------------------------------------------------------------------------
 * y (n_rows, n_channels) fp32 row-major = the Linear output.  Two launches each way with the per-channel fp64 sums in
 * between, so that a data-parallel job can all-reduce them (synchronised BN = single-device global-batch semantics):
 *   forward_reduce : sums[s][0][c] = sum_rows y, sums[s][1][c] = sum_rows y^2 for s < lcrec_bn_splits(n_rows, n_channels)
 *                    row blocks (sums: lcrec_bn_sums_elems(n_channels) doubles);
 *   forward_apply  : mean, biased variance over n_rows_total (>= n_rows: pass the global count and ONE block of reduced sums
 *                    under DP), out = relu?((y - mean) / sqrt(var + eps) * gamma + beta), save_mean / save_invstd (C) for the
 *                    backward, running_mean / running_var (nullable) <- (1 - momentum) r + momentum stat (unbiased variance),
 *                    exactly torch.nn.BatchNorm1d;
 *   backward_reduce: sums = {sum g, sum g xhat}, g = gy * (out > 0) when relu, xhat = (y - mean) invstd;
 *   backward_apply : g_beta, g_gamma (nullable) and gx (nullable) = gamma invstd (g - g_beta / N - xhat g_gamma / N). */
int64_t lcrec_bn_sums_elems(int n_channels);
int lcrec_bn_splits(int64_t n_rows, int n_channels);
int lcrec_bn_forward_reduce(const float* y, int64_t n_rows, int n_channels, double* sums, void* stream);
int lcrec_bn_forward_apply(const float* y, const double* sums, int n_splits, int64_t n_rows, int64_t n_rows_total,
                           int n_channels, const float* gamma, const float* beta, double eps, double momentum, int relu,
                           float* out, float* save_mean, float* save_invstd, float* running_mean, float* running_var,
                           void* stream);
int lcrec_bn_backward_reduce(const float* y, const float* gy, const float* out, int relu, const float* save_mean,
                             const float* save_invstd, int64_t n_rows, int n_channels, double* sums, void* stream);
int lcrec_bn_backward_apply(const float* y, const float* gy, const float* out, int relu, const double* sums, int n_splits,
                            int64_t n_rows, int64_t n_rows_total, int n_channels, const float* gamma, const float* save_mean,
                            const float* save_invstd, float* gx, float* g_gamma, float* g_beta, void* stream);

/* ---- a10 (training): reconstruction loss of RQVAE.compute_loss (index/models/rqvae.py:74-85) ---------------------------
 * loss (1 fp32, device) = mean over `total` = n * in_dim elements of (out - x)^2 (loss_type 0, F.mse_loss) or |out - x|
 * (1, F.l1_loss); fp64 partial sums in a fixed order.  backward: grad = (*upstream, or 1 when NULL) * d loss / d out. */
int64_t lcrec_recon_loss_workspace_bytes(int64_t total);
int lcrec_recon_loss(const float* out, const float* x, int64_t total, int loss_type, float* loss, void* ws, int64_t ws_bytes,
                     void* stream);
int lcrec_recon_loss_backward(const float* out, const float* x, int64_t total, int loss_type, const float* upstream,
                              float* grad, void* stream);

/* ---- a4: distances only (index/models/vq.py:71-73), (n, K) fp32 ------------------------ */
int lcrec_vq_distances(const float* r, int64_t n, int e_dim, const float* codebook, int n_codes,
                       float* d, void* stream);

/* ---- a5+a6+a7: Sinkhorn assignment -------------------------------------------------------
 * lcrec_sinkhorn_dense: drop-in for sinkhorn_algorithm(distances, epsilon, iters)
 * (index/models/layers.py:85-108) on an fp64 (B, K) matrix; q may alias distances.
 * ws: workspace of lcrec_sinkhorn_workspace_bytes(B, K).  If argmax != NULL also writes
 * torch.argmax(Q, -1) (vq.py:83, lowest index on ties, NaN counts as maximum).
 * flags (nullable, 1 int32): bit0 = NaN/Inf seen in Q (vq.py:81).
 */
int64_t lcrec_sinkhorn_workspace_bytes(int64_t n_rows, int n_codes);
int lcrec_sinkhorn_dense(const double* distances, int64_t n_rows, int n_codes, double epsilon,
                         int iters, double* q, int64_t* argmax, int32_t* flags, void* ws,
                         int64_t ws_bytes, void* stream);
/* center_distance_for_constraint (vq.py:51-61): fp32 in, centred fp64 out (the .double() of
 * vq.py:78).  status (1 int32, device): set to 1 when amplitude <= 0. */
/* sinkhorn_algorithm (layers.py:85-108) on ONE (n_rows_global x n_codes) problem whose rows are split over the ranks
 * of a data-parallel job (the DP form of the training step, trainer.py:114): row steps are local, the initial total
 * and the per-iteration column marginals are summed inside the kernel through peer memory (NVLink P2P on symmetric
 * buffers, rank-ordered sum => identical marginals on all ranks).  peers_dev: device array of `world` pointers to the
 * ranks' symmetric buffers (lcrec_sinkhorn_dist_symmetric_bytes each, zeroed once); epoch = steps published on these
 * buffers so far: 0 for the first call, then EXACTLY the previous call's epoch + its iters + 1 (the double-buffered slots
 * alternate on the absolute step, so consecutive calls may overlap without a barrier in between).  Collective: every rank calls it with its own rows.  Workspace as lcrec_sinkhorn_workspace_bytes. */
/* argmax per row of sinkhorn_algorithm(distances, epsilon, iters) - all that vq.py:83 consumes in the training forward - as ONE
 * thread-block cluster (<= 16 CTAs): exp(-d / eps) in shared memory, column marginals exchanged through distributed shared memory
 * with a cluster barrier per iteration; scaling-vector iterations + the reference's last column step evaluated literally (exact
 * ties as in layers.py:85-108).  Falls back to lcrec_sinkhorn_dense (scratch plan in ws) when the problem does not fit
 * (n_rows / 16 x n_codes doubles > 200 KB), iters == 0, or lcrec_sinkhorn_set_dense_cluster(0). */
int64_t lcrec_sinkhorn_dense_argmax_workspace_bytes(int64_t n_rows, int n_codes);
int lcrec_sinkhorn_dense_argmax(const double* distances, int64_t n_rows, int n_codes, double epsilon, int iters,
                                int64_t* argmax, int32_t* flags, void* ws, int64_t ws_bytes, void* stream);
int lcrec_sinkhorn_set_dense_cluster(int on);
/* Large codebooks (2048 ... 8192 codes per cluster CTA, e.g. BASELINE configs[4]: 8192 x 256) in lcrec_sinkhorn_groups*: 1 (default) =
 * fp32 distances of ALL colliding rows in one register-tiled pass (each output one fma chain in ascending dimension, as everywhere)
 * + one thread-block cluster of 1 / 2 / 4 / 8 CTAs per group of <= 3 / 6 / 12 / 24 rows with exp(-dc / eps) in shared memory and the
 * row sums exchanged through distributed shared memory (register-resident variants for the classes that hold most groups);
 * 0 = the CTA kernel for every group, 2 = the cluster path in the literal divide form, 3 = shared-memory cluster kernels only
 * (cross-checks). */
int lcrec_sinkhorn_set_wide(int on);
int64_t lcrec_sinkhorn_dist_symmetric_bytes(int n_codes);
int lcrec_sinkhorn_dense_dist(const double* distances, int64_t n_rows_local, int64_t n_rows_global, int n_codes,
                              double epsilon, int iters, double* q, int64_t* argmax, int32_t* flags,
                              void* const* peers_dev, int world, int rank, uint64_t epoch, void* ws, int64_t ws_bytes,
                              void* stream);
int lcrec_center_distances(const float* d, int64_t n_rows, int n_codes, double* centred,
                           int32_t* status, void* ws, int64_t ws_bytes, void* stream);

/* lcrec_sinkhorn_groups: one independent Sinkhorn problem per collision group
 * (index/generate_indices.py:116-119 -> vq.py:71-83 on the group's rows).
 * resid: (n_items, e_dim) residuals entering the last level; group g owns rows
 * members[offsets[g] .. offsets[g+1]).  Writes new_code[item] for every member.
 * n_groups_dev: device int64 holding the group count (<= max_groups, the launch bound). */
int64_t lcrec_sinkhorn_groups_workspace_bytes(int64_t max_rows, int n_codes);
/* same, restricted to the groups g with g % part_mod == part_rem, and with an optional bound on the rows of the
 * largest group (max_group_rows, 0 = unknown) that lets the library skip size classes that cannot occur */
int lcrec_sinkhorn_groups_ex(const float* resid, int e_dim, const float* codebook, int n_codes,
                             const int64_t* offsets, const int64_t* members, const int64_t* n_groups_dev,
                             int64_t max_groups, int64_t max_rows, int64_t max_group_rows, double epsilon, int iters,
                             int64_t* codes, int n_levels, int level, int part_mod, int part_rem, int32_t* flags,
                             void* ws, int64_t ws_bytes, void* stream);
int lcrec_sinkhorn_groups(const float* resid, int e_dim, const float* codebook, int n_codes,
                          const int64_t* offsets, const int64_t* members, const int64_t* n_groups_dev,
                          int64_t max_groups, int64_t max_rows, double epsilon, int iters,
                          int64_t* codes, int n_levels, int level, int32_t* flags, void* ws,
                          int64_t ws_bytes, void* stream);

/* Same, restricted to groups g with g % part_mod == part_rem: the multi-GPU split of one round
 * (every rank sees the same CSR, resolves its share, last-level code deltas are all-reduced). */
int lcrec_sinkhorn_groups_part(const float* resid, int e_dim, const float* codebook, int n_codes,
                               const int64_t* offsets, const int64_t* members, const int64_t* n_groups_dev,
                               int64_t max_groups, int64_t max_rows, double epsilon, int iters,
                               int64_t* codes, int n_levels, int level, int part_mod, int part_rem,
                               int32_t* flags, void* ws, int64_t ws_bytes, void* stream);

/* Arithmetic form of the per-group Sinkhorn kernels:
 *   0  the reference's literal in-place divides (layers.py:93-107) for every group: bit-faithful plan;
 *   1  scaling-vector iterations + literal last column step (fastest; ulp-level ties of Q may resolve
 *      differently: 0 of 1.7 M rows on realistic data, ~1e-5 on duplicate-heavy data);
 *   2  (default) filtered: form 1 for groups of <= 8 rows, then every group whose argmax is not provably the
 *      literal kernel's (lead <= 1e-9 relative and not a robust exact tie) is re-run with form 0; larger
 *      groups always use form 0.  Same codes as mode 0 (tested), close to the speed of mode 1. */
int lcrec_sinkhorn_set_mode(int mode);

/* ---- a12/a14: collision bookkeeping (generate_indices.py:18-42, trainer.py:141-150) -----
 * Packs (n, L) int64 codes into u64 keys, radix-sorts (key, item) and emits collision groups
 * in CSR form: groups ordered by key, members ascending (the reference orders groups by
 * first occurrence; groups are disjoint so the order does not change any result).
 * counts (device, 4 int64): [n_unique, n_groups, n_colliding_rows, max_multiplicity].
 */
int64_t lcrec_collisions_workspace_bytes(int64_t n);
int lcrec_collisions(const int64_t* codes, int64_t n, int n_levels, const int32_t* n_codes,
                     int64_t* offsets /* n+1 */, int64_t* members /* n */, int64_t* counts,
                     void* ws, int64_t ws_bytes, void* stream);
/* Prefix segments: runs (>= 2 items) of equal first n_levels-1 codes, same CSR / counts layout as lcrec_collisions.
 * While the collision rounds rewrite the last level only (generate_indices.py:116-119 re-assigns with use_sk on the
 * last level), two items can collide only inside one segment; built once after PASS 0. */
int lcrec_prefix_segments(const int64_t* codes, int64_t n, int n_levels, const int32_t* n_codes,
                          int64_t* seg_offsets /* n+1 */, int64_t* seg_members /* n */, int64_t* counts,
                          void* ws, int64_t ws_bytes, void* stream);
/* Collision groups of codes[:, level] inside those segments (no global sort): same outputs as lcrec_collisions
 * (group order differs; members of a group are in ascending item order).  counts: 8 int64, counts[5] = 1 when a
 * segment was too large for the on-chip sort (> 1024 items): result incomplete, call lcrec_collisions instead. */
int64_t lcrec_segment_collisions_workspace_bytes(int64_t max_segments);
int lcrec_collisions_in_segments(const int64_t* codes, int64_t n, int n_levels, int level,
                                 const int64_t* seg_offsets, const int64_t* seg_members, const int64_t* n_segs_dev,
                                 int64_t max_segments, int64_t* offsets, int64_t* members, int64_t* counts,
                                 void* ws, int64_t ws_bytes, void* stream);
/* same with an explicit active list (device int32 arrays): only the segments named by active_in / n_active_in are
 * examined (NULL = all), the segments that still contain a collision are appended to active_out / n_active_out
 * (NULL = not wanted; *n_active_out must be 0 on entry) - a segment without a collision cannot acquire one later. */
int lcrec_collisions_in_segments_active(const int64_t* codes, int64_t n, int n_levels, int level,
                                        const int64_t* seg_offsets, const int64_t* seg_members,
                                        const int64_t* n_segs_dev, int64_t max_segments, const int32_t* active_in,
                                        const int32_t* n_active_in, int32_t* active_out, int32_t* n_active_out,
                                        int64_t* offsets, int64_t* members, int64_t* counts, void* ws, int64_t ws_bytes,
                                        void* stream);
/* sorted (key, item) pairs only; keys_out/items_out (n) */
int lcrec_sort_codes(const int64_t* codes, int64_t n, int n_levels, const int32_t* n_codes,
                     uint64_t* keys_out, uint32_t* items_out, void* ws, int64_t ws_bytes, void* stream);

/* ---- a15: whole index generation, HOST buffers (index/generate_indices.py:85-128) -------
 * x_host: (n, dims[0]) fp32 in pageable or pinned host memory; codes_host: (n, L) int64.
 * The _ex forms take the embeddings as `const void* x, int dtype` (0 = fp32, 1 = fp16, 2 = bf16, as in
 * lcrec_mlp_forward_ex): half-precision embeddings are read, and for run_host copied to the device, as they are
 * (half the bytes of fp32).  Codes and stats are bit-identical to the fp32 entry run on the input upcast to fp32.
 * dtype outside {0, 1, 2}: LCREC_ERR_ARG, before anything touches the device; half input needs encoder engine 1.
 * Each fp32 entry is its _ex form with dtype 0.
 * Streams the embeddings to the device in chunks, PASS 0 argmin, then up to max_rounds
 * collision rounds with per-group Sinkhorn on the last level.  stats_host (nullable, 8 int64):
 * [rounds_run, n_unique_final, groups_round1, rows_round1, total_sinkhorn_rows, max_multiplicity,
 *  nan_flag, 0].
 */
typedef struct lcrec_indexer lcrec_indexer_t;
int lcrec_indexer_create(lcrec_mlp_t* encoder, int e_dim, int n_levels, const float* const* codebooks,
                         const int32_t* n_codes, double last_epsilon, int sk_iters,
                         int64_t max_items, int64_t chunk_rows, lcrec_indexer_t** out);
int lcrec_indexer_destroy(lcrec_indexer_t* ix);
/* device-resident input */
int lcrec_indexer_run_device(lcrec_indexer_t* ix, const float* x, int64_t n, int max_rounds,
                             int64_t* codes, int64_t* stats_host, void* stream);
/* host-resident input and output */
int lcrec_indexer_run_host(lcrec_indexer_t* ix, const float* x_host, int64_t n, int max_rounds,
                           int64_t* codes_host, int64_t* stats_host, void* stream);
int lcrec_indexer_run_device_ex(lcrec_indexer_t* ix, const void* x, int dtype, int64_t n, int max_rounds,
                                int64_t* codes, int64_t* stats_host, void* stream);
int lcrec_indexer_run_host_ex(lcrec_indexer_t* ix, const void* x_host, int dtype, int64_t n, int max_rounds,
                              int64_t* codes_host, int64_t* stats_host, void* stream);
/* building blocks of the loop, for multi-GPU drivers and tests */
int lcrec_indexer_pass0(lcrec_indexer_t* ix, const float* x, int64_t n, int64_t row_offset, void* stream);
int lcrec_indexer_pass0_ex(lcrec_indexer_t* ix, const void* x, int dtype, int64_t n, int64_t row_offset, void* stream);
int lcrec_indexer_round(lcrec_indexer_t* ix, int64_t n, int64_t* counts_host, void* stream);
/* The collision rounds alone (generate_indices.py:108-128) on caller-owned device arrays: codes (n, L) int64 updated
 * in place, resid (n, e_dim) = residual entering the last level; n <= max_items.  stats_host as in run_host. */
int lcrec_indexer_resolve(lcrec_indexer_t* ix, int64_t* codes, const float* resid, int64_t n, int max_rounds,
                          int64_t* stats_host, void* stream);
/* 1 (default): from the second round on, collisions are searched inside the prefix segments (no global re-sort);
 * 0: every round re-sorts all items.  Results are identical; process-wide switch for cross-checks. */
int lcrec_indexer_set_segments(int on);
/* Later rounds of generate_indices.py:108-128 without a host read per round.  Once the first check inside the prefix segments has
 * passed, a round can be enqueued blind (check -> Sinkhorn with worst-case launch bounds, group counts read on the device):
 * 0 = one host read of the counts per round; 1 = every remaining round enqueued blind on the caller's stream (measured no faster:
 * the host's launch rate becomes the bound); 2 (default) = as soon as a round has <= 888 groups the blind round is captured once
 * into a CUDA graph and the remaining rounds are graph replays in batches of 6 with one host read per batch.  Results and stats
 * are identical (tests/test_gpu_loop_ledger.py).  Applies to last-level codebooks of <= 256 codes; process-wide switch. */
int lcrec_indexer_set_speculative(int on);
int64_t* lcrec_indexer_codes(lcrec_indexer_t* ix);      /* (max_items, L) int64 device */
float* lcrec_indexer_resid(lcrec_indexer_t* ix);        /* (max_items, e_dim) fp32 device */
/* ---- f1: k-means codebook initialisation (index/models/layers.py:69-82 -> sklearn.cluster.KMeans(n_clusters,
 * max_iter).fit; scikit-learn `_kmeans_single_lloyd`) ------------------------------------------------------------------
 * The k-means++ seeding stays with scikit-learn on the host (it consumes numpy's global RNG like the reference); the
 * Lloyd iterations run here with sklearn's structure (centred data, lowest-index nearest centre, per-cluster sums in item
 * order times the reciprocal count, empty clusters take the farthest points, stop on unchanged labels or on a total
 * squared centre shift <= tol, final E-step if the stop was not strict).
 * lcrec_kmeans_center: xc = x - column means (n, e_dim); mean (e_dim) device; *mean_variance_host = mean of the column
 * variances (sklearn's tol is 1e-4 times that).  lcrec_kmeans_lloyd: centers (n_codes, e_dim) holds the seeds on entry (in
 * the centred frame) and the result on exit, `add_mean` (nullable) is added at the end; labels_out (nullable, n int64),
 * *inertia_host, *n_iter_host as KMeans.inertia_ / n_iter_.  Synchronises the stream once per iteration (24 bytes D2H). */
int64_t lcrec_kmeans_workspace_bytes(int64_t n, int e_dim, int n_codes);
int lcrec_kmeans_center(const float* x, int64_t n, int e_dim, float* xc, float* mean, double* mean_variance_host,
                        void* workspace, int64_t workspace_bytes, void* stream);
int lcrec_kmeans_lloyd(const float* xc, int64_t n, int e_dim, float* centers, int n_codes, int max_iter, double tol,
                       const float* add_mean, int64_t* labels_out, double* inertia_host, int* n_iter_host,
                       void* workspace, int64_t workspace_bytes, void* stream);
/* k-means++ seeding with scikit-learn's arithmetic from random numbers drawn up front (sklearn `_kmeans_plusplus`: one
 * uniform for the first centre - the caller turns it into first_index exactly like RandomState.choice - then n_trials =
 * 2 + int(log(K)) uniforms per further centre; `draws` is a DEVICE array of (n_clusters - 1) x n_trials doubles in drawing
 * order).  xc: centred rows (n, e_dim); indices (n_clusters int64, device) receives the chosen rows, centers (nullable)
 * their vectors.  No host read inside: three launches per centre are enqueued back to back.
 * NOT YET RUN ON HARDWARE in round 1 (restated and pinned on the CPU: oracle.kmeanspp_predrawn). */
int64_t lcrec_kmeanspp_workspace_bytes(int64_t n, int n_trials);
int lcrec_kmeanspp_seed(const float* xc, int64_t n, int e_dim, int n_clusters, int64_t first_index, const double* draws,
                        int n_trials, int64_t* indices, float* centers, void* workspace, int64_t workspace_bytes,
                        void* stream);
/* ---- f3: EMA codebook variant (index_improve/models/vq.py) ----------------------------------
 * lcrec_ema_update: the `self.training and use_ema` block of the improved VectorQuantizer.forward
 * (index_improve/models/vq.py:146-187) in place on the module's buffers: per-code counts of `indices` (n,) int64,
 * cluster_size (K,) <- cluster_size * decay + (1 - decay) * counts, the per-code sums of latent (n, e_dim) in ascending
 * item order (= CPU index_add_, bit-reproducible, no atomics), ema_w (K, e_dim) <- ema_w * decay + (1 - decay) * sums,
 * and for codes with cluster_size > epsilon: codebook <- codebook * (1 - r) + ema_w / (cluster_size + epsilon) * r,
 * r = 1 - decay.  Scalars are rounded to fp32 where the reference's Python doubles meet fp32 tensors.  n < 2^31.
 * lcrec_codebook_usage: get_codebook_usage (vq.py:205-217) and the dead-code test of _reset_unused_codes
 * (vq.py:83-87): used_codes (1 int64, device) = #{cs / (sum cs + epsilon) > reset_threshold}; unused_mask (nullable,
 * K bytes) = usage < reset_threshold.  The replacement vectors of a reset are drawn by the caller (torch RNG). */
int lcrec_ema_update(const float* latent, const int64_t* indices, int64_t n, int n_codes, int e_dim,
                     double ema_decay, double epsilon, float* cluster_size, float* ema_w, float* codebook,
                     void* stream);
int lcrec_codebook_usage(const float* cluster_size, int n_codes, double epsilon, double reset_threshold,
                         int64_t* used_codes, uint8_t* unused_mask, void* stream);
/* ---- f4: embedding producer hand-off (data_process/amazon_text_emb.py:91-96) -----------------
 * Masked mean pool of a PLM's last hidden state: pooled[b] = sum_t mask[b][t] * hidden[b][t][:] / sum_t mask[b][t]
 * (hidden (n_seq, seq_len, hidden_dim) of dtype 0 = fp32, 1 = fp16, 2 = bf16, row-major; mask (n_seq, seq_len) int64 as
 * the tokenizer returns it; accumulation and result in fp32).  out[b * out_stride + c] = (accumulate ? out : 0) + pooled,
 * then / divide_by if divide_by > 0: the mean over an item's text fields (:96) is `accumulate` on every field after the
 * first and divide_by = n_fields on the last.  `out` may be rows of the (N, in_dim) fp32 embedding matrix that
 * lcrec_indexer_run_device reads - no .npy round trip.  Padded positions are not read.  workspace: partial sums when a
 * small batch is split along the sequence (lcrec_masked_mean_pool_workspace_bytes). */
int64_t lcrec_masked_mean_pool_workspace_bytes(int64_t n_seq, int64_t seq_len, int hidden_dim);
int lcrec_masked_mean_pool(const void* hidden, int dtype, const int64_t* mask, int64_t n_seq, int64_t seq_len,
                           int hidden_dim, float* out, int64_t out_stride, int accumulate, double divide_by,
                           void* workspace, int64_t workspace_bytes, void* stream);
/* ---- a16 / f2: `.index.json` text on the device (index/generate_indices.py:83,138-145) -------------------------------
 * The bytes json.dump({item: ["<a_%d>", "<b_%d>", ...]}) writes (int keys as strings, separators ", " and ": "), formatted
 * from the code table in HBM: out (device, out_cap bytes; NULL for a sizing call), total_bytes_dev (1 int64, device) = the
 * exact length; nothing is written past out_cap.  n_levels <= 5 (the reference's prefix list). */
int64_t lcrec_index_json_workspace_bytes(int64_t n);
int lcrec_index_json(const int64_t* codes, int64_t n, int n_levels, char* out, int64_t out_cap, int64_t* total_bytes_dev,
                     void* ws, int64_t ws_bytes, void* stream);
/* ---- (e) multi-GPU hand-over of PASS-0 results to the owners of the prefix buckets (lcrec_b200/distributed.py) -----------
 * pack: owner = hash(first L-1 codes) mod world; STABLE partition of this rank's n items by owner straight into `send` =
 * `world` slabs of lcrec_exchange_slab_bytes(slab_rows, L, D) bytes: [16 B header: int64 row count, int64 overflow flag][records:
 * L int64 codes + D fp32 residual, lcrec_exchange_record_bytes each]; slot[i] = owner * slab_rows + position (-1: slab overflow).
 * ONE equal-split all-to-all moves the slabs.  unpack: received slabs -> (rows x L) codes + (rows x D) residuals in source-rank
 * order (= ascending global item id for contiguous shards).  pack_last / scatter_last: the resolved last-level codes travel back
 * in (world x slab_rows) int64 slabs along the same routes and land in the origin's table through slot[]. */
int64_t lcrec_exchange_record_bytes(int n_levels, int e_dim);
int64_t lcrec_exchange_slab_bytes(int64_t slab_rows, int n_levels, int e_dim);
int64_t lcrec_exchange_workspace_bytes(int64_t n, int world);
int lcrec_exchange_pack(const int64_t* codes, const float* resid, int64_t n, int n_levels, int e_dim, const int32_t* n_codes,
                        int world, int64_t slab_rows, void* send, int32_t* slot, int64_t* counts_dev, void* ws, int64_t ws_bytes,
                        void* stream);
int lcrec_exchange_unpack(const void* recv, int world, int64_t slab_rows, int n_levels, int e_dim, int64_t* codes, float* resid,
                          int64_t cap_rows, void* stream);
int lcrec_exchange_pack_last(const int64_t* codes, int n_levels, const void* recv, int world, int64_t slab_rows, int e_dim,
                             int64_t* back, int64_t n_rows_hint, void* stream);
int lcrec_exchange_scatter_last(const int64_t* back_recv, const int32_t* slot, int64_t n, int n_levels, int64_t* codes, void* stream);
/* A/B switch for codebooks of <= 256 codes: 0 = collision groups of 9..32 rows run on the shared-memory CTA kernel as in round 1,
 * 1 = on the column kernels (one thread per code, kernel matrix in registers), 2 (default) = additionally every group of a call
 * with few (<= 888) groups - the late collision rounds, bound by the latency of one group.  Results are identical. */
int lcrec_sinkhorn_set_col(int on);
/* Self-check of the shared-reciprocal IEEE division of the per-group Sinkhorn kernels (its last column step divides every row
 * of a column by the same sum): counts[0] += pairs (a[i], b[i]) whose quotient differs from the device's IEEE a / b although
 * the range check of the fast sequence passed (must stay 0), counts[1] += pairs the range check sends to the fallback.
 * counts: 2 x u64 on the device, accumulated (zero them first). */
int lcrec_ddiv_probe(const double* a, const double* b, int64_t n, uint64_t* counts, void* stream);
/* Measured fp64 FMA peak of the device in FLOP/s (8 independent DFMA chains per thread, 148 x 8 CTAs): the denominator of the
 * fp64-pipe fraction bench.py reports for the per-group Sinkhorn (MEASURED_PEAKS.json carries no fp64 figure).  ws: >= 8 B x SMs x 2048.
 * Synchronises the stream. */
int lcrec_fp64_peak_probe(double* flops_out, void* ws, int64_t ws_bytes, void* stream);
/* Per-stage device timing with CUDA events on the launching stream (bench.py's live roofline).
 * Tags: 0 = operand split of the input, 1+l = MLP layer l, 17 = splits of the tail layers, 20 = fused RQ,
 * 21 = collision checks, 22 / 23 = per-group Sinkhorn of the first / the later rounds.  collect() synchronises and ADDS elapsed ms / call counts (32 each). */
int lcrec_profile_enable(int on);
int lcrec_profile_collect(double* ms, int64_t* calls);
/* number of kernels this library has launched on the calling process so far */
int64_t lcrec_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* LCREC_B200_H */
