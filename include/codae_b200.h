/*
 * codae_b200.h -- C ABI of libcodae_b200.so: the B200 (sm_100a) implementation of CODAE's
 * data-parallel hot path (denoising-autoencoder training step + complementarity inference).
 *
 * The reference (victordeleau/MUI-DeepAutoEncoder) is pure Python on stock PyTorch: it has no FFI.
 * Its "plugin boundary" for this path is the set of library calls its Python makes on device
 * tensors.  Each entry point below names the reference call site (paths relative to the reference
 * root) whose device work it replaces.  INTEGRATION.md shows the ctypes stub a maintainer adds.
 *
 * Conventions
 *   - every pointer is a raw DEVICE pointer borrowed from the caller (PyTorch allocations); the
 *     library never frees or keeps them.  `stream` is a cudaStream_t passed as void*.
 *   - all matrices are row-major; `ld*` is the row pitch in ELEMENTS.  Tensor-core paths need
 *     pitches that are multiples of 16 bytes (the caller pads; see *_EINVAL).
 *   - every call is asynchronous on `stream`, allocates nothing and never synchronises the host,
 *     so a whole training step can be captured into a CUDA graph.
 *   - return value: 0 or a negative CODAE_E* code; text via codae_last_error().  Nothing aborts,
 *     nothing throws, and there is no CPU or non-sm_100 fallback (CODAE_EARCH instead).
 *   - reductions use fixed trees: results are bitwise reproducible run to run for fixed shapes.
 */
#ifndef CODAE_B200_H
#define CODAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CODAE_VERSION 100 /* 0.1.0 */

typedef struct codae_ctx codae_ctx;

enum codae_status { CODAE_OK = 0, CODAE_EINVAL = -1, CODAE_EARCH = -2, CODAE_ECUDA = -3, CODAE_ENOMEM = -4 };
/* CODAE_F32X3: an fp32 tensor held as THREE bf16 planes (hi, mid, lo; x = hi + mid + lo to 2^-24 |x|), plane p at
 * base + p * plane_stride elements.  The operand format of the fp32-parity tensor-core engine (codae_linear_*_x3). */
enum codae_dtype { CODAE_F32 = 0, CODAE_BF16 = 1, CODAE_F32X3 = 2 };
enum codae_act { CODAE_ACT_NONE = 0, CODAE_ACT_RELU = 1 };
enum codae_metric { CODAE_METRIC_SQERR = 0, CODAE_METRIC_COSINE = 1 };
enum codae_vartype { CODAE_VAR_REGRESSION = 0, CODAE_VAR_CLASSIFICATION = 1 };
/* GEMM engines (a shape/dtype specialisation chosen by the library, reported for tests/bench) */
enum codae_engine { CODAE_ENGINE_SIMT_F32 = 0, CODAE_ENGINE_TCGEN05_BF16 = 1, CODAE_ENGINE_TCGEN05_F32X3 = 2 };

/* ---- context ------------------------------------------------------------------------------ */
int codae_version(void);
/* Binds to `device`; fails with CODAE_EARCH unless it is compute capability 10.x. */
int codae_ctx_create(int device, codae_ctx** out);
int codae_ctx_destroy(codae_ctx* ctx);
const char* codae_last_error(const codae_ctx* ctx); /* ctx may be NULL: last process-wide error */
int codae_ctx_sm_count(const codae_ctx* ctx);
/* Tuning switches, on by default unless noted (tests flip them to compare code paths):
 *   CODAE_OPT_SPLITK  contractions with too few output tiles to occupy the GPU (the small-batch layers of
 *                     embedding.yaml / modanet) spread their k-blocks over a thread-block cluster and reduce the partial
 *                     tiles through distributed shared memory, in rank order (bitwise reproducible);
 *   CODAE_OPT_PDL     training-step kernels are launched as programmatic dependents: their prologue overlaps the tail
 *                     of the previous kernel and they wait (griddepcontrol.wait) before touching global memory;
 *   CODAE_OPT_PERSISTENT  contractions with more than 2 output tiles per SM run one persistent CTA per SM with the
 *                     accumulator double-buffered in TMEM, so a tile's epilogue overlaps the next tile's MMAs;
 *   CODAE_OPT_WEIGHT_PREFETCH  (needs CODAE_OPT_PDL) codae_linear_fwd / codae_linear_dgrad on the tensor-core engine request
 *                     the TMA loads of their WEIGHT tiles before griddepcontrol.wait, i.e. while the stream predecessors
 *                     that produce the activations are still finishing.  Sound because every entry point that writes
 *                     weights (codae_adam_step, codae_clip_adam_step, codae_cast_bf16) makes the next launch on its stream
 *                     a full (non-programmatic) dependency.  A caller that writes the bf16 weight buffer with kernels of
 *                     its own must either switch this off or call codae_cast_bf16 / an optimizer entry point afterwards.
 *   CODAE_OPT_TMA_STORE  single-pass f32 output tiles of the tensor-core engine (the weight gradients of the small-batch
 *                     step) are staged in shared memory in the 128-byte-swizzle layout and leave through
 *                     cp.async.bulk.tensor stores instead of per-thread 128-bit stores (the N & 3 tail columns of a row
 *                     are stored by the threads: TMA clips ragged row ends at 16-byte granularity).  Same values, bit for
 *                     bit; measured 98.8 -> 64.2 us for the ten weight gradients of the embedding.yaml step.
 *   CODAE_OPT_TMA_STORE_PERSISTENT  (default on: 7.155 -> 6.970 ms/step at 10 x 4096^2, B = 8192) the same for the persistent kernel
 *                     of the large contractions: every epilogue warp stages 32 rows x 128 bytes per store in one of two
 *                     boxes of its own and issues the bulk store itself (f32 and bf16 outputs, all fused epilogues).
 *   CODAE_OPT_CTA_PAIR  (default on) 256-wide persistent contractions run as CTA PAIRS: a cluster of two CTAs on one TPC works
 *                     on a 256 x 256 tile with tcgen05.mma.cta_group::2 (M = 256) -- each CTA stages its own 128 rows of A and
 *                     only HALF of B (32 KB instead of 48 KB of shared-memory traffic per k-block, six ring slots instead of
 *                     four), the leader issues the MMAs, each CTA drains its own half of the accumulator.  Same k order per
 *                     output element, bit-identical results; measured on a B200 at M = 8192, 4096 x 4096: fwd 1443 -> 1645,
 *                     dgrad 1364 -> 1569, wgrad 1215 -> 1406 TFLOP/s; polyvore-shaped step 7.55 -> 6.60-6.75 ms. */
enum codae_option { CODAE_OPT_SPLITK = 0, CODAE_OPT_PDL = 1, CODAE_OPT_PERSISTENT = 2, CODAE_OPT_WEIGHT_PREFETCH = 3,
                    CODAE_OPT_TMA_STORE = 4, CODAE_OPT_TMA_STORE_PERSISTENT = 5, CODAE_OPT_CTA_PAIR = 6 };
int codae_ctx_set_option(codae_ctx* ctx, int option, int value);
/* Tells the library that `stream` has just been made to wait (event / stream wait) for work on ANOTHER stream that writes
 * layer weights -- e.g. an optimizer launch on a side stream.  The next launch on `stream` is then issued with a full stream
 * dependency instead of a programmatic one, so that its weight-tile prefetch (CODAE_OPT_WEIGHT_PREFETCH) cannot run ahead of
 * that wait.  Weight writers on the SAME stream are tracked by the library itself. */
int codae_weights_written(codae_ctx* ctx, void* stream);
/* Current value (0 / 1) of a tuning switch, CODAE_EINVAL for an unknown option. */
int codae_ctx_get_option(const codae_ctx* ctx, int option);
/* Which engine codae_linear_* will use for (dtype, M, N, K). */
int codae_linear_engine(const codae_ctx* ctx, int dtype, int M, int N, int K);

/* ---- K1: corruption ------------------------------------------------------------------------ */
/* Replaces the un-seeded `random.sample` draw of Corrupter.mask_to_use
 * (codae/tool/data_tool.py:222-226) by a Philox4x32-10 stream: out[i, :] (int16 [n_obs, nb_run]) is a
 * permutation of range(nb_run) that depends only on (seed, first_obs + i).  nb_run <= 1024. */
int codae_mask_table_philox(codae_ctx* ctx, uint64_t seed, int64_t first_obs, int64_t n_obs, int nb_run,
                            int16_t* out, void* stream);

/* Fused batch gather + slot-mask corruption.  Replaces collate_embedding's torch.stack
 * (codae/tool/data_tool.py:96-103), Corrupter.get_masks (data_tool.py:239-262) and model.corrupt
 * (codae/model/embedding_denoising_autoencoder.py:226-239).
 *   data      [n_rows, ld_data] f32   resident dataset (ConcatenatedEmbeddingDataset.data)
 *   batch_idx [B] int64 or NULL       observation ids (NULL: observations 0..B-1); an id outside [0, n_rows) traps the kernel
 *                                     (launch failure) rather than gathering foreign memory -- the reference raises IndexError
 *   mask_table[n_rows, nb_run] int16  mask id of (observation, run)
 *   mask_bits [nb_run] u64            bit v set <=> variable v is zeroed by that mask (V <= 64)
 *   col_var   [io] u8                 variable index of every column
 *   out_cx    [B, ld_cx] f32|bf16     x * mask (a multiply: -0.0 / NaN propagate like the reference)
 *   out_x     [B, ld_x] f32 or NULL   gathered clean rows
 *   out_mask_id [B] int32 or NULL     mask id applied to every row                              */
int codae_corrupt_fwd(codae_ctx* ctx, const float* data, int64_t n_rows, int64_t ld_data, const int64_t* batch_idx, int B,
                      const int16_t* mask_table, int nb_run, int run, const uint64_t* mask_bits,
                      const uint8_t* col_var, int io, void* out_cx, int cx_dtype, int64_t ld_cx, float* out_x,
                      int64_t ld_x, int32_t* out_mask_id, void* stream);

/* Dense masks for the legacy API: Corrupter.get_masks (data_tool.py:239-262).
 *   out_masks [k_max, B, io] f32 (row i of plane k-1 holds the mask iff its subset has k variables)
 *   out_fmask [B, io] f32 = sum over k.  nb_missing [nb_run] u8.                                */
int codae_dense_masks(codae_ctx* ctx, const int64_t* batch_idx, int B, const int16_t* mask_table, int nb_run,
                      int run, const uint64_t* mask_bits, const uint8_t* nb_missing, const uint8_t* col_var, int io,
                      int k_max, float* out_masks, float* out_fmask, void* stream);

/* out = x * mask, elementwise over n floats: model.corrupt for caller-supplied dense masks
 * (embedding_denoising_autoencoder.py:239, mixed_variable_denoising_autoencoder.py:262). */
int codae_mul_mask(codae_ctx* ctx, const float* x, const float* mask, float* out, int64_t n, void* stream);

/* ---- K1-loss: reconstruction loss, its gradient and the monitors ------------------------------ */
/* MSELoss("mean")(x, y) forward + backward and the host-side monitor sums, in one pass.
 * Replaces script/train_dae_on_embedding.py:206 (loss), :210 (first backward node) and
 * :217-223 (full / partial error sums, there computed on the host after two D2H copies).
 *   x        clean rows: x[i, :] = data[batch_idx ? batch_idx[i] : i, :]   (f32, pitch ld_x)
 *   y        [B, ld_y] f32|bf16 reconstructions
 *   mask_id  [B] int32 (from codae_corrupt_fwd); mask_bits/col_var as above
 *   dy       [B, ld_dy] f32|bf16 or NULL:  grad_scale * (y - x)   (grad_scale = 2 / (B_global * io))
 *   acc      double[4]:  acc[0] += sum (x-y)^2 ; acc[1] += sum (1-m)(x-y)^2 ; acc[2] += B ;
 *                        acc[3]  = this call's sum (x-y)^2  (loss = acc[3] / (B*io))
 *   workspace >= codae_loss_workspace_bytes()                                                     */
size_t codae_loss_workspace_bytes(const codae_ctx* ctx);
int codae_mse_loss_fwd_bwd(codae_ctx* ctx, const float* x, int64_t ld_x, const int64_t* batch_idx, const void* y,
                           int y_dtype, int64_t ld_y, const int32_t* mask_id, const uint64_t* mask_bits,
                           const uint8_t* col_var, int B, int io, float grad_scale, void* dy, int dy_dtype,
                           int64_t ld_dy, double* acc, void* workspace, size_t ws_bytes, void* stream);

/* CombinedCriterion(reduction="mean") forward + backward (codae/tool/metering.py:155-180;
 * script/train_dae_on_abalone.py:215,219).  Per-variable RMSE over the batch / softmax-NLL, weighted.
 *   var_pos/var_size/var_type [V] int32 ; weight [V] f32 ; x,y [B, ld] f32 ; dy [B, ld] f32
 *   loss_out: float[1 + V] = {loss, l_0 .. l_{V-1}}.  Single-CTA kernel: meant for tabular widths. */
int codae_mixed_loss_fwd_bwd(codae_ctx* ctx, const float* x, const float* y, int B, int io, int64_t ld, int V,
                             const int32_t* var_pos, const int32_t* var_size, const int32_t* var_type,
                             const float* weight, float* dy, float* loss_out, void* stream);

/* Monitor pass of the abalone loop (train_dae_on_abalone.py:227-236): Normalizer.undo on columns
 * [norm_first, io) (data_tool.py:80-90), CombinedCriterion(reduction="none") (metering.py:131-152),
 * get_per_k / get_partial (metering.py:187-204), accumulated on the device.
 *   out_loss [B, V] f32 (required; the as_numpy matrix, also the kernel's staging buffer)
 *   acc double[2 + 2*k_max*V]: {ftl, ptl, ftl_per_k[k_max][V], ptl_per_k[k_max][V]}  (+=)            */
int codae_mixed_monitor(codae_ctx* ctx, const float* x, const float* y, int B, int io, int64_t ld, int V,
                        const int32_t* var_pos, const int32_t* var_size, const int32_t* var_type,
                        const float* norm_scale, const float* norm_min, int norm_first, const int32_t* mask_id,
                        const uint64_t* mask_bits, const uint8_t* nb_missing, int k_max, float* out_loss, double* acc,
                        void* stream);

/* ---- K2: encoder / decoder contractions ------------------------------------------------------- */
/* dtype = CODAE_F32 : operands and outputs f32 (exact-fp32 engine).
 * dtype = CODAE_BF16: X, W, dY bf16 operands, fp32 accumulation on tcgen05 tensor cores; the output type
 *                     is `out_dtype`.  M = batch rows, N = out features, K = in features.
 * Y[M,N] = act(X[M,K] . W[N,K]^T + bias[N])      nn.Linear forward + ReLU(inplace)
 *                                                (embedding_denoising_autoencoder.py:63-129,166,183)   */
int codae_linear_fwd(codae_ctx* ctx, const void* X, int64_t ldx, const void* W, int64_t ldw, const float* bias,
                     void* Y, int64_t ldy, int M, int N, int K, int act, int dtype, int out_dtype, void* stream);
/* dX[M,K] = (dY[M,N] . W[N,K]) * (A_prev > 0 ? 1 : 0)   autograd's mm + threshold_backward for loss.backward()
 * (train_dae_on_embedding.py:210).  A_prev [M,K] = this layer's input (post-ReLU output of the previous
 * layer), same dtype as the operands, or NULL when the previous layer has no ReLU.                       */
int codae_linear_dgrad(codae_ctx* ctx, const void* dY, int64_t lddy, const void* W, int64_t ldw, const void* A_prev,
                       int64_t lda, void* dX, int64_t lddx, int M, int N, int K, int dtype, int out_dtype,
                       void* stream);
/* dW[N,K] = dY[M,N]^T . X[M,K]  (f32 out, pitch lddw) and db[N] = column sums of dY (f32).
 * The weight/bias gradient of nn.Linear in loss.backward().                                           */
int codae_linear_wgrad(codae_ctx* ctx, const void* dY, int64_t lddy, const void* X, int64_t ldx, float* dW,
                       int64_t lddw, float* db, int M, int N, int K, int dtype, void* stream);
/* codae_linear_wgrad on the tensor-core engine that also leaves sum(dW^2) behind, so that clip_grad_norm_
 * (train_dae_on_embedding.py:212-213) needs no pass of its own over the gradients on a single GPU: every CTA of the
 * launch writes the sum of squares of the gradient elements it stored into sq_partials[cta] (double, fixed reduction
 * tree).  n_slots must equal codae_linear_wgrad_sq_slots(ctx, M, N, K, dtype) -- the number of CTAs the launch has under
 * the context's current options; 0 means the engine for that shape cannot do it (use codae_linear_wgrad and
 * codae_clip_adam_step).  The bias gradient is the constant-1 column of the augmented contraction (no db argument).
 * Consumer: codae_adam_step_partials. */
int codae_linear_wgrad_sq_slots(const codae_ctx* ctx, int M, int N, int K, int dtype);
int codae_linear_wgrad_sq(codae_ctx* ctx, const void* dY, int64_t lddy, const void* X, int64_t ldx, float* dW,
                          int64_t lddw, int M, int N, int K, int dtype, double* sq_partials, int n_slots,
                          void* stream);
/* The same three contractions at the REFERENCE'S precision (fp32, config/embedding.yaml has no dtype) on the tensor cores:
 * every operand is a CODAE_F32X3 triple of bf16 planes and each k-step issues six tcgen05 MMAs (hi.hi | hi.mid, mid.hi, mid.mid,
 * hi.lo, lo.hi) into two fp32 TMEM accumulators that the epilogue adds -- products are exact, accumulation is fp32, the
 * dropped terms and the representation error are 2^-24: results track torch's fp32 nn.Linear to fp32 rounding (1e-5 gate in
 * tests/test_gpu_f32x3.py), where the bf16 engine is a 1e-2 mode.  Same shapes / pitches / epilogues as codae_linear_fwd,
 * _dgrad, _wgrad[_sq]; *_plane = elements between planes (multiple of 8).  out_dtype: CODAE_F32 (the last layer: the loss reads
 * fp32) or CODAE_F32X3 (the next contraction's operand).  A_prev_hi = plane 0 of this layer's input (x > 0 <=> hi > 0).
 * sq_partials may be NULL (n_slots ignored); otherwise as codae_linear_wgrad_sq with dtype CODAE_F32X3 for the slot count. */
int codae_linear_fwd_x3(codae_ctx* ctx, const void* X, int64_t ldx, int64_t x_plane, const void* W, int64_t ldw, int64_t w_plane,
                        void* Y, int64_t ldy, int64_t y_plane, int M, int N, int K, int act, int out_dtype, void* stream);
int codae_linear_dgrad_x3(codae_ctx* ctx, const void* dY, int64_t lddy, int64_t dy_plane, const void* W, int64_t ldw,
                          int64_t w_plane, const void* A_prev_hi, int64_t lda, void* dX, int64_t lddx, int64_t dx_plane, int M,
                          int N, int K, int out_dtype, void* stream);
int codae_linear_wgrad_x3(codae_ctx* ctx, const void* dY, int64_t lddy, int64_t dy_plane, const void* X, int64_t ldx,
                          int64_t x_plane, float* dW, int64_t lddw, int M, int N, int K, double* sq_partials, int n_slots,
                          void* stream);
/* f32 -> CODAE_F32X3 planes of n elements (weight shadow of the fp32-parity engine, activation / gradient split of the legacy
 * autograd path); n and plane_stride multiples of 4. */
int codae_split_x3(codae_ctx* ctx, const float* src, void* dst, int64_t n, int64_t plane_stride, void* stream);
/* Tabular widths (abalone: Linear layers of at most 11 x 11): the WHOLE network in one launch, exact fp32 FMA arithmetic.
 * Replaces the per-layer codae_linear_fwd / codae_linear_dgrad / codae_linear_wgrad launches of
 * MixedVariableDenoisingAutoencoder.forward (codae/model/mixed_variable_denoising_autoencoder.py:133-181) and of
 * loss.backward() (script/train_dae_on_abalone.py:219).  Parameters and gradients use the augmented flat layout (layer l:
 * W'[out, ld] at w_off, bias in column bcol; activations [B, ld_act] carry the constant-1 column):
 *   fwd: acts[l+1][r, o] = act_l(sum_{k <= bcol} acts[l][r, k] W'_l[o, k])                      acts: L+1 device pointers (host array)
 *   bwd: dW'_l[o, k] = sum_r g_l[r, o] acts[l][r, k] ;  g_{l-1}[r, k] = (sum_o g_l[r, o] W'_l[o, k]) * (acts[l][r, k] > 0 if ReLU
 *        follows layer l-1), with g_l in g3[l % 3] ([B, ld_g] f32; g3[(L-1) % 3] holds dL/dy on entry)
 * Default for tabular widths (FusedStep(tiny_mlp=None)): parity-checked on a B200 against the reference's abalone goldens
 * (tests/test_gpu_variants.py); the arithmetic (csrc/tiny_mlp.h) is also unit-tested on the CPU. */
typedef struct codae_tiny_layer {
    int64_t w_off;
    int32_t ld, bcol, in, out, relu;
} codae_tiny_layer;
int codae_tiny_mlp_fwd(codae_ctx* ctx, const codae_tiny_layer* layers, int n_layers, const float* flat, float* const* acts,
                       int64_t ld_act, int B, void* stream);
int codae_tiny_mlp_bwd(codae_ctx* ctx, const codae_tiny_layer* layers, int n_layers, const float* flat, float* gflat,
                       float* const* acts, int64_t ld_act, float* const* g3, int64_t ld_g, int B, void* stream);
/* f32 -> bf16 copy of n elements (weight shadow / activation cast). */
int codae_cast_bf16(codae_ctx* ctx, const float* src, void* dst, int64_t n, void* stream);

/* ---- K4: clip_grad_norm_ + Adam over flat buffers ----------------------------------------------- */
/* out_sqnorm (f32[1]) = sum g^2 over the flat gradient buffer: clip_grad_norm_(params, 1)
 * (train_dae_on_embedding.py:212-213).  workspace >= codae_sqnorm_workspace_bytes().          */
size_t codae_sqnorm_workspace_bytes(const codae_ctx* ctx);
int codae_grad_sqnorm(codae_ctx* ctx, const float* g, int64_t n, float* out_sqnorm, void* workspace,
                      size_t ws_bytes, void* stream);
/* torch.optim.Adam(lr, weight_decay).step() with the clip scale folded in (train_dae_on_embedding.py:
 * 160-163,215).  g_eff = g * grad_scale * min(1, max_norm / (sqrt(sqnorm)*grad_scale + 1e-6));
 * g_eff += wd*p ; m = lerp(m, g_eff, 1-b1) ; v = b2*v + (1-b2) g_eff^2 ;
 * p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps).
 *   max_norm < 0 or sqnorm == NULL: no clipping.  p_shadow (or NULL): the copy of p the tensor-core GEMMs read, rewritten
 *   with the update -- shadow_dtype CODAE_BF16: bf16 [n]; CODAE_F32X3: three bf16 planes [3][n] (fp32-parity engine).
 *   Hyper-parameters are doubles: the bias corrections are derived in double like torch's Python code,
 *   then rounded to f32 once.  `step` is 1-based; step_dev (device int32, or NULL) overrides it so that a
 *   captured CUDA graph can advance the step count without new scalar arguments.                       */
int codae_adam_step(codae_ctx* ctx, float* p, const float* g, float* m, float* v, void* p_shadow, int shadow_dtype, int64_t n,
                    double lr, double beta1, double beta2, double eps, double weight_decay, int step, double max_norm,
                    const float* sqnorm, double grad_scale, const int32_t* step_dev, void* stream);
/* codae_grad_sqnorm + codae_adam_step in ONE cooperative launch (grid barrier between the norm and the update): same
 * arithmetic and argument meaning; sqnorm_out (f32[1]) receives sum g^2.  max_norm < 0 computes the norm but does not clip.
 * workspace >= codae_sqnorm_workspace_bytes(). */
int codae_clip_adam_step(codae_ctx* ctx, float* p, const float* g, float* m, float* v, void* p_shadow, int shadow_dtype, int64_t n, double lr,
                         double beta1, double beta2, double eps, double weight_decay, int step, double max_norm,
                         float* sqnorm_out, void* workspace, size_t ws_bytes, double grad_scale, const int32_t* step_dev,
                         void* stream);
/* codae_clip_adam_step without the norm pass: sum g^2 = the sum of `n_partials` doubles written by the
 * codae_linear_wgrad_sq launches of this step (summed in index order by every CTA: reproducible).  Same arithmetic
 * and argument meaning otherwise; sqnorm_out (f32[1]) receives the sum.  Not for data-parallel runs (the norm must
 * be taken after the gradient all-reduce). */
int codae_adam_step_partials(codae_ctx* ctx, float* p, const float* g, float* m, float* v, void* p_shadow, int shadow_dtype, int64_t n,
                             double lr, double beta1, double beta2, double eps, double weight_decay, int step,
                             double max_norm, const double* sq_partials, int n_partials, float* sqnorm_out,
                             double grad_scale, const int32_t* step_dev, void* stream);
/* *counter += delta on the device (the Adam step counter of a CUDA-graph-captured training step). */
int codae_counter_add(codae_ctx* ctx, int32_t* counter, int delta, void* stream);

/* ---- K4 under data parallelism: reduce-scatter + clip + Adam + all-gather as ONE kernel over NVLink peer memory ----------
 * Replaces, per step, the reference-equivalent DP sequence  all-reduce(grads) -> clip_grad_norm_ -> Adam.step on every replica
 * (train_dae_on_embedding.py:209-215 under one process per GPU).  Rank r owns elements [r S, (r+1) S) of the flat buffers,
 * S = codae_dp_shard_elems(n, world): it sums that shard of every rank's gradient buffer through peer loads (rank order,
 * deterministic), exchanges the shard's sum of squares with the peers (same clip scale, bit for bit, on every rank), applies
 * Adam to the shard (p: this rank's f32 master [n], only the shard is updated; m, v: SHARD-sized moments [S]) and stores the
 * new weights into EVERY rank's weight buffer w_out[q] ([n] bf16 shadow -- CODAE_BF16 -- or the f32 master itself --
 * CODAE_F32, then w_out[rank] == p).  When the kernel ends on a rank, that rank's weight buffer is complete and no peer reads
 * its gradients any more.  grads / w_out / signals are device pointers valid in THIS process for every rank's buffer (CUDA IPC /
 * torch symmetric memory); signals[q]: CODAE_DP_SIGNAL_BYTES bytes, zeroed once before the first call, owned by the library
 * afterwards.  Every rank must call it the same number of times; cross-GPU waits are bounded (CODAE_DP_TIMEOUT_S, default 30 s:
 * the kernel traps and the next CUDA call reports it).  Cooperative launch, no host synchronisation, CUDA-graph capturable.
 * n % 8 == 0 (the flat layout pads rows to 64 elements), world <= CODAE_DP_MAX_WORLD. */
#define CODAE_DP_MAX_WORLD 8
#define CODAE_DP_SIGNAL_BYTES 512
typedef struct codae_dp_peers {
    int32_t world, rank;
    const float* grads[CODAE_DP_MAX_WORLD];
    void* w_out[CODAE_DP_MAX_WORLD];
    void* signals[CODAE_DP_MAX_WORLD];
    /* NVSwitch multicast (NVLS) addresses of the SAME gradient / weight buffers, or NULL.  When both are given the kernel
     * reduces its shard with one multimem.ld_reduce per 16 bytes (the switch adds the ranks' values: each rank receives its
     * shard once, not world - 1 times) and broadcasts the new weights with one multicast store per 16 bytes.  The sum is
     * formed inside the switch instead of in rank order; every rank still reduces only its own shard, so replicas stay
     * bitwise equal.  Used from 8 ranks on (measured: the multimem path moves fewer bytes but at a lower rate -- slower than the
     * peer loops at 2 and 4 GPUs, faster at 8); CODAE_DP_NVLS=0|1 overrides.  torch symmetric memory: handle.multicast_ptr. */
    const float* grads_mc;
    void* w_mc;
} codae_dp_peers;
size_t codae_dp_workspace_bytes(const codae_ctx* ctx);
int64_t codae_dp_shard_elems(int64_t n, int world);
int codae_dp_adam_step(codae_ctx* ctx, const codae_dp_peers* peers, float* p, float* m, float* v, int w_dtype, int64_t n,
                       double lr, double beta1, double beta2, double eps, double weight_decay, int step, double max_norm,
                       float* sqnorm_out, void* workspace, size_t ws_bytes, double grad_scale, const int32_t* step_dev,
                       void* stream);

/* ---- K3: complementarity inference -------------------------------------------------------------- */
/* Scores every row of a catalog shard against Q query vectors and keeps the best k per query.
 * Generalises RankingLoss.get (codae/tool/metering.py:46-79) into the stage-IV entry point the README
 * names (README.md:14-16,30-32; script absent from the reference).
 *   catalog [n_rows, ld] f32|bf16 ; query [Q, E] f32 ; score_j = sum_d (q_d - cat_jd * inv_scale)^2
 *   (SQERR, lower is better) or cosine similarity (higher is better; metering.py:67-69).
 *   out_score [Q, k] f32, out_idx [Q, k] int64 = row_offset + local row; sorted best first,
 *   ties -> lower index.  Unused slots (n_rows < k): idx = -1.  1 <= k <= 128, E <= 4096, E % 4 == 0.  */
size_t codae_score_topk_workspace_bytes(const codae_ctx* ctx, int Q, int k);
int codae_score_topk(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                     int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k,
                     float* out_score, int64_t* out_idx, void* workspace, size_t ws_bytes, void* stream);
/* Batched top-k on tensor cores: the same results as codae_score_topk -- the same scores bit for bit, the same indices, ties
 * by (score, index) -- for many queries in about one pass over the catalog.  A tcgen05 contraction of the queries (as hi / mid
 * bf16 planes) against the catalog PROPOSES k' = min(2k + 32, 128) candidates per query, ranked by a bound on the sweep's
 * fp32 score; the proposals are re-scored with the sweep's own arithmetic and the query is CERTIFIED when the exact k-th score
 * is strictly better than the bound of every row left out (or when the shard has at most k' rows).
 *   Arguments, layouts and E / ld / alignment rules: as codae_score_topk.  1 <= k <= CODAE_TOPK_BATCHED_MAX_K.
 *   n_uncertified: device int, set to the number of queries that could not be certified; uncertified: device int [Q], its
 *   first *n_uncertified entries are those query numbers (in no particular order).  Their out_score / out_idx rows are
 *   unspecified: compute them with codae_score_topk (codae.tool.ComplementarityScorer.topk_local_batched does).
 *   workspace >= codae_score_topk_batched_workspace_bytes(ctx, cat_dtype, n_rows, E, Q, k), 256-byte aligned; after the call
 *   it begins with the merged proposals: float key[Q][k'] then, at offset round_up(4 Q k', 256), int64 idx[Q][k'] (best
 *   first; key = the bound, never better than the row's exact score; idx -1 = empty).  fp32 catalogs are split into planes
 *   chunk by chunk in the workspace (at most 512 MB of it).
 *   Anything outside these limits returns CODAE_EINVAL; the call never switches to another algorithm by itself. */
#define CODAE_TOPK_BATCHED_MAX_K 64
size_t codae_score_topk_batched_workspace_bytes(const codae_ctx* ctx, int cat_dtype, int64_t n_rows, int E, int Q, int k);
int codae_score_topk_batched(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                             int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k,
                             float* out_score, int64_t* out_idx, int* n_uncertified, int* uncertified, void* workspace,
                             size_t ws_bytes, void* stream);
/* Filtered top-k: codae_score_topk / codae_score_topk_batched / codae_swap_error_topk with a say in which rows may be returned,
 * e.g. leaving out the item the query outfit already holds, or keeping only items in stock.  Each takes its unfiltered
 * sibling's arguments plus, before the outputs:
 *   allow      uint8 [n_rows] indexed by LOCAL row (row j of `catalog`; swap: catalog row first_row + b), nonzero = eligible;
 *              NULL = every row is eligible.
 *   exclude    int64 [Q][n_exclude] GLOBAL indices (row_offset + local row) per query -- the same tensor fits every shard;
 *              swap scoring has one outfit: [n_exclude].  Entries < 0 are padding; entries outside the shard never match.
 *   n_exclude  0 <= n_exclude <= CODAE_TOPK_MAX_EXCLUDE; exclude is NULL exactly when n_exclude == 0.
 * A filtered-out row behaves as if it were absent from the catalog: it never appears in the output; with fewer than k eligible
 * rows the trailing slots are the usual empty ones (idx = -1, score = the unfiltered call's empty-slot value); ties stay
 * (score, index).  The score of a row does not depend on which other rows are scored, so a filtered call equals, bit for bit,
 * the unfiltered call on the catalog compacted to its eligible rows with the indices mapped back; the batched filtered call
 * equals the filtered sweep bit for bit (its uncertified queries are recomputed with codae_score_topk_filtered, the same allow
 * and their rows of exclude).  Workspace sizes are those of the unfiltered calls.  row_offset must be >= 0.  Bad filter
 * arguments return CODAE_EINVAL.  No filter (allow NULL, n_exclude 0) runs exactly the unfiltered code.              */
#define CODAE_TOPK_MAX_EXCLUDE 256
int codae_score_topk_filtered(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                              int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k,
                              const uint8_t* allow, const int64_t* exclude, int n_exclude, float* out_score, int64_t* out_idx,
                              void* workspace, size_t ws_bytes, void* stream);
int codae_score_topk_batched_filtered(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                                      int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k,
                                      const uint8_t* allow, const int64_t* exclude, int n_exclude, float* out_score,
                                      int64_t* out_idx, int* n_uncertified, int* uncertified, void* workspace, size_t ws_bytes,
                                      void* stream);
/* Deterministic merge of G per-shard lists [G, Q, k] (e.g. after an all-gather) into [Q, k]. */
int codae_topk_merge(codae_ctx* ctx, const float* scores, const int64_t* idx, int G, int Q, int k, int metric,
                     float* out_score, int64_t* out_idx, void* stream);
/* out_rank[q] = #{ j in subset : score(true_idx[q]) strictly better than score(j) } -- the rank inside
 * RankingLoss.get (metering.py:72-75).  subset_idx int64 [n_subset] or NULL (all rows).  Q <= 1024.   */
int codae_score_rank(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                     const float* query, int Q, float inv_scale, int metric, const int64_t* true_idx,
                     const int64_t* subset_idx, int64_t n_subset, int64_t* out_rank, void* stream);
/* Rank mode for large query batches (Q >= 64 per category; every validation batch of train_dae_on_embedding.py:241-261 calls
 * RankingLoss.get): the Q x n cosine numerators are ONE contraction on the fp32-parity tensor-core engine
 * (codae_linear_fwd_x3 with X = queries, W = [subset rows ; the Q true rows] as CODAE_F32X3 planes, f32 output [Q, n + Q]);
 * codae_row_sqnorm supplies |c|^2 / |q|^2 (out[r] = sum_d X[r, d]^2) and codae_rank_count the ranks:
 *   out_rank[q] = #{ j < n : cos(q, true_q) > cos(q, c_j) },  cos = dot / max(sqrt(|c|^2 |q|^2), 1e-8)  (metering.py:67-75),
 *   dot(q, c_j) = scores[q, j], dot(q, true_q) = scores[q, n + q]; cc [n + Q] f32, qq [Q] f32.  Cosine only. */
int codae_row_sqnorm(codae_ctx* ctx, const float* X, int64_t ld, int64_t rows, int E, float* out, void* stream);
int codae_rank_count(codae_ctx* ctx, const float* scores, int64_t ld, int Q, int64_t n, const float* cc, const float* qq,
                     int64_t* out_rank, void* stream);

/* Candidate SWAPS scored by full reconstruction error (the GEMM-bound reading of stage IV): candidate j replaces slot
 * `slot` of the (scaled) outfit, the DAE reconstructs the swapped outfit (codae_linear_fwd per layer, batched over the
 * candidates), and the swap's score is sum_d (DAE(x'_j)_d - x'_j,d)^2 over all io dimensions (lower is better).
 *   codae_swap_build      x'[b, :] for candidates first_row .. first_row+B-1 of `catalog` ([.., ld_cat] f32|bf16, un-scaled,
 *                         multiplied by inv_scale), written as f32|bf16 with pitch ld_x (columns >= io untouched)
 *   codae_swap_error_topk errors of the B reconstructions y [B, ld_y] f32 and the best k of them:
 *                         out_score [k], out_idx [k] = row_offset + first_row + b, best first, ties -> lower index,
 *                         unused slots idx = -1.  workspace >= codae_score_topk_workspace_bytes(ctx, 1, k).
 * Lists of several candidate chunks / ranks are combined with codae_topk_merge.                                  */
int codae_swap_build(codae_ctx* ctx, const float* outfit, const void* catalog, int cat_dtype, int64_t ld_cat, int64_t first_row,
                     int B, int E, int slot, int io, float inv_scale, void* out_x, int x_dtype, int64_t ld_x, void* stream);
int codae_swap_error_topk(codae_ctx* ctx, const float* outfit, const void* catalog, int cat_dtype, int64_t ld_cat,
                          int64_t first_row, int B, int E, int slot, int io, float inv_scale, const float* y, int64_t ld_y,
                          int64_t row_offset, int k, float* out_score, int64_t* out_idx, void* workspace, size_t ws_bytes,
                          void* stream);
/* codae_swap_error_topk with allow [rows of catalog] and exclude [n_exclude]: see the filtered top-k above. */
int codae_swap_error_topk_filtered(codae_ctx* ctx, const float* outfit, const void* catalog, int cat_dtype, int64_t ld_cat,
                                   int64_t first_row, int B, int E, int slot, int io, float inv_scale, const float* y,
                                   int64_t ld_y, int64_t row_offset, int k, const uint8_t* allow, const int64_t* exclude,
                                   int n_exclude, float* out_score, int64_t* out_idx, void* workspace, size_t ws_bytes,
                                   void* stream);
/* Swaps over per-outfit candidate lists (re-ranking: retrieve M rows per outfit cheaply, score those M by swap error).  Any set of
 * (outfit, candidate) pairs goes through the same GEMM chain in chunks of B rows, however the pairs are spread over outfits:
 *   outfits    [Q, ld_outfit] f32, scaled rows (io columns used); one slot for every outfit.
 *   candidates int64 [Q][m] GLOBAL catalog row ids (row_offset + local row), entries < 0 are padding; the same list fits every
 *              shard.  Pairs are numbered p = q * m + j (0 <= p < Q m <= INT32_MAX).
 *   pos        int64 [B]: built row b holds pair pos[b].  Its outfit is q = pos[b] / m, its local catalog row
 *              candidates[pos[b]] - row_offset.
 * A pos outside [0, Q m) or a local row outside [0, n_rows) is never dereferenced: the row is built as zeros and no error is written
 * for it (pos and candidates are device data; the host cannot check them without a synchronisation).
 *   codae_swap_build_pairs  x'[b, :] = outfit q with the slot columns replaced by catalog row * inv_scale, f32|bf16, pitch ld_x --
 *                           codae_swap_build's values for that outfit and row.
 *   codae_swap_error_pairs  err[pos[b]] = the swap error of built row b from y [B, ld_y] f32; err is [Q m] f32, set to NaN by the
 *                           caller, so pairs that are not built stay NaN.
 *   codae_swap_pairs_topk   per outfit, the best k (1 <= k <= 128) pairs by (error, candidate id): out_score / out_idx [Q][k],
 *                           best first, NaN errors and ids < 0 skipped, unused slots (+inf, -1); a duplicated id is returned once
 *                           per listing.  Lists of several ranks are combined with codae_topk_merge (CODAE_METRIC_SQERR).
 * Numerics: a pair's error is computed exactly as codae_swap_error_topk computes a candidate's -- the same build values, the same
 * codae_linear_fwd chain, the same per-lane fmaf order and warp_sum over io.  A GEMM row's result depends only on that row and on
 * the launch's shape (the tensor-core plan follows the row count through its 128-row tile count), so (a) pairs in chunks of
 * the same tile counts get the same bits
 * wherever they sit and whatever the other rows of the chunk are, and in particular one outfit listing rows row_offset ..
 * row_offset + n_rows - 1 in order gives the sweep's errors and ids bit for bit; (b) otherwise errors agree with the fp64
 * reference to the engine's tolerance.  Bad shapes, k, NULL arguments return CODAE_EINVAL.                          */
int codae_swap_build_pairs(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, const void* catalog, int cat_dtype,
                           int64_t ld_cat, int64_t n_rows, int64_t row_offset, const int64_t* candidates, int m, const int64_t* pos,
                           int B, int E, int slot, int io, float inv_scale, void* out_x, int x_dtype, int64_t ld_x, void* stream);
int codae_swap_error_pairs(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, const void* catalog, int cat_dtype,
                           int64_t ld_cat, int64_t n_rows, int64_t row_offset, const int64_t* candidates, int m, const int64_t* pos,
                           int B, int E, int slot, int io, float inv_scale, const float* y, int64_t ld_y, float* err, void* stream);
int codae_swap_pairs_topk(codae_ctx* ctx, const float* err, const int64_t* candidates, int Q, int m, int k, float* out_score,
                          int64_t* out_idx, void* stream);

/* Outfit COMPATIBILITY by leave-one-slot-out reconstruction: how well do the S items of a complete outfit go together, and which
 * one fits least?  Slot s of the outfit is hidden (multiplied by 0), the DAE reconstructs the outfit, and the distance of the
 * reconstructed slot s from the item that was there is that slot's error; a compatible outfit has small errors.  The input rows
 * come from codae_corrupt_fwd: with mask_table int16 [Q, S] (every row 0 .. S-1), mask_bits [S] = 1 << s and col_var [io] = c / E,
 * launch s (data = the Q outfit rows, batch_idx NULL, run s) writes rows [s Q, (s+1) Q) of the GEMM chain's input -- bit for bit
 * what predict_slot(model, outfits, s, E) feeds the model (the same multiply: -0.0, NaN and inf propagate alike).
 *   outfits [Q, ld_outfit] f32   the scaled outfit rows (S E columns used)
 *   y       [S Q, ld_y] f32      the reconstructions, slot-major: row s Q + i is outfit i with slot s hidden
 *   err     [Q, S] f32           err[i, s] = sum_{d < E} (y[s Q + i, s E + d] - outfits[i, s E + d])^2 (lane-strided fmaf, warp tree)
 *   score   [Q] f32              err[i, 0] + err[i, 1] + ... + err[i, S-1], summed in slot order in fp32 (lower: more compatible)
 *   odd     [Q] int64            argmax_s err[i, s], ties -> the lower slot (the odd item out)
 * A NaN error makes that outfit's score NaN and its odd -1.  An outfit holding a NaN or inf in its S E columns gets NaN for every
 * err (score NaN, odd -1): the GEMM chain's ReLU (fmaxf) maps NaN to 0, so its reconstructions may be finite but say nothing.  Q >= 1, 1 <= S <= 64 (the corruption kernel's variable limit),
 * E % 4 == 0, ld_outfit and ld_y >= S E, buffers naturally aligned; CODAE_EINVAL otherwise.
 * Numerics: a GEMM row depends only on that row and on the launch's 128-row tile count, so for a fixed chunk layout an outfit's
 * err / score / odd do not depend on the other outfits of its launch or their order, and repeat bit for bit run to run; err
 * agrees with an fp64 restatement to the engine's tolerance (1e-5 relative for the fp32-parity and FFMA engines, 1e-2 for bf16);
 * score and odd follow from the returned err bit for bit. */
int codae_outfit_loo_error(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const float* y, int64_t ld_y,
                           float* err, float* score, int64_t* odd, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CODAE_B200_H */
