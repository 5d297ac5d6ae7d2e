/* rigl_b200 -- C ABI of the B200-native RigL hot path.
 *
 * The reference (google-research/rigl) is pure Python/TensorFlow and has no FFI
 * of its own; these entry points are what a binding for its two hot paths
 * would call.  Each declaration cites the reference interface it replaces
 * (file:line into the reference tree).  Conventions:
 *   - plain pointers and sizes only; every tensor is caller-owned DEVICE memory
 *     (allocated by PyTorch in this repo); nothing is retained past a call
 *     except by the explicit plan objects, which hold pointers, not ownership;
 *   - every function returns 0 on success, a negative rigl_status otherwise;
 *     rigl_last_error() gives the message (thread-local);
 *   - launches go to the `stream` argument (a cudaStream_t passed as void*),
 *     no host synchronisation inside, safe under CUDA-graph capture unless
 *     stated;
 *   - weights / masks / gradients are float32, flattened in the reference's own
 *     layout: HWIO [kh,kw,Cin,Cout] for conv kernels, [in,out] for dense
 *     (Cout fastest) -- the flat index IS the tie-break order of tf.nn.top_k.
 *   - a mask is a bitmap: bit (i & 31) of word (i >> 5) <=> mask.flat[i] == 1;
 *     word count = rigl_mask_words(n); bits >= n are zero.
 */
#ifndef RIGL_B200_H_
#define RIGL_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define RIGL_API __attribute__((visibility("default")))
#else
#define RIGL_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  RIGL_OK = 0,
  RIGL_ERR_INVALID_ARG = -1,
  RIGL_ERR_CUDA = -2,
  RIGL_ERR_WORKSPACE = -3,
  RIGL_ERR_UNSUPPORTED = -4,
  RIGL_ERR_DRIVER = -5
} rigl_status;

/* Library version (major*10000 + minor*100 + patch). */
RIGL_API int rigl_version(void);
/* Message of the last failing call on this thread ("" if none). */
RIGL_API const char* rigl_last_error(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
RIGL_API uint64_t rigl_launch_count(void);

/* ------------------------------------------------------------------------
 * Mask bitmaps  (reference: the float32 `mask` variable of
 * tf.contrib.model_pruning masked layers; rigl/sparse_utils.py:39-45,71-87)
 * ---------------------------------------------------------------------- */
/* Words (uint32) a bitmap of n bits occupies; padded to a multiple of 4 words. */
RIGL_API int64_t rigl_mask_words(int64_t n);
/* bits <- (src[i] != 0).  Replaces tf.assign(mask, new_mask), sparse_utils.py:359-362. */
RIGL_API int rigl_mask_pack_f32(const float* src, int64_t n, uint32_t* bits, void* stream);
/* dst[i] <- bit ? 1.0f : 0.0f.  Replaces reading the mask variable. */
RIGL_API int rigl_mask_unpack_f32(const uint32_t* bits, int64_t n, float* dst, void* stream);
/* *out_count_dev <- popcount(bits) (one int32 on the device).  Replaces
 * reduce_sum(mask): sparse_utils.py:39-45, sparse_optimizers_base.py:286,
 * imagenet_resnet/utils.py:83-90. */
RIGL_API int rigl_mask_popcount(const uint32_t* bits, int64_t n, int32_t* out_count_dev, void* stream);
/* dst[i] <- bit ? src[i] : 0  (dL/dweights = mask * dL/d(masked_weights)),
 * the masked gradient the wrapped optimizer consumes; sparse_optimizers_base.py:480. */
RIGL_API int rigl_apply_mask_f32(const float* src, const uint32_t* bits, int64_t n, float* dst,
                        float scale, void* stream);

/* ------------------------------------------------------------------------
 * Periodic mask update: drop (magnitude top-k) + grow (dense-gradient top-k)
 * Replaces SparseSETOptimizerBase._get_update_op (sparse_optimizers_base.py:
 * 276-343) together with generic_mask_update (:260-274, :523-538),
 * get_grow_tensor (:355-400, :540-553) and reset_momentum (:345-353, :555-564)
 * for ALL masked layers in one batched launch sequence.
 * ---------------------------------------------------------------------- */
typedef struct {
  float* weights;            /* [n] in/out: grown entries are overwritten        */
  const float* score_grow;   /* [n] dense dL/d(mask*w) (RigL) | U[0,1) (SET) | mask (Static); ranked by
                                |score_grow| unless RIGL_LAYER_GROW_SCORE_SIGNED is set in `flags` */
  uint32_t* mask_bits;       /* [rigl_mask_words(n)] in/out                      */
  const float* noise;        /* [n] added to |mask*w| before ranking, or NULL    */
  float* slots[2];           /* optimizer slots reset at new connections, or NULL */
  const float* grow_values;  /* [n] used by RIGL_GROW_TENSOR, else NULL          */
  const float* score_drop;   /* [n] explicit drop scores (overrides |mask*w|+noise), or NULL:
                                the `_get_update_op(score_drop, ...)` entry, base.py:276 */
  int64_t n;                 /* elements, 1 <= n < 2^31                          */
  int32_t n_prune_override;  /* >= 0: use this n_prune; -1: int32(float32(n_ones)*drop_fraction) */
  int32_t flags;             /* RIGL_LAYER_* bits */
  uint32_t noise_key;        /* per-layer key of the in-kernel drop-score noise (rigl_mask_update_run_noise) */
  uint32_t reserved;
  const float* grad;         /* [n] gradient read by RIGL_GROW_GRAD_SCALE / _SIGN and by the slot reset
                                (slot <- grad * acc_scale), base.py:540-564; NULL: score_grow is the gradient
                                (the RigL / Momentum callers, whose grow score IS the dense gradient) */
} rigl_layer_desc;

/* rigl_layer_desc.flags */
#define RIGL_LAYER_GROW_SCORE_SIGNED 1  /* rank score_grow verbatim (signed), as `_get_update_op(score_drop,
                                           score_grow, ...)` (base.py:276-343) does with caller-built scores,
                                           e.g. the rigl_tf2 updaters' -|g|; default ranks |score_grow| */
#define RIGL_LAYER_DROP_ONLY 2          /* grow nothing: mask <- the kept set (top n_ones - n_prune of the drop
                                           scores); weights and slots are not touched */
#define RIGL_LAYER_ALL_ACTIVE 4         /* rank EVERY position as if the mask were all ones (n_ones = n).  With
                                           DROP_ONLY and n_prune_override = get_n_zeros(n, sparsity) this is the
                                           "mask = top-k of a score" of SparseSnipOptimizer (|g*w|, score_drop) and
                                           SparseDNWOptimizer (|w|: no score_drop), sparse_optimizers.py:286-316,
                                           :436-465 */

typedef enum {
  RIGL_GROW_ZEROS = 0,       /* 'zeros'            base.py:372-373 */
  RIGL_GROW_TENSOR = 1,      /* caller-supplied    (random_normal/uniform/initial_dist draws) */
  RIGL_GROW_GRAD_SCALE = 2,  /* 'grad_scale_<d>'   base.py:542-545: g / d */
  RIGL_GROW_GRAD_SIGN = 3    /* 'grad_sign_<d>'    base.py:546-549: sign(g) / d */
} rigl_grow_mode;

typedef struct rigl_mask_plan rigl_mask_plan;

/* Builds the device-side layer table and block schedule for a fixed set of
 * layers (pointers are captured).  Not capturable (allocates). */
RIGL_API int rigl_mask_plan_create(const rigl_layer_desc* layers, int n_layers, rigl_mask_plan** out);
RIGL_API int rigl_mask_plan_destroy(rigl_mask_plan* plan);
/* Caller-owned scratch needed by rigl_mask_update_run (device memory, 256B aligned). */
RIGL_API size_t rigl_mask_plan_workspace_bytes(const rigl_mask_plan* plan);
/* One full update of every layer in the plan.
 *   drop_fraction : float32 value of self.drop_fraction for this step (host-computed,
 *                   base.py:232-258); n_prune = int32(float32(n_ones) * drop_fraction).
 *   acc_scale     : initial_acc_scale; slots[.] <- score_grow * acc_scale at new connections.
 *   reinit_when_same : base.py:328-333 (SparseStaticOptimizer passes 1).
 * Per-layer results (n_ones, n_prune, n_keep, ...) are left in the workspace;
 * see rigl_mask_plan_read_stats. */
RIGL_API int rigl_mask_update_run(rigl_mask_plan* plan, float drop_fraction, int grow_mode,
                         float grow_divisor, float acc_scale, int reinit_when_same,
                         void* workspace, size_t workspace_bytes, void* stream);
/* Same, with the drop-score noise of generic_mask_update (noise_std, base.py:260-274, 523-538) drawn IN-KERNEL
 * for every layer whose `noise` pointer is NULL (and that has no explicit score_drop): element i of a layer gets
 * noise_std * N(0,1) from a counter-based generator keyed by (noise_seed, layer noise_key, i) -- no noise tensor
 * is written or read.  noise_std = 0 behaves like rigl_mask_update_run. */
RIGL_API int rigl_mask_update_run_noise(rigl_mask_plan* plan, float drop_fraction, int grow_mode,
                         float grow_divisor, float acc_scale, int reinit_when_same, float noise_std,
                         uint64_t noise_seed, void* workspace, size_t workspace_bytes, void* stream);
/* out[i] <- exactly the noise rigl_mask_update_run_noise adds to element i of a layer with this key
 * (tests and the CPU oracle consume it; the product path never materialises it). */
RIGL_API int rigl_mask_noise_fill(float* out, int64_t n, uint32_t layer_noise_key, float noise_std,
                         uint64_t noise_seed, void* stream);
/* Copies 8 int32 per layer {n_ones, n_prune, n_keep, drop_candidates, grow_candidates,
 * drop_bucket, grow_bucket, 0} to host (synchronises the stream). */
RIGL_API int rigl_mask_plan_read_stats(const rigl_mask_plan* plan, const void* workspace,
                              int32_t* out_host, void* stream);

/* ------------------------------------------------------------------------
 * Masked weight operands (mask fused into the fp32 -> bf16 weight load)
 * Replaces `masked_weights = mask * weights` of tf.contrib.model_pruning
 * (call sites rigl/imagenet_resnet/pruning_layers.py:140-157, 223-233).
 * ---------------------------------------------------------------------- */
/* Bytes of the packed operand blob for a [taps, cin, cout] weight tensor. */
RIGL_API size_t rigl_packed_weights_bytes(int taps, int cin, int cout);
/* From HWIO fp32 weights + bitmap, writes the packed blob (256B-aligned sections):
 *   w_fprop bf16 [taps][cout][cin_pad]  (K = cin contiguous)   B operand of fprop
 *   w_dgrad bf16 [taps][cin][cout_pad]  (K = cout contiguous)  B operand of dgrad
 *   tile_nnz u32 [taps][ceil(cout/64)][ceil(cin/64)]  surviving weights per 64x64
 *            weight tile -- the per-tile gate: all-zero tiles are never fetched.
 * cin_pad / cout_pad = rounded up to a multiple of 8 (16-byte rows); padding = 0. */
RIGL_API int rigl_pack_masked_weights(const float* w_hwio, const uint32_t* mask_bits, int taps,
                                      int cin, int cout, void* packed, void* stream);

/* The same for ALL masked layers of a model in ONE launch (the reference rebuilds every layer's
 * `mask * weights` once per step; per-layer launches cost more than the 200 MB they move).  Pointers are
 * captured at plan creation, like rigl_mask_plan.  Not capturable: create (allocates); capturable: run. */
typedef struct {
  const float* weights;        /* [taps][cin][cout] fp32 (HWIO / [in,out]) */
  const uint32_t* mask_bits;   /* [rigl_mask_words(taps*cin*cout)] */
  void* packed;                /* rigl_packed_weights_bytes(taps, cin, cout) bytes, 256B aligned */
  int32_t taps, cin, cout, reserved;
} rigl_pack_desc;
typedef struct rigl_pack_plan rigl_pack_plan;
RIGL_API int rigl_pack_plan_create(const rigl_pack_desc* layers, int n_layers, rigl_pack_plan** out);
RIGL_API int rigl_pack_plan_destroy(rigl_pack_plan* plan);
RIGL_API int rigl_pack_plan_run(rigl_pack_plan* plan, void* stream);

/* ------------------------------------------------------------------------
 * Wrapped-optimizer step with the masked gradient fused in.
 * Replaces tf.train.MomentumOptimizer(use_nesterov=True).apply_gradients on
 * dL/dweights = mask * dL/d(mask*weights) (imagenet_train_eval.py:355-365,
 * sparse_optimizers_base.py:478-485) for EVERY parameter of a model in one launch:
 *   g = (bit ? grad * grad_scale : 0) + weight_decay * w;  accum = momentum * accum + g;
 *   w -= lr * (nesterov ? g + momentum * accum : accum).
 * The learning rate is read from device memory (graph replays follow a schedule).
 * ---------------------------------------------------------------------- */
typedef struct {
  float* param;                /* [n] in/out */
  float* momentum;             /* [n] in/out accumulator (the 'momentum' slot of the reference) */
  const float* grad;           /* [n] gradient; the DENSE gradient when mask_bits != NULL */
  const uint32_t* mask_bits;   /* NULL (dense parameter) or the layer's bitmap */
  int64_t n;
  float weight_decay;
  float grad_scale;            /* multiplies grad (1/replicas for the summed dense gradients) */
} rigl_sgd_desc;
typedef struct rigl_sgd_plan rigl_sgd_plan;
RIGL_API int rigl_sgd_plan_create(const rigl_sgd_desc* params, int n_params, rigl_sgd_plan** out);
RIGL_API int rigl_sgd_plan_destroy(rigl_sgd_plan* plan);
RIGL_API int rigl_sgd_plan_run(rigl_sgd_plan* plan, const float* lr_dev, float momentum, int nesterov, void* stream);

/* ------------------------------------------------------------------------
 * Masked conv2d / linear as implicit GEMM (tcgen05 on sm_100a; a CUDA-core
 * kernel serves shapes whose row pitch is not a 16-byte multiple).
 * Replaces layers.masked_conv2d / masked_fully_connected fprop and its two
 * gradient GEMMs (pruning_layers.py:72-172, 175-248; sparse_optimizers_base.py:
 * 478-485 for the dense wgrad RigL needs).
 * Activations: NHWC bf16.  Square kernels and strides (pruning_layers.py:143-144).
 * A dense layer is the 1x1 case with in_h = in_w = 1 and batch = rows.
 * ---------------------------------------------------------------------- */
typedef struct {
  int32_t batch, in_h, in_w, cin;     /* x  [batch,in_h,in_w,cin]   bf16 NHWC */
  int32_t out_h, out_w, cout;         /* y  [batch,out_h,out_w,cout] bf16 NHWC */
  int32_t ksize, stride, pad;         /* square; pad = zero rows/cols BEFORE the image: (k-1)/2 for
                                         conv2d_fixed_padding (resnet_model.py:83-108,278-281), TF 'SAME'
                                         pad_total/2, 0 for 'VALID'; the far edge is padded implicitly */
  int32_t x_pitch;                    /* elements between consecutive pixels of x (0 => cin); lets a
                                         zero-padded buffer (e.g. the im2col matrix) be addressed */
} rigl_conv_desc;

RIGL_API size_t rigl_conv_workspace_bytes(const rigl_conv_desc* d);
/* y = conv(x, mask*W) (+ bias[cout]).  `packed` from rigl_pack_masked_weights.
 * y_bf16 and/or y_f32 receive the result (either may be NULL, not both). */
RIGL_API int rigl_masked_conv2d_fprop(const rigl_conv_desc* d, const void* x, const void* packed,
                                      void* y_bf16, float* y_f32, const float* bias, void* ws,
                                      size_t ws_bytes, void* stream);
/* fprop that also emits the batch-norm statistics of its output from the epilogue
 * (SURVEY 8f row 1: the BN stats pass over y disappears): bn_partial[rows][2][cout] fp32 receives
 * per-CTA column sums and sums of squares of the fp32 accumulators, *bn_rows_out (host) the number
 * of rows written (<= rigl_bn_partial_rows()).  Tensor-core path only (RIGL_ERR_UNSUPPORTED else). */
RIGL_API int rigl_bn_partial_rows(void);
RIGL_API int rigl_masked_conv2d_fprop_bnstats(const rigl_conv_desc* d, const void* x, const void* packed,
                                              void* y_bf16, float* bn_partial, int* bn_rows_out, void* ws,
                                              size_t ws_bytes, void* stream);
/* The statistics epilogue is used only where it is profitable (reduction length taps*cin >= 512, or >= 256 with
 * <= 128 output channels; otherwise RIGL_ERR_UNSUPPORTED and the caller runs the plain call + a stats pass).
 * on != 0: for every supported shape (tests; same as RIGL_BN_STATS_ALWAYS=1). */
RIGL_API int rigl_set_bn_stats_always(int on);
/* Inference: y = [relu](conv(x, mask*W) * scale[c] + shift[c] (+ residual)), bf16 out, fp32 math, one rounding.
 * scale / shift / residual may be NULL (scale 1, shift 0, no residual); y, scale, shift and residual must be
 * 16-byte aligned, and residual ([batch,out_h,out_w,cout] bf16) must not overlap y.  RIGL_ERR_UNSUPPORTED where
 * the shape runs on the halo kernels or where the fused epilogue measured slower than the plain call +
 * rigl_bn_apply (policy in DESIGN.md 3.8); the caller then runs those two.  RIGL_AFFINE_ALWAYS=1 lifts the
 * profitability rule (measurement). */
RIGL_API int rigl_masked_conv2d_fprop_affine(const rigl_conv_desc* d, const void* x, const void* packed,
                                             const float* scale, const float* shift, const void* residual,
                                             int relu, void* y_bf16, void* ws, size_t ws_bytes, void* stream);
/* dx = conv^T(dy, mask*W). */
RIGL_API int rigl_masked_conv2d_dgrad(const rigl_conv_desc* d, const void* dy, const void* packed,
                                      void* dx, void* ws, size_t ws_bytes, void* stream);
/* dw[kh,kw,cin,cout] (fp32, HWIO, DENSE -- every position, as RigL's grow needs)
 * = sum over pixels x (x) dy.  beta=0 overwrites, beta=1 accumulates into dw. */
RIGL_API int rigl_conv2d_wgrad_dense(const rigl_conv_desc* d, const void* x, const void* dy,
                                     float* dw, float beta, void* ws, size_t ws_bytes, void* stream);
/* Patch matrix of a conv whose channel count cannot be addressed by TMA (the 7x7x3 stem,
 * resnet_model.py:620-633): out[pixel][(kh*k+kw)*cin + ci] = x[n, ho*s+kh-pad, wo*s+kw-pad, ci]
 * (0 outside), bf16, row pitch out_pitch >= k*k*cin (extra columns zeroed).  The conv then
 * runs as a masked dense layer over [pixels, k*k*cin] with the SAME HWIO weights and mask. */
RIGL_API int rigl_im2col_nhwc(const rigl_conv_desc* d, const void* x, void* out, int64_t out_pitch,
                              void* stream);
/* EXPERIMENTAL (opt-in in the host mirror: layers.STEM_S2D_PATH; not yet validated on hardware).
 * The 7x7 / stride-2 / 3-channel stem (conv2d_fixed_padding, resnet_model.py:619-629) without a
 * patch matrix: rigl_stem_s2d_fold_input folds the zero-padded input 2x2 -> 16 channels
 * ([N,(H+6)/2,(W+6)/2,16] bf16, rigl_stem_s2d_folded_bytes), the conv becomes a 4x4 stride-1 conv
 * whose 16 taps are fed from one shared-memory halo tile; rigl_stem_s2d_pack_weights writes the
 * [16 taps][cout][16] operand from the SAME HWIO weights + bitmap; _wgrad returns the dense
 * [7,7,cin,cout] gradient.  Requires ksize 7, stride 2, pad 3, cin <= 3, cout <= 64, even extents,
 * out_w <= 125. */
RIGL_API int rigl_stem_s2d_supported(const rigl_conv_desc* d);
RIGL_API size_t rigl_stem_s2d_folded_bytes(const rigl_conv_desc* d);
RIGL_API size_t rigl_stem_s2d_packed_bytes(const rigl_conv_desc* d);
RIGL_API size_t rigl_stem_s2d_workspace_bytes(const rigl_conv_desc* d);
RIGL_API int rigl_stem_s2d_fold_input(const rigl_conv_desc* d, const void* x, void* xs, void* stream);
RIGL_API int rigl_stem_s2d_pack_weights(const rigl_conv_desc* d, const float* w_hwio,
                                        const uint32_t* mask_bits, void* packed, void* stream);
RIGL_API int rigl_stem_s2d_fprop(const rigl_conv_desc* d, const void* xs, const void* packed, void* y,
                                 void* stream);
RIGL_API int rigl_stem_s2d_wgrad(const rigl_conv_desc* d, const void* xs, const void* dy, float* dw,
                                 float beta, void* ws, size_t ws_bytes, void* stream);

/* Small-Cin convs (cin <= 8, ksize <= 8: the 7x7x3 stem, resnet_model.py:620-633) WITHOUT a
 * patch matrix: the input is copied once into a zero-bordered 8-channel buffer `xp`
 * (rigl_smallc_padded_bytes); window tensor maps with a W stride of `stride` pixels then feed
 * the same tcgen05 kernels with ksize "taps" of K = 64 = 8 pixels x 8 channels.  `packed` here
 * is the stem-specific operand written by rigl_smallc_pack_weights from the SAME HWIO weights
 * and mask.  dw is the dense HWIO gradient as in rigl_conv2d_wgrad_dense. */
RIGL_API int rigl_smallc_supported(const rigl_conv_desc* d);
RIGL_API size_t rigl_smallc_padded_bytes(const rigl_conv_desc* d);
RIGL_API size_t rigl_smallc_packed_bytes(const rigl_conv_desc* d);
RIGL_API size_t rigl_smallc_workspace_bytes(const rigl_conv_desc* d);
RIGL_API int rigl_smallc_pad_input(const rigl_conv_desc* d, const void* x, void* xp, void* stream);
RIGL_API int rigl_smallc_pack_weights(const rigl_conv_desc* d, const float* w_hwio,
                                      const uint32_t* mask_bits, void* packed, void* stream);
RIGL_API int rigl_smallc_fprop(const rigl_conv_desc* d, const void* xp, const void* packed, void* y,
                               void* stream);
RIGL_API int rigl_smallc_wgrad(const rigl_conv_desc* d, const void* xp, const void* dy, float* dw,
                               float beta, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------
 * Fused batch-norm (+ReLU, +residual) over NHWC bf16 activations viewed as [rows, channels]
 * Replaces batch_norm_relu (rigl/imagenet_resnet/resnet_model.py:41-80) and the
 * relu(inputs + shortcut) block tail (:501).  channels % 8 == 0.  SURVEY 8(f) row 1.
 * ---------------------------------------------------------------------- */
RIGL_API size_t rigl_bn_workspace_bytes(int64_t rows, int channels);
/* Training forward: batch statistics of y, running-stat update (momentum = 1 - decay, may be
 * NULL), out = [relu](gamma*(y-mean)*rstd + beta (+ residual)).  save_* [channels] fp32 are kept
 * for the backward pass (scale = gamma*rstd, shift = beta - mean*scale). */
RIGL_API int rigl_bn_forward_train(const void* y, const void* residual, const float* gamma,
                                   const float* beta, int64_t rows, int channels, float eps,
                                   float momentum, int relu, float* running_mean, float* running_var,
                                   float* save_mean, float* save_rstd, float* save_scale,
                                   float* save_shift, void* out, void* ws, size_t ws_bytes, void* relu_bits,
                                   void* stream);
/* relu_bits (optional, uint8 [rows*channels/8]): bit k of byte i <- out[8i+k] > 0.  The residual-form backward
 * needs nothing else of the block output, so it reads this bitmap (1/16 of the bytes) instead of re-reading it. */
/* Training forward from conv-epilogue partial sums (rigl_masked_conv2d_fprop_bnstats). */
RIGL_API int rigl_bn_forward_train_partials(const void* y, const void* residual, const float* gamma,
                                            const float* beta, const float* partial, int partial_rows,
                                            int64_t rows, int channels, float eps, float momentum, int relu,
                                            float* running_mean, float* running_var, float* save_mean,
                                            float* save_rstd, float* save_scale, float* save_shift, void* out,
                                            void* relu_bits, void* stream);
/* Inference / given statistics: out = [relu](y*scale + shift (+ residual)). */
RIGL_API int rigl_bn_apply(const void* y, const void* residual, const float* scale, const float* shift,
                           int64_t rows, int channels, int relu, void* out, void* stream);
/* Backward.  da = gradient of the output; y = the saved BN input; act = the saved output
 * (required only in the residual form).  dresidual != NULL selects the residual form and
 * receives the gradient of the shortcut.  Writes dy, dgamma, dbeta. */
RIGL_API int rigl_bn_backward(const void* da, const void* y, const void* act, const float* save_mean,
                              const float* save_rstd, const float* save_scale, const float* save_shift,
                              int64_t rows, int channels, int relu, void* dy, void* dresidual,
                              float* dgamma, float* dbeta, void* ws, size_t ws_bytes, void* stream);
/* Same with the output gradient given as TWO addends, da + da2 (da2 may be NULL): the output of a
 * residual block feeds both the next block's first conv and its shortcut, and TensorFlow's
 * gradient aggregation (an AddN per forked tensor) would otherwise be a separate elementwise pass.
 * The sum is rounded to bf16 exactly like that separate add.  Residual form only. */
RIGL_API int rigl_bn_backward2(const void* da, const void* da2, const void* y, const void* act,
                               const float* save_mean, const float* save_rstd, const float* save_scale,
                               const float* save_shift, int64_t rows, int channels, int relu, void* dy,
                               void* dresidual, float* dgamma, float* dbeta, void* ws, size_t ws_bytes,
                               const void* relu_bits, void* stream);
/* relu_bits: the bitmap written by the forward pass; when given, `act` is not read (may be NULL). */

/* Max pooling, NHWC bf16, TF 'SAME' padding (out = ceil(in/stride), pad_before = pad_total/2).
 * Replaces tf.layers.max_pooling2d(pool_size=3, strides=2, padding='SAME'),
 * resnet_model.py:636-642.  argmax: one byte per OUTPUT element (window-relative index of the
 * first maximum), consumed by the backward gather; NULL (inference) skips writing it.  channels % 8 == 0. */
RIGL_API int rigl_maxpool_same_forward(const void* x, int n, int h, int w, int c, int ksize, int stride,
                                       void* y, uint8_t* argmax, void* stream);
RIGL_API int rigl_maxpool_same_backward(const void* dy, const uint8_t* argmax, int n, int h, int w, int c,
                                        int ksize, int stride, void* dx, void* stream);

/* ------------------------------------------------------------------------
 * Depthwise 3x3 convolution (stride 1 / 2, explicit padding 1), NHWC bf16, fp32 master weights [C][1][3][3]
 * (flat index c*9 + kh*3 + kw), rounded to bf16 on load; fp32 accumulation.  Replaces
 * depthwise_conv2d_fixed_padding of the reference's MobileNet-v1 (mobilenetv1_model.py:120-153; not a masked
 * op there).  channels % 8 == 0.  x [n,h,w,c], y / dy [n,oh,ow,c] with oh = (h - 1)/stride + 1.
 * ---------------------------------------------------------------------- */
RIGL_API size_t rigl_depthwise3x3_workspace_bytes(int n, int h, int w, int c, int stride);
RIGL_API int rigl_depthwise3x3_fprop(const void* x, const float* weights, int n, int h, int w, int c, int stride,
                                     void* y, void* stream);
RIGL_API int rigl_depthwise3x3_dgrad(const void* dy, const float* weights, int n, int h, int w, int c, int stride,
                                     void* dx, void* stream);
/* dw <- beta * dw + dL/dweights (fp32, deterministic order); beta in {0, 1}. */
RIGL_API int rigl_depthwise3x3_wgrad(const void* x, const void* dy, int n, int h, int w, int c, int stride,
                                     float* dw, float beta, void* ws, size_t ws_bytes, void* stream);

/* 1 to route every conv call through the CUDA-core kernels (debug cross-check). */
RIGL_API int rigl_set_force_simt(int on);

#ifdef __cplusplus
}
#endif
#endif  /* RIGL_B200_H_ */
