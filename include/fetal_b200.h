/*
 * fetal_b200.h — C ABI of libfetalb200.so: the B200-native replacement for the numeric
 * backend underneath the reference's hot path (Keras/TensorFlow under fetal_net.model +
 * fetal_net.metrics, and the NumPy inner loop of fetal_net.prediction.patch_wise_prediction).
 *
 * The reference has no FFI of its own (pure Python; SURVEY.md §8b): the two seams it offers are
 *   (i)  `getattr(fetal_net.model, config['model_name'])(...)` -> Keras-Model duck type
 *        (fetal/train_fetal.py:31-39, fetal_net/training.py:74-75), whose members
 *        `.predict`, `.train_on_batch`/`.fit_generator`, `.evaluate`, `.load_weights`/`.save`
 *        are used at fetal_net/prediction.py:361, fetal_net/training.py:110-124,
 *        fetal/experiments/train_adv.py:227,257;
 *   (ii) `patch_wise_prediction(model, data, patch_shape, overlap_factor, batch_size, ...)`
 *        (fetal_net/prediction.py:118-210).
 * Every entry point below names the reference interface it stands in for. All signatures are
 * plain C: pointers + sizes, no torch / numpy types. Every function returns 0 on success and a
 * negative FM_E* code on failure; `fm_last_error()` returns the message for the calling thread.
 *
 * Threading: one fm_ctx per GPU / process rank; calls on one ctx must come from one host thread
 * at a time (the reference calls model.predict / train_on_batch from the main thread only).
 */
#ifndef FETAL_B200_H
#define FETAL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FM_OK 0
#define FM_EINVAL (-1)   /* bad argument / unsupported shape            */
#define FM_ECUDA (-2)    /* CUDA runtime or driver error                */
#define FM_ENOMEM (-3)   /* device or host allocation failed            */
#define FM_ESTATE (-4)   /* call order violated (e.g. backward w/o fwd) */
#define FM_ECOMM (-5)    /* NCCL error / libnccl not loadable           */

typedef struct fm_ctx fm_ctx;
typedef struct fm_model fm_model;

/* ---- context ------------------------------------------------------------------------------ */

/* Replaces: Keras/TF session creation (implicit in `import keras`; fetal/utils.py:59-66). */
int fm_ctx_create(int device, fm_ctx** out);
int fm_ctx_destroy(fm_ctx* ctx);
const char* fm_last_error(void);
/* SM count / compute capability of the ctx device: out[0]=major, out[1]=minor, out[2]=#SM. */
int fm_ctx_device_info(fm_ctx* ctx, int out[3]);
/* cudaStream_t the model's kernels are launched on (as an integer handle, for event timing). */
uint64_t fm_ctx_stream(fm_ctx* ctx);
int fm_ctx_synchronize(fm_ctx* ctx);
/* Number of kernels this library has launched on ctx since creation (bench `gpu_launches`). */
int64_t fm_ctx_launch_count(fm_ctx* ctx);

/* Per-launch timing (bench.py's roofline leg): when enabled, every kernel launch on ctx is
 * bracketed by CUDA events; record i gives name, out[0]=ms, out[1]=algorithmic FLOPs,
 * out[2]=algorithmic bytes of that launch. Enabling/disabling clears the records. */
int fm_ctx_profile_enable(fm_ctx* ctx, int on);
int fm_ctx_profile_count(fm_ctx* ctx);
int fm_ctx_profile_get(fm_ctx* ctx, int i, char name[48], double out[3]);

/* ---- model -------------------------------------------------------------------------------- */

/* Builder spec. Replaces the kwargs of unet_model_3d (fetal_net/model/unet3d/unet.py:17-20):
 * input_shape=(in_channels,X,Y,Z), depth, n_base_filters, n_labels. pool_size is (2,2,2),
 * deconvolution=False, batch_normalization=False, activation 'sigmoid' (the defaults the
 * reference's train_fetal.py path uses, fetal/train_fetal.py:33-39). */
typedef struct fm_unet3d_spec {
  int32_t in_channels;    /* 1 on the reference's path                       */
  int32_t X, Y, Z;        /* patch extent; each divisible by 2^(depth-1)     */
  int32_t depth;          /* default 4                                       */
  int32_t n_base_filters; /* builder default 32; BASELINE configs use 16     */
  int32_t n_labels;       /* 1                                               */
} fm_unet3d_spec;

/* Replaces: unet_model_3d(...) + model.compile(Adam, loss=dice_coefficient_loss)
 * (fetal_net/model/unet3d/unet.py:40-86). Weights start as zeros: call fm_model_set_weights. */
int fm_model_create_unet3d(fm_ctx* ctx, const fm_unet3d_spec* spec, fm_model** out);
int fm_model_destroy(fm_model* m);

/* Builder switches of unet_model_3d / unet_model_2d beyond the spec (unet3d/unet.py:17-20, unet/unet.py:22-25).
 * FM_UNET_DECONVOLUTION: deconvolution=True - get_up_convolution returns Deconvolution3D / Deconvolution2D(filters =
 * channels of the coarse tensor, kernel_size 2, strides 2) instead of UpSampling (unet3d/unet.py:57-59,132-136). The
 * layer table then holds an "up<d>" layer in front of every "dec<d>a"; its kernel has the Keras Conv3DTranspose
 * layout (2,2,2,Cout,Cin). It runs as ONE 1x1x1 tensor-core convolution to (8 x C) channels (4 x C in 2D) - a k = 2,
 * s = 2 transposed convolution writes every output voxel from exactly one input voxel - plus a depth-to-space
 * shuffle; backward is the reverse shuffle, a 1x1x1 wgrad and a 1x1x1 dgrad.
 * FM_UNET_BATCH_NORMALIZATION: batch_normalization=True - every create_convolution_block is Conv -> BatchNormalization(
 * axis=1) -> ReLU (unet3d/unet.py:102-113). Keras semantics: batch statistics (biased variance, eps 1e-3 under the root)
 * in training passes, moving statistics (momentum 0.99, sample-size-corrected variance) at inference. The layer table
 * lists, behind every block's conv, a "<conv>_norm" pseudo-layer (kernel = gamma, bias = beta) and a "<conv>_moving"
 * pseudo-layer (kernel = moving_mean, bias = moving_variance; never touched by the optimizer). Single-process training
 * only: fm_train_step_dp refuses (the statistics would have to span the global batch). */
#define FM_UNET_DECONVOLUTION 1
#define FM_UNET_BATCH_NORMALIZATION 2
int fm_model_create_unet3d_ex(fm_ctx* ctx, const fm_unet3d_spec* spec, int flags, fm_model** out);

/* Builder spec of the 2D / "2.5D" U-Net. Replaces the kwargs of unet_model_2d
 * (fetal_net/model/unet/unet.py:22-25): input_shape=(H,W,in_channels) with the slices (and the previous-slice
 * truth, fetal_net/generator.py:305-306) as channels; Permute + Conv2D/MaxPooling2D/UpSampling2D stack. */
typedef struct fm_unet2d_spec {
  int32_t H, W;           /* each divisible by 2^(depth-1)                          */
  int32_t in_channels;    /* patch_depth (+ prev_truth_size), 1..16                 */
  int32_t depth;          /* default 4                                              */
  int32_t n_base_filters; /* default 32                                             */
  int32_t n_labels;       /* 1                                                      */
} fm_unet2d_spec;

/* Replaces: unet_model_2d(...) + model.compile (fetal_net/model/unet/unet.py:49-88). Input [B,H,W,in_channels],
 * output [B,H,W,n_labels] (the Permute((3,1,2)) / Permute((2,3,1)) pair of the reference is a layout no-op here:
 * device tensors are channels-last). All entry points below accept either model kind. */
int fm_model_create_unet2d(fm_ctx* ctx, const fm_unet2d_spec* spec, fm_model** out);
int fm_model_create_unet2d_ex(fm_ctx* ctx, const fm_unet2d_spec* spec, int flags, fm_model** out);

/* Builder spec of the Isensee-2017 residual 3D U-Net. Replaces the kwargs of isensee2017_model_3d
 * (fetal_net/model/unet3d/isensee2017.py:15-18). Inference and training (every fm_predict* / fm_patchwise_predict* /
 * fm_train_* / fm_evaluate entry point). The layer table lists every Conv3D followed by its InstanceNormalization
 * pseudo-layer (kernel = gamma, bias = beta). */
typedef struct fm_isensee3d_spec {
  int32_t in_channels;            /* 1                                        */
  int32_t X, Y, Z;                /* each divisible by 2^(depth-1)            */
  int32_t depth;                  /* default 5                                */
  int32_t n_base_filters;         /* default 16                               */
  int32_t n_segmentation_levels;  /* default 1; BASELINE config 3 uses 3      */
  int32_t n_labels;               /* 1                                        */
} fm_isensee3d_spec;
int fm_model_create_isensee3d(fm_ctx* ctx, const fm_isensee3d_spec* spec, fm_model** out);

/* Builder spec of the 2D Isensee-2017 net. Replaces the kwargs of isensee2017_model
 * (fetal_net/model/unet/isensee.py:14-16; config_utils.py:66-69 selects it as model_name for 2D runs):
 * input_shape=(H,W,in_channels) with the slices as channels, Conv2D 3x3 / 1x1 blocks with InstanceNormalization +
 * LeakyReLU, strides (2,2) between levels, SpatialDropout2D in the context modules, UpSampling2D, 1x1 heads.
 * n_segmentation_levels = the number of heads that reach the output: with the reference's default summation=False only
 * the finest head does (pass 1); with summation=True the coarser heads are upsampled and added (pass the builder's
 * n_segmentation_levels). Input [B,H,W,in_channels], output [B,H,W,1]. */
typedef struct fm_isensee2d_spec {
  int32_t H, W;                   /* each divisible by 2^(depth-1)            */
  int32_t in_channels;            /* 1..16                                    */
  int32_t depth;                  /* default 5                                */
  int32_t n_base_filters;         /* default 16                               */
  int32_t n_segmentation_levels;  /* heads summed into the output (see above) */
  int32_t n_labels;               /* 1                                        */
} fm_isensee2d_spec;
int fm_model_create_isensee2d(fm_ctx* ctx, const fm_isensee2d_spec* spec, fm_model** out);

/* Layer table, Keras creation order (conv3d_1 ... conv3d_15). */
int fm_model_num_layers(fm_model* m);
/* info[0]=cin, info[1]=cout, info[2]=kernel extent code (33: 3x3x3, 31: 3x3, 11: 1x1[x1], 0: InstanceNormalization gamma/beta), info[3]=param offset
 * of kernel, info[4]=param offset of bias (offsets into the flat fp32 parameter buffer). */
int fm_model_layer_info(fm_model* m, int layer, char name[32], int64_t info[5]);
int64_t fm_model_num_params(fm_model* m);

/* Replaces: Model.set_weights / load_weights (fetal/train_fetal.py:43, fetal_net/training.py:83).
 * `kernel` is in **Keras layout** (k0,k1,k2,Cin,Cout) fp32, `bias` (Cout). Host pointers. */
int fm_model_set_weights(fm_model* m, int layer, const float* kernel, const float* bias);
/* Replaces: Model.get_weights / save (fetal_net/training.py:30-32 ModelCheckpoint). */
int fm_model_get_weights(fm_model* m, int layer, float* kernel, float* bias);
/* Gradients of the last backward pass, Keras layout (test hook; TF autodiff has no equivalent). */
int fm_model_get_grads(fm_model* m, int layer, float* kernel, float* bias);
/* Resets Adam moments and the iteration counter (a fresh model.compile). */
int fm_model_reset_optimizer(fm_model* m);
/* Optimizer state of one layer, Keras layout like the weights: Adam first / second moments (kernel, bias) and the step
 * counter. Replaces the optimizer part of Keras' model.save() / load_model() that the reference's resume path relies on
 * (load_old_model(get_last_model_path(...)), fetal/train_fetal.py:25-28, fetal_net/training.py:45-65). */
int fm_model_get_adam_state(fm_model* m, int layer, float* m_kernel, float* m_bias, float* v_kernel, float* v_bias);
int fm_model_set_adam_state(fm_model* m, int layer, const float* m_kernel, const float* m_bias, const float* v_kernel,
                            const float* v_bias);
int fm_model_get_iterations(fm_model* m);
int fm_model_set_iterations(fm_model* m, int iterations);
/* Replaces: the `dropout_rate` kwarg of isensee2017_model_3d -> SpatialDropout3D(rate) between the two convs of
 * every context module (fetal_net/model/unet3d/isensee2017.py:15,51,103-105). Active in training passes only
 * (fm_train_*), one keep/scale factor per (sample, channel) drawn from a counter-based hash of (seed, step, level);
 * rate 0 (the default here) switches it off. Plain U-Net models ignore it. */
int fm_model_set_dropout(fm_model* m, float rate, uint64_t seed);
/* No counterpart in the reference (Keras picks its own conv algorithms). fast = 0 (default): predict / evaluate /
 * patch_wise_prediction issue their tensor-core MMAs in a fixed order - the same input gives the same bits on every
 * run. fast = 1: inference takes the three-issuer mode of the training passes (about a quarter more conv throughput);
 * results then differ in the last bf16 bit from run to run, exactly like a training pass. Tolerances against the
 * oracle are unaffected. FETAL_B200_DETERMINISTIC=1 overrides it. */
int fm_model_set_inference_mode(fm_model* m, int fast);
/* Replaces: the `loss_function` argument of the builders, looked up by getattr(fetal_net.metrics, config['loss'])
 * (fetal/train_fetal.py:31, fetal_net/training.py:51-58):
 *   kind 0  dice_coefficient_loss                       (fetal_net/metrics.py:31-32)                    [default]
 *   kind 1  dice_and_xent(y_true, y_pred, xent_weight)   = -dice + xent_weight * mean(binary_crossentropy)
 *                                                        (fetal_net/metrics.py:68-78)
 *   kind 2  dice_and_xent_mask(weight_mask, xent_weight, dist_sigma): the cross-entropy of every voxel is weighted by
 *           exp(-weight_mask / dist_sigma) (fetal_net/metrics.py:89-95); the mask is the model's second input
 *           (`mask_shape`, fetal_net/model/unet3d/isensee2017.py:85-88) and is handed over per step with
 *           fm_model_set_weight_mask.
 * The reported loss (out_metrics[0]) becomes the combined one; out_metrics[3] stays the soft Dice coefficient, which
 * Keras appends to the metrics when the loss is not the Dice loss (unet3d/unet.py:82-83, isensee2017.py:82-83). In a
 * data-parallel step the cross-entropy sum travels in the same all-reduce as the Dice sums (9 doubles). */
int fm_model_set_loss(fm_model* m, int kind, float xent_weight, float dist_sigma);
/* Replaces: the second element of the `[x, mask]` input list a two-input Keras model is trained on
 * (isensee2017.py:85-88): float32 [batch, X, Y, Z] distances, uploaded for the next training / evaluation call of
 * that batch size and kept until replaced. FM_EINVAL unless the loss kind is 2. */
int fm_model_set_weight_mask(fm_model* m, const float* mask, int batch);

/* ---- inference ---------------------------------------------------------------------------- */

/* Replaces: model.predict(ndarray[B,Cin,X,Y,Z]) -> float32 [B,n_labels,X,Y,Z]
 * (fetal_net/prediction.py:354-361). Host pointers; H2D + forward + D2H inside the call.
 * With n_labels == 1 the channels-first and channels-last output layouts coincide. */
int fm_predict(fm_model* m, const float* x, int batch, float* y);

/* Page-locked host memory: a result array allocated here receives the device->host copies of fm_patchwise_predict
 * directly (no staging copy, no first-touch page faults); fetal_net.prediction keeps a pool of such arrays behind the
 * NumPy arrays it returns (the reference returns fresh np.zeros arrays, prediction.py:174-175). */
int fm_host_alloc(size_t bytes, void** out);
int fm_host_free(void* p);

/* Sliding-window plan. Replaces get_set_of_patch_indices_full + the overlap arithmetic
 * (fetal_net/prediction.py:88-95,135-137,161-163). `padded` is the extent of the padded volume,
 * `pred` the model's prediction extent (== patch for the 3D models). Writes up to `cap` corner
 * triples (x-major product order) to `out_idx` and the total count to `out_n`. Pure host code. */
int fm_patch_plan(const int32_t padded[3], const int32_t patch[3], const int32_t pred[3],
                  double overlap_factor, int32_t* out_idx, int64_t cap, int64_t* out_n);

/* Replaces the body of patch_wise_prediction (fetal_net/prediction.py:161-210): gather patches from the
 * (virtually padded) volume, run the network, overlap-add in float64 in patch order, divide by the int count.
 * `vol` is the UNPADDED float32 volume [X,Y,Z] (host); padding is virtual: `halo_pad` = {before,after} x 3 axes
 * of the first np.pad (prediction.py:138-141, filled with pad_value[0]) and `fit_pad` likewise for pad_for_fit
 * (prediction.py:142-146, filled with pad_value[1]). 3D models predict the whole patch (halo_pad all zero);
 * 2D models take patches (H, W, patch_depth), predict (H, W, 1) and need the z halo (ceil,floor)((patch_depth-1)/2).
 * `idx` are the n patch corners from fm_patch_plan (coordinates in the padded volume).
 * `truth` (host float32 [X,Y,Z], may be NULL): previous-slice conditioning of the 2.5D path — the slices
 * [z + prev_truth_index, +prev_truth_size) of the identically padded (with 0) truth volume are appended as input
 * channels (prediction.py:106-110,148-156).
 * `out` receives float64 [X+fit, Y+fit, Z+fit, n_labels] (host) - the caller crops pad_for_fit
 * (prediction.py:198-207). `batch` = patches per network launch (reference default 5; result is batch-invariant).
 * `shard_rank`/`shard_count`: this rank handles patches [rank*n/count, (rank+1)*n/count) and `out` then holds
 * the partial SUM (not divided) when shard_count > 1; use shard 0 of 1 for the single-GPU drop-in.
 * `out_count` (int16, same extent, may be NULL) receives the full count map. */
int fm_patchwise_predict(fm_model* m, const float* vol, const int32_t vol_dims[3],
                         const int32_t halo_pad[6], const int32_t fit_pad[6],
                         const double pad_value[2], const int32_t* idx, int64_t n, int batch,
                         int shard_rank, int shard_count, const float* truth, int prev_truth_index,
                         int prev_truth_size, double* out, int16_t* out_count);

/* Reassembly alone (test hook for bit-exactness): `preds` float32 [n,P0,P1,P2,C] (host) are
 * overlap-added exactly as fetal_net/prediction.py:188-193,210 does. */
int fm_reassemble(fm_ctx* ctx, const float* preds, const int32_t* idx, int64_t n,
                  const int32_t pred_shape[3], int channels, const int32_t out_dims[3],
                  double* out, int16_t* out_count);
/* Patch gather alone (test hook): replaces get_patch_from_3d_data on the padded volume
 * (fetal_net/utils/patches.py:57-72) - out float32 [n,P0,P1,P2] (host). */
int fm_gather_patches(fm_ctx* ctx, const float* vol, const int32_t vol_dims[3],
                      const int32_t halo_pad[6], const int32_t fit_pad[6],
                      const double pad_value[2], const int32_t* idx, int64_t n,
                      const int32_t patch[3], float* out);

/* ---- post-processing ---------------------------------------------------------------------- */

/* Replaces: postprocess_prediction(pred, gaussian_std, threshold, fill_holes, connected_component)
 * (fetal_net/postprocess.py:13): scipy.ndimage.gaussian_filter (mode 'reflect', truncate 4, axes 0, 1, 2, each pass
 * rounded to the input dtype), `> threshold` in the input dtype, binary_fill_holes (6-connected background) and the
 * largest 6-connected component (lowest first voxel in C order on a tie), bit-exact with scipy.
 * `weights` are the 2 radius + 1 normalised Gaussian weights as scipy computes them with numpy.exp (so they are taken
 * from the caller, not recomputed here); radius 0 with weight 1.0 is the identity (sigma 0). */
typedef struct fm_postprocess_spec {
  int32_t radius;
  const double* weights; /* 2 radius + 1, host */
  double threshold;
  int32_t fill_holes;
  int32_t connected_component;
} fm_postprocess_spec;
#define FM_DTYPE_FLOAT32 0
#define FM_DTYPE_FLOAT64 1
/* `pred` host [dims] of `dtype`, `mask` host uint8 [dims]. `n_components` (may be NULL) receives the number of
 * foreground components before the largest one is selected, or -1 when connected_component is 0. With
 * connected_component set and no foreground the mask is all zero and n_components 0 (the reference raises).
 * Volumes of up to 2^31 - 1 voxels. */
int fm_postprocess(fm_ctx* ctx, const void* pred, int dtype, const int32_t dims[3], const fm_postprocess_spec* spec,
                   uint8_t* mask, int64_t* n_components);
/* fm_patchwise_predict (single GPU, n_labels 1) followed by fm_postprocess of its cropped result, without the float64
 * map leaving the device: `mask` host uint8 [vol_dims]; `prob` (may be NULL) receives exactly what `out` of
 * fm_patchwise_predict would (the padded [X+fit, Y+fit, Z+fit, 1] float64 map). */
int fm_patchwise_segment(fm_model* m, const float* vol, const int32_t vol_dims[3], const int32_t halo_pad[6],
                         const int32_t fit_pad[6], const double pad_value[2], const int32_t* idx, int64_t n, int batch,
                         const float* truth, int prev_truth_index, int prev_truth_size,
                         const fm_postprocess_spec* spec, uint8_t* mask, double* prob, int64_t* n_components);
/* Gaussian filter alone (test hook): `out` host [dims] of `dtype` = scipy.ndimage.gaussian_filter(in, sigma). */
int fm_op_gaussian3d(fm_ctx* ctx, const void* in, int dtype, const int32_t dims[3], int radius, const double* weights,
                     void* out);

/* ---- training ----------------------------------------------------------------------------- */

/* Replaces: model.train_on_batch(x, y) as driven by fit_generator (fetal_net/training.py:110-124):
 * forward, soft-Dice loss (fetal_net/metrics.py:11-15,31-32), backward, Keras-2 Adam.
 * x [B,Cin,X,Y,Z], t [B,n_labels,X,Y,Z] float32 host. out_metrics[4] = loss, binary_accuracy,
 * vod_coefficient, dice_coefficient (the Keras metrics of unet3d/unet.py:81-83). */
/* Pipelining: when x and t are pinned (page-locked) host buffers, the upload goes through two device staging buffers
 * on a copy stream and the call returns as soon as the Dice statistics of THIS step's forward pass are on the host;
 * backward, Adam and the weight repack keep running and are stream-ordered before every later call on the model
 * (predict, get_weights, the next step), whose upload then overlaps them. x / t may be reused when the call returns.
 * Pageable buffers (plain NumPy batches, what the reference's generator yields) are first copied by a few host threads
 * into pinned ping-pong buffers owned by the model and then take the same route; FETAL_B200_NO_PIPELINE=1 selects the
 * fully synchronous route. */
int fm_train_step(fm_model* m, const float* x, const float* t, int batch, float lr,
                  float out_metrics[4]);

/* The same step split at its two exchange points, for data-parallel training (one process per
 * GPU). fm_train_forward leaves the LOCAL sums {sum(t*p), sum(t), sum(p), sum(tb*pb), sum(tb),
 * sum(pb), sum(correct), count} as 8 float64 at fm_model_loss_sums(); the caller all-reduces
 * them (SUM) so every rank back-propagates the GLOBAL Dice (metrics.py flattens the whole
 * batch), then fm_train_backward launches the backward pass; the caller all-reduces (SUM) the
 * flat fp32 gradient buffer fm_model_grad_buffer() bucket by bucket — fm_stream_wait_bucket
 * makes a foreign stream wait until bucket `b`'s gradients are final — and finally
 * fm_train_apply runs Adam after making the compute stream wait on `after_stream`. */
int fm_train_forward(fm_model* m, const float* x, const float* t, int batch);
int fm_train_backward(fm_model* m);
int fm_train_apply(fm_model* m, float lr, uint64_t after_stream, float out_metrics[4]);
/* Optional early return for the split step (data-parallel trainers): call fm_train_metrics_async after the
 * all-reduce of the statistics has been queued on the compute stream (it queues their copy to pinned host memory),
 * run fm_train_backward / the gradient all-reduces / fm_train_apply(..., NULL), and finish with
 * fm_train_metrics_wait, which blocks only until that copy has landed: backward, Adam and the repack keep running
 * and are stream-ordered before every later call on the model, so the next step's upload (pinned inputs) overlaps
 * them. Replaces nothing in the reference (Keras' train_on_batch is synchronous); same numbers as the metrics
 * argument of fm_train_apply. */
int fm_train_metrics_async(fm_model* m);
int fm_train_metrics_wait(fm_model* m, float out_metrics[4]);
int fm_model_loss_sums(fm_model* m, uint64_t* dev_ptr);               /* 8 x float64, device */
int fm_model_grad_buffer(fm_model* m, uint64_t* dev_ptr, int64_t* n); /* n x float32, device */
int fm_model_num_buckets(fm_model* m);
int fm_model_bucket_range(fm_model* m, int bucket, int64_t* offset, int64_t* count);
int fm_stream_wait_bucket(fm_model* m, uint64_t stream, int bucket);
/* Device-resident variants (x, t already float32 in HBM): what bench.py's `value` times. */
int fm_train_step_device(fm_model* m, uint64_t x_dev, uint64_t t_dev, int batch, float lr,
                         float out_metrics[4]);
int fm_predict_device(fm_model* m, uint64_t x_dev, int batch, uint64_t y_dev);

/* Replaces: model.evaluate / test_on_batch (validation loop of fit_generator). */
int fm_evaluate(fm_model* m, const float* x, const float* t, int batch, float out_metrics[4]);

/* ---- training patches cut on the device ---------------------------------------------------------------------------
 * Replaces the inner loop of the reference's training generator (fetal_net/generator.py:222-348: add_data ->
 * extract_patch -> get_patch_from_3d_data, convert_data) for cases that fit in HBM: the data / truth volumes are uploaded
 * once (float32, the dtype Keras feeds), the host keeps drawing the case order, the random corners and the skip-blank
 * rejections with the reference's own np.random call sequence (fetal_net/device_sampler.py), and one kernel cuts the
 * whole batch - data patch, target slice(s) at truth_index, previous-truth slice(s) at prev_truth_index appended as
 * extra input channels (generator.py:305-306), out-of-range slices edge-replicated (utils/patches.py:75-91) - into the
 * model's input / target buffers. No host<->device traffic per step besides 32 bytes of arguments per sample. */
typedef struct fm_volset fm_volset;
/* Optional per-sample cheap augmentations applied while cutting (not the reference's nilearn / imgaug pipeline):
 * flip bit 0 / 1 / 2 = x / y / z (data, previous truth and target alike), data *= intensity_scale, data += noise_sigma *
 * N(0,1) (counter-based hash of noise_seed). A NULL pointer means none. */
typedef struct fm_sample_aug {
  uint32_t flip;
  float intensity_scale;
  float noise_sigma;
  uint32_t noise_seed;
} fm_sample_aug;
int fm_volset_create(fm_ctx* ctx, int n_cases, fm_volset** out);
int fm_volset_destroy(fm_volset* s);
/* data, truth: host float32 [X,Y,Z] of case `index` (data_file.root.data[index] / .truth[index]). */
int fm_volset_set_case(fm_volset* s, int index, const float* data, const float* truth, const int32_t dims[3]);
/* Test hook: cuts `batch` samples (case[b], corner[b][3]) into host buffers x_out [B,P0,P1,P2+prev_truth_size] and
 * y_out [B,P0,P1,truth_size]. */
int fm_volset_gather(fm_volset* s, const int32_t* cases, const int32_t* corners, const fm_sample_aug* aug, int batch,
                     const int32_t patch[3], int truth_index, int truth_size, int prev_truth_index, int prev_truth_size,
                     float* x_out, float* y_out);
/* Replaces: next(generator) + model.train_on_batch(x, y) for one batch whose samples are cut on the device. The patch
 * extent follows from the model (3D: (X, Y, Z), truth_size must be Z and prev_truth_size 0; 2D: (H, W, in_channels -
 * prev_truth_size), truth_size 1). Data-parallel when the ctx has a communicator (like fm_train_step_dp). */
int fm_train_step_sampled(fm_model* m, fm_volset* s, const int32_t* cases, const int32_t* corners,
                          const fm_sample_aug* aug, int batch, int truth_index, int truth_size, int prev_truth_index,
                          int prev_truth_size, float lr, float out_metrics[4]);

/* ---- data parallelism (one process per GPU; NCCL over NVLink 5 / NVSwitch) -----------------------------------
 * The reference is single-process (fetal_net/training.py:115-117: workers=1, use_multiprocessing=False); these entry
 * points are the multi-GPU extension of the same two calls (train_on_batch, patch_wise_prediction). libnccl.so.2 is
 * resolved with dlopen at the first call (FETAL_B200_NCCL_LIB overrides the name). The 128-byte id is created on one
 * rank and carried to the others by the host program (torch.distributed store, MPI, a file ...). */
#define FM_COMM_UID_BYTES 128
int fm_comm_unique_id(uint8_t out[FM_COMM_UID_BYTES]);
int fm_comm_init(fm_ctx* ctx, int rank, int nranks, const uint8_t uid[FM_COMM_UID_BYTES]);
int fm_comm_destroy(fm_ctx* ctx);
/* out[0] = rank, out[1] = ranks (1 without a communicator), out[2] = NCCL version code. */
int fm_comm_info(fm_ctx* ctx, int out[3]);
/* on = 0 turns every collective of this ctx into a no-op (bench.py measures the EXPOSED communication time of a
 * step as the difference; results are then meaningless). */
int fm_comm_enable(fm_ctx* ctx, int on);
/* cudaStream_t of the gradient all-reduces (integer handle, for event timing). */
uint64_t fm_comm_stream(fm_ctx* ctx);
/* Average duration of `iters` in-place fp32 SUM all-reduces of `bytes` on the communication stream. */
int fm_comm_allreduce_bench(fm_ctx* ctx, int64_t bytes, int iters, float* ms_per_iter);
/* Copies rank `root`'s parameters (and Adam state) to every rank: the replicas start identical. */
int fm_comm_broadcast_params(fm_model* m, int root);

/* Replaces: model.train_on_batch(x, y) on THIS rank's shard of the global batch. Forward; all-reduce of the 8 Dice
 * sums so that every rank back-propagates the GLOBAL soft Dice (fetal_net/metrics.py:11-15 flattens the batch axis);
 * backward; SUM all-reduce of the flat fp32 gradient buffer in fm_model_num_buckets() contiguous buckets on the
 * communication stream, each as soon as its last layer's gradients are final (overlapping the rest of backward);
 * the identical Keras-Adam step on every rank. out_metrics are the GLOBAL loss / accuracy / VOD / Dice. With pinned
 * x / t the call returns when the statistics are on the host (like fm_train_step). Without a communicator it is
 * fm_train_step. */
int fm_train_step_dp(fm_model* m, const float* x, const float* t, int batch, float lr, float out_metrics[4]);

/* fm_patchwise_predict with the patch list sharded contiguously over the ranks of the ctx communicator: every rank
 * overlap-adds its patches into a private float64 partial sum on its GPU, one ncclReduce to `root`, which divides by
 * the (analytic, never communicated) counts and copies the result to `out`; `out` / `out_count` are ignored on the
 * other ranks (may be NULL). */
int fm_patchwise_predict_dp(fm_model* m, const float* vol, const int32_t vol_dims[3], const int32_t halo_pad[6],
                            const int32_t fit_pad[6], const double pad_value[2], const int32_t* idx, int64_t n,
                            int batch, int root, const float* truth, int prev_truth_index, int prev_truth_size,
                            double* out, int16_t* out_count);

/* ---- per-op hooks (parity tests call the kernels one at a time through these) --------------
 * All pointers are HOST pointers; tensors are channels-last (NDHWC) fp32 on the host and are
 * converted to the device storage type (bf16) inside the call. Each replaces one Keras layer
 * call of create_convolution_block / unet_model_3d (fetal_net/model/unet3d/unet.py:51,61,102,138)
 * or its TF autodiff counterpart. `impl`:
 *   0 = tcgen05 per-tap tensor-core kernel;
 *   1 = SIMT check kernel;
 *   2 = plane-marching kernel, bit-reproducible issue order (predict / evaluate); for wgrad, the marching weight
 *       gradient with the bias gradient folded in;
 *   3 = plane-marching kernel in the issue order of training passes (fprop / dgrad; wgrad takes the SIMT kernel).
 */
int fm_op_conv3d_fprop(fm_ctx* ctx, int impl, const float* x, const float* x2, const float* w_keras,
                       const float* bias, int N, int X, int Y, int Z, int C1, int C2, int Cout,
                       int ksize, int relu, float* y);
int fm_op_conv3d_dgrad(fm_ctx* ctx, int impl, const float* dy, const float* w_keras,
                       const float* mask, int N, int X, int Y, int Z, int Cin, int Cout,
                       float* dx);
int fm_op_conv3d_wgrad(fm_ctx* ctx, int impl, const float* x, const float* dy, int N, int X, int Y,
                       int Z, int Cin, int Cout, float* dw_keras, float* dbias);
/* First Conv3D of the network on the single-channel float32 input x [N,X,Y,Z] (create_convolution_block on the
 * (1, X, Y, Z) input, unet.py:102): y [N,X,Y,Z,Cout] = act(conv + bias) when y != NULL; the weight gradient
 * dw_keras (3,3,3,1,Cout) for dy [N,X,Y,Z,Cout] when both are != NULL. */
int fm_op_conv3d_first(fm_ctx* ctx, const float* x, const float* w_keras, const float* bias, int N, int X, int Y, int Z,
                       int Cout, int relu, float* y, const float* dy, float* dw_keras);
/* Decoder convolution Conv3D(3x3x3, 'same') over concatenate([UpSampling3D(2)(coarse), skip], axis=1)
 * (fetal_net/model/unet3d/unet.py:59-62,138 with get_up_convolution's UpSampling3D) computed WITHOUT the upsampled
 * tensor: per parity class of the fine voxel the 27 taps over the upsampled source collapse into 8 taps over the coarse
 * tensor with summed weights (3.4x fewer MACs on that source). Channels-last float32 in/out, bf16 arithmetic inside.
 * coarse [N,X/2,Y/2,Z/2,Cc], skip [N,X,Y,Z,Cs], w_keras (3,3,3,Cc+Cs,Cout), y / dy [N,X,Y,Z,Cout]. */
int fm_op_conv3d_up_fprop(fm_ctx* ctx, const float* coarse, const float* skip, const float* w_keras, const float* bias,
                          int N, int X, int Y, int Z, int Cc, int Cs, int Cout, int relu, float* y);
/* Its backward towards the coarse tensor: dcoarse [N,X/2,Y/2,Z/2,Cc] (ReLU-masked by coarse > 0 when apply_mask) and the
 * weight gradient of the up-source channels dw_up_keras (3,3,3,Cc,Cout); either output may be NULL. */
int fm_op_conv3d_up_bwd(fm_ctx* ctx, const float* coarse, const float* dy, const float* w_keras, int N, int X, int Y,
                        int Z, int Cc, int Cs, int Cout, int apply_mask, float* dcoarse, float* dw_up_keras);

int fm_op_maxpool3d(fm_ctx* ctx, const float* x, int N, int X, int Y, int Z, int C, float* y);
int fm_op_maxpool3d_bwd(fm_ctx* ctx, const float* x, const float* dy, const float* dskip, int N,
                        int X, int Y, int Z, int C, float* dx);
int fm_op_upsample3d(fm_ctx* ctx, const float* x, int N, int X, int Y, int Z, int C, float* y);
int fm_op_upsample3d_bwd(fm_ctx* ctx, const float* dy, const float* act, int N, int X, int Y, int Z,
                         int C, float* dx);
int fm_op_dice(fm_ctx* ctx, const float* p, const float* t, int64_t n, double sums[8],
               float* dloss_dp);
/* dice_and_xent / dice_and_xent_mask (fetal_net/metrics.py:68-95) on probabilities p: sums[0..7] as fm_op_dice,
 * sums[8] = sum_i w_i * binary_crossentropy(t_i, p_i), w_i = exp(-mask_i / dist_sigma) (1 when mask == NULL);
 * dloss_dz (optional) = d(-dice + xent_weight * sums[8] / n) / d(logit) through the sigmoid. */
int fm_op_dice_xent(fm_ctx* ctx, const float* p, const float* t, const float* mask, int64_t n, float xent_weight,
                    float dist_sigma, double sums[9], float* dloss_dz);
int fm_op_adam(fm_ctx* ctx, float* p, const float* g, float* mm, float* vv, int64_t n,
               int iterations, float lr);

#ifdef __cplusplus
}
#endif
#endif /* FETAL_B200_H */
