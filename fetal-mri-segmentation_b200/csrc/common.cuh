// common.cuh — shared host/device helpers for libfetalb200 (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/fetal_b200.h"

typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
void fm_set_error(const char* fmt, ...);

#define FM_CUDA(expr)                                                                         \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      fm_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));     \
      return FM_ECUDA;                                                                        \
    }                                                                                         \
  } while (0)

#define FM_CHECK(cond, code, ...)                                                             \
  do {                                                                                        \
    if (!(cond)) {                                                                            \
      fm_set_error(__VA_ARGS__);                                                              \
      return (code);                                                                          \
    }                                                                                         \
  } while (0)

#define FM_TRY(expr)                                                                          \
  do {                                                                                        \
    int _r = (expr);                                                                          \
    if (_r != FM_OK) return _r;                                                               \
  } while (0)

struct ProfRec {
  const char* name;
  double flops, bytes;
  cudaEvent_t e0, e1;
};

struct fm_ctx {
  int device = 0;
  // optional per-launch timing (fm_ctx_profile_*): CUDA events around every kernel launch
  bool profile = false;
  std::vector<ProfRec> prof;
  int sm_major = 0, sm_minor = 0, num_sms = 0;
  cudaStream_t stream = nullptr;
  // side stream for host->device copies that the head of the compute stream does not need yet (training targets)
  cudaStream_t copy_stream = nullptr;
  // device->host copies of finished output slabs (patch-wise inference) run on their own stream, so that they never
  // hold back the next slab's upload
  cudaStream_t d2h_stream = nullptr;
  cudaEvent_t copy_fence = nullptr, copy_done = nullptr;
  int64_t launches = 0;
  // scratch for deterministic two-stage reductions
  double* red_scratch = nullptr;  // [kRedScratchRows][8] per-block partial loss statistics
  // pinned staging for host<->device copies
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
  // data-parallel communicator (comm.cu): ncclComm_t, its side stream (gradient buckets overlap backward) and an event
  void* comm = nullptr;
  int comm_rank = 0, comm_size = 1;
  bool comm_enabled = true;  // false: collectives are skipped (bench.py measures the exposed communication time)
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t comm_ev = nullptr;
  // device workspace of the post-processing kernels (postprocess.cu), grown on demand
  void* pp_ws = nullptr;
  size_t pp_ws_bytes = 0;
};

// sampler.cu: cuts a batch of training samples out of device-resident cases into device buffers
int sampler_gather_device(fm_volset* s, const int32_t* cases, const int32_t* corners, const fm_sample_aug* aug, int batch,
                          const int32_t patch[3], int truth_index, int truth_size, int prev_truth_index,
                          int prev_truth_size, float* x_dev, float* y_dev);

// comm.cu: in-place SUM collectives on the ctx communicator (no-ops without one); dtype 0 = float32, 1 = float64
int comm_allreduce(fm_ctx* ctx, void* buf, size_t count, int dtype, cudaStream_t stream);
int comm_reduce(fm_ctx* ctx, void* buf, size_t count, int dtype, int root, cudaStream_t stream);
int comm_broadcast(fm_ctx* ctx, void* buf, size_t count, int dtype, int root, cudaStream_t stream);

int fm_ctx_pinned(fm_ctx* ctx, size_t bytes, void** out);

// Programmatic dependent launch: the kernel may be scheduled while its stream predecessor drains, runs its
// prologue (barrier init, TMEM allocation, resident-weight loads), and blocks in `griddepcontrol.wait` (tcp::pdl_wait)
// before it touches anything the predecessor wrote. FETAL_B200_NO_PDL=1 launches it as a plain kernel.
// first statement of a simple kernel launched through launch_pdl: wait for the predecessor, then let the successor in
#define FM_PDL_SYNC()                                              \
  do {                                                             \
    asm volatile("griddepcontrol.wait;" ::: "memory");             \
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); \
  } while (0)

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                     Args&&... args) {
  static const bool off = [] {
    const char* e = getenv("FETAL_B200_NO_PDL");
    return e && e[0] == '1';
  }();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = off ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Kernel-extent code used by all conv launchers: 3 = 3x3x3, 1 = 1x1x1, 31 = 3x3x1 (Conv2D on a Z = 1 volume:
// the 2.5D U-Net, fetal_net/model/unet/unet.py:103). Tap index = (kx * kxy + ky) * kz + kzi.
// 2 = 2x2x2 and 21 = 2x2x1: the stride-2 transposed convolutions (Deconvolution3D / Deconvolution2D,
// get_up_convolution(deconvolution=True), unet3d/unet.py:132-136) - tap = parity class of the output voxel.
__host__ __device__ static inline int kext_xy(int kcode) { return kcode == 31 ? 3 : (kcode == 21 ? 2 : kcode); }
__host__ __device__ static inline int kext_z(int kcode) { return (kcode == 31 || kcode == 21) ? 1 : kcode; }
__host__ __device__ static inline int kext_taps(int kcode) { return kext_xy(kcode) * kext_xy(kcode) * kext_z(kcode); }

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------------------------------
// Work split of the plane-marching kernels. A problem is `cols` columns (sample, y tile, z tile) of X planes each; a CTA
// marches along x inside a column. Every column is cut into nxc chunks of xchunk planes; work unit u = chunk * cols +
// column, CTA r of G takes units r, r + G, ... - a wave of G units covers neighbouring columns at the SAME x range, so
// the y / z halos they share are re-read from L2 (DRAM traffic = algorithmic bytes); nxc is chosen on the host for wave
// efficiency. `it` counts the CTA's units from 0. Returns false when the CTA is done.
// ------------------------------------------------------------------------------------------
struct PlaneSplit {
  int X, cols, nxc, xchunk;
};
#ifdef __CUDACC__
__device__ __forceinline__ bool plane_split_next(const PlaneSplit& s, int rank, int G, int it, int& col, int& xa, int& xb) {
  const int u = rank + it * G;
  if (u >= s.cols * s.nxc) return false;
  const int xc = u / s.cols;
  col = u - xc * s.cols;
  xa = xc * s.xchunk;
  xb = min(s.X, xa + s.xchunk);
  return true;
}
#endif
// host side: fills `s` for `G` CTAs (halo = planes a chunk re-loads, in units of a plane's cost)
static inline void plane_split_setup(PlaneSplit* s, int cols, int X, int G, double halo) {
  s->X = X;
  s->cols = cols;
  double best = -1.0;
  int best_nxc = 1;
  for (int nxc = 1; nxc <= 32; nxc *= 2) {
    const int xc = (X + nxc - 1) / nxc;
    if (xc < 4 && nxc > 1) break;
    const int units = cols * ((X + xc - 1) / xc);
    const int waves = (units + G - 1) / G;
    const double eff = (double)units / ((double)waves * G) * (double)xc / ((double)xc + halo);
    if (eff > best) {
      best = eff;
      best_nxc = nxc;
    }
  }
  s->xchunk = (X + best_nxc - 1) / best_nxc;
  s->nxc = (X + s->xchunk - 1) / s->xchunk;
}

// Per-launch profiling hooks: `flops` / `bytes` are the ALGORITHMIC figures of the launch.
int fm_prof_begin(fm_ctx* ctx, const char* name, double flops, double bytes);
int fm_prof_end(fm_ctx* ctx);
struct ProfScope {
  fm_ctx* ctx;
  ProfScope(fm_ctx* c, const char* name, double flops, double bytes) : ctx(c) {
    if (ctx->profile) fm_prof_begin(ctx, name, flops, bytes);
  }
  ~ProfScope() {
    if (ctx->profile) fm_prof_end(ctx);
  }
};

// Launch-error check that also counts the launch (bench.py reports gpu_launches from this).
#define FM_LAUNCH_OK(ctx)                                                                     \
  do {                                                                                        \
    (ctx)->launches++;                                                                        \
    cudaError_t _e = cudaGetLastError();                                                      \
    if (_e != cudaSuccess) {                                                                  \
      fm_set_error("%s:%d: kernel launch failed: %s", __FILE__, __LINE__,                     \
                   cudaGetErrorString(_e));                                                   \
      return FM_ECUDA;                                                                        \
    }                                                                                         \
  } while (0)

// ------------------------------------------------------------------------------------------
// tensor descriptors (device storage is channels-last: [N][X][Y][Z][C], C contiguous)
// ------------------------------------------------------------------------------------------
struct Dims5 {
  int N, X, Y, Z, C;
  int64_t voxels() const { return (int64_t)N * X * Y * Z; }
  int64_t elems() const { return voxels() * C; }
};

// ------------------------------------------------------------------------------------------
// kernel launch wrappers implemented across the .cu files (all asynchronous on ctx->stream)
// ------------------------------------------------------------------------------------------

// bandwidth.cu
int k_cast_f32_to_bf16(fm_ctx*, const float* in, bf16* out, int64_t n);
int k_cast_bf16_to_f32(fm_ctx*, const bf16* in, float* out, int64_t n);
// pz = pooling factor along z: 2 (MaxPooling3D / UpSampling3D) or 1 (the 2D layers of the 2.5D U-Net)
int k_maxpool3d_fwd(fm_ctx*, const bf16* x, bf16* y, Dims5 in, int pz = 2);
// dx = relu'(x) * ( dskip(optional) + route(dy) ): fused MaxPooling3D backward + skip-gradient add
int k_maxpool3d_bwd(fm_ctx*, const bf16* x, const bf16* dy, const bf16* dskip, bf16* dx, Dims5 in,
                    int relu_mask, int pz = 2);
int k_upsample3d_fwd(fm_ctx*, const bf16* x, bf16* y, Dims5 in, int pz = 2);
// dx[v] = (act? act[v]>0 : 1) * sum_{children} dy[child]; `in` = coarse dims
int k_upsample3d_bwd(fm_ctx*, const bf16* dy, const bf16* act, bf16* dx, Dims5 coarse,
                     int dy_C, int dy_cofs, int pz = 2);
// fp32 [vox][Cin] -> bf16 [vox][Cpad], channels >= Cin zero (first layer of the 2.5D U-Net: 6 -> 16 channels)
int k_pad_cast(fm_ctx*, const float* in, bf16* out, int64_t vox, int Cin, int Cpad);
// dice_and_xent / dice_and_xent_mask (metrics.py:68-95): loss = -dice + weight * mean(w * binary_crossentropy(t, p)),
// w = exp(-mask / dist_sigma) per voxel (mask: the second model input of isensee2017.py:85-88) or 1 without a mask.
// weight == 0 selects the plain soft-Dice loss; the statistics then carry a zero in the cross-entropy slot.
struct XentSpec {
  float weight = 0.f;
  float inv_sigma = 0.f;
  const float* mask = nullptr;
};
constexpr int kNumLossSums = 9;
constexpr int kRedScratchRows = 4096;  // rows of fm_ctx::red_scratch (one per block of the partial-sum kernels)
#ifdef __CUDACC__
// Keras K.binary_crossentropy on probabilities (TF backend): p is clipped to [1e-7, 1 - 1e-7] (fp32), turned back into
// a logit and fed to sigmoid_cross_entropy_with_logits, i.e. -(t log p + (1 - t) log(1 - p)) on the clipped p; its
// gradient w.r.t. the pre-sigmoid logit is (p - t), and zero where the clip is active.
__device__ __forceinline__ float xent_term(float t, float p) {
  const float pc = fminf(fmaxf(p, 1e-7f), 1.f - 1e-7f);
  return -(t * logf(pc) + (1.f - t) * log1pf(-pc));
}
__device__ __forceinline__ float xent_grad(float t, float p) {
  return (p >= 1e-7f && p <= 1.f - 1e-7f) ? p - t : 0.f;
}
__device__ __forceinline__ float xent_voxel_weight(const XentSpec& xs, int64_t i) {
  return xs.mask != nullptr ? __expf(-__ldg(xs.mask + i) * xs.inv_sigma) : 1.f;
}
#endif
// loss statistics over p,t (fp32): sums[9] (double) = {tp, t, p, tbpb, tb, pb, correct, count, sum w*bce}
int k_dice_sums(fm_ctx*, const float* p, const float* t, int64_t n, double* sums, int accumulate,
                XentSpec xs = XentSpec());
// dL/dz = dL/dp * p (1-p) with global sums (closed form, metrics.py:11-15) [+ weight/count * w * (p - t)]
int k_dice_bwd(fm_ctx*, const float* p, const float* t, const double* sums, int64_t n, float* dz,
               int through_sigmoid, XentSpec xs = XentSpec());
int k_adam(fm_ctx*, float* p, const float* g, float* m, float* v, int64_t n, int iterations,
           float lr);
int k_zero(fm_ctx*, void* p, size_t bytes);
// InstanceNormalization(axis=1) + LeakyReLU(0.3) (+ residual add) of a raw conv output (Isensee blocks)
// `stats` (optional, [N][C][2]) receives (mean, 1/(std+eps)) for the backward pass; `chan_scale` (optional, [N][C])
// is the SpatialDropout3D keep/scale factor applied after the activation
int k_instnorm_lrelu(fm_ctx*, const bf16* x, const float* gamma, const float* beta, const bf16* add, bf16* y, int N,
                     int64_t vox_per_sample, int C, float* scratch, size_t scratch_floats, float* stats = nullptr,
                     const float* chan_scale = nullptr);
int k_instnorm_lrelu_bwd(fm_ctx*, const bf16* x, const float* stats, const float* gamma, const float* beta,
                         const bf16* gy, const bf16* gy2, const float* chan_scale, bf16* dx, float* dgamma,
                         float* dbeta, int N, int64_t vox_per_sample, int C, float* scratch, size_t scratch_floats);
// BatchNormalization(axis=1) + ReLU of a raw conv output (create_convolution_block(batch_normalization=True)):
// training = batch statistics (kept in `stats` [N][C][2] = (mean, rsqrt(var + eps)), identical rows) and the moving
// averages are updated in place; inference = the moving statistics. Scratch as for the instance norm.
int k_batchnorm_relu(fm_ctx*, const bf16* x, const float* gamma, const float* beta, float* moving_mean, float* moving_var,
                     bf16* y, int N, int64_t vox_per_sample, int C, float* scratch, size_t scratch_floats, float* stats,
                     int training);
int k_batchnorm_relu_bwd(fm_ctx*, const bf16* x, const float* stats, const float* gamma, const float* beta, const bf16* gy,
                         const bf16* gy2, bf16* dx, float* dgamma, float* dbeta, int N, int64_t vox_per_sample, int C,
                         float* scratch, size_t scratch_floats);
int k_zero_insert(fm_ctx*, const bf16* coarse, bf16* fine, Dims5 coarse_dims, int pz = 2);
int k_add_bf16(fm_ctx*, const bf16* a, const bf16* b, bf16* out, int64_t n);
int k_sumpool_f32(fm_ctx*, const float* fine, float* coarse, int N, int X, int Y, int Z, int pz = 2);
int k_dropout_scale(fm_ctx*, float* scale, int n, float rate, uint64_t seed);
// Deconvolution3D/2D (kernel 2, stride 2) = a 1x1x1 conv to taps*C channels followed by a depth-to-space shuffle:
// fine[n][2x+a][2y+b][pz*z+c][co] = z8[n][x][y][z][cls*C + co] + bias[co], cls = (a*2 + b)*pz + c. `coarse` = dims of z8
// with C = channels per class. The reverse shuffle carries the gradient back.
int k_depth_to_space(fm_ctx*, const bf16* z8, const float* bias, bf16* fine, Dims5 coarse, int pz);
int k_space_to_depth(fm_ctx*, const bf16* fine, bf16* g8, Dims5 coarse, int pz);
// x[n][v][c] *= scale[n][c] in place (SpatialDropout2D of the 2D U-Net, forward and backward)
int k_channel_scale(fm_ctx*, bf16* x, const float* scale, int N, int64_t vox_per_sample, int C);
int k_seg_upsample_add(fm_ctx*, const float* fine, const float* coarse, float* out, int N, int X, int Y, int Z,
                       int pz = 2);
int k_sigmoid(fm_ctx*, const float* z, float* p, int64_t n);
// out[(patch voxel (i,j)) * out_pitch + out_cofs + k]: with out_pitch = patch[2], out_cofs = 0 this is the plain
// [n,P0,P1,P2] gather; the 2.5D path writes the slices and the previous-truth slices as channels of one row
int k_gather_patches(fm_ctx*, const float* vol, const int32_t vol_dims[3], const int32_t halo_pad[6],
                     const int32_t fit_pad[6], float pad0, float pad1, const int32_t* idx_dev,
                     int64_t n, const int32_t patch[3], float* out, int out_pitch = 0, int out_cofs = 0,
                     int z_shift = 0);
int k_reassemble(fm_ctx*, const float* preds, const int32_t* idx_host, int64_t n_total,
                 int64_t shard_lo, int64_t shard_hi, int64_t pred_base, const int32_t pred_shape[3],
                 int channels, const int32_t out_dims[3], double* out_dev, int16_t* count_dev,
                 int divide);
int k_divide_by_count(fm_ctx*, double* out, const int16_t* count, int64_t nvox, int channels);
// the same reassembly prepared once (per-axis start lists / covering ranges on the device) and run slab by slab
struct ReasmPlan;
int k_reassemble_prepare(fm_ctx*, const int32_t* idx_host, int64_t n_total, const int32_t pred_shape[3], int channels,
                         const int32_t out_dims[3], ReasmPlan** out_plan);
void k_reassemble_release(ReasmPlan* plan);
// distinct x corners (ascending), their number and the patches per x corner (the list is x-major)
int k_reassemble_groups(const ReasmPlan* plan, const int32_t** xstarts, int* n_groups, int* patches_per_group);
int k_reassemble_rows(fm_ctx*, const ReasmPlan* plan, const float* preds, int64_t shard_lo, int64_t shard_hi,
                      int64_t pred_base, double* out_dev, int16_t* count_dev, int divide, int x_lo, int x_hi);

// postprocess.cu: postprocess_prediction (fetal_net/postprocess.py:13) on a float32 (dtype 0) / float64 (dtype 1) field.
// Views of the ctx-owned workspace for volumes of up to nvox voxels and filters of up to `radius`.
struct PostprocBuffers {
  void *field0, *field1;      // nvox doubles each (float32 fields use the first half)
  int32_t *labels, *aux;      // union-find parents; border marks / component sizes
  uint8_t* mask;              // nvox result
  double* weights;            // 2 radius + 1
  unsigned long long* stats;  // [0] components found, [1] (size << 32 | ~root) of the kept component
};
int pp_buffers(fm_ctx*, int64_t nvox, int radius, PostprocBuffers* out);
// gaussian_filter of the [dims] box of `src` (element strides sx, sy, 1) into the compact out_field (device); src may
// be b.field1
int k_gaussian3d(fm_ctx*, const PostprocBuffers& b, const void* src, int dtype, int64_t sx, int64_t sy,
                 const int32_t dims[3], int radius, const double* weights_host, void* out_field);
// the whole post-processing of the box: result in b.mask, component count and choice in b.stats
int k_postprocess(fm_ctx*, const PostprocBuffers& b, const void* src, int dtype, int64_t sx, int64_t sy,
                  const int32_t dims[3], const fm_postprocess_spec* spec);

// tta.cu: flip test-time augmentation (predict_flips, fetal_net/prediction.py:65-85). Masks: bit a = axis a reversed.
// out [dims] = in [dims] flipped by `mask`
int k_flip_volume(fm_ctx*, const float* in, float* out, const int32_t dims[3], int mask);
// out [dims] = the [dims] box at fit_lo of the [map_dims] map, flipped by `mask`
int k_flip_crop(fm_ctx*, const double* map, const int32_t map_dims[3], const int32_t fit_lo[3], double* out,
                const int32_t dims[3], int mask);
// out[i] = np.median over k < passes (1 .. 8) of stack[k * pitch + i]; pitch % 4 == 0, stack and out 32-byte aligned
int k_median_passes(fm_ctx*, const double* stack, int64_t pitch, int passes, int64_t nvox, double* out);

// conv_simt.cu
// first layer: fp32 single/multi-channel input (channels-last), small Cin; out bf16 + ReLU
int k_conv3d_simt_fprop(fm_ctx*, const void* x, int x_is_f32, const bf16* x2, const bf16* w_packed,
                        const float* bias, bf16* y, float* y_f32, int N, int X, int Y, int Z, int C1,
                        int C2, int Cout, int ksize, int relu, const bf16* mask);
int k_conv3d_simt_wgrad(fm_ctx*, const void* x, int x_is_f32, const bf16* dy, float* dw_packed,
                        int N, int X, int Y, int Z, int Cin, int Cin_total, int cin_ofs, int Cout,
                        int ksize);
int k_bias_grad(fm_ctx*, const bf16* dy, float* db, int64_t voxels, int C);
// 1x1x1 head: z = w.x + b ; p = sigmoid(z) (fp32 out)
int k_head_fwd(fm_ctx*, const bf16* x, const float* w, const float* b, float* p, int64_t voxels,
               int C, int apply_sigmoid = 1);
// training forward: head + sigmoid + the 8 loss statistics of k_dice_sums in one pass over the activations
int k_head_fwd_dice(fm_ctx*, const bf16* x, const float* w, const float* b, const float* t, float* p, int64_t voxels,
                    int C, double* sums, XentSpec xs = XentSpec());
int k_dice_finalize(fm_ctx*, int nblocks, double n_elems, double* sums);
// head backward: dx[v,c] = dz[v] * w[c] * (x[v,c] > 0); dw[c] = sum_v dz[v] x[v,c]; db = sum dz.
// With `t` and `sums`: `dz` holds the probabilities and dL/dz of the soft-Dice loss is formed inside (fused dice_bwd)
int k_head_bwd(fm_ctx*, const bf16* x, const float* dz, const float* w, bf16* dx, float* dw,
               float* db, int64_t voxels, int C, int mode = 0, const float* t = nullptr, const double* sums = nullptr,
               XentSpec xs = XentSpec());
// weight repack: master fp32 [Cout][taps][Cin] -> bf16 fprop pack (same layout) and bf16 dgrad
// pack(s) [Cin_s][taps flipped][Cout] per source
// all layers in ONE launch (after every Adam step): per layer the fprop pack, the dgrad pack(s) and, where the
// plane-marching kernels run, their packs [chunk][dz][dy][kx = 2,1,0][row][kc] — see k_repack_weights / k_repack_march
struct RepackDesc {
  int64_t w_off;   // offset of the master kernel [Cout][taps][C1+C2] in the flat fp32 parameter buffer
  int cout, taps, c1, c2;
  bf16 *wf, *wd0, *wd1, *mf0, *mf1, *md0, *md1;  // null = not needed
  int kcf0, kcf1, kcd0, kcd1;                    // K-chunk widths of the four marching packs (conv_march_kc)
  int block0;      // first 256-thread block of this layer in the fused grid
};
int k_repack_all(fm_ctx*, const float* params, const RepackDesc* table_dev, int nlayers, int total_blocks,
                 double total_weights);
int k_repack_weights(fm_ctx*, const float* w, bf16* w_f, bf16* w_d0, bf16* w_d1, int Cout, int taps,
                     int C1, int C2);

// conv_tc.cu
struct ConvTcPlan;  // opaque cached TMA descriptors for one conv launch configuration
int conv_tc_supported(int C1, int C2, int Cout, int ksize);
// N,X,Y,Z = OUTPUT extent. stride 2 (TF 'SAME', Isensee in-convs) reads an input of extent Xin x Yin x Zin.
// relu: 0 = none, 1 = ReLU
int k_conv3d_tc_fprop(fm_ctx*, const bf16* x1, const bf16* x2, const bf16* w_packed,
                      const float* bias, bf16* y, const bf16* mask, int N, int X, int Y, int Z,
                      int C1, int C2, int Cout, int ksize, int relu, int out_C, int out_cofs, int stride = 1,
                      int Xin = 0, int Yin = 0, int Zin = 0);
int k_conv3d_tc_wgrad(fm_ctx*, const bf16* x, const bf16* dy, float* dw_packed, int N, int X, int Y,
                      int Z, int Cin, int Cin_total, int cin_ofs, int Cout, int ksize);
// Decoder convolution over concatenate([UpSampling3D(2)(coarse), skip]) (unet3d/unet.py:59-62,138) computed WITHOUT
// the upsampled tensor: per parity class of the fine voxel the 27 taps over the upsampled source collapse into 8 taps over
// the coarse tensor with summed weights. X, Y, Z = FINE extents; packs from k_repack_up (tap = class * 8 + j).
int conv_up_supported(int X, int Y, int Z, int Cc, int Cs, int Cout);
int k_repack_up(fm_ctx*, const float* w_master, bf16* w_up_f, bf16* w_up_d, int Cout, int Cc, int Ct);
// the same for up to 8 layers in one launch (w_off = offset of the layer's master kernel in `params`)
struct RepackUpDesc {
  int64_t w_off;
  bf16 *wf, *wd;
  int cout, cc, ct, block0;
};
struct RepackUpTable {
  RepackUpDesc d[8];
  int n;
};
int k_repack_up_table(fm_ctx*, const float* params, const RepackUpTable& tab);
int k_conv3d_up_fprop(fm_ctx*, const bf16* coarse, const bf16* skip, const bf16* w_up, const bf16* w_packed,
                      const float* bias, bf16* y, int N, int X, int Y, int Z, int Cc, int Cs, int Cout, int relu);
int k_conv3d_up_dgrad(fm_ctx*, const bf16* dy, const bf16* w_up_d, bf16* dcoarse, const bf16* mask, int N, int X,
                      int Y, int Z, int Cout, int Cc);
// dw_up [Cout][64][Cc] fp32, zeroed by the caller; k_fold_up_wgrad adds it onto dW[co][27][Ct] (channels [0, Cc))
int k_conv3d_up_wgrad(fm_ctx*, const bf16* coarse, const bf16* dy, float* dw_up, int N, int X, int Y, int Z, int Cc,
                      int Cout);
int k_fold_up_wgrad(fm_ctx*, const float* dw_up, float* dw_master, int Cout, int Cc, int Ct);

// conv_first_tc.cu: first conv (Cin = 1, fp32 volume) and its weight gradient through an im2col tile + tcgen05
int conv_first_tc_supported(int X, int Y, int Z, int Cout);
int k_conv3d_first_tc(fm_ctx*, const float* x, const bf16* w_packed, const float* bias, bf16* y, int N, int X, int Y,
                      int Z, int Cout, int relu);
int k_conv3d_first_tc_wgrad(fm_ctx*, const float* x, const bf16* dy, float* dw, int N, int X, int Y, int Z, int Cout);

// conv_march.cu: plane-marching fprop / dgrad of 3x3x3 convs whose filter bank fits in shared memory
int conv_march_supported(int X, int Y, int Z, int C1, int C2, int Cout, int ksize);
int64_t conv_march_pack_elems(int Cs, int Cout);
// K-chunk width of a source with Cs channels in a marching conv (C1 [+ C2] -> Cout): 64 (128-byte slab rows) unless the
// resident filter bank leaves fewer than two slab slots per dz ring, then 32 (half-size slots, twice as many)
int conv_march_kc(int C1, int C2, int Cout, int Cs);
int k_repack_march(fm_ctx*, const bf16* P, bf16* Wm, int Nrows, int Ktot, int kofs, int Cs, int KC);
// reproducible: the MMAs reach the tensor pipe in a fixed order, so the output is identical run to run (predict /
// evaluate / patch_wise_prediction); otherwise, for Cout <= 32, the order follows three interleaved issue streams
// (training passes)
int k_conv3d_march(fm_ctx*, const bf16* x1, const bf16* x2, const bf16* wm1, const bf16* wm2, const float* bias,
                   bf16* y, const bf16* mask, int N, int X, int Y, int Z, int C1, int C2, int Cout, int relu,
                   int out_C, int out_cofs, bool reproducible);

// conv_wgrad_march.cu
int conv_wgrad_march_supported(int X, int Y, int Z, int Cin, int Cout, int ksize);
// db (optional): the bias gradient [Cout] = column sums of dY, accumulated (atomics) by the same launch
int k_conv3d_wgrad_march(fm_ctx*, const bf16* x, const bf16* dy, float* dw_packed, int N, int X, int Y, int Z,
                         int Cin, int Cin_total, int cin_ofs, int Cout, float* db = nullptr);
