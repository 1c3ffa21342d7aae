// api.cu — C ABI of libfetalb200.so (see include/fetal_b200.h): context, the plain 3D U-Net
// (fetal_net/model/unet3d/unet.py:40-70) as a static launch plan over the kernels in conv_tc.cu /
// conv_simt.cu / bandwidth.cu, the training step (forward, soft-Dice, backward, Keras-Adam) and the
// patch-wise sliding-window inference (fetal_net/prediction.py:118-210).
#include <stdarg.h>

#include <algorithm>
#include <cmath>

#include "common.cuh"
#include <chrono>
#include <thread>

// ---------------------------------------------------------------------------------------------
// error string (per thread)
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";

void fm_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* fm_last_error(void) { return g_err; }

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
extern "C" int fm_ctx_create(int device, fm_ctx** out) {
  FM_CHECK(out != nullptr, FM_EINVAL, "fm_ctx_create: out is NULL");
  int count = 0;
  FM_CUDA(cudaGetDeviceCount(&count));
  FM_CHECK(device >= 0 && device < count, FM_EINVAL, "fm_ctx_create: device %d of %d", device, count);
  FM_CUDA(cudaSetDevice(device));
  fm_ctx* ctx = new fm_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  FM_CUDA(cudaGetDeviceProperties(&prop, device));
  ctx->sm_major = prop.major;
  ctx->sm_minor = prop.minor;
  ctx->num_sms = prop.multiProcessorCount;
  if (prop.major != 10) {
    fm_set_error("fetalb200 is built for sm_100a only; device %d is sm_%d%d (%s)", device, prop.major,
                 prop.minor, prop.name);
    delete ctx;
    return FM_ECUDA;
  }
  FM_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  FM_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  FM_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
  FM_CUDA(cudaEventCreateWithFlags(&ctx->copy_fence, cudaEventDisableTiming));
  FM_CUDA(cudaEventCreateWithFlags(&ctx->copy_done, cudaEventDisableTiming));
  FM_CUDA(cudaMalloc((void**)&ctx->red_scratch, kRedScratchRows * 8 * sizeof(double)));
  *out = ctx;
  return FM_OK;
}

extern "C" int fm_ctx_destroy(fm_ctx* ctx) {
  if (!ctx) return FM_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  fm_comm_destroy(ctx);
  if (ctx->comm_stream) cudaStreamDestroy(ctx->comm_stream);
  if (ctx->comm_ev) cudaEventDestroy(ctx->comm_ev);
  if (ctx->red_scratch) cudaFree(ctx->red_scratch);
  if (ctx->pp_ws) cudaFree(ctx->pp_ws);
  for (auto& r : ctx->prof) {
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
  if (ctx->copy_fence) cudaEventDestroy(ctx->copy_fence);
  if (ctx->copy_done) cudaEventDestroy(ctx->copy_done);
  delete ctx;
  return FM_OK;
}

extern "C" int fm_ctx_device_info(fm_ctx* ctx, int out[3]) {
  FM_CHECK(ctx && out, FM_EINVAL, "fm_ctx_device_info: NULL argument");
  out[0] = ctx->sm_major;
  out[1] = ctx->sm_minor;
  out[2] = ctx->num_sms;
  return FM_OK;
}
extern "C" uint64_t fm_ctx_stream(fm_ctx* ctx) { return ctx ? (uint64_t)(uintptr_t)ctx->stream : 0; }
extern "C" int fm_ctx_synchronize(fm_ctx* ctx) {
  FM_CHECK(ctx, FM_EINVAL, "fm_ctx_synchronize: NULL ctx");
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  return FM_OK;
}
extern "C" int64_t fm_ctx_launch_count(fm_ctx* ctx) { return ctx ? ctx->launches : -1; }

int fm_prof_begin(fm_ctx* ctx, const char* name, double flops, double bytes) {
  ProfRec r;
  r.name = name;
  r.flops = flops;
  r.bytes = bytes;
  FM_CUDA(cudaEventCreate(&r.e0));
  FM_CUDA(cudaEventCreate(&r.e1));
  FM_CUDA(cudaEventRecord(r.e0, ctx->stream));
  ctx->prof.push_back(r);
  return FM_OK;
}
int fm_prof_end(fm_ctx* ctx) {
  if (ctx->prof.empty()) return FM_OK;
  FM_CUDA(cudaEventRecord(ctx->prof.back().e1, ctx->stream));
  return FM_OK;
}
extern "C" int fm_ctx_profile_enable(fm_ctx* ctx, int on) {
  FM_CHECK(ctx, FM_EINVAL, "NULL ctx");
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  for (auto& r : ctx->prof) {
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  ctx->prof.clear();
  ctx->profile = on != 0;
  return FM_OK;
}
extern "C" int fm_ctx_profile_count(fm_ctx* ctx) { return ctx ? (int)ctx->prof.size() : -1; }
extern "C" int fm_ctx_profile_get(fm_ctx* ctx, int i, char name[48], double out[3]) {
  FM_CHECK(ctx && i >= 0 && i < (int)ctx->prof.size() && name && out, FM_EINVAL, "profile record %d", i);
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  float ms = 0.f;
  FM_CUDA(cudaEventElapsedTime(&ms, ctx->prof[i].e0, ctx->prof[i].e1));
  memset(name, 0, 48);
  strncpy(name, ctx->prof[i].name, 47);
  out[0] = ms;
  out[1] = ctx->prof[i].flops;
  out[2] = ctx->prof[i].bytes;
  return FM_OK;
}

// Large host copies into freshly allocated caller memory are page-fault bound (~5 GB/s on one thread);
// faults on disjoint ranges proceed in parallel, so split the copy over a few short-lived threads.
static void host_copy(void* dst, const void* src, size_t bytes) {
  const size_t kMin = (size_t)4 << 20;
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t nt = std::min<size_t>({(size_t)8, (size_t)hw, bytes / kMin});
  if (nt <= 1) {
    memcpy(dst, src, bytes);
    return;
  }
  const size_t chunk = ((bytes + nt - 1) / nt + 4095) & ~(size_t)4095;
  std::vector<std::thread> th;
  for (size_t i = 1; i < nt; ++i) {
    const size_t o = i * chunk;
    if (o >= bytes) break;
    th.emplace_back([=] { memcpy((char*)dst + o, (const char*)src + o, std::min(chunk, bytes - o)); });
  }
  memcpy(dst, src, std::min(chunk, bytes));
  for (auto& t : th) t.join();
}

int fm_ctx_pinned(fm_ctx* ctx, size_t bytes, void** out) {
  if (ctx->pinned_bytes < bytes) {
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr;
    ctx->pinned_bytes = 0;
    FM_CUDA(cudaMallocHost(&ctx->pinned, bytes));
    ctx->pinned_bytes = bytes;
  }
  *out = ctx->pinned;
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------
// small device-buffer helper
// ---------------------------------------------------------------------------------------------
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  int ensure(size_t count) {
    if (count <= n) return FM_OK;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
    if (e != cudaSuccess) {
      fm_set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
      return FM_ENOMEM;
    }
    n = count;
    return FM_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
};

// ---------------------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------------------
struct Layer {
  char name[32];
  int c1, c2, cout, k;  // c2 > 0: second (skip) source of a concat
  int level;            // resolution level (0 = full)
  int64_t w_off, b_off; // offsets in the flat fp32 parameter buffer (kernel packed [Cout][taps][Cin])
  bf16 *w_f = nullptr, *w_d0 = nullptr, *w_d1 = nullptr;  // bf16 packs (fprop, dgrad per source)
  // plane-marching kernel (conv_march.cu): packs per source for fprop / dgrad, null when not applicable
  bf16 *w_mf[2] = {nullptr, nullptr}, *w_md[2] = {nullptr, nullptr};
  bool march_f = false, march_d[2] = {false, false};
  // decoder conv over [UpSampling3D(coarse), skip] computed at coarse resolution (conv_tc.cu, FpropParams::upmode):
  // class-combined packs [Cout][64][c1] / [c1][64][Cout] and the fp32 gradient of the 64 class taps
  bool up_coarse = false;
  bool up_dgrad = false;  // only the gradient towards the coarse tensor runs at coarse resolution (fprop / wgrad march)
  bf16 *w_up_f = nullptr, *w_up_d = nullptr;
  float* dw_up = nullptr;
  int cin_real = 0;     // true input channels when c1 is zero-padded to 16 (first layer of the 2.5D U-Net)
  // 1: normalisation pseudo-layer (InstanceNormalization of the Isensee nets, BatchNormalization of a U-Net built with
  // batch_normalization=True): kernel = gamma, bias = beta (cout each). 2: the BatchNormalization's non-trainable
  // moving statistics: kernel = moving_mean, bias = moving_variance (zero gradient; updated by the forward pass)
  int is_norm = 0;
  int stride = 1;       // 2: TF-'SAME' strided conv (Isensee in-convs)
  int deconv = 0;       // Deconvolution3D/2D (k = 2 or 21, stride 2): master kernel [class][Cout][Cin] = the Keras layout
  int cin() const { return c1 + c2; }
  int taps() const { return kext_taps(k); }
  int cin_keras() const { return cin_real ? cin_real : cin(); }
  int64_t wcount() const { return is_norm ? cout : (int64_t)cout * taps() * cin(); }
};

struct fm_model {
  fm_ctx* ctx = nullptr;
  fm_unet3d_spec spec;
  std::vector<Layer> layers;  // Keras creation order
  int64_t nparams = 0;
  float *params = nullptr, *grads = nullptr, *adam_m = nullptr, *adam_v = nullptr;
  bf16* wpack = nullptr;  // arena for all bf16 packs
  RepackDesc* repack_tab = nullptr;  // device table for the fused repack launch
  int repack_n = 0, repack_blocks = 0;
  double repack_weights = 0.0;
  int iterations = 0;
  bool packs_dirty = true;

  // activations, allocated for `cap` samples
  int cap = 0;
  bool train_alloc = false;
  int kind = 0;   // 0: plain U-Net (3D or 2D); 1: Isensee-2017 residual 3D U-Net (forward / inference only)
  int nseg = 1;   // Isensee: n_segmentation_levels
  std::vector<DevBuf<bf16>> isIn, isC1, isSum, isUp, isU, isLoc1, isLoc2;
  std::vector<DevBuf<float>> isSeg;
  DevBuf<bf16> isRaw;
  DevBuf<float> isScratch, isAcc;
  // Isensee training: per-layer raw conv outputs + (mean, 1/std) for the norm backward, SpatialDropout3D scales per
  // level, gradient scratch (three per level, the 2f-channel upsample gradient, zero-inserted strided gradients)
  std::vector<DevBuf<bf16>> isRawL, gIsA, gIsB, gIsC, gIsUp;
  std::vector<DevBuf<float>> isStatsL, isDropL, gSeg;
  DevBuf<bf16> gIsRaw, gIsZero;
  float dropout_rate = 0.f;
  uint64_t dropout_seed = 0x5EEDull;
  // 2D U-Net: SpatialDropout2D keep/scale factors [B][C] after enc<d>a (slot d) and dec<d>a (slot depth + d)
  std::vector<DevBuf<float>> dropU;
  // deconvolution=True (get_up_convolution, unet3d/unet.py:132-136): the 1x1x1 conv output before the depth-to-space
  // shuffle, and the shuffled gradient on the way back
  bool deconvolution = false;
  DevBuf<bf16> dcZ, dcG;
  // batch_normalization=True (create_convolution_block, unet3d/unet.py:103-104): every conv block is Conv -> BN -> ReLU.
  // Raw conv outputs + batch statistics per layer (training), one raw scratch (inference), the gradient of a raw output
  bool batch_norm = false;
  std::vector<DevBuf<bf16>> bnRawL;
  std::vector<DevBuf<float>> bnStatsL;
  DevBuf<bf16> bnRaw, bnGRaw;
  DevBuf<float> bnScratch;
  bool unet_dropout() const { return kind == 0 && kcode == 31 && dropout_rate > 0.f; }
  int kcode = 3;  // 3: Conv3D 3x3x3 (unet_model_3d); 31: Conv2D 3x3 on a Z = 1 volume (unet_model_2d)
  int pz = 2;     // pooling factor along z
  int cin_real = 1;
  DevBuf<bf16> x_pad;  // 2D model: input cast to bf16 and zero-padded to 16 channels
  DevBuf<float> x_in, t_in, prob, dz;
  std::vector<DevBuf<bf16>> encA, encB, pool, up, decA, decB;          // forward
  std::vector<DevBuf<bf16>> gEncA, gEncB, gPool, gUp, gSkip, gDecA, gDecB;  // gradients
  double* sums = nullptr;  // kNumLossSums doubles (device): 7 Dice / VOD / accuracy sums, the count, sum w * bce
  double sums_host[kNumLossSums];
  // loss: 0 dice_coefficient_loss, 1 dice_and_xent, 2 dice_and_xent_mask (weight mask = second model input)
  int loss_kind = 0;
  float xent_weight = 0.f, xent_inv_sigma = 0.f;
  DevBuf<float> mask_in;
  bool mask_valid = false;
  int mask_batch = 0;
  XentSpec xent() const {
    XentSpec xs;
    if (loss_kind != 0) {
      xs.weight = xent_weight;
      xs.inv_sigma = xent_inv_sigma;
      xs.mask = loss_kind == 2 ? mask_in.p : nullptr;
    }
    return xs;
  }
  // fm_train_step pipelining (pinned host inputs): two device staging buffers filled by the copy stream while the
  // previous step is still in its backward pass; the call returns once the Dice statistics of ITS forward pass are
  // on the host, the rest of the step (backward, Adam, repack) keeps running and is ordered before any later call
  DevBuf<float> stage_x[2], stage_t[2];
  // pageable host inputs are first copied (a few host threads) into these pinned ping-pong buffers, so that they take
  // the same pipelined route; host_stage_done[b] = the H2D copies out of buffer b have completed
  float* host_stage[2] = {nullptr, nullptr};
  size_t host_stage_floats[2] = {0, 0};
  cudaEvent_t host_stage_done[2] = {nullptr, nullptr};
  cudaEvent_t stage_ready[2] = {nullptr, nullptr}, stage_free[2] = {nullptr, nullptr}, sums_ready = nullptr;
  double* sums_pin = nullptr;
  int stage_idx = 0;
  bool metrics_pending = false;

  // sliding-window workspace (grow-only): volume, corners, per-patch probabilities, fp64 sums, counts
  DevBuf<float> pw_vol, pw_pred;
  DevBuf<int32_t> pw_idx;
  DevBuf<double> pw_out;
  DevBuf<int16_t> pw_cnt;
  std::vector<cudaEvent_t> pw_events;  // [0] upload, [1] rows ready, [2..] one per finished output slab
  // flip test-time augmentation (grow-only): the flipped copy of the volume, the un-flipped maps [passes][pitch]
  DevBuf<float> tta_vol;
  DevBuf<double> tta_stack;

  // backward bucket events (one per layer, reverse creation order)
  std::vector<cudaEvent_t> layer_done;
  std::vector<std::pair<int, int>> buckets;  // [first layer, last layer] inclusive, creation order
  cudaEvent_t ev_tmp = nullptr;
  int last_batch = 0;
  bool fwd_valid = false;
  // training passes use the shared-accumulator marching kernel (faster; fp32 summation order not fixed), inference
  // the bit-reproducible one
  bool train_pass = false;
  // fm_model_set_inference_mode(m, 1): predict / evaluate / patch_wise_prediction also take the three-issuer mode
  // (about 25 % more conv throughput, results no longer bit-identical from run to run)
  bool fast_inference = false;
  // training forward with the targets already in t_in: the head kernel also produces the loss statistics
  bool targets_ready = false, stats_done = false;

  int depth() const { return spec.depth; }
  Dims5 dims(int level, int C, int B) const {
    return Dims5{B, spec.X >> level, spec.Y >> level, pz == 2 ? spec.Z >> level : spec.Z, C};
  }
  int64_t vox(int level) const {
    return (int64_t)(spec.X >> level) * (spec.Y >> level) * (pz == 2 ? spec.Z >> level : spec.Z);
  }
};

static int layer_index(fm_model* m, const char* name) {
  for (size_t i = 0; i < m->layers.size(); ++i)
    if (strcmp(m->layers[i].name, name) == 0) return (int)i;
  return -1;
}
static Layer& L(fm_model* m, const char* fmt, int d) {
  char nm[32];
  snprintf(nm, sizeof(nm), fmt, d);
  return m->layers[layer_index(m, nm)];
}

// Training passes (and fast inference) let the marching kernel issue its MMAs in three interleaved streams where it
// applies (Cout <= 32): 20-30 % faster, but the order in which the three MMA warps' products land in an accumulator is
// not fixed, so activations differ in the last bf16 bit from run to run. FETAL_B200_DETERMINISTIC=1 keeps training on
// the bit-reproducible issue order (the fp32 red.add order of the weight gradients is then the only run-to-run
// difference).
static bool reproducible_pass(const fm_model* m) {
  static const bool det = [] {
    const char* e = getenv("FETAL_B200_DETERMINISTIC");
    return e && e[0] == '1';
  }();
  return !(m->train_pass || m->fast_inference) || det;
}

static int build_unet(fm_ctx* ctx, const fm_unet3d_spec* spec, int kcode, int flags, fm_model** out);

extern "C" int fm_model_create_unet3d(fm_ctx* ctx, const fm_unet3d_spec* spec, fm_model** out) {
  return fm_model_create_unet3d_ex(ctx, spec, 0, out);
}
extern "C" int fm_model_create_unet2d(fm_ctx* ctx, const fm_unet2d_spec* spec2, fm_model** out) {
  return fm_model_create_unet2d_ex(ctx, spec2, 0, out);
}

extern "C" int fm_model_create_unet3d_ex(fm_ctx* ctx, const fm_unet3d_spec* spec, int flags, fm_model** out) {
  FM_CHECK(ctx && spec && out, FM_EINVAL, "fm_model_create_unet3d: NULL argument");
  FM_CHECK((flags & ~(FM_UNET_DECONVOLUTION | FM_UNET_BATCH_NORMALIZATION)) == 0, FM_EINVAL,
           "fm_model_create_unet3d_ex: unknown flags 0x%x", flags);
  FM_CHECK(spec->in_channels == 1, FM_EINVAL,
           "in_channels=%d: only the reference's single-modality path (1) is built", spec->in_channels);
  const int div = 1 << (spec->depth > 0 ? spec->depth - 1 : 0);
  FM_CHECK(spec->X > 0 && spec->Y > 0 && spec->Z > 0 && spec->X % div == 0 && spec->Y % div == 0 &&
               spec->Z % div == 0,
           FM_EINVAL, "input extent %dx%dx%d must be divisible by 2^(depth-1)=%d (unet3d/unet.py:32-33)",
           spec->X, spec->Y, spec->Z, div);
  return build_unet(ctx, spec, 3, flags, out);
}

extern "C" int fm_model_create_unet2d_ex(fm_ctx* ctx, const fm_unet2d_spec* spec2, int flags, fm_model** out) {
  FM_CHECK(ctx && spec2 && out, FM_EINVAL, "fm_model_create_unet2d: NULL argument");
  FM_CHECK((flags & ~(FM_UNET_DECONVOLUTION | FM_UNET_BATCH_NORMALIZATION)) == 0, FM_EINVAL,
           "fm_model_create_unet2d_ex: unknown flags 0x%x", flags);
  FM_CHECK(spec2->in_channels >= 1 && spec2->in_channels <= 16, FM_EINVAL,
           "in_channels=%d: the slices-as-channels input supports 1..16 channels", spec2->in_channels);
  const int div = 1 << (spec2->depth > 0 ? spec2->depth - 1 : 0);
  FM_CHECK(spec2->H > 0 && spec2->W > 0 && spec2->H % div == 0 && spec2->W % div == 0, FM_EINVAL,
           "input extent %dx%d must be divisible by 2^(depth-1)=%d", spec2->H, spec2->W, div);
  fm_unet3d_spec s;
  s.in_channels = spec2->in_channels;
  s.X = spec2->H;
  s.Y = spec2->W;
  s.Z = 1;
  s.depth = spec2->depth;
  s.n_base_filters = spec2->n_base_filters;
  s.n_labels = spec2->n_labels;
  return build_unet(ctx, &s, 31, flags, out);
}

static int build_unet(fm_ctx* ctx, const fm_unet3d_spec* spec, int kcode, int flags, fm_model** out) {
  FM_CHECK(spec->depth >= 2 && spec->depth <= 6, FM_EINVAL, "depth %d unsupported", spec->depth);
  FM_CHECK(spec->n_labels == 1, FM_EINVAL, "n_labels=%d: only 1 is built", spec->n_labels);
  FM_CHECK(spec->n_base_filters == 16 || spec->n_base_filters == 32, FM_EINVAL,
           "n_base_filters=%d: 16 or 32", spec->n_base_filters);
  FM_CUDA(cudaSetDevice(ctx->device));
  fm_model* m = new fm_model();
  m->ctx = ctx;
  m->spec = *spec;
  m->kcode = kcode;
  m->pz = kcode == 31 ? 1 : 2;
  m->cin_real = spec->in_channels;
  m->deconvolution = (flags & FM_UNET_DECONVOLUTION) != 0;
  m->batch_norm = (flags & FM_UNET_BATCH_NORMALIZATION) != 0;
  const int D = spec->depth, nf = spec->n_base_filters;
  auto add = [&](const char* fmt, int d, int c1, int c2, int cout, int k, int level) {
    Layer l;
    memset(l.name, 0, sizeof(l.name));
    snprintf(l.name, sizeof(l.name), fmt, d);
    l.c1 = c1;
    l.c2 = c2;
    l.cout = cout;
    l.k = k;
    l.level = level;
    l.w_off = m->nparams;
    m->nparams += l.wcount();
    l.b_off = m->nparams;
    m->nparams += cout;
    // keep every layer's block 16-byte aligned for the vectorised Adam / allreduce views
    m->nparams = (m->nparams + 3) & ~(int64_t)3;
    m->layers.push_back(l);
    if (m->batch_norm && (k == 3 || k == 31)) {
      // BatchNormalization(axis=1) behind the conv of every block: (gamma, beta) and (moving_mean, moving_variance)
      for (int kind = 1; kind <= 2; ++kind) {
        Layer g;
        memset(g.name, 0, sizeof(g.name));
        snprintf(g.name, sizeof(g.name), kind == 1 ? "%s_norm" : "%s_moving", l.name);
        g.is_norm = kind;
        g.c1 = cout;
        g.c2 = 0;
        g.cout = cout;
        g.k = 1;
        g.level = level;
        g.w_off = m->nparams;
        m->nparams += cout;
        g.b_off = m->nparams;
        m->nparams = (m->nparams + cout + 3) & ~(int64_t)3;
        m->layers.push_back(g);
      }
    }
  };
  // the 2D model feeds its first conv from a 16-channel zero-padded copy of the input (tensor-core K granule)
  int c = kcode == 31 ? 16 : spec->in_channels;
  std::vector<int> skipc;
  for (int d = 0; d < D; ++d) {
    const int f1 = nf << d, f2 = f1 * 2;
    add("enc%da", d, c, 0, f1, kcode, d);
    add("enc%db", d, f1, 0, f2, kcode, d);
    skipc.push_back(f2);
    c = f2;
  }
  for (int d = D - 2; d >= 0; --d) {
    if (m->deconvolution) {
      // Deconvolution3D(filters = channels of the coarse tensor, kernel 2, strides 2), created before the block that
      // consumes it (unet.py:57-59): 8 (4 in 2D) parity-class 1x1x1 matrices, bias, no activation
      add("up%d", d, c, 0, c, kcode == 31 ? 21 : 2, d + 1);
      m->layers.back().deconv = 1;
    }
    add("dec%da", d, c, skipc[d], skipc[d], kcode, d);  // concat order [up, skip] (unet.py:61)
    add("dec%db", d, skipc[d], 0, skipc[d], kcode, d);
    c = skipc[d];
  }
  add("final", 0, c, 0, spec->n_labels, 1, 0);
  if (kcode == 31) m->layers[0].cin_real = spec->in_channels;

  const size_t pb = (size_t)m->nparams * sizeof(float);
  FM_CUDA(cudaMalloc((void**)&m->params, pb));
  FM_CUDA(cudaMalloc((void**)&m->grads, pb));
  FM_CUDA(cudaMalloc((void**)&m->adam_m, pb));
  FM_CUDA(cudaMalloc((void**)&m->adam_v, pb));
  FM_CUDA(cudaMemset(m->params, 0, pb));
  FM_CUDA(cudaMemset(m->grads, 0, pb));
  FM_CUDA(cudaMemset(m->adam_m, 0, pb));
  FM_CUDA(cudaMemset(m->adam_v, 0, pb));
  // bf16 packs: fprop + dgrad copies of every kernel
  int64_t pack_elems = 0;
  for (auto& l : m->layers) pack_elems += 2 * ((l.wcount() + 63) & ~(int64_t)63);
  FM_CUDA(cudaMalloc((void**)&m->wpack, (size_t)pack_elems * sizeof(bf16)));
  FM_CUDA(cudaMemset(m->wpack, 0, (size_t)pack_elems * sizeof(bf16)));
  bf16* wp = m->wpack;
  for (auto& l : m->layers) {
    const int64_t padded = (l.wcount() + 63) & ~(int64_t)63;
    l.w_f = wp;
    wp += padded;
    l.w_d0 = wp;
    l.w_d1 = wp + (int64_t)l.c1 * l.taps() * l.cout;
    wp += padded;
  }
  for (auto& l : m->layers) {
    if (l.is_norm || l.k != 3 || l.c1 < 16) continue;
    const int X = spec->X >> l.level, Y = spec->Y >> l.level, Z = m->pz == 2 ? spec->Z >> l.level : spec->Z;
    const int cs[2] = {l.c1, l.c2};
    if (conv_march_supported(X, Y, Z, l.c1, l.c2, l.cout, l.k)) {
      l.march_f = true;
      for (int s = 0; s < (l.c2 ? 2 : 1); ++s)
        FM_CUDA(cudaMalloc((void**)&l.w_mf[s], (size_t)conv_march_pack_elems(cs[s], l.cout) * sizeof(bf16)));
    }
    for (int s = 0; s < (l.c2 ? 2 : 1); ++s)
      if (conv_march_supported(X, Y, Z, l.cout, 0, cs[s], l.k)) {
        l.march_d[s] = true;
        FM_CUDA(cudaMalloc((void**)&l.w_md[s], (size_t)conv_march_pack_elems(l.cout, cs[s]) * sizeof(bf16)));
      }
  }
  // decoder convs whose filter bank is too large for the marching kernel run at COARSE resolution on their upsampled
  // source (dec1a, dec2a of the shipped model)
  for (auto& l : m->layers) {
    if (strncmp(l.name, "dec", 3) != 0 || l.c2 == 0 || l.k != 3 || m->pz != 2 || m->deconvolution || m->batch_norm ||
        l.is_norm)
      continue;
    const int X = spec->X >> l.level, Y = spec->Y >> l.level, Z = spec->Z >> l.level;
    if (!conv_up_supported(X, Y, Z, l.c1, l.c2, l.cout)) continue;
    const size_t n = (size_t)l.cout * 64 * l.c1;
    FM_CUDA(cudaMalloc((void**)&l.w_up_d, n * sizeof(bf16)));
    if (l.march_f) {
      // small filter bank (dec0a): forward and weight gradient stay on the marching kernels over the materialised
      // upsampled tensor; the gradient towards the coarse tensor still drops from 27 fine taps + a sum-pool pass to
      // 64 class taps per COARSE voxel
      l.up_dgrad = true;
      continue;
    }
    l.up_coarse = true;
    FM_CUDA(cudaMalloc((void**)&l.w_up_f, n * sizeof(bf16)));
    FM_CUDA(cudaMalloc((void**)&l.dw_up, n * sizeof(float)));
  }
  FM_CUDA(cudaMalloc((void**)&m->sums, kNumLossSums * sizeof(double)));
  FM_CUDA(cudaMemset(m->sums, 0, kNumLossSums * sizeof(double)));
  m->encA.resize(D);
  m->encB.resize(D);
  m->pool.resize(D);
  m->up.resize(D);
  m->decA.resize(D);
  m->decB.resize(D);
  m->gEncA.resize(D);
  m->gEncB.resize(D);
  m->gPool.resize(D);
  m->gUp.resize(D);
  m->gSkip.resize(D);
  m->gDecA.resize(D);
  m->gDecB.resize(D);
  m->bnRawL.resize(m->layers.size());
  m->bnStatsL.resize(m->layers.size());
  m->layer_done.resize(m->layers.size());
  for (auto& e : m->layer_done) FM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  FM_CUDA(cudaEventCreateWithFlags(&m->ev_tmp, cudaEventDisableTiming));
  // gradient buckets: consecutive layers in backward (= reverse creation) order, ~1/4 of the
  // parameters each; every bucket is one contiguous range of the flat buffer.
  {
    const int nl = (int)m->layers.size();
    const int64_t target = m->nparams / 4 + 1;
    int hi = nl - 1;
    int64_t acc = 0;
    for (int i = nl - 1; i >= 0; --i) {
      acc += m->layers[i].wcount() + m->layers[i].cout;
      if (acc >= target || i == 0) {
        m->buckets.push_back({i, hi});
        hi = i - 1;
        acc = 0;
      }
    }
  }
  *out = m;
  return FM_OK;
}

extern "C" int fm_model_destroy(fm_model* m) {
  if (!m) return FM_OK;
  cudaSetDevice(m->ctx->device);
  cudaStreamSynchronize(m->ctx->stream);
  cudaFree(m->params);
  cudaFree(m->grads);
  cudaFree(m->adam_m);
  cudaFree(m->adam_v);
  cudaFree(m->wpack);
  cudaFree(m->repack_tab);
  cudaFree(m->sums);
  for (auto& l : m->layers) {
    for (int s = 0; s < 2; ++s) {
      if (l.w_mf[s]) cudaFree(l.w_mf[s]);
      if (l.w_md[s]) cudaFree(l.w_md[s]);
    }
    if (l.w_up_f) cudaFree(l.w_up_f);
    if (l.w_up_d) cudaFree(l.w_up_d);
    if (l.dw_up) cudaFree(l.dw_up);
  }
  for (auto* v : {&m->isIn, &m->isC1, &m->isSum, &m->isUp, &m->isU, &m->isLoc1, &m->isLoc2})
    for (auto& b : *v) b.release();
  for (auto& b : m->isSeg) b.release();
  for (auto* v : {&m->isRawL, &m->gIsA, &m->gIsB, &m->gIsC, &m->gIsUp})
    for (auto& b : *v) b.release();
  for (auto* v : {&m->isStatsL, &m->isDropL, &m->gSeg, &m->dropU, &m->bnStatsL})
    for (auto& b : *v) b.release();
  m->gIsRaw.release();
  m->gIsZero.release();
  m->isRaw.release();
  m->isScratch.release();
  m->isAcc.release();
  m->pw_vol.release();
  m->pw_pred.release();
  m->pw_idx.release();
  m->pw_out.release();
  m->pw_cnt.release();
  m->tta_vol.release();
  m->tta_stack.release();
  m->x_in.release();
  m->bnRaw.release();
  m->bnGRaw.release();
  m->bnScratch.release();
  for (auto& b : m->bnRawL) b.release();
  m->dcZ.release();
  m->dcG.release();
  m->mask_in.release();
  m->x_pad.release();
  m->t_in.release();
  m->prob.release();
  m->dz.release();
  for (auto* v : {&m->encA, &m->encB, &m->pool, &m->up, &m->decA, &m->decB, &m->gEncA, &m->gEncB,
                  &m->gPool, &m->gUp, &m->gSkip, &m->gDecA, &m->gDecB})
    for (auto& b : *v) b.release();
  for (auto& e : m->layer_done) cudaEventDestroy(e);
  for (auto& e : m->pw_events)
    if (e) cudaEventDestroy(e);
  for (int b = 0; b < 2; ++b) {
    m->stage_x[b].release();
    m->stage_t[b].release();
    if (m->stage_ready[b]) cudaEventDestroy(m->stage_ready[b]);
    if (m->stage_free[b]) cudaEventDestroy(m->stage_free[b]);
  }
  if (m->sums_ready) cudaEventDestroy(m->sums_ready);
  if (m->sums_pin) cudaFreeHost(m->sums_pin);
  for (int b = 0; b < 2; ++b) {
    if (m->host_stage[b]) cudaFreeHost(m->host_stage[b]);
    if (m->host_stage_done[b]) cudaEventDestroy(m->host_stage_done[b]);
  }
  if (m->ev_tmp) cudaEventDestroy(m->ev_tmp);
  delete m;
  return FM_OK;
}

extern "C" int fm_model_num_layers(fm_model* m) { return m ? (int)m->layers.size() : -1; }
extern "C" int64_t fm_model_num_params(fm_model* m) {
  if (!m) return -1;
  int64_t n = 0;
  for (auto& l : m->layers) n += l.is_norm ? 2 * (int64_t)l.cout : (int64_t)l.cout * l.taps() * l.cin_keras() + l.cout;
  return n;
}
extern "C" int fm_model_layer_info(fm_model* m, int layer, char name[32], int64_t info[5]) {
  FM_CHECK(m && layer >= 0 && layer < (int)m->layers.size(), FM_EINVAL, "layer %d out of range", layer);
  const Layer& l = m->layers[layer];
  if (name) memcpy(name, l.name, 32);
  if (info) {
    info[0] = l.cin_keras();
    info[1] = l.cout;
    // 33: 3x3x3, 31: 3x3(x1), 22 / 21: deconvolution, 11: 1x1x1, 0: norm (gamma, beta), -1: BN moving (mean, variance)
    info[2] = l.is_norm == 2 ? -1 : (l.is_norm ? 0 : kext_xy(l.k) * 10 + kext_z(l.k));
    info[3] = l.w_off;
    info[4] = l.b_off;
  }
  return FM_OK;
}

// Keras layout (k0,k1,k2,Cin,Cout) <-> packed [Cout][tap=(k0*K+k1)*K+k2][Cin]
// `Cin` = channels of the Keras kernel, `Cpad` >= Cin = channels of the packed kernel (extra channels zero)
static void keras_to_packed(const float* kern, float* packed, int K, int Cin, int Cout, int Cpad = 0) {
  const int taps = kext_taps(K);
  if (Cpad < Cin) Cpad = Cin;
  for (int tap = 0; tap < taps; ++tap)
    for (int co = 0; co < Cout; ++co)
      for (int ci = 0; ci < Cpad; ++ci)
        packed[((int64_t)co * taps + tap) * Cpad + ci] = ci < Cin ? kern[((int64_t)tap * Cin + ci) * Cout + co] : 0.f;
}
static void packed_to_keras(const float* packed, float* kern, int K, int Cin, int Cout, int Cpad = 0) {
  const int taps = kext_taps(K);
  if (Cpad < Cin) Cpad = Cin;
  for (int tap = 0; tap < taps; ++tap)
    for (int ci = 0; ci < Cin; ++ci)
      for (int co = 0; co < Cout; ++co)
        kern[((int64_t)tap * Cin + ci) * Cout + co] = packed[((int64_t)co * taps + tap) * Cpad + ci];
}

extern "C" int fm_model_set_weights(fm_model* m, int layer, const float* kernel, const float* bias) {
  FM_CHECK(m && layer >= 0 && layer < (int)m->layers.size() && kernel && bias, FM_EINVAL,
           "fm_model_set_weights: bad argument");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  Layer& l = m->layers[layer];
  if (l.is_norm) {
    FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
    FM_CUDA(cudaMemcpy(m->params + l.w_off, kernel, (size_t)l.cout * 4, cudaMemcpyHostToDevice));
    FM_CUDA(cudaMemcpy(m->params + l.b_off, bias, (size_t)l.cout * 4, cudaMemcpyHostToDevice));
    return FM_OK;
  }
  std::vector<float> packed((size_t)l.wcount());
  if (l.deconv)  // Keras Conv3DTranspose kernel (2,2,2,Cout,Cin) is already [class][Cout][Cin]
    memcpy(packed.data(), kernel, packed.size() * sizeof(float));
  else
    keras_to_packed(kernel, packed.data(), l.k, l.cin_keras(), l.cout, l.cin());
  FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
  FM_CUDA(cudaMemcpy(m->params + l.w_off, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice));
  FM_CUDA(cudaMemcpy(m->params + l.b_off, bias, (size_t)l.cout * 4, cudaMemcpyHostToDevice));
  m->packs_dirty = true;
  return FM_OK;
}
static int get_flat(fm_model* m, const float* flat, int layer, float* kernel, float* bias) {
  FM_CHECK(m && layer >= 0 && layer < (int)m->layers.size(), FM_EINVAL, "layer %d out of range", layer);
  FM_CUDA(cudaSetDevice(m->ctx->device));
  Layer& l = m->layers[layer];
  FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
  if (kernel && l.is_norm) {
    FM_CUDA(cudaMemcpy(kernel, flat + l.w_off, (size_t)l.cout * 4, cudaMemcpyDeviceToHost));
  } else if (kernel) {
    std::vector<float> packed((size_t)l.wcount());
    FM_CUDA(cudaMemcpy(packed.data(), flat + l.w_off, packed.size() * 4, cudaMemcpyDeviceToHost));
    if (l.deconv)
      memcpy(kernel, packed.data(), packed.size() * sizeof(float));
    else
      packed_to_keras(packed.data(), kernel, l.k, l.cin_keras(), l.cout, l.cin());
  }
  if (bias) FM_CUDA(cudaMemcpy(bias, flat + l.b_off, (size_t)l.cout * 4, cudaMemcpyDeviceToHost));
  return FM_OK;
}
extern "C" int fm_model_get_weights(fm_model* m, int layer, float* kernel, float* bias) {
  return get_flat(m, m ? m->params : nullptr, layer, kernel, bias);
}
extern "C" int fm_model_get_grads(fm_model* m, int layer, float* kernel, float* bias) {
  return get_flat(m, m ? m->grads : nullptr, layer, kernel, bias);
}
extern "C" int fm_model_set_dropout(fm_model* m, float rate, uint64_t seed) {
  FM_CHECK(m, FM_EINVAL, "NULL model");
  FM_CHECK(rate >= 0.f && rate < 1.f, FM_EINVAL, "dropout rate %g outside [0,1)", (double)rate);
  m->dropout_rate = rate;
  m->dropout_seed = seed;
  return FM_OK;
}

extern "C" int fm_model_set_inference_mode(fm_model* m, int fast) {
  FM_CHECK(m, FM_EINVAL, "NULL model");
  m->fast_inference = fast != 0;
  return FM_OK;
}

extern "C" int fm_model_set_loss(fm_model* m, int kind, float xent_weight, float dist_sigma) {
  FM_CHECK(m, FM_EINVAL, "NULL model");
  FM_CHECK(kind >= 0 && kind <= 2, FM_EINVAL, "fm_model_set_loss: kind %d (0 dice, 1 dice_and_xent, 2 dice_and_xent_mask)", kind);
  FM_CHECK(kind != 2 || dist_sigma > 0.f, FM_EINVAL, "fm_model_set_loss: dist_sigma must be positive");
  m->loss_kind = kind;
  m->xent_weight = kind ? xent_weight : 0.f;
  m->xent_inv_sigma = kind == 2 ? 1.f / dist_sigma : 0.f;
  m->mask_valid = false;
  return FM_OK;
}

extern "C" int fm_model_set_weight_mask(fm_model* m, const float* mask, int batch) {
  FM_CHECK(m && mask && batch > 0, FM_EINVAL, "fm_model_set_weight_mask: bad argument");
  FM_CHECK(m->loss_kind == 2, FM_EINVAL, "fm_model_set_weight_mask: the model's loss takes no weight mask");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  const size_t n = (size_t)batch * m->vox(0);
  if (n > m->mask_in.n) {
    // the previous step may still read the old buffer
    FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
    FM_TRY(m->mask_in.ensure(n));
  }
  FM_CUDA(cudaMemcpyAsync(m->mask_in.p, mask, n * sizeof(float), cudaMemcpyHostToDevice, m->ctx->stream));
  m->mask_valid = true;
  m->mask_batch = batch;
  return FM_OK;
}

extern "C" int fm_model_reset_optimizer(fm_model* m) {
  FM_CHECK(m, FM_EINVAL, "NULL model");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  const size_t pb = (size_t)m->nparams * sizeof(float);
  FM_CUDA(cudaMemsetAsync(m->adam_m, 0, pb, m->ctx->stream));
  FM_CUDA(cudaMemsetAsync(m->adam_v, 0, pb, m->ctx->stream));
  m->iterations = 0;
  return FM_OK;
}

static int refresh_packs(fm_model* m) {
  if (!m->packs_dirty) return FM_OK;
  if (!m->repack_tab) {
    // built on first use: one descriptor per conv layer that keeps bf16 packs, one fused launch from then on
    std::vector<RepackDesc> tab;
    int blocks = 0;
    double weights = 0.0;
    for (auto& l : m->layers) {
      if (l.is_norm || (l.k == 1 && l.cout == 1)) continue;  // norm parameters / heads are read as fp32
      RepackDesc d;
      d.w_off = l.w_off;
      // a deconvolution is repacked as the 1x1x1 conv it runs as: [class * Cout + co][1][Cin]
      d.cout = l.deconv ? l.cout * l.taps() : l.cout;
      d.taps = l.deconv ? 1 : l.taps();
      d.c1 = l.c1;
      d.c2 = l.c2;
      d.wf = l.w_f;
      d.wd0 = l.w_d0;
      d.wd1 = l.c2 ? l.w_d1 : nullptr;
      d.mf0 = l.march_f ? l.w_mf[0] : nullptr;
      d.mf1 = l.march_f && l.c2 ? l.w_mf[1] : nullptr;
      d.md0 = l.march_d[0] ? l.w_md[0] : nullptr;
      d.md1 = l.c2 && l.march_d[1] ? l.w_md[1] : nullptr;
      d.kcf0 = conv_march_kc(l.c1, l.c2, l.cout, l.c1);
      d.kcf1 = l.c2 ? conv_march_kc(l.c1, l.c2, l.cout, l.c2) : 0;
      d.kcd0 = conv_march_kc(l.cout, 0, l.c1, l.cout);
      d.kcd1 = l.c2 ? conv_march_kc(l.cout, 0, l.c2, l.cout) : 0;
      d.block0 = blocks;
      blocks += d.taps * ceil_div(d.cout, 32) * ceil_div(l.cin(), 32);  // 32 x 32 (co, c) tiles per tap
      weights += (double)l.wcount();
      tab.push_back(d);
    }
    FM_CUDA(cudaMalloc((void**)&m->repack_tab, tab.size() * sizeof(RepackDesc)));
    FM_CUDA(cudaMemcpy(m->repack_tab, tab.data(), tab.size() * sizeof(RepackDesc), cudaMemcpyHostToDevice));
    m->repack_n = (int)tab.size();
    m->repack_blocks = blocks;
    m->repack_weights = weights;
  }
  if (m->repack_n > 0)  // (0 only for a model without convs)
    FM_TRY(k_repack_all(m->ctx, m->params, m->repack_tab, m->repack_n, m->repack_blocks, m->repack_weights));
  RepackUpTable ut;
  memset(&ut, 0, sizeof(ut));
  for (auto& l : m->layers) {
    if (!(l.up_coarse || l.up_dgrad)) continue;
    if (ut.n == 8) {
      FM_TRY(k_repack_up_table(m->ctx, m->params, ut));
      ut.n = 0;
    }
    RepackUpDesc& d = ut.d[ut.n];
    d.w_off = l.w_off;
    d.wf = l.w_up_f;
    d.wd = l.w_up_d;
    d.cout = l.cout;
    d.cc = l.c1;
    d.ct = l.cin();
    d.block0 = ut.n ? ut.d[ut.n - 1].block0 + (int)ceil_div64((int64_t)ut.d[ut.n - 1].cout * 64 * ut.d[ut.n - 1].cc, 256) : 0;
    ++ut.n;
  }
  FM_TRY(k_repack_up_table(m->ctx, m->params, ut));
  m->packs_dirty = false;
  return FM_OK;
}

static int ensure_capacity_isensee(fm_model* m, int B, bool train);

static int ensure_capacity(fm_model* m, int B, bool train) {
  if (m->kind == 1) return ensure_capacity_isensee(m, B, train);
  if (B <= m->cap && (!train || m->train_alloc)) return FM_OK;
  FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
  const int cap = std::max(B, m->cap);
  const int D = m->depth();
  const size_t v0 = (size_t)m->vox(0);
  FM_TRY(m->x_in.ensure((size_t)cap * v0 * m->cin_real));
  if (m->kcode == 31) FM_TRY(m->x_pad.ensure((size_t)cap * v0 * 16));
  FM_TRY(m->prob.ensure((size_t)cap * v0));
  for (int d = 0; d < D; ++d) {
    const size_t v = (size_t)m->vox(d) * cap;
    const Layer &la = L(m, "enc%da", d), &lb = L(m, "enc%db", d);
    FM_TRY(m->encA[d].ensure(v * la.cout));
    FM_TRY(m->encB[d].ensure(v * lb.cout));
    if (d < D - 1) {
      FM_TRY(m->pool[d].ensure((size_t)m->vox(d + 1) * cap * lb.cout));
      const Layer &da = L(m, "dec%da", d), &db = L(m, "dec%db", d);
      if (!da.up_coarse) FM_TRY(m->up[d].ensure(v * da.c1));
      if (m->deconvolution) FM_TRY(m->dcZ.ensure(v * da.c1));
      FM_TRY(m->decA[d].ensure(v * da.cout));
      FM_TRY(m->decB[d].ensure(v * db.cout));
    }
  }
  if (m->batch_norm) {
    size_t biggest = 0, cmax = 0;
    for (size_t i = 0; i < m->layers.size(); ++i) {
      const Layer& l = m->layers[i];
      if (l.is_norm != 1) continue;
      const size_t n = (size_t)cap * m->vox(l.level) * l.cout;
      biggest = std::max(biggest, n);
      cmax = std::max(cmax, (size_t)l.cout);
      if (train || m->train_alloc) {
        FM_TRY(m->bnRawL[i].ensure(n));
        FM_TRY(m->bnStatsL[i].ensure((size_t)cap * l.cout * 2));
      }
    }
    FM_TRY(m->bnRaw.ensure(biggest));
    if (train || m->train_alloc) FM_TRY(m->bnGRaw.ensure(biggest));
    FM_TRY(m->bnScratch.ensure((size_t)cap * cmax * 2 * 1030));
  }
  if (train || m->train_alloc) {
    FM_TRY(m->t_in.ensure((size_t)cap * v0));  // (no dL/dz tensor: the head backward forms the Dice gradient itself)
    for (int d = 0; d < D; ++d) {
      const size_t v = (size_t)m->vox(d) * cap;
      const Layer &la = L(m, "enc%da", d), &lb = L(m, "enc%db", d);
      FM_TRY(m->gEncA[d].ensure(v * la.cout));
      FM_TRY(m->gEncB[d].ensure(v * lb.cout));
      if (d < D - 1) {
        FM_TRY(m->gPool[d].ensure((size_t)m->vox(d + 1) * cap * lb.cout));
        const Layer &da = L(m, "dec%da", d), &db = L(m, "dec%db", d);
        if (!da.up_coarse && !da.up_dgrad) FM_TRY(m->gUp[d].ensure(v * da.c1));
        if (m->deconvolution) FM_TRY(m->dcG.ensure(v * da.c1));
        FM_TRY(m->gSkip[d].ensure(v * da.c2));
        FM_TRY(m->gDecA[d].ensure(v * da.cout));
        FM_TRY(m->gDecB[d].ensure(v * db.cout));
      }
    }
    m->train_alloc = true;
  }
  m->cap = cap;
  return FM_OK;
}

// conv block forward: Conv3D + bias + ReLU (create_convolution_block, unet.py:102-113)
static int conv_fwd(fm_model* m, const Layer& l, const bf16* x1, const bf16* x2, bf16* y, int B, int relu = 1) {
  fm_ctx* ctx = m->ctx;
  const Dims5 d = m->dims(l.level, l.cout, B);
  const float* bias = m->params + l.b_off;
  if (l.march_f)
    return k_conv3d_march(ctx, x1, x2, l.w_mf[0], l.w_mf[1], bias, y, nullptr, B, d.X, d.Y, d.Z, l.c1, l.c2, l.cout, relu,
                          l.cout, 0, reproducible_pass(m));
  if (conv_tc_supported(l.c1, l.c2, l.cout, l.k))
    return k_conv3d_tc_fprop(ctx, x1, x2, l.w_f, bias, y, nullptr, B, d.X, d.Y, d.Z, l.c1, l.c2, l.cout,
                             l.k, relu, l.cout, 0);
  return k_conv3d_simt_fprop(ctx, x1, 0, x2, l.w_f, bias, y, nullptr, B, d.X, d.Y, d.Z, l.c1, l.c2,
                             l.cout, l.k, relu, nullptr);
}

// one conv block of a U-Net built with batch_normalization=True: Conv (+bias, no activation) -> raw ->
// BatchNormalization + ReLU -> y. A training pass keeps the raw output and the batch statistics of every block.
static int bn_block_fwd(fm_model* m, const Layer& l, const void* x1, int x1_f32, const bf16* x2, bf16* y, int B) {
  fm_ctx* ctx = m->ctx;
  const int li = (int)(&l - &m->layers[0]);
  const Layer &nl = m->layers[li + 1], &ml = m->layers[li + 2];
  const Dims5 d = m->dims(l.level, l.cout, B);
  bf16* raw = m->train_pass ? m->bnRawL[li + 1].p : m->bnRaw.p;
  if (x1_f32)  // the first conv of the 3D model reads the fp32 single-channel input
    FM_TRY(k_conv3d_simt_fprop(ctx, x1, 1, nullptr, l.w_f, m->params + l.b_off, raw, nullptr, B, d.X, d.Y, d.Z, l.c1, 0,
                               l.cout, l.k, 0, nullptr));
  else
    FM_TRY(conv_fwd(m, l, (const bf16*)x1, x2, raw, B, 0));
  return k_batchnorm_relu(ctx, raw, m->params + nl.w_off, m->params + nl.b_off, m->params + ml.w_off,
                          m->params + ml.b_off, y, B, m->vox(l.level), l.cout, m->bnScratch.p, m->bnScratch.n,
                          m->train_pass ? m->bnStatsL[li + 1].p : nullptr, m->train_pass ? 1 : 0);
}

static int forward_unet_bn(fm_model* m, int B) {
  fm_ctx* ctx = m->ctx;
  const int D = m->depth();
  FM_TRY(refresh_packs(m));
  const bf16* cur = nullptr;
  for (int d = 0; d < D; ++d) {
    const Layer &la = L(m, "enc%da", d), &lb = L(m, "enc%db", d);
    if (d == 0 && m->kcode == 31) {
      FM_TRY(k_pad_cast(ctx, m->x_in.p, m->x_pad.p, (int64_t)B * m->vox(0), m->cin_real, 16));
      FM_TRY(bn_block_fwd(m, la, m->x_pad.p, 0, nullptr, m->encA[0].p, B));
    } else if (d == 0) {
      FM_TRY(bn_block_fwd(m, la, m->x_in.p, 1, nullptr, m->encA[0].p, B));
    } else {
      FM_TRY(bn_block_fwd(m, la, cur, 0, nullptr, m->encA[d].p, B));
    }
    FM_TRY(bn_block_fwd(m, lb, m->encA[d].p, 0, nullptr, m->encB[d].p, B));
    cur = m->encB[d].p;
    if (d < D - 1) {
      FM_TRY(k_maxpool3d_fwd(ctx, m->encB[d].p, m->pool[d].p, m->dims(d, lb.cout, B), m->pz));
      cur = m->pool[d].p;
    }
  }
  for (int d = D - 2; d >= 0; --d) {
    const Layer &da = L(m, "dec%da", d), &db = L(m, "dec%db", d);
    if (m->deconvolution) {
      const Layer& lu = L(m, "up%d", d);
      const Dims5 dc = m->dims(d + 1, lu.cout, B);
      FM_TRY(k_conv3d_tc_fprop(ctx, cur, nullptr, lu.w_f, nullptr, m->dcZ.p, nullptr, B, dc.X, dc.Y, dc.Z, lu.c1, 0,
                               lu.cout * lu.taps(), 1, 0, lu.cout * lu.taps(), 0));
      FM_TRY(k_depth_to_space(ctx, m->dcZ.p, m->params + lu.b_off, m->up[d].p, dc, m->pz));
    } else {
      FM_TRY(k_upsample3d_fwd(ctx, cur, m->up[d].p, m->dims(d + 1, da.c1, B), m->pz));
    }
    FM_TRY(bn_block_fwd(m, da, m->up[d].p, 0, m->encB[d].p, m->decA[d].p, B));
    FM_TRY(bn_block_fwd(m, db, m->decA[d].p, 0, nullptr, m->decB[d].p, B));
    cur = m->decB[d].p;
  }
  const Layer& lf = m->layers.back();
  if (m->train_pass && m->targets_ready) {
    FM_TRY(k_head_fwd_dice(ctx, cur, m->params + lf.w_off, m->params + lf.b_off, m->t_in.p, m->prob.p,
                           (int64_t)B * m->vox(0), lf.c1, m->sums, m->xent()));
    m->stats_done = true;
    return FM_OK;
  }
  return k_head_fwd(ctx, cur, m->params + lf.w_off, m->params + lf.b_off, m->prob.p, (int64_t)B * m->vox(0), lf.c1);
}

static int forward_isensee(fm_model* m, int B);

// SpatialDropout2D(rate) behind the first conv block of every level of the 2D U-Net (unet/unet.py:60-61,76-77):
// one keep/scale factor per (sample, channel), drawn per step from the counter-based hash, applied in place. The
// stored activation is the dropped one, so the next conv's weight gradient and the ReLU mask of the gradient
// (kept channels are scaled by a positive factor) need no change; the gradient itself is scaled on the way back.
static int unet_dropout_fwd(fm_model* m, int slot, bf16* act, const Layer& l, int B) {
  if ((int)m->dropU.size() <= slot) m->dropU.resize(slot + 1);
  FM_TRY(m->dropU[slot].ensure((size_t)B * l.cout));
  FM_TRY(k_dropout_scale(m->ctx, m->dropU[slot].p, B * l.cout, m->dropout_rate,
                         m->dropout_seed + (uint64_t)m->iterations * 64 + (uint64_t)slot));
  return k_channel_scale(m->ctx, act, m->dropU[slot].p, B, m->vox(l.level), l.cout);
}

// forward pass on x_in (fp32 [B, X, Y, Z], C = 1) -> prob (fp32 [B, X, Y, Z])
static int forward(fm_model* m, int B) {
  if (m->kind == 1) return forward_isensee(m, B);
  if (m->batch_norm) return forward_unet_bn(m, B);
  fm_ctx* ctx = m->ctx;
  const int D = m->depth();
  FM_TRY(refresh_packs(m));
  const bf16* cur = nullptr;
  for (int d = 0; d < D; ++d) {
    const Layer &la = L(m, "enc%da", d), &lb = L(m, "enc%db", d);
    const Dims5 dd = m->dims(d, la.cout, B);
    if (d == 0 && m->kcode == 31) {
      FM_TRY(k_pad_cast(ctx, m->x_in.p, m->x_pad.p, dd.voxels(), m->cin_real, 16));
      FM_TRY(conv_fwd(m, la, m->x_pad.p, nullptr, m->encA[0].p, B));
    } else if (d == 0) {
      FM_TRY(k_conv3d_simt_fprop(ctx, m->x_in.p, 1, nullptr, la.w_f, m->params + la.b_off, m->encA[0].p,
                                 nullptr, B, dd.X, dd.Y, dd.Z, la.c1, 0, la.cout, la.k, 1, nullptr));
    } else {
      FM_TRY(conv_fwd(m, la, cur, nullptr, m->encA[d].p, B));
    }
    if (m->train_pass && m->unet_dropout()) FM_TRY(unet_dropout_fwd(m, d, m->encA[d].p, la, B));
    FM_TRY(conv_fwd(m, lb, m->encA[d].p, nullptr, m->encB[d].p, B));
    cur = m->encB[d].p;
    if (d < D - 1) {
      FM_TRY(k_maxpool3d_fwd(ctx, m->encB[d].p, m->pool[d].p, m->dims(d, lb.cout, B), m->pz));
      cur = m->pool[d].p;
    }
  }
  for (int d = D - 2; d >= 0; --d) {
    const Layer &da = L(m, "dec%da", d), &db = L(m, "dec%db", d);
    if (da.up_coarse) {
      // no upsampled tensor: the conv reads the coarse tensor with class-combined weights (8 taps instead of 27)
      const Dims5 dd = m->dims(d, da.cout, B);
      FM_TRY(k_conv3d_up_fprop(ctx, cur, m->encB[d].p, da.w_up_f, da.w_f, m->params + da.b_off, m->decA[d].p, B, dd.X,
                               dd.Y, dd.Z, da.c1, da.c2, da.cout, 1));
    } else if (m->deconvolution) {
      // Deconvolution3D: 1x1x1 conv of the coarse tensor to (classes x C) channels, then depth-to-space (+ bias)
      const Layer& lu = L(m, "up%d", d);
      const Dims5 dc = m->dims(d + 1, lu.cout, B);
      FM_TRY(k_conv3d_tc_fprop(ctx, cur, nullptr, lu.w_f, nullptr, m->dcZ.p, nullptr, B, dc.X, dc.Y, dc.Z, lu.c1, 0,
                               lu.cout * lu.taps(), 1, 0, lu.cout * lu.taps(), 0));
      FM_TRY(k_depth_to_space(ctx, m->dcZ.p, m->params + lu.b_off, m->up[d].p, dc, m->pz));
      FM_TRY(conv_fwd(m, da, m->up[d].p, m->encB[d].p, m->decA[d].p, B));
    } else {
      FM_TRY(k_upsample3d_fwd(ctx, cur, m->up[d].p, m->dims(d + 1, da.c1, B), m->pz));
      FM_TRY(conv_fwd(m, da, m->up[d].p, m->encB[d].p, m->decA[d].p, B));
    }
    if (m->train_pass && m->unet_dropout()) FM_TRY(unet_dropout_fwd(m, D + d, m->decA[d].p, da, B));
    FM_TRY(conv_fwd(m, db, m->decA[d].p, nullptr, m->decB[d].p, B));
    cur = m->decB[d].p;
  }
  const Layer& lf = m->layers.back();
  if (m->train_pass && m->targets_ready) {
    // head + sigmoid + Dice / VOD / accuracy sums in one pass (unet.py:68-69 + metrics.py:11-28)
    FM_TRY(k_head_fwd_dice(ctx, cur, m->params + lf.w_off, m->params + lf.b_off, m->t_in.p, m->prob.p,
                           (int64_t)B * m->vox(0), lf.c1, m->sums, m->xent()));
    m->stats_done = true;
    return FM_OK;
  }
  FM_TRY(k_head_fwd(ctx, cur, m->params + lf.w_off, m->params + lf.b_off, m->prob.p,
                    (int64_t)B * m->vox(0), lf.c1));
  return FM_OK;
}

// wgrad + bias grad of one conv layer (only_src >= 0: the weight gradient of that source alone, plus the bias)
static int conv_wgrad(fm_model* m, const Layer& l, const bf16* x1, const bf16* x2, const bf16* dy, int B,
                      int only_src = -1) {
  fm_ctx* ctx = m->ctx;
  const Dims5 d = m->dims(l.level, l.cout, B);
  float* dw = m->grads + l.w_off;
  const bf16* xs[2] = {x1, x2};
  const int cs[2] = {l.c1, l.c2};
  int cofs = 0;
  bool bias_done = false;
  for (int s = 0; s < (l.c2 ? 2 : 1); ++s) {
    if (only_src >= 0 && s != only_src) {
      cofs += cs[s];
      continue;
    }
    if (conv_wgrad_march_supported(d.X, d.Y, d.Z, cs[s], l.cout, l.k)) {
      // the marching kernel also sums dY over the voxels (bias gradient) while the tiles sit in shared memory
      FM_TRY(k_conv3d_wgrad_march(ctx, xs[s], dy, dw, B, d.X, d.Y, d.Z, cs[s], l.cin(), cofs, l.cout,
                                  bias_done ? nullptr : m->grads + l.b_off));
      bias_done = true;
    } else if (conv_tc_supported(cs[s], 0, l.cout, l.k))
      FM_TRY(k_conv3d_tc_wgrad(ctx, xs[s], dy, dw, B, d.X, d.Y, d.Z, cs[s], l.cin(), cofs, l.cout, l.k));
    else
      FM_TRY(k_conv3d_simt_wgrad(ctx, xs[s], 0, dy, dw, B, d.X, d.Y, d.Z, cs[s], l.cin(), cofs, l.cout,
                                 l.k));
    cofs += cs[s];
  }
  if (!bias_done) FM_TRY(k_bias_grad(ctx, dy, m->grads + l.b_off, d.voxels(), l.cout));
  return FM_OK;
}

static int conv_wgrad_source(fm_model* m, const Layer& l, int src, const bf16* x, const bf16* dy, int B) {
  return conv_wgrad(m, l, src == 0 ? x : nullptr, src == 1 ? x : nullptr, dy, B, src);
}

// dgrad of one source of a conv layer: dx = conv(dy, W flipped^T) [* ReLU mask of `mask`]
static int conv_dgrad(fm_model* m, const Layer& l, int src, const bf16* dy, const bf16* mask, bf16* dx,
                      int B) {
  fm_ctx* ctx = m->ctx;
  const Dims5 d = m->dims(l.level, l.cout, B);
  const int cs = src == 0 ? l.c1 : l.c2;
  const bf16* wd = src == 0 ? l.w_d0 : l.w_d1;
  if (l.march_d[src])
    return k_conv3d_march(ctx, dy, nullptr, l.w_md[src], nullptr, nullptr, dx, mask, B, d.X, d.Y, d.Z, l.cout, 0, cs, 0,
                          cs, 0, reproducible_pass(m));
  if (conv_tc_supported(l.cout, 0, cs, l.k))
    return k_conv3d_tc_fprop(ctx, dy, nullptr, wd, nullptr, dx, mask, B, d.X, d.Y, d.Z, l.cout, 0, cs, l.k,
                             0, cs, 0);
  return k_conv3d_simt_fprop(ctx, dy, 0, nullptr, wd, nullptr, dx, nullptr, B, d.X, d.Y, d.Z, l.cout, 0,
                             cs, l.k, 0, mask);
}

static int mark_layer_done(fm_model* m, const Layer& l) {
  const int i = (int)(&l - &m->layers[0]);
  FM_CUDA(cudaEventRecord(m->layer_done[i], m->ctx->stream));
  return FM_OK;
}

static int backward_isensee(fm_model* m, int B);

// BatchNormalization + ReLU backward of block `l` (gy [+ gy2] = gradient of the block's activation) -> m->bnGRaw, the
// gradient of the raw conv output; gamma / beta gradients. The conv bias in front of the normalisation has an
// analytically zero gradient (conv_wgrad still sums it: rounding noise, as in Keras).
static int bn_block_bwd(fm_model* m, const Layer& l, const bf16* gy, const bf16* gy2, int B) {
  const int li = (int)(&l - &m->layers[0]);
  const Layer& nl = m->layers[li + 1];
  FM_TRY(k_batchnorm_relu_bwd(m->ctx, m->bnRawL[li + 1].p, m->bnStatsL[li + 1].p, m->params + nl.w_off,
                              m->params + nl.b_off, gy, gy2, m->bnGRaw.p, m->grads + nl.w_off, m->grads + nl.b_off, B,
                              m->vox(l.level), l.cout, m->bnScratch.p, m->bnScratch.n));
  FM_TRY(mark_layer_done(m, m->layers[li + 2]));
  return mark_layer_done(m, nl);
}

// Backward pass of a U-Net built with batch_normalization=True: the ReLU derivative lives in the normalisation
// backward (it is recomputed from the raw conv output and the batch statistics), so every dgrad / pooling / upsampling
// gradient runs WITHOUT an activation mask; the decoder's upsampled source is materialised.
static int backward_unet_bn(fm_model* m, int B) {
  fm_ctx* ctx = m->ctx;
  const int D = m->depth();
  const int64_t n0 = (int64_t)B * m->vox(0);
  FM_TRY(k_zero(ctx, m->grads, (size_t)m->nparams * sizeof(float)));
  const Layer& lf = m->layers.back();
  FM_TRY(k_head_bwd(ctx, m->decB[0].p, m->prob.p, m->params + lf.w_off, m->gDecB[0].p, m->grads + lf.w_off,
                    m->grads + lf.b_off, n0, lf.c1, 1, m->t_in.p, m->sums, m->xent()));
  FM_TRY(mark_layer_done(m, lf));
  for (int d = 0; d <= D - 2; ++d) {
    const Layer &da = L(m, "dec%da", d), &db = L(m, "dec%db", d);
    FM_TRY(bn_block_bwd(m, db, m->gDecB[d].p, nullptr, B));
    FM_TRY(conv_wgrad(m, db, m->decA[d].p, nullptr, m->bnGRaw.p, B));
    FM_TRY(mark_layer_done(m, db));
    FM_TRY(conv_dgrad(m, db, 0, m->bnGRaw.p, nullptr, m->gDecA[d].p, B));
    FM_TRY(bn_block_bwd(m, da, m->gDecA[d].p, nullptr, B));
    FM_TRY(conv_wgrad(m, da, m->up[d].p, m->encB[d].p, m->bnGRaw.p, B));
    FM_TRY(mark_layer_done(m, da));
    FM_TRY(conv_dgrad(m, da, 0, m->bnGRaw.p, nullptr, m->gUp[d].p, B));
    FM_TRY(conv_dgrad(m, da, 1, m->bnGRaw.p, nullptr, m->gSkip[d].p, B));
    const bool bottom = (d + 1 == D - 1);
    const bf16* act = bottom ? m->encB[D - 1].p : m->decB[d + 1].p;
    bf16* gdst = bottom ? m->gEncB[D - 1].p : m->gDecB[d + 1].p;
    if (m->deconvolution) {
      const Layer& lu = L(m, "up%d", d);
      const Dims5 dc = m->dims(d + 1, lu.cout, B);
      const int c8 = lu.cout * lu.taps();
      FM_TRY(k_bias_grad(ctx, m->gUp[d].p, m->grads + lu.b_off, (int64_t)B * m->vox(d), lu.cout));
      FM_TRY(k_space_to_depth(ctx, m->gUp[d].p, m->dcG.p, dc, m->pz));
      FM_TRY(k_conv3d_tc_wgrad(ctx, act, m->dcG.p, m->grads + lu.w_off, B, dc.X, dc.Y, dc.Z, lu.c1, lu.c1, 0, c8, 1));
      FM_TRY(mark_layer_done(m, lu));
      FM_TRY(k_conv3d_tc_fprop(ctx, m->dcG.p, nullptr, lu.w_d0, nullptr, gdst, nullptr, B, dc.X, dc.Y, dc.Z, c8, 0, lu.c1,
                               1, 0, lu.c1, 0));
    } else {
      FM_TRY(k_upsample3d_bwd(ctx, m->gUp[d].p, nullptr, gdst, m->dims(d + 1, da.c1, B), da.c1, 0, m->pz));
    }
  }
  for (int d = D - 1; d >= 0; --d) {
    const Layer &la = L(m, "enc%da", d), &lb = L(m, "enc%db", d);
    if (d < D - 1)  // gradient of encB[d]: skip path + MaxPooling backward (no mask)
      FM_TRY(k_maxpool3d_bwd(ctx, m->encB[d].p, m->gPool[d].p, m->gSkip[d].p, m->gEncB[d].p, m->dims(d, lb.cout, B), 0,
                             m->pz));
    FM_TRY(bn_block_bwd(m, lb, m->gEncB[d].p, nullptr, B));
    FM_TRY(conv_wgrad(m, lb, m->encA[d].p, nullptr, m->bnGRaw.p, B));
    FM_TRY(mark_layer_done(m, lb));
    FM_TRY(conv_dgrad(m, lb, 0, m->bnGRaw.p, nullptr, m->gEncA[d].p, B));
    FM_TRY(bn_block_bwd(m, la, m->gEncA[d].p, nullptr, B));
    if (d > 0) {
      FM_TRY(conv_wgrad(m, la, m->pool[d - 1].p, nullptr, m->bnGRaw.p, B));
      FM_TRY(mark_layer_done(m, la));
      FM_TRY(conv_dgrad(m, la, 0, m->bnGRaw.p, nullptr, m->gPool[d - 1].p, B));
    } else if (m->kcode == 31) {
      FM_TRY(conv_wgrad(m, la, m->x_pad.p, nullptr, m->bnGRaw.p, B));
      FM_TRY(mark_layer_done(m, la));
    } else {
      const Dims5 dd = m->dims(0, la.cout, B);
      FM_TRY(k_conv3d_simt_wgrad(ctx, m->x_in.p, 1, m->bnGRaw.p, m->grads + la.w_off, B, dd.X, dd.Y, dd.Z, la.c1, la.c1, 0,
                                 la.cout, la.k));
      FM_TRY(k_bias_grad(ctx, m->bnGRaw.p, m->grads + la.b_off, dd.voxels(), la.cout));
      FM_TRY(mark_layer_done(m, la));
    }
  }
  return FM_OK;
}

static int backward(fm_model* m, int B) {
  if (m->kind == 1) return backward_isensee(m, B);
  if (m->batch_norm) return backward_unet_bn(m, B);
  fm_ctx* ctx = m->ctx;
  const int D = m->depth();
  const int64_t n0 = (int64_t)B * m->vox(0);
  FM_TRY(k_zero(ctx, m->grads, (size_t)m->nparams * sizeof(float)));
  const Layer& lf = m->layers.back();
  // head backward with the soft-Dice gradient formed inside (closed form through the sigmoid with the GLOBAL sums):
  // gradient lands masked by the ReLU of dec0b (or encB[0] when depth == 1)
  FM_TRY(k_head_bwd(ctx, m->decB[0].p, m->prob.p, m->params + lf.w_off, m->gDecB[0].p, m->grads + lf.w_off,
                    m->grads + lf.b_off, n0, lf.c1, 0, m->t_in.p, m->sums, m->xent()));
  FM_TRY(mark_layer_done(m, lf));
  for (int d = 0; d <= D - 2; ++d) {
    const Layer &da = L(m, "dec%da", d), &db = L(m, "dec%db", d);
    // dec_b: input decA[d]
    FM_TRY(conv_wgrad(m, db, m->decA[d].p, nullptr, m->gDecB[d].p, B));
    FM_TRY(mark_layer_done(m, db));
    FM_TRY(conv_dgrad(m, db, 0, m->gDecB[d].p, m->decA[d].p, m->gDecA[d].p, B));
    if (m->unet_dropout()) FM_TRY(k_channel_scale(ctx, m->gDecA[d].p, m->dropU[D + d].p, B, m->vox(d), da.cout));
    // dec_a: inputs [up[d], encB[d]]; the coarser tensor that was upsampled and its ReLU mask
    const bool bottom = (d + 1 == D - 1);
    const bf16* act = bottom ? m->encB[D - 1].p : m->decB[d + 1].p;
    bf16* gdst = bottom ? m->gEncB[D - 1].p : m->gDecB[d + 1].p;
    if (da.up_coarse) {
      // weight gradient of the up-source channels from the 64 class taps at coarse resolution, folded onto the 27
      // taps; the skip channels and the bias through the ordinary kernels; the gradient towards the coarse tensor
      // straight from dY (no gUp tensor, no sum-pool pass)
      const Dims5 dd = m->dims(d, da.cout, B);
      FM_TRY(k_zero(ctx, da.dw_up, (size_t)da.cout * 64 * da.c1 * sizeof(float)));
      FM_TRY(k_conv3d_up_wgrad(ctx, act, m->gDecA[d].p, da.dw_up, B, dd.X, dd.Y, dd.Z, da.c1, da.cout));
      FM_TRY(k_fold_up_wgrad(ctx, da.dw_up, m->grads + da.w_off, da.cout, da.c1, da.cin()));
      FM_TRY(conv_wgrad_source(m, da, 1, m->encB[d].p, m->gDecA[d].p, B));
      FM_TRY(mark_layer_done(m, da));
      FM_TRY(k_conv3d_up_dgrad(ctx, m->gDecA[d].p, da.w_up_d, gdst, act, B, dd.X, dd.Y, dd.Z, da.cout, da.c1));
      FM_TRY(conv_dgrad(m, da, 1, m->gDecA[d].p, nullptr, m->gSkip[d].p, B));
      continue;
    }
    FM_TRY(conv_wgrad(m, da, m->up[d].p, m->encB[d].p, m->gDecA[d].p, B));
    FM_TRY(mark_layer_done(m, da));
    if (da.up_dgrad) {
      const Dims5 dd = m->dims(d, da.cout, B);
      FM_TRY(k_conv3d_up_dgrad(ctx, m->gDecA[d].p, da.w_up_d, gdst, act, B, dd.X, dd.Y, dd.Z, da.cout, da.c1));
      FM_TRY(conv_dgrad(m, da, 1, m->gDecA[d].p, nullptr, m->gSkip[d].p, B));
      continue;
    }
    FM_TRY(conv_dgrad(m, da, 0, m->gDecA[d].p, nullptr, m->gUp[d].p, B));
    FM_TRY(conv_dgrad(m, da, 1, m->gDecA[d].p, nullptr, m->gSkip[d].p, B));
    if (m->deconvolution) {
      // Deconvolution3D backward: bias gradient = column sums of the fine gradient; the shuffled gradient is the dY
      // of a 1x1x1 conv with (classes x C) outputs: weight gradient against the coarse activation, data gradient
      // (+ ReLU mask of the coarse block) through the transposed matrix
      const Layer& lu = L(m, "up%d", d);
      const Dims5 dc = m->dims(d + 1, lu.cout, B);
      const int c8 = lu.cout * lu.taps();
      FM_TRY(k_bias_grad(ctx, m->gUp[d].p, m->grads + lu.b_off, (int64_t)B * m->vox(d), lu.cout));
      FM_TRY(k_space_to_depth(ctx, m->gUp[d].p, m->dcG.p, dc, m->pz));
      FM_TRY(k_conv3d_tc_wgrad(ctx, act, m->dcG.p, m->grads + lu.w_off, B, dc.X, dc.Y, dc.Z, lu.c1, lu.c1, 0, c8, 1));
      FM_TRY(mark_layer_done(m, lu));
      FM_TRY(k_conv3d_tc_fprop(ctx, m->dcG.p, nullptr, lu.w_d0, nullptr, gdst, act, B, dc.X, dc.Y, dc.Z, c8, 0, lu.c1, 1,
                               0, lu.c1, 0));
      continue;
    }
    // through UpSampling3D into the coarser tensor that was upsampled (+ its ReLU mask)
    FM_TRY(k_upsample3d_bwd(ctx, m->gUp[d].p, act, gdst, m->dims(d + 1, da.c1, B), da.c1, 0, m->pz));
  }
  for (int d = D - 1; d >= 0; --d) {
    const Layer &la = L(m, "enc%da", d), &lb = L(m, "enc%db", d);
    if (d < D - 1) {
      // gradient of encB[d]: skip path + MaxPooling3D backward, masked by its ReLU
      FM_TRY(k_maxpool3d_bwd(ctx, m->encB[d].p, m->gPool[d].p, m->gSkip[d].p, m->gEncB[d].p,
                             m->dims(d, lb.cout, B), 1, m->pz));
    }
    FM_TRY(conv_wgrad(m, lb, m->encA[d].p, nullptr, m->gEncB[d].p, B));
    FM_TRY(mark_layer_done(m, lb));
    FM_TRY(conv_dgrad(m, lb, 0, m->gEncB[d].p, m->encA[d].p, m->gEncA[d].p, B));
    if (m->unet_dropout()) FM_TRY(k_channel_scale(ctx, m->gEncA[d].p, m->dropU[d].p, B, m->vox(d), la.cout));
    if (d > 0) {
      FM_TRY(conv_wgrad(m, la, m->pool[d - 1].p, nullptr, m->gEncA[d].p, B));
      FM_TRY(mark_layer_done(m, la));
      FM_TRY(conv_dgrad(m, la, 0, m->gEncA[d].p, nullptr, m->gPool[d - 1].p, B));
    } else if (m->kcode == 31) {
      FM_TRY(conv_wgrad(m, la, m->x_pad.p, nullptr, m->gEncA[0].p, B));
      FM_TRY(mark_layer_done(m, la));
    } else {
      const Dims5 dd = m->dims(0, la.cout, B);
      FM_TRY(k_conv3d_simt_wgrad(ctx, m->x_in.p, 1, m->gEncA[0].p, m->grads + la.w_off, B, dd.X, dd.Y, dd.Z,
                                 la.c1, la.c1, 0, la.cout, la.k));
      FM_TRY(k_bias_grad(ctx, m->gEncA[0].p, m->grads + la.b_off, dd.voxels(), la.cout));
      FM_TRY(mark_layer_done(m, la));
    }
  }
  return FM_OK;
}

static void metrics_from_sums(const double s[kNumLossSums], float out[4], float xent_weight = 0.f) {
  const double dice = (2.0 * s[0] + 1.0) / (s[1] + s[2] + 1.0);
  const double uni = s[4] + s[5] - s[3];
  // loss = -dice (metrics.py:31-32) [+ xent_weight * mean(w * bce): dice_and_xent, metrics.py:68-78]
  out[0] = (float)(-dice + (xent_weight != 0.f && s[7] > 0 ? (double)xent_weight * s[8] / s[7] : 0.0));
  out[1] = (float)(s[7] > 0 ? s[6] / s[7] : 0);  // binary_accuracy
  out[2] = (float)((s[3] + 1.0) / (uni + 1.0));  // vod_coefficient (metrics.py:18-28)
  out[3] = (float)dice;
}

static int upload(fm_model* m, const float* src, float* dst, size_t count) {
  // pageable -> device through the runtime's own staging; callers that care pass pinned memory
  FM_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(float), cudaMemcpyHostToDevice, m->ctx->stream));
  return FM_OK;
}


// ---------------------------------------------------------------------------------------------
// Isensee-2017 residual 3D U-Net, forward / inference (fetal_net/model/unet3d/isensee2017.py:39-79):
// conv block = Conv3D(+bias) -> InstanceNormalization(axis=1) -> LeakyReLU(0.3) (isensee2017.py:12);
// level: in_conv (stride 2 from level 1, TF 'SAME') -> context module (2 blocks; SpatialDropout3D is
// identity at inference) -> residual Add; decoder: UpSampling3D -> block -> concat [skip, up] ->
// localisation module (3^3 block, 1^3 block) -> Conv3D(n_labels, 1) heads summed coarse-to-fine; sigmoid.
// Layer table in Keras creation order, every conv followed by its norm pseudo-layer (gamma, beta).
// ---------------------------------------------------------------------------------------------
struct IsenseeBuild {
  int X, Y, Z, in_channels, depth, n_base_filters, n_segmentation_levels, kcode;
};
static int build_isensee(fm_ctx* ctx, const IsenseeBuild* spec, fm_model** out);

// whether the data gradient towards a source of cs channels (first source c1 channels) runs on the marching kernel;
// decided once per layer when the model is built (X, Y, Z = the extent the dgrad runs at)
static bool isensee_dgrad_marches(int X, int Y, int Z, int c1, int cs, int cout, int k) {
  return k == 3 && c1 >= 16 && conv_march_supported(X, Y, Z, cout, 0, cs, k);
}

extern "C" int fm_model_create_isensee3d(fm_ctx* ctx, const fm_isensee3d_spec* spec, fm_model** out) {
  FM_CHECK(ctx && spec && out, FM_EINVAL, "fm_model_create_isensee3d: NULL argument");
  FM_CHECK(spec->in_channels == 1 && spec->n_labels == 1, FM_EINVAL, "isensee: in_channels and n_labels must be 1");
  IsenseeBuild b{spec->X, spec->Y, spec->Z, 1, spec->depth, spec->n_base_filters, spec->n_segmentation_levels, 3};
  return build_isensee(ctx, &b, out);
}

// isensee2017_model (fetal_net/model/unet/isensee.py:14-86): the same graph in 2D on slices-as-channels input -
// Conv2D 3x3 / 1x1 blocks, strides (2, 2), UpSampling2D, SpatialDropout2D - run on a Z = 1 volume with kernel-extent
// code 31 and no pooling along z, like the 2D U-Net. The input's `in_channels` slices are zero-padded to 16 channels.
extern "C" int fm_model_create_isensee2d(fm_ctx* ctx, const fm_isensee2d_spec* spec, fm_model** out) {
  FM_CHECK(ctx && spec && out, FM_EINVAL, "fm_model_create_isensee2d: NULL argument");
  FM_CHECK(spec->n_labels == 1, FM_EINVAL, "isensee2d: n_labels must be 1");
  FM_CHECK(spec->in_channels >= 1 && spec->in_channels <= 16, FM_EINVAL, "isensee2d: in_channels %d outside [1,16]",
           spec->in_channels);
  IsenseeBuild b{spec->H, spec->W, 1, spec->in_channels, spec->depth, spec->n_base_filters,
                 spec->n_segmentation_levels, 31};
  return build_isensee(ctx, &b, out);
}

static int build_isensee(fm_ctx* ctx, const IsenseeBuild* spec, fm_model** out) {
  const int kcode = spec->kcode, pz = kcode == 31 ? 1 : 2;
  FM_CHECK(spec->depth >= 2 && spec->depth <= 6, FM_EINVAL, "isensee: depth %d unsupported", spec->depth);
  FM_CHECK(spec->n_base_filters == 16 || spec->n_base_filters == 32, FM_EINVAL, "isensee: n_base_filters 16 or 32");
  FM_CHECK(spec->n_segmentation_levels >= 1 && spec->n_segmentation_levels <= spec->depth - 1, FM_EINVAL,
           "isensee: n_segmentation_levels %d out of range", spec->n_segmentation_levels);
  const int div = 1 << (spec->depth - 1);
  FM_CHECK(spec->X % div == 0 && spec->Y % div == 0 && (pz == 1 || spec->Z % div == 0) && spec->X > 0, FM_EINVAL,
           "isensee: input extent %dx%dx%d must be divisible by 2^(depth-1)=%d", spec->X, spec->Y, spec->Z, div);
  FM_CUDA(cudaSetDevice(ctx->device));
  fm_model* m = new fm_model();
  m->ctx = ctx;
  m->kind = 1;
  m->kcode = kcode;
  m->pz = pz;
  m->cin_real = spec->in_channels;
  m->nseg = spec->n_segmentation_levels;
  m->spec.in_channels = spec->in_channels;
  m->spec.X = spec->X;
  m->spec.Y = spec->Y;
  m->spec.Z = spec->Z;
  m->spec.depth = spec->depth;
  m->spec.n_base_filters = spec->n_base_filters;
  m->spec.n_labels = 1;
  const int D = spec->depth, nf = spec->n_base_filters;
  auto add_conv = [&](const char* fmt, int d, int c1, int c2, int cout, int k, int level, int stride, bool norm) {
    Layer l;
    memset(l.name, 0, sizeof(l.name));
    snprintf(l.name, sizeof(l.name), fmt, d);
    l.c1 = c1;
    l.c2 = c2;
    l.cout = cout;
    l.k = k;
    l.level = level;
    l.stride = stride;
    l.w_off = m->nparams;
    m->nparams += l.wcount();
    l.b_off = m->nparams;
    m->nparams = (m->nparams + cout + 3) & ~(int64_t)3;
    m->layers.push_back(l);
    if (norm) {
      Layer g;
      memset(g.name, 0, sizeof(g.name));
      snprintf(g.name, sizeof(g.name), "%s_norm", l.name);
      g.is_norm = 1;
      g.c1 = cout;
      g.c2 = 0;
      g.cout = cout;
      g.k = 1;
      g.level = level;
      g.w_off = m->nparams;
      m->nparams += cout;
      g.b_off = m->nparams;
      m->nparams = (m->nparams + cout + 3) & ~(int64_t)3;
      m->layers.push_back(g);
    }
  };
  // 2D: the first conv reads a 16-channel zero-padded bf16 copy of the input (tensor-core K granule)
  int c = kcode == 31 ? 16 : 1;
  for (int l = 0; l < D; ++l) {
    const int f = nf << l;
    add_conv("l%d_in", l, c, 0, f, kcode, l, l == 0 ? 1 : 2, true);
    if (l == 0 && kcode == 31) m->layers[m->layers.size() - 2].cin_real = spec->in_channels;
    add_conv("l%d_ctx1", l, f, 0, f, kcode, l, 1, true);
    add_conv("l%d_ctx2", l, f, 0, f, kcode, l, 1, true);
    c = f;
  }
  for (int l = D - 2; l >= 0; --l) {
    const int f = nf << l;
    add_conv("u%d_up", l, c, 0, f, kcode, l, 1, true);
    add_conv("u%d_loc1", l, f, f, f, kcode, l, 1, true);  // concat order [skip, up] (isensee2017.py:62)
    add_conv("u%d_loc2", l, f, 0, f, 1, l, 1, true);
    c = f;
    if (l < m->nseg) add_conv("u%d_seg", l, f, 0, 1, 1, l, 1, false);
  }
  const size_t pb = (size_t)m->nparams * sizeof(float);
  float** bufs[4] = {&m->params, &m->grads, &m->adam_m, &m->adam_v};
  for (auto b : bufs) {
    FM_CUDA(cudaMalloc((void**)b, pb));
    FM_CUDA(cudaMemset(*b, 0, pb));
  }
  FM_CUDA(cudaMalloc((void**)&m->sums, kNumLossSums * sizeof(double)));
  FM_CUDA(cudaMemset(m->sums, 0, kNumLossSums * sizeof(double)));
  int64_t pack_elems = 0;
  for (auto& l : m->layers)
    if (!l.is_norm) pack_elems += 2 * ((l.wcount() + 63) & ~(int64_t)63);
  FM_CUDA(cudaMalloc((void**)&m->wpack, (size_t)pack_elems * sizeof(bf16)));
  FM_CUDA(cudaMemset(m->wpack, 0, (size_t)pack_elems * sizeof(bf16)));
  bf16* wp = m->wpack;
  for (auto& l : m->layers) {
    if (l.is_norm) continue;
    const int64_t padded = (l.wcount() + 63) & ~(int64_t)63;
    l.w_f = wp;
    wp += padded;
    if (l.c1 >= 16) {  // dgrad packs (none for the Cin = 1 first conv)
      l.w_d0 = wp;
      l.w_d1 = wp + (int64_t)l.c1 * l.taps() * l.cout;
    }
    wp += padded;
    if (l.k != 3 || l.c1 < 16) continue;  // (the 2D family, k = 31, runs on the per-tap kernels)
    // the backward of a stride-2 conv runs as a stride-1 dgrad over the zero-inserted gradient, one level finer
    const int dl = l.stride == 2 ? l.level - 1 : l.level;
    const int X = spec->X >> l.level, Y = spec->Y >> l.level, Z = spec->Z >> l.level;
    const int Xd = spec->X >> dl, Yd = spec->Y >> dl, Zd = spec->Z >> dl;
    const int cs[2] = {l.c1, l.c2};
    if (l.stride == 1 && conv_march_supported(X, Y, Z, l.c1, l.c2, l.cout, l.k)) {
      l.march_f = true;
      for (int s = 0; s < (l.c2 ? 2 : 1); ++s)
        FM_CUDA(cudaMalloc((void**)&l.w_mf[s], (size_t)conv_march_pack_elems(cs[s], l.cout) * sizeof(bf16)));
    }
    for (int s = 0; s < (l.c2 ? 2 : 1); ++s)
      if (isensee_dgrad_marches(Xd, Yd, Zd, l.c1, cs[s], l.cout, l.k)) {
        l.march_d[s] = true;
        FM_CUDA(cudaMalloc((void**)&l.w_md[s], (size_t)conv_march_pack_elems(l.cout, cs[s]) * sizeof(bf16)));
      }
  }
  m->layer_done.resize(m->layers.size());
  for (auto& e : m->layer_done) FM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  {  // gradient buckets as for the plain U-Net: backward runs in reverse creation order
    const int nl = (int)m->layers.size();
    const int64_t target = m->nparams / 4 + 1;
    int hi = nl - 1;
    int64_t acc = 0;
    for (int i = nl - 1; i >= 0; --i) {
      acc += m->layers[i].wcount() + m->layers[i].cout;
      if (acc >= target || i == 0) {
        m->buckets.push_back({i, hi});
        hi = i - 1;
        acc = 0;
      }
    }
  }
  m->isRawL.resize(m->layers.size());
  m->isStatsL.resize(m->layers.size());
  m->gIsA.resize(D);
  m->gIsB.resize(D);
  m->gIsC.resize(D);
  m->gIsUp.resize(D);
  m->isDropL.resize(D);
  m->gSeg.resize(D);
  m->isIn.resize(D);
  m->isC1.resize(D);
  m->isSum.resize(D);
  m->isUp.resize(D);
  m->isU.resize(D);
  m->isLoc1.resize(D);
  m->isLoc2.resize(D);
  m->isSeg.resize(D);
  FM_CUDA(cudaEventCreateWithFlags(&m->ev_tmp, cudaEventDisableTiming));
  *out = m;
  return FM_OK;
}

static int ensure_capacity_isensee(fm_model* m, int B, bool train) {
  if (B <= m->cap && (!train || m->train_alloc)) return FM_OK;
  FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
  B = std::max(B, m->cap);
  const int D = m->depth(), nf = m->spec.n_base_filters;
  const size_t v0 = (size_t)m->vox(0);
  if (train || m->train_alloc) {
    FM_TRY(m->t_in.ensure((size_t)B * v0));
    FM_TRY(m->dz.ensure((size_t)B * v0));
    FM_TRY(m->gIsRaw.ensure((size_t)B * v0 * nf));
    FM_TRY(m->gIsZero.ensure((size_t)B * v0 * nf * 2));
    for (size_t i = 0; i < m->layers.size(); ++i) {
      const Layer& l = m->layers[i];
      if (l.is_norm || (l.k == 1 && l.cout == 1)) continue;
      FM_TRY(m->isRawL[i].ensure((size_t)B * m->vox(l.level) * l.cout));
      FM_TRY(m->isStatsL[i].ensure((size_t)B * l.cout * 2));
    }
    for (int l = 0; l < D; ++l) {
      const size_t n = (size_t)B * m->vox(l) * (nf << l);
      FM_TRY(m->gIsA[l].ensure(n));
      FM_TRY(m->gIsB[l].ensure(n));
      FM_TRY(m->gIsC[l].ensure(n));
      FM_TRY(m->isDropL[l].ensure((size_t)B * (nf << l)));
      if (l < D - 1) FM_TRY(m->gIsUp[l].ensure(2 * n));
      if (l >= 1 && l < m->nseg) FM_TRY(m->gSeg[l].ensure((size_t)B * m->vox(l)));
    }
    m->train_alloc = true;
  }
  FM_TRY(m->x_in.ensure((size_t)B * v0 * m->cin_real));
  if (m->kcode == 31) FM_TRY(m->x_pad.ensure((size_t)B * v0 * 16));
  FM_TRY(m->prob.ensure((size_t)B * v0));
  FM_TRY(m->isAcc.ensure((size_t)B * v0));
  FM_TRY(m->isRaw.ensure((size_t)B * v0 * nf));
  FM_TRY(m->isScratch.ensure((size_t)B * (nf << (D - 1)) * 2 * 1028));
  for (int l = 0; l < D; ++l) {
    const size_t n = (size_t)B * m->vox(l) * (nf << l);
    FM_TRY(m->isIn[l].ensure(n));
    FM_TRY(m->isC1[l].ensure(n));
    FM_TRY(m->isSum[l].ensure(n));
    if (l < D - 1) {
      FM_TRY(m->isUp[l].ensure((size_t)B * m->vox(l) * (nf << (l + 1))));
      FM_TRY(m->isU[l].ensure(n));
      FM_TRY(m->isLoc1[l].ensure(n));
      FM_TRY(m->isLoc2[l].ensure(n));
      if (l < m->nseg) FM_TRY(m->isSeg[l].ensure((size_t)B * m->vox(l)));
    }
  }
  m->cap = B;
  return FM_OK;
}

// one Isensee conv block: Conv3D (+bias) -> raw -> InstanceNorm + LeakyReLU (* dropout scale) (+ residual add) -> y.
// A training pass keeps the raw conv output and the norm statistics of every block for the backward pass.
static int isensee_block(fm_model* m, const Layer& l, const Layer& nl, const bf16* x1, const bf16* x2, const bf16* add,
                         bf16* y, int B, const float* chan_scale = nullptr) {
  fm_ctx* ctx = m->ctx;
  const Dims5 d = m->dims(l.level, l.cout, B);
  const float* bias = m->params + l.b_off;
  const int li = (int)(&l - &m->layers[0]);
  bf16* raw = m->train_pass ? m->isRawL[li].p : m->isRaw.p;
  float* stats = m->train_pass ? m->isStatsL[li].p : nullptr;
  if (l.c1 == 1) {
    // Cin = 1: bandwidth kernel, raw output (no activation)
    FM_TRY(k_conv3d_simt_fprop(ctx, x1, 1, nullptr, l.w_f, bias, raw, nullptr, B, d.X, d.Y, d.Z, 1, 0, l.cout, 3, 0,
                               nullptr));
  } else if (l.march_f) {
    FM_TRY(k_conv3d_march(ctx, x1, x2, l.w_mf[0], l.w_mf[1], bias, raw, nullptr, B, d.X, d.Y, d.Z, l.c1, l.c2, l.cout, 0,
                          l.cout, 0, reproducible_pass(m)));
  } else if (conv_tc_supported(l.c1, l.c2, l.cout, l.k)) {
    FM_TRY(k_conv3d_tc_fprop(ctx, x1, x2, l.w_f, bias, raw, nullptr, B, d.X, d.Y, d.Z, l.c1, l.c2, l.cout, l.k, 0,
                             l.cout, 0, l.stride, d.X * l.stride, d.Y * l.stride, m->pz == 2 ? d.Z * l.stride : d.Z));
  } else {
    FM_CHECK(l.stride == 1, FM_EINVAL, "isensee: strided conv %s has no fallback", l.name);
    FM_TRY(k_conv3d_simt_fprop(ctx, x1, 0, x2, l.w_f, bias, raw, nullptr, B, d.X, d.Y, d.Z, l.c1, l.c2, l.cout, l.k, 0,
                               nullptr));
  }
  return k_instnorm_lrelu(ctx, raw, m->params + nl.w_off, m->params + nl.b_off, add, y, B, m->vox(l.level), l.cout,
                          m->isScratch.p, m->isScratch.n, stats, chan_scale);
}

static int forward_isensee(fm_model* m, int B) {
  fm_ctx* ctx = m->ctx;
  const int D = m->depth();
  FM_TRY(refresh_packs(m));
  auto LI = [&](const char* fmt, int d) {
    char nm[32];
    snprintf(nm, sizeof(nm), fmt, d);
    return layer_index(m, nm);
  };
  const bf16* cur = nullptr;
  for (int l = 0; l < D; ++l) {
    const int i_in = LI("l%d_in", l), i_c1 = LI("l%d_ctx1", l), i_c2 = LI("l%d_ctx2", l);
    const Layer &lin = m->layers[i_in], &lc1 = m->layers[i_c1], &lc2 = m->layers[i_c2];
    const bf16* src = cur;
    if (l == 0 && m->kcode == 31) {
      FM_TRY(k_pad_cast(ctx, m->x_in.p, m->x_pad.p, (int64_t)B * m->vox(0), m->cin_real, 16));
      src = m->x_pad.p;
    } else if (l == 0) {
      src = (const bf16*)m->x_in.p;  // fp32 single-channel input, read by the Cin = 1 kernel
    }
    FM_TRY(isensee_block(m, lin, m->layers[i_in + 1], src, nullptr, nullptr, m->isIn[l].p, B));
    // SpatialDropout3D between the two context convs (isensee2017.py:103-105): training passes only
    const float* drop = nullptr;
    if (m->train_pass && m->dropout_rate > 0.f) {
      FM_TRY(k_dropout_scale(ctx, m->isDropL[l].p, B * lc1.cout, m->dropout_rate,
                             m->dropout_seed + (uint64_t)m->iterations * 64 + (uint64_t)l));
      drop = m->isDropL[l].p;
    }
    FM_TRY(isensee_block(m, lc1, m->layers[i_c1 + 1], m->isIn[l].p, nullptr, nullptr, m->isC1[l].p, B, drop));
    // context output + residual: summation = in_conv + context (isensee2017.py:55)
    FM_TRY(isensee_block(m, lc2, m->layers[i_c2 + 1], m->isC1[l].p, nullptr, m->isIn[l].p, m->isSum[l].p, B));
    cur = m->isSum[l].p;
  }
  for (int l = D - 2; l >= 0; --l) {
    const int i_up = LI("u%d_up", l), i_l1 = LI("u%d_loc1", l), i_l2 = LI("u%d_loc2", l);
    const Layer& lup = m->layers[i_up];
    FM_TRY(k_upsample3d_fwd(ctx, cur, m->isUp[l].p, m->dims(l + 1, lup.c1, B), m->pz));
    FM_TRY(isensee_block(m, lup, m->layers[i_up + 1], m->isUp[l].p, nullptr, nullptr, m->isU[l].p, B));
    FM_TRY(isensee_block(m, m->layers[i_l1], m->layers[i_l1 + 1], m->isSum[l].p, m->isU[l].p, nullptr, m->isLoc1[l].p, B));
    FM_TRY(isensee_block(m, m->layers[i_l2], m->layers[i_l2 + 1], m->isLoc1[l].p, nullptr, nullptr, m->isLoc2[l].p, B));
    cur = m->isLoc2[l].p;
    if (l < m->nseg) {
      const Layer& ls = m->layers[LI("u%d_seg", l)];
      FM_TRY(k_head_fwd(ctx, cur, m->params + ls.w_off, m->params + ls.b_off, m->isSeg[l].p, (int64_t)B * m->vox(l),
                        ls.c1, 0));
    }
  }
  // deep-supervision sum, coarse to fine (isensee2017.py:68-77), then sigmoid (:79)
  const float* acc = m->isSeg[m->nseg - 1].p;
  for (int l = m->nseg - 2; l >= 0; --l) {
    const Dims5 d = m->dims(l, 1, B);
    float* dst = (l == 0) ? m->isAcc.p : m->isSeg[l].p;  // in place on the finer map is safe (element-wise)
    FM_TRY(k_seg_upsample_add(ctx, m->isSeg[l].p, acc, dst, B, d.X, d.Y, d.Z, m->pz));
    acc = dst;
  }
  FM_TRY(k_sigmoid(ctx, acc, m->prob.p, (int64_t)B * m->vox(0)));
  return FM_OK;
}


// ---------------------------------------------------------------------------------------------
// Isensee backward. Per block: (InstanceNorm + LeakyReLU [+ dropout]) backward -> gradient of the raw conv output
// (gIsRaw), bias / weight gradients, dgrad to the block input(s). Fan-outs: in_conv feeds ctx1 and the residual
// add; summation[l] feeds the next level's stride-2 in_conv and the decoder's concat (or the first upsampling at
// the bottom); loc2[l] feeds its segmentation head and the next upsampling. The stride-2 convs go backward as
// stride-1 dgrad / wgrad over the zero-inserted gradient (k_zero_insert), one level finer.
// Gradients are produced in reverse layer-creation order, so the all-reduce buckets work as for the plain U-Net.
// ---------------------------------------------------------------------------------------------
// Kernel choice of the Isensee weight / data gradients, shared with the per-op hook fm_op_conv_strided so that the
// hook runs what the model runs. Weight gradient of one source (cs of cin_total channels at cofs): marching, per-tap
// tensor-core or SIMT kernel.
static int isensee_wgrad_route(fm_ctx* ctx, const bf16* x, const bf16* dy, float* dw, int B, int X, int Y, int Z, int cs,
                               int cin_total, int cofs, int cout, int k) {
  if (conv_wgrad_march_supported(X, Y, Z, cs, cout, k))
    return k_conv3d_wgrad_march(ctx, x, dy, dw, B, X, Y, Z, cs, cin_total, cofs, cout);
  if (conv_tc_supported(cs, 0, cout, k))
    return k_conv3d_tc_wgrad(ctx, x, dy, dw, B, X, Y, Z, cs, cin_total, cofs, cout, k);
  return k_conv3d_simt_wgrad(ctx, x, 0, dy, dw, B, X, Y, Z, cs, cin_total, cofs, cout, k);
}

// data gradient towards one source: w_md = its marching pack (null: per-tap tensor-core or SIMT kernel on w_d)
static int isensee_dgrad_route(fm_ctx* ctx, const bf16* dy, const bf16* w_md, const bf16* w_d, bf16* dx, int B, int X,
                               int Y, int Z, int cout, int cs, int k, bool reproducible) {
  if (w_md != nullptr)
    return k_conv3d_march(ctx, dy, nullptr, w_md, nullptr, nullptr, dx, nullptr, B, X, Y, Z, cout, 0, cs, 0, cs, 0,
                          reproducible);
  if (conv_tc_supported(cout, 0, cs, k))
    return k_conv3d_tc_fprop(ctx, dy, nullptr, w_d, nullptr, dx, nullptr, B, X, Y, Z, cout, 0, cs, k, 0, cs, 0);
  return k_conv3d_simt_fprop(ctx, dy, 0, nullptr, w_d, nullptr, dx, nullptr, B, X, Y, Z, cout, 0, cs, k, 0, nullptr);
}

static int is_wgrad(fm_model* m, const Layer& l, int level, const bf16* x1, const bf16* x2, const bf16* dy, int B) {
  const Dims5 d = m->dims(level, l.cout, B);
  const bf16* xs[2] = {x1, x2};
  const int cs[2] = {l.c1, l.c2};
  int cofs = 0;
  // no bias gradient here: every Isensee conv feeds an InstanceNormalization, which removes a per-channel constant -
  // the gradient of such a bias is exactly zero (the heads, which have a live bias, are 1x1x1 kernels handled elsewhere)
  for (int s = 0; s < (l.c2 ? 2 : 1); ++s) {
    FM_TRY(isensee_wgrad_route(m->ctx, xs[s], dy, m->grads + l.w_off, B, d.X, d.Y, d.Z, cs[s], l.cin(), cofs, l.cout,
                               l.k));
    cofs += cs[s];
  }
  return FM_OK;
}

static int is_dgrad(fm_model* m, const Layer& l, int level, int src, const bf16* dy, bf16* dx, int B) {
  const Dims5 d = m->dims(level, l.cout, B);
  return isensee_dgrad_route(m->ctx, dy, l.march_d[src] ? l.w_md[src] : nullptr, src == 0 ? l.w_d0 : l.w_d1, dx, B, d.X,
                             d.Y, d.Z, l.cout, src == 0 ? l.c1 : l.c2, l.k, reproducible_pass(m));
}

// norm + activation backward of block `li` -> m->gIsRaw (gradient of the raw conv output); gamma/beta/bias gradients
static int is_block_bwd(fm_model* m, int li, const bf16* gy, const bf16* gy2, const float* chan_scale, int B) {
  const Layer &l = m->layers[li], &nl = m->layers[li + 1];
  FM_TRY(k_instnorm_lrelu_bwd(m->ctx, m->isRawL[li].p, m->isStatsL[li].p, m->params + nl.w_off, m->params + nl.b_off, gy,
                              gy2, chan_scale, m->gIsRaw.p, m->grads + nl.w_off, m->grads + nl.b_off, B, m->vox(l.level),
                              l.cout, m->isScratch.p, m->isScratch.n));
  FM_TRY(mark_layer_done(m, nl));
  // no bias-gradient pass: the conv bias sits in front of an InstanceNormalization, which removes any per-channel
  // constant - its gradient is exactly zero (the buffer was zeroed at the start of the backward pass); summing gIsRaw
  // over the voxels would only return the rounding noise of a sum that vanishes analytically
  return FM_OK;
}

static int backward_isensee(fm_model* m, int B) {
  fm_ctx* ctx = m->ctx;
  const int D = m->depth();
  const int64_t n0 = (int64_t)B * m->vox(0);
  auto LI = [&](const char* fmt, int d) {
    char nm[32];
    snprintf(nm, sizeof(nm), fmt, d);
    return layer_index(m, nm);
  };
  FM_TRY(k_zero(ctx, m->grads, (size_t)m->nparams * sizeof(float)));
  // d(loss)/d(summed logits); the deep-supervision sum hands the same gradient, 2^3 sum-pooled, to every head
  FM_TRY(k_dice_bwd(ctx, m->prob.p, m->t_in.p, m->sums, n0, m->dz.p, 1, m->xent()));
  std::vector<const float*> gseg(D, nullptr);
  gseg[0] = m->dz.p;
  for (int l = 1; l < m->nseg; ++l) {
    const Dims5 d = m->dims(l, 1, B);
    FM_TRY(k_sumpool_f32(ctx, gseg[l - 1], m->gSeg[l].p, B, d.X, d.Y, d.Z, m->pz));
    gseg[l] = m->gSeg[l].p;
  }
  for (int l = 0; l <= D - 2; ++l) {
    const int i_up = LI("u%d_up", l), i_l1 = LI("u%d_loc1", l), i_l2 = LI("u%d_loc2", l);
    const Layer &lup = m->layers[i_up], &ll1 = m->layers[i_l1], &ll2 = m->layers[i_l2];
    // gradient of loc2[l] (gIsA[l]): upsampling path (already stored for l > 0) + segmentation head
    if (l < m->nseg) {
      const Layer& ls = m->layers[LI("u%d_seg", l)];
      FM_TRY(k_head_bwd(ctx, m->isLoc2[l].p, gseg[l], m->params + ls.w_off, m->gIsA[l].p, m->grads + ls.w_off,
                        m->grads + ls.b_off, (int64_t)B * m->vox(l), ls.c1, l > 0 ? 2 : 1));
      FM_TRY(mark_layer_done(m, ls));
    }
    FM_TRY(is_block_bwd(m, i_l2, m->gIsA[l].p, nullptr, nullptr, B));
    FM_TRY(is_wgrad(m, ll2, l, m->isLoc1[l].p, nullptr, m->gIsRaw.p, B));
    FM_TRY(mark_layer_done(m, ll2));
    FM_TRY(is_dgrad(m, ll2, l, 0, m->gIsRaw.p, m->gIsB[l].p, B));
    FM_TRY(is_block_bwd(m, i_l1, m->gIsB[l].p, nullptr, nullptr, B));
    FM_TRY(is_wgrad(m, ll1, l, m->isSum[l].p, m->isU[l].p, m->gIsRaw.p, B));
    FM_TRY(mark_layer_done(m, ll1));
    FM_TRY(is_dgrad(m, ll1, l, 0, m->gIsRaw.p, m->gIsC[l].p, B));  // skip part of d(summation[l])
    FM_TRY(is_dgrad(m, ll1, l, 1, m->gIsRaw.p, m->gIsA[l].p, B));  // d(up block output)
    FM_TRY(is_block_bwd(m, i_up, m->gIsA[l].p, nullptr, nullptr, B));
    FM_TRY(is_wgrad(m, lup, l, m->isUp[l].p, nullptr, m->gIsRaw.p, B));
    FM_TRY(mark_layer_done(m, lup));
    FM_TRY(is_dgrad(m, lup, l, 0, m->gIsRaw.p, m->gIsUp[l].p, B));
    bf16* gdst = (l + 1 == D - 1) ? m->gIsC[D - 1].p : m->gIsA[l + 1].p;
    FM_TRY(k_upsample3d_bwd(ctx, m->gIsUp[l].p, nullptr, gdst, m->dims(l + 1, lup.c1, B), lup.c1, 0, m->pz));
  }
  for (int l = D - 1; l >= 0; --l) {
    const int i_in = LI("l%d_in", l), i_c1 = LI("l%d_ctx1", l), i_c2 = LI("l%d_ctx2", l);
    const Layer &lin = m->layers[i_in], &lc1 = m->layers[i_c1], &lc2 = m->layers[i_c2];
    const bf16* gsum = m->gIsC[l].p;  // complete d(summation[l])
    FM_TRY(is_block_bwd(m, i_c2, gsum, nullptr, nullptr, B));
    FM_TRY(is_wgrad(m, lc2, l, m->isC1[l].p, nullptr, m->gIsRaw.p, B));
    FM_TRY(mark_layer_done(m, lc2));
    FM_TRY(is_dgrad(m, lc2, l, 0, m->gIsRaw.p, m->gIsA[l].p, B));
    const float* drop = m->dropout_rate > 0.f ? m->isDropL[l].p : nullptr;
    FM_TRY(is_block_bwd(m, i_c1, m->gIsA[l].p, nullptr, drop, B));
    FM_TRY(is_wgrad(m, lc1, l, m->isIn[l].p, nullptr, m->gIsRaw.p, B));
    FM_TRY(mark_layer_done(m, lc1));
    FM_TRY(is_dgrad(m, lc1, l, 0, m->gIsRaw.p, m->gIsB[l].p, B));
    // in_conv output feeds ctx1 and the residual add
    FM_TRY(is_block_bwd(m, i_in, m->gIsB[l].p, gsum, nullptr, B));
    if (l == 0 && m->kcode == 31) {
      FM_TRY(is_wgrad(m, lin, 0, m->x_pad.p, nullptr, m->gIsRaw.p, B));  // the zero-padded 16-channel input copy
      FM_TRY(mark_layer_done(m, lin));
    } else if (l == 0) {
      const Dims5 dd = m->dims(0, lin.cout, B);
      FM_TRY(k_conv3d_simt_wgrad(ctx, m->x_in.p, 1, m->gIsRaw.p, m->grads + lin.w_off, B, dd.X, dd.Y, dd.Z, 1, 1, 0,
                                 lin.cout, 3));
      FM_TRY(mark_layer_done(m, lin));
    } else {
      FM_TRY(k_zero_insert(ctx, m->gIsRaw.p, m->gIsZero.p, m->dims(l, lin.cout, B), m->pz));
      FM_TRY(is_wgrad(m, lin, l - 1, m->isSum[l - 1].p, nullptr, m->gIsZero.p, B));
      FM_TRY(mark_layer_done(m, lin));
      FM_TRY(is_dgrad(m, lin, l - 1, 0, m->gIsZero.p, m->gIsA[l - 1].p, B));
      FM_TRY(k_add_bf16(ctx, m->gIsC[l - 1].p, m->gIsA[l - 1].p, m->gIsC[l - 1].p,
                        (int64_t)B * m->vox(l - 1) * lin.c1));
    }
  }
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------
// inference
// ---------------------------------------------------------------------------------------------
extern "C" int fm_predict_device(fm_model* m, uint64_t x_dev, int batch, uint64_t y_dev) {
  FM_CHECK(m && batch > 0, FM_EINVAL, "fm_predict_device: bad argument");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  FM_TRY(ensure_capacity(m, batch, false));
  const size_t n = (size_t)batch * m->vox(0);
  FM_CUDA(cudaMemcpyAsync(m->x_in.p, (const void*)(uintptr_t)x_dev, n * m->cin_real * 4, cudaMemcpyDeviceToDevice,
                          m->ctx->stream));
  FM_TRY(forward(m, batch));
  if (y_dev)
    FM_CUDA(cudaMemcpyAsync((void*)(uintptr_t)y_dev, m->prob.p, n * 4, cudaMemcpyDeviceToDevice,
                            m->ctx->stream));
  m->fwd_valid = false;
  return FM_OK;
}

extern "C" int fm_predict(fm_model* m, const float* x, int batch, float* y) {
  FM_CHECK(m && x && y && batch > 0, FM_EINVAL, "fm_predict: bad argument");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  FM_TRY(ensure_capacity(m, batch, false));
  const size_t n = (size_t)batch * m->vox(0);
  FM_TRY(upload(m, x, m->x_in.p, n * m->cin_real));
  FM_TRY(forward(m, batch));
  FM_CUDA(cudaMemcpyAsync(y, m->prob.p, n * 4, cudaMemcpyDeviceToHost, m->ctx->stream));
  FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
  m->fwd_valid = false;
  return FM_OK;
}

extern "C" int fm_patch_plan(const int32_t padded[3], const int32_t patch[3], const int32_t pred[3],
                             double overlap_factor, int32_t* out_idx, int64_t cap, int64_t* out_n) {
  FM_CHECK(padded && patch && pred && out_n, FM_EINVAL, "fm_patch_plan: NULL argument");
  std::vector<int32_t> starts[3];
  for (int a = 0; a < 3; ++a) {
    const int min_ov = patch[a] - pred[a];
    const int max_ov = patch[a] - 1;
    // prediction.py:137: (overlap_factor * (max - min)).astype(int) truncates toward zero
    const int ov = min_ov + (int)(overlap_factor * (double)(max_ov - min_ov));
    const int step = patch[a] - ov;
    const int stop = padded[a] - patch[a];
    FM_CHECK(step > 0, FM_EINVAL, "fm_patch_plan: non-positive step on axis %d (overlap_factor %g)", a,
             overlap_factor);
    FM_CHECK(stop >= 0, FM_EINVAL, "fm_patch_plan: padded extent %d smaller than patch %d on axis %d",
             padded[a], patch[a], a);
    for (int s = 0; s <= stop; s += step) starts[a].push_back(s);  // range(0, stop+1, step)
    if (stop % step > 0) starts[a].push_back(stop);                // prediction.py:93-94
  }
  const int64_t n = (int64_t)starts[0].size() * starts[1].size() * starts[2].size();
  *out_n = n;
  if (out_idx == nullptr) return FM_OK;
  FM_CHECK(cap >= n, FM_EINVAL, "fm_patch_plan: capacity %lld < %lld patches", (long long)cap, (long long)n);
  int64_t i = 0;
  for (int32_t x : starts[0])
    for (int32_t y : starts[1])
      for (int32_t z : starts[2]) {
        out_idx[i * 3] = x;
        out_idx[i * 3 + 1] = y;
        out_idx[i * 3 + 2] = z;
        ++i;
      }
  return FM_OK;
}

extern "C" int fm_gather_patches(fm_ctx* ctx, const float* vol, const int32_t vol_dims[3],
                                 const int32_t halo_pad[6], const int32_t fit_pad[6],
                                 const double pad_value[2], const int32_t* idx, int64_t n,
                                 const int32_t patch[3], float* out) {
  FM_CHECK(ctx && vol && vol_dims && halo_pad && fit_pad && pad_value && idx && patch && out && n > 0,
           FM_EINVAL, "fm_gather_patches: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  const size_t nv = (size_t)vol_dims[0] * vol_dims[1] * vol_dims[2];
  const size_t np = (size_t)n * patch[0] * patch[1] * patch[2];
  DevBuf<float> dvol, dout;
  DevBuf<int32_t> didx;
  FM_TRY(dvol.ensure(nv));
  FM_TRY(dout.ensure(np));
  FM_TRY(didx.ensure((size_t)n * 3));
  FM_CUDA(cudaMemcpyAsync(dvol.p, vol, nv * 4, cudaMemcpyHostToDevice, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(didx.p, idx, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
  int r = k_gather_patches(ctx, dvol.p, vol_dims, halo_pad, fit_pad, (float)pad_value[0],
                           (float)pad_value[1], didx.p, n, patch, dout.p);
  if (r == FM_OK) {
    cudaError_t e = cudaMemcpyAsync(out, dout.p, np * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      fm_set_error("fm_gather_patches: %s", cudaGetErrorString(e));
      r = FM_ECUDA;
    }
  }
  cudaStreamSynchronize(ctx->stream);
  dvol.release();
  dout.release();
  didx.release();
  return r;
}

extern "C" int fm_reassemble(fm_ctx* ctx, const float* preds, const int32_t* idx, int64_t n,
                             const int32_t pred_shape[3], int channels, const int32_t out_dims[3],
                             double* out, int16_t* out_count) {
  FM_CHECK(ctx && preds && idx && pred_shape && out_dims && out && n > 0 && channels > 0, FM_EINVAL,
           "fm_reassemble: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  const size_t np = (size_t)n * pred_shape[0] * pred_shape[1] * pred_shape[2] * channels;
  const size_t nvox = (size_t)out_dims[0] * out_dims[1] * out_dims[2];
  DevBuf<float> dp;
  DevBuf<double> dout;
  DevBuf<int16_t> dcnt;
  FM_TRY(dp.ensure(np));
  FM_TRY(dout.ensure(nvox * channels));
  FM_TRY(dcnt.ensure(nvox));
  FM_CUDA(cudaMemcpyAsync(dp.p, preds, np * 4, cudaMemcpyHostToDevice, ctx->stream));
  int r = k_reassemble(ctx, dp.p, idx, n, 0, n, 0, pred_shape, channels, out_dims, dout.p, dcnt.p, 1);
  if (r == FM_OK) {
    cudaError_t e = cudaMemcpyAsync(out, dout.p, nvox * channels * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && out_count)
      e = cudaMemcpyAsync(out_count, dcnt.p, nvox * 2, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      fm_set_error("fm_reassemble: %s", cudaGetErrorString(e));
      r = FM_ECUDA;
    }
  }
  cudaStreamSynchronize(ctx->stream);
  dp.release();
  dout.release();
  dcnt.release();
  return r;
}

// ---------------------------------------------------------------------------------------------
// post-processing (postprocess.cu)
// ---------------------------------------------------------------------------------------------
static int check_pp_spec(const fm_postprocess_spec* spec, const int32_t dims[3]) {
  FM_CHECK(spec && spec->weights && spec->radius >= 0, FM_EINVAL, "post-processing: bad spec");
  FM_CHECK(dims[0] > 0 && dims[1] > 0 && dims[2] > 0, FM_EINVAL, "post-processing: dims %d x %d x %d", dims[0],
           dims[1], dims[2]);
  FM_CHECK((int64_t)dims[0] * dims[1] * dims[2] <= INT32_MAX, FM_EINVAL,
           "post-processing: %d x %d x %d voxels exceed 2^31 - 1", dims[0], dims[1], dims[2]);
  return FM_OK;
}

// mask (and the component count) of the last k_postprocess to the host, through the pinned staging area at `pin`
static int pp_download(fm_ctx* ctx, const PostprocBuffers& b, size_t nvox, const fm_postprocess_spec* spec, char* pin,
                       uint8_t* mask, int64_t* n_components) {
  FM_CUDA(cudaMemcpyAsync(pin, b.stats, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(pin + 256, b.mask, nvox, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  host_copy(mask, pin + 256, nvox);
  if (n_components) *n_components = spec->connected_component ? (int64_t)((unsigned long long*)pin)[0] : -1;
  return FM_OK;
}

extern "C" int fm_postprocess(fm_ctx* ctx, const void* pred, int dtype, const int32_t dims[3],
                              const fm_postprocess_spec* spec, uint8_t* mask, int64_t* n_components) {
  FM_CHECK(ctx && pred && dims && mask, FM_EINVAL, "fm_postprocess: bad argument");
  FM_CHECK(dtype == FM_DTYPE_FLOAT32 || dtype == FM_DTYPE_FLOAT64, FM_EINVAL, "fm_postprocess: dtype %d", dtype);
  FM_TRY(check_pp_spec(spec, dims));
  FM_CUDA(cudaSetDevice(ctx->device));
  const size_t nvox = (size_t)dims[0] * dims[1] * dims[2], es = dtype == FM_DTYPE_FLOAT64 ? 8 : 4;
  PostprocBuffers b;
  FM_TRY(pp_buffers(ctx, (int64_t)nvox, spec->radius, &b));
  // pinned staging: [map | stats | mask]
  const size_t in_bytes = (nvox * es + 4095) & ~(size_t)4095;
  void* pin = nullptr;
  FM_TRY(fm_ctx_pinned(ctx, in_bytes + 256 + nvox, &pin));
  host_copy(pin, pred, nvox * es);
  FM_CUDA(cudaMemcpyAsync(b.field1, pin, nvox * es, cudaMemcpyHostToDevice, ctx->stream));
  FM_TRY(k_postprocess(ctx, b, b.field1, dtype, (int64_t)dims[1] * dims[2], dims[2], dims, spec));
  return pp_download(ctx, b, nvox, spec, (char*)pin + in_bytes, mask, n_components);
}

extern "C" int fm_op_gaussian3d(fm_ctx* ctx, const void* in, int dtype, const int32_t dims[3], int radius,
                                const double* weights, void* out) {
  FM_CHECK(ctx && in && dims && weights && out && radius >= 0, FM_EINVAL, "fm_op_gaussian3d: bad argument");
  FM_CHECK(dtype == FM_DTYPE_FLOAT32 || dtype == FM_DTYPE_FLOAT64, FM_EINVAL, "fm_op_gaussian3d: dtype %d", dtype);
  fm_postprocess_spec spec = {radius, weights, 0.0, 0, 0};
  FM_TRY(check_pp_spec(&spec, dims));
  FM_CUDA(cudaSetDevice(ctx->device));
  const size_t nvox = (size_t)dims[0] * dims[1] * dims[2], es = dtype == FM_DTYPE_FLOAT64 ? 8 : 4;
  PostprocBuffers b;
  FM_TRY(pp_buffers(ctx, (int64_t)nvox, radius, &b));
  FM_CUDA(cudaMemcpyAsync(b.field1, in, nvox * es, cudaMemcpyHostToDevice, ctx->stream));
  FM_TRY(k_gaussian3d(ctx, b, b.field1, dtype, (int64_t)dims[1] * dims[2], dims[2], dims, radius, weights, b.field0));
  FM_CUDA(cudaMemcpyAsync(out, b.field0, nvox * es, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  return FM_OK;
}

// reduce_root < 0: `out` receives this shard's result (the average for shard 0 of 1, the partial SUM otherwise).
// reduce_root >= 0: the partial sums are reduced on the ctx communicator to that rank, which divides by the counts and
// is the only one to copy anything back to the host.
// pp != null (fm_patchwise_segment; single GPU): the cropped result is post-processed on the device into `pp_mask`;
// `out` is then optional.
static bool is_pinned_host(const void* p);

// patch extent in the padded volume (`nslices` deep for the 2D model), the prediction extent it yields
// (prediction.py:131-134) and the padded output extent (prediction.py:169); checks the halo pads against them
static int pw_extents(const fm_model* m, int nslices, const int32_t vol_dims[3], const int32_t halo_pad[6],
                      const int32_t fit_pad[6], int32_t patch[3], int32_t pred[3], int32_t out_dims[3]) {
  const bool is2d = m->kcode == 31;
  patch[0] = pred[0] = m->spec.X;
  patch[1] = pred[1] = m->spec.Y;
  patch[2] = nslices;
  pred[2] = is2d ? 1 : m->spec.Z;
  for (int a = 0; a < 3; ++a) {
    FM_CHECK(halo_pad[2 * a] + halo_pad[2 * a + 1] == patch[a] - pred[a], FM_EINVAL,
             "fm_patchwise_predict: halo pad on axis %d must total patch - prediction = %d", a, patch[a] - pred[a]);
    out_dims[a] = vol_dims[a] + fit_pad[2 * a] + fit_pad[2 * a + 1];
  }
  return FM_OK;
}

// Patches per network launch for `nloc` patches in `ngroups` x groups of `ppg`, given the caller's `batch`.
static int pw_sub_batch(const fm_model* m, int batch, int64_t nloc, int ngroups, int ppg) {
  if (batch <= ppg || ngroups < 3) return batch;
  // cut so that a sub-batch fills the SMs in whole waves: the marching kernels run one 16 x 8 column per CTA, a
  // patch has cpp columns, and q patches (q = SMs / gcd(SMs, cpp); 37 for 64^3 patches on 148 SMs) are a whole
  // number of waves for them and for the 128-voxel tiles of the deeper levels. The first cut keeps ~3/4 of the
  // patches (its finished output slabs travel back while the remainder runs); 2D models keep whole x groups.
  const int64_t cpp = m->kcode == 31 ? 0 : (int64_t)(m->spec.Y / 16) * (m->spec.Z / 8);
  int64_t q = 0;
  if (cpp > 0) {
    int64_t a = m->ctx->num_sms, b = cpp;
    while (b) {
      const int64_t t = a % b;
      a = b;
      b = t;
    }
    q = m->ctx->num_sms / a;
  }
  if (q > 0 && nloc > q)
    return (int)std::min<int64_t>(batch, q * std::max<int64_t>(1, std::min<int64_t>(2, (nloc * 3 / 4) / q)));
  if (q == 0) return (int)std::min<int64_t>(batch, (int64_t)ppg * std::max(1, ngroups / 8));
  return batch;
}

static int patchwise_impl(fm_model* m, const float* vol, const int32_t vol_dims[3], const int32_t halo_pad[6],
                          const int32_t fit_pad[6], const double pad_value[2], const int32_t* idx, int64_t n, int batch,
                          int shard_rank, int shard_count, int reduce_root, const float* truth, int prev_truth_index,
                          int prev_truth_size, double* out, int16_t* out_count,
                          const fm_postprocess_spec* pp = nullptr, uint8_t* pp_mask = nullptr,
                          int64_t* pp_components = nullptr) {
  const bool want_out = (reduce_root < 0 || shard_rank == reduce_root) && (out || !pp);
  FM_CHECK(m && vol && vol_dims && halo_pad && fit_pad && pad_value && idx && (out || !want_out) && n > 0 && batch > 0,
           FM_EINVAL, "fm_patchwise_predict: bad argument");
  if (pp) {
    FM_CHECK(pp_mask && shard_count == 1 && reduce_root < 0, FM_EINVAL,
             "fm_patchwise_segment: needs a mask and a single shard");
    FM_TRY(check_pp_spec(pp, vol_dims));
  }
  FM_CHECK(shard_count >= 1 && shard_rank >= 0 && shard_rank < shard_count, FM_EINVAL,
           "fm_patchwise_predict: shard %d of %d", shard_rank, shard_count);
  fm_ctx* ctx = m->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  const bool is2d = m->kcode == 31;
  const int nslices = is2d ? m->cin_real - (truth ? prev_truth_size : 0) : m->spec.Z;
  FM_CHECK(!truth || (is2d && prev_truth_size > 0 && prev_truth_size < m->cin_real), FM_EINVAL,
           "fm_patchwise_predict: truth conditioning needs a 2D model with in_channels > prev_truth_size");
  // The truth slices are gathered with zero fill outside the padded truth volume; the reference edge-replicates there
  // (get_patch_from_3d_data -> fix_out_of_bound_patch_attempt, mode='edge'). The two agree as long as the slices stay
  // inside the patch's own z range, whose halo is zero-padded on both sides - anything else is refused, not approximated.
  FM_CHECK(!truth || (prev_truth_index >= 0 && prev_truth_index + prev_truth_size <= nslices), FM_EINVAL,
           "fm_patchwise_predict: previous-truth slices [%d, %d) must lie inside the patch depth %d", prev_truth_index,
           prev_truth_index + prev_truth_size, nslices);
  int32_t patch[3], pred[3], out_dims[3];
  FM_TRY(pw_extents(m, nslices, vol_dims, halo_pad, fit_pad, patch, pred, out_dims));
  const size_t nv = (size_t)vol_dims[0] * vol_dims[1] * vol_dims[2];
  const size_t nout = (size_t)out_dims[0] * out_dims[1] * out_dims[2];
  const size_t pv = (size_t)pred[0] * pred[1] * pred[2];  // predicted voxels per patch
  const int64_t lo = n * shard_rank / shard_count, hi = n * (shard_rank + 1) / shard_count;
  const int64_t nloc = hi - lo;
  batch = (int)std::min<int64_t>(batch, std::max<int64_t>(nloc, 1));
  // the reassembly plan also validates the corner list (x-major Cartesian product, every voxel covered)
  ReasmPlan* plan = nullptr;
  FM_TRY(k_reassemble_prepare(ctx, idx, n, pred, 1, out_dims, &plan));
  struct PlanGuard {
    ReasmPlan* p;
    ~PlanGuard() { k_reassemble_release(p); }
  } plan_guard{plan};
  const int32_t* xstarts = nullptr;
  int ngroups = 0, ppg = 0;
  k_reassemble_groups(plan, &xstarts, &ngroups, &ppg);
  // PIPELINE: the patch list is x-major, so output rows below the x corner of the next unprocessed patch are final.
  // A large caller batch is therefore cut into sub-batches of whole x groups: the volume is uploaded slab by slab on
  // the copy stream just ahead of the patches that need it, and finished output slabs are overlap-added, copied back
  // and un-staged while the network still works on later patches. The network is bit-reproducible and batch-invariant,
  // so the result does not depend on the cut.
  batch = pw_sub_batch(m, batch, nloc, ngroups, ppg);
  FM_TRY(ensure_capacity(m, batch, false));
  DevBuf<float>&dvol = m->pw_vol, &dpred = m->pw_pred;
  DevBuf<int32_t>& didx = m->pw_idx;
  DevBuf<double>& dout = m->pw_out;
  DevBuf<int16_t>& dcnt = m->pw_cnt;
  FM_TRY(dvol.ensure(nv * (truth ? 2 : 1)));
  FM_TRY(dpred.ensure(std::max<size_t>(1, (size_t)nloc) * pv));
  FM_TRY(didx.ensure((size_t)n * 3));
  FM_TRY(dout.ensure(nout));
  FM_TRY(dcnt.ensure(nout));
  const bool trace = getenv("FETAL_B200_TRACE") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto t_start = now();
  auto lap = [&](const char* what) {
    if (!trace) return;
    auto t = now();
    fprintf(stderr, "[fm_patchwise_predict] %-22s %8.3f ms\n", what,
            std::chrono::duration<double, std::milli>(t - t_start).count());
    t_start = t;
  };
  // host <-> device through the context's pinned staging buffer (pageable cudaMemcpy runs at a fraction of PCIe):
  // [volume | truth | float64 result | int16 counts | post-processing stats + mask]
  const size_t in_bytes = (nv * sizeof(float) * (truth ? 2 : 1) + 4095) & ~(size_t)4095;
  const size_t out_bytes = pp && !out ? 0 : nout * sizeof(double), cnt_bytes = out_count ? nout * sizeof(int16_t) : 0;
  const size_t cnt_off = in_bytes + ((out_bytes + 4095) & ~(size_t)4095);
  const size_t pp_off = cnt_off + ((cnt_bytes + 4095) & ~(size_t)4095);
  void* pin = nullptr;
  FM_TRY(fm_ctx_pinned(ctx, pp ? pp_off + 256 + nv : cnt_off + cnt_bytes, &pin));
  char* pin_in = (char*)pin;
  char* pin_out = (char*)pin + in_bytes;
  char* pin_cnt = (char*)pin + cnt_off;
  if ((int)m->pw_events.size() < ngroups + 2) {
    const size_t old = m->pw_events.size();
    m->pw_events.resize((size_t)ngroups + 2, nullptr);
    for (size_t i = old; i < m->pw_events.size(); ++i)
      FM_CUDA(cudaEventCreateWithFlags(&m->pw_events[i], cudaEventDisableTiming));
  }
  cudaEvent_t ev_up = m->pw_events[0], ev_rows = m->pw_events[1];
  lap("workspace");
  FM_CUDA(cudaMemcpyAsync(didx.p, idx, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
  if (shard_count > 1) FM_CUDA(cudaMemsetAsync(dout.p, 0, nout * 8, ctx->stream));  // partial sums accumulate
  // the copy stream starts behind everything queued so far (nothing of an earlier call may still read the buffers)
  FM_CUDA(cudaEventRecord(ctx->copy_fence, ctx->stream));
  FM_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_fence, 0));
  const size_t row_floats = (size_t)vol_dims[1] * vol_dims[2];
  const int x_off = halo_pad[0] + fit_pad[0];  // padded x = volume x + x_off
  int rows_up = 0;
  auto upload_to = [&](int need_rows) -> int {
    need_rows = std::min(need_rows, (int)vol_dims[0]);
    if (need_rows <= rows_up) return FM_OK;
    const size_t off = (size_t)rows_up * row_floats, cnt = (size_t)(need_rows - rows_up) * row_floats;
    host_copy(pin_in + off * 4, vol + off, cnt * 4);
    FM_CUDA(cudaMemcpyAsync(dvol.p + off, pin_in + off * 4, cnt * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
    if (truth) {
      host_copy(pin_in + (nv + off) * 4, truth + off, cnt * 4);
      FM_CUDA(cudaMemcpyAsync(dvol.p + nv + off, pin_in + (nv + off) * 4, cnt * 4, cudaMemcpyHostToDevice,
                              ctx->copy_stream));
    }
    FM_CUDA(cudaEventRecord(ev_up, ctx->copy_stream));
    FM_CUDA(cudaStreamWaitEvent(ctx->stream, ev_up, 0));
    rows_up = need_rows;
    return FM_OK;
  };
  // finished output slabs: (first row, rows, event after their D2H copy)
  struct Slab {
    int x0, rows;
    cudaEvent_t done;
  };
  std::vector<Slab> slabs;
  size_t unstaged = 0;
  const size_t plane = (size_t)out_dims[1] * out_dims[2];
  const bool stream_out = want_out && shard_count == 1;  // slab-wise D2H only when no cross-rank reduce follows
  // a page-locked result (fm_host_alloc, what fetal_net.prediction hands in) receives the slabs directly: no staging
  // copy, no first-touch page faults of a fresh 33 MB array
  const bool out_pinned = want_out && is_pinned_host(out) && (!out_count || is_pinned_host(out_count));
  if (out_pinned) {
    pin_out = (char*)out;
    pin_cnt = (char*)out_count;
  }
  auto unstage = [&](bool block) {
    while (unstaged < slabs.size()) {
      const Slab& sl = slabs[unstaged];
      if (block) {
        cudaEventSynchronize(sl.done);
      } else if (cudaEventQuery(sl.done) != cudaSuccess) {
        cudaGetLastError();
        break;
      }
      const size_t o = (size_t)sl.x0 * plane, c = (size_t)sl.rows * plane;
      if (!out_pinned) {
        host_copy(out + o, pin_out + o * 8, c * 8);
        if (out_count) host_copy(out_count + o, pin_cnt + o * 2, c * 2);
      }
      ++unstaged;
    }
  };
  int x_done = 0;
  for (int64_t b0 = lo; b0 < hi; b0 += batch) {
    const int nb = (int)std::min<int64_t>(batch, hi - b0);
    // rows of the volume the patches of this sub-batch read: up to the last patch's corner + its extent
    FM_TRY(upload_to(idx[(b0 + nb - 1) * 3] - x_off + patch[0]));
    // 3D: [nb,P0,P1,P2] == the network's [nb,X,Y,Z] input. 2D: [nb,H,W,(slices | truth slices)] channels-last
    FM_TRY(k_gather_patches(ctx, dvol.p, vol_dims, halo_pad, fit_pad, (float)pad_value[0], (float)pad_value[1],
                            didx.p + b0 * 3, nb, patch, m->x_in.p, is2d ? m->cin_real : 0, 0, 0));
    if (truth) {
      const int32_t tpatch[3] = {patch[0], patch[1], prev_truth_size};
      FM_TRY(k_gather_patches(ctx, dvol.p + nv, vol_dims, halo_pad, fit_pad, 0.f, 0.f, didx.p + b0 * 3, nb, tpatch,
                              m->x_in.p, m->cin_real, nslices, prev_truth_index));
    }
    FM_TRY(forward(m, nb));
    FM_CUDA(cudaMemcpyAsync(dpred.p + (size_t)(b0 - lo) * pv, m->prob.p, (size_t)nb * pv * 4,
                            cudaMemcpyDeviceToDevice, ctx->stream));
    // output rows below the next unprocessed patch's x corner are final (for this shard)
    const int x_final = b0 + nb < hi ? std::min<int>(idx[(b0 + nb) * 3], out_dims[0]) : out_dims[0];
    if (x_final > x_done) {
      FM_TRY(k_reassemble_rows(ctx, plan, dpred.p, lo, hi, lo, dout.p, dcnt.p, shard_count == 1 ? 1 : 0, x_done, x_final));
      if (stream_out) {
        const size_t o = (size_t)x_done * plane, c = (size_t)(x_final - x_done) * plane;
        FM_CUDA(cudaEventRecord(ev_rows, ctx->stream));
        FM_CUDA(cudaStreamWaitEvent(ctx->d2h_stream, ev_rows, 0));
        FM_CUDA(cudaMemcpyAsync(pin_out + o * 8, dout.p + o, c * 8, cudaMemcpyDeviceToHost, ctx->d2h_stream));
        if (out_count)
          FM_CUDA(cudaMemcpyAsync(pin_cnt + o * 2, dcnt.p + o, c * 2, cudaMemcpyDeviceToHost, ctx->d2h_stream));
        cudaEvent_t done = m->pw_events[2 + slabs.size() % (size_t)ngroups];
        FM_CUDA(cudaEventRecord(done, ctx->d2h_stream));
        slabs.push_back(Slab{x_done, x_final - x_done, done});
      }
      x_done = x_final;
    }
    unstage(false);
  }
  lap("enqueue (upload / gather / forward / overlap-add)");
  if (pp) {
    // the float64 map stays on the device: its pad_for_fit crop (prediction.py:198-207) is post-processed in place,
    // while the slabs of `out` (when asked for) are still on their way back
    PostprocBuffers b;
    FM_TRY(pp_buffers(ctx, (int64_t)nv, pp->radius, &b));
    const double* box = dout.p + (size_t)fit_pad[0] * plane + (size_t)fit_pad[2] * out_dims[2] + fit_pad[4];
    FM_TRY(k_postprocess(ctx, b, box, FM_DTYPE_FLOAT64, (int64_t)plane, out_dims[2], vol_dims, pp));
    if (stream_out) unstage(true);
    FM_TRY(pp_download(ctx, b, nv, pp, (char*)pin + pp_off, pp_mask, pp_components));
    lap("post-process + D2H");
    m->fwd_valid = false;
    return FM_OK;
  }
  if (stream_out) {
    unstage(true);
    FM_CUDA(cudaStreamSynchronize(ctx->stream));
    lap("drain (D2H + unstage)");
    m->fwd_valid = false;
    return FM_OK;
  }
  if (reduce_root >= 0 && shard_count > 1) {
    FM_TRY(comm_reduce(ctx, dout.p, nout, 1, reduce_root, ctx->stream));
    if (want_out) FM_TRY(k_divide_by_count(ctx, dout.p, dcnt.p, (int64_t)nout, 1));
  }
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  lap("reduce");
  m->fwd_valid = false;
  if (!want_out) return FM_OK;
  FM_CUDA(cudaMemcpyAsync(pin_out, dout.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (out_count) FM_CUDA(cudaMemcpyAsync(pin_cnt, dcnt.p, cnt_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  lap("d2h");
  if (!out_pinned) {
    host_copy(out, pin_out, out_bytes);
    if (out_count) host_copy(out_count, pin_cnt, cnt_bytes);
  }
  lap("unstage result");
  return FM_OK;
}

// Page-locked host memory for callers that want results without a staging copy (fetal_net.prediction keeps a pool).
extern "C" int fm_host_alloc(size_t bytes, void** out) {
  FM_CHECK(out && bytes > 0, FM_EINVAL, "fm_host_alloc: bad argument");
  FM_CUDA(cudaMallocHost(out, bytes));
  return FM_OK;
}
extern "C" int fm_host_free(void* p) {
  if (p) FM_CUDA(cudaFreeHost(p));
  return FM_OK;
}

extern "C" int fm_patchwise_predict(fm_model* m, const float* vol, const int32_t vol_dims[3],
                                    const int32_t halo_pad[6], const int32_t fit_pad[6],
                                    const double pad_value[2], const int32_t* idx, int64_t n, int batch,
                                    int shard_rank, int shard_count, const float* truth, int prev_truth_index,
                                    int prev_truth_size, double* out, int16_t* out_count) {
  return patchwise_impl(m, vol, vol_dims, halo_pad, fit_pad, pad_value, idx, n, batch, shard_rank, shard_count, -1, truth,
                        prev_truth_index, prev_truth_size, out, out_count);
}

extern "C" int fm_patchwise_predict_dp(fm_model* m, const float* vol, const int32_t vol_dims[3],
                                       const int32_t halo_pad[6], const int32_t fit_pad[6],
                                       const double pad_value[2], const int32_t* idx, int64_t n, int batch, int root,
                                       const float* truth, int prev_truth_index, int prev_truth_size, double* out,
                                       int16_t* out_count) {
  FM_CHECK(m, FM_EINVAL, "fm_patchwise_predict_dp: NULL model");
  fm_ctx* ctx = m->ctx;
  const int ranks = ctx->comm ? ctx->comm_size : 1;
  FM_CHECK(root >= 0 && root < ranks, FM_EINVAL, "fm_patchwise_predict_dp: root %d of %d ranks", root, ranks);
  return patchwise_impl(m, vol, vol_dims, halo_pad, fit_pad, pad_value, idx, n, batch, ctx->comm_rank, ranks, root, truth,
                        prev_truth_index, prev_truth_size, out, out_count);
}

extern "C" int fm_patchwise_segment(fm_model* m, const float* vol, const int32_t vol_dims[3], const int32_t halo_pad[6],
                                    const int32_t fit_pad[6], const double pad_value[2], const int32_t* idx, int64_t n,
                                    int batch, const float* truth, int prev_truth_index, int prev_truth_size,
                                    const fm_postprocess_spec* spec, uint8_t* mask, double* prob, int64_t* n_components) {
  FM_CHECK(spec && mask, FM_EINVAL, "fm_patchwise_segment: NULL spec or mask");
  return patchwise_impl(m, vol, vol_dims, halo_pad, fit_pad, pad_value, idx, n, batch, 0, 1, -1, truth, prev_truth_index,
                        prev_truth_size, prob, nullptr, spec, mask, n_components);
}

// Flip test-time augmentation: `passes` sliding-window predictions of the volume flipped by in_flip[k], each cropped and
// un-flipped by out_flip[k] into slot k of a device stack, then the per-voxel median and (spec) its post-processing.
// Flipping keeps the volume's shape and multiset of values, so the pads, the patch list and the reassembly plan of the
// unflipped volume serve every pass; the flip is applied to the unpadded volume and the gather pads it as usual.
extern "C" int fm_patchwise_predict_flips(fm_model* m, const float* vol, const int32_t vol_dims[3],
                                          const int32_t halo_pad[6], const int32_t fit_pad[6], const double pad_value[2],
                                          const int32_t* idx, int64_t n, int batch, int passes, const int32_t* in_flip,
                                          const int32_t* out_flip, double* maps, double* median,
                                          const fm_postprocess_spec* spec, uint8_t* mask, int64_t* n_components) {
  FM_CHECK(m && vol && vol_dims && halo_pad && fit_pad && pad_value && idx && in_flip && out_flip && n > 0 && batch > 0,
           FM_EINVAL, "fm_patchwise_predict_flips: bad argument");
  FM_CHECK(passes >= 1 && passes <= 8, FM_EINVAL, "fm_patchwise_predict_flips: %d passes (1 .. 8)", passes);
  for (int k = 0; k < passes; ++k)
    FM_CHECK(in_flip[k] >= 0 && in_flip[k] <= 7 && out_flip[k] >= 0 && out_flip[k] <= 7, FM_EINVAL,
             "fm_patchwise_predict_flips: pass %d has flip masks %d / %d (0 .. 7)", k, in_flip[k], out_flip[k]);
  FM_CHECK(vol_dims[0] > 0 && vol_dims[1] > 0 && vol_dims[2] > 0, FM_EINVAL,
           "fm_patchwise_predict_flips: volume %d x %d x %d", vol_dims[0], vol_dims[1], vol_dims[2]);
  if (spec) {
    FM_CHECK(mask, FM_EINVAL, "fm_patchwise_predict_flips: post-processing needs a mask");
    FM_TRY(check_pp_spec(spec, vol_dims));
  }
  fm_ctx* ctx = m->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  const bool is2d = m->kcode == 31;
  int32_t patch[3], pred[3], out_dims[3];
  FM_TRY(pw_extents(m, is2d ? m->cin_real : m->spec.Z, vol_dims, halo_pad, fit_pad, patch, pred, out_dims));
  const int32_t fit_lo[3] = {fit_pad[0], fit_pad[2], fit_pad[4]};
  const size_t nv = (size_t)vol_dims[0] * vol_dims[1] * vol_dims[2];
  const size_t nout = (size_t)out_dims[0] * out_dims[1] * out_dims[2];
  const size_t pv = (size_t)pred[0] * pred[1] * pred[2];
  const int64_t pitch = ((int64_t)nv + 3) & ~(int64_t)3;  // slot stride of the stack: whole 32-byte quads
  ReasmPlan* plan = nullptr;
  FM_TRY(k_reassemble_prepare(ctx, idx, n, pred, 1, out_dims, &plan));
  struct PlanGuard {
    ReasmPlan* p;
    ~PlanGuard() { k_reassemble_release(p); }
  } plan_guard{plan};
  const int32_t* xstarts = nullptr;
  int ngroups = 0, ppg = 0;
  k_reassemble_groups(plan, &xstarts, &ngroups, &ppg);
  batch = pw_sub_batch(m, (int)std::min<int64_t>(batch, n), n, ngroups, ppg);
  FM_TRY(ensure_capacity(m, batch, false));
  FM_TRY(m->pw_vol.ensure(nv));
  FM_TRY(m->tta_vol.ensure(nv));
  FM_TRY(m->pw_pred.ensure((size_t)n * pv));
  FM_TRY(m->pw_idx.ensure((size_t)n * 3));
  FM_TRY(m->pw_out.ensure(nout));
  FM_TRY(m->pw_cnt.ensure(nout));
  FM_TRY(m->tta_stack.ensure((size_t)passes * pitch));
  if (m->pw_events.size() < 2) {
    const size_t old = m->pw_events.size();
    m->pw_events.resize(2, nullptr);
    for (size_t i = old; i < 2; ++i) FM_CUDA(cudaEventCreateWithFlags(&m->pw_events[i], cudaEventDisableTiming));
  }
  cudaEvent_t ev_slot = m->pw_events[1];
  double* stack = m->tta_stack.p;
  double* dmed = m->pw_out.p;  // the median replaces the last pass's padded map once that is in the stack
  // pinned staging: [volume | one float64 map (median / maps into pageable memory) | post-processing stats + mask]
  const size_t in_bytes = (nv * sizeof(float) + 4095) & ~(size_t)4095;
  const size_t map_bytes = (nv * sizeof(double) + 4095) & ~(size_t)4095;
  void* pin = nullptr;
  FM_TRY(fm_ctx_pinned(ctx, in_bytes + map_bytes + 256 + nv, &pin));
  char* pin_map = (char*)pin + in_bytes;
  host_copy(pin, vol, nv * sizeof(float));
  FM_CUDA(cudaMemcpyAsync(m->pw_vol.p, pin, nv * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(m->pw_idx.p, idx, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
  // a page-locked `maps` receives slot k on the copy-back stream while pass k + 1 computes
  const bool maps_pinned = maps && is_pinned_host(maps);
  for (int k = 0; k < passes; ++k) {
    const float* src = m->pw_vol.p;
    if (in_flip[k]) {
      FM_TRY(k_flip_volume(ctx, m->pw_vol.p, m->tta_vol.p, vol_dims, in_flip[k]));
      src = m->tta_vol.p;
    }
    for (int64_t b0 = 0; b0 < n; b0 += batch) {
      const int nb = (int)std::min<int64_t>(batch, n - b0);
      FM_TRY(k_gather_patches(ctx, src, vol_dims, halo_pad, fit_pad, (float)pad_value[0], (float)pad_value[1],
                              m->pw_idx.p + b0 * 3, nb, patch, m->x_in.p, is2d ? m->cin_real : 0, 0, 0));
      FM_TRY(forward(m, nb));
      FM_CUDA(cudaMemcpyAsync(m->pw_pred.p + (size_t)b0 * pv, m->prob.p, (size_t)nb * pv * 4, cudaMemcpyDeviceToDevice,
                              ctx->stream));
    }
    FM_TRY(k_reassemble_rows(ctx, plan, m->pw_pred.p, 0, n, 0, m->pw_out.p, m->pw_cnt.p, 1, 0, out_dims[0]));
    double* slot = stack + (size_t)k * pitch;
    FM_TRY(k_flip_crop(ctx, m->pw_out.p, out_dims, fit_lo, slot, vol_dims, out_flip[k]));
    if (maps_pinned) {
      FM_CUDA(cudaEventRecord(ev_slot, ctx->stream));
      FM_CUDA(cudaStreamWaitEvent(ctx->d2h_stream, ev_slot, 0));
      FM_CUDA(cudaMemcpyAsync(maps + (size_t)k * nv, slot, nv * sizeof(double), cudaMemcpyDeviceToHost,
                              ctx->d2h_stream));
    }
  }
  FM_TRY(k_median_passes(ctx, stack, pitch, passes, (int64_t)nv, dmed));
  const bool median_pinned = median && is_pinned_host(median);
  if (median)
    FM_CUDA(cudaMemcpyAsync(median_pinned ? (void*)median : (void*)pin_map, dmed, nv * sizeof(double),
                            cudaMemcpyDeviceToHost, ctx->stream));
  if (spec) {
    PostprocBuffers b;
    FM_TRY(pp_buffers(ctx, (int64_t)nv, spec->radius, &b));
    FM_TRY(k_postprocess(ctx, b, dmed, FM_DTYPE_FLOAT64, (int64_t)vol_dims[1] * vol_dims[2], vol_dims[2], vol_dims,
                         spec));
    FM_TRY(pp_download(ctx, b, nv, spec, pin_map + map_bytes, mask, n_components));
  }
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  if (median && !median_pinned) host_copy(median, pin_map, nv * sizeof(double));
  if (maps && !maps_pinned)
    for (int k = 0; k < passes; ++k) {
      FM_CUDA(cudaMemcpyAsync(pin_map, stack + (size_t)k * pitch, nv * sizeof(double), cudaMemcpyDeviceToHost,
                              ctx->stream));
      FM_CUDA(cudaStreamSynchronize(ctx->stream));
      host_copy(maps + (size_t)k * nv, pin_map, nv * sizeof(double));
    }
  FM_CUDA(cudaStreamSynchronize(ctx->d2h_stream));
  m->fwd_valid = false;
  return FM_OK;
}

extern "C" int fm_op_median_passes(fm_ctx* ctx, const double* in, int passes, int64_t nvox, double* out) {
  FM_CHECK(ctx && in && out && nvox > 0, FM_EINVAL, "fm_op_median_passes: bad argument");
  FM_CHECK(passes >= 1 && passes <= 8, FM_EINVAL, "fm_op_median_passes: %d passes (1 .. 8)", passes);
  FM_CUDA(cudaSetDevice(ctx->device));
  const int64_t pitch = (nvox + 3) & ~(int64_t)3;
  DevBuf<double> d;
  FM_TRY(d.ensure((size_t)(passes + 1) * pitch));
  int r = FM_OK;
  cudaError_t e = cudaSuccess;
  for (int k = 0; k < passes && e == cudaSuccess; ++k)
    e = cudaMemcpyAsync(d.p + k * pitch, in + k * nvox, (size_t)nvox * 8, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) r = k_median_passes(ctx, d.p, pitch, passes, nvox, d.p + passes * pitch);
  if (e == cudaSuccess && r == FM_OK)
    e = cudaMemcpyAsync(out, d.p + passes * pitch, (size_t)nvox * 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    fm_set_error("fm_op_median_passes: %s", cudaGetErrorString(e));
    r = FM_ECUDA;
  }
  cudaStreamSynchronize(ctx->stream);
  d.release();
  return r;
}

// ---------------------------------------------------------------------------------------------
// training
// ---------------------------------------------------------------------------------------------
// `t_host` (optional): targets still on the host. They are first needed by the Dice sums at the end of the forward
// pass, so they are copied on the side stream AFTER the network has been queued — the transfer (and, for pageable
// memory, the host-side staging) overlaps the forward kernels. The side stream first waits for everything queued on
// the compute stream before this step, which may still read the previous targets.
static int train_forward_dev(fm_model* m, int batch, const float* t_host = nullptr) {
  fm_ctx* ctx = m->ctx;
  FM_CHECK(m->loss_kind != 2 || (m->mask_valid && m->mask_batch == batch), FM_ESTATE,
           "dice_and_xent_mask: call fm_model_set_weight_mask with this batch's weight mask before the step");
  if (t_host) {
    FM_CUDA(cudaEventRecord(ctx->copy_fence, ctx->stream));
    FM_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_fence, 0));
  }
  m->train_pass = true;
  m->targets_ready = t_host == nullptr;  // already uploaded: the head kernel also sums the loss statistics
  m->stats_done = false;
  const int rf = forward(m, batch);
  m->train_pass = false;
  m->targets_ready = false;
  FM_TRY(rf);
  if (t_host) {
    FM_CUDA(cudaMemcpyAsync(m->t_in.p, t_host, (size_t)batch * m->vox(0) * sizeof(float), cudaMemcpyHostToDevice,
                            ctx->copy_stream));
    FM_CUDA(cudaEventRecord(ctx->copy_done, ctx->copy_stream));
    FM_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->copy_done, 0));
  }
  if (!m->stats_done)
    FM_TRY(k_dice_sums(m->ctx, m->prob.p, m->t_in.p, (int64_t)batch * m->vox(0), m->sums, 0, m->xent()));
  m->stats_done = false;
  m->last_batch = batch;
  m->fwd_valid = true;
  return FM_OK;
}

static bool is_pinned_host(const void* p);
static bool is_pinned_host(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

static bool pipeline_enabled() {
  static const bool off = [] {
    const char* e = getenv("FETAL_B200_NO_PIPELINE");
    return e && e[0] == '1';
  }();
  return !off;
}

// pinned host inputs -> working buffers through one of two device staging buffers: the H2D copies run on the copy
// stream as soon as the step that last used that staging buffer has consumed it (two steps ago), i.e. concurrently
// with whatever the compute stream is still doing for the previous step; the compute stream then takes a device copy
static int stage_inputs(fm_model* m, const float* x, const float* t, int batch) {
  fm_ctx* ctx = m->ctx;
  const bool pageable = !is_pinned_host(x) || !is_pinned_host(t);
  if (!m->sums_ready) {
    for (int b = 0; b < 2; ++b) {
      FM_CUDA(cudaEventCreateWithFlags(&m->stage_ready[b], cudaEventDisableTiming));
      FM_CUDA(cudaEventCreateWithFlags(&m->stage_free[b], cudaEventDisableTiming));
    }
    FM_CUDA(cudaEventCreateWithFlags(&m->sums_ready, cudaEventDisableTiming));
    FM_CUDA(cudaMallocHost((void**)&m->sums_pin, kNumLossSums * sizeof(double)));
  }
  const size_t n = (size_t)batch * m->vox(0), nx = n * m->cin_real;
  const int b = (m->stage_idx ^= 1);
  FM_TRY(m->stage_x[b].ensure(nx));
  FM_TRY(m->stage_t[b].ensure(n));
  if (pageable) {
    // a caller feeding plain NumPy batches (the reference's generator does): host threads copy them into a pinned
    // buffer while the GPU still works on the previous step, then the same asynchronous route as pinned inputs
    if (m->host_stage_floats[b] < nx + n) {
      if (m->host_stage[b]) {
        FM_CUDA(cudaEventSynchronize(m->host_stage_done[b]));
        FM_CUDA(cudaFreeHost(m->host_stage[b]));
        m->host_stage[b] = nullptr;
      }
      FM_CUDA(cudaMallocHost((void**)&m->host_stage[b], (nx + n) * sizeof(float)));
      m->host_stage_floats[b] = nx + n;
      if (!m->host_stage_done[b]) FM_CUDA(cudaEventCreateWithFlags(&m->host_stage_done[b], cudaEventDisableTiming));
    } else {
      FM_CUDA(cudaEventSynchronize(m->host_stage_done[b]));  // the copies of two steps ago have left the buffer
    }
    host_copy(m->host_stage[b], x, nx * sizeof(float));
    host_copy(m->host_stage[b] + nx, t, n * sizeof(float));
    x = m->host_stage[b];
    t = m->host_stage[b] + nx;
  }
  FM_CUDA(cudaStreamWaitEvent(ctx->copy_stream, m->stage_free[b], 0));
  FM_CUDA(cudaMemcpyAsync(m->stage_x[b].p, x, nx * sizeof(float), cudaMemcpyHostToDevice, ctx->copy_stream));
  FM_CUDA(cudaMemcpyAsync(m->stage_t[b].p, t, n * sizeof(float), cudaMemcpyHostToDevice, ctx->copy_stream));
  FM_CUDA(cudaEventRecord(m->stage_ready[b], ctx->copy_stream));
  if (pageable) FM_CUDA(cudaEventRecord(m->host_stage_done[b], ctx->copy_stream));
  FM_CUDA(cudaStreamWaitEvent(ctx->stream, m->stage_ready[b], 0));
  FM_CUDA(cudaMemcpyAsync(m->x_in.p, m->stage_x[b].p, nx * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(m->t_in.p, m->stage_t[b].p, n * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
  FM_CUDA(cudaEventRecord(m->stage_free[b], ctx->stream));
  return FM_OK;
}

extern "C" int fm_train_forward(fm_model* m, const float* x, const float* t, int batch) {
  FM_CHECK(m && x && t && batch > 0, FM_EINVAL, "fm_train_forward: bad argument");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  FM_TRY(ensure_capacity(m, batch, true));
  const size_t n = (size_t)batch * m->vox(0);
  if (pipeline_enabled()) {
    FM_TRY(stage_inputs(m, x, t, batch));
    return train_forward_dev(m, batch);
  }
  FM_TRY(upload(m, x, m->x_in.p, n * m->cin_real));
  return train_forward_dev(m, batch, t);
}

// Data-parallel early return: after the caller's all-reduce of the statistics (queued on the compute stream),
// fm_train_metrics_async queues their copy to pinned host memory; fm_train_metrics_wait blocks only until that copy
// has landed - the rest of the step keeps running and is ordered before every later call on the model.
extern "C" int fm_train_metrics_async(fm_model* m) {
  FM_CHECK(m && m->fwd_valid, FM_ESTATE, "fm_train_metrics_async needs a preceding fm_train_forward");
  fm_ctx* ctx = m->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  if (!m->sums_ready) {
    for (int b = 0; b < 2; ++b) {
      FM_CUDA(cudaEventCreateWithFlags(&m->stage_ready[b], cudaEventDisableTiming));
      FM_CUDA(cudaEventCreateWithFlags(&m->stage_free[b], cudaEventDisableTiming));
    }
    FM_CUDA(cudaEventCreateWithFlags(&m->sums_ready, cudaEventDisableTiming));
    FM_CUDA(cudaMallocHost((void**)&m->sums_pin, kNumLossSums * sizeof(double)));
  }
  FM_CUDA(cudaMemcpyAsync(m->sums_pin, m->sums, kNumLossSums * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaEventRecord(m->sums_ready, ctx->stream));
  m->metrics_pending = true;
  return FM_OK;
}
extern "C" int fm_train_metrics_wait(fm_model* m, float out_metrics[4]) {
  FM_CHECK(m && out_metrics, FM_EINVAL, "fm_train_metrics_wait: bad argument");
  FM_CHECK(m->metrics_pending, FM_ESTATE, "fm_train_metrics_wait without fm_train_metrics_async");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  FM_CUDA(cudaEventSynchronize(m->sums_ready));
  metrics_from_sums(m->sums_pin, out_metrics, m->loss_kind ? m->xent_weight : 0.f);
  m->metrics_pending = false;
  return FM_OK;
}

extern "C" int fm_train_backward(fm_model* m) {
  FM_CHECK(m, FM_EINVAL, "NULL model");
  FM_CHECK(m->fwd_valid, FM_ESTATE, "fm_train_backward called without a preceding fm_train_forward");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  m->train_pass = true;
  const int rb = backward(m, m->last_batch);
  m->train_pass = false;
  FM_TRY(rb);
  m->fwd_valid = false;
  return FM_OK;
}

extern "C" int fm_train_apply(fm_model* m, float lr, uint64_t after_stream, float out_metrics[4]) {
  FM_CHECK(m, FM_EINVAL, "NULL model");
  fm_ctx* ctx = m->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  if (after_stream) {
    FM_CUDA(cudaEventRecord(m->ev_tmp, (cudaStream_t)(uintptr_t)after_stream));
    FM_CUDA(cudaStreamWaitEvent(ctx->stream, m->ev_tmp, 0));
  }
  FM_TRY(k_adam(ctx, m->params, m->grads, m->adam_m, m->adam_v, m->nparams, m->iterations, lr));
  m->iterations++;
  m->packs_dirty = true;
  FM_TRY(refresh_packs(m));
  if (out_metrics) {
    FM_CUDA(cudaMemcpyAsync(m->sums_host, m->sums, kNumLossSums * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaStreamSynchronize(ctx->stream));
    metrics_from_sums(m->sums_host, out_metrics, m->loss_kind ? m->xent_weight : 0.f);
  }
  return FM_OK;
}

extern "C" int fm_model_loss_sums(fm_model* m, uint64_t* dev_ptr) {
  FM_CHECK(m && dev_ptr, FM_EINVAL, "NULL argument");
  *dev_ptr = (uint64_t)(uintptr_t)m->sums;
  return FM_OK;
}
extern "C" int fm_model_grad_buffer(fm_model* m, uint64_t* dev_ptr, int64_t* n) {
  FM_CHECK(m && dev_ptr && n, FM_EINVAL, "NULL argument");
  *dev_ptr = (uint64_t)(uintptr_t)m->grads;
  *n = m->nparams;
  return FM_OK;
}
extern "C" int fm_model_num_buckets(fm_model* m) { return m ? (int)m->buckets.size() : -1; }
extern "C" int fm_model_bucket_range(fm_model* m, int bucket, int64_t* offset, int64_t* count) {
  FM_CHECK(m && bucket >= 0 && bucket < (int)m->buckets.size() && offset && count, FM_EINVAL,
           "bucket %d out of range", bucket);
  const Layer& first = m->layers[m->buckets[bucket].first];
  const int last_i = m->buckets[bucket].second;
  const int64_t end = last_i + 1 < (int)m->layers.size() ? m->layers[last_i + 1].w_off : m->nparams;
  *offset = first.w_off;
  *count = end - first.w_off;
  return FM_OK;
}
extern "C" int fm_stream_wait_bucket(fm_model* m, uint64_t stream, int bucket) {
  FM_CHECK(m && bucket >= 0 && bucket < (int)m->buckets.size(), FM_EINVAL, "bucket %d out of range", bucket);
  // backward runs in reverse creation order: the bucket is final when its FIRST layer is done
  FM_CUDA(cudaStreamWaitEvent((cudaStream_t)(uintptr_t)stream, m->layer_done[m->buckets[bucket].first], 0));
  return FM_OK;
}

extern "C" int fm_train_step_device(fm_model* m, uint64_t x_dev, uint64_t t_dev, int batch, float lr,
                                    float out_metrics[4]) {
  FM_CHECK(m && x_dev && t_dev && batch > 0, FM_EINVAL, "fm_train_step_device: bad argument");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  FM_TRY(ensure_capacity(m, batch, true));
  const size_t n = (size_t)batch * m->vox(0);
  FM_CUDA(cudaMemcpyAsync(m->x_in.p, (const void*)(uintptr_t)x_dev, n * m->cin_real * 4, cudaMemcpyDeviceToDevice,
                          m->ctx->stream));
  FM_CUDA(cudaMemcpyAsync(m->t_in.p, (const void*)(uintptr_t)t_dev, n * 4, cudaMemcpyDeviceToDevice,
                          m->ctx->stream));
  FM_TRY(train_forward_dev(m, batch));
  FM_TRY(fm_train_backward(m));
  return fm_train_apply(m, lr, 0, out_metrics);
}

extern "C" int fm_train_step(fm_model* m, const float* x, const float* t, int batch, float lr,
                             float out_metrics[4]) {
  FM_CHECK(m && x && t && batch > 0, FM_EINVAL, "fm_train_step: bad argument");
  if (!pipeline_enabled() || !out_metrics) {
    FM_TRY(fm_train_forward(m, x, t, batch));
    FM_TRY(fm_train_backward(m));
    return fm_train_apply(m, lr, 0, out_metrics);
  }
  fm_ctx* ctx = m->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  FM_TRY(ensure_capacity(m, batch, true));
  FM_TRY(stage_inputs(m, x, t, batch));
  FM_TRY(train_forward_dev(m, batch));
  FM_CUDA(cudaMemcpyAsync(m->sums_pin, m->sums, kNumLossSums * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaEventRecord(m->sums_ready, ctx->stream));
  FM_TRY(fm_train_backward(m));
  FM_TRY(fm_train_apply(m, lr, 0, nullptr));
  FM_CUDA(cudaEventSynchronize(m->sums_ready));  // the inputs were consumed long before: x / t may be reused
  metrics_from_sums(m->sums_pin, out_metrics, m->loss_kind ? m->xent_weight : 0.f);
  return FM_OK;
}

// The data-parallel tail of a step whose forward pass has been queued (statistics in m->sums): all-reduce of the Dice
// sums, backward, bucketed gradient all-reduce overlapped with it, Adam, metrics.
static int dp_step_after_forward(fm_model* m, float lr, float out_metrics[4]);

extern "C" int fm_train_step_dp(fm_model* m, const float* x, const float* t, int batch, float lr,
                                float out_metrics[4]) {
  FM_CHECK(!(m && m->batch_norm), FM_EINVAL,
           "fm_train_step_dp: batch_normalization=True needs batch statistics over the GLOBAL batch (not built): "
           "a data-parallel step on local statistics would not equal the single-process reference");
  FM_CHECK(m && x && t && batch > 0 && out_metrics, FM_EINVAL, "fm_train_step_dp: bad argument");
  fm_ctx* ctx = m->ctx;
  if (!ctx->comm || ctx->comm_size == 1) return fm_train_step(m, x, t, batch, lr, out_metrics);
  FM_TRY(fm_train_forward(m, x, t, batch));
  return dp_step_after_forward(m, lr, out_metrics);
}

extern "C" int fm_train_step_sampled(fm_model* m, fm_volset* s, const int32_t* cases, const int32_t* corners,
                                     const fm_sample_aug* aug, int batch, int truth_index, int truth_size,
                                     int prev_truth_index, int prev_truth_size, float lr, float out_metrics[4]) {
  FM_CHECK(m && s && cases && corners && batch > 0 && out_metrics, FM_EINVAL, "fm_train_step_sampled: bad argument");
  fm_ctx* ctx = m->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  const bool is2d = m->kcode == 31;
  FM_CHECK(m->kind == 0 || !is2d, FM_EINVAL, "fm_train_step_sampled: unsupported model kind");
  int32_t patch[3];
  if (is2d) {
    FM_CHECK(truth_size == 1 && prev_truth_size >= 0 && prev_truth_size < m->cin_real, FM_EINVAL,
             "fm_train_step_sampled: a 2D model takes truth_size 1 and prev_truth_size < in_channels (%d)", m->cin_real);
    patch[0] = m->spec.X;
    patch[1] = m->spec.Y;
    patch[2] = m->cin_real - prev_truth_size;
  } else {
    FM_CHECK(prev_truth_size == 0 && truth_size == m->spec.Z, FM_EINVAL,
             "fm_train_step_sampled: a 3D model takes truth_size == Z (%d) and no previous-truth channels", m->spec.Z);
    patch[0] = m->spec.X;
    patch[1] = m->spec.Y;
    patch[2] = m->spec.Z;
  }
  FM_TRY(ensure_capacity(m, batch, true));
  FM_TRY(sampler_gather_device(s, cases, corners, aug, batch, patch, truth_index, truth_size, prev_truth_index,
                               prev_truth_size, m->x_in.p, m->t_in.p));
  FM_TRY(train_forward_dev(m, batch));
  if (ctx->comm && ctx->comm_size > 1) return dp_step_after_forward(m, lr, out_metrics);
  if (!pipeline_enabled()) {
    FM_TRY(fm_train_backward(m));
    return fm_train_apply(m, lr, 0, out_metrics);
  }
  // like fm_train_step: return as soon as the statistics of THIS forward pass are on the host; backward, Adam and the
  // repack keep running while the caller draws the next batch
  FM_TRY(fm_train_metrics_async(m));
  FM_TRY(fm_train_backward(m));
  FM_TRY(fm_train_apply(m, lr, 0, nullptr));
  return fm_train_metrics_wait(m, out_metrics);
}

static int dp_step_after_forward(fm_model* m, float lr, float out_metrics[4]) {
  fm_ctx* ctx = m->ctx;
  FM_CHECK(!m->batch_norm, FM_EINVAL,
           "data-parallel step: batch_normalization=True needs batch statistics over the GLOBAL batch (not built)");
  // 8 float64: the GLOBAL Dice statistics every rank back-propagates (64 bytes; latency only)
  FM_TRY(comm_allreduce(ctx, m->sums, kNumLossSums, 1, ctx->stream));
  FM_TRY(fm_train_metrics_async(m));
  FM_TRY(fm_train_backward(m));
  // gradient buckets in completion order (backward runs in reverse creation order): each all-reduce waits only for
  // the event of the bucket's first layer and overlaps whatever backward still has queued on the compute stream
  for (size_t b = 0; b < m->buckets.size(); ++b) {
    const Layer& first = m->layers[m->buckets[b].first];
    const int last_i = m->buckets[b].second;
    const int64_t end = last_i + 1 < (int)m->layers.size() ? m->layers[last_i + 1].w_off : m->nparams;
    FM_CUDA(cudaStreamWaitEvent(ctx->comm_stream, m->layer_done[m->buckets[b].first], 0));
    FM_TRY(comm_allreduce(ctx, m->grads + first.w_off, (size_t)(end - first.w_off), 0, ctx->comm_stream));
  }
  FM_TRY(fm_train_apply(m, lr, (uint64_t)(uintptr_t)ctx->comm_stream, nullptr));
  return fm_train_metrics_wait(m, out_metrics);
}

extern "C" int fm_comm_broadcast_params(fm_model* m, int root) {
  FM_CHECK(m, FM_EINVAL, "fm_comm_broadcast_params: NULL model");
  fm_ctx* ctx = m->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  FM_TRY(comm_broadcast(ctx, m->params, (size_t)m->nparams, 0, root, ctx->stream));
  FM_TRY(comm_broadcast(ctx, m->adam_m, (size_t)m->nparams, 0, root, ctx->stream));
  FM_TRY(comm_broadcast(ctx, m->adam_v, (size_t)m->nparams, 0, root, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  m->packs_dirty = true;
  return FM_OK;
}

// Adam moments of one layer in Keras layout, and the step counter: what Keras' model.save() keeps besides the weights
// (the reference resumes with load_old_model(get_last_model_path(...)), fetal/train_fetal.py:25-28)
extern "C" int fm_model_get_adam_state(fm_model* m, int layer, float* m_kernel, float* m_bias, float* v_kernel,
                                       float* v_bias) {
  FM_TRY(get_flat(m, m ? m->adam_m : nullptr, layer, m_kernel, m_bias));
  return get_flat(m, m ? m->adam_v : nullptr, layer, v_kernel, v_bias);
}
static int set_flat(fm_model* m, float* flat, int layer, const float* kernel, const float* bias) {
  FM_CHECK(m && layer >= 0 && layer < (int)m->layers.size() && kernel && bias, FM_EINVAL, "layer %d out of range", layer);
  FM_CUDA(cudaSetDevice(m->ctx->device));
  Layer& l = m->layers[layer];
  FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
  if (l.is_norm) {
    FM_CUDA(cudaMemcpy(flat + l.w_off, kernel, (size_t)l.cout * 4, cudaMemcpyHostToDevice));
  } else {
    std::vector<float> packed((size_t)l.wcount());
    keras_to_packed(kernel, packed.data(), l.k, l.cin_keras(), l.cout, l.cin());
    FM_CUDA(cudaMemcpy(flat + l.w_off, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice));
  }
  FM_CUDA(cudaMemcpy(flat + l.b_off, bias, (size_t)l.cout * 4, cudaMemcpyHostToDevice));
  return FM_OK;
}
extern "C" int fm_model_set_adam_state(fm_model* m, int layer, const float* m_kernel, const float* m_bias,
                                       const float* v_kernel, const float* v_bias) {
  FM_TRY(set_flat(m, m ? m->adam_m : nullptr, layer, m_kernel, m_bias));
  return set_flat(m, m ? m->adam_v : nullptr, layer, v_kernel, v_bias);
}
extern "C" int fm_model_get_iterations(fm_model* m) { return m ? m->iterations : -1; }
extern "C" int fm_model_set_iterations(fm_model* m, int iterations) {
  FM_CHECK(m && iterations >= 0, FM_EINVAL, "fm_model_set_iterations: bad argument");
  m->iterations = iterations;
  return FM_OK;
}

extern "C" int fm_evaluate(fm_model* m, const float* x, const float* t, int batch, float out_metrics[4]) {
  FM_CHECK(m && x && t && batch > 0 && out_metrics, FM_EINVAL, "fm_evaluate: bad argument");
  FM_CUDA(cudaSetDevice(m->ctx->device));
  FM_TRY(ensure_capacity(m, batch, true));
  const size_t n = (size_t)batch * m->vox(0);
  FM_TRY(upload(m, x, m->x_in.p, n * m->cin_real));
  FM_TRY(upload(m, t, m->t_in.p, n));
  FM_CHECK(m->loss_kind != 2 || (m->mask_valid && m->mask_batch == batch), FM_ESTATE,
           "dice_and_xent_mask: call fm_model_set_weight_mask with this batch's weight mask before fm_evaluate");
  FM_TRY(forward(m, batch));  // inference kernels: same bits as fm_predict
  FM_TRY(k_dice_sums(m->ctx, m->prob.p, m->t_in.p, (int64_t)n, m->sums, 0, m->xent()));
  m->fwd_valid = false;
  FM_CUDA(cudaMemcpyAsync(m->sums_host, m->sums, kNumLossSums * sizeof(double), cudaMemcpyDeviceToHost, m->ctx->stream));
  FM_CUDA(cudaStreamSynchronize(m->ctx->stream));
  metrics_from_sums(m->sums_host, out_metrics, m->loss_kind ? m->xent_weight : 0.f);
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------
// per-op hooks (host fp32 channels-last in/out; bf16 on the device)
// ---------------------------------------------------------------------------------------------
namespace {
struct OpScratch {
  fm_ctx* ctx;
  std::vector<void*> ptrs;
  explicit OpScratch(fm_ctx* c) : ctx(c) {}
  ~OpScratch() {
    cudaStreamSynchronize(ctx->stream);
    for (void* p : ptrs) cudaFree(p);
  }
  template <typename T>
  int alloc(T** out, size_t count) {
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e != cudaSuccess) {
      fm_set_error("cudaMalloc failed: %s", cudaGetErrorString(e));
      return FM_ENOMEM;
    }
    ptrs.push_back(p);
    *out = (T*)p;
    return FM_OK;
  }
  // host fp32 -> device bf16
  int up_bf16(const float* h, size_t count, bf16** out) {
    float* tmp;
    FM_TRY(alloc(&tmp, count));
    FM_TRY(alloc(out, count));
    FM_CUDA(cudaMemcpyAsync(tmp, h, count * 4, cudaMemcpyHostToDevice, ctx->stream));
    return k_cast_f32_to_bf16(ctx, tmp, *out, (int64_t)count);
  }
  int up_f32(const float* h, size_t count, float** out) {
    FM_TRY(alloc(out, count));
    FM_CUDA(cudaMemcpyAsync(*out, h, count * 4, cudaMemcpyHostToDevice, ctx->stream));
    return FM_OK;
  }
  // device bf16 -> host fp32
  int down_bf16(const bf16* d, size_t count, float* h) {
    float* tmp;
    FM_TRY(alloc(&tmp, count));
    FM_TRY(k_cast_bf16_to_f32(ctx, d, tmp, (int64_t)count));
    FM_CUDA(cudaMemcpyAsync(h, tmp, count * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaStreamSynchronize(ctx->stream));
    return FM_OK;
  }
};
}  // namespace

extern "C" int fm_op_conv3d_fprop(fm_ctx* ctx, int impl, const float* x, const float* x2,
                                  const float* w_keras, const float* bias, int N, int X, int Y, int Z,
                                  int C1, int C2, int Cout, int ksize, int relu, float* y) {
  FM_CHECK(ctx && x && w_keras && y, FM_EINVAL, "fm_op_conv3d_fprop: NULL argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t vox = (size_t)N * X * Y * Z;
  const int taps = kext_taps(ksize), Ct = C1 + C2;
  std::vector<float> packed((size_t)Cout * taps * Ct);
  keras_to_packed(w_keras, packed.data(), ksize, Ct, Cout);
  bf16 *dx1 = nullptr, *dx2 = nullptr, *dw = nullptr, *dy = nullptr;
  float* dbias = nullptr;
  FM_TRY(s.up_bf16(x, vox * C1, &dx1));
  if (C2 > 0) FM_TRY(s.up_bf16(x2, vox * C2, &dx2));
  FM_TRY(s.up_bf16(packed.data(), packed.size(), &dw));
  if (bias) FM_TRY(s.up_f32(bias, Cout, &dbias));
  FM_TRY(s.alloc(&dy, vox * Cout));
  if (impl == 2 || impl == 3) {  // marching kernel: 2 = bit-reproducible, 3 = the issue order of training passes
    FM_CHECK(conv_march_supported(X, Y, Z, C1, C2, Cout, ksize), FM_EINVAL, "march kernel does not cover this shape");
    bf16 *wm1 = nullptr, *wm2 = nullptr;
    FM_TRY(s.alloc(&wm1, (size_t)conv_march_pack_elems(C1, Cout)));
    FM_TRY(k_repack_march(ctx, dw, wm1, Cout, Ct, 0, C1, conv_march_kc(C1, C2, Cout, C1)));
    if (C2 > 0) {
      FM_TRY(s.alloc(&wm2, (size_t)conv_march_pack_elems(C2, Cout)));
      FM_TRY(k_repack_march(ctx, dw, wm2, Cout, Ct, C1, C2, conv_march_kc(C1, C2, Cout, C2)));
    }
    FM_TRY(k_conv3d_march(ctx, dx1, dx2, wm1, wm2, dbias, dy, nullptr, N, X, Y, Z, C1, C2, Cout, relu, Cout, 0,
                          impl != 3));
  } else if (impl == 0)
    FM_TRY(k_conv3d_tc_fprop(ctx, dx1, dx2, dw, dbias, dy, nullptr, N, X, Y, Z, C1, C2, Cout, ksize, relu,
                             Cout, 0));
  else
    FM_TRY(k_conv3d_simt_fprop(ctx, dx1, 0, dx2, dw, dbias, dy, nullptr, N, X, Y, Z, C1, C2, Cout, ksize,
                               relu, nullptr));
  return s.down_bf16(dy, vox * Cout, y);
}

extern "C" int fm_op_conv_dgrad(fm_ctx* ctx, int impl, const float* dy, const float* w_keras, const float* mask, int N,
                                int X, int Y, int Z, int Cin, int Cout, int ksize, float* dx) {
  FM_CHECK(ctx && dy && w_keras && dx, FM_EINVAL, "fm_op_conv_dgrad: NULL argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t vox = (size_t)N * X * Y * Z;
  const int taps = kext_taps(ksize);
  std::vector<float> packed((size_t)Cout * taps * Cin);
  keras_to_packed(w_keras, packed.data(), ksize, Cin, Cout);
  float* dwm = nullptr;
  bf16 *wd = nullptr, *ddy = nullptr, *dmask = nullptr, *ddx = nullptr;
  FM_TRY(s.up_f32(packed.data(), packed.size(), &dwm));
  FM_TRY(s.alloc(&wd, packed.size()));
  FM_TRY(k_repack_weights(ctx, dwm, nullptr, wd, nullptr, Cout, taps, Cin, 0));
  FM_TRY(s.up_bf16(dy, vox * Cout, &ddy));
  if (mask) FM_TRY(s.up_bf16(mask, vox * Cin, &dmask));
  FM_TRY(s.alloc(&ddx, vox * Cin));
  if (impl == 2 || impl == 3) {
    FM_CHECK(conv_march_supported(X, Y, Z, Cout, 0, Cin, ksize), FM_EINVAL, "march kernel does not cover this shape");
    bf16* wm = nullptr;
    FM_TRY(s.alloc(&wm, (size_t)conv_march_pack_elems(Cout, Cin)));
    FM_TRY(k_repack_march(ctx, wd, wm, Cin, Cout, 0, Cout, conv_march_kc(Cout, 0, Cin, Cout)));
    FM_TRY(k_conv3d_march(ctx, ddy, nullptr, wm, nullptr, nullptr, ddx, dmask, N, X, Y, Z, Cout, 0, Cin, 0, Cin, 0,
                          impl != 3));
  } else if (impl == 0)
    FM_TRY(k_conv3d_tc_fprop(ctx, ddy, nullptr, wd, nullptr, ddx, dmask, N, X, Y, Z, Cout, 0, Cin, ksize, 0,
                             Cin, 0));
  else
    FM_TRY(k_conv3d_simt_fprop(ctx, ddy, 0, nullptr, wd, nullptr, ddx, nullptr, N, X, Y, Z, Cout, 0, Cin,
                               ksize, 0, dmask));
  return s.down_bf16(ddx, vox * Cin, dx);
}

extern "C" int fm_op_conv_wgrad(fm_ctx* ctx, int impl, const float* x, const float* dy, int N, int X, int Y, int Z,
                                int Cin, int Cout, int ksize, float* dw_keras, float* dbias) {
  FM_CHECK(ctx && x && dy && dw_keras, FM_EINVAL, "fm_op_conv_wgrad: NULL argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t vox = (size_t)N * X * Y * Z;
  const int taps = kext_taps(ksize);
  bf16 *dx = nullptr, *ddy = nullptr;
  float *dw = nullptr, *db = nullptr;
  FM_TRY(s.up_bf16(x, vox * Cin, &dx));
  FM_TRY(s.up_bf16(dy, vox * Cout, &ddy));
  const size_t wn = (size_t)Cout * taps * Cin;
  FM_TRY(s.alloc(&dw, wn));
  FM_TRY(s.alloc(&db, Cout));
  FM_TRY(k_zero(ctx, dw, wn * 4));
  FM_TRY(k_zero(ctx, db, (size_t)Cout * 4));
  if (impl == 2)  // the marching kernel also produces the bias gradient (column sums of dY)
    FM_TRY(k_conv3d_wgrad_march(ctx, dx, ddy, dw, N, X, Y, Z, Cin, Cin, 0, Cout, db));
  else if (impl == 0)
    FM_TRY(k_conv3d_tc_wgrad(ctx, dx, ddy, dw, N, X, Y, Z, Cin, Cin, 0, Cout, ksize));
  else
    FM_TRY(k_conv3d_simt_wgrad(ctx, dx, 0, ddy, dw, N, X, Y, Z, Cin, Cin, 0, Cout, ksize));
  if (impl != 2) FM_TRY(k_bias_grad(ctx, ddy, db, (int64_t)vox, Cout));
  std::vector<float> packed(wn);
  FM_CUDA(cudaMemcpyAsync(packed.data(), dw, wn * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (dbias) FM_CUDA(cudaMemcpyAsync(dbias, db, (size_t)Cout * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  packed_to_keras(packed.data(), dw_keras, ksize, Cin, Cout);
  return FM_OK;
}

// the 3x3x3 forms of the two hooks above
extern "C" int fm_op_conv3d_dgrad(fm_ctx* ctx, int impl, const float* dy, const float* w_keras, const float* mask, int N,
                                  int X, int Y, int Z, int Cin, int Cout, float* dx) {
  return fm_op_conv_dgrad(ctx, impl, dy, w_keras, mask, N, X, Y, Z, Cin, Cout, 3, dx);
}
extern "C" int fm_op_conv3d_wgrad(fm_ctx* ctx, int impl, const float* x, const float* dy, int N, int X, int Y, int Z,
                                  int Cin, int Cout, float* dw_keras, float* dbias) {
  return fm_op_conv_wgrad(ctx, impl, x, dy, N, X, Y, Z, Cin, Cout, 3, dw_keras, dbias);
}

// First convolution of the network (one fp32 input channel): y = act(conv3x3x3(x) + bias) and / or the weight gradient
// dw_keras (3,3,3,1,Cout) for a given dy [N,X,Y,Z,Cout] (test hook for conv_first_tc.cu / the SIMT kernels behind it).
extern "C" int fm_op_conv3d_first(fm_ctx* ctx, const float* x, const float* w_keras, const float* bias, int N, int X,
                                  int Y, int Z, int Cout, int relu, float* y, const float* dy, float* dw_keras) {
  FM_CHECK(ctx && x && ((y && w_keras && bias) || (dy && dw_keras)), FM_EINVAL, "fm_op_conv3d_first: NULL argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t vox = (size_t)N * X * Y * Z;
  float* dx = nullptr;
  FM_TRY(s.up_f32(x, vox, &dx));
  if (y) {
    std::vector<float> packed((size_t)Cout * 27);
    keras_to_packed(w_keras, packed.data(), 3, 1, Cout);
    bf16 *wf = nullptr, *out = nullptr;
    float* dbias = nullptr;
    FM_TRY(s.up_bf16(packed.data(), packed.size(), &wf));
    FM_TRY(s.up_f32(bias, Cout, &dbias));
    FM_TRY(s.alloc(&out, vox * Cout));
    FM_TRY(k_conv3d_simt_fprop(ctx, dx, 1, nullptr, wf, dbias, out, nullptr, N, X, Y, Z, 1, 0, Cout, 3, relu, nullptr));
    FM_TRY(s.down_bf16(out, vox * Cout, y));
  }
  if (dy && dw_keras) {
    bf16* ddy = nullptr;
    float* dw = nullptr;
    FM_TRY(s.up_bf16(dy, vox * Cout, &ddy));
    FM_TRY(s.alloc(&dw, (size_t)Cout * 27));
    FM_TRY(k_zero(ctx, dw, (size_t)Cout * 27 * 4));
    FM_TRY(k_conv3d_simt_wgrad(ctx, dx, 1, ddy, dw, N, X, Y, Z, 1, 1, 0, Cout, 3));
    std::vector<float> host((size_t)Cout * 27);
    FM_CUDA(cudaMemcpyAsync(host.data(), dw, host.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaStreamSynchronize(ctx->stream));
    packed_to_keras(host.data(), dw_keras, 3, 1, Cout);
  }
  return FM_OK;
}

// Decoder convolution over concatenate([UpSampling3D(2)(coarse), skip]) computed at coarse resolution (test hooks for
// k_conv3d_up_*). coarse [N, X/2, Y/2, Z/2, Cc], skip [N, X, Y, Z, Cs], w_keras (3,3,3,Cc+Cs,Cout), y [N, X, Y, Z, Cout].
extern "C" int fm_op_conv3d_up_fprop(fm_ctx* ctx, const float* coarse, const float* skip, const float* w_keras,
                                     const float* bias, int N, int X, int Y, int Z, int Cc, int Cs, int Cout, int relu,
                                     float* y) {
  FM_CHECK(ctx && coarse && skip && w_keras && y, FM_EINVAL, "fm_op_conv3d_up_fprop: NULL argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t vox = (size_t)N * X * Y * Z;
  const int Ct = Cc + Cs;
  std::vector<float> packed((size_t)Cout * 27 * Ct);
  keras_to_packed(w_keras, packed.data(), 3, Ct, Cout);
  bf16 *dc = nullptr, *dsk = nullptr, *wf = nullptr, *wup = nullptr, *dy = nullptr;
  float *wm = nullptr, *dbias = nullptr;
  FM_TRY(s.up_bf16(coarse, vox / 8 * Cc, &dc));
  FM_TRY(s.up_bf16(skip, vox * Cs, &dsk));
  FM_TRY(s.up_bf16(packed.data(), packed.size(), &wf));
  FM_TRY(s.up_f32(packed.data(), packed.size(), &wm));
  FM_TRY(s.alloc(&wup, (size_t)Cout * 64 * Cc));
  if (bias) FM_TRY(s.up_f32(bias, Cout, &dbias));
  FM_TRY(s.alloc(&dy, vox * Cout));
  FM_TRY(k_repack_up(ctx, wm, wup, nullptr, Cout, Cc, Ct));
  FM_TRY(k_conv3d_up_fprop(ctx, dc, dsk, wup, wf, dbias, dy, N, X, Y, Z, Cc, Cs, Cout, relu));
  return s.down_bf16(dy, vox * Cout, y);
}

// Backward of the same layer towards the coarse tensor: dcoarse [N, X/2, Y/2, Z/2, Cc] (times coarse > 0 when
// apply_mask) and the weight gradient of the up-source channels dw_up_keras (3,3,3,Cc,Cout).
extern "C" int fm_op_conv3d_up_bwd(fm_ctx* ctx, const float* coarse, const float* dy, const float* w_keras, int N,
                                   int X, int Y, int Z, int Cc, int Cs, int Cout, int apply_mask, float* dcoarse,
                                   float* dw_up_keras) {
  FM_CHECK(ctx && coarse && dy && w_keras, FM_EINVAL, "fm_op_conv3d_up_bwd: NULL argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t vox = (size_t)N * X * Y * Z;
  const int Ct = Cc + Cs;
  std::vector<float> packed((size_t)Cout * 27 * Ct);
  keras_to_packed(w_keras, packed.data(), 3, Ct, Cout);
  bf16 *dc = nullptr, *ddy = nullptr, *wupd = nullptr, *dgc = nullptr;
  float *wm = nullptr, *dwu = nullptr, *dw = nullptr;
  FM_TRY(s.up_bf16(coarse, vox / 8 * Cc, &dc));
  FM_TRY(s.up_bf16(dy, vox * Cout, &ddy));
  FM_TRY(s.up_f32(packed.data(), packed.size(), &wm));
  FM_TRY(s.alloc(&wupd, (size_t)Cout * 64 * Cc));
  FM_TRY(k_repack_up(ctx, wm, nullptr, wupd, Cout, Cc, Ct));
  if (dcoarse) {
    FM_TRY(s.alloc(&dgc, vox / 8 * Cc));
    FM_TRY(k_conv3d_up_dgrad(ctx, ddy, wupd, dgc, apply_mask ? dc : nullptr, N, X, Y, Z, Cout, Cc));
    FM_TRY(s.down_bf16(dgc, vox / 8 * Cc, dcoarse));
  }
  if (dw_up_keras) {
    const size_t nu = (size_t)Cout * 64 * Cc, nw = (size_t)Cout * 27 * Cc;
    FM_TRY(s.alloc(&dwu, nu));
    FM_TRY(s.alloc(&dw, nw));
    FM_TRY(k_zero(ctx, dwu, nu * 4));
    FM_TRY(k_zero(ctx, dw, nw * 4));
    FM_TRY(k_conv3d_up_wgrad(ctx, dc, ddy, dwu, N, X, Y, Z, Cc, Cout));
    FM_TRY(k_fold_up_wgrad(ctx, dwu, dw, Cout, Cc, Cc));
    std::vector<float> host(nw);
    FM_CUDA(cudaMemcpyAsync(host.data(), dw, nw * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaStreamSynchronize(ctx->stream));
    packed_to_keras(host.data(), dw_up_keras, 3, Cc, Cout);
  }
  return FM_OK;
}

// pz = pooling factor along z: 2 (MaxPooling3D / UpSampling3D) or 1 (the 2D models); X, Y, Z = the finer extent for
// the pool hooks, the coarser one for the upsample hooks
extern "C" int fm_op_maxpool(fm_ctx* ctx, const float* x, int N, int X, int Y, int Z, int C, int pz, float* y) {
  FM_CHECK(ctx && x && y, FM_EINVAL, "fm_op_maxpool: NULL argument");
  FM_CHECK(pz == 1 || pz == 2, FM_EINVAL, "fm_op_maxpool: pz=%d", pz);
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z * C, nc = n / (4 * pz);
  bf16 *dx = nullptr, *dy = nullptr;
  FM_TRY(s.up_bf16(x, n, &dx));
  FM_TRY(s.alloc(&dy, nc));
  FM_TRY(k_maxpool3d_fwd(ctx, dx, dy, Dims5{N, X, Y, Z, C}, pz));
  return s.down_bf16(dy, nc, y);
}

extern "C" int fm_op_maxpool_bwd(fm_ctx* ctx, const float* x, const float* dy, const float* dskip,
                                   int N, int X, int Y, int Z, int C, int pz, float* dx) {
  FM_CHECK(ctx && x && dy && dx, FM_EINVAL, "fm_op_maxpool_bwd: NULL argument");
  FM_CHECK(pz == 1 || pz == 2, FM_EINVAL, "fm_op_maxpool_bwd: pz=%d", pz);
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z * C, nc = n / (4 * pz);
  bf16 *bx = nullptr, *bdy = nullptr, *bsk = nullptr, *bdx = nullptr;
  FM_TRY(s.up_bf16(x, n, &bx));
  FM_TRY(s.up_bf16(dy, nc, &bdy));
  if (dskip) FM_TRY(s.up_bf16(dskip, n, &bsk));
  FM_TRY(s.alloc(&bdx, n));
  FM_TRY(k_maxpool3d_bwd(ctx, bx, bdy, bsk, bdx, Dims5{N, X, Y, Z, C}, 1, pz));
  return s.down_bf16(bdx, n, dx);
}

extern "C" int fm_op_upsample(fm_ctx* ctx, const float* x, int N, int X, int Y, int Z, int C, int pz, float* y) {
  FM_CHECK(ctx && x && y, FM_EINVAL, "fm_op_upsample: NULL argument");
  FM_CHECK(pz == 1 || pz == 2, FM_EINVAL, "fm_op_upsample: pz=%d", pz);
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z * C, nf = n * 4 * pz;
  bf16 *dx = nullptr, *dy = nullptr;
  FM_TRY(s.up_bf16(x, n, &dx));
  FM_TRY(s.alloc(&dy, nf));
  FM_TRY(k_upsample3d_fwd(ctx, dx, dy, Dims5{N, X, Y, Z, C}, pz));
  return s.down_bf16(dy, nf, y);
}

extern "C" int fm_op_upsample_bwd(fm_ctx* ctx, const float* dy, const float* act, int N, int X, int Y,
                                    int Z, int C, int pz, float* dx) {
  FM_CHECK(ctx && dy && dx, FM_EINVAL, "fm_op_upsample_bwd: NULL argument");
  FM_CHECK(pz == 1 || pz == 2, FM_EINVAL, "fm_op_upsample_bwd: pz=%d", pz);
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z * C;  // coarse elements
  bf16 *bdy = nullptr, *bact = nullptr, *bdx = nullptr;
  FM_TRY(s.up_bf16(dy, n * 4 * pz, &bdy));
  if (act) FM_TRY(s.up_bf16(act, n, &bact));
  FM_TRY(s.alloc(&bdx, n));
  FM_TRY(k_upsample3d_bwd(ctx, bdy, bact, bdx, Dims5{N, X, Y, Z, C}, C, 0, pz));
  return s.down_bf16(bdx, n, dx);
}

// the MaxPooling3D / UpSampling3D forms (pz = 2) of the four hooks above
extern "C" int fm_op_maxpool3d(fm_ctx* ctx, const float* x, int N, int X, int Y, int Z, int C, float* y) {
  return fm_op_maxpool(ctx, x, N, X, Y, Z, C, 2, y);
}
extern "C" int fm_op_maxpool3d_bwd(fm_ctx* ctx, const float* x, const float* dy, const float* dskip, int N, int X, int Y,
                                   int Z, int C, float* dx) {
  return fm_op_maxpool_bwd(ctx, x, dy, dskip, N, X, Y, Z, C, 2, dx);
}
extern "C" int fm_op_upsample3d(fm_ctx* ctx, const float* x, int N, int X, int Y, int Z, int C, float* y) {
  return fm_op_upsample(ctx, x, N, X, Y, Z, C, 2, y);
}
extern "C" int fm_op_upsample3d_bwd(fm_ctx* ctx, const float* dy, const float* act, int N, int X, int Y, int Z, int C,
                                    float* dx) {
  return fm_op_upsample_bwd(ctx, dy, act, N, X, Y, Z, C, 2, dx);
}

extern "C" int fm_op_dice(fm_ctx* ctx, const float* p, const float* t, int64_t n, double sums[8],
                          float* dloss_dp) {
  FM_CHECK(ctx && p && t && sums && n > 0, FM_EINVAL, "fm_op_dice: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  float *dp = nullptr, *dt = nullptr, *dg = nullptr;
  double* ds = nullptr;
  FM_TRY(s.up_f32(p, (size_t)n, &dp));
  FM_TRY(s.up_f32(t, (size_t)n, &dt));
  FM_TRY(s.alloc(&ds, kNumLossSums));
  FM_TRY(k_dice_sums(ctx, dp, dt, n, ds, 0));
  FM_CUDA(cudaMemcpyAsync(sums, ds, 64, cudaMemcpyDeviceToHost, ctx->stream));
  if (dloss_dp) {
    FM_TRY(s.alloc(&dg, (size_t)n));
    FM_TRY(k_dice_bwd(ctx, dp, dt, ds, n, dg, 0));
    FM_CUDA(cudaMemcpyAsync(dloss_dp, dg, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  return FM_OK;
}

extern "C" int fm_op_dice_xent(fm_ctx* ctx, const float* p, const float* t, const float* mask, int64_t n,
                               float xent_weight, float dist_sigma, double sums[9], float* dloss_dz) {
  FM_CHECK(ctx && p && t && sums && n > 0, FM_EINVAL, "fm_op_dice_xent: bad argument");
  FM_CHECK(mask == nullptr || dist_sigma > 0.f, FM_EINVAL, "fm_op_dice_xent: dist_sigma must be positive");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  float *dp = nullptr, *dt = nullptr, *dm = nullptr, *dg = nullptr;
  double* ds = nullptr;
  FM_TRY(s.up_f32(p, (size_t)n, &dp));
  FM_TRY(s.up_f32(t, (size_t)n, &dt));
  if (mask) FM_TRY(s.up_f32(mask, (size_t)n, &dm));
  XentSpec xs;
  xs.weight = xent_weight;
  xs.inv_sigma = mask ? 1.f / dist_sigma : 0.f;
  xs.mask = dm;
  FM_TRY(s.alloc(&ds, kNumLossSums));
  FM_TRY(k_dice_sums(ctx, dp, dt, n, ds, 0, xs));
  FM_CUDA(cudaMemcpyAsync(sums, ds, kNumLossSums * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  if (dloss_dz) {
    FM_TRY(s.alloc(&dg, (size_t)n));
    FM_TRY(k_dice_bwd(ctx, dp, dt, ds, n, dg, 1, xs));
    FM_CUDA(cudaMemcpyAsync(dloss_dz, dg, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  return FM_OK;
}

extern "C" int fm_op_adam(fm_ctx* ctx, float* p, const float* g, float* mm, float* vv, int64_t n,
                          int iterations, float lr) {
  FM_CHECK(ctx && p && g && mm && vv && n > 0, FM_EINVAL, "fm_op_adam: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  float *dp, *dg, *dm, *dv;
  FM_TRY(s.up_f32(p, (size_t)n, &dp));
  FM_TRY(s.up_f32(g, (size_t)n, &dg));
  FM_TRY(s.up_f32(mm, (size_t)n, &dm));
  FM_TRY(s.up_f32(vv, (size_t)n, &dv));
  FM_TRY(k_adam(ctx, dp, dg, dm, dv, n, iterations, lr));
  FM_CUDA(cudaMemcpyAsync(p, dp, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(mm, dm, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(vv, dv, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  return FM_OK;
}

// Scratch of the normalisation kernels: per-(sample, block) partials for at most 1024 blocks per sample (norm_blocks)
// plus the per-(sample, channel) coefficients of the forward (2) or backward (4) pass.
static size_t norm_scratch_floats(int N, int C) { return (size_t)N * C * (2 * 1024 + 4); }

// InstanceNormalization + LeakyReLU(0.3) of the Isensee blocks (isensee_block): y = act(norm(x)) * chan_scale + add.
// add [N,vox,C] and chan_scale [N,C] may be NULL; stats [N,C,2] (optional) = (mean, 1/(std + eps)).
extern "C" int fm_op_instnorm_lrelu(fm_ctx* ctx, const float* x, const float* gamma, const float* beta, const float* add,
                                    const float* chan_scale, int N, int64_t vox, int C, float* y, float* stats) {
  FM_CHECK(ctx && x && gamma && beta && y && N > 0 && vox > 0, FM_EINVAL, "fm_op_instnorm_lrelu: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * vox * C, ns = norm_scratch_floats(N, C);
  bf16 *bx = nullptr, *badd = nullptr, *by = nullptr;
  float *dg = nullptr, *db = nullptr, *dcs = nullptr, *scratch = nullptr, *dst = nullptr;
  FM_TRY(s.up_bf16(x, n, &bx));
  if (add) FM_TRY(s.up_bf16(add, n, &badd));
  if (chan_scale) FM_TRY(s.up_f32(chan_scale, (size_t)N * C, &dcs));
  FM_TRY(s.up_f32(gamma, C, &dg));
  FM_TRY(s.up_f32(beta, C, &db));
  FM_TRY(s.alloc(&scratch, ns));
  FM_TRY(s.alloc(&dst, (size_t)N * C * 2));
  FM_TRY(s.alloc(&by, n));
  FM_TRY(k_instnorm_lrelu(ctx, bx, dg, db, badd, by, N, vox, C, scratch, ns, dst, dcs));
  if (stats) FM_CUDA(cudaMemcpyAsync(stats, dst, (size_t)N * C * 2 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  return s.down_bf16(by, n, y);
}

// Its backward (is_block_bwd): the forward runs first for the device's own statistics; gy2 (the second incoming
// gradient of a fan-out) and chan_scale may be NULL. dgamma / dbeta [C] are zeroed here (the kernel accumulates).
extern "C" int fm_op_instnorm_lrelu_bwd(fm_ctx* ctx, const float* x, const float* gamma, const float* beta,
                                        const float* gy, const float* gy2, const float* chan_scale, int N, int64_t vox,
                                        int C, float* dx, float* dgamma, float* dbeta) {
  FM_CHECK(ctx && x && gamma && beta && gy && dx && dgamma && dbeta && N > 0 && vox > 0, FM_EINVAL,
           "fm_op_instnorm_lrelu_bwd: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * vox * C, ns = norm_scratch_floats(N, C);
  bf16 *bx = nullptr, *bgy = nullptr, *bgy2 = nullptr, *by = nullptr, *bdx = nullptr;
  float *dg = nullptr, *db = nullptr, *dcs = nullptr, *scratch = nullptr, *dst = nullptr, *dgg = nullptr;
  FM_TRY(s.up_bf16(x, n, &bx));
  FM_TRY(s.up_bf16(gy, n, &bgy));
  if (gy2) FM_TRY(s.up_bf16(gy2, n, &bgy2));
  if (chan_scale) FM_TRY(s.up_f32(chan_scale, (size_t)N * C, &dcs));
  FM_TRY(s.up_f32(gamma, C, &dg));
  FM_TRY(s.up_f32(beta, C, &db));
  FM_TRY(s.alloc(&scratch, ns));
  FM_TRY(s.alloc(&dst, (size_t)N * C * 2));
  FM_TRY(s.alloc(&dgg, 2 * (size_t)C));
  FM_TRY(s.alloc(&by, n));
  FM_TRY(s.alloc(&bdx, n));
  FM_TRY(k_instnorm_lrelu(ctx, bx, dg, db, nullptr, by, N, vox, C, scratch, ns, dst, dcs));
  FM_TRY(k_zero(ctx, dgg, 2 * (size_t)C * 4));
  FM_TRY(k_instnorm_lrelu_bwd(ctx, bx, dst, dg, db, bgy, bgy2, dcs, bdx, dgg, dgg + C, N, vox, C, scratch, ns));
  FM_CUDA(cudaMemcpyAsync(dgamma, dgg, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(dbeta, dgg + C, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
  return s.down_bf16(bdx, n, dx);
}

// BatchNormalization + ReLU (bn_block_fwd): training = batch statistics, and moving_mean / moving_var [C] (in/out)
// take the Keras moving-average step; inference = the moving statistics.
extern "C" int fm_op_batchnorm_relu(fm_ctx* ctx, int training, const float* x, const float* gamma, const float* beta,
                                    float* moving_mean, float* moving_var, int N, int64_t vox, int C, float* y) {
  FM_CHECK(ctx && x && gamma && beta && moving_mean && moving_var && y && N > 0 && vox > 0, FM_EINVAL,
           "fm_op_batchnorm_relu: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * vox * C, ns = norm_scratch_floats(N, C);
  bf16 *bx = nullptr, *by = nullptr;
  float *dg = nullptr, *db = nullptr, *dmm = nullptr, *dmv = nullptr, *scratch = nullptr, *dst = nullptr;
  FM_TRY(s.up_bf16(x, n, &bx));
  FM_TRY(s.up_f32(gamma, C, &dg));
  FM_TRY(s.up_f32(beta, C, &db));
  FM_TRY(s.up_f32(moving_mean, C, &dmm));
  FM_TRY(s.up_f32(moving_var, C, &dmv));
  FM_TRY(s.alloc(&scratch, ns));
  FM_TRY(s.alloc(&dst, (size_t)N * C * 2));
  FM_TRY(s.alloc(&by, n));
  FM_TRY(k_batchnorm_relu(ctx, bx, dg, db, dmm, dmv, by, N, vox, C, scratch, ns, training ? dst : nullptr,
                          training ? 1 : 0));
  FM_CUDA(cudaMemcpyAsync(moving_mean, dmm, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(moving_var, dmv, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
  return s.down_bf16(by, n, y);
}

// Its backward (bn_block_bwd) after a training forward that supplies the batch statistics; gy2 may be NULL.
// dgamma / dbeta [C] are zeroed here (the kernel adds into them).
extern "C" int fm_op_batchnorm_relu_bwd(fm_ctx* ctx, const float* x, const float* gamma, const float* beta,
                                        const float* gy, const float* gy2, int N, int64_t vox, int C, float* dx,
                                        float* dgamma, float* dbeta) {
  FM_CHECK(ctx && x && gamma && beta && gy && dx && dgamma && dbeta && N > 0 && vox > 0, FM_EINVAL,
           "fm_op_batchnorm_relu_bwd: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * vox * C, ns = norm_scratch_floats(N, C);
  bf16 *bx = nullptr, *bgy = nullptr, *bgy2 = nullptr, *by = nullptr, *bdx = nullptr;
  float *dg = nullptr, *db = nullptr, *scratch = nullptr, *dst = nullptr, *dgg = nullptr;
  FM_TRY(s.up_bf16(x, n, &bx));
  FM_TRY(s.up_bf16(gy, n, &bgy));
  if (gy2) FM_TRY(s.up_bf16(gy2, n, &bgy2));
  FM_TRY(s.up_f32(gamma, C, &dg));
  FM_TRY(s.up_f32(beta, C, &db));
  FM_TRY(s.alloc(&scratch, ns));
  FM_TRY(s.alloc(&dst, (size_t)N * C * 2));
  FM_TRY(s.alloc(&dgg, 2 * (size_t)C));
  FM_TRY(s.alloc(&by, n));
  FM_TRY(s.alloc(&bdx, n));
  FM_TRY(k_batchnorm_relu(ctx, bx, dg, db, nullptr, nullptr, by, N, vox, C, scratch, ns, dst, 1));
  FM_TRY(k_zero(ctx, dgg, 2 * (size_t)C * 4));
  FM_TRY(k_batchnorm_relu_bwd(ctx, bx, dst, dg, db, bgy, bgy2, bdx, dgg, dgg + C, N, vox, C, scratch, ns));
  FM_CUDA(cudaMemcpyAsync(dgamma, dgg, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaMemcpyAsync(dbeta, dgg + C, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
  return s.down_bf16(bdx, n, dx);
}

// Stride-2 TF-'SAME' convolution of the Isensee in-convs (isensee_block, relu 0): x [N,Xin,Yin,Zin,Cin] (even extents;
// Zin is not strided for ksize 31), w_keras (3,3[,3],Cin,Cout), y [N,Xin/2,Yin/2,Zout,Cout]. With dy (same shape as y):
// the backward of backward_isensee - zero insertion, then the stride-1 data gradient dx [N,Xin,Yin,Zin,Cin] and weight
// gradient dw_keras on the kernels the model picks for that extent.
extern "C" int fm_op_conv_strided(fm_ctx* ctx, const float* x, const float* w_keras, const float* bias, int N, int Xin,
                                  int Yin, int Zin, int Cin, int Cout, int ksize, float* y, const float* dy, float* dx,
                                  float* dw_keras) {
  FM_CHECK(ctx && x && w_keras && (ksize == 3 || ksize == 31), FM_EINVAL, "fm_op_conv_strided: bad argument");
  FM_CHECK(Xin % 2 == 0 && Yin % 2 == 0 && (ksize == 31 || Zin % 2 == 0), FM_EINVAL, "fm_op_conv_strided: odd extent");
  FM_CHECK(!dy || (dx && dw_keras), FM_EINVAL, "fm_op_conv_strided: dy needs dx and dw_keras");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const int pz = ksize == 31 ? 1 : 2, X = Xin / 2, Y = Yin / 2, Z = Zin / pz, taps = kext_taps(ksize);
  const size_t vin = (size_t)N * Xin * Yin * Zin, vout = (size_t)N * X * Y * Z, wn = (size_t)Cout * taps * Cin;
  std::vector<float> packed(wn);
  keras_to_packed(w_keras, packed.data(), ksize, Cin, Cout);
  bf16 *bx = nullptr, *wf = nullptr, *wd = nullptr;
  float* wm = nullptr;
  FM_TRY(s.up_bf16(x, vin * Cin, &bx));
  FM_TRY(s.up_f32(packed.data(), wn, &wm));
  FM_TRY(s.alloc(&wf, wn));
  FM_TRY(s.alloc(&wd, wn));
  FM_TRY(k_repack_weights(ctx, wm, wf, wd, nullptr, Cout, taps, Cin, 0));
  if (y) {
    FM_CHECK(conv_tc_supported(Cin, 0, Cout, ksize), FM_EINVAL, "fm_op_conv_strided: no strided kernel for %d -> %d",
             Cin, Cout);
    bf16* by = nullptr;
    float* db = nullptr;
    if (bias) FM_TRY(s.up_f32(bias, Cout, &db));
    FM_TRY(s.alloc(&by, vout * Cout));
    FM_TRY(k_conv3d_tc_fprop(ctx, bx, nullptr, wf, db, by, nullptr, N, X, Y, Z, Cin, 0, Cout, ksize, 0, Cout, 0, 2, Xin,
                             Yin, Zin));
    FM_TRY(s.down_bf16(by, vout * Cout, y));
  }
  if (dy) {
    bf16 *bdy = nullptr, *bz = nullptr, *bdx = nullptr, *wmd = nullptr;
    float* dw = nullptr;
    FM_TRY(s.up_bf16(dy, vout * Cout, &bdy));
    FM_TRY(s.alloc(&bz, vin * Cout));
    FM_TRY(s.alloc(&bdx, vin * Cin));
    FM_TRY(s.alloc(&dw, wn));
    FM_TRY(k_zero(ctx, dw, wn * 4));
    FM_TRY(k_zero_insert(ctx, bdy, bz, Dims5{N, X, Y, Z, Cout}, pz));
    FM_TRY(isensee_wgrad_route(ctx, bx, bz, dw, N, Xin, Yin, Zin, Cin, Cin, 0, Cout, ksize));
    if (isensee_dgrad_marches(Xin, Yin, Zin, Cin, Cin, Cout, ksize)) {
      FM_TRY(s.alloc(&wmd, (size_t)conv_march_pack_elems(Cout, Cin)));
      FM_TRY(k_repack_march(ctx, wd, wmd, Cin, Cout, 0, Cout, conv_march_kc(Cout, 0, Cin, Cout)));
    }
    FM_TRY(isensee_dgrad_route(ctx, bz, wmd, wd, bdx, N, Xin, Yin, Zin, Cout, Cin, ksize, false));
    FM_TRY(s.down_bf16(bdx, vin * Cin, dx));
    std::vector<float> host(wn);
    FM_CUDA(cudaMemcpyAsync(host.data(), dw, wn * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaStreamSynchronize(ctx->stream));
    packed_to_keras(host.data(), dw_keras, ksize, Cin, Cout);
  }
  return FM_OK;
}

// Deconvolution3D / Deconvolution2D (kernel 2, stride 2, C -> C channels) as the U-Nets run it: the 1x1x1 conv of the
// coarse x [N,X,Y,Z,C] to 4*pz*C channels, then depth-to-space with the bias -> y [N,2X,2Y,pz*Z,C]. w_keras is the
// Keras kernel (2,2[,2],C,C) = (..., Cout, Cin). With dy [N,2X,2Y,pz*Z,C]: the backward of backward_unet /
// backward_unet_bn - bias gradient, space-to-depth, the 1x1x1 weight gradient and the data gradient dx (masked by
// x > 0 when relu_mask, as behind a ReLU block of the plain U-Net).
extern "C" int fm_op_deconv(fm_ctx* ctx, const float* x, const float* w_keras, const float* bias, int N, int X, int Y,
                            int Z, int C, int pz, float* y, const float* dy, int relu_mask, float* dx, float* dw_keras,
                            float* dbias) {
  FM_CHECK(ctx && x && w_keras && (pz == 1 || pz == 2), FM_EINVAL, "fm_op_deconv: bad argument");
  FM_CHECK(!dy || (dx && dw_keras && dbias), FM_EINVAL, "fm_op_deconv: dy needs dx, dw_keras and dbias");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const int c8 = 4 * pz * C;
  const Dims5 dc{N, X, Y, Z, C};
  const size_t vc = (size_t)N * X * Y * Z, nf = vc * c8, wn = (size_t)c8 * C;
  bf16 *bx = nullptr, *wf = nullptr, *wd = nullptr, *bz = nullptr;
  float* wm = nullptr;
  FM_TRY(s.up_bf16(x, vc * C, &bx));
  FM_TRY(s.up_f32(w_keras, wn, &wm));  // the Keras kernel is the master layout [class][Cout][Cin]
  FM_TRY(s.alloc(&wf, wn));
  FM_TRY(s.alloc(&wd, wn));
  FM_TRY(k_repack_weights(ctx, wm, wf, wd, nullptr, c8, 1, C, 0));
  FM_TRY(s.alloc(&bz, nf));
  if (y) {
    FM_CHECK(bias, FM_EINVAL, "fm_op_deconv: y needs the bias");
    bf16* by = nullptr;
    float* db = nullptr;
    FM_TRY(s.up_f32(bias, C, &db));
    FM_TRY(s.alloc(&by, nf));
    FM_TRY(k_conv3d_tc_fprop(ctx, bx, nullptr, wf, nullptr, bz, nullptr, N, X, Y, Z, C, 0, c8, 1, 0, c8, 0));
    FM_TRY(k_depth_to_space(ctx, bz, db, by, dc, pz));
    FM_TRY(s.down_bf16(by, nf, y));
  }
  if (dy) {
    bf16 *bdy = nullptr, *bdx = nullptr;
    float *dw = nullptr, *db = nullptr;
    FM_TRY(s.up_bf16(dy, nf, &bdy));
    FM_TRY(s.alloc(&bdx, vc * C));
    FM_TRY(s.alloc(&dw, wn));
    FM_TRY(s.alloc(&db, C));
    FM_TRY(k_zero(ctx, dw, wn * 4));
    FM_TRY(k_zero(ctx, db, (size_t)C * 4));
    FM_TRY(k_bias_grad(ctx, bdy, db, (int64_t)nf / C, C));
    FM_TRY(k_space_to_depth(ctx, bdy, bz, dc, pz));
    FM_TRY(k_conv3d_tc_wgrad(ctx, bx, bz, dw, N, X, Y, Z, C, C, 0, c8, 1));
    FM_TRY(k_conv3d_tc_fprop(ctx, bz, nullptr, wd, nullptr, bdx, relu_mask ? bx : nullptr, N, X, Y, Z, c8, 0, C, 1, 0, C,
                             0));
    FM_CUDA(cudaMemcpyAsync(dw_keras, dw, wn * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaMemcpyAsync(dbias, db, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_TRY(s.down_bf16(bdx, vc * C, dx));
  }
  return FM_OK;
}

// The raw shuffles of the deconvolution, without bias: depth-to-space of z8 [N,X,Y,Z,4*pz*C] -> fine
// [N,2X,2Y,pz*Z,C] (to_space = 1) or its inverse (to_space = 0, fine -> z8).
extern "C" int fm_op_depth_space(fm_ctx* ctx, int to_space, const float* in, int N, int X, int Y, int Z, int C, int pz,
                                 float* out) {
  FM_CHECK(ctx && in && out && (pz == 1 || pz == 2), FM_EINVAL, "fm_op_depth_space: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z * C * 4 * pz;
  bf16 *bi = nullptr, *bo = nullptr;
  FM_TRY(s.up_bf16(in, n, &bi));
  FM_TRY(s.alloc(&bo, n));
  if (to_space)
    FM_TRY(k_depth_to_space(ctx, bi, nullptr, bo, Dims5{N, X, Y, Z, C}, pz));
  else
    FM_TRY(k_space_to_depth(ctx, bi, bo, Dims5{N, X, Y, Z, C}, pz));
  return s.down_bf16(bo, n, out);
}

// Zero insertion of the strided-conv backward: coarse [N,X,Y,Z,C] -> fine [N,2X,2Y,pz*Z,C], fine[2v+1] = coarse[v].
extern "C" int fm_op_zero_insert(fm_ctx* ctx, const float* coarse, int N, int X, int Y, int Z, int C, int pz,
                                 float* fine) {
  FM_CHECK(ctx && coarse && fine && (pz == 1 || pz == 2), FM_EINVAL, "fm_op_zero_insert: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z * C;
  bf16 *bc = nullptr, *bf = nullptr;
  FM_TRY(s.up_bf16(coarse, n, &bc));
  FM_TRY(s.alloc(&bf, n * 4 * pz));
  FM_TRY(k_zero_insert(ctx, bc, bf, Dims5{N, X, Y, Z, C}, pz));
  return s.down_bf16(bf, n * 4 * pz, fine);
}

// The 1x1x1 single-output heads. Forward when p != NULL: p = [sigmoid](x . w + b) (k_head_fwd), or with targets t the
// training form k_head_fwd_dice (always through the sigmoid) that also returns the 8 loss statistics in sums.
// Backward when dz != NULL (k_head_bwd): dx = dz * w (mode 0: masked by x > 0; mode 1: plain; mode 2: added to dx, which
// is then in/out), dw [C] = sum dz * x and db [1] = sum dz.
extern "C" int fm_op_head(fm_ctx* ctx, const float* x, const float* w, const float* b, int64_t voxels, int C,
                          int apply_sigmoid, const float* t, float* p, double sums[8], const float* dz, int mode, float* dx,
                          float* dw, float* db) {
  FM_CHECK(ctx && x && w && voxels > 0, FM_EINVAL, "fm_op_head: bad argument");
  FM_CHECK(!p || b, FM_EINVAL, "fm_op_head: the forward needs b");
  FM_CHECK(!t || (p && sums), FM_EINVAL, "fm_op_head: t needs p and sums");
  FM_CHECK(!dz || (dx && dw && db && mode >= 0 && mode <= 2), FM_EINVAL, "fm_op_head: dz needs dx, dw, db, mode 0-2");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)voxels * C;
  bf16* bx = nullptr;
  float *dwt = nullptr, *dbias = nullptr;
  FM_TRY(s.up_bf16(x, n, &bx));
  FM_TRY(s.up_f32(w, C, &dwt));
  if (p) {
    float *dp = nullptr, *dt = nullptr;
    FM_TRY(s.up_f32(b, 1, &dbias));
    FM_TRY(s.alloc(&dp, (size_t)voxels));
    if (t) {
      double* ds = nullptr;
      FM_TRY(s.up_f32(t, (size_t)voxels, &dt));
      FM_TRY(s.alloc(&ds, kNumLossSums));
      FM_TRY(k_head_fwd_dice(ctx, bx, dwt, dbias, dt, dp, voxels, C, ds));
      FM_CUDA(cudaMemcpyAsync(sums, ds, 8 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    } else {
      FM_TRY(k_head_fwd(ctx, bx, dwt, dbias, dp, voxels, C, apply_sigmoid));
    }
    FM_CUDA(cudaMemcpyAsync(p, dp, (size_t)voxels * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  if (dz) {
    float *ddz = nullptr, *dg = nullptr;
    bf16* bdx = nullptr;
    FM_TRY(s.up_f32(dz, (size_t)voxels, &ddz));
    if (mode == 2)
      FM_TRY(s.up_bf16(dx, n, &bdx));
    else
      FM_TRY(s.alloc(&bdx, n));
    FM_TRY(s.alloc(&dg, (size_t)C + 1));
    FM_TRY(k_zero(ctx, dg, ((size_t)C + 1) * 4));
    FM_TRY(k_head_bwd(ctx, bx, ddz, dwt, bdx, dg, dg + C, voxels, C, mode));
    FM_CUDA(cudaMemcpyAsync(dw, dg, (size_t)C * 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_CUDA(cudaMemcpyAsync(db, dg + C, 4, cudaMemcpyDeviceToHost, ctx->stream));
    FM_TRY(s.down_bf16(bdx, n, dx));
  }
  return FM_OK;
}

// Deep-supervision plumbing of the Isensee nets (fp32 single-channel maps): out [N,X,Y,Z] = fine + the coarse map
// [N,X/2,Y/2,Z/pz] upsampled, and the gradient of that upsampling: coarse [N,X,Y,Z] = 2x2(x2) sum-pool of fine
// [N,2X,2Y,pz*Z].
extern "C" int fm_op_seg_upsample_add(fm_ctx* ctx, const float* fine, const float* coarse, int N, int X, int Y, int Z,
                                      int pz, float* out) {
  FM_CHECK(ctx && fine && coarse && out && (pz == 1 || pz == 2), FM_EINVAL, "fm_op_seg_upsample_add: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z;
  float *df = nullptr, *dc = nullptr, *dout = nullptr;
  FM_TRY(s.up_f32(fine, n, &df));
  FM_TRY(s.up_f32(coarse, n / (4 * pz), &dc));
  FM_TRY(s.alloc(&dout, n));
  FM_TRY(k_seg_upsample_add(ctx, df, dc, dout, N, X, Y, Z, pz));
  FM_CUDA(cudaMemcpyAsync(out, dout, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  return FM_OK;
}

extern "C" int fm_op_sumpool_f32(fm_ctx* ctx, const float* fine, int N, int X, int Y, int Z, int pz, float* coarse) {
  FM_CHECK(ctx && fine && coarse && (pz == 1 || pz == 2), FM_EINVAL, "fm_op_sumpool_f32: bad argument");
  FM_CUDA(cudaSetDevice(ctx->device));
  OpScratch s(ctx);
  const size_t n = (size_t)N * X * Y * Z;
  float *df = nullptr, *dc = nullptr;
  FM_TRY(s.up_f32(fine, n * 4 * pz, &df));
  FM_TRY(s.alloc(&dc, n));
  FM_TRY(k_sumpool_f32(ctx, df, dc, N, X, Y, Z, pz));
  FM_CUDA(cudaMemcpyAsync(coarse, dc, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  FM_CUDA(cudaStreamSynchronize(ctx->stream));
  return FM_OK;
}
