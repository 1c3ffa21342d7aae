// sampler.cu — training patches cut on the device (SURVEY.md §8f rank 3).
//
// The reference's training generator (fetal_net/generator.py:222-348) keeps every case in host memory, draws a random
// patch corner per sample (np.random.randint, generator.py:266-269), slices the data patch, the truth slice(s) at
// `truth_index` and - for the 2.5D models - the previous-truth slice(s) at `prev_truth_index` with
// get_patch_from_3d_data (edge-replicated where a slice sticks out, utils/patches.py:57-91), concatenates the previous
// truth to the data on the last axis (generator.py:305-306) and stacks a batch (convert_data, generator.py:380-401).
// At a few milliseconds per training step that host loop (and the H2D copy of every batch) is the bottleneck, so here
// the cases live in HBM (float32, the dtype Keras feeds) and ONE kernel cuts the whole batch straight into the
// model's input / target buffers. The random decisions stay on the host (fetal_net/device_sampler.py draws case order,
// corners and the skip-blank rejections with the reference's own np.random call sequence), so the device only needs
// (case, corner) per sample: index mapping bit-exact by construction, values bit-exact float32 copies.
//
// Optional cheap augmentations on the way (NOT the reference's nilearn / imgaug pipeline, generator.py:271-295, which
// stays on the host through the overlay): axis flips, an intensity scale, additive Gaussian noise from a counter-based
// hash - all per sample, parameters drawn by the host. A second kernel (sample_patches_warp_kernel) adds the library's
// own geometric augmentation: every output element reads its source through a per-sample affine map and an optional
// elastic displacement (fm_sample_warp, include/fetal_b200.h), data trilinearly, truth at the nearest sample.
#include <cmath>
#include <vector>

#include "common.cuh"

struct fm_volset {
  fm_ctx* ctx = nullptr;
  struct Case {
    float *data = nullptr, *truth = nullptr;
    int32_t dims[3] = {0, 0, 0};
  };
  std::vector<Case> cases;
  // device table of the cases (pointers + dims), rebuilt when a case changes
  struct DevCase {
    const float *data, *truth;
    int32_t dims[3];
    int32_t pad;
  };
  DevCase* table = nullptr;
  bool table_dirty = true;
  // per-sample (case, corner[3], flip bits) + float (scale, sigma) staging on the device, followed by the warps
  int32_t* d_args = nullptr;
  size_t d_args_bytes = 0;
};

namespace {

constexpr int kThreadsS = 256;

struct SampleGeom {
  int32_t patch[3];          // P0, P1, P2 of the data patch
  int32_t truth_index, truth_size, prev_index, prev_size;  // prev_size == 0: no previous-truth channels
  int32_t x_pitch;           // P2 + prev_size (last-axis extent of the network input)
};

__device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}
// standard normal from two counter-based uniforms (Box-Muller)
__device__ __forceinline__ float gauss(uint32_t seed, uint32_t idx) {
  const uint32_t a = hash32(idx * 2u + seed), b = hash32(idx * 2u + 1u + seed * 0x9e3779b9u);
  const float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777217.0f), u2 = (float)(b >> 8) * (1.0f / 16777216.0f);
  return sqrtf(-2.0f * __logf(u1)) * __cosf(6.28318530718f * u2);
}

// args per sample: int32 [8] = {case, cx, cy, cz, flip bits (1: x, 2: y, 4: z), noise seed, bits of scale, bits of sigma}
// x: [B][P0][P1][P2 + prev_size] (data patch | previous-truth slices), y: [B][P0][P1][truth_size]
// Batches of up to kInlineSamples samples carry their arguments in the kernel parameters (no staging buffer, no
// synchronisation with the previous step); larger ones read them from `args`.
constexpr int kInlineSamples = 64;
struct SampleArgs {
  int32_t v[kInlineSamples * 8];
};
__global__ void __launch_bounds__(kThreadsS) sample_patches_kernel(const fm_volset::DevCase* __restrict__ cases,
                                                                   const int32_t* __restrict__ args,
                                                                   const __grid_constant__ SampleArgs inl, SampleGeom gm,
                                                                   float* __restrict__ x, float* __restrict__ y) {
  const int b = blockIdx.y;
  const int32_t* a = args != nullptr ? args + b * 8 : inl.v + b * 8;
  const fm_volset::DevCase cs = cases[a[0]];
  const int cx = a[1], cy = a[2], cz = a[3], flip = a[4];
  const uint32_t seed = (uint32_t)a[5];
  const float scale = __int_as_float(a[6]), sigma = __int_as_float(a[7]);
  const int P0 = gm.patch[0], P1 = gm.patch[1], P2 = gm.patch[2];
  const int rowx = gm.x_pitch, rowy = gm.truth_size;
  const int64_t nx = (int64_t)P0 * P1 * rowx, ny = (int64_t)P0 * P1 * rowy;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < nx + ny; g += (int64_t)gridDim.x * blockDim.x) {
    const bool is_y = g >= nx;
    const int64_t q = is_y ? g - nx : g;
    const int row = is_y ? rowy : rowx;
    const int k = (int)(q % row);
    const int64_t ij = q / row;
    int j = (int)(ij % P1), i = (int)(ij / P1);
    // flips act on the assembled sample (data, previous truth and target alike), like flipping the arrays on the host
    if (flip & 1) i = P0 - 1 - i;
    if (flip & 2) j = P1 - 1 - j;
    const float* src;
    int zz;
    bool is_data = false;
    if (is_y) {
      src = cs.truth;
      zz = cz + gm.truth_index + ((flip & 4) ? rowy - 1 - k : k);
    } else if (k < P2) {
      src = cs.data;
      zz = cz + ((flip & 4) ? P2 - 1 - k : k);
      is_data = true;
    } else {
      src = cs.truth;
      const int kk = k - P2;
      zz = cz + gm.prev_index + ((flip & 4) ? gm.prev_size - 1 - kk : kk);
    }
    // get_patch_from_3d_data completes a patch that sticks out with the nearest edge sample (np.pad(mode='edge')):
    // clamping the coordinates yields the same values
    const int xx = min(max(cx + i, 0), cs.dims[0] - 1);
    const int yy = min(max(cy + j, 0), cs.dims[1] - 1);
    zz = min(max(zz, 0), cs.dims[2] - 1);
    float v = __ldg(src + ((int64_t)xx * cs.dims[1] + yy) * cs.dims[2] + zz);
    if (is_data) {
      v *= scale;
      if (sigma > 0.f) v += sigma * gauss(seed, (uint32_t)q);
    }
    (is_y ? y + (int64_t)b * ny : x + (int64_t)b * nx)[q] = v;
  }
}

// Per-sample warp as the kernel takes it: the matrix, c + offset (c = the centre of the data box, rounded once from
// float64) and the elastic parameters.
struct WarpArgs {
  float m[9];
  float ct[3];
  float alpha[3];
  uint32_t seed;
  int32_t grid;
};
struct WarpInline {
  WarpArgs w[kInlineSamples];
};
constexpr int kMaxGrid = 8;
// kernel parameters: 4 pointers + the inline arguments + the geometry; the parameter block holds at most 32764 bytes
static_assert(4 * sizeof(void*) + sizeof(SampleArgs) + sizeof(WarpInline) + sizeof(SampleGeom) <= 32764,
              "sample_patches_warp_kernel: inline arguments exceed the kernel parameter limit");

__device__ __forceinline__ float lerpf(float a, float b, float f) { return fmaf(f, b - a, a); }

// The sample_patches_kernel cut with a warp: the element that the unwarped kernel reads at volume position q (after
// the flips) reads s = c + t + M (q + d(q) - c). q - c is formed from the patch-local indices and the half-extents
// (exact in float32), so an identity, integer-offset or axis-permuting warp reproduces the unwarped cut bit for bit.
__global__ void __launch_bounds__(kThreadsS) sample_patches_warp_kernel(
    const fm_volset::DevCase* __restrict__ cases, const int32_t* __restrict__ args, const WarpArgs* __restrict__ warps,
    const __grid_constant__ SampleArgs inl, const __grid_constant__ WarpInline winl, SampleGeom gm,
    float* __restrict__ x, float* __restrict__ y) {
  __shared__ float ctrl[3 * kMaxGrid * kMaxGrid * kMaxGrid];  // [axis][gx][gy][gz] elastic control values
  const int b = blockIdx.y;
  const int32_t* a = args != nullptr ? args + b * 8 : inl.v + b * 8;
  const WarpArgs& w = warps != nullptr ? warps[b] : winl.w[b];
  const fm_volset::DevCase cs = cases[a[0]];
  const int flip = a[4];
  const uint32_t seed = (uint32_t)a[5];
  const float scale = __int_as_float(a[6]), sigma = __int_as_float(a[7]);
  float M[9];
#pragma unroll
  for (int t = 0; t < 9; ++t) M[t] = w.m[t];
  const float ct0 = w.ct[0], ct1 = w.ct[1], ct2 = w.ct[2];
  const float al0 = w.alpha[0], al1 = w.alpha[1], al2 = w.alpha[2];
  const int G = w.grid, G3 = G * G * G;
  const int P0 = gm.patch[0], P1 = gm.patch[1], P2 = gm.patch[2];
  if (G > 0) {  // uniform over the block (one sample per blockIdx.y)
    const uint32_t hs = hash32(w.seed);
    for (int t = threadIdx.x; t < 3 * G3; t += blockDim.x) {  // t = 3 g + axis
      const uint32_t h = hash32(hs ^ (uint32_t)t);
      ctrl[(t % 3) * G3 + t / 3] = (float)(h >> 8) * (1.0f / 8388608.0f) - 1.0f;  // exact: 24-bit value in [-1, 1)
    }
    __syncthreads();
  }
  // patch-local position -> control-grid coordinate: p (G - 1) / (P - 1), 0 on an axis with P = 1
  const float gs0 = P0 > 1 ? (float)(G - 1) / (float)(P0 - 1) : 0.f;
  const float gs1 = P1 > 1 ? (float)(G - 1) / (float)(P1 - 1) : 0.f;
  const float gs2 = P2 > 1 ? (float)(G - 1) / (float)(P2 - 1) : 0.f;
  const float gmax = (float)(G - 1);
  const float h0 = 0.5f * (float)(P0 - 1), h1 = 0.5f * (float)(P1 - 1), h2 = 0.5f * (float)(P2 - 1);
  const int n0 = cs.dims[0], n1 = cs.dims[1], n2 = cs.dims[2];
  const float m0 = (float)(n0 - 1), m1 = (float)(n1 - 1), m2 = (float)(n2 - 1);
  const int rowx = gm.x_pitch, rowy = gm.truth_size;
  const int64_t nx = (int64_t)P0 * P1 * rowx, ny = (int64_t)P0 * P1 * rowy;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < nx + ny; g += (int64_t)gridDim.x * blockDim.x) {
    const bool is_y = g >= nx;
    const int64_t q = is_y ? g - nx : g;
    const int row = is_y ? rowy : rowx;
    const int k = (int)(q % row);
    const int64_t ij = q / row;
    int j = (int)(ij % P1), i = (int)(ij / P1);
    if (flip & 1) i = P0 - 1 - i;
    if (flip & 2) j = P1 - 1 - j;
    const float* src;
    int pz;  // patch-local z of the element (q_z - corner_z)
    bool is_data = false;
    if (is_y) {
      src = cs.truth;
      pz = gm.truth_index + ((flip & 4) ? rowy - 1 - k : k);
    } else if (k < P2) {
      src = cs.data;
      pz = (flip & 4) ? P2 - 1 - k : k;
      is_data = true;
    } else {
      src = cs.truth;
      const int kk = k - P2;
      pz = gm.prev_index + ((flip & 4) ? gm.prev_size - 1 - kk : kk);
    }
    float r0 = (float)i - h0, r1 = (float)j - h1, r2 = (float)pz - h2;  // q - c
    if (G > 0) {
      const float u0 = fminf(fmaxf((float)i * gs0, 0.f), gmax);
      const float u1 = fminf(fmaxf((float)j * gs1, 0.f), gmax);
      const float u2 = fminf(fmaxf((float)pz * gs2, 0.f), gmax);
      const int g0 = min((int)u0, G - 2), g1 = min((int)u1, G - 2), g2 = min((int)u2, G - 2);
      const float f0 = u0 - (float)g0, f1 = u1 - (float)g1, f2 = u2 - (float)g2;
      const int c000 = (g0 * G + g1) * G + g2;
      float d[3];
#pragma unroll
      for (int ax = 0; ax < 3; ++ax) {
        const float* c = ctrl + ax * G3 + c000;
        const float v00 = lerpf(c[0], c[1], f2), v01 = lerpf(c[G], c[G + 1], f2);
        const float v10 = lerpf(c[G * G], c[G * G + 1], f2), v11 = lerpf(c[G * G + G], c[G * G + G + 1], f2);
        d[ax] = lerpf(lerpf(v00, v01, f1), lerpf(v10, v11, f1), f0);
      }
      r0 = fmaf(al0, d[0], r0);
      r1 = fmaf(al1, d[1], r1);
      r2 = fmaf(al2, d[2], r2);
    }
    // source position, clamped to the volume (np.pad(mode='edge') / map_coordinates(mode='nearest'))
    const float s0 = fminf(fmaxf(ct0 + fmaf(M[0], r0, fmaf(M[1], r1, M[2] * r2)), 0.f), m0);
    const float s1 = fminf(fmaxf(ct1 + fmaf(M[3], r0, fmaf(M[4], r1, M[5] * r2)), 0.f), m1);
    const float s2 = fminf(fmaxf(ct2 + fmaf(M[6], r0, fmaf(M[7], r1, M[8] * r2)), 0.f), m2);
    float v;
    if (is_data) {
      const int x0 = (int)s0, y0 = (int)s1, z0 = (int)s2;  // s >= 0: truncation is floor
      const float fx = s0 - (float)x0, fy = s1 - (float)y0, fz = s2 - (float)z0;
      const int x1 = min(x0 + 1, n0 - 1), y1 = min(y0 + 1, n1 - 1), dz = min(z0 + 1, n2 - 1) - z0;
      const float* p00 = src + ((int64_t)x0 * n1 + y0) * n2 + z0;
      const float* p01 = src + ((int64_t)x0 * n1 + y1) * n2 + z0;
      const float* p10 = src + ((int64_t)x1 * n1 + y0) * n2 + z0;
      const float* p11 = src + ((int64_t)x1 * n1 + y1) * n2 + z0;
      const float v00 = lerpf(__ldg(p00), __ldg(p00 + dz), fz), v01 = lerpf(__ldg(p01), __ldg(p01 + dz), fz);
      const float v10 = lerpf(__ldg(p10), __ldg(p10 + dz), fz), v11 = lerpf(__ldg(p11), __ldg(p11 + dz), fz);
      v = lerpf(lerpf(v00, v01, fy), lerpf(v10, v11, fy), fx) * scale;
      if (sigma > 0.f) v += sigma * gauss(seed, (uint32_t)q);
    } else {
      const int xx = min((int)floorf(s0 + 0.5f), n0 - 1), yy = min((int)floorf(s1 + 0.5f), n1 - 1);
      const int zz = min((int)floorf(s2 + 0.5f), n2 - 1);
      v = __ldg(src + ((int64_t)xx * n1 + yy) * n2 + zz);
    }
    (is_y ? y + (int64_t)b * ny : x + (int64_t)b * nx)[q] = v;
  }
}

int check_warp(const fm_sample_warp& w, int b) {
  for (int t = 0; t < 9; ++t)
    FM_CHECK(std::isfinite(w.matrix[t]), FM_EINVAL, "sampler: warp of sample %d: non-finite matrix", b);
  for (int t = 0; t < 3; ++t) {
    FM_CHECK(std::isfinite(w.offset[t]), FM_EINVAL, "sampler: warp of sample %d: non-finite offset", b);
    FM_CHECK(std::isfinite(w.elastic_alpha[t]) && w.elastic_alpha[t] >= 0.f, FM_EINVAL,
             "sampler: warp of sample %d: elastic_alpha must be finite and >= 0", b);
  }
  FM_CHECK(w.elastic_grid == 0 || (w.elastic_grid >= 2 && w.elastic_grid <= kMaxGrid), FM_EINVAL,
           "sampler: warp of sample %d: elastic_grid %d is not 0 or 2..%d", b, w.elastic_grid, kMaxGrid);
  return FM_OK;
}

int build_table(fm_volset* s) {
  if (!s->table_dirty) return FM_OK;
  std::vector<fm_volset::DevCase> host(s->cases.size());
  for (size_t i = 0; i < s->cases.size(); ++i) {
    host[i].data = s->cases[i].data;
    host[i].truth = s->cases[i].truth;
    for (int a = 0; a < 3; ++a) host[i].dims[a] = s->cases[i].dims[a];
    host[i].pad = 0;
  }
  if (!s->table) FM_CUDA(cudaMalloc((void**)&s->table, host.size() * sizeof(fm_volset::DevCase)));
  FM_CUDA(cudaMemcpy(s->table, host.data(), host.size() * sizeof(fm_volset::DevCase), cudaMemcpyHostToDevice));
  s->table_dirty = false;
  return FM_OK;
}

}  // namespace

extern "C" int fm_volset_create(fm_ctx* ctx, int n_cases, fm_volset** out) {
  FM_CHECK(ctx && out && n_cases > 0, FM_EINVAL, "fm_volset_create: bad argument");
  fm_volset* s = new fm_volset();
  s->ctx = ctx;
  s->cases.resize((size_t)n_cases);
  *out = s;
  return FM_OK;
}

extern "C" int fm_volset_destroy(fm_volset* s) {
  if (!s) return FM_OK;
  cudaSetDevice(s->ctx->device);
  cudaStreamSynchronize(s->ctx->stream);
  for (auto& c : s->cases) {
    if (c.data) cudaFree(c.data);
    if (c.truth) cudaFree(c.truth);
  }
  if (s->table) cudaFree(s->table);
  if (s->d_args) cudaFree(s->d_args);
  delete s;
  return FM_OK;
}

extern "C" int fm_volset_set_case(fm_volset* s, int index, const float* data, const float* truth, const int32_t dims[3]) {
  FM_CHECK(s && data && truth && dims && index >= 0 && index < (int)s->cases.size(), FM_EINVAL,
           "fm_volset_set_case: bad argument");
  FM_CHECK(dims[0] > 0 && dims[1] > 0 && dims[2] > 0, FM_EINVAL, "fm_volset_set_case: empty volume");
  FM_CUDA(cudaSetDevice(s->ctx->device));
  FM_CUDA(cudaStreamSynchronize(s->ctx->stream));
  fm_volset::Case& c = s->cases[(size_t)index];
  if (c.data) cudaFree(c.data);
  if (c.truth) cudaFree(c.truth);
  c.data = c.truth = nullptr;
  const size_t n = (size_t)dims[0] * dims[1] * dims[2];
  FM_CUDA(cudaMalloc((void**)&c.data, n * sizeof(float)));
  FM_CUDA(cudaMalloc((void**)&c.truth, n * sizeof(float)));
  FM_CUDA(cudaMemcpy(c.data, data, n * sizeof(float), cudaMemcpyHostToDevice));
  FM_CUDA(cudaMemcpy(c.truth, truth, n * sizeof(float), cudaMemcpyHostToDevice));
  for (int a = 0; a < 3; ++a) c.dims[a] = dims[a];
  s->table_dirty = true;
  return FM_OK;
}

// Cuts `batch` samples into x_dev [B][P0][P1][P2 + prev_size] and y_dev [B][P0][P1][truth_size] (device pointers).
int sampler_gather_device(fm_volset* s, const int32_t* cases, const int32_t* corners, const fm_sample_aug* aug,
                          const fm_sample_warp* warp, int batch, const int32_t patch[3], int truth_index,
                          int truth_size, int prev_truth_index, int prev_truth_size, float* x_dev, float* y_dev) {
  FM_CHECK(s && cases && corners && patch && batch > 0 && x_dev && y_dev, FM_EINVAL, "sampler: bad argument");
  FM_CHECK(truth_size > 0 && prev_truth_size >= 0 && patch[0] > 0 && patch[1] > 0 && patch[2] > 0, FM_EINVAL,
           "sampler: bad patch / truth extents");
  fm_ctx* ctx = s->ctx;
  FM_CUDA(cudaSetDevice(ctx->device));
  for (int b = 0; b < batch; ++b) {
    FM_CHECK(cases[b] >= 0 && cases[b] < (int)s->cases.size() && s->cases[(size_t)cases[b]].data != nullptr, FM_EINVAL,
             "sampler: case %d of sample %d is not loaded", cases[b], b);
    if (warp) FM_TRY(check_warp(warp[b], b));
  }
  FM_TRY(build_table(s));
  // per-sample arguments: inside the kernel parameters for ordinary batches (the call never waits for the previous
  // step, which is still in its backward pass when the next batch is drawn); through a pinned staging area otherwise
  SampleArgs inl;
  WarpInline winl;
  const bool inline_args = batch <= kInlineSamples;
  const size_t arg_bytes = (size_t)batch * 32, bytes = arg_bytes + (warp ? (size_t)batch * sizeof(WarpArgs) : 0);
  void* pin = nullptr;
  if (!inline_args) {
    FM_CUDA(cudaStreamSynchronize(ctx->stream));  // the previous step's copy out of the staging area has completed
    FM_TRY(fm_ctx_pinned(ctx, bytes, &pin));
  }
  int32_t* h = inline_args ? inl.v : (int32_t*)pin;
  WarpArgs* hw = inline_args ? winl.w : (WarpArgs*)((char*)pin + arg_bytes);
  for (int b = 0; b < batch; ++b) {
    h[b * 8] = cases[b];
    h[b * 8 + 1] = corners[b * 3];
    h[b * 8 + 2] = corners[b * 3 + 1];
    h[b * 8 + 3] = corners[b * 3 + 2];
    const float scale = aug ? aug[b].intensity_scale : 1.0f, sigma = aug ? aug[b].noise_sigma : 0.0f;
    h[b * 8 + 4] = aug ? (int32_t)(aug[b].flip & 7u) : 0;
    h[b * 8 + 5] = aug ? (int32_t)aug[b].noise_seed : 0;
    memcpy(&h[b * 8 + 6], &scale, 4);
    memcpy(&h[b * 8 + 7], &sigma, 4);
    if (warp) {
      const fm_sample_warp& w = warp[b];
      for (int t = 0; t < 9; ++t) hw[b].m[t] = w.matrix[t];
      for (int t = 0; t < 3; ++t) {
        hw[b].ct[t] = (float)((double)corners[b * 3 + t] + 0.5 * (patch[t] - 1) + (double)w.offset[t]);
        hw[b].alpha[t] = w.elastic_alpha[t];
      }
      hw[b].seed = w.elastic_seed;
      hw[b].grid = w.elastic_grid;
    }
  }
  if (!inline_args) {
    if (s->d_args_bytes < bytes) {
      if (s->d_args) cudaFree(s->d_args);
      s->d_args = nullptr;
      s->d_args_bytes = 0;
      FM_CUDA(cudaMalloc((void**)&s->d_args, bytes));
      s->d_args_bytes = bytes;
    }
    FM_CUDA(cudaMemcpyAsync(s->d_args, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  SampleGeom gm;
  for (int a = 0; a < 3; ++a) gm.patch[a] = patch[a];
  gm.truth_index = truth_index;
  gm.truth_size = truth_size;
  gm.prev_index = prev_truth_index;
  gm.prev_size = prev_truth_size;
  gm.x_pitch = patch[2] + prev_truth_size;
  const int64_t per = (int64_t)patch[0] * patch[1] * (gm.x_pitch + truth_size);
  if (!warp) {
    const dim3 grid((unsigned)std::min<int64_t>(ceil_div64(per, kThreadsS), 4096), (unsigned)batch);
    ProfScope prof(ctx, "sample_patches", 0.0, (double)batch * per * 8.0);
    sample_patches_kernel<<<grid, kThreadsS, 0, ctx->stream>>>(s->table, inline_args ? nullptr : s->d_args, inl, gm,
                                                               x_dev, y_dev);
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  // four elements per thread: a block expands its sample's elastic control grid once for 1024 output elements
  const dim3 grid((unsigned)std::min<int64_t>(ceil_div64(per, 4 * kThreadsS), 4096), (unsigned)batch);
  ProfScope prof(ctx, "sample_patches_warp", 0.0, (double)batch * per * 8.0);
  sample_patches_warp_kernel<<<grid, kThreadsS, 0, ctx->stream>>>(
      s->table, inline_args ? nullptr : s->d_args, inline_args ? nullptr : (const WarpArgs*)((char*)s->d_args + arg_bytes),
      inl, winl, gm, x_dev, y_dev);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

extern "C" int fm_volset_gather(fm_volset* s, const int32_t* cases, const int32_t* corners, const fm_sample_aug* aug,
                                int batch, const int32_t patch[3], int truth_index, int truth_size, int prev_truth_index,
                                int prev_truth_size, float* x_out, float* y_out) {
  return fm_volset_gather_warp(s, cases, corners, aug, nullptr, batch, patch, truth_index, truth_size, prev_truth_index,
                               prev_truth_size, x_out, y_out);
}

extern "C" int fm_volset_gather_warp(fm_volset* s, const int32_t* cases, const int32_t* corners,
                                     const fm_sample_aug* aug, const fm_sample_warp* warp, int batch,
                                     const int32_t patch[3], int truth_index, int truth_size, int prev_truth_index,
                                     int prev_truth_size, float* x_out, float* y_out) {
  FM_CHECK(s && x_out && y_out && patch && batch > 0, FM_EINVAL, "fm_volset_gather: bad argument");
  FM_CUDA(cudaSetDevice(s->ctx->device));
  const size_t nx = (size_t)batch * patch[0] * patch[1] * (patch[2] + prev_truth_size);
  const size_t ny = (size_t)batch * patch[0] * patch[1] * truth_size;
  float *dx = nullptr, *dy = nullptr;
  FM_CUDA(cudaMalloc((void**)&dx, nx * sizeof(float)));
  cudaError_t e = cudaMalloc((void**)&dy, ny * sizeof(float));
  int rc = e == cudaSuccess ? FM_OK : FM_ENOMEM;
  if (rc == FM_OK)
    rc = sampler_gather_device(s, cases, corners, aug, warp, batch, patch, truth_index, truth_size, prev_truth_index,
                               prev_truth_size, dx, dy);
  if (rc == FM_OK) {
    e = cudaMemcpyAsync(x_out, dx, nx * sizeof(float), cudaMemcpyDeviceToHost, s->ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(y_out, dy, ny * sizeof(float), cudaMemcpyDeviceToHost, s->ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->ctx->stream);
    if (e != cudaSuccess) {
      fm_set_error("fm_volset_gather: %s", cudaGetErrorString(e));
      rc = FM_ECUDA;
    }
  }
  cudaStreamSynchronize(s->ctx->stream);
  cudaFree(dx);
  if (dy) cudaFree(dy);
  return rc;
}
