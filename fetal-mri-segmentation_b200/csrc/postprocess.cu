// postprocess.cu — the reference's postprocess_prediction (fetal_net/postprocess.py:13) on the device:
// scipy.ndimage.gaussian_filter (mode 'reflect', axes 0, 1, 2), threshold, binary_fill_holes and the largest
// 6-connected component, bit-exact with scipy.
//
// Gaussian: one launch per axis, one thread per output voxel. The sum runs in scipy's correlate1d order for a symmetric
// kernel - acc = x[i] * w[0], then acc += (x[i - l] + x[i + l]) * w[l] for l = r .. 1 - in double with explicitly rounded
// operations (nvcc would otherwise contract to DFMA and change the last bit); the output of every pass is rounded to the
// input dtype, as scipy writes each axis into an array of that dtype. The last pass compares with the threshold in the
// input dtype and writes the uint8 mask instead of the field.
//
// Connected components: union-find over voxel indices. Links always go from the larger to the smaller index through
// atomicMin, so every root ends up as the smallest linear index of its component - the order in which scipy.ndimage.label
// numbers components - whatever order the atomics land in. Hole filling labels the background the same way and turns
// every background component without a border voxel into foreground; then the foreground is labelled, component sizes
// are counted with warp-aggregated atomics and one packed 64-bit atomicMax over (size, ~root) picks the largest
// component, the lowest root on a tie (np.argmax keeps the first label).
#include "common.cuh"

namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ int reflect_index(int j, int n) {
  if (j >= 0 && j < n) return j;
  const int p = 2 * n;
  int m = j % p;
  if (m < 0) m += p;
  return m < n ? m : p - 1 - m;
}

__device__ __forceinline__ float round_to(double v, float) { return __double2float_rn(v); }
__device__ __forceinline__ double round_to(double v, double) { return v; }

// One axis of the separable filter. `src` is addressed with strides (sx, sy, 1) - the first pass reads a box inside a
// larger buffer - `dst` / `mask` are compact [X][Y][Z]. `w` points at the centre weight (w[-r .. r]).
template <typename T>
__global__ void __launch_bounds__(kThreads) gauss_pass_kernel(const T* __restrict__ src, int64_t sx, int64_t sy,
                                                              T* __restrict__ dst, uint8_t* __restrict__ mask,
                                                              int X, int Y, int Z, int axis,
                                                              int r, const double* __restrict__ w, double threshold) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= (int64_t)X * Y * Z) return;
  const int z = (int)(i % Z);
  const int y = (int)((i / Z) % Y);
  const int x = (int)(i / ((int64_t)Z * Y));
  const int64_t stride = axis == 0 ? sx : (axis == 1 ? sy : 1);
  const int pos = axis == 0 ? x : (axis == 1 ? y : z);
  const int n = axis == 0 ? X : (axis == 1 ? Y : Z);
  const T* line = src + (int64_t)x * sx + (int64_t)y * sy + z - (int64_t)pos * stride;
  double acc = __dmul_rn((double)__ldg(line + (int64_t)pos * stride), __ldg(w));
  if (pos - r >= 0 && pos + r < n) {
    for (int l = r; l >= 1; --l) {
      const double s = __dadd_rn((double)__ldg(line + (int64_t)(pos - l) * stride),
                                 (double)__ldg(line + (int64_t)(pos + l) * stride));
      acc = __dadd_rn(acc, __dmul_rn(s, __ldg(w + l)));
    }
  } else {
    for (int l = r; l >= 1; --l) {
      const double s = __dadd_rn((double)__ldg(line + (int64_t)reflect_index(pos - l, n) * stride),
                                 (double)__ldg(line + (int64_t)reflect_index(pos + l, n) * stride));
      acc = __dadd_rn(acc, __dmul_rn(s, __ldg(w + l)));
    }
  }
  const T out = round_to(acc, T());
  if (mask) {
    mask[i] = out > round_to(threshold, T()) ? 1 : 0;
  } else {
    dst[i] = out;
  }
}

__device__ __forceinline__ int32_t find_root(const int32_t* labels, int32_t i) {
  int32_t p = __ldcg(labels + i);
  while (p != i) {
    i = p;
    p = __ldcg(labels + i);
  }
  return i;
}

__device__ __forceinline__ void unite(int32_t* labels, int32_t a, int32_t b) {
  while (true) {
    a = find_root(labels, a);
    b = find_root(labels, b);
    if (a == b) return;
    if (a > b) {
      const int32_t t = a;
      a = b;
      b = t;
    }
    const int32_t old = atomicMin(labels + b, a);
    if (old == b) return;
    b = old;  // b was linked meanwhile: retry from its new parent
  }
}

// Initial forest: every voxel of class `cls` points at the first voxel of its run along z (one warp per (x, y) row,
// 32 z at a time; run starts come from the ballot of the class bits).
__global__ void __launch_bounds__(kThreads) cc_runs_kernel(const uint8_t* __restrict__ mask, uint8_t cls,
                                                           int32_t* __restrict__ labels, int64_t rows, int Z) {
  const int64_t row = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;  // uniform per warp
  const int64_t base = row * Z;
  int32_t carry = -1;       // start of the run that reaches the end of the previous chunk
  for (int z0 = 0; z0 < Z; z0 += 32) {
    const bool in = z0 + lane < Z && mask[base + z0 + lane] == cls;
    const unsigned bits = __ballot_sync(0xffffffffu, in);
    const unsigned starts = bits & ~((bits << 1) | (carry >= 0 ? 1u : 0u));
    if (in) {
      const unsigned upto = starts & (0xffffffffu >> (31 - lane));
      labels[base + z0 + lane] = upto ? (int32_t)(base + z0 + 31 - __clz(upto)) : carry;
    }
    if (bits >> 31)
      carry = starts ? (int32_t)(base + z0 + 31 - __clz(starts)) : carry;
    else
      carry = -1;
  }
}

// Voxels of class `cls` join their -y and -x neighbours of the same class. A contact is skipped when the voxels below
// both (at z - 1) are of the class too: the two runs are then joined at z - 1 already (by induction down to the first z
// of the contact), so only the first voxel of every contact between two runs issues a union.
__global__ void __launch_bounds__(kThreads) cc_union_kernel(const uint8_t* __restrict__ mask, uint8_t cls,
                                                            int32_t* labels, int X, int Y, int Z) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= (int64_t)X * Y * Z || mask[i] != cls) return;
  const int z = (int)(i % Z);
  const int y = (int)((i / Z) % Y);
  const int x = (int)(i / ((int64_t)Z * Y));
  const bool below = z > 0 && mask[i - 1] == cls;
  const int64_t sy = Z, sx = (int64_t)Y * Z;
  if (y > 0 && mask[i - sy] == cls && !(below && mask[i - sy - 1] == cls)) unite(labels, (int32_t)i, (int32_t)(i - sy));
  if (x > 0 && mask[i - sx] == cls && !(below && mask[i - sx - 1] == cls)) unite(labels, (int32_t)i, (int32_t)(i - sx));
}

// labels[i] = root for voxels of class `cls`; with `sizes`, each root also receives its voxel count
__global__ void __launch_bounds__(kThreads) cc_flatten_kernel(const uint8_t* __restrict__ mask, uint8_t cls,
                                                              int32_t* labels, int32_t* sizes, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  int32_t root = -1;
  if (i < n && mask[i] == cls) {
    root = find_root(labels, (int32_t)i);
    labels[i] = root;
  }
  if (sizes) {
    // one atomic per distinct root in the warp: a component can hold millions of voxels
    const unsigned peers = __match_any_sync(0xffffffffu, root);
    if (root >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(sizes + root, __popc(peers));
  }
}

// marks[root] = 1 for background components that reach the array border
__global__ void __launch_bounds__(kThreads) fill_mark_kernel(const uint8_t* __restrict__ mask,
                                                             const int32_t* __restrict__ labels, int32_t* marks, int X,
                                                             int Y, int Z) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= (int64_t)X * Y * Z || mask[i] != 0) return;
  const int z = (int)(i % Z);
  const int y = (int)((i / Z) % Y);
  const int x = (int)(i / ((int64_t)Z * Y));
  if (x == 0 || y == 0 || z == 0 || x == X - 1 || y == Y - 1 || z == Z - 1) marks[labels[i]] = 1;
}

// enclosed background becomes foreground
__global__ void __launch_bounds__(kThreads) fill_apply_kernel(uint8_t* mask, const int32_t* __restrict__ labels,
                                                              const int32_t* __restrict__ marks, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i < n && mask[i] == 0 && marks[labels[i]] == 0) mask[i] = 1;
}

// stats[0] += number of foreground roots, stats[1] = max over roots of (size << 32 | ~root)
__global__ void __launch_bounds__(kThreads) cc_select_kernel(const uint8_t* __restrict__ mask,
                                                             const int32_t* __restrict__ labels,
                                                             const int32_t* __restrict__ sizes,
                                                             unsigned long long* stats, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const bool root = i < n && mask[i] && labels[i] == (int32_t)i;
  unsigned long long key = root ? ((unsigned long long)(uint32_t)sizes[i] << 32) | (uint32_t)~(uint32_t)i : 0ull;
  const unsigned roots = __ballot_sync(0xffffffffu, root);
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
    key = other > key ? other : key;
  }
  if ((threadIdx.x & 31) == 0 && roots) {
    atomicAdd(stats, (unsigned long long)__popc(roots));
    atomicMax(stats + 1, key);
  }
}

__global__ void __launch_bounds__(kThreads) cc_keep_kernel(uint8_t* mask, const int32_t* __restrict__ labels,
                                                           const unsigned long long* __restrict__ stats, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= n || !mask[i]) return;
  const int32_t keep = (int32_t)~(uint32_t)(stats[1] & 0xffffffffull);
  mask[i] = labels[i] == keep ? 1 : 0;
}

inline unsigned grid_of(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

int pp_buffers(fm_ctx* ctx, int64_t nvox, int radius, PostprocBuffers* b) {
  FM_CHECK(nvox > 0 && nvox <= INT32_MAX, FM_EINVAL, "post-processing: %lld voxels (1 .. 2^31 - 1 supported)",
           (long long)nvox);
  FM_CHECK(radius >= 0 && radius <= (1 << 20), FM_EINVAL, "post-processing: filter radius %d", radius);
  const size_t field = align256((size_t)nvox * sizeof(double)), lab = align256((size_t)nvox * sizeof(int32_t));
  const size_t msk = align256((size_t)nvox), wts = align256((size_t)(2 * radius + 1) * sizeof(double));
  const size_t total = 2 * field + 2 * lab + msk + wts + 256;
  if (ctx->pp_ws_bytes < total) {
    if (ctx->pp_ws) cudaFree(ctx->pp_ws);
    ctx->pp_ws = nullptr;
    ctx->pp_ws_bytes = 0;
    cudaError_t e = cudaMalloc(&ctx->pp_ws, total);
    if (e != cudaSuccess) {
      fm_set_error("post-processing workspace: cudaMalloc(%zu bytes) failed: %s", total, cudaGetErrorString(e));
      return FM_ENOMEM;
    }
    ctx->pp_ws_bytes = total;
  }
  char* p = (char*)ctx->pp_ws;
  b->field0 = p;
  b->field1 = p + field;
  b->labels = (int32_t*)(p + 2 * field);
  b->aux = (int32_t*)(p + 2 * field + lab);
  b->mask = (uint8_t*)(p + 2 * field + 2 * lab);
  b->weights = (double*)(p + 2 * field + 2 * lab + msk);
  b->stats = (unsigned long long*)(p + 2 * field + 2 * lab + msk + wts);
  return FM_OK;
}

// The three axis passes: src (strides sx, sy, 1) -> field0 -> field1 -> out_field, or -> mask when out_field is null.
// src may be field1 (it is consumed by the first pass).
static int gaussian_passes(fm_ctx* ctx, const PostprocBuffers& b, const void* src, int dtype, int64_t sx, int64_t sy,
                           const int32_t dims[3], int radius, const double* weights_host, void* out_field,
                           double threshold) {
  const int X = dims[0], Y = dims[1], Z = dims[2];
  const int64_t n = (int64_t)X * Y * Z;
  const size_t es = dtype == 1 ? sizeof(double) : sizeof(float);
  FM_CUDA(cudaMemcpyAsync(b.weights, weights_host, (size_t)(2 * radius + 1) * sizeof(double), cudaMemcpyHostToDevice,
                          ctx->stream));
  const double* wc = b.weights + radius;
  static const char* names[3] = {"gaussian_x", "gaussian_y", "gaussian_z_threshold"};
  for (int axis = 0; axis < 3; ++axis) {
    const void* in = axis == 0 ? src : (axis == 1 ? b.field0 : b.field1);
    const int64_t isx = axis == 0 ? sx : (int64_t)Y * Z, isy = axis == 0 ? sy : Z;
    void* dst = axis == 0 ? b.field0 : (axis == 1 ? b.field1 : out_field);
    uint8_t* mask = axis == 2 && !out_field ? b.mask : nullptr;
    // algorithmic bytes: the line is read once and the result written once (the 2r neighbours come from L1 / L2)
    const double bytes = (double)n * (es + (mask ? 1 : es));
    ProfScope ps(ctx, axis == 2 && !mask ? "gaussian_z" : names[axis], (double)n * (3 * radius + 1), bytes);
    if (dtype == 1)
      gauss_pass_kernel<double><<<grid_of(n), kThreads, 0, ctx->stream>>>(
          (const double*)in, isx, isy, (double*)dst, mask, X, Y, Z, axis, radius, wc, threshold);
    else
      gauss_pass_kernel<float><<<grid_of(n), kThreads, 0, ctx->stream>>>(
          (const float*)in, isx, isy, (float*)dst, mask, X, Y, Z, axis, radius, wc, threshold);
    FM_LAUNCH_OK(ctx);
  }
  return FM_OK;
}

int k_gaussian3d(fm_ctx* ctx, const PostprocBuffers& b, const void* src, int dtype, int64_t sx, int64_t sy,
                 const int32_t dims[3], int radius, const double* weights_host, void* out_field) {
  return gaussian_passes(ctx, b, src, dtype, sx, sy, dims, radius, weights_host, out_field, 0.0);
}

// labels of the voxels of class `cls`: z-run forest, unions across runs, flatten (+ component sizes)
static int label_class(fm_ctx* ctx, const PostprocBuffers& b, uint8_t cls, const int32_t dims[3], int32_t* sizes) {
  const int64_t n = (int64_t)dims[0] * dims[1] * dims[2];
  {
    ProfScope ps(ctx, cls ? "cc_runs_fg" : "cc_runs_bg", 0.0, (double)n * (1 + 4));
    cc_runs_kernel<<<grid_of((int64_t)dims[0] * dims[1] * 32), kThreads, 0, ctx->stream>>>(
        b.mask, cls, b.labels, (int64_t)dims[0] * dims[1], dims[2]);
    FM_LAUNCH_OK(ctx);
  }
  {
    ProfScope ps(ctx, cls ? "cc_union_fg" : "cc_union_bg", 0.0, (double)n * (1 + 4));
    cc_union_kernel<<<grid_of(n), kThreads, 0, ctx->stream>>>(b.mask, cls, b.labels, dims[0], dims[1], dims[2]);
    FM_LAUNCH_OK(ctx);
  }
  {
    ProfScope ps(ctx, sizes ? "cc_flatten_count_fg" : "cc_flatten_bg", 0.0, (double)n * (1 + 4 + 4));
    cc_flatten_kernel<<<grid_of(n), kThreads, 0, ctx->stream>>>(b.mask, cls, b.labels, sizes, n);
    FM_LAUNCH_OK(ctx);
  }
  return FM_OK;
}

int k_postprocess(fm_ctx* ctx, const PostprocBuffers& b, const void* src, int dtype, int64_t sx, int64_t sy,
                  const int32_t dims[3], const fm_postprocess_spec* spec) {
  const int64_t n = (int64_t)dims[0] * dims[1] * dims[2];
  const bool fill = spec->fill_holes != 0, cc = spec->connected_component != 0;
  FM_CUDA(cudaMemsetAsync(b.stats, 0, 2 * sizeof(unsigned long long), ctx->stream));
  FM_TRY(gaussian_passes(ctx, b, src, dtype, sx, sy, dims, spec->radius, spec->weights, nullptr, spec->threshold));
  if (fill) {
    FM_TRY(label_class(ctx, b, 0, dims, nullptr));
    FM_CUDA(cudaMemsetAsync(b.aux, 0, (size_t)n * sizeof(int32_t), ctx->stream));
    {
      ProfScope ps(ctx, "fill_mark", 0.0, (double)n * (1 + 4));
      fill_mark_kernel<<<grid_of(n), kThreads, 0, ctx->stream>>>(b.mask, b.labels, b.aux, dims[0], dims[1], dims[2]);
      FM_LAUNCH_OK(ctx);
    }
    {
      ProfScope ps(ctx, "fill_apply", 0.0, (double)n * (1 + 4 + 4 + 1));
      fill_apply_kernel<<<grid_of(n), kThreads, 0, ctx->stream>>>(b.mask, b.labels, b.aux, n);
      FM_LAUNCH_OK(ctx);
    }
  }
  if (cc) {
    FM_CUDA(cudaMemsetAsync(b.aux, 0, (size_t)n * sizeof(int32_t), ctx->stream));
    FM_TRY(label_class(ctx, b, 1, dims, b.aux));
    {
      ProfScope ps(ctx, "cc_select", 0.0, (double)n * (1 + 4 + 4));
      cc_select_kernel<<<grid_of(n), kThreads, 0, ctx->stream>>>(b.mask, b.labels, b.aux, b.stats, n);
      FM_LAUNCH_OK(ctx);
    }
    {
      ProfScope ps(ctx, "cc_keep", 0.0, (double)n * (1 + 4 + 1));
      cc_keep_kernel<<<grid_of(n), kThreads, 0, ctx->stream>>>(b.mask, b.labels, b.stats, n);
      FM_LAUNCH_OK(ctx);
    }
  }
  return FM_OK;
}
