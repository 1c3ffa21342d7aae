// tta.cu — flip test-time augmentation of the sliding window (the reference's predict_flips, fetal_net/prediction.py:65-85,
// and the per-voxel median its callers take, predict_nifti2.py:86-87): the per-pass flip of the input volume, the
// un-flip of each pass's cropped map into a stack [passes][X][Y][Z], and the median over the stack. All three are pure
// data movement or comparisons plus one explicitly rounded add and halving, so the results are bit-exact with NumPy.
// Flip masks: bit a set = axis a (x, y, z) reversed.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;

struct FlipGeom {
  int X, Y, Z;
  int fx, fy, fz;
};

__device__ __forceinline__ void flip_coords(const FlipGeom& g, int64_t i, int* x, int* y, int* z) {
  const int zz = (int)(i % g.Z);
  const int64_t r = i / g.Z;
  const int yy = (int)(r % g.Y);
  const int xx = (int)(r / g.Y);
  *x = g.fx ? g.X - 1 - xx : xx;
  *y = g.fy ? g.Y - 1 - yy : yy;
  *z = g.fz ? g.Z - 1 - zz : zz;
}

// out[x][y][z] = in[flipped x][flipped y][flipped z] over the [X][Y][Z] volume
__global__ void __launch_bounds__(kThreads) flip_volume_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                               FlipGeom g) {
  const int64_t n = (int64_t)g.X * g.Y * g.Z;
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    int x, y, z;
    flip_coords(g, i, &x, &y, &z);
    out[i] = __ldg(in + ((int64_t)x * g.Y + y) * g.Z + z);
  }
}

// out[x][y][z] = map[f0 + flipped x][f1 + flipped y][f2 + flipped z]: the pad_for_fit crop of the padded [MX][MY][MZ]
// map, un-flipped
__global__ void __launch_bounds__(kThreads) flip_crop_kernel(const double* __restrict__ map, int MY, int MZ, int f0,
                                                             int f1, int f2, double* __restrict__ out, FlipGeom g) {
  const int64_t n = (int64_t)g.X * g.Y * g.Z;
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    int x, y, z;
    flip_coords(g, i, &x, &y, &z);
    out[i] = __ldg(map + ((int64_t)(f0 + x) * MY + (f1 + y)) * MZ + (f2 + z));
  }
}

// np.median of P values: NaN if any value is NaN, else the middle of the sorted values, or for even P
// (s[P/2-1] + s[P/2]) / 2 — the mean numpy takes of the two partitioned middle elements (x 0.5 is the exact halving;
// the explicit roundings keep nvcc from fusing anything). Signed zeros compare equal in both sorts, so an odd-P median
// whose middle run mixes -0.0 and +0.0 may differ from NumPy in the sign of that zero.
template <int P>
__device__ __forceinline__ double median_of(double v[P]) {
  bool nan = false;
#pragma unroll
  for (int i = 0; i < P; ++i) nan = nan || v[i] != v[i];
  // odd-even transposition sort: P rounds of compare-exchange put P values in order
#pragma unroll
  for (int r = 0; r < P; ++r)
#pragma unroll
    for (int i = r & 1; i + 1 < P; i += 2) {
      const double lo = fmin(v[i], v[i + 1]), hi = fmax(v[i], v[i + 1]);
      v[i] = lo;
      v[i + 1] = hi;
    }
  const double med = (P & 1) ? v[P / 2] : __dmul_rn(__dadd_rn(v[P / 2 - 1], v[P / 2]), 0.5);
  return nan ? __longlong_as_double(0x7ff8000000000000ll) : med;
}

// out[i] = median over k of stack[k * pitch + i]. Four consecutive voxels per thread, two 16-byte loads per pass
// (pitch % 4 == 0 and a 32-byte aligned stack make every quad aligned); the last partial quad goes voxel by voxel.
template <int P>
__global__ void __launch_bounds__(kThreads) median_passes_kernel(const double* __restrict__ stack, int64_t pitch,
                                                                 int64_t nvox, double* __restrict__ out) {
  const int64_t nq = (nvox + 3) / 4;
  for (int64_t q = (int64_t)blockIdx.x * kThreads + threadIdx.x; q < nq; q += (int64_t)gridDim.x * kThreads) {
    const int64_t i = q * 4;
    if (i + 4 <= nvox) {
      double v[4][P];
#pragma unroll
      for (int k = 0; k < P; ++k) {
        const double2 a = __ldcs(reinterpret_cast<const double2*>(stack + k * pitch + i));
        const double2 b = __ldcs(reinterpret_cast<const double2*>(stack + k * pitch + i) + 1);
        v[0][k] = a.x;
        v[1][k] = a.y;
        v[2][k] = b.x;
        v[3][k] = b.y;
      }
      double r[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) r[e] = median_of<P>(v[e]);
      reinterpret_cast<double2*>(out + i)[0] = make_double2(r[0], r[1]);
      reinterpret_cast<double2*>(out + i)[1] = make_double2(r[2], r[3]);
    } else {
      for (int64_t j = i; j < nvox; ++j) {
        double v[P];
#pragma unroll
        for (int k = 0; k < P; ++k) v[k] = stack[k * pitch + j];
        out[j] = median_of<P>(v);
      }
    }
  }
}

inline unsigned grid_cap(int64_t work) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>((work + kThreads - 1) / kThreads, 148 * 32));
}

inline FlipGeom flip_geom(const int32_t dims[3], int mask) {
  return FlipGeom{dims[0], dims[1], dims[2], mask & 1, (mask >> 1) & 1, (mask >> 2) & 1};
}

}  // namespace

int k_flip_volume(fm_ctx* ctx, const float* in, float* out, const int32_t dims[3], int mask) {
  const int64_t n = (int64_t)dims[0] * dims[1] * dims[2];
  ProfScope prof(ctx, "flip_volume", 0.0, (double)n * 8.0);
  flip_volume_kernel<<<grid_cap(n), kThreads, 0, ctx->stream>>>(in, out, flip_geom(dims, mask));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_flip_crop(fm_ctx* ctx, const double* map, const int32_t map_dims[3], const int32_t fit_lo[3], double* out,
                const int32_t dims[3], int mask) {
  const int64_t n = (int64_t)dims[0] * dims[1] * dims[2];
  ProfScope prof(ctx, "flip_crop", 0.0, (double)n * 16.0);
  flip_crop_kernel<<<grid_cap(n), kThreads, 0, ctx->stream>>>(map, map_dims[1], map_dims[2], fit_lo[0], fit_lo[1],
                                                               fit_lo[2], out, flip_geom(dims, mask));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_median_passes(fm_ctx* ctx, const double* stack, int64_t pitch, int passes, int64_t nvox, double* out) {
  FM_CHECK(passes >= 1 && passes <= 8 && pitch % 4 == 0 && pitch >= nvox && ((uintptr_t)stack & 31) == 0 &&
               ((uintptr_t)out & 31) == 0,
           FM_EINVAL, "median_passes: %d passes, pitch %lld", passes, (long long)pitch);
  ProfScope prof(ctx, "median_passes", 0.0, (double)nvox * 8.0 * (passes + 1));
  const unsigned grid = grid_cap((nvox + 3) / 4);
  switch (passes) {
#define FM_MEDIAN_CASE(P)                                                                           \
  case P:                                                                                           \
    median_passes_kernel<P><<<grid, kThreads, 0, ctx->stream>>>(stack, pitch, nvox, out);          \
    break;
    FM_MEDIAN_CASE(1) FM_MEDIAN_CASE(2) FM_MEDIAN_CASE(3) FM_MEDIAN_CASE(4)
    FM_MEDIAN_CASE(5) FM_MEDIAN_CASE(6) FM_MEDIAN_CASE(7) FM_MEDIAN_CASE(8)
#undef FM_MEDIAN_CASE
  }
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
