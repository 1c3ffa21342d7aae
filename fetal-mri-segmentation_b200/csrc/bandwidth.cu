// bandwidth.cu — HBM-bound kernels of the hot path: MaxPooling3D / UpSampling3D forward+backward,
// soft-Dice statistics and backward, Keras-Adam, patch gather and overlap-add reassembly.
// Device layout everywhere: channels-last [N][X][Y][Z][C] (C contiguous), bf16 activations.
// All kernels move 16-byte vectors per thread along the contiguous (C, then Z) direction.
#include "common.cuh"

#include <algorithm>

namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ uint4 ldg16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void stg16(void* p, uint4 v) { *reinterpret_cast<uint4*>(p) = v; }

__device__ __forceinline__ void unpack8(uint4 v, float f[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float f[8]) {
  uint4 v;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return v;
}

// ---------------------------------------------------------------------------------------------
// casts
// ---------------------------------------------------------------------------------------------
__global__ void cast_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, int64_t n) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i + 8 <= n) {
    float4 a = __ldg(reinterpret_cast<const float4*>(in + i));
    float4 b = __ldg(reinterpret_cast<const float4*>(in + i + 4));
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    stg16(out + i, pack8(f));
  } else {
    for (; i < n; ++i) out[i] = __float2bfloat16(in[i]);
  }
}
__global__ void cast_bf16_f32_kernel(const bf16* __restrict__ in, float* __restrict__ out, int64_t n) {
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i + 8 <= n) {
    float f[8];
    unpack8(ldg16(in + i), f);
    *reinterpret_cast<float4*>(out + i) = make_float4(f[0], f[1], f[2], f[3]);
    *reinterpret_cast<float4*>(out + i + 4) = make_float4(f[4], f[5], f[6], f[7]);
  } else {
    for (; i < n; ++i) out[i] = __bfloat162float(in[i]);
  }
}

// fp32 [vox][Cin] -> bf16 [vox][Cpad] with zero channel padding (2.5D U-Net input: slices-as-channels)
__global__ void pad_cast_kernel(const float* __restrict__ in, bf16* __restrict__ out, int64_t vox, int Cin, int Cpad) {
  const int64_t total = vox * Cpad;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(g % Cpad);
    const int64_t v = g / Cpad;
    out[g] = __float2bfloat16(c < Cin ? __ldg(in + v * Cin + c) : 0.f);
  }
}

// ---------------------------------------------------------------------------------------------
// MaxPooling3D((2,2,2)) — Keras call site fetal_net/model/unet3d/unet.py:51 (valid, stride 2)
// one thread = one pooled voxel x 8 channels (16 B); the two z-children of a window are adjacent
// in memory so every warp-level request is a run of full 32 B sectors.
// ---------------------------------------------------------------------------------------------
template <int pz>
__global__ void maxpool3d_fwd_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, int N, int X,
                                     int Y, int Z, int C) {
  FM_PDL_SYNC();
  const int c8n = C >> 3;
  const int Xo = X >> 1, Yo = Y >> 1, Zo = Z / pz;
  const int64_t total = (int64_t)N * Xo * Yo * Zo * c8n;
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int c8 = (int)(g % c8n);
  int64_t v = g / c8n;
  const int zo = (int)(v % Zo);
  v /= Zo;
  const int yo = (int)(v % Yo);
  v /= Yo;
  const int xo = (int)(v % Xo);
  const int n = (int)(v / Xo);
  __nv_bfloat162 m[4];
  bool first = true;
#pragma unroll
  for (int dx = 0; dx < 2; ++dx)
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dz = 0; dz < 2; ++dz) {
        if (dz >= pz) continue;
        const int64_t vi = (((int64_t)n * X + 2 * xo + dx) * Y + 2 * yo + dy) * Z + pz * zo + dz;
        uint4 t = ldg16(x + vi * C + c8 * 8);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
        if (first) {
#pragma unroll
          for (int i = 0; i < 4; ++i) m[i] = h[i];
          first = false;
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) m[i] = __hmax2(m[i], h[i]);
        }
      }
  uint4 o;
  __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
  for (int i = 0; i < 4; ++i) oh[i] = m[i];
  const int64_t vo = (((int64_t)n * Xo + xo) * Yo + yo) * Zo + zo;
  stg16(y + vo * C + c8 * 8, o);
}

// Backward of MaxPooling3D fused with the skip-connection gradient add and the ReLU mask of the
// producing conv block: dx = [x>0] * (dskip + [x is the first max of its window] * dy).
// TWO threads per (pooled voxel, 8 channels): lane pair (l, l^1) = the x-halves ddx = 0 / 1 of the window. Each loads
// its four children of x and dskip plus dy (9 x 16 B in flight per thread, all issued before the first use), finds its
// local first maximum and swaps it with the partner by shuffle; the ddx = 0 half wins ties (= first maximum in the
// window's k order). ~60 registers -> 4 resident blocks per SM instead of 2: the kernel is latency-bound on its loads.
template <int pz>
__global__ void __launch_bounds__(kThreads, 4) maxpool3d_bwd_kernel(const bf16* __restrict__ x,
                                                                    const bf16* __restrict__ dy,
                                     const bf16* __restrict__ dskip, bf16* __restrict__ dx, int N,
                                     int X, int Y, int Z, int C, int relu_mask) {
  FM_PDL_SYNC();
  const int c8n = C >> 3;
  const int Xo = X >> 1, Yo = Y >> 1, Zo = Z / pz;
  const int64_t total = (int64_t)N * Xo * Yo * Zo * c8n * 2;
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = g < total;  // (total is even and blockDim is even: a lane pair is live or dead together)
  if (!live) g = total - 2 + (threadIdx.x & 1);
  const int half = (int)(g & 1);
  int64_t v = g >> 1;
  const int c8 = (int)(v % c8n);
  v /= c8n;
  const int zo = (int)(v % Zo);
  v /= Zo;
  const int yo = (int)(v % Yo);
  v /= Yo;
  const int xo = (int)(v % Xo);
  const int n = (int)(v / Xo);
  // element offset of child j (= ddy * 2 + ddz) of this half: base + (ddy * Z + ddz) * C
  const int64_t base = ((((int64_t)n * X + 2 * xo + half) * Y + 2 * yo) * Z + pz * zo) * C + c8 * 8;
  const int sy = Z * C;
#define FM_CHILD_OFS(j) (base + (((j) >> 1) * sy + ((j) & 1) * C))
  uint4 xr[4], sk[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if ((j & 1) < pz) {
      xr[j] = ldg16(x + FM_CHILD_OFS(j));
      sk[j] = dskip != nullptr ? ldg16(dskip + FM_CHILD_OFS(j)) : make_uint4(0u, 0u, 0u, 0u);
    }
  }
  const int64_t vo = (((int64_t)n * Xo + xo) * Yo + yo) * Zo + zo;
  float g8[8];
  unpack8(ldg16(dy + vo * C + c8 * 8), g8);
  float best[8];
  int arg[8];
  unpack8(xr[0], best);
#pragma unroll
  for (int c = 0; c < 8; ++c) arg[c] = 0;
#pragma unroll
  for (int j = 1; j < 4; ++j) {
    if ((j & 1) >= pz) continue;  // pz == 1: the z-child does not exist
    float t[8];
    unpack8(xr[j], t);
#pragma unroll
    for (int c = 0; c < 8; ++c)
      if (t[c] > best[c]) {  // strict: the FIRST maximum keeps the gradient
        best[c] = t[c];
        arg[c] = j;
      }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const float other = __shfl_xor_sync(0xffffffffu, best[c], 1);
    const bool mine = half == 0 ? best[c] >= other : best[c] > other;
    if (!mine) arg[c] = -1;
  }
  if (!live) return;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if ((j & 1) >= pz) continue;
    float o[8], t[8];
    unpack8(sk[j], o);
    unpack8(xr[j], t);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (arg[c] == j) o[c] += g8[c];
      if (relu_mask && !(t[c] > 0.f)) o[c] = 0.f;
    }
    stg16(dx + FM_CHILD_OFS(j), pack8(o));
  }
#undef FM_CHILD_OFS
}

// ---------------------------------------------------------------------------------------------
// UpSampling3D((2,2,2)) nearest — Keras call site fetal_net/model/unet3d/unet.py:138
// ---------------------------------------------------------------------------------------------
template <int pz>
__global__ void upsample3d_fwd_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, int N, int X,
                                      int Y, int Z, int C) {
  FM_PDL_SYNC();
  const int c8n = C >> 3;
  const int64_t total = (int64_t)N * X * Y * Z * c8n;
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int c8 = (int)(g % c8n);
  int64_t v = g / c8n;
  const int z = (int)(v % Z);
  int64_t r = v / Z;
  const int yy = (int)(r % Y);
  r /= Y;
  const int xx = (int)(r % X);
  const int n = (int)(r / X);
  const uint4 t = ldg16(x + v * C + c8 * 8);
  const int X2 = 2 * X, Y2 = 2 * Y, Z2 = pz * Z;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int ddx = k >> 2, ddy = (k >> 1) & 1, ddz = k & 1;
    if (ddz >= pz) continue;
    const int64_t vo = (((int64_t)n * X2 + 2 * xx + ddx) * Y2 + 2 * yy + ddy) * Z2 + pz * z + ddz;
    stg16(y + vo * C + c8 * 8, t);
  }
}

// backward: 2^3 sum-pool of dy (fp32 accumulate), optionally masked by ReLU of the coarse activation
template <int pz>
__global__ void upsample3d_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ act,
                                      bf16* __restrict__ dx, int N, int X, int Y, int Z, int C,
                                      int dyC, int dy_cofs) {
  FM_PDL_SYNC();
  const int c8n = C >> 3;
  const int64_t total = (int64_t)N * X * Y * Z * c8n;
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int c8 = (int)(g % c8n);
  int64_t v = g / c8n;
  const int z = (int)(v % Z);
  int64_t r = v / Z;
  const int yy = (int)(r % Y);
  r /= Y;
  const int xx = (int)(r % X);
  const int n = (int)(r / X);
  const int X2 = 2 * X, Y2 = 2 * Y, Z2 = pz * Z;
  float acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int ddx = k >> 2, ddy = (k >> 1) & 1, ddz = k & 1;
    if (ddz >= pz) continue;
    const int64_t vo = (((int64_t)n * X2 + 2 * xx + ddx) * Y2 + 2 * yy + ddy) * Z2 + pz * z + ddz;
    float f[8];
    unpack8(ldg16(dy + vo * dyC + dy_cofs + c8 * 8), f);
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] += f[c];
  }
  if (act != nullptr) {
    float a[8];
    unpack8(ldg16(act + v * C + c8 * 8), a);
#pragma unroll
    for (int c = 0; c < 8; ++c)
      if (!(a[c] > 0.f)) acc[c] = 0.f;
  }
  stg16(dx + v * C + c8 * 8, pack8(acc));
}


// Block fold of per-thread (a[8], b[8]) partials over the threads that share a channel group (tid % c8n), c8n a power
// of two <= 64: xor-shuffles inside a warp, one shared-memory hop across warps, fixed order -> deterministic.
// Returns true in the c8n threads (tid < c8n) that hold the block totals of channel group `tid`.
__device__ __forceinline__ bool fold_channel_groups(float a[8], float b[8], float* sh, int c8n) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (c8n < 32) {
    for (int o = c8n; o < 32; o <<= 1)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        a[i] += __shfl_xor_sync(0xffffffffu, a[i], o);
        b[i] += __shfl_xor_sync(0xffffffffu, b[i], o);
      }
    if (lane < c8n)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        sh[(warp * c8n + lane) * 16 + i] = a[i];
        sh[(warp * c8n + lane) * 16 + 8 + i] = b[i];
      }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sh[threadIdx.x * 16 + i] = a[i];
      sh[threadIdx.x * 16 + 8 + i] = b[i];
    }
  }
  __syncthreads();
  if ((int)threadIdx.x >= c8n) return false;
  const int groups = c8n < 32 ? kThreads / 32 : kThreads / c8n;  // rows of sh holding this channel group
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = b[i] = 0.f;
  for (int k = 0; k < groups; ++k)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      a[i] += sh[(k * c8n + threadIdx.x) * 16 + i];
      b[i] += sh[(k * c8n + threadIdx.x) * 16 + 8 + i];
    }
  return true;
}

// ---------------------------------------------------------------------------------------------
// InstanceNormalization(axis=1) + LeakyReLU(0.3) — keras_contrib layer used by every Isensee conv block
// (fetal_net/model/unet3d/isensee2017.py:12, unet3d/unet.py:107-111): per (sample, channel) mean / biased
// variance over the voxels, y = (x - mean) / (sqrt(var) + 1e-3) * gamma + beta   (eps added to the STD).
// Deterministic two-stage reduction: per-block partial (sum, sum of squares) in fp32 over <= 4096 voxels,
// combined in fp64 in a fixed order; then one fused normalise + LeakyReLU (+ residual add) pass.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) instnorm_partial_kernel(const bf16* __restrict__ x, float* __restrict__ part,
                                                                    int64_t vox_per_sample, int C, int64_t vox_per_block,
                                                                    int blocks_per_sample) {
  extern __shared__ float sh[];  // [kThreads][16]
  const int c8n = C >> 3;
  const int lanes = kThreads / c8n;
  const int c8 = threadIdx.x % c8n, l = threadIdx.x / c8n;
  const int n = blockIdx.y, blk = blockIdx.x;
  const int64_t v0 = (int64_t)blk * vox_per_block;
  const int64_t v1 = min(vox_per_sample, v0 + vox_per_block);
  const bf16* xs = x + (int64_t)n * vox_per_sample * C;
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  if (l < lanes) {
    // four independent 16-byte loads in flight per thread (the pass is latency-bound otherwise: one load per trip)
    int64_t v = v0 + l;
    for (; v + 3 * (int64_t)lanes < v1; v += 4 * (int64_t)lanes) {
      uint4 r[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) r[u] = ldg16(xs + (v + u * (int64_t)lanes) * C + c8 * 8);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float f[8];
        unpack8(r[u], f);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          s[i] += f[i];
          q[i] += f[i] * f[i];
        }
      }
    }
    for (; v < v1; v += lanes) {
      float f[8];
      unpack8(ldg16(xs + v * C + c8 * 8), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s[i] += f[i];
        q[i] += f[i] * f[i];
      }
    }
  }
  if (fold_channel_groups(s, q, sh, c8n)) {
    float* o = part + (((int64_t)n * blocks_per_sample + blk) * C + threadIdx.x * 8) * 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      o[2 * i] = s[i];
      o[2 * i + 1] = q[i];
    }
  }
}

// coefficients per (n, c), ss[4 (n C + c) ...] = (scale, mean, beta, 0) with scale = gamma / (sqrt(var) + eps): the
// apply pass forms y = (x - mean) * scale + beta. (A folded shift beta - mean * scale would leave y with an fp32 error
// of ~|mean| * scale * 2^-24, which exceeds a bf16 ulp of y where the std is small against the mean.)
// One warp per (n, c): lane l folds partials l, l+32, ... in fp64, then a fixed-order butterfly (deterministic).
__global__ void instnorm_final_kernel(const float* __restrict__ part, const float* __restrict__ gamma,
                                      const float* __restrict__ beta, float* __restrict__ ss,
                                      float* __restrict__ stats, int N, int C, int blocks_per_sample,
                                      double inv_count, float eps) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= N * C) return;
  const int n = i / C, c = i % C;
  double s = 0.0, q = 0.0;
  for (int b = lane; b < blocks_per_sample; b += 32) {
    const float2 o = *reinterpret_cast<const float2*>(part + (((int64_t)n * blocks_per_sample + b) * C + c) * 2);
    s += (double)o.x;
    q += (double)o.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  if (lane != 0) return;
  const double mean = s * inv_count;
  const double var = fmax(q * inv_count - mean * mean, 0.0);
  const double scale = (double)gamma[c] / (sqrt(var) + (double)eps);
  ss[4 * i] = (float)scale;
  ss[4 * i + 1] = (float)mean;
  ss[4 * i + 2] = beta[c];
  ss[4 * i + 3] = 0.f;
  if (stats != nullptr) {  // kept for the backward pass: (mean, 1 / (sqrt(var) + eps))
    stats[2 * i] = (float)mean;
    stats[2 * i + 1] = (float)(1.0 / (sqrt(var) + (double)eps));
  }
}

// grid (blocks per sample, N): a thread keeps its 8 channels' (scale, shift[, dropout scale]) in registers and walks
// the voxels of its block
__global__ void __launch_bounds__(kThreads) instnorm_apply_kernel(const bf16* __restrict__ x, const float* __restrict__ ss,
                                                                  const bf16* __restrict__ add,
                                                                  const float* __restrict__ chan_scale,
                                                                  bf16* __restrict__ y, int64_t vox_per_sample, int C,
                                                                  int64_t vox_per_block, float slope) {
  const int c8n = C >> 3;
  const int lanes = kThreads / c8n;
  const int c8 = threadIdx.x % c8n, l = threadIdx.x / c8n;
  if (l >= lanes) return;
  const int n = blockIdx.y;
  float sc[8], mu[8], be[8], cs[8];
  const float4* sp = reinterpret_cast<const float4*>(ss + ((int64_t)n * C + c8 * 8) * 4);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 t = __ldg(sp + i);  // (scale, mean, beta, 0) of one channel
    sc[i] = t.x, mu[i] = t.y, be[i] = t.z;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) cs[i] = chan_scale ? __ldg(chan_scale + (int64_t)n * C + c8 * 8 + i) : 1.f;
  const int64_t v0 = (int64_t)n * vox_per_sample + (int64_t)blockIdx.x * vox_per_block;
  const int64_t v1 = min((int64_t)(n + 1) * vox_per_sample, v0 + vox_per_block);
  // a block covers 4 voxels per thread (norm_apply_blocks): all loads of the thread are issued before the first use
  uint4 rx[4], ra[4];
  int64_t vv[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    vv[u] = v0 + l + u * (int64_t)lanes;
    if (vv[u] < v1) {
      rx[u] = ldg16(x + vv[u] * C + c8 * 8);
      if (add != nullptr) ra[u] = ldg16(add + vv[u] * C + c8 * 8);
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    if (vv[u] >= v1) continue;
    float f[8], a[8];
    unpack8(rx[u], f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float t = (f[i] - mu[i]) * sc[i] + be[i];
      f[i] = (t > 0.f ? t : slope * t) * cs[i];
    }
    if (add != nullptr) {
      unpack8(ra[u], a);
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] += a[i];
    }
    stg16(y + vv[u] * C + c8 * 8, pack8(f));
  }
  for (int64_t v = v0 + l + 4 * (int64_t)lanes; v < v1; v += lanes) {  // (blocks larger than 4 voxels per thread)
    float f[8], a[8];
    unpack8(ldg16(x + v * C + c8 * 8), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float t = (f[i] - mu[i]) * sc[i] + be[i];
      f[i] = (t > 0.f ? t : slope * t) * cs[i];
    }
    if (add != nullptr) {
      unpack8(ldg16(add + v * C + c8 * 8), a);
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] += a[i];
    }
    stg16(y + v * C + c8 * 8, pack8(f));
  }
}


// ---------------------------------------------------------------------------------------------
// InstanceNorm + LeakyReLU backward. With s = sqrt(var) + eps, xh = (x - mean) / s, z = gamma * xh + beta and
// g = dL/dz = (gy [+ gy2]) * chan_scale * (z > 0 ? 1 : slope):
//   dgamma = sum g * xh,  dbeta = sum g,
//   dx = (gamma / s) * (g - mean_v(g) - xh * (s / sigma) * mean_v(g * xh))      (eps sits on the STD, so the
//   variance term carries s / sigma = 1 + eps / sigma instead of 1)
// Two passes over (x, gy): per-(sample, block) partial sums of (g, g * xh), fp64 combine, then the apply pass.
// ---------------------------------------------------------------------------------------------
struct NormBwdArgs {
  const bf16* x;          // raw conv output
  const float* stats;     // [N][C][2] (mean, 1/s)
  const float* gamma;
  const float* beta;
  const bf16* gy;
  const bf16* gy2;        // optional second gradient (fan-out of the block output)
  const float* chan_scale;
  int64_t vox_per_sample;
  int C;
  float slope;
};

struct NormConst {
  float mean[8], inv_s[8], gamma[8], beta[8], cs[8];
};
__device__ __forceinline__ void norm_load_const(const NormBwdArgs& a, int n, int c8, NormConst& k) {
  const float4* sp = reinterpret_cast<const float4*>(a.stats + ((int64_t)n * a.C + c8 * 8) * 2);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 st = __ldg(sp + i);  // (mean, 1/s) of two channels
    k.mean[2 * i] = st.x, k.inv_s[2 * i] = st.y, k.mean[2 * i + 1] = st.z, k.inv_s[2 * i + 1] = st.w;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ch = c8 * 8 + i;
    k.gamma[i] = __ldg(a.gamma + ch);
    k.beta[i] = __ldg(a.beta + ch);
    k.cs[i] = a.chan_scale ? __ldg(a.chan_scale + (int64_t)n * a.C + ch) : 1.f;
  }
}
struct NormBwdRaw {
  uint4 x, gy, gy2;
};
__device__ __forceinline__ void norm_bwd_load(const NormBwdArgs& a, int64_t v, int c8, NormBwdRaw& r) {
  r.x = ldg16(a.x + v * a.C + c8 * 8);
  r.gy = ldg16(a.gy + v * a.C + c8 * 8);
  if (a.gy2 != nullptr) r.gy2 = ldg16(a.gy2 + v * a.C + c8 * 8);
}
__device__ __forceinline__ void norm_bwd_compute(const NormBwdArgs& a, const NormConst& k, const NormBwdRaw& r, float g[8],
                                                 float xh[8]) {
  float x[8], t[8];
  unpack8(r.x, x);
  unpack8(r.gy, g);
  if (a.gy2 != nullptr) {
    unpack8(r.gy2, t);
#pragma unroll
    for (int i = 0; i < 8; ++i) g[i] += t[i];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    xh[i] = (x[i] - k.mean[i]) * k.inv_s[i];
    const float z = k.gamma[i] * xh[i] + k.beta[i];
    g[i] *= (z > 0.f ? 1.f : a.slope) * k.cs[i];
  }
}
__device__ __forceinline__ void norm_bwd_g(const NormBwdArgs& a, const NormConst& k, int64_t v, int c8, float g[8],
                                           float xh[8]) {
  NormBwdRaw r;
  norm_bwd_load(a, v, c8, r);
  norm_bwd_compute(a, k, r, g, xh);
}

__global__ void __launch_bounds__(kThreads) instnorm_bwd_partial_kernel(NormBwdArgs a, float* __restrict__ part,
                                                                        int64_t vox_per_block, int blocks_per_sample) {
  extern __shared__ float sh[];  // [kThreads][16]
  const int C = a.C, c8n = C >> 3;
  const int lanes = kThreads / c8n;
  const int c8 = threadIdx.x % c8n, l = threadIdx.x / c8n;
  const int n = blockIdx.y, blk = blockIdx.x;
  const int64_t v0 = (int64_t)n * a.vox_per_sample + (int64_t)blk * vox_per_block;
  const int64_t v1 = min((int64_t)(n + 1) * a.vox_per_sample, v0 + vox_per_block);
  float s1[8], s2[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s1[i] = s2[i] = 0.f;
  if (l < lanes) {
    NormConst k;
    norm_load_const(a, n, c8, k);
    int64_t v = v0 + l;
    for (; v + (int64_t)lanes < v1; v += 2 * (int64_t)lanes) {  // two voxels per trip: 4-6 loads in flight per thread
      NormBwdRaw r0, r1;
      norm_bwd_load(a, v, c8, r0);
      norm_bwd_load(a, v + lanes, c8, r1);
      float g[8], xh[8];
      norm_bwd_compute(a, k, r0, g, xh);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s1[i] += g[i];
        s2[i] += g[i] * xh[i];
      }
      norm_bwd_compute(a, k, r1, g, xh);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s1[i] += g[i];
        s2[i] += g[i] * xh[i];
      }
    }
    for (; v < v1; v += lanes) {
      float g[8], xh[8];
      norm_bwd_g(a, k, v, c8, g, xh);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s1[i] += g[i];
        s2[i] += g[i] * xh[i];
      }
    }
  }
  if (fold_channel_groups(s1, s2, sh, c8n)) {
    float* o = part + (((int64_t)n * blocks_per_sample + blk) * C + threadIdx.x * 8) * 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      o[2 * i] = s1[i];
      o[2 * i + 1] = s2[i];
    }
  }
}

// coef[n][c] = (gamma / s, mean(g), (s / sigma) * mean(g * xh)); dgamma / dbeta accumulate over the samples.
// One warp per (n, c), fixed-order fold of the block partials.
__global__ void instnorm_bwd_final_kernel(const float* __restrict__ part, const float* __restrict__ stats,
                                          const float* __restrict__ gamma, float* __restrict__ coef,
                                          float* __restrict__ dgamma, float* __restrict__ dbeta, int N, int C,
                                          int blocks_per_sample, double inv_count, float eps) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= N * C) return;
  const int n = i / C, c = i % C;
  double s1 = 0.0, s2 = 0.0;
  for (int b = lane; b < blocks_per_sample; b += 32) {
    const float2 o = *reinterpret_cast<const float2*>(part + (((int64_t)n * blocks_per_sample + b) * C + c) * 2);
    s1 += (double)o.x;
    s2 += (double)o.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if (lane != 0) return;
  const double inv_s = (double)stats[2 * i + 1];
  const double s = 1.0 / inv_s;
  const double sigma = fmax(s - (double)eps, 1e-12);
  coef[4 * i] = (float)((double)gamma[c] * inv_s);
  coef[4 * i + 1] = (float)(s1 * inv_count);
  coef[4 * i + 2] = (float)(s / sigma * s2 * inv_count);
  coef[4 * i + 3] = 0.f;
  atomicAdd(dgamma + c, (float)s2);
  atomicAdd(dbeta + c, (float)s1);
}

// grid (blocks per sample, N), like the partial pass
__global__ void __launch_bounds__(kThreads) instnorm_bwd_apply_kernel(NormBwdArgs a, const float* __restrict__ coef,
                                                                      bf16* __restrict__ dx, int64_t vox_per_block) {
  const int c8n = a.C >> 3;
  const int lanes = kThreads / c8n;
  const int c8 = threadIdx.x % c8n, l = threadIdx.x / c8n;
  if (l >= lanes) return;
  const int n = blockIdx.y;
  NormConst k;
  norm_load_const(a, n, c8, k);
  float ca[8], cm1[8], cm2[8];
  const float4* cp = reinterpret_cast<const float4*>(coef + ((int64_t)n * a.C + c8 * 8) * 4);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 t = __ldg(cp + i);
    ca[i] = t.x, cm1[i] = t.y, cm2[i] = t.z;
  }
  const int64_t v0 = (int64_t)n * a.vox_per_sample + (int64_t)blockIdx.x * vox_per_block;
  const int64_t v1 = min((int64_t)(n + 1) * a.vox_per_sample, v0 + vox_per_block);
  int64_t v = v0 + l;
  for (; v + (int64_t)lanes < v1; v += 2 * (int64_t)lanes) {  // two voxels per trip
    NormBwdRaw r0, r1;
    norm_bwd_load(a, v, c8, r0);
    norm_bwd_load(a, v + lanes, c8, r1);
    float g[8], xh[8];
    norm_bwd_compute(a, k, r0, g, xh);
#pragma unroll
    for (int i = 0; i < 8; ++i) g[i] = ca[i] * (g[i] - cm1[i] - xh[i] * cm2[i]);
    stg16(dx + v * a.C + c8 * 8, pack8(g));
    norm_bwd_compute(a, k, r1, g, xh);
#pragma unroll
    for (int i = 0; i < 8; ++i) g[i] = ca[i] * (g[i] - cm1[i] - xh[i] * cm2[i]);
    stg16(dx + (v + lanes) * a.C + c8 * 8, pack8(g));
  }
  for (; v < v1; v += lanes) {
    float g[8], xh[8];
    norm_bwd_g(a, k, v, c8, g, xh);
#pragma unroll
    for (int i = 0; i < 8; ++i) g[i] = ca[i] * (g[i] - cm1[i] - xh[i] * cm2[i]);
    stg16(dx + v * a.C + c8 * 8, pack8(g));
  }
}

// transposed-conv helper for the stride-2 in-convs: fine[2v + 1] = coarse[v] per axis, zero elsewhere. A stride-1
// 'same' dgrad / wgrad over this tensor equals the stride-2 (TF SAME, pad_before = 0) conv's dgrad / wgrad.
// (pz = 1: the 2D family - z is not strided.)
__global__ void zero_insert_kernel(const bf16* __restrict__ coarse, bf16* __restrict__ fine, int N, int X, int Y, int Z,
                                   int C, int pz) {
  const int c8n = C >> 3;
  const int64_t total = (int64_t)N * X * Y * Z * 4 * pz * c8n;  // fine voxels x 16-byte groups
  const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= total) return;
  const int c8 = (int)(gi % c8n);
  int64_t v = gi / c8n;
  const int z = (int)(v % (pz * Z));
  int64_t r = v / (pz * Z);
  const int y = (int)(r % (2 * Y));
  r /= 2 * Y;
  const int x = (int)(r % (2 * X));
  const int n = (int)(r / (2 * X));
  uint4 o = make_uint4(0u, 0u, 0u, 0u);
  if ((x & y & (pz == 2 ? z : 1) & 1) != 0) {
    const int64_t vc = (((int64_t)n * X + (x >> 1)) * Y + (y >> 1)) * Z + (pz == 2 ? (z >> 1) : z);
    o = ldg16(coarse + vc * C + c8 * 8);
  }
  stg16(fine + v * C + c8 * 8, o);
}

__global__ void add_bf16_kernel(const bf16* __restrict__ a, const bf16* __restrict__ b, bf16* __restrict__ out,
                                int64_t n8) {
  const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= n8) return;
  float fa[8], fb[8];
  unpack8(ldg16(a + gi * 8), fa);
  unpack8(ldg16(b + gi * 8), fb);
#pragma unroll
  for (int i = 0; i < 8; ++i) fa[i] += fb[i];
  stg16(out + gi * 8, pack8(fa));
}

// gradient of the nearest-neighbour upsampling of a single-channel fp32 map: 2^3 sum-pool
__global__ void sumpool_f32_kernel(const float* __restrict__ fine, float* __restrict__ coarse, int N, int X, int Y,
                                   int Z, int pz) {  // coarse extents; pz = 1: 2x2 sum-pool in x, y only
  const int64_t total = (int64_t)N * X * Y * Z;
  const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= total) return;
  const int z = (int)(gi % Z);
  int64_t r = gi / Z;
  const int y = (int)(r % Y);
  r /= Y;
  const int x = (int)(r % X);
  const int n = (int)(r / X);
  float acc = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int64_t vf = (((int64_t)n * 2 * X + 2 * x + (k >> 1)) * 2 * Y + 2 * y + (k & 1)) * pz * Z + pz * z;
    if (pz == 2) {
      const float2 t = __ldg(reinterpret_cast<const float2*>(fine + vf));
      acc += t.x + t.y;
    } else {
      acc += __ldg(fine + vf);
    }
  }
  coarse[gi] = acc;
}

// SpatialDropout3D keep mask: scale[n][c] = keep ? 1 / (1 - rate) : 0, from a counter-based hash of (seed, index)
__global__ void dropout_scale_kernel(float* __restrict__ scale, int n, float rate, uint64_t seed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t h = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(i + 1);  // splitmix64
  h = (h ^ (h >> 30)) * 0xBF58476D1CE4E5B9ull;
  h = (h ^ (h >> 27)) * 0x94D049BB133111EBull;
  h ^= h >> 31;
  const float u = (float)(h >> 40) * (1.0f / 16777216.0f);
  scale[i] = u >= rate ? 1.f / (1.f - rate) : 0.f;
}

// segmentation-head plumbing of the Isensee net (isensee2017.py:68-79): fp32 single-channel maps
// out[v] = fine[v] + coarse[v >> 1 per axis]   /   p = sigmoid(z)
__global__ void seg_upsample_add_kernel(const float* __restrict__ fine, const float* __restrict__ coarse,
                                        float* __restrict__ out, int N, int X, int Y, int Z, int pz) {
  const int64_t total = (int64_t)N * X * Y * Z;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int z = (int)(g % Z);
  int64_t r = g / Z;
  const int y = (int)(r % Y);
  r /= Y;
  const int x = (int)(r % X);
  const int n = (int)(r / X);
  const int zc = pz == 2 ? (z >> 1) : z, Zc = pz == 2 ? (Z >> 1) : Z;
  const int64_t vc = (((int64_t)n * (X >> 1) + (x >> 1)) * (Y >> 1) + (y >> 1)) * Zc + zc;
  out[g] = fine[g] + __ldg(coarse + vc);
}
// the same two steps for L > 1 labels: maps [N][X][Y][Z][L] (label fastest); one thread per element, every label summed
// with the arithmetic of the one-label kernels
__global__ void seg_upsample_add_labels_kernel(const float* __restrict__ fine, const float* __restrict__ coarse,
                                               float* __restrict__ out, int N, int X, int Y, int Z, int pz, int L) {
  const int64_t total = (int64_t)N * X * Y * Z * L;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int l = (int)(g % L);
  int64_t r = g / L;
  const int z = (int)(r % Z);
  r /= Z;
  const int y = (int)(r % Y);
  r /= Y;
  const int x = (int)(r % X);
  const int n = (int)(r / X);
  const int zc = pz == 2 ? (z >> 1) : z, Zc = pz == 2 ? (Z >> 1) : Z;
  const int64_t vc = (((int64_t)n * (X >> 1) + (x >> 1)) * (Y >> 1) + (y >> 1)) * Zc + zc;
  out[g] = fine[g] + __ldg(coarse + vc * L + l);
}
__global__ void sumpool_f32_labels_kernel(const float* __restrict__ fine, float* __restrict__ coarse, int N, int X,
                                          int Y, int Z, int pz, int L) {  // coarse extents
  const int64_t total = (int64_t)N * X * Y * Z * L;
  const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= total) return;
  const int l = (int)(gi % L);
  int64_t r = gi / L;
  const int z = (int)(r % Z);
  r /= Z;
  const int y = (int)(r % Y);
  r /= Y;
  const int x = (int)(r % X);
  const int n = (int)(r / X);
  float acc = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int64_t vf = (((int64_t)n * 2 * X + 2 * x + (k >> 1)) * 2 * Y + 2 * y + (k & 1)) * pz * Z + pz * z;
    if (pz == 2)
      acc += __ldg(fine + vf * L + l) + __ldg(fine + (vf + 1) * L + l);
    else
      acc += __ldg(fine + vf * L + l);
  }
  coarse[gi] = acc;
}
__global__ void sigmoid_kernel(const float* __restrict__ z, float* __restrict__ p, int64_t n) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n) p[g] = 1.f / (1.f + __expf(-z[g]));
}

// ---------------------------------------------------------------------------------------------
// soft-Dice statistics — fetal_net/metrics.py:11-15 (dice), :18-28 (vod), Keras binary_accuracy
// deterministic two-stage reduction: per-block partials in double, then one block sums them.
// ---------------------------------------------------------------------------------------------
constexpr int kRedBlocks = 592;  // 4 x 148 SMs

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(kThreads) dice_partial_kernel(const float* __restrict__ p,
                                                                const float* __restrict__ t,
                                                                int64_t n, double* __restrict__ part, XentSpec xs) {
  FM_PDL_SYNC();
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const int64_t nv = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float4 pp = __ldg(reinterpret_cast<const float4*>(p) + i);
    const float4 tt = __ldg(reinterpret_cast<const float4*>(t) + i);
    const float pa[4] = {pp.x, pp.y, pp.z, pp.w};
    const float ta[4] = {tt.x, tt.y, tt.z, tt.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float pb = pa[k] > 0.5f ? 1.f : 0.f;
      const float tb = ta[k] > 0.5f ? 1.f : 0.f;
      s[0] += ta[k] * pa[k];
      s[1] += ta[k];
      s[2] += pa[k];
      s[3] += tb * pb;
      s[4] += tb;
      s[5] += pb;
      s[6] += (ta[k] == pb) ? 1.f : 0.f;
      if (xs.weight != 0.f) s[7] += xent_voxel_weight(xs, i * 4 + k) * xent_term(ta[k], pa[k]);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    for (int64_t i = nv << 2; i < n; ++i) {
      const float pb = p[i] > 0.5f ? 1.f : 0.f, tb = t[i] > 0.5f ? 1.f : 0.f;
      s[0] += t[i] * p[i];
      s[1] += t[i];
      s[2] += p[i];
      s[3] += tb * pb;
      s[4] += tb;
      s[5] += pb;
      s[6] += (t[i] == pb) ? 1.f : 0.f;
      if (xs.weight != 0.f) s[7] += xent_voxel_weight(xs, i) * xent_term(t[i], p[i]);
    }
  }
  __shared__ double sh[kThreads / 32][8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const double w = warp_sum((double)s[k]);
    if (lane == 0) sh[warp][k] = w;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    double a = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) a += sh[w][threadIdx.x];
    part[(int64_t)blockIdx.x * 8 + threadIdx.x] = a;
  }
}

__global__ void __launch_bounds__(256) dice_final_kernel(const double* __restrict__ part, int nblocks, double n_elems,
                                                         double* __restrict__ sums, int accumulate) {
  FM_PDL_SYNC();
  // 32 strided partial chains per statistic, then a fixed-order fold: deterministic, ~20 dependent adds deep
  __shared__ double sh[32][8];
  // partial slot 7 = sum w * binary cross-entropy (zero under the plain Dice loss) -> sums[8]; sums[7] = element count
  const int k = threadIdx.x & 7, j = threadIdx.x >> 3;
  double a = 0.0;
  for (int b = j; b < nblocks; b += 32) a += part[(int64_t)b * 8 + k];
  sh[j][k] = a;
  __syncthreads();
  if (threadIdx.x < 8) {
    double s = 0.0;
    for (int g = 0; g < 32; ++g) s += sh[g][threadIdx.x];
    const int dst = threadIdx.x == 7 ? 8 : threadIdx.x;
    sums[dst] = accumulate ? sums[dst] + s : s;
  } else if (threadIdx.x == 8) {
    sums[7] = accumulate ? sums[7] + n_elems : n_elems;
  }
}

// Multi-label statistics (1 < L <= kMaxLabels, label of element i = i mod L): the 8 partials of dice_partial_kernel over
// all elements, then (tp, t, p) per label; 8 + 3 L per block (write_label_partials).
__global__ void __launch_bounds__(kThreads) dice_partial_labels_kernel(const float* __restrict__ p,
                                                                       const float* __restrict__ t, int64_t n, int L,
                                                                       double* __restrict__ part, XentSpec xs) {
  FM_PDL_SYNC();
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float sl[3 * kMaxLabels];
#pragma unroll
  for (int i = 0; i < 3 * kMaxLabels; ++i) sl[i] = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float pv = __ldg(p + i), tt = __ldg(t + i);
    const float pb = pv > 0.5f ? 1.f : 0.f, tb = tt > 0.5f ? 1.f : 0.f;
    s[0] += tt * pv;
    s[1] += tt;
    s[2] += pv;
    s[3] += tb * pb;
    s[4] += tb;
    s[5] += pb;
    s[6] += (tt == pb) ? 1.f : 0.f;
    if (xs.weight != 0.f) s[7] += xent_voxel_weight(xs, i) * xent_term(tt, pv);
    const int l = (int)(i % L);
#pragma unroll
    for (int k = 0; k < kMaxLabels; ++k)
      if (k == l) {
        sl[3 * k] += tt * pv;
        sl[3 * k + 1] += tt;
        sl[3 * k + 2] += pv;
      }
  }
  write_label_partials<kThreads>(s, sl, L, part);
}

// fixed-order fold of nblocks rows of K = 8 + 3 L partials: 32 strided chains per statistic, then the chains in order.
// Partial slot 7 (sum w * bce) -> sums[8], sums[7] = element count, slot 8 + j -> sums[kNumLossSums + j].
__global__ void __launch_bounds__(1024) dice_final_labels_kernel(const double* __restrict__ part, int nblocks, int K,
                                                                 double n_elems, double* __restrict__ sums) {
  FM_PDL_SYNC();
  __shared__ double sh[32][8 + 3 * kMaxLabels];
  const int k = threadIdx.x & 31, j = threadIdx.x >> 5;
  if (k < K) {
    double a = 0.0;
    for (int b = j; b < nblocks; b += 32) a += part[(int64_t)b * K + k];
    sh[j][k] = a;
  }
  __syncthreads();
  if ((int)threadIdx.x < K) {
    double s = 0.0;
    for (int g = 0; g < 32; ++g) s += sh[g][threadIdx.x];
    sums[threadIdx.x < 7 ? threadIdx.x : threadIdx.x + 1] = s;
  } else if ((int)threadIdx.x == K) {
    sums[7] = n_elems;
  }
}

// [B][L][V] -> [B][V][L] (to_device) or back; one thread per element of `out`
__global__ void label_transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t V, int L,
                                       int64_t total, int to_device) {
  for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
    const int64_t per = V * L, b = o / per, r = o - b * per;
    int64_t v, l;
    if (to_device) {
      v = r / L;
      l = r - v * L;
    } else {
      l = r / V;
      v = r - l * V;
    }
    out[o] = __ldg(in + b * per + (to_device ? l * V + v : v * L + l));
  }
}

// dL/dz for L = -dice(t, sigmoid(z)): closed form of metrics.py:11-15,31-32 with smooth = 1
__global__ void dice_bwd_kernel(const float* __restrict__ p, const float* __restrict__ t,
                                const double* __restrict__ sums, int64_t n, float* __restrict__ dz,
                                int through_sigmoid, XentSpec xs) {
  FM_PDL_SYNC();
  const double I = sums[0], S = sums[1] + sums[2] + 1.0;
  const float a = (float)(-2.0 / S);               // coefficient of t_i
  const float b = (float)((2.0 * I + 1.0) / (S * S));  // constant term
  // cross-entropy term of dice_and_xent (through the sigmoid only): weight / count * w_i * (p_i - t_i)
  const float xc = xs.weight != 0.f ? (float)((double)xs.weight / sums[7]) : 0.f;
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 4 <= n) {
    const float4 pp = __ldg(reinterpret_cast<const float4*>(p + i));
    const float4 tt = __ldg(reinterpret_cast<const float4*>(t + i));
    float4 o;
    o.x = a * tt.x + b;
    o.y = a * tt.y + b;
    o.z = a * tt.z + b;
    o.w = a * tt.w + b;
    if (through_sigmoid) {
      o.x *= pp.x * (1.f - pp.x);
      o.y *= pp.y * (1.f - pp.y);
      o.z *= pp.z * (1.f - pp.z);
      o.w *= pp.w * (1.f - pp.w);
      if (xc != 0.f) {
        o.x += xc * xent_voxel_weight(xs, i) * xent_grad(tt.x, pp.x);
        o.y += xc * xent_voxel_weight(xs, i + 1) * xent_grad(tt.y, pp.y);
        o.z += xc * xent_voxel_weight(xs, i + 2) * xent_grad(tt.z, pp.z);
        o.w += xc * xent_voxel_weight(xs, i + 3) * xent_grad(tt.w, pp.w);
      }
    }
    *reinterpret_cast<float4*>(dz + i) = o;
  } else {
    for (; i < n; ++i) {
      float o = a * t[i] + b;
      if (through_sigmoid) {
        o *= p[i] * (1.f - p[i]);
        if (xc != 0.f) o += xc * xent_voxel_weight(xs, i) * xent_grad(t[i], p[i]);
      }
      dz[i] = o;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Keras-2 Adam (SURVEY.md App. A.9): epsilon outside the bias correction, lr_t folded on host
// ---------------------------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float lr_t, float b1, float b2,
                            float eps) {
  FM_PDL_SYNC();
  int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 4 <= n) {
    float4 pp = *reinterpret_cast<float4*>(p + i);
    const float4 gg = __ldg(reinterpret_cast<const float4*>(g + i));
    float4 mm = *reinterpret_cast<float4*>(m + i);
    float4 vv = *reinterpret_cast<float4*>(v + i);
#define FM_ADAM1(c)                                   \
  mm.c = b1 * mm.c + (1.f - b1) * gg.c;               \
  vv.c = b2 * vv.c + (1.f - b2) * gg.c * gg.c;        \
  pp.c = pp.c - lr_t * mm.c / (sqrtf(vv.c) + eps);
    FM_ADAM1(x) FM_ADAM1(y) FM_ADAM1(z) FM_ADAM1(w)
#undef FM_ADAM1
    *reinterpret_cast<float4*>(p + i) = pp;
    *reinterpret_cast<float4*>(m + i) = mm;
    *reinterpret_cast<float4*>(v + i) = vv;
  } else {
    for (; i < n; ++i) {
      const float gg = g[i];
      const float mm = b1 * m[i] + (1.f - b1) * gg;
      const float vv = b2 * v[i] + (1.f - b2) * gg * gg;
      m[i] = mm;
      v[i] = vv;
      p[i] = p[i] - lr_t * mm / (sqrtf(vv) + eps);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// patch gather — get_patch_from_3d_data on the virtually padded volume
// (fetal_net/utils/patches.py:57-72; padding of fetal_net/prediction.py:138-146)
// ---------------------------------------------------------------------------------------------
struct GatherGeom {
  int vol[3], halo[3], fit[3], padded[3], patch[3];
  int halo_dims[3];
};

__global__ void gather_patches_kernel(const float* __restrict__ vol, GatherGeom gm, float pad0,
                                      float pad1, const int32_t* __restrict__ idx, int64_t n,
                                      float* __restrict__ out, int out_pitch, int out_cofs, int z_shift) {
  // one patch per blockIdx.y (strided when there are more patches than grid rows); 32-bit arithmetic inside a patch
  // (64-bit div/mod by run-time extents costs ~100 instructions each)
  const uint32_t pv = (uint32_t)gm.patch[0] * (uint32_t)gm.patch[1] * (uint32_t)gm.patch[2];
  for (int64_t pi = blockIdx.y; pi < n; pi += gridDim.y)
  for (uint32_t r0 = blockIdx.x * blockDim.x + threadIdx.x; r0 < pv; r0 += gridDim.x * blockDim.x) {
    uint32_t r = r0;
    const int k = (int)(r % (uint32_t)gm.patch[2]);
    r /= (uint32_t)gm.patch[2];
    const int j = (int)(r % (uint32_t)gm.patch[1]);
    const int i = (int)(r / (uint32_t)gm.patch[1]);
    // coordinate in the fit-padded array -> halo-padded array -> original volume
    const int c[3] = {idx[pi * 3 + 0] + i, idx[pi * 3 + 1] + j, idx[pi * 3 + 2] + k + z_shift};
    float val;
    int h[3], o[3];
    bool in_halo = true, in_vol = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      h[a] = c[a] - gm.fit[a];
      in_halo = in_halo && h[a] >= 0 && h[a] < gm.halo_dims[a];
      o[a] = h[a] - gm.halo[a];
      in_vol = in_vol && o[a] >= 0 && o[a] < gm.vol[a];
    }
    if (!in_halo)
      val = pad1;
    else if (!in_vol)
      val = pad0;
    else
      val = __ldg(vol + ((int64_t)o[0] * gm.vol[1] + o[1]) * gm.vol[2] + o[2]);
    out[((pi * gm.patch[0] + i) * (int64_t)gm.patch[1] + j) * out_pitch + out_cofs + k] = val;
  }
}

// four z-consecutive patch voxels per thread (patch[2] % 4 == 0): the index arithmetic and the x / y range tests are
// shared, the store is one 16-byte write when the destination allows it
__global__ void __launch_bounds__(kThreads) gather_patches4_kernel(const float* __restrict__ vol, GatherGeom gm, float pad0,
                                                                   float pad1, const int32_t* __restrict__ idx, int64_t n,
                                                                   float* __restrict__ out, int out_pitch, int out_cofs,
                                                                   int z_shift, int vec_store) {
  const uint32_t k4n = (uint32_t)gm.patch[2] >> 2;
  const uint32_t pv4 = (uint32_t)gm.patch[0] * (uint32_t)gm.patch[1] * k4n;
  for (int64_t pi = blockIdx.y; pi < n; pi += gridDim.y) {
    const int c0b = __ldg(idx + pi * 3 + 0), c1b = __ldg(idx + pi * 3 + 1), c2b = __ldg(idx + pi * 3 + 2) + z_shift;
    for (uint32_t r0 = blockIdx.x * blockDim.x + threadIdx.x; r0 < pv4; r0 += gridDim.x * blockDim.x) {
      uint32_t r = r0;
      const int k = (int)(r % k4n) * 4;
      r /= k4n;
      const int j = (int)(r % (uint32_t)gm.patch[1]);
      const int i = (int)(r / (uint32_t)gm.patch[1]);
      const int h0 = c0b + i - gm.fit[0], h1 = c1b + j - gm.fit[1];
      const int o0 = h0 - gm.halo[0], o1 = h1 - gm.halo[1];
      const bool halo_xy = h0 >= 0 && h0 < gm.halo_dims[0] && h1 >= 0 && h1 < gm.halo_dims[1];
      const bool vol_xy = o0 >= 0 && o0 < gm.vol[0] && o1 >= 0 && o1 < gm.vol[1];
      const float* row = vol + ((int64_t)o0 * gm.vol[1] + o1) * gm.vol[2];
      float val[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int h2 = c2b + k + e - gm.fit[2], o2 = h2 - gm.halo[2];
        if (!(halo_xy && h2 >= 0 && h2 < gm.halo_dims[2]))
          val[e] = pad1;
        else if (!(vol_xy && o2 >= 0 && o2 < gm.vol[2]))
          val[e] = pad0;
        else
          val[e] = __ldg(row + o2);
      }
      float* dst = out + ((pi * gm.patch[0] + i) * (int64_t)gm.patch[1] + j) * out_pitch + out_cofs + k;
      if (vec_store) {
        *reinterpret_cast<float4*>(dst) = make_float4(val[0], val[1], val[2], val[3]);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) dst[e] = val[e];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// overlap-add / average reassembly — fetal_net/prediction.py:188-193,210
// output-stationary: every output voxel walks the (contiguous) range of patches covering it per
// axis, adding float32 predictions in float64 in ascending patch order — the same order the
// reference's `+=` loop uses — so the sum (and sum / count) is bit-identical. No atomics.
// ---------------------------------------------------------------------------------------------
struct ReasmGeom {
  int out[3], pred[3], np[3];
  int channels;
};

__global__ void reassemble_kernel(const float* __restrict__ preds, ReasmGeom gm,
                                  const int32_t* __restrict__ starts,   // [3][max np]
                                  const int32_t* __restrict__ cover,    // [3][max dim][2] lo,hi
                                  int starts_pitch, int cover_pitch, int64_t shard_lo,
                                  int64_t shard_hi, int64_t pred_base, double* __restrict__ out,
                                  int16_t* __restrict__ count, int divide, int x_lo, int x_hi) {
  // blockIdx.y walks x in [x_lo, x_hi); 32-bit arithmetic inside one (y, z, channel) plane
  const int64_t pvox = (int64_t)gm.pred[0] * gm.pred[1] * gm.pred[2];
  const uint32_t plane = (uint32_t)gm.out[1] * (uint32_t)gm.out[2] * (uint32_t)gm.channels;
  for (int x = x_lo + blockIdx.y; x < x_hi; x += gridDim.y)
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < plane; q += gridDim.x * blockDim.x) {
    const int ch = (int)(q % (uint32_t)gm.channels);
    uint32_t r = q / (uint32_t)gm.channels;
    const int z = (int)(r % (uint32_t)gm.out[2]);
    const int y = (int)(r / (uint32_t)gm.out[2]);
    const int64_t v = (int64_t)x * gm.out[1] * gm.out[2] + r;
    const int64_t g = (int64_t)x * plane + q;
    const int xlo = cover[(0 * cover_pitch + x) * 2], xhi = cover[(0 * cover_pitch + x) * 2 + 1];
    const int ylo = cover[(1 * cover_pitch + y) * 2], yhi = cover[(1 * cover_pitch + y) * 2 + 1];
    const int zlo = cover[(2 * cover_pitch + z) * 2], zhi = cover[(2 * cover_pitch + z) * 2 + 1];
    double acc = 0.0;
    for (int ix = xlo; ix < xhi; ++ix) {
      const int px = x - starts[0 * starts_pitch + ix];
      for (int iy = ylo; iy < yhi; ++iy) {
        const int py = y - starts[1 * starts_pitch + iy];
        for (int iz = zlo; iz < zhi; ++iz) {
          const int64_t patch = ((int64_t)ix * gm.np[1] + iy) * gm.np[2] + iz;
          if (patch < shard_lo || patch >= shard_hi) continue;
          const int pz = z - starts[2 * starts_pitch + iz];
          const int64_t off = (((patch - pred_base) * pvox) +
                               ((int64_t)px * gm.pred[1] + py) * gm.pred[2] + pz) * gm.channels + ch;
          acc += (double)__ldg(preds + off);
        }
      }
    }
    const int cnt = (xhi - xlo) * (yhi - ylo) * (zhi - zlo);
    if (count != nullptr && ch == 0) count[v] = (int16_t)cnt;
    if (divide)
      out[g] = acc / (double)cnt;
    else
      out[g] += acc;
  }
}

// single-channel maps with out[2] % 4 == 0: four z-consecutive outputs per thread share the x / y covering sets and
// the index arithmetic; every output still adds its patches in ascending patch order (ix, iy, iz) in fp64 and
// divides by its analytic count, so the result is bit-identical to reassemble_kernel
__global__ void __launch_bounds__(kThreads) reassemble4_kernel(const float* __restrict__ preds, ReasmGeom gm,
                                                               const int32_t* __restrict__ starts,
                                                               const int32_t* __restrict__ cover, int starts_pitch,
                                                               int cover_pitch, int64_t shard_lo, int64_t shard_hi,
                                                               int64_t pred_base, double* __restrict__ out,
                                                               int16_t* __restrict__ count, int divide, int x_lo,
                                                               int x_hi) {
  const int64_t pvox = (int64_t)gm.pred[0] * gm.pred[1] * gm.pred[2];
  const uint32_t z4n = (uint32_t)gm.out[2] >> 2;
  const uint32_t plane4 = (uint32_t)gm.out[1] * z4n;
  for (int x = x_lo + blockIdx.y; x < x_hi; x += gridDim.y) {
    const int2 cx = __ldg(reinterpret_cast<const int2*>(cover + (0 * cover_pitch + x) * 2));
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < plane4; q += gridDim.x * blockDim.x) {
      const int z = (int)(q % z4n) * 4;
      const int y = (int)(q / z4n);
      const int2 cy = __ldg(reinterpret_cast<const int2*>(cover + (1 * cover_pitch + y) * 2));
      int2 cz[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) cz[e] = __ldg(reinterpret_cast<const int2*>(cover + (2 * cover_pitch + z + e) * 2));
      double acc[4] = {0.0, 0.0, 0.0, 0.0};
      for (int ix = cx.x; ix < cx.y; ++ix) {
        const int px = x - __ldg(starts + 0 * starts_pitch + ix);
        for (int iy = cy.x; iy < cy.y; ++iy) {
          const int py = y - __ldg(starts + 1 * starts_pitch + iy);
          const int64_t prow = ((int64_t)px * gm.pred[1] + py) * gm.pred[2];
          const int64_t pxy = ((int64_t)ix * gm.np[1] + iy) * gm.np[2];
#pragma unroll
          for (int e = 0; e < 4; ++e)
            for (int iz = cz[e].x; iz < cz[e].y; ++iz) {
              const int64_t patch = pxy + iz;
              if (patch < shard_lo || patch >= shard_hi) continue;
              const int pz = z + e - __ldg(starts + 2 * starts_pitch + iz);
              acc[e] += (double)__ldg(preds + (patch - pred_base) * pvox + prow + pz);
            }
        }
      }
      const int64_t v = ((int64_t)x * gm.out[1] + y) * gm.out[2] + z;
      const int nxy = (cx.y - cx.x) * (cy.y - cy.x);
      double res[4];
      short cn[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int cnt = nxy * (cz[e].y - cz[e].x);
        cn[e] = (short)cnt;
        if (!divide) {
          res[e] = out[v + e] + acc[e];
        } else if ((cnt & (cnt - 1)) == 0) {
          // power-of-two count (the usual case: 1 or 2 covering patches per axis): the quotient is the exact product
          // with 2^-k, bit-identical to the IEEE division and ~40 instructions cheaper
          res[e] = acc[e] * __longlong_as_double((long long)(1023 - (31 - __clz(cnt))) << 52);
        } else {
          res[e] = acc[e] / (double)cnt;
        }
      }
      reinterpret_cast<double2*>(out + v)[0] = make_double2(res[0], res[1]);
      reinterpret_cast<double2*>(out + v)[1] = make_double2(res[2], res[3]);
      if (count != nullptr) *reinterpret_cast<short4*>(count + v) = make_short4(cn[0], cn[1], cn[2], cn[3]);
    }
  }
}

__global__ void divide_by_count_kernel(double* __restrict__ out, const int16_t* __restrict__ count,
                                       int64_t nvox, int channels) {
  const int64_t total = nvox * channels;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (int64_t)gridDim.x * blockDim.x)
    out[g] = out[g] / (double)count[g / channels];
}

inline int grid_for(int64_t work_items, int cap = 1 << 30) {
  int64_t b = ceil_div64(work_items, kThreads);
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// launch wrappers
// ---------------------------------------------------------------------------------------------
int k_cast_f32_to_bf16(fm_ctx* ctx, const float* in, bf16* out, int64_t n) {
  cast_f32_bf16_kernel<<<grid_for(ceil_div64(n, 8)), kThreads, 0, ctx->stream>>>(in, out, n);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_cast_bf16_to_f32(fm_ctx* ctx, const bf16* in, float* out, int64_t n) {
  cast_bf16_f32_kernel<<<grid_for(ceil_div64(n, 8)), kThreads, 0, ctx->stream>>>(in, out, n);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_maxpool3d_fwd(fm_ctx* ctx, const bf16* x, bf16* y, Dims5 in, int pz) {
  FM_CHECK(in.C % 8 == 0 && in.X % 2 == 0 && in.Y % 2 == 0 && in.Z % pz == 0 && (pz == 1 || pz == 2), FM_EINVAL,
           "maxpool3d: need C%%8==0 and even extents (got C=%d %dx%dx%d)", in.C, in.X, in.Y, in.Z);
  const int64_t total = in.elems() / (32 * pz);
  ProfScope prof(ctx, "maxpool3d_fwd", 0.0, (double)in.elems() * 2.0 * 1.125);
  if (pz == 2)
    FM_CUDA(launch_pdl(maxpool3d_fwd_kernel<2>, dim3(grid_for(total)), dim3(kThreads), 0, ctx->stream, x, y, in.N, in.X, in.Y, in.Z, in.C));
  else
    FM_CUDA(launch_pdl(maxpool3d_fwd_kernel<1>, dim3(grid_for(total)), dim3(kThreads), 0, ctx->stream, x, y, in.N, in.X, in.Y, in.Z, in.C));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_maxpool3d_bwd(fm_ctx* ctx, const bf16* x, const bf16* dy, const bf16* dskip, bf16* dx, Dims5 in,
                    int relu_mask, int pz) {
  FM_CHECK(in.C % 8 == 0 && in.X % 2 == 0 && in.Y % 2 == 0 && in.Z % pz == 0 && (pz == 1 || pz == 2), FM_EINVAL,
           "maxpool3d_bwd: need C%%8==0 and even extents");
  const int64_t total = in.elems() / (32 * pz) * 2;  // two threads per (pooled voxel, 8 channels)
  ProfScope prof(ctx, "maxpool3d_bwd", 0.0, (double)in.elems() * 2.0 * (dskip ? 3.125 : 2.125));
  if (pz == 2)
    FM_CUDA(launch_pdl(maxpool3d_bwd_kernel<2>, dim3(grid_for(total)), dim3(kThreads), 0, ctx->stream, x, dy, dskip, dx, in.N, in.X, in.Y, in.Z,
                                                                          in.C, relu_mask));
  else
    FM_CUDA(launch_pdl(maxpool3d_bwd_kernel<1>, dim3(grid_for(total)), dim3(kThreads), 0, ctx->stream, x, dy, dskip, dx, in.N, in.X, in.Y, in.Z,
                                                                          in.C, relu_mask));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_upsample3d_fwd(fm_ctx* ctx, const bf16* x, bf16* y, Dims5 in, int pz) {
  FM_CHECK(in.C % 8 == 0, FM_EINVAL, "upsample3d: need C%%8==0");
  ProfScope prof(ctx, "upsample3d_fwd", 0.0, (double)in.elems() * 2.0 * 9.0);
  if (pz == 2)
    FM_CUDA(launch_pdl(upsample3d_fwd_kernel<2>, dim3(grid_for(in.elems() / 8)), dim3(kThreads), 0, ctx->stream, x, y, in.N, in.X, in.Y, in.Z, in.C));
  else
    FM_CUDA(launch_pdl(upsample3d_fwd_kernel<1>, dim3(grid_for(in.elems() / 8)), dim3(kThreads), 0, ctx->stream, x, y, in.N, in.X, in.Y, in.Z, in.C));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_upsample3d_bwd(fm_ctx* ctx, const bf16* dy, const bf16* act, bf16* dx, Dims5 coarse, int dy_C,
                     int dy_cofs, int pz) {
  FM_CHECK(coarse.C % 8 == 0 && dy_C % 8 == 0 && dy_cofs % 8 == 0, FM_EINVAL,
           "upsample3d_bwd: channel counts must be multiples of 8");
  ProfScope prof(ctx, "upsample3d_bwd", 0.0, (double)coarse.elems() * 2.0 * (act ? 10.0 : 9.0));
  if (pz == 2)
    FM_CUDA(launch_pdl(upsample3d_bwd_kernel<2>, dim3(grid_for(coarse.elems() / 8)), dim3(kThreads), 0, ctx->stream, 
        dy, act, dx, coarse.N, coarse.X, coarse.Y, coarse.Z, coarse.C, dy_C, dy_cofs));
  else
    FM_CUDA(launch_pdl(upsample3d_bwd_kernel<1>, dim3(grid_for(coarse.elems() / 8)), dim3(kThreads), 0, ctx->stream, 
        dy, act, dx, coarse.N, coarse.X, coarse.Y, coarse.Z, coarse.C, dy_C, dy_cofs));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_dice_sums(fm_ctx* ctx, const float* p, const float* t, int64_t n, double* sums, int accumulate, XentSpec xs,
                int L) {
  if (L != 1) {
    FM_CHECK(L >= 2 && L <= kMaxLabels && !accumulate && n % L == 0, FM_EINVAL,
             "dice_sums: %d labels over %lld elements (accumulate %d)", L, (long long)n, accumulate);
    ProfScope prof(ctx, "dice_sums_labels", 0.0, (double)n * (xs.mask ? 12.0 : 8.0));
    FM_CUDA(launch_pdl(dice_partial_labels_kernel, dim3(kRedBlocks), dim3(kThreads), 0, ctx->stream, p, t, n, L,
                       ctx->red_scratch, xs));
    FM_LAUNCH_OK(ctx);
    return k_dice_finalize_labels(ctx, kRedBlocks, (double)n, sums, L);
  }
  ProfScope prof(ctx, "dice_sums", 0.0, (double)n * (xs.mask ? 12.0 : 8.0));
  FM_CUDA(launch_pdl(dice_partial_kernel, dim3(kRedBlocks), dim3(kThreads), 0, ctx->stream, p, t, n, ctx->red_scratch, xs));
  FM_LAUNCH_OK(ctx);
  FM_CUDA(launch_pdl(dice_final_kernel, dim3(1), dim3(256), 0, ctx->stream, ctx->red_scratch, kRedBlocks, (double)n, sums,
                                              accumulate));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
// fixed-order fold of `nblocks` x 8 partial statistics in ctx->red_scratch (written by head_fwd_dice_kernel)
int k_dice_finalize(fm_ctx* ctx, int nblocks, double n_elems, double* sums) {
  FM_CUDA(launch_pdl(dice_final_kernel, dim3(1), dim3(256), 0, ctx->stream, ctx->red_scratch, nblocks, n_elems, sums, 0));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_dice_finalize_labels(fm_ctx* ctx, int nblocks, double n_elems, double* sums, int L) {
  FM_CUDA(launch_pdl(dice_final_labels_kernel, dim3(1), dim3(1024), 0, ctx->stream, ctx->red_scratch, nblocks, 8 + 3 * L,
                     n_elems, sums));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_label_transpose(fm_ctx* ctx, const float* in, float* out, int B, int64_t V, int L, int to_device) {
  const int64_t total = (int64_t)B * V * L;
  ProfScope prof(ctx, "label_transpose", 0.0, (double)total * 8.0);
  label_transpose_kernel<<<grid_for(total, 148 * 16), kThreads, 0, ctx->stream>>>(in, out, V, L, total, to_device);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_dice_bwd(fm_ctx* ctx, const float* p, const float* t, const double* sums, int64_t n, float* dz,
               int through_sigmoid, XentSpec xs) {
  FM_CHECK(xs.weight == 0.f || through_sigmoid, FM_EINVAL, "dice_bwd: the cross-entropy term is formed through the sigmoid");
  ProfScope prof(ctx, "dice_bwd", 0.0, (double)n * (xs.mask ? 16.0 : 12.0));
  FM_CUDA(launch_pdl(dice_bwd_kernel, dim3(grid_for(ceil_div64(n, 4))), dim3(kThreads), 0, ctx->stream, p, t, sums, n, dz,
                                                                           through_sigmoid, xs));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_adam(fm_ctx* ctx, float* p, const float* g, float* m, float* v, int64_t n, int iterations,
           float lr) {
  const double b1 = 0.9, b2 = 0.999;
  const double t = (double)iterations + 1.0;
  const float lr_t = (float)((double)lr * sqrt(1.0 - pow(b2, t)) / (1.0 - pow(b1, t)));
  ProfScope prof(ctx, "adam", 0.0, (double)n * 28.0);
  FM_CUDA(launch_pdl(adam_kernel, dim3(grid_for(ceil_div64(n, 4))), dim3(kThreads), 0, ctx->stream, p, g, m, v, n, lr_t, 0.9f,
                                                                       0.999f, 1e-7f));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_zero(fm_ctx* ctx, void* p, size_t bytes) {
  FM_CUDA(cudaMemsetAsync(p, 0, bytes, ctx->stream));
  return FM_OK;
}

int k_pad_cast(fm_ctx* ctx, const float* in, bf16* out, int64_t vox, int Cin, int Cpad) {
  ProfScope prof(ctx, "pad_cast", 0.0, (double)vox * (Cin * 4.0 + Cpad * 2.0));
  pad_cast_kernel<<<grid_for(vox * Cpad, 148 * 32), kThreads, 0, ctx->stream>>>(in, out, vox, Cin, Cpad);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_gather_patches(fm_ctx* ctx, const float* vol, const int32_t vol_dims[3],
                     const int32_t halo_pad[6], const int32_t fit_pad[6], float pad0, float pad1,
                     const int32_t* idx_dev, int64_t n, const int32_t patch[3], float* out, int out_pitch,
                     int out_cofs, int z_shift) {
  if (out_pitch <= 0) out_pitch = patch[2];
  GatherGeom gm;
  for (int a = 0; a < 3; ++a) {
    gm.vol[a] = vol_dims[a];
    gm.halo[a] = halo_pad[2 * a];
    gm.fit[a] = fit_pad[2 * a];
    gm.halo_dims[a] = vol_dims[a] + halo_pad[2 * a] + halo_pad[2 * a + 1];
    gm.padded[a] = gm.halo_dims[a] + fit_pad[2 * a] + fit_pad[2 * a + 1];
    gm.patch[a] = patch[a];
  }
  const int64_t total = n * (int64_t)patch[0] * patch[1] * patch[2];
  ProfScope prof(ctx, "gather_patches", 0.0, (double)total * 8.0);
  const int64_t pv = (int64_t)patch[0] * patch[1] * patch[2];
  FM_CHECK(pv < ((int64_t)1 << 31), FM_EINVAL, "gather_patches: patch of %lld voxels", (long long)pv);
  if (patch[2] % 4 == 0) {
    const int vec = out_pitch % 4 == 0 && out_cofs % 4 == 0 && ((uintptr_t)out & 15) == 0;
    const dim3 grid((unsigned)grid_for(pv / 4, 1024), (unsigned)std::min<int64_t>(n, 32768));
    gather_patches4_kernel<<<grid, kThreads, 0, ctx->stream>>>(vol, gm, pad0, pad1, idx_dev, n, out, out_pitch, out_cofs,
                                                              z_shift, vec);
  } else {
    const dim3 grid((unsigned)grid_for(pv, 1024), (unsigned)std::min<int64_t>(n, 32768));
    gather_patches_kernel<<<grid, kThreads, 0, ctx->stream>>>(vol, gm, pad0, pad1, idx_dev, n, out, out_pitch, out_cofs,
                                                             z_shift);
  }
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// Host side of the reassembly: turns the corner list into per-axis start lists + per-coordinate
// covering ranges (the corners of fm_patch_plan are always a Cartesian product in x-major order;
// anything else is rejected). Prepared once per call; the overlap-add itself can then run slab by slab
// (rows [x_lo, x_hi) of the output) as soon as the patches covering a slab have been predicted.
struct ReasmPlan {
  int32_t *d_starts = nullptr, *d_cover = nullptr;
  int maxnp = 0, maxdim = 0;
  ReasmGeom gm;
  std::vector<int32_t> xstarts;  // distinct x corners, ascending
  int64_t n_total = 0;
};

int k_reassemble_prepare(fm_ctx* ctx, const int32_t* idx_host, int64_t n_total, const int32_t pred_shape[3],
                         int channels, const int32_t out_dims[3], ReasmPlan** out_plan) {
  std::vector<int32_t> st[3];
  for (int a = 0; a < 3; ++a) {
    for (int64_t i = 0; i < n_total; ++i) {
      const int32_t v = idx_host[i * 3 + a];
      bool seen = false;
      for (int32_t s : st[a]) seen = seen || (s == v);
      if (!seen) st[a].push_back(v);
    }
    for (size_t i = 1; i < st[a].size(); ++i)
      FM_CHECK(st[a][i] > st[a][i - 1], FM_EINVAL, "reassemble: patch corners not ascending on axis %d", a);
  }
  const int64_t np0 = st[0].size(), np1 = st[1].size(), np2 = st[2].size();
  FM_CHECK(np0 * np1 * np2 == n_total, FM_EINVAL,
           "reassemble: corner list is not a Cartesian product (%lld*%lld*%lld != %lld)",
           (long long)np0, (long long)np1, (long long)np2, (long long)n_total);
  for (int64_t i = 0; i < n_total; ++i) {
    const int64_t i2 = i % np2, i1 = (i / np2) % np1, i0 = i / (np2 * np1);
    FM_CHECK(idx_host[i * 3] == st[0][i0] && idx_host[i * 3 + 1] == st[1][i1] &&
                 idx_host[i * 3 + 2] == st[2][i2],
             FM_EINVAL, "reassemble: corner list is not in x-major product order at %lld", (long long)i);
  }
  int maxnp = (int)std::max(np0, std::max(np1, np2));
  int maxdim = std::max(out_dims[0], std::max(out_dims[1], out_dims[2]));
  std::vector<int32_t> starts(3 * (size_t)maxnp, 0), cover(3 * (size_t)maxdim * 2, 0);
  for (int a = 0; a < 3; ++a) {
    for (size_t i = 0; i < st[a].size(); ++i) starts[(size_t)a * maxnp + i] = st[a][i];
    for (int c = 0; c < out_dims[a]; ++c) {
      int lo = (int)st[a].size(), hi = 0;
      for (int i = 0; i < (int)st[a].size(); ++i)
        if (st[a][i] <= c && c < st[a][i] + pred_shape[a]) {
          lo = std::min(lo, i);
          hi = std::max(hi, i + 1);
        }
      FM_CHECK(hi > lo, FM_EINVAL, "Found zeros in count");  // prediction.py:196
      for (int i = lo; i < hi; ++i)
        FM_CHECK(st[a][i] <= c && c < st[a][i] + pred_shape[a], FM_EINVAL,
                 "reassemble: covering set not contiguous");
      cover[((size_t)a * maxdim + c) * 2] = lo;
      cover[((size_t)a * maxdim + c) * 2 + 1] = hi;
    }
  }
  ReasmPlan* pl = new ReasmPlan();
  cudaError_t e = cudaMalloc((void**)&pl->d_starts, starts.size() * 4);
  if (e == cudaSuccess) e = cudaMalloc((void**)&pl->d_cover, cover.size() * 4);
  // synchronous copies: the host vectors go out of scope below (a few hundred bytes)
  if (e == cudaSuccess) e = cudaMemcpy(pl->d_starts, starts.data(), starts.size() * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(pl->d_cover, cover.data(), cover.size() * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    fm_set_error("reassemble: %s", cudaGetErrorString(e));
    k_reassemble_release(pl);
    return FM_ECUDA;
  }
  for (int a = 0; a < 3; ++a) {
    pl->gm.out[a] = out_dims[a];
    pl->gm.pred[a] = pred_shape[a];
  }
  pl->gm.np[0] = (int)np0;
  pl->gm.np[1] = (int)np1;
  pl->gm.np[2] = (int)np2;
  pl->gm.channels = channels;
  pl->maxnp = maxnp;
  pl->maxdim = maxdim;
  pl->xstarts = st[0];
  pl->n_total = n_total;
  (void)ctx;
  *out_plan = pl;
  return FM_OK;
}

void k_reassemble_release(ReasmPlan* pl) {
  if (!pl) return;
  if (pl->d_starts) cudaFree(pl->d_starts);
  if (pl->d_cover) cudaFree(pl->d_cover);
  delete pl;
}

int k_reassemble_groups(const ReasmPlan* pl, const int32_t** xstarts, int* n_groups, int* patches_per_group) {
  *xstarts = pl->xstarts.data();
  *n_groups = pl->gm.np[0];
  *patches_per_group = pl->gm.np[1] * pl->gm.np[2];
  return FM_OK;
}

// overlap-add (+ count, + divide) of the output rows [x_lo, x_hi). `preds` holds patches [pred_base, ...) of the plan.
int k_reassemble_rows(fm_ctx* ctx, const ReasmPlan* pl, const float* preds, int64_t shard_lo, int64_t shard_hi,
                      int64_t pred_base, double* out_dev, int16_t* count_dev, int divide, int x_lo, int x_hi) {
  const ReasmGeom& gm = pl->gm;
  FM_CHECK(x_lo >= 0 && x_hi <= gm.out[0] && x_lo < x_hi, FM_EINVAL, "reassemble: rows [%d, %d) of %d", x_lo, x_hi, gm.out[0]);
  const int channels = gm.channels;
  const double frac = (double)(x_hi - x_lo) / (double)gm.out[0];
  const int64_t total = (int64_t)gm.out[0] * gm.out[1] * gm.out[2] * channels;
  ProfScope prof(ctx, "reassemble", 0.0,
                 frac * ((double)(shard_hi - shard_lo) * gm.pred[0] * gm.pred[1] * gm.pred[2] * channels * 4.0 + (double)total * 8.0));
  const int64_t plane = (int64_t)gm.out[1] * gm.out[2] * channels;
  FM_CHECK(plane < ((int64_t)1 << 31), FM_EINVAL, "reassemble: plane of %lld elements", (long long)plane);
  const int rows = x_hi - x_lo;
  if (channels == 1 && gm.out[2] % 4 == 0 && ((uintptr_t)out_dev & 15) == 0 && ((uintptr_t)count_dev & 7) == 0) {
    const dim3 rgrid((unsigned)grid_for(plane / 4, 256), (unsigned)std::min<int>(rows, 32768));
    reassemble4_kernel<<<rgrid, kThreads, 0, ctx->stream>>>(preds, gm, pl->d_starts, pl->d_cover, pl->maxnp, pl->maxdim,
                                                           shard_lo, shard_hi, pred_base, out_dev, count_dev, divide, x_lo,
                                                           x_hi);
  } else {
    const dim3 rgrid((unsigned)grid_for(plane, 256), (unsigned)std::min<int>(rows, 32768));
    reassemble_kernel<<<rgrid, kThreads, 0, ctx->stream>>>(preds, gm, pl->d_starts, pl->d_cover, pl->maxnp, pl->maxdim,
                                                          shard_lo, shard_hi, pred_base, out_dev, count_dev, divide, x_lo,
                                                          x_hi);
  }
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_reassemble(fm_ctx* ctx, const float* preds, const int32_t* idx_host, int64_t n_total,
                 int64_t shard_lo, int64_t shard_hi, int64_t pred_base,
                 const int32_t pred_shape[3], int channels, const int32_t out_dims[3],
                 double* out_dev, int16_t* count_dev, int divide) {
  ReasmPlan* pl = nullptr;
  FM_TRY(k_reassemble_prepare(ctx, idx_host, n_total, pred_shape, channels, out_dims, &pl));
  const int rc = k_reassemble_rows(ctx, pl, preds, shard_lo, shard_hi, pred_base, out_dev, count_dev, divide, 0, out_dims[0]);
  cudaStreamSynchronize(ctx->stream);  // the plan's tables are freed below
  k_reassemble_release(pl);
  return rc;
}

int k_divide_by_count(fm_ctx* ctx, double* out, const int16_t* count, int64_t nvox, int channels) {
  divide_by_count_kernel<<<grid_for(nvox * channels, 148 * 16), kThreads, 0, ctx->stream>>>(
      out, count, nvox, channels);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// x: raw conv output [N][vox][C] bf16 -> y = LeakyReLU(InstanceNorm(x)) (+ add). `scratch` >= N*C*(2*blocks + 4) floats.
static int norm_blocks(int64_t vox_per_sample, int64_t* vpb) {
  int bps = (int)std::min<int64_t>(std::max<int64_t>(1, vox_per_sample / 512), 1024);
  *vpb = ceil_div64(vox_per_sample, bps);
  return (int)ceil_div64(vox_per_sample, *vpb);
}
// the element-wise passes want many more, smaller blocks: ~4 voxels per thread
static int norm_apply_blocks(int64_t vox_per_sample, int C, int64_t* vpb) {
  const int lanes = kThreads / (C / 8);
  *vpb = (int64_t)lanes * 4;
  return (int)ceil_div64(vox_per_sample, *vpb);
}

// gradient of k_instnorm_lrelu w.r.t. the raw conv output (dx), gamma and beta (accumulated into dgamma / dbeta).
// `scratch` >= N*C*(2*blocks + 4) floats.
int k_instnorm_lrelu_bwd(fm_ctx* ctx, const bf16* x, const float* stats, const float* gamma, const float* beta,
                         const bf16* gy, const bf16* gy2, const float* chan_scale, bf16* dx, float* dgamma,
                         float* dbeta, int N, int64_t vox_per_sample, int C, float* scratch, size_t scratch_floats) {
  FM_CHECK(C >= 8 && C <= 512 && (C & (C - 1)) == 0, FM_EINVAL, "instnorm bwd: C=%d must be a power of two in [8,512]", C);
  int64_t vpb;
  const int bps = norm_blocks(vox_per_sample, &vpb);
  const size_t need = (size_t)N * C * (2 * (size_t)bps + 4);
  FM_CHECK(scratch_floats >= need, FM_EINVAL, "instnorm bwd: scratch too small (%zu < %zu floats)", scratch_floats, need);
  float* part = scratch;
  float* coef = scratch + (size_t)N * C * 2 * bps;
  NormBwdArgs a{x, stats, gamma, beta, gy, gy2, chan_scale, vox_per_sample, C, 0.3f};
  ProfScope prof(ctx, "instnorm_lrelu_bwd", 0.0, (double)N * vox_per_sample * C * (gy2 ? 14.0 : 10.0));
  instnorm_bwd_partial_kernel<<<dim3(bps, N), kThreads, kThreads * 16 * sizeof(float), ctx->stream>>>(a, part, vpb, bps);
  FM_LAUNCH_OK(ctx);
  instnorm_bwd_final_kernel<<<ceil_div(N * C * 32, 128), 128, 0, ctx->stream>>>(part, stats, gamma, coef, dgamma, dbeta,
                                                                                 N, C, bps, 1.0 / (double)vox_per_sample,
                                                                                 1e-3f);
  FM_LAUNCH_OK(ctx);
  int64_t vpa;
  const int bpa = norm_apply_blocks(vox_per_sample, C, &vpa);
  instnorm_bwd_apply_kernel<<<dim3(bpa, N), kThreads, 0, ctx->stream>>>(a, coef, dx, vpa);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_zero_insert(fm_ctx* ctx, const bf16* coarse, bf16* fine, Dims5 c, int pz) {
  FM_CHECK(c.C % 8 == 0, FM_EINVAL, "zero_insert: C=%d", c.C);
  ProfScope prof(ctx, "zero_insert", 0.0, (double)c.elems() * 2.0 * (1.0 + 4.0 * pz));
  zero_insert_kernel<<<grid_for(c.elems() / 8 * 4 * pz), kThreads, 0, ctx->stream>>>(coarse, fine, c.N, c.X, c.Y, c.Z,
                                                                                     c.C, pz);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_add_bf16(fm_ctx* ctx, const bf16* a, const bf16* b, bf16* out, int64_t n) {
  FM_CHECK(n % 8 == 0, FM_EINVAL, "add_bf16: n %% 8");
  ProfScope prof(ctx, "add_bf16", 0.0, (double)n * 6.0);
  add_bf16_kernel<<<grid_for(n / 8), kThreads, 0, ctx->stream>>>(a, b, out, n / 8);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_sumpool_f32(fm_ctx* ctx, const float* fine, float* coarse, int N, int X, int Y, int Z, int pz, int L) {
  if (L != 1) {
    const int64_t total = (int64_t)N * X * Y * Z * L;
    ProfScope prof(ctx, "sumpool_f32_labels", 0.0, (double)total * (4.0 + 16.0 * pz));
    sumpool_f32_labels_kernel<<<grid_for(total), kThreads, 0, ctx->stream>>>(fine, coarse, N, X, Y, Z, pz, L);
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  ProfScope prof(ctx, "sumpool_f32", 0.0, (double)N * X * Y * Z * (4.0 + 16.0 * pz));
  sumpool_f32_kernel<<<grid_for((int64_t)N * X * Y * Z), kThreads, 0, ctx->stream>>>(fine, coarse, N, X, Y, Z, pz);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// SpatialDropout2D of the 2D U-Net (unet/unet.py:60-61,76-77): x[n][v][c] *= scale[n][c], in place; the same kernel
// scales the gradient on the way back
__global__ void channel_scale_kernel(bf16* __restrict__ x, const float* __restrict__ scale, int64_t vox_per_sample,
                                     int C, int64_t total8) {
  const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= total8) return;
  const int c8n = C >> 3;
  const int c8 = (int)(gi % c8n);
  const int64_t n = gi / c8n / vox_per_sample;
  float f[8];
  unpack8(ldg16(x + gi * 8), f);
  const float* sc = scale + n * C + c8 * 8;
#pragma unroll
  for (int i = 0; i < 8; ++i) f[i] *= __ldg(sc + i);
  stg16(x + gi * 8, pack8(f));
}

int k_channel_scale(fm_ctx* ctx, bf16* x, const float* scale, int N, int64_t vox_per_sample, int C) {
  FM_CHECK(C % 8 == 0, FM_EINVAL, "channel_scale: C=%d must be a multiple of 8", C);
  const int64_t total8 = (int64_t)N * vox_per_sample * (C / 8);
  ProfScope prof(ctx, "channel_scale", 0.0, (double)total8 * 32.0);
  channel_scale_kernel<<<grid_for(total8), kThreads, 0, ctx->stream>>>(x, scale, vox_per_sample, C, total8);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// Deconvolution (k = 2, s = 2) shuffles: one thread per 16-byte channel group of a FINE voxel.
template <bool TO_SPACE>
__global__ void depth_space_kernel(const bf16* __restrict__ src, const float* __restrict__ bias, bf16* __restrict__ dst,
                                   int N, int X, int Y, int Z, int C, int pz) {  // X, Y, Z = coarse extents
  const int c8n = C >> 3;
  const int64_t total = (int64_t)N * X * Y * Z * 4 * pz * c8n;
  const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= total) return;
  const int c8 = (int)(gi % c8n);
  int64_t v = gi / c8n;  // fine voxel index
  const int fz = (int)(v % (pz * Z));
  int64_t r = v / (pz * Z);
  const int fy = (int)(r % (2 * Y));
  r /= 2 * Y;
  const int fx = (int)(r % (2 * X));
  const int n = (int)(r / (2 * X));
  const int a = fx & 1, b = fy & 1, c = pz == 2 ? (fz & 1) : 0;
  const int cls = (a * 2 + b) * pz + c;
  const int64_t vc = (((int64_t)n * X + (fx >> 1)) * Y + (fy >> 1)) * Z + (pz == 2 ? (fz >> 1) : fz);
  const int64_t coarse_ofs = (vc * (4 * pz) + cls) * C + c8 * 8;
  const int64_t fine_ofs = v * C + c8 * 8;
  if (TO_SPACE) {
    float f[8];
    unpack8(ldg16(src + coarse_ofs), f);
    if (bias != nullptr) {
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] += __ldg(bias + c8 * 8 + i);
    }
    stg16(dst + fine_ofs, pack8(f));
  } else {
    stg16(dst + coarse_ofs, ldg16(src + fine_ofs));
  }
}

int k_depth_to_space(fm_ctx* ctx, const bf16* z8, const float* bias, bf16* fine, Dims5 c, int pz) {
  FM_CHECK(c.C % 8 == 0, FM_EINVAL, "depth_to_space: C=%d", c.C);
  const int64_t total = c.elems() / 8 * 4 * pz;
  ProfScope prof(ctx, "depth_to_space", 0.0, (double)total * 32.0);
  depth_space_kernel<true><<<grid_for(total), kThreads, 0, ctx->stream>>>(z8, bias, fine, c.N, c.X, c.Y, c.Z, c.C, pz);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_space_to_depth(fm_ctx* ctx, const bf16* fine, bf16* g8, Dims5 c, int pz) {
  FM_CHECK(c.C % 8 == 0, FM_EINVAL, "space_to_depth: C=%d", c.C);
  const int64_t total = c.elems() / 8 * 4 * pz;
  ProfScope prof(ctx, "space_to_depth", 0.0, (double)total * 32.0);
  depth_space_kernel<false><<<grid_for(total), kThreads, 0, ctx->stream>>>(fine, nullptr, g8, c.N, c.X, c.Y, c.Z, c.C, pz);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_dropout_scale(fm_ctx* ctx, float* scale, int n, float rate, uint64_t seed) {
  dropout_scale_kernel<<<ceil_div(n, 128), 128, 0, ctx->stream>>>(scale, n, rate, seed);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_instnorm_lrelu(fm_ctx* ctx, const bf16* x, const float* gamma, const float* beta, const bf16* add, bf16* y,
                     int N, int64_t vox_per_sample, int C, float* scratch, size_t scratch_floats, float* stats,
                     const float* chan_scale) {
  FM_CHECK(C >= 8 && C <= 512 && (C & (C - 1)) == 0, FM_EINVAL, "instnorm: C=%d must be a power of two in [8,512]", C);
  int64_t vpb;
  const int bps = norm_blocks(vox_per_sample, &vpb);
  const size_t need = (size_t)N * C * (2 * (size_t)bps + 4);
  FM_CHECK(scratch_floats >= need, FM_EINVAL, "instnorm: scratch too small (%zu < %zu floats)", scratch_floats, need);
  float* part = scratch;
  float* ss = scratch + (size_t)N * C * 2 * bps;
  ProfScope prof(ctx, "instnorm_lrelu", 0.0, (double)N * vox_per_sample * C * (add ? 8.0 : 6.0));
  instnorm_partial_kernel<<<dim3(bps, N), kThreads, kThreads * 16 * sizeof(float), ctx->stream>>>(x, part, vox_per_sample,
                                                                                               C, vpb, bps);
  FM_LAUNCH_OK(ctx);
  instnorm_final_kernel<<<ceil_div(N * C * 32, 128), 128, 0, ctx->stream>>>(part, gamma, beta, ss, stats, N, C, bps,
                                                                             1.0 / (double)vox_per_sample, 1e-3f);
  FM_LAUNCH_OK(ctx);
  int64_t vpa;
  const int bpa = norm_apply_blocks(vox_per_sample, C, &vpa);
  instnorm_apply_kernel<<<dim3(bpa, N), kThreads, 0, ctx->stream>>>(x, ss, add, chan_scale, y, vox_per_sample, C, vpa,
                                                                     0.3f);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------
// BatchNormalization(axis=1) + ReLU — create_convolution_block(batch_normalization=True), unet3d/unet.py:103-104,112.
// Keras 2.x semantics: training: per-channel mean / BIASED variance over (batch, voxels),
// y = (x - mean) * rsqrt(var + 1e-3) * gamma + beta; moving_mean / moving_variance <- 0.99 * old + 0.01 * batch value,
// the variance fed to the moving average carries Keras' sample-size correction n / (n - (1 + eps)); inference: the
// moving statistics. The per-(sample, block) partial pass, the apply pass and the backward partial / apply passes are
// the instance-norm kernels above (slope 0 = ReLU); only the folds differ: they run over the samples too, and
// eps sits under the square root.
// ---------------------------------------------------------------------------------------------
// Per-channel fold of the (n, block) partial pairs part[b][C][2] in fp64, one warp per channel: lane l takes pairs l,
// l + 32, ... in (n, block) order, then a fixed xor butterfly (deterministic; every lane ends with the same totals).
// The single-pass final kernels and batchnorm_fold_kernel all fold through this function, so the statistics of a
// data-parallel step with one rank are bit-identical to those of a single-process step.
__device__ __forceinline__ void bn_fold(const float* __restrict__ part, int pairs, int C, int c, int lane, double& a,
                                        double& b) {
  a = 0.0, b = 0.0;
  for (int i = lane; i < pairs; i += 32) {
    const float2 o = *reinterpret_cast<const float2*>(part + ((int64_t)i * C + c) * 2);
    a += (double)o.x;
    b += (double)o.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
}

// Global statistics (data-parallel training): this shard's per-channel totals into sums[2C + 1] = (sum_c a, sum_c b,
// count), ready for a SUM all-reduce over the ranks. (a, b) = (x, x^2) forward, (g, g * xh) backward; the backward
// also adds this shard's totals into dgamma / dbeta (the gradient all-reduce sums them over the ranks once).
__global__ void batchnorm_fold_kernel(const float* __restrict__ part, int pairs, int C, double count,
                                      double* __restrict__ sums, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  double a, b;
  bn_fold(part, pairs, C, c, lane, a, b);
  if (lane != 0) return;
  sums[c] = a;
  sums[C + c] = b;
  if (c == 0) sums[2 * C] = count;
  if (dgamma != nullptr) {
    dgamma[c] += (float)b;
    dbeta[c] += (float)a;
  }
}

// One warp per channel. ss / stats are written for every sample (identical rows) so that the apply kernels are shared.
// Training folds the partials of this batch, or with `sums` != nullptr takes the (all-reduced) totals and count of the
// global batch from sums[2C + 1].
__global__ void batchnorm_final_kernel(const float* __restrict__ part, const double* __restrict__ sums,
                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                       float* __restrict__ moving_mean, float* __restrict__ moving_var,
                                       float* __restrict__ ss, float* __restrict__ stats, int N, int C,
                                       int blocks_per_sample, double count, float eps, float momentum, int training) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  double mean, var;
  if (training) {
    double s, q;
    if (sums != nullptr) {
      s = sums[c], q = sums[C + c], count = sums[2 * C];
    } else {
      bn_fold(part, N * blocks_per_sample, C, c, lane, s, q);
    }
    mean = s / count;
    var = fmax(q / count - mean * mean, 0.0);
  } else {
    mean = (double)moving_mean[c];
    var = (double)moving_var[c];
  }
  const double rstd = 1.0 / sqrt(var + (double)eps);
  const double scale = (double)gamma[c] * rstd;
  for (int n = lane; n < N; n += 32) {
    ss[((int64_t)n * C + c) * 4] = (float)scale;
    ss[((int64_t)n * C + c) * 4 + 1] = (float)mean;
    ss[((int64_t)n * C + c) * 4 + 2] = beta[c];
    ss[((int64_t)n * C + c) * 4 + 3] = 0.f;
    if (stats != nullptr) {
      stats[((int64_t)n * C + c) * 2] = (float)mean;
      stats[((int64_t)n * C + c) * 2 + 1] = (float)rstd;
    }
  }
  if (training && lane == 0 && moving_mean != nullptr) {
    const double unbiased = var * (count / (count - (1.0 + (double)eps)));
    moving_mean[c] = (float)((double)moving_mean[c] * momentum + mean * (1.0 - (double)momentum));
    moving_var[c] = (float)((double)moving_var[c] * momentum + unbiased * (1.0 - (double)momentum));
  }
}

// coef[n][c] = (gamma * rstd, mean(g), mean(g * xh)) for every sample; dgamma = sum g * xh, dbeta = sum g (stored).
// With `sums` the means are those of the global batch and dgamma / dbeta are left alone (batchnorm_fold_kernel added
// this shard's totals).
__global__ void batchnorm_bwd_final_kernel(const float* __restrict__ part, const double* __restrict__ sums,
                                           const float* __restrict__ stats, const float* __restrict__ gamma,
                                           float* __restrict__ coef, float* __restrict__ dgamma,
                                           float* __restrict__ dbeta, int N, int C, int blocks_per_sample,
                                           double count) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (c >= C) return;
  double s1, s2;
  if (sums != nullptr) {
    s1 = sums[c], s2 = sums[C + c], count = sums[2 * C];
  } else {
    bn_fold(part, N * blocks_per_sample, C, c, lane, s1, s2);
  }
  const float a = (float)((double)gamma[c] * (double)stats[2 * c + 1]);  // sample 0's row: all rows are equal
  for (int n = lane; n < N; n += 32) {
    float* o = coef + ((int64_t)n * C + c) * 4;
    o[0] = a;
    o[1] = (float)(s1 / count);
    o[2] = (float)(s2 / count);
    o[3] = 0.f;
  }
  if (lane == 0 && sums == nullptr) {
    dgamma[c] += (float)s2;
    dbeta[c] += (float)s1;
  }
}

static int batchnorm_check(int C, int N, int64_t vox_per_sample, size_t scratch_floats, int64_t* vpb, int* bps) {
  FM_CHECK(C >= 8 && C <= 512 && (C & (C - 1)) == 0, FM_EINVAL, "batchnorm: C=%d must be a power of two in [8,512]", C);
  *bps = norm_blocks(vox_per_sample, vpb);
  const size_t need = (size_t)N * C * (2 * (size_t)*bps + 4);
  FM_CHECK(scratch_floats >= need, FM_EINVAL, "batchnorm: scratch too small (%zu < %zu floats)", scratch_floats, need);
  return FM_OK;
}

int k_batchnorm_sums(fm_ctx* ctx, const bf16* x, int N, int64_t vox_per_sample, int C, float* scratch,
                     size_t scratch_floats, double* sums) {
  int64_t vpb;
  int bps;
  FM_TRY(batchnorm_check(C, N, vox_per_sample, scratch_floats, &vpb, &bps));
  float* part = scratch;
  ProfScope prof(ctx, "batchnorm_sums", 0.0, (double)N * vox_per_sample * C * 2.0);
  instnorm_partial_kernel<<<dim3(bps, N), kThreads, kThreads * 16 * sizeof(float), ctx->stream>>>(x, part, vox_per_sample,
                                                                                               C, vpb, bps);
  FM_LAUNCH_OK(ctx);
  batchnorm_fold_kernel<<<ceil_div(C * 32, 128), 128, 0, ctx->stream>>>(part, N * bps, C,
                                                                      (double)N * (double)vox_per_sample, sums, nullptr,
                                                                      nullptr);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_batchnorm_relu(fm_ctx* ctx, const bf16* x, const float* gamma, const float* beta, float* moving_mean,
                     float* moving_var, bf16* y, int N, int64_t vox_per_sample, int C, float* scratch,
                     size_t scratch_floats, float* stats, int training, const double* sums) {
  int64_t vpb;
  int bps;
  FM_TRY(batchnorm_check(C, N, vox_per_sample, scratch_floats, &vpb, &bps));
  FM_CHECK(sums == nullptr || training, FM_EINVAL, "batchnorm: global sums need a training pass");
  float* part = scratch;
  float* ss = scratch + (size_t)N * C * 2 * bps;
  const bool fold = training && sums == nullptr;
  ProfScope prof(ctx, "batchnorm_relu", 0.0, (double)N * vox_per_sample * C * (fold ? 6.0 : 4.0));
  if (fold) {
    instnorm_partial_kernel<<<dim3(bps, N), kThreads, kThreads * 16 * sizeof(float), ctx->stream>>>(x, part, vox_per_sample,
                                                                                                 C, vpb, bps);
    FM_LAUNCH_OK(ctx);
  }
  batchnorm_final_kernel<<<ceil_div(C * 32, 128), 128, 0, ctx->stream>>>(part, sums, gamma, beta, moving_mean, moving_var,
                                                                       ss, stats, N, C, bps,
                                                                       (double)N * (double)vox_per_sample, 1e-3f, 0.99f,
                                                                       training);
  FM_LAUNCH_OK(ctx);
  int64_t vpa;
  const int bpa = norm_apply_blocks(vox_per_sample, C, &vpa);
  instnorm_apply_kernel<<<dim3(bpa, N), kThreads, 0, ctx->stream>>>(x, ss, nullptr, nullptr, y, vox_per_sample, C, vpa, 0.f);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_batchnorm_bwd_sums(fm_ctx* ctx, const bf16* x, const float* stats, const float* gamma, const float* beta,
                         const bf16* gy, const bf16* gy2, float* dgamma, float* dbeta, int N, int64_t vox_per_sample,
                         int C, float* scratch, size_t scratch_floats, double* sums) {
  int64_t vpb;
  int bps;
  FM_TRY(batchnorm_check(C, N, vox_per_sample, scratch_floats, &vpb, &bps));
  float* part = scratch;
  NormBwdArgs a{x, stats, gamma, beta, gy, gy2, nullptr, vox_per_sample, C, 0.f};
  ProfScope prof(ctx, "batchnorm_bwd_sums", 0.0, (double)N * vox_per_sample * C * (gy2 ? 6.0 : 4.0));
  instnorm_bwd_partial_kernel<<<dim3(bps, N), kThreads, kThreads * 16 * sizeof(float), ctx->stream>>>(a, part, vpb, bps);
  FM_LAUNCH_OK(ctx);
  batchnorm_fold_kernel<<<ceil_div(C * 32, 128), 128, 0, ctx->stream>>>(part, N * bps, C,
                                                                      (double)N * (double)vox_per_sample, sums, dgamma,
                                                                      dbeta);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_batchnorm_relu_bwd(fm_ctx* ctx, const bf16* x, const float* stats, const float* gamma, const float* beta,
                         const bf16* gy, const bf16* gy2, bf16* dx, float* dgamma, float* dbeta, int N,
                         int64_t vox_per_sample, int C, float* scratch, size_t scratch_floats, const double* sums) {
  int64_t vpb;
  int bps;
  FM_TRY(batchnorm_check(C, N, vox_per_sample, scratch_floats, &vpb, &bps));
  float* part = scratch;
  float* coef = scratch + (size_t)N * C * 2 * bps;
  NormBwdArgs a{x, stats, gamma, beta, gy, gy2, nullptr, vox_per_sample, C, 0.f};
  ProfScope prof(ctx, "batchnorm_relu_bwd", 0.0,
                 (double)N * vox_per_sample * C * ((gy2 ? 14.0 : 10.0) - (sums ? (gy2 ? 6.0 : 4.0) : 0.0)));
  if (sums == nullptr) {
    instnorm_bwd_partial_kernel<<<dim3(bps, N), kThreads, kThreads * 16 * sizeof(float), ctx->stream>>>(a, part, vpb, bps);
    FM_LAUNCH_OK(ctx);
  }
  batchnorm_bwd_final_kernel<<<ceil_div(C * 32, 128), 128, 0, ctx->stream>>>(part, sums, stats, gamma, coef, dgamma, dbeta,
                                                                           N, C, bps, (double)N * (double)vox_per_sample);
  FM_LAUNCH_OK(ctx);
  int64_t vpa;
  const int bpa = norm_apply_blocks(vox_per_sample, C, &vpa);
  instnorm_bwd_apply_kernel<<<dim3(bpa, N), kThreads, 0, ctx->stream>>>(a, coef, dx, vpa);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_seg_upsample_add(fm_ctx* ctx, const float* fine, const float* coarse, float* out, int N, int X, int Y, int Z,
                       int pz, int L) {
  if (L != 1) {
    const int64_t total = (int64_t)N * X * Y * Z * L;
    seg_upsample_add_labels_kernel<<<grid_for(total), kThreads, 0, ctx->stream>>>(fine, coarse, out, N, X, Y, Z, pz, L);
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  const int64_t total = (int64_t)N * X * Y * Z;
  seg_upsample_add_kernel<<<grid_for(total), kThreads, 0, ctx->stream>>>(fine, coarse, out, N, X, Y, Z, pz);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
int k_sigmoid(fm_ctx* ctx, const float* z, float* p, int64_t n) {
  sigmoid_kernel<<<grid_for(n), kThreads, 0, ctx->stream>>>(z, p, n);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
