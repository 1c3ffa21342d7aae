// conv_simt.cu — the convolutions that are NOT tensor-core shaped, plus small helpers:
//   * first layer (Cin = 1, K = 27): bandwidth kernel, fp32 volume in -> bf16 NDHWC out
//   * N = 1 head: 1x1x1 conv + sigmoid fused, and its backward (+ ReLU mask of the producer)
//   * bias gradients, weight repacking
//   * a generic direct-convolution fprop / wgrad pair used (a) for shapes the tcgen05 kernels do
//     not cover and (b) as the on-GPU cross-check of the tcgen05 kernels in tests (`impl = 1`).
// Keras call sites: Conv3D in create_convolution_block (fetal_net/model/unet3d/unet.py:102) and
// the final Conv3D(n_labels,(1,1,1)) + sigmoid (unet.py:68-69).
#include "common.cuh"

namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ float ldx(const void* x, int is_f32, int64_t i) {
  return is_f32 ? __ldg(reinterpret_cast<const float*>(x) + i)
                : __bfloat162float(reinterpret_cast<const bf16*>(x)[i]);
}

// --------------------------------------------------------------------------------------------
// generic direct conv (cross-correlation, 'same' zero padding, stride 1), one thread per
// (voxel, cout). Weights packed [Cout][taps][Cin_total] bf16, tap = (kx*K + ky)*K + kz.
// --------------------------------------------------------------------------------------------
__global__ void conv3d_simt_fprop_kernel(const void* __restrict__ x, int x_is_f32,
                                         const bf16* __restrict__ x2, const bf16* __restrict__ w,
                                         const float* __restrict__ bias, bf16* __restrict__ y,
                                         float* __restrict__ y32, int N, int X, int Y, int Z, int C1,
                                         int C2, int Cout, int K, int relu,
                                         const bf16* __restrict__ mask) {
  const int64_t total = (int64_t)N * X * Y * Z * Cout;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int co = (int)(g % Cout);
  int64_t v = g / Cout;
  const int z = (int)(v % Z);
  int64_t r = v / Z;
  const int yy = (int)(r % Y);
  r /= Y;
  const int xx = (int)(r % X);
  const int n = (int)(r / X);
  const int Kxy = kext_xy(K), Kz = kext_z(K);
  const int pad = Kxy / 2, padz = Kz / 2, Ct = C1 + C2, taps = Kxy * Kxy * Kz;
  float acc = bias ? bias[co] : 0.f;
  for (int kx = 0; kx < Kxy; ++kx) {
    const int xi = xx + kx - pad;
    if (xi < 0 || xi >= X) continue;
    for (int ky = 0; ky < Kxy; ++ky) {
      const int yi = yy + ky - pad;
      if (yi < 0 || yi >= Y) continue;
      for (int kz = 0; kz < Kz; ++kz) {
        const int zi = z + kz - padz;
        if (zi < 0 || zi >= Z) continue;
        const int tap = (kx * Kxy + ky) * Kz + kz;
        const int64_t vi = (((int64_t)n * X + xi) * Y + yi) * Z + zi;
        const bf16* wr = w + ((int64_t)co * taps + tap) * Ct;
        for (int c = 0; c < C1; ++c) acc += ldx(x, x_is_f32, vi * C1 + c) * __bfloat162float(wr[c]);
        for (int c = 0; c < C2; ++c)
          acc += __bfloat162float(x2[vi * C2 + c]) * __bfloat162float(wr[C1 + c]);
      }
    }
  }
  if (relu) acc = fmaxf(acc, 0.f);
  if (mask && !(__bfloat162float(mask[g]) > 0.f)) acc = 0.f;
  if (y) y[g] = __float2bfloat16(acc);
  if (y32) y32[g] = acc;
}

// generic wgrad: dw[co][tap][cin_ofs+ci] += sum_v dy[v][co] * x[v+shift(tap)][ci].
// One warp per output element and voxel chunk; lanes stride over the voxels of the chunk.
__global__ void conv3d_simt_wgrad_kernel(const void* __restrict__ x, int x_is_f32,
                                         const bf16* __restrict__ dy, float* __restrict__ dw, int N,
                                         int X, int Y, int Z, int Cin, int Ct, int cofs, int Cout,
                                         int K, int64_t vox_per_chunk) {
  const int Kxy = kext_xy(K), Kz = kext_z(K);
  const int taps = Kxy * Kxy * Kz, pad = Kxy / 2, padz = Kz / 2;
  const int64_t n_out = (int64_t)Cout * taps * Cin;
  const int warps_per_block = blockDim.x >> 5;
  const int64_t o = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  if (o >= n_out) return;
  const int lane = threadIdx.x & 31;
  const int ci = (int)(o % Cin);
  const int tap = (int)((o / Cin) % taps);
  const int co = (int)(o / ((int64_t)Cin * taps));
  const int kz = tap % Kz, ky = (tap / Kz) % Kxy, kx = tap / (Kz * Kxy);
  const int64_t nvox = (int64_t)N * X * Y * Z;
  const int64_t v0 = (int64_t)blockIdx.y * vox_per_chunk;
  const int64_t v1 = min(nvox, v0 + vox_per_chunk);
  float acc = 0.f;
  for (int64_t v = v0 + lane; v < v1; v += 32) {
    const int z = (int)(v % Z);
    int64_t r = v / Z;
    const int yy = (int)(r % Y);
    r /= Y;
    const int xx = (int)(r % X);
    const int n = (int)(r / X);
    const int xi = xx + kx - pad, yi = yy + ky - pad, zi = z + kz - padz;
    if (xi < 0 || xi >= X || yi < 0 || yi >= Y || zi < 0 || zi >= Z) continue;
    const int64_t vi = (((int64_t)n * X + xi) * Y + yi) * Z + zi;
    acc += __bfloat162float(dy[v * Cout + co]) * ldx(x, x_is_f32, vi * Cin + ci);
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
  if (lane == 0) atomicAdd(dw + ((int64_t)co * taps + tap) * Ct + cofs + ci, acc);
}

// --------------------------------------------------------------------------------------------
// first layer: Cin = 1 fp32 volume, 3x3x3, COUT in {16, 32}. One thread per voxel computes all
// COUT outputs from 27 L1-cached neighbours; weights live in smem as fp32 [27][COUT] and are
// read as LDS.128 broadcasts. Writes COUT bf16 (32/64 B) per voxel.
// --------------------------------------------------------------------------------------------
template <int COUT>
__global__ void __launch_bounds__(kThreads) conv3d_first_kernel(const float* __restrict__ x,
                                                                const bf16* __restrict__ w,
                                                                const float* __restrict__ bias,
                                                                bf16* __restrict__ y, int N, int X,
                                                                int Y, int Z, int relu) {
  FM_PDL_SYNC();
  __shared__ __align__(16) float ws[27 * COUT];
  __shared__ float bs[COUT];
  for (int i = threadIdx.x; i < 27 * COUT; i += blockDim.x) {
    const int tap = i / COUT, co = i % COUT;
    ws[i] = __bfloat162float(w[co * 27 + tap]);  // packed [Cout][27][1]
  }
  if (threadIdx.x < COUT) bs[threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  const int64_t nvox = (int64_t)N * X * Y * Z;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvox;
       v += (int64_t)gridDim.x * blockDim.x) {
    const int z = (int)(v % Z);
    int64_t r = v / Z;
    const int yy = (int)(r % Y);
    r /= Y;
    const int xx = (int)(r % X);
    const int n = (int)(r / X);
    float acc[COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) acc[c] = bs[c];
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int xi = xx + kx - 1;
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int yi = yy + ky - 1;
#pragma unroll
        for (int kz = 0; kz < 3; ++kz) {
          const int zi = z + kz - 1;
          float xv = 0.f;
          if (xi >= 0 && xi < X && yi >= 0 && yi < Y && zi >= 0 && zi < Z)
            xv = __ldg(x + (((int64_t)n * X + xi) * Y + yi) * Z + zi);
          const float4* wr = reinterpret_cast<const float4*>(ws + ((kx * 3 + ky) * 3 + kz) * COUT);
#pragma unroll
          for (int q = 0; q < COUT / 4; ++q) {
            const float4 ww = wr[q];
            acc[4 * q + 0] += xv * ww.x;
            acc[4 * q + 1] += xv * ww.y;
            acc[4 * q + 2] += xv * ww.z;
            acc[4 * q + 3] += xv * ww.w;
          }
        }
      }
    }
    uint4* out = reinterpret_cast<uint4*>(y + v * COUT);
#pragma unroll
    for (int q = 0; q < COUT / 8; ++q) {
      uint4 o;
      __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a = acc[8 * q + 2 * i], b = acc[8 * q + 2 * i + 1];
        if (relu) {
          a = fmaxf(a, 0.f);
          b = fmaxf(b, 0.f);
        }
        h[i] = __floats2bfloat162_rn(a, b);
      }
      out[q] = o;
    }
  }
}


// --------------------------------------------------------------------------------------------
// first-layer wgrad (Cin = 1): dW[co][tap] = sum_v dY[v][co] * x[v + shift(tap)].
// A warp owns one class = (kx, ky, 16-channel slice); every lane takes TWO z-adjacent voxels per trip (Z even), so
// the index arithmetic and the x loads are shared by 96 FMAs and a lane reads 64 contiguous bytes of dY. The
// 3 (kz) x 16 partial sums of the class stay in registers for the whole (persistent) block; at the end every warp
// butterfly-reduces them and issues fp32 red.add (27 * COUT per block).
// --------------------------------------------------------------------------------------------
template <int COUT>
__global__ void __launch_bounds__(32 * 9 * (COUT / 16)) conv3d_first_wgrad_kernel(const float* __restrict__ x,
                                                                                 const bf16* __restrict__ dy,
                                                                                 float* __restrict__ dw, int N, int X,
                                                                                 int Y, int Z) {
  FM_PDL_SYNC();
  constexpr int CS = 16;
  const int cls = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kx = cls % 3, ky = (cls / 3) % 3, cslice = cls / 9;
  float acc[3][CS];
#pragma unroll
  for (int t = 0; t < 3; ++t)
#pragma unroll
    for (int c = 0; c < CS; ++c) acc[t][c] = 0.f;
  // 32-bit index arithmetic (the launcher guarantees < 2^31 voxels): 64-bit div/mod costs ~100 instructions each
  const uint32_t Zh = (uint32_t)Z >> 1;
  const uint32_t npairs = (uint32_t)N * X * Y * Zh, stride = gridDim.x * 32u;
  for (uint32_t p = blockIdx.x * 32u + (uint32_t)lane; p < npairs; p += stride) {
    const int z = (int)(p % Zh) * 2;
    uint32_t r = p / Zh;
    const int yy = (int)(r % (uint32_t)Y);
    r /= (uint32_t)Y;
    const int xx = (int)(r % (uint32_t)X);
    const int n = (int)(r / (uint32_t)X);
    const int xi = xx + kx - 1, yi = yy + ky - 1;
    if (xi < 0 || xi >= X || yi < 0 || yi >= Y) continue;
    const bf16* gp = dy + (int64_t)p * 2 * COUT + cslice * CS;
    const uint4 a0 = __ldg(reinterpret_cast<const uint4*>(gp)), a1 = __ldg(reinterpret_cast<const uint4*>(gp + 8));
    const uint4 b0 = __ldg(reinterpret_cast<const uint4*>(gp + COUT)),
                b1 = __ldg(reinterpret_cast<const uint4*>(gp + COUT + 8));
    const float* xb = x + (((int64_t)n * X + xi) * Y + yi) * Z + z;
    const float2 xm = __ldg(reinterpret_cast<const float2*>(xb));  // x[z], x[z+1] (z even: 8-byte aligned)
    const float xl = z > 0 ? __ldg(xb - 1) : 0.f;
    const float xr = z + 2 < Z ? __ldg(xb + 2) : 0.f;
    const uint32_t wa[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const uint32_t wb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float ga0 = __uint_as_float(wa[j] << 16), ga1 = __uint_as_float(wa[j] & 0xffff0000u);
      const float gb0 = __uint_as_float(wb[j] << 16), gb1 = __uint_as_float(wb[j] & 0xffff0000u);
      // voxel z sees x[z-1], x[z], x[z+1]; voxel z+1 sees x[z], x[z+1], x[z+2]
      acc[0][2 * j] += xl * ga0 + xm.x * gb0;
      acc[1][2 * j] += xm.x * ga0 + xm.y * gb0;
      acc[2][2 * j] += xm.y * ga0 + xr * gb0;
      acc[0][2 * j + 1] += xl * ga1 + xm.x * gb1;
      acc[1][2 * j + 1] += xm.x * ga1 + xm.y * gb1;
      acc[2][2 * j + 1] += xm.y * ga1 + xr * gb1;
    }
  }
#pragma unroll
  for (int t = 0; t < 3; ++t)
#pragma unroll
    for (int c = 0; c < CS; ++c) {
      float a = acc[t][c];
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) a += __shfl_xor_sync(0xffffffffu, a, s);
      if (lane == ((t * CS + c) & 31)) atomicAdd(dw + (cslice * CS + c) * 27 + kx * 9 + ky * 3 + t, a);  // [Cout][27][1]
    }
}

// --------------------------------------------------------------------------------------------
// bias gradient: db[c] += sum_v dy[v][c]. Threads are laid out (voxel-lane, channel) with the
// channel fastest so each warp reads a contiguous run of rows.
// --------------------------------------------------------------------------------------------
__global__ void bias_grad_kernel(const bf16* __restrict__ dy, float* __restrict__ db, int64_t voxels,
                                 int C, int64_t vox_per_block) {
  extern __shared__ float sh[];
  const int lanes = blockDim.x / C;
  const int c = threadIdx.x % C, l = threadIdx.x / C;
  const int64_t v0 = (int64_t)blockIdx.x * vox_per_block;
  const int64_t v1 = min(voxels, v0 + vox_per_block);
  float acc = 0.f;
  if (l < lanes)
    for (int64_t v = v0 + l; v < v1; v += lanes) acc += __bfloat162float(dy[v * C + c]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  if (l == 0) {
    for (int k = 1; k < lanes; ++k) acc += sh[k * C + c];
    atomicAdd(db + c, acc);
  }
}

// Vector form for C = 8*G, G a power of two <= 32: thread i reads 16-byte element i, i+stride, ...
// of the flat [voxels*G] array; stride is a multiple of G, so a thread's channel group (lane % G)
// never changes and eight fp32 accumulators suffice. Lanes sharing a group fold by xor-shuffle.
__global__ void __launch_bounds__(kThreads) bias_grad_vec_kernel(const uint4* __restrict__ dy,
                                                                 float* __restrict__ db,
                                                                 int64_t nvec, int G) {
  __shared__ float sh[256];
  sh[threadIdx.x] = 0.f;
  // launched as a programmatic dependent (launch_pdl): sits between two tensor-core kernels of the backward pass
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  auto add8 = [&](const uint4& t) {
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      acc[2 * j] += __uint_as_float(w[j] << 16);
      acc[2 * j + 1] += __uint_as_float(w[j] & 0xffff0000u);
    }
  };
  for (; i + 3 * stride < nvec; i += 4 * stride) {
    const uint4 t0 = __ldg(dy + i), t1 = __ldg(dy + i + stride), t2 = __ldg(dy + i + 2 * stride),
                t3 = __ldg(dy + i + 3 * stride);
    add8(t0), add8(t1), add8(t2), add8(t3);
  }
  for (; i < nvec; i += stride) add8(__ldg(dy + i));
  for (int o = G; o < 32; o <<= 1)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  if (lane < G)
#pragma unroll
    for (int j = 0; j < 8; ++j) atomicAdd(&sh[lane * 8 + j], acc[j]);
  __syncthreads();
  if ((int)threadIdx.x < G * 8) atomicAdd(db + threadIdx.x, sh[threadIdx.x]);
}

// --------------------------------------------------------------------------------------------
// head: Conv3D(1,(1,1,1)) + sigmoid (unet.py:68-69). C/8 lanes cooperate on one voxel, each
// loading 16 B; shuffle-reduce; one fp32 probability per voxel.
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) head_fwd_kernel(const bf16* __restrict__ x,
                                                            const float* __restrict__ w,
                                                            const float* __restrict__ b,
                                                            float* __restrict__ p, int64_t voxels,
                                                            int C, int apply_sigmoid) {
  FM_PDL_SYNC();
  const int lpv = C >> 3;  // lanes per voxel (power of two <= 32)
  const int sub = threadIdx.x % lpv;
  float wv[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) wv[i] = __ldg(w + sub * 8 + i);
  const float bb = __ldg(b);
  const int64_t vpb = blockDim.x / lpv;
  // every thread of the block runs the same trip count (the shuffles below need full warps); four voxels per trip
  // so that four 16-byte loads are in flight per thread
  constexpr int U = 4;
  for (int64_t base = (int64_t)blockIdx.x * vpb * U; base < voxels; base += (int64_t)gridDim.x * vpb * U) {
    uint4 t[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * vpb + threadIdx.x / lpv;
      t[u] = v < voxels ? __ldg(reinterpret_cast<const uint4*>(x + v * C + sub * 8)) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * vpb + threadIdx.x / lpv;
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t[u]);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        acc += f.x * wv[2 * i] + f.y * wv[2 * i + 1];
      }
      for (int s = lpv >> 1; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      if (sub == 0 && v < voxels) p[v] = apply_sigmoid ? 1.f / (1.f + __expf(-(acc + bb))) : acc + bb;
    }
  }
}

// Training forward: the 1x1x1 head, the sigmoid AND the partial sums of the soft-Dice / VOD / accuracy statistics in
// one pass (Conv3D(n_labels, 1) + Activation('sigmoid') of unet3d/unet.py:68-69 + dice_coefficient / vod_coefficient /
// binary_accuracy of metrics.py:11-28). Per block: 7 double partial sums at part[block * 8 ...], folded in a fixed order
// by dice_final_kernel (deterministic, no atomics). p is still written: the backward pass needs it.
__global__ void __launch_bounds__(kThreads) head_fwd_dice_kernel(const bf16* __restrict__ x, const float* __restrict__ w,
                                                                 const float* __restrict__ b,
                                                                 const float* __restrict__ t, float* __restrict__ p,
                                                                 int64_t voxels, int C, double* __restrict__ part,
                                                                 XentSpec xs) {
  FM_PDL_SYNC();
  const int lpv = C >> 3;  // lanes per voxel (power of two <= 32)
  const int sub = threadIdx.x % lpv;
  float wv[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) wv[i] = __ldg(w + sub * 8 + i);
  const float bb = __ldg(b);
  const int64_t vpb = blockDim.x / lpv;
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  constexpr int U = 4;
  for (int64_t base = (int64_t)blockIdx.x * vpb * U; base < voxels; base += (int64_t)gridDim.x * vpb * U) {
    uint4 xv[U];
    float tv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * vpb + threadIdx.x / lpv;
      const bool ok = v < voxels;
      xv[u] = ok ? __ldg(reinterpret_cast<const uint4*>(x + v * C + sub * 8)) : make_uint4(0u, 0u, 0u, 0u);
      tv[u] = ok && sub == 0 ? __ldg(t + v) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * vpb + threadIdx.x / lpv;
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&xv[u]);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        acc += f.x * wv[2 * i] + f.y * wv[2 * i + 1];
      }
      for (int sft = lpv >> 1; sft > 0; sft >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, sft);
      if (sub == 0 && v < voxels) {
        const float pv = 1.f / (1.f + __expf(-(acc + bb)));
        p[v] = pv;
        const float tt = tv[u];
        const float pb = pv > 0.5f ? 1.f : 0.f, tb = tt > 0.5f ? 1.f : 0.f;
        s[0] += tt * pv;
        s[1] += tt;
        s[2] += pv;
        s[3] += tb * pb;
        s[4] += tb;
        s[5] += pb;
        s[6] += (tt == pb) ? 1.f : 0.f;
        if (xs.weight != 0.f) s[7] += xent_voxel_weight(xs, v) * xent_term(tt, pv);
      }
    }
  }
  __shared__ double shd[kThreads / 32][8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    double wsum = (double)s[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
    if (lane == 0) shd[warp][k] = wsum;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    double a = 0.0;
    for (int wi = 0; wi < kThreads / 32; ++wi) a += shd[wi][threadIdx.x];
    part[(int64_t)blockIdx.x * 8 + threadIdx.x] = a;
  }
}

// Thread-per-voxel form of the two head kernels for C in {16, 32, 64} (every model of the BASELINE configs): one thread reads
// its voxel's C channels with C/8 16-byte loads (the sectors a warp's loads share are consumed back to back out of L1),
// keeps the weights in registers, and - in the training form - updates the loss statistics for its own voxel. The
// lanes-per-voxel kernels above spend 13.7 warp instructions per voxel (shuffle folds, and the sigmoid / statistics
// section runs with one active lane in C/8); this one about 3: they were 60 % issue-bound at 3.3-4.3 TB/s.
template <int C, bool DICE>
__global__ void __launch_bounds__(kThreads) head_fwd_tpv_kernel(const bf16* __restrict__ x, const float* __restrict__ w,
                                                                const float* __restrict__ b, const float* __restrict__ t,
                                                                float* __restrict__ p, int64_t voxels, int apply_sigmoid,
                                                                double* __restrict__ part, XentSpec xs) {
  FM_PDL_SYNC();
  float wv[C];
#pragma unroll
  for (int i = 0; i < C; ++i) wv[i] = __ldg(w + i);
  const float bb = __ldg(b);
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < voxels; v += (int64_t)gridDim.x * blockDim.x) {
    uint4 r[C / 8];
    const uint4* src = reinterpret_cast<const uint4*>(x + v * C);
#pragma unroll
    for (int j = 0; j < C / 8; ++j) r[j] = __ldg(src + j);
    const float tt = DICE ? __ldg(t + v) : 0.f;
    float acc = bb;
#pragma unroll
    for (int j = 0; j < C / 8; ++j) {
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r[j]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        acc += f.x * wv[j * 8 + 2 * i] + f.y * wv[j * 8 + 2 * i + 1];
      }
    }
    const float pv = (DICE || apply_sigmoid) ? 1.f / (1.f + __expf(-acc)) : acc;
    p[v] = pv;
    if (DICE) {
      const float pb = pv > 0.5f ? 1.f : 0.f, tb = tt > 0.5f ? 1.f : 0.f;
      s[0] += tt * pv;
      s[1] += tt;
      s[2] += pv;
      s[3] += tb * pb;
      s[4] += tb;
      s[5] += pb;
      s[6] += (tt == pb) ? 1.f : 0.f;
      if (xs.weight != 0.f) s[7] += xent_voxel_weight(xs, v) * xent_term(tt, pv);
    }
  }
  if (DICE) {
    __shared__ double shd[kThreads / 32][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      double wsum = (double)s[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
      if (lane == 0) shd[warp][k] = wsum;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
      double a = 0.0;
      for (int wi = 0; wi < kThreads / 32; ++wi) a += shd[wi][threadIdx.x];
      part[(int64_t)blockIdx.x * 8 + threadIdx.x] = a;
    }
  }
}

// Multi-label form of head_fwd_tpv_kernel (1 < L <= kMaxLabels outputs per voxel, w = [L][C], p / t = [voxel][L]): the
// voxel's C channels are read once, and label l accumulates them exactly as the one-label kernel does with w + l C and
// b[l], so each label's map is bit-identical to a one-label head with that label's weights. The weights live in shared
// memory; the label loops are unrolled to kMaxLabels behind a guard so the per-label sums stay in registers. The
// training form writes 8 + 3 L partials per block (write_label_partials), folded by dice_final_labels_kernel.
template <int C, bool DICE>
__global__ void __launch_bounds__(kThreads) head_fwd_labels_kernel(const bf16* __restrict__ x, const float* __restrict__ w,
                                                                   const float* __restrict__ b,
                                                                   const float* __restrict__ t, float* __restrict__ p,
                                                                   int64_t voxels, int L, int apply_sigmoid,
                                                                   double* __restrict__ part, XentSpec xs) {
  FM_PDL_SYNC();
  __shared__ float wsh[kMaxLabels * C];
  __shared__ float bsh[kMaxLabels];
  for (int i = threadIdx.x; i < L * C; i += blockDim.x) wsh[i] = __ldg(w + i);
  if ((int)threadIdx.x < L) bsh[threadIdx.x] = __ldg(b + threadIdx.x);
  __syncthreads();
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float sl[3 * kMaxLabels];
#pragma unroll
  for (int i = 0; i < 3 * kMaxLabels; ++i) sl[i] = 0.f;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < voxels; v += (int64_t)gridDim.x * blockDim.x) {
    uint4 r[C / 8];
    const uint4* src = reinterpret_cast<const uint4*>(x + v * C);
#pragma unroll
    for (int j = 0; j < C / 8; ++j) r[j] = __ldg(src + j);
#pragma unroll
    for (int l = 0; l < kMaxLabels; ++l) {
      if (l >= L) break;
      const float* wl = wsh + l * C;
      float acc = bsh[l];
#pragma unroll
      for (int j = 0; j < C / 8; ++j) {
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r[j]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 f = __bfloat1622float2(h[i]);
          acc += f.x * wl[j * 8 + 2 * i] + f.y * wl[j * 8 + 2 * i + 1];
        }
      }
      const float pv = (DICE || apply_sigmoid) ? 1.f / (1.f + __expf(-acc)) : acc;
      const int64_t e = v * L + l;
      p[e] = pv;
      if (DICE) {
        const float tt = __ldg(t + e);
        const float pb = pv > 0.5f ? 1.f : 0.f, tb = tt > 0.5f ? 1.f : 0.f;
        s[0] += tt * pv;
        s[1] += tt;
        s[2] += pv;
        s[3] += tb * pb;
        s[4] += tb;
        s[5] += pb;
        s[6] += (tt == pb) ? 1.f : 0.f;
        if (xs.weight != 0.f) s[7] += xent_voxel_weight(xs, e) * xent_term(tt, pv);
        sl[3 * l] += tt * pv;
        sl[3 * l + 1] += tt;
        sl[3 * l + 2] += pv;
      }
    }
  }
  if (DICE) write_label_partials<kThreads>(s, sl, L, part);
}

// Multi-label inference form of head_fwd_kernel (C/8 lanes per voxel) for the channel counts the thread-per-voxel form
// does not take (the Isensee heads of 128 or more channels): label l accumulates and shuffle-reduces exactly as the
// one-label kernel does with w + l C and b[l].
__global__ void __launch_bounds__(kThreads) head_fwd_labels_lpv_kernel(const bf16* __restrict__ x,
                                                                       const float* __restrict__ w,
                                                                       const float* __restrict__ b,
                                                                       float* __restrict__ p, int64_t voxels, int C,
                                                                       int L, int apply_sigmoid) {
  FM_PDL_SYNC();
  const int lpv = C >> 3;
  const int sub = threadIdx.x % lpv;
  const int64_t vpb = blockDim.x / lpv;
  constexpr int U = 4;
  for (int64_t base = (int64_t)blockIdx.x * vpb * U; base < voxels; base += (int64_t)gridDim.x * vpb * U) {
    uint4 t[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = base + u * vpb + threadIdx.x / lpv;
      t[u] = v < voxels ? __ldg(reinterpret_cast<const uint4*>(x + v * C + sub * 8)) : make_uint4(0u, 0u, 0u, 0u);
    }
    for (int l = 0; l < L; ++l) {
      float wv[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) wv[i] = __ldg(w + l * C + sub * 8 + i);
      const float bb = __ldg(b + l);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t v = base + u * vpb + threadIdx.x / lpv;
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t[u]);
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 f = __bfloat1622float2(h[i]);
          acc += f.x * wv[2 * i] + f.y * wv[2 * i + 1];
        }
        for (int s = lpv >> 1; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
        if (sub == 0 && v < voxels) p[v * L + l] = apply_sigmoid ? 1.f / (1.f + __expf(-(acc + bb))) : acc + bb;
      }
    }
  }
}

// Multi-label head backward (1 < L <= kMaxLabels, C a power of two in [8, 256]): C/8 lanes per voxel as in
// head_bwd_kernel; g[l] is formed from p and t per label with the global sums, dx[c] = sum_l g[l] w[l][c] (labels in
// ascending order), and each thread keeps dw / db partials for all labels of its 8 channels.
__global__ void __launch_bounds__(kThreads) head_bwd_labels_kernel(const bf16* __restrict__ x,
                                                                   const float* __restrict__ dz,
                                                                   const float* __restrict__ w, bf16* __restrict__ dx,
                                                                   float* __restrict__ dw, float* __restrict__ db,
                                                                   int64_t voxels, int C, int L, int mode,
                                                                   const float* __restrict__ pt,
                                                                   const double* __restrict__ sums, XentSpec xs) {
  FM_PDL_SYNC();
  __shared__ float wsh[kMaxLabels * 256];
  for (int i = threadIdx.x; i < L * C; i += blockDim.x) wsh[i] = __ldg(w + i);
  float ga = 0.f, gbc = 0.f, xc = 0.f;
  if (pt != nullptr) {
    const double I = sums[0], S = sums[1] + sums[2] + 1.0;
    ga = (float)(-2.0 / S);
    gbc = (float)((2.0 * I + 1.0) / (S * S));
    if (xs.weight != 0.f) xc = (float)((double)xs.weight / sums[7]);
  }
  const int lpv = C >> 3;
  const int sub = threadIdx.x % lpv;
  float gw[kMaxLabels][8], gb[kMaxLabels];
#pragma unroll
  for (int l = 0; l < kMaxLabels; ++l) {
    gb[l] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) gw[l][i] = 0.f;
  }
  __syncthreads();
  const int64_t vstride = (int64_t)gridDim.x * (blockDim.x / lpv);
  for (int64_t v = (int64_t)blockIdx.x * (blockDim.x / lpv) + threadIdx.x / lpv; v < voxels; v += vstride) {
    const uint4 xr = __ldg(reinterpret_cast<const uint4*>(x + v * C + sub * 8));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&xr);
    float f[8], d[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 q = __bfloat1622float2(h[i]);
      f[2 * i] = q.x;
      f[2 * i + 1] = q.y;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = 0.f;
#pragma unroll
    for (int l = 0; l < kMaxLabels; ++l) {
      if (l >= L) break;
      const int64_t e = v * L + l;
      float g = __ldg(dz + e);
      if (pt != nullptr) {
        const float p0 = g, tv = __ldg(pt + e);
        g = (ga * tv + gbc) * p0 * (1.f - p0);
        if (xc != 0.f) g += xc * xent_voxel_weight(xs, e) * xent_grad(tv, p0);
      }
      const float* wl = wsh + l * C + sub * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        gw[l][i] += g * f[i];
        d[i] += g * wl[i];
      }
      if (sub == 0) gb[l] += g;
    }
    uint4 o;
    __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      oh[i] = __floats2bfloat162_rn(mode != 0 || f[2 * i] > 0.f ? d[2 * i] : 0.f,
                                    mode != 0 || f[2 * i + 1] > 0.f ? d[2 * i + 1] : 0.f);
    if (mode == 2) {
      const uint4 prev = *reinterpret_cast<const uint4*>(dx + v * C + sub * 8);
      const __nv_bfloat162* ph = reinterpret_cast<const __nv_bfloat162*>(&prev);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 a = __bfloat1622float2(ph[i]), c = __bfloat1622float2(oh[i]);
        oh[i] = __floats2bfloat162_rn(a.x + c.x, a.y + c.y);
      }
    }
    *reinterpret_cast<uint4*>(dx + v * C + sub * 8) = o;
  }
  // block reduction, one label at a time: threads with equal `sub` hold partial sums of the same 8 channels
  __shared__ float sh[kThreads][9];
#pragma unroll
  for (int l = 0; l < kMaxLabels; ++l) {
    if (l >= L) break;
#pragma unroll
    for (int i = 0; i < 8; ++i) sh[threadIdx.x][i] = gw[l][i];
    sh[threadIdx.x][8] = gb[l];
    __syncthreads();
    if ((int)threadIdx.x < lpv) {
      float a[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int tt = threadIdx.x; tt < kThreads; tt += lpv)
#pragma unroll
        for (int i = 0; i < 9; ++i) a[i] += sh[tt][i];
#pragma unroll
      for (int i = 0; i < 8; ++i) atomicAdd(dw + l * C + threadIdx.x * 8 + i, a[i]);
      if (threadIdx.x == 0) atomicAdd(db + l, a[8]);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kThreads) head_bwd_kernel(const bf16* __restrict__ x,
                                                            const float* __restrict__ dz,
                                                            const float* __restrict__ w,
                                                            bf16* __restrict__ dx,
                                                            float* __restrict__ dw,
                                                            float* __restrict__ db, int64_t voxels,
                                                            int C, int mode, const float* __restrict__ pt,
                                                            const double* __restrict__ sums, XentSpec xs) {
  FM_PDL_SYNC();
  // mode 0: dx = g*w masked by ReLU(x) (plain U-Net head); 1: dx = g*w; 2: dx += g*w (Isensee seg heads)
  // `pt` != NULL: `dz` holds the probabilities p, `pt` the targets t and g = dL/dz is formed here - the closed-form
  // gradient of L = -dice(t, sigmoid(z)) (metrics.py:11-15,31-32, smooth = 1) with the GLOBAL sums - instead of being
  // read from a dz tensor written by a separate dice_bwd launch
  float ga = 0.f, gbc = 0.f, xc = 0.f;
  if (pt != nullptr) {
    const double I = sums[0], S = sums[1] + sums[2] + 1.0;
    ga = (float)(-2.0 / S);
    gbc = (float)((2.0 * I + 1.0) / (S * S));
    // dice_and_xent: + weight / count * w_i * (p_i - t_i) (metrics.py:68-78 through the sigmoid)
    if (xs.weight != 0.f) xc = (float)((double)xs.weight / sums[7]);
  }
  const int lpv = C >> 3;
  const int sub = threadIdx.x % lpv;
  float wv[8], gw[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    wv[i] = __ldg(w + sub * 8 + i);
    gw[i] = 0.f;
  }
  float gb = 0.f;
  const int64_t vstride = (int64_t)gridDim.x * (blockDim.x / lpv);
  constexpr int U = 4;  // voxels per trip: all loads of a trip are issued before the first is consumed
  for (int64_t vb = (int64_t)blockIdx.x * (blockDim.x / lpv) + threadIdx.x / lpv; vb < voxels; vb += U * vstride) {
    float gg[U], tv[U];
    uint4 tt[U];
    bool has[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t v = vb + u * vstride;
      has[u] = v < voxels;
      gg[u] = has[u] ? __ldg(dz + v) : 0.f;
      tv[u] = (pt != nullptr && has[u]) ? __ldg(pt + v) : 0.f;
      tt[u] = has[u] ? __ldg(reinterpret_cast<const uint4*>(x + v * C + sub * 8)) : make_uint4(0u, 0u, 0u, 0u);
    }
    if (pt != nullptr) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float p0 = gg[u];
        gg[u] = (ga * tv[u] + gbc) * p0 * (1.f - p0);
        if (xc != 0.f && has[u]) gg[u] += xc * xent_voxel_weight(xs, vb + u * vstride) * xent_grad(tv[u], p0);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!has[u]) break;
      const int64_t v = vb + u * vstride;
      const float g = gg[u];
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&tt[u]);
      uint4 o;
      __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        gw[2 * i] += g * f.x;
        gw[2 * i + 1] += g * f.y;
        oh[i] = __floats2bfloat162_rn(mode != 0 || f.x > 0.f ? g * wv[2 * i] : 0.f,
                                      mode != 0 || f.y > 0.f ? g * wv[2 * i + 1] : 0.f);
      }
      if (sub == 0) gb += g;
      if (mode == 2) {
        const uint4 prev = *reinterpret_cast<const uint4*>(dx + v * C + sub * 8);
        const __nv_bfloat162* ph = reinterpret_cast<const __nv_bfloat162*>(&prev);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 a = __bfloat1622float2(ph[i]), b = __bfloat1622float2(oh[i]);
          oh[i] = __floats2bfloat162_rn(a.x + b.x, a.y + b.y);
        }
      }
      *reinterpret_cast<uint4*>(dx + v * C + sub * 8) = o;
    }
  }
  // block reduction: threads with equal `sub` hold partial sums of the same 8 channels
  __shared__ float sh[kThreads][9];
#pragma unroll
  for (int i = 0; i < 8; ++i) sh[threadIdx.x][i] = gw[i];
  sh[threadIdx.x][8] = gb;
  __syncthreads();
  if ((int)threadIdx.x < lpv) {
    float a[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int tt = threadIdx.x; tt < kThreads; tt += lpv)
#pragma unroll
      for (int i = 0; i < 9; ++i) a[i] += sh[tt][i];
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(dw + threadIdx.x * 8 + i, a[i]);
    if (threadIdx.x == 0) atomicAdd(db, a[8]);
  }
}

// --------------------------------------------------------------------------------------------
// weight repack: master fp32 [Cout][taps][Ct] -> bf16 fprop pack (same order) and the dgrad packs
// Wd_s[ci][tap'][co] = W[co][taps-1-tap'][cofs_s + ci]  (spatially flipped, in/out swapped)
// --------------------------------------------------------------------------------------------
__global__ void repack_weights_kernel(const float* __restrict__ w, bf16* __restrict__ wf,
                                      bf16* __restrict__ wd0, bf16* __restrict__ wd1, int Cout,
                                      int taps, int C1, int C2) {
  const int Ct = C1 + C2;
  const int64_t total = (int64_t)Cout * taps * Ct;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int c = (int)(g % Ct);
  const int tap = (int)((g / Ct) % taps);
  const int co = (int)(g / ((int64_t)Ct * taps));
  const bf16 v = __float2bfloat16(w[g]);
  if (wf) wf[g] = v;
  const int tf = taps - 1 - tap;
  if (c < C1) {
    if (wd0) wd0[((int64_t)c * taps + tf) * Cout + co] = v;
  } else {
    if (wd1) wd1[((int64_t)(c - C1) * taps + tf) * Cout + co] = v;
  }
}

// One block = one 32 (co) x 32 (c) tile of one tap of one layer: the master weights are read along c (coalesced), the
// fprop pack and the marching fprop pack are written along c, and - through a shared-memory transpose - the dgrad pack
// and the marching dgrad pack along co. (The first version wrote the transposed packs as scattered 2-byte stores:
// 11 % of the HBM roofline.)
__global__ void __launch_bounds__(kThreads) repack_all_kernel(const float* __restrict__ params,
                                                              const RepackDesc* __restrict__ tab, int nlayers) {
  FM_PDL_SYNC();
  __shared__ float tile[32][33];
  int li = 0;
  while (li + 1 < nlayers && (int)blockIdx.x >= tab[li + 1].block0) ++li;
  const RepackDesc d = tab[li];
  const int Ct = d.c1 + d.c2;
  const int nct = (Ct + 31) >> 5, ncot = (d.cout + 31) >> 5;
  int t = blockIdx.x - d.block0;
  const int ctile = t % nct;
  t /= nct;
  const int cotile = t % ncot;
  const int tap = t / ncot;
  const int tf = d.taps - 1 - tap;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  {
    const int c = ctile * 32 + tx;
    const bool second = c >= d.c1;
    const int cs = second ? c - d.c1 : c;
    bf16* mf = second ? d.mf1 : d.mf0;
    const int kcf = second ? d.kcf1 : d.kcf0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int co = cotile * 32 + ty + 8 * r;
      float v = 0.f;
      if (c < Ct && co < d.cout) {
        const int64_t g = ((int64_t)co * d.taps + tap) * Ct + c;
        v = params[d.w_off + g];
        const bf16 b = __float2bfloat16(v);
        if (d.wf) d.wf[g] = b;
        if (mf) mf[march_pack_index(second ? d.c2 : d.c1, d.srf, co, tap, cs, kcf)] = b;
      }
      tile[ty + 8 * r][tx] = v;
    }
  }
  __syncthreads();
  {
    const int co = cotile * 32 + tx;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int c = ctile * 32 + ty + 8 * r;
      if (c >= Ct || co >= d.cout) continue;
      const bool second = c >= d.c1;
      const int cs = second ? c - d.c1 : c;
      const bf16 b = __float2bfloat16(tile[tx][ty + 8 * r]);
      bf16* wd = second ? d.wd1 : d.wd0;
      if (wd) wd[((int64_t)cs * d.taps + tf) * d.cout + co] = b;
      bf16* md = second ? d.md1 : d.md0;
      if (md) md[march_pack_index(d.cout, second ? d.srd1 : d.srd0, cs, tf, co, second ? d.kcd1 : d.kcd0)] = b;
    }
  }
}

inline int grid_for(int64_t work_items, int cap = 1 << 30) {
  int64_t b = ceil_div64(work_items, kThreads);
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace

int k_conv3d_simt_fprop(fm_ctx* ctx, const void* x, int x_is_f32, const bf16* x2, const bf16* w_packed,
                        const float* bias, bf16* y, float* y_f32, int N, int X, int Y, int Z, int C1,
                        int C2, int Cout, int ksize, int relu, const bf16* mask) {
  if (x_is_f32 && C1 == 1 && C2 == 0 && ksize == 3 && y != nullptr && y_f32 == nullptr &&
      mask == nullptr && bias != nullptr && (Cout == 16 || Cout == 32)) {
    if (conv_first_tc_supported(X, Y, Z, Cout))  // im2col tile in shared memory + tcgen05 (conv_first_tc.cu)
      return k_conv3d_first_tc(ctx, (const float*)x, w_packed, bias, y, N, X, Y, Z, Cout, relu);
    const int64_t nvox = (int64_t)N * X * Y * Z;
    const int grid = grid_for(nvox, ctx->num_sms * 16);
    ProfScope prof(ctx, "conv3d_first", 2.0 * 27 * Cout * (double)nvox, (double)nvox * (4.0 + 2.0 * Cout));
    if (Cout == 16)
      FM_CUDA(launch_pdl(conv3d_first_kernel<16>, dim3(grid), dim3(kThreads), 0, ctx->stream, (const float*)x, w_packed, bias, y,
                                                                 N, X, Y, Z, relu));
    else
      FM_CUDA(launch_pdl(conv3d_first_kernel<32>, dim3(grid), dim3(kThreads), 0, ctx->stream, (const float*)x, w_packed, bias, y,
                                                                 N, X, Y, Z, relu));
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  const int64_t total = (int64_t)N * X * Y * Z * Cout;
  ProfScope prof(ctx, "conv3d_simt_fprop", 2.0 * kext_taps(ksize) * (C1 + C2) * (double)total, 0.0);
  conv3d_simt_fprop_kernel<<<grid_for(total), kThreads, 0, ctx->stream>>>(
      x, x_is_f32, x2, w_packed, bias, y, y_f32, N, X, Y, Z, C1, C2, Cout, ksize, relu, mask);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_conv3d_simt_wgrad(fm_ctx* ctx, const void* x, int x_is_f32, const bf16* dy, float* dw_packed,
                        int N, int X, int Y, int Z, int Cin, int Cin_total, int cin_ofs, int Cout,
                        int ksize) {
  const int taps = kext_taps(ksize);
  const int64_t n_out = (int64_t)Cout * taps * Cin;
  const int64_t nvox = (int64_t)N * X * Y * Z;
  if (x_is_f32 && Cin == 1 && Cin_total == 1 && cin_ofs == 0 && ksize == 3 && (Cout == 16 || Cout == 32) &&
      nvox < (int64_t)1 << 31 && Z % 2 == 0) {
    if (conv_first_tc_supported(X, Y, Z, Cout))  // im2col tile in shared memory + tcgen05 (conv_first_tc.cu)
      return k_conv3d_first_tc_wgrad(ctx, (const float*)x, dy, dw_packed, N, X, Y, Z, Cout);
    ProfScope prof(ctx, "conv3d_first_wgrad", 2.0 * 27 * Cout * (double)nvox, (double)nvox * (4.0 + 2.0 * Cout));
    const int grid = (int)std::min<int64_t>(ceil_div64(nvox, 64), (int64_t)ctx->num_sms * (Cout == 16 ? 4 : 2));
    if (Cout == 16)
      FM_CUDA(launch_pdl(conv3d_first_wgrad_kernel<16>, dim3(grid), dim3(32 * 9), 0, ctx->stream, (const float*)x, dy, dw_packed, N, X, Y, Z));
    else
      FM_CUDA(launch_pdl(conv3d_first_wgrad_kernel<32>, dim3(grid), dim3(32 * 18), 0, ctx->stream, (const float*)x, dy, dw_packed, N, X, Y, Z));
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  // enough voxel chunks that small layers (the 432 outputs of the first layer) still fill the GPU
  int64_t chunks = std::max<int64_t>(1, (int64_t)ctx->num_sms * 64 / std::max<int64_t>(1, n_out / 8));
  chunks = std::min<int64_t>(chunks, std::max<int64_t>(1, nvox / 1024));
  chunks = std::min<int64_t>(chunks, 65535);
  const int64_t vpc = ceil_div64(nvox, chunks);
  dim3 grid((unsigned)ceil_div64(n_out, kThreads / 32), (unsigned)ceil_div64(nvox, vpc));
  ProfScope prof(ctx, "conv3d_simt_wgrad", 2.0 * (double)n_out * (double)nvox, 0.0);
  conv3d_simt_wgrad_kernel<<<grid, kThreads, 0, ctx->stream>>>(x, x_is_f32, dy, dw_packed, N, X, Y, Z,
                                                              Cin, Cin_total, cin_ofs, Cout, ksize,
                                                              vpc);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_bias_grad(fm_ctx* ctx, const bf16* dy, float* db, int64_t voxels, int C) {
  FM_CHECK(C >= 1 && C <= 1024, FM_EINVAL, "bias_grad: C=%d unsupported", C);
  if (C >= 8 && C <= 256 && (C & (C - 1)) == 0 && ((uintptr_t)dy & 15) == 0) {
    const int64_t nvec = voxels * (C / 8);
    const int64_t blocks = std::max<int64_t>(1, std::min<int64_t>((int64_t)ctx->num_sms * 8, nvec / (kThreads * 4)));
    ProfScope prof(ctx, "bias_grad", 0.0, (double)voxels * C * 2.0);
    FM_CUDA(launch_pdl(bias_grad_vec_kernel, dim3((unsigned)blocks), dim3(kThreads), 0, ctx->stream,
                       reinterpret_cast<const uint4*>(dy), db, nvec, C / 8));
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  const int lanes = std::max(1, kThreads / C);
  const int threads = C * lanes;
  int64_t blocks = std::min<int64_t>((int64_t)ctx->num_sms * 8, std::max<int64_t>(1, voxels / (lanes * 8)));
  const int64_t vpb = ceil_div64(voxels, blocks);
  blocks = ceil_div64(voxels, vpb);
  ProfScope prof(ctx, "bias_grad", 0.0, (double)voxels * C * 2.0);
  bias_grad_kernel<<<(unsigned)blocks, threads, threads * sizeof(float), ctx->stream>>>(dy, db, voxels,
                                                                                       C, vpb);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// the multi-label head forward (L > 1); with `t` the training form, whose partials land in ctx->red_scratch
static int head_fwd_labels(fm_ctx* ctx, const bf16* x, const float* w, const float* b, const float* t, float* p,
                           int64_t voxels, int C, int L, int apply_sigmoid, XentSpec xs, int* grid_out) {
  FM_CHECK(L >= 2 && L <= kMaxLabels, FM_EINVAL, "head: %d labels (1 .. %d)", L, kMaxLabels);
  FM_CHECK(C >= 8 && C <= 256 && (C & (C - 1)) == 0, FM_EINVAL,
           "head: channel count %d must be a power of two in [8,256]", C);
  if (!t && !(C >= 16 && C <= 64)) {  // inference form, lanes-per-voxel
    const int64_t vpb = kThreads / (C / 8);
    const int grid = (int)std::min<int64_t>(ceil_div64(voxels, vpb), (int64_t)ctx->num_sms * 32);
    ProfScope prof(ctx, "head_fwd_labels", 2.0 * C * L * (double)voxels, (double)voxels * (C * 2.0 + L * 4.0));
    FM_CUDA(launch_pdl(head_fwd_labels_lpv_kernel, dim3(grid), dim3(kThreads), 0, ctx->stream, x, w, b, p, voxels, C, L,
                       apply_sigmoid));
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  FM_CHECK(C == 16 || C == 32 || C == 64, FM_EINVAL,
           "head: the training form of %d labels needs 16, 32 or 64 input channels, not %d", L, C);
  // one partial row of 8 + 3 L doubles per block in the reduction scratch
  const int rows = kRedScratchRows * 8 / (8 + 3 * L);
  const int grid = (int)std::min<int64_t>(ceil_div64(voxels, kThreads), (int64_t)std::min(rows, 16 * ctx->num_sms));
  const bool dice = t != nullptr;
  ProfScope prof(ctx, dice ? "head_fwd_dice_labels" : "head_fwd_labels", 2.0 * C * L * (double)voxels,
                 (double)voxels * (C * 2.0 + L * (dice ? 8.0 : 4.0)));
  double* part = dice ? ctx->red_scratch : nullptr;
#define FM_HEAD_LABELS(CC)                                                                                           \
  if (C == CC) {                                                                                                     \
    if (dice)                                                                                                        \
      FM_CUDA(launch_pdl(head_fwd_labels_kernel<CC, true>, dim3(grid), dim3(kThreads), 0, ctx->stream, x, w, b, t, p, \
                         voxels, L, 1, part, xs));                                                                   \
    else                                                                                                             \
      FM_CUDA(launch_pdl(head_fwd_labels_kernel<CC, false>, dim3(grid), dim3(kThreads), 0, ctx->stream, x, w, b, t,   \
                         p, voxels, L, apply_sigmoid, part, xs));                                                    \
  }
  FM_HEAD_LABELS(16)
  FM_HEAD_LABELS(32)
  FM_HEAD_LABELS(64)
#undef FM_HEAD_LABELS
  FM_LAUNCH_OK(ctx);
  if (grid_out) *grid_out = grid;
  return FM_OK;
}

int k_head_fwd(fm_ctx* ctx, const bf16* x, const float* w, const float* b, float* p, int64_t voxels,
               int C, int apply_sigmoid, int L) {
  if (L != 1) return head_fwd_labels(ctx, x, w, b, nullptr, p, voxels, C, L, apply_sigmoid, XentSpec(), nullptr);
  FM_CHECK(C >= 8 && C <= 256 && (C & (C - 1)) == 0, FM_EINVAL,
           "head: channel count %d must be a power of two in [8,256]", C);
  const int lpv = C / 8;
  const int64_t vpb = kThreads / lpv;
  const int grid = (int)std::min<int64_t>(ceil_div64(voxels, vpb), (int64_t)ctx->num_sms * 32);
  ProfScope prof(ctx, "head_fwd", 2.0 * C * (double)voxels, (double)voxels * (C * 2.0 + 4.0));
  if (C >= 16 && C <= 64) {  // thread-per-voxel form (instantiated for 16, 32 and 64 channels)
    const int g2 = (int)std::min<int64_t>(ceil_div64(voxels, kThreads), (int64_t)ctx->num_sms * 16);
    const XentSpec none;
    if (C == 16)
      FM_CUDA(launch_pdl(head_fwd_tpv_kernel<16, false>, dim3(g2), dim3(kThreads), 0, ctx->stream, x, w, b,
                         (const float*)nullptr, p, voxels, apply_sigmoid, (double*)nullptr, none));
    else if (C == 32)
      FM_CUDA(launch_pdl(head_fwd_tpv_kernel<32, false>, dim3(g2), dim3(kThreads), 0, ctx->stream, x, w, b,
                         (const float*)nullptr, p, voxels, apply_sigmoid, (double*)nullptr, none));
    else
      FM_CUDA(launch_pdl(head_fwd_tpv_kernel<64, false>, dim3(g2), dim3(kThreads), 0, ctx->stream, x, w, b,
                         (const float*)nullptr, p, voxels, apply_sigmoid, (double*)nullptr, none));
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  FM_CUDA(launch_pdl(head_fwd_kernel, dim3(grid), dim3(kThreads), 0, ctx->stream, x, w, b, p, voxels, C, apply_sigmoid));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// head + sigmoid + Dice / VOD / accuracy partial sums in one pass; `sums` receives the 8 folded statistics
int k_head_fwd_dice(fm_ctx* ctx, const bf16* x, const float* w, const float* b, const float* t, float* p,
                    int64_t voxels, int C, double* sums, XentSpec xs, int L) {
  if (L != 1) {
    int grid = 0;
    FM_TRY(head_fwd_labels(ctx, x, w, b, t, p, voxels, C, L, 1, xs, &grid));
    return k_dice_finalize_labels(ctx, grid, (double)voxels * L, sums, L);
  }
  FM_CHECK(C >= 8 && C <= 256 && (C & (C - 1)) == 0, FM_EINVAL,
           "head: channel count %d must be a power of two in [8,256]", C);
  const int lpv = C / 8;
  const int64_t vpb = kThreads / lpv;
  // one wave of resident blocks (64 registers x 256 threads: 4 blocks per SM): a grid-stride kernel launched with 1024
  // blocks on 592 slots ran 1.73 waves, the second one three-quarters empty
  const int grid = (int)std::min<int64_t>(ceil_div64(voxels, vpb * 4), (int64_t)std::min(1024, 4 * ctx->num_sms));
  if (C >= 16 && C <= 64) {  // thread-per-voxel form; one partial row per block of the reduction scratch
    const int g2 = (int)std::min<int64_t>(ceil_div64(voxels, kThreads), (int64_t)std::min(kRedScratchRows, 16 * ctx->num_sms));
    {
      ProfScope prof(ctx, "head_fwd_dice", 2.0 * C * (double)voxels, (double)voxels * (C * 2.0 + 8.0));
      if (C == 16)
        FM_CUDA(launch_pdl(head_fwd_tpv_kernel<16, true>, dim3(g2), dim3(kThreads), 0, ctx->stream, x, w, b, t, p, voxels, 1,
                           ctx->red_scratch, xs));
      else if (C == 32)
        FM_CUDA(launch_pdl(head_fwd_tpv_kernel<32, true>, dim3(g2), dim3(kThreads), 0, ctx->stream, x, w, b, t, p, voxels, 1,
                           ctx->red_scratch, xs));
      else
        FM_CUDA(launch_pdl(head_fwd_tpv_kernel<64, true>, dim3(g2), dim3(kThreads), 0, ctx->stream, x, w, b, t, p, voxels, 1,
                           ctx->red_scratch, xs));
      FM_LAUNCH_OK(ctx);
    }
    return k_dice_finalize(ctx, g2, (double)voxels, sums);
  }
  {
    ProfScope prof(ctx, "head_fwd_dice", 2.0 * C * (double)voxels, (double)voxels * (C * 2.0 + 8.0));
    FM_CUDA(launch_pdl(head_fwd_dice_kernel, dim3(grid), dim3(kThreads), 0, ctx->stream, x, w, b, t, p, voxels, C,
                       ctx->red_scratch, xs));
    FM_LAUNCH_OK(ctx);
  }
  return k_dice_finalize(ctx, grid, (double)voxels, sums);
}

int k_head_bwd(fm_ctx* ctx, const bf16* x, const float* dz, const float* w, bf16* dx, float* dw,
               float* db, int64_t voxels, int C, int mode, const float* t, const double* sums, XentSpec xs, int L) {
  FM_CHECK(C >= 8 && C <= 256 && (C & (C - 1)) == 0, FM_EINVAL,
           "head_bwd: channel count %d must be a power of two in [8,256]", C);
  const int lpv = C / 8;
  const int64_t vpb = kThreads / lpv;
  const int grid = (int)std::min<int64_t>(ceil_div64(voxels, vpb), (int64_t)ctx->num_sms * 8);
  if (L != 1) {
    FM_CHECK(L >= 2 && L <= kMaxLabels, FM_EINVAL, "head_bwd: %d labels (1 .. %d)", L, kMaxLabels);
    ProfScope prof(ctx, t ? "head_bwd_dice_labels" : "head_bwd_labels", 4.0 * C * L * (double)voxels,
                   (double)voxels * (C * 4.0 + L * (t ? 8.0 : 4.0)));
    FM_CUDA(launch_pdl(head_bwd_labels_kernel, dim3(grid), dim3(kThreads), 0, ctx->stream, x, dz, w, dx, dw, db, voxels,
                       C, L, mode, t, sums, xs));
    FM_LAUNCH_OK(ctx);
    return FM_OK;
  }
  ProfScope prof(ctx, t ? "head_bwd_dice" : "head_bwd", 4.0 * C * (double)voxels,
                 (double)voxels * (C * 4.0 + (t ? 8.0 : 4.0)));
  FM_CUDA(launch_pdl(head_bwd_kernel, dim3(grid), dim3(kThreads), 0, ctx->stream, x, dz, w, dx, dw, db, voxels, C, mode, t,
                     sums, xs));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_repack_all(fm_ctx* ctx, const float* params, const RepackDesc* table_dev, int nlayers, int total_blocks,
                 double total_weights) {
  ProfScope prof(ctx, "repack_all", 0.0, total_weights * 12.0);
  FM_CUDA(launch_pdl(repack_all_kernel, dim3(total_blocks), dim3(kThreads), 0, ctx->stream, params, table_dev, nlayers));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_repack_weights(fm_ctx* ctx, const float* w, bf16* w_f, bf16* w_d0, bf16* w_d1, int Cout, int taps,
                     int C1, int C2) {
  const int64_t total = (int64_t)Cout * taps * (C1 + C2);
  ProfScope prof(ctx, "repack_weights", 0.0, (double)total * 8.0);
  repack_weights_kernel<<<grid_for(total), kThreads, 0, ctx->stream>>>(w, w_f, w_d0, w_d1, Cout, taps,
                                                                      C1, C2);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
