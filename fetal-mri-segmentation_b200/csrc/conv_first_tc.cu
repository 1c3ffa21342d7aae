// conv_first_tc.cu — the first convolution of the network (Cin = 1, 3x3x3, Cout = 16 / 32) and its weight gradient on
// the tensor cores.
//
// With one input channel the GEMM K is only 27, so the layer is not "tensor-core shaped" and round 1 ran it as SIMT
// kernels: 432 (x Cout/16) fp32 FMAs per voxel, instruction-bound at 13 % (fprop) and 7.5 % (wgrad) of the HBM
// roofline that actually bounds it (4 B in + 2 Cout B out per voxel). Here four builder warps expand each tile of
// 128 voxels (16 y x 8 z of one x plane) into an im2col tile in shared memory - [128 voxels][64 taps] bf16, 128-byte
// swizzled rows, taps 27..63 zero - and ONE operand layout serves both directions:
//   fprop :  Y[v, co]   = act(sum_t A[v, t] W[co, t] + b[co])   A K-major   (M = 128 voxels, K = 32 taps: 2 MMAs)
//   wgrad :  dW[co, t]  = sum_v A[v, t] dY[v, co]                A MN-major  (M = taps, K = 128 voxels: 8 MMAs),
//            dY tile TMA-loaded as the MN-major B operand, accumulator resident in TMEM for the CTA's whole life.
// The volume is rounded to bf16 on the way into the tile (every other activation of the network is bf16 as well).
// Replaces: the first Conv3D of create_convolution_block (fetal_net/model/unet3d/unet.py:102) on the (1, X, Y, Z)
// input and its TF autodiff weight gradient.
#include <algorithm>

#include "tc_ptx.cuh"

using namespace tcp;

namespace {

constexpr int kFY = 16, kFZ = 8;          // tile: 16 (y) x 8 (z) voxels of one x plane = 128 GEMM rows
constexpr int kBuildWarps = 4;            // warps 0-3 build the im2col tile (one voxel row per thread)
constexpr int kThreadsF = 32 * (kBuildWarps + 1 + 4);  // + MMA / TMA warp 4, + epilogue warps 5-8
constexpr uint32_t kATile = 128u * 128u;  // 16 KB
constexpr int kABufs = 3;                 // im2col ring
constexpr int kDyRingF = 4;

struct alignas(64) FirstParams {
  CUtensorMap tmDY;  // wgrad: dY [N][X][Y][Z][Cout], box (Cout, 8, 16, 1, 1)
  const float* x;    // [N][X][Y][Z] fp32
  const bf16* w;     // packed [Cout][27]
  const float* bias;
  bf16* y;
  float* dw;         // [Cout][27] fp32 (atomics)
  int N, X, Y, Z, Cout, relu;
  int ty, tz, tiles;
};

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// The builders first stage the tile's input halo - 3 planes x 18 y x 10 z, zero outside the volume (= padding 'same'),
// rounded to bf16 - in shared memory (5 coalesced loads per thread, issued one tile ahead so their latency hides
// behind the previous tile's gather), then every thread assembles the im2col row of its voxel from 27 16-bit shared
// loads: ~100 instructions per voxel instead of the ~320 of gathering from global memory with bounds checks.
constexpr int kHZ = 12;                          // padded z pitch of the halo (10 used)
constexpr uint32_t kHaloBytes = 3u * 18u * kHZ * 2u;  // 1296 B
constexpr int kHaloPerThread = 5;                // 540 halo elements over 128 builder threads

__device__ __forceinline__ void halo_load(const FirstParams& p, int n, int x, int y0, int z0, int tid, float v[kHaloPerThread]) {
#pragma unroll
  for (int k = 0; k < kHaloPerThread; ++k) {
    const int e = tid + k * 128;
    const int kx = e / 180, rem = e % 180;
    const int yy = rem / 10, zz = rem % 10;
    const int xi = x + kx - 1, yi = y0 + yy - 1, zi = z0 + zz - 1;
    const bool ok = e < 540 && xi >= 0 && xi < p.X && yi >= 0 && yi < p.Y && zi >= 0 && zi < p.Z;
    v[k] = ok ? __ldg(p.x + (((int64_t)n * p.X + xi) * p.Y + yi) * p.Z + zi) : 0.f;
  }
}
__device__ __forceinline__ void halo_store(uint32_t halo, int tid, const float v[kHaloPerThread]) {
#pragma unroll
  for (int k = 0; k < kHaloPerThread; ++k) {
    const int e = tid + k * 128;
    if (e < 540) {
      const int kx = e / 180, rem = e % 180;
      const int yy = rem / 10, zz = rem % 10;
      const bf16 h = __float2bfloat16(v[k]);
      asm volatile("st.shared.u16 [%0], %1;" ::"r"(halo + (uint32_t)(((kx * 18 + yy) * kHZ + zz) * 2)),
                   "h"(*reinterpret_cast<const unsigned short*>(&h))
                   : "memory");
    }
  }
}
// im2col row of the voxel (ry, rz) of the tile from the staged halo into the 128-byte swizzled row `row` of the tile
// at `tile` (16-byte chunk index ^= row & 7); taps 27..31 zero
__device__ __forceinline__ void build_row(uint32_t halo, uint32_t tile, int row, int ry, int rz) {
  uint32_t h[28];
#pragma unroll
  for (int kx = 0; kx < 3; ++kx)
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const uint32_t a = halo + (uint32_t)(((kx * 18 + ry + ky) * kHZ + rz) * 2);
#pragma unroll
      for (int kz = 0; kz < 3; ++kz) {
        unsigned short u;
        asm volatile("ld.shared.u16 %0, [%1];" : "=h"(u) : "r"(a + 2u * (uint32_t)kz));
        h[(kx * 3 + ky) * 3 + kz] = u;
      }
    }
  h[27] = 0u;
  const uint32_t rbase = tile + (uint32_t)row * 128u;
  const uint32_t sw = (uint32_t)(row & 7);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t w4[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int t = 8 * c + 2 * j;
      w4[j] = t + 1 < 28 ? (h[t] | (h[t + 1] << 16)) : (t < 28 ? h[t] : 0u);
    }
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(rbase + (((uint32_t)c ^ sw) << 4)), "r"(w4[0]),
                 "r"(w4[1]), "r"(w4[2]), "r"(w4[3])
                 : "memory");
  }
}

__device__ __forceinline__ void decode_tile(const FirstParams& p, int tile, int& n, int& x, int& y0, int& z0) {
  const int iz = tile % p.tz;
  int t = tile / p.tz;
  const int iy = t % p.ty;
  t /= p.ty;
  x = t % p.X;
  n = t / p.X;
  y0 = iy * kFY;
  z0 = iz * kFZ;
}

// MODE 0: fprop, MODE 1: wgrad
template <int MODE>
__global__ void __launch_bounds__(kThreadsF, 1) conv3d_first_tc_kernel(const __grid_constant__ FirstParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // smem: kABufs im2col tiles + one always-zero tile (the second 64-row M block of the last ring slot in wgrad), then
  // the weight tile (fprop: [Cout][64 taps], 128-byte rows) or the dY ring (wgrad: kDyRingF x [128][Cout]), barriers
  const uint32_t a_base = smem0;
  const uint32_t w_base = a_base + (uint32_t)(kABufs + 1) * kATile;
  const uint32_t dy_tile = 128u * (uint32_t)p.Cout * 2u;
  const uint32_t halo_base = w_base + (MODE == 0 ? 32u * 128u : (uint32_t)kDyRingF * dy_tile);  // two halo buffers
  const uint32_t bar0 = (halo_base + 2u * kHaloBytes + 15u) & ~15u;
  auto afull = [&](int b) { return bar0 + 8u * (uint32_t)b; };
  auto aempty = [&](int b) { return bar0 + 8u * (uint32_t)(kABufs + b); };
  auto tfull = [&](int a) { return bar0 + 8u * (uint32_t)(2 * kABufs + a); };
  auto tempty = [&](int a) { return bar0 + 8u * (uint32_t)(2 * kABufs + 2 + a); };
  auto dyfull = [&](int s) { return bar0 + 8u * (uint32_t)(2 * kABufs + 4 + s); };
  auto dyempty = [&](int s) { return bar0 + 8u * (uint32_t)(2 * kABufs + 4 + kDyRingF + s); };
  const uint32_t tmem_slot = bar0 + 8u * (uint32_t)(2 * kABufs + 4 + 2 * kDyRingF);
  const uint32_t tmem_cols = MODE == 0 ? (p.Cout == 16 ? 32u : 64u) : 32u;

  // zero every im2col buffer once: the builders only ever write the four chunks of taps 0..31
  for (uint32_t i = threadIdx.x; i < (uint32_t)(kABufs + 1) * kATile / 16u; i += blockDim.x)
    asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a_base + i * 16u), "r"(0u) : "memory");
  if (MODE == 0) {
    // weights [Cout][27] -> K-major tile [Cout rows][64 taps] (128-byte swizzled rows), taps 27..63 zero
    for (uint32_t i = threadIdx.x; i < 32u * 128u / 16u; i += blockDim.x)
      asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(w_base + i * 16u), "r"(0u) : "memory");
  }
  __syncthreads();
  if (MODE == 0) {
    for (int i = threadIdx.x; i < p.Cout * 27; i += blockDim.x) {
      const int co = i / 27, t = i % 27;
      const uint32_t addr = w_base + (uint32_t)co * 128u + ((((uint32_t)t >> 3) ^ (uint32_t)(co & 7)) << 4) + ((uint32_t)t & 7u) * 2u;
      const bf16 wv = p.w[i];
      asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(*reinterpret_cast<const unsigned short*>(&wv)) : "memory");
    }
  }
  if (warp == kBuildWarps) {
    if (lane == 0) {
      for (int b = 0; b < kABufs; ++b) {
        mbar_init(afull(b), kBuildWarps * 32);
        mbar_init(aempty(b), 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull(a), 1);
        mbar_init(tempty(a), 128);
      }
      for (int s = 0; s < kDyRingF; ++s) {
        mbar_init(dyfull(s), 1);
        mbar_init(dyempty(s), 1);
      }
      fence_barrier_init();
      if (MODE == 1) prefetch_tmap(&p.tmDY);
    }
    __syncwarp();
    tmem_alloc(tmem_slot, tmem_cols);
  }
  fence_async_smem();  // the zero fill and the weight tile are read by the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);

  if (warp_u < kBuildWarps) {
    // ===== builders: one im2col row per thread and tile =====
    pdl_wait();  // (wgrad: x is the network input, but dY's producer must have finished before ITS consumer starts)
    if (warp_u == 0) pdl_launch_dependents();
    const int row = threadIdx.x;  // 0..127 = y * 8 + z inside the tile
    const int ry = row / kFZ, rz = row % kFZ;
    float hv[kHaloPerThread];
    int n, x, y0, z0;
    if ((int)blockIdx.x < p.tiles) {
      decode_tile(p, blockIdx.x, n, x, y0, z0);
      halo_load(p, n, x, y0, z0, row, hv);
    }
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++it) {
      const uint32_t b = it % (uint32_t)kABufs, ph = (it / (uint32_t)kABufs) & 1u;
      const uint32_t halo = halo_base + (it & 1u) * kHaloBytes;
      halo_store(halo, row, hv);
      // the next tile's halo is already in flight while this one is gathered
      const int next = tile + gridDim.x;
      if (next < p.tiles) {
        decode_tile(p, next, n, x, y0, z0);
        halo_load(p, n, x, y0, z0, row, hv);
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // the four builder warps: halo complete (two buffers alternate)
      mbar_wait(aempty(b), ph ^ 1u);
      build_row(halo, a_base + b * kATile, row, ry, rz);
      fence_async_smem();
      mbar_arrive(afull(b));
    }
  } else if (warp_u == kBuildWarps) {
    // ===== MMA warp (and, for wgrad, the TMA producer of the dY tiles: both loops are interleaved) =====
    const uint32_t a_hi = desc_hi(1024u, layout_code(128));
    uint32_t it = 0;
    if (MODE == 0) {
      const uint32_t idesc = make_idesc(128, p.Cout, 0, 0);
      const uint32_t b_lo = desc_lo(w_base, 16u);
      for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++it) {
        const uint32_t b = it % (uint32_t)kABufs, ph = (it / (uint32_t)kABufs) & 1u;
        const uint32_t acc = it & 1u, acc_ph = (it >> 1) & 1u;
        mbar_wait(tempty(acc), acc_ph ^ 1u);
        mbar_wait(afull(b), ph);
        tc_fence_after();
        const uint32_t a_lo = desc_lo(a_base + b * kATile, 16u);
        const uint32_t d = tmem_base + acc * (uint32_t)p.Cout;
        umma_bf16_lh_elect(d, a_lo, a_hi, b_lo, a_hi, idesc, 0u);
        umma_bf16_lh_elect(d, a_lo + 2u, a_hi, b_lo + 2u, a_hi, idesc, 1u);
        umma_commit_elect(aempty(b));
        umma_commit_elect(tfull(acc));
      }
    } else {
      pdl_wait();
      const uint32_t idesc = make_idesc(128, p.Cout, 1, 1);
      const uint32_t b_row = (uint32_t)p.Cout * 2u, b_sbo = 8u * b_row;
      const uint32_t b_hi = desc_hi(b_sbo, layout_code((int)b_row));
      const uint32_t b_step = (2u * b_sbo) >> 4;
      // prime the dY ring
      int ahead = blockIdx.x;
      uint32_t issued = 0;
      auto issue_dy = [&]() {
        if (ahead >= p.tiles) return;
        const uint32_t s = issued % (uint32_t)kDyRingF, sph = (issued / (uint32_t)kDyRingF) & 1u;
        int n, x, y0, z0;
        decode_tile(p, ahead, n, x, y0, z0);
        mbar_wait(dyempty(s), sph ^ 1u);
        mbar_expect_tx_elect(dyfull(s), dy_tile);
        tma_load_5d_elect(w_base + s * dy_tile, &p.tmDY, dyfull(s), 0, z0, y0, x, n);
        ++issued;
        ahead += gridDim.x;
      };
      for (int i = 0; i < kDyRingF - 1; ++i) issue_dy();
      for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++it) {
        issue_dy();
        const uint32_t b = it % (uint32_t)kABufs, ph = (it / (uint32_t)kABufs) & 1u;
        const uint32_t s = it % (uint32_t)kDyRingF, sph = (it / (uint32_t)kDyRingF) & 1u;
        mbar_wait(afull(b), ph);
        mbar_wait(dyfull(s), sph);
        tc_fence_after();
        // A: M block 0 = this tile's 64 tap columns, M block 1 (LBO = one tile further) = whatever follows - its
        // accumulator rows 64..127 are never read
        uint32_t a_lo = desc_lo(a_base + b * kATile, kATile);
        uint32_t b_lo = desc_lo(w_base + s * dy_tile, dy_tile);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          umma_bf16_lh_elect(tmem_base, a_lo, a_hi, b_lo, b_hi, idesc, (it > 0 || ks > 0) ? 1u : 0u);
          a_lo += 128u;  // 16 voxels = two 8-row groups of 1024 B
          b_lo += b_step;
        }
        umma_commit_elect(aempty(b));
        umma_commit_elect(dyempty(s));
      }
      umma_commit_elect(tfull(0));
    }
  } else {
    // ===== epilogue warps =====
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    if (MODE == 0) {
      const int ry = row / kFZ, rz = row % kFZ;
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++it) {
        const uint32_t acc = it & 1u, acc_ph = (it >> 1) & 1u;
        int n, x, y0, z0;
        decode_tile(p, tile, n, x, y0, z0);
        const int64_t v = (((int64_t)n * p.X + x) * p.Y + y0 + ry) * p.Z + z0 + rz;
        mbar_wait(tfull(acc), acc_ph);
        tc_fence_after();
        for (int c16 = 0; c16 < p.Cout / 16; ++c16) {
          uint32_t r[16];
          tmem_ld16(lane_base + acc * (uint32_t)p.Cout + (uint32_t)c16 * 16u, r);
          tmem_ld_wait();
          uint4 o[2];
          __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(o);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float a = __uint_as_float(r[2 * j]) + __ldg(p.bias + c16 * 16 + 2 * j);
            float b = __uint_as_float(r[2 * j + 1]) + __ldg(p.bias + c16 * 16 + 2 * j + 1);
            if (p.relu) {
              a = fmaxf(a, 0.f);
              b = fmaxf(b, 0.f);
            }
            oh[j] = __floats2bfloat162_rn(a, b);
          }
          uint4* op = reinterpret_cast<uint4*>(p.y + v * p.Cout + c16 * 16);
          op[0] = o[0];
          op[1] = o[1];
        }
        tc_fence_before();
        mbar_arrive(tempty(acc));
      }
    } else {
      mbar_wait(tfull(0), 0);
      tc_fence_after();
      if ((int)blockIdx.x < p.tiles) {
        for (int c16 = 0; c16 < p.Cout / 16; ++c16) {
          uint32_t r[16];
          tmem_ld16(lane_base + (uint32_t)c16 * 16u, r);
          tmem_ld_wait();
          if (row < 27) {
#pragma unroll
            for (int j = 0; j < 16; ++j) atomicAdd(p.dw + (c16 * 16 + j) * 27 + row, __uint_as_float(r[j]));
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kBuildWarps) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

size_t first_smem(int mode, int Cout) {
  return (size_t)(kABufs + 1) * kATile + (mode == 0 ? 32u * 128u : (size_t)kDyRingF * 128u * Cout * 2u) + 2 * kHaloBytes +
         1024 + 256 + 16;
}

int fill(FirstParams& p, int N, int X, int Y, int Z, int Cout) {
  memset(&p, 0, sizeof(p));
  p.N = N;
  p.X = X;
  p.Y = Y;
  p.Z = Z;
  p.Cout = Cout;
  p.ty = Y / kFY;
  p.tz = Z / kFZ;
  p.tiles = N * X * p.ty * p.tz;
  return FM_OK;
}

}  // namespace

int conv_first_tc_supported(int X, int Y, int Z, int Cout) {
  return X > 0 && Y % kFY == 0 && Z % kFZ == 0 && (Cout == 16 || Cout == 32);
}

int k_conv3d_first_tc(fm_ctx* ctx, const float* x, const bf16* w_packed, const float* bias, bf16* y, int N, int X, int Y,
                      int Z, int Cout, int relu) {
  FM_CHECK(conv_first_tc_supported(X, Y, Z, Cout) && bias != nullptr, FM_EINVAL, "conv3d first tc: unsupported %dx%dx%d Cout=%d",
           X, Y, Z, Cout);
  FirstParams p;
  FM_TRY(fill(p, N, X, Y, Z, Cout));
  p.x = x;
  p.w = w_packed;
  p.bias = bias;
  p.y = y;
  p.relu = relu;
  const size_t smem = first_smem(0, Cout);
  static bool attr_set = false;
  if (!attr_set) {
    FM_CUDA(cudaFuncSetAttribute(conv3d_first_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)first_smem(0, 32)));
    attr_set = true;
  }
  const double nvox = (double)N * X * Y * Z;
  const int grid = std::min(p.tiles, 3 * ctx->num_sms);
  ProfScope prof(ctx, "conv3d_first", 2.0 * 27 * Cout * nvox, nvox * (4.0 + 2.0 * Cout));
  FM_CUDA(launch_pdl(conv3d_first_tc_kernel<0>, dim3(grid), dim3(kThreadsF), smem, ctx->stream, p));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// dw [Cout][27] fp32 += sum_v dY[v][co] * x[v + tap]
int k_conv3d_first_tc_wgrad(fm_ctx* ctx, const float* x, const bf16* dy, float* dw, int N, int X, int Y, int Z, int Cout) {
  FM_CHECK(conv_first_tc_supported(X, Y, Z, Cout), FM_EINVAL, "conv3d first tc wgrad: unsupported %dx%dx%d Cout=%d", X, Y, Z,
           Cout);
  FirstParams p;
  FM_TRY(fill(p, N, X, Y, Z, Cout));
  p.x = x;
  p.dw = dw;
  EncodeTiledFn enc = encode_tiled();
  FM_CHECK(enc != nullptr, FM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[5] = {(cuuint64_t)Cout, (cuuint64_t)Z, (cuuint64_t)Y, (cuuint64_t)X, (cuuint64_t)N};
  cuuint64_t strides[4] = {(cuuint64_t)Cout * 2, (cuuint64_t)Z * Cout * 2, (cuuint64_t)Y * Z * Cout * 2,
                           (cuuint64_t)X * Y * Z * Cout * 2};
  cuuint32_t box[5] = {(cuuint32_t)Cout, (cuuint32_t)kFZ, (cuuint32_t)kFY, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(&p.tmDY, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)dy, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_row_bytes(Cout * 2),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FM_CHECK(r == CUDA_SUCCESS, FM_ECUDA, "cuTensorMapEncodeTiled(first wgrad) failed: %d", (int)r);
  const size_t smem = first_smem(1, Cout);
  static bool attr_set = false;
  if (!attr_set) {
    FM_CUDA(cudaFuncSetAttribute(conv3d_first_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)first_smem(1, 32)));
    attr_set = true;
  }
  const double nvox = (double)N * X * Y * Z;
  const int grid = std::min(p.tiles, 2 * ctx->num_sms);
  ProfScope prof(ctx, "conv3d_first_wgrad", 2.0 * 27 * Cout * nvox, nvox * (4.0 + 2.0 * Cout));
  FM_CUDA(launch_pdl(conv3d_first_tc_kernel<1>, dim3(grid), dim3(kThreadsF), smem, ctx->stream, p));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
