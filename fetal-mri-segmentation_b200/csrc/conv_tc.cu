// conv_tc.cu — Conv3D as implicit GEMM on the 5th-generation tensor cores (sm_100a):
// tcgen05.mma with TMEM accumulators, operands staged in shared memory by TMA, mbarrier pipeline,
// warp-specialised (1 TMA producer warp, 1 MMA issuer warp, 4 epilogue warps), persistent CTAs.
//
//   fprop :  Y[v, co]  = act( sum_{tap, ci} X[v + shift(tap), ci] * W[co, tap, ci] + b[co] )
//            GEMM view  M = voxels (tile = 128-voxel box), N = Cout, K = taps * Cin.
//            A tile (128 voxels x KC channels, K-major) is ONE 5-D TMA box of the channels-last
//            activation tensor at tap-shifted coordinates — out-of-bounds rows are zero-filled by
//            TMA, which is exactly Keras' padding='same'. Up to two input tensors (K range split)
//            make the skip `concatenate([up, skip], axis=1)` (unet3d/unet.py:61) zero-copy.
//   dgrad :  the same kernel on dY with spatially flipped, in/out-swapped weights; the epilogue
//            applies the ReLU mask of the producing block instead of bias+ReLU.
//   wgrad :  dW[co, tap, ci] = sum_v dY[v, co] * X[v + shift(tap), ci]
//            GEMM view  M = (tap, ci) stacked to 128 rows, N = Cout, K = voxels. Both operands are
//            MN-major (the voxel axis is K and channels are contiguous in memory), accumulators for
//            up to 512/N tap groups stay in TMEM for the whole voxel range of the CTA (split-K over
//            CTAs, fp32 red.add into the gradient buffer).
//
// Keras call site replaced: Conv3D(n_filters, kernel, padding='same') in create_convolution_block
// (fetal_net/model/unet3d/unet.py:102) and its TF autodiff gradients.
#include <algorithm>

#include "tc_ptx.cuh"

namespace {

using namespace tcp;

constexpr int kTileM = 128;      // voxels per M tile == TMEM lanes
constexpr int kThreadsTc = 192;  // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr uint32_t kABytes = kTileM * 128;  // A slot: 128 rows x 128 B (largest swizzle span)

struct alignas(64) FpropParams {
  CUtensorMap tmA[2];  // activation sources (5-D: C, Z, Y, X, N)
  CUtensorMap tmW[2];  // packed weights per source (3-D: Cin_total, taps, Cout)
  int nsrc;
  int nchunks[2];  // C_s / KC_s
  int KC[2];       // channels per K chunk (16, 32 or 64)
  int wcofs[2];    // channel offset of the source inside the weight Cin axis
  int N, X, Y, Z;
  int bx, by, bz, tx, ty, tz;
  int m_tiles, n_tiles, block_n;
  int ksize, ntaps;
  int out_C, out_cofs;
  int relu;
  int stages;
  int stride;         // 1, or 2 = strided conv with TF 'SAME' padding (Isensee in-convs, isensee2017.py:51)
  int stride_z;       // = stride, or 1 for the 3x3x1 kernels of the 2D family (strides=(2, 2), unet/isensee.py:49)
  int pbx, pby, pbz;  // 'before' padding per axis (k/2 for stride 1; TF SAME for stride 2)
  // Decoder convolutions over concatenate([UpSampling3D(2)(coarse), skip]) WITHOUT the upsampled tensor
  // (unet3d/unet.py:59-62,138): a fine voxel 2c+p of parity class p only ever sees the 2x2x2 coarse neighbourhood
  // c + {p-1, p} per axis, so per class the 27 taps over the upsampled source collapse into 8 taps over the coarse
  // tensor with summed weights W'_p[j] (3.4x fewer MACs on that source).
  //   upmode 1 (fprop): a tile is 128 coarse positions of ONE class; source 0 = coarse tensor, 8 taps at c0 + j - 1 + p
  //            (weights [Cout][class*8 + j][Cc]); source 1 = the skip tensor read with traversal stride 2 at
  //            2*c0 + p + t - 1 for the 27 ordinary taps; the epilogue writes the fine voxels 2c + p.
  //   upmode 2 (dgrad to the coarse tensor): a tile is 128 coarse positions; the source is dY read with traversal
  //            stride 2 at 2*(c0 - d) + q, d = j - 1 + q, for the 64 (class q, tap j) pairs (weights transposed).
  int upmode;
  int ntaps_s[2];     // taps per source (== ntaps unless upmode)
  int oX, oY, oZ;     // extents of the OUTPUT tensor (fine grid in upmode 1; == X, Y, Z otherwise)
  const float* bias;
  bf16* out;
  const bf16* mask;
};

// ---------------------------------------------------------------------------------------------
// fprop / dgrad kernel
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreadsTc, 1) conv3d_tc_fprop_kernel(
    const __grid_constant__ FpropParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t b_bytes = (uint32_t)p.block_n * 128u;
  const uint32_t stage_bytes = kABytes + b_bytes;
  const uint32_t bar0 = smem0 + (uint32_t)p.stages * stage_bytes;
  // barrier map: full[s], empty[s], tmem_full[2], tmem_empty[2], then the TMEM base address word
  auto full_bar = [&](int s) { return bar0 + 8u * (uint32_t)s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (uint32_t)(p.stages + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (uint32_t)(2 * p.stages + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (uint32_t)(2 * p.stages + 2 + a); };
  const uint32_t tmem_slot = bar0 + 8u * (uint32_t)(2 * p.stages + 4);

  uint32_t tmem_cols = 32;
  while (tmem_cols < 2u * (uint32_t)p.block_n) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.nsrc; ++s) {
      prefetch_tmap(&p.tmA[s]);
      prefetch_tmap(&p.tmW[s]);
    }
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < p.stages; ++s) {
        mbar_init(full_bar(s), 1);
        mbar_init(empty_bar(s), 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull_bar(a), 1);
        mbar_init(tempty_bar(a), 128);
      }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const int total_tiles = p.m_tiles * p.n_tiles;  // m_tiles counts (coarse tile, class) pairs in upmode 1
  const int kxy = kext_xy(p.ksize), kzz = kext_z(p.ksize);
  const int pad = kxy >> 1, padz = kzz >> 1;

  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);

  if (warp_u == 0) {
    // ===== TMA producer warp (converged; one elected lane issues) =====
    pdl_wait();  // activations come from the previous kernel in the stream
    pdl_launch_dependents();
    uint32_t stage = 0, ph = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int n_tile = tile % p.n_tiles;
      int m = tile / p.n_tiles;
      int cls = 0;
      if (p.upmode == 1) {
        cls = m & 7;
        m >>= 3;
      }
      const int iz = m % p.tz;
      m /= p.tz;
      const int iy = m % p.ty;
      m /= p.ty;
      const int ix = m % p.tx;
      const int n = m / p.tx;
      const int x0 = ix * p.bx * p.stride - p.pbx, y0 = iy * p.by * p.stride - p.pby,
                z0 = iz * p.bz * p.stride_z - p.pbz;
      const int px = cls >> 2, py = (cls >> 1) & 1, pz = cls & 1;
      for (int s = 0; s < p.nsrc; ++s) {
        const uint32_t tx_bytes = (uint32_t)(kTileM + p.block_n) * (uint32_t)p.KC[s] * 2u;
        for (int ch = 0; ch < p.nchunks[s]; ++ch) {
          if (p.upmode == 0) {
            int tap = 0;
            for (int kx = 0; kx < kxy; ++kx)
              for (int ky = 0; ky < kxy; ++ky)
                for (int kz = 0; kz < kzz; ++kz, ++tap) {
                  mbar_wait(empty_bar(stage), ph ^ 1u);
                  mbar_expect_tx_elect(full_bar(stage), tx_bytes);
                  const uint32_t a_dst = smem0 + stage * stage_bytes;
                  tma_load_5d_elect(a_dst, &p.tmA[s], full_bar(stage), ch * p.KC[s], z0 + kz, y0 + ky, x0 + kx, n);
                  tma_load_3d_elect(a_dst + kABytes, &p.tmW[s], full_bar(stage), p.wcofs[s] + ch * p.KC[s], tap,
                                    n_tile * p.block_n);
                  if (++stage == (uint32_t)p.stages) {
                    stage = 0;
                    ph ^= 1u;
                  }
                }
          } else {
            // x0, y0, z0 are the coarse tile origin here (stride 1, no padding)
            for (int tap = 0; tap < p.ntaps_s[s]; ++tap) {
              int ax, ay, az, wtap;
              if (p.upmode == 1 && s == 0) {        // coarse source, 8 taps of this class
                ax = x0 + (tap >> 2) - 1 + px;
                ay = y0 + ((tap >> 1) & 1) - 1 + py;
                az = z0 + (tap & 1) - 1 + pz;
                wtap = cls * 8 + tap;
              } else if (p.upmode == 1) {           // skip source at fine resolution, every second voxel
                ax = 2 * x0 + px + tap / 9 - 1;
                ay = 2 * y0 + py + (tap / 3) % 3 - 1;
                az = 2 * z0 + pz + tap % 3 - 1;
                wtap = tap;
              } else {                              // dY at fine resolution: class q = tap / 8, coarse tap j = tap % 8
                const int q = tap >> 3, j = tap & 7;
                const int qx = q >> 2, qy = (q >> 1) & 1, qz = q & 1;
                ax = 2 * (x0 - ((j >> 2) - 1 + qx)) + qx;
                ay = 2 * (y0 - (((j >> 1) & 1) - 1 + qy)) + qy;
                az = 2 * (z0 - ((j & 1) - 1 + qz)) + qz;
                wtap = tap;
              }
              mbar_wait(empty_bar(stage), ph ^ 1u);
              mbar_expect_tx_elect(full_bar(stage), tx_bytes);
              const uint32_t a_dst = smem0 + stage * stage_bytes;
              tma_load_5d_elect(a_dst, &p.tmA[s], full_bar(stage), ch * p.KC[s], az, ay, ax, n);
              tma_load_3d_elect(a_dst + kABytes, &p.tmW[s], full_bar(stage), p.wcofs[s] + ch * p.KC[s], wtap,
                                n_tile * p.block_n);
              if (++stage == (uint32_t)p.stages) {
                stage = 0;
                ph ^= 1u;
              }
            }
          }
        }
      }
    }
  } else if (warp_u == 1) {
    // ===== MMA warp (converged; tcgen05.mma / commit predicated on one elected lane) =====
    const uint32_t idesc = make_idesc(kTileM, p.block_n, 0, 0);
    uint32_t stage = 0, ph = 0, tcount = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tcount) {
      const uint32_t acc = tcount & 1u, acc_ph = (tcount >> 1) & 1u;
      mbar_wait(tempty_bar(acc), acc_ph ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * (uint32_t)p.block_n;
      uint32_t accumulate = 0;
      for (int s = 0; s < p.nsrc; ++s) {
        const uint32_t row_bytes = (uint32_t)p.KC[s] * 2u;
        const uint32_t hi32 = desc_hi(8u * row_bytes, layout_code((int)row_bytes));
        const int nk = p.KC[s] >> 4;
        const int nst = p.nchunks[s] * p.ntaps_s[s];
        for (int i = 0; i < nst; ++i) {
          mbar_wait(full_bar(stage), ph);
          tc_fence_after();
          const uint32_t a_lo = desc_lo(smem0 + stage * stage_bytes, 16u);
          const uint32_t b_lo = a_lo + (kABytes >> 4);
          for (int k = 0; k < nk; ++k) {
            umma_bf16_lh_elect(d_tmem, a_lo + 2u * (uint32_t)k, hi32, b_lo + 2u * (uint32_t)k, hi32, idesc,
                               accumulate);
            accumulate = 1;
          }
          umma_commit_elect(empty_bar(stage));  // frees the smem slot once these MMAs retire
          if (++stage == (uint32_t)p.stages) {
            stage = 0;
            ph ^= 1u;
          }
        }
      }
      umma_commit_elect(tfull_bar(acc));  // accumulator complete -> epilogue
    }
  } else {
    // ===== epilogue: TMEM -> registers -> bias/ReLU (fprop) or ReLU mask (dgrad) -> bf16 -> HBM =====
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const int rz = row % p.bz, ry = (row / p.bz) % p.by, rx = row / (p.bz * p.by);
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tcount) {
      const uint32_t acc = tcount & 1u, acc_ph = (tcount >> 1) & 1u;
      const int n_tile = tile % p.n_tiles;
      int m = tile / p.n_tiles;
      int cls = 0;
      if (p.upmode == 1) {
        cls = m & 7;
        m >>= 3;
      }
      const int iz = m % p.tz;
      m /= p.tz;
      const int iy = m % p.ty;
      m /= p.ty;
      const int ix = m % p.tx;
      const int n = m / p.tx;
      int x = ix * p.bx + rx, y = iy * p.by + ry, z = iz * p.bz + rz;
      const bool valid = (x < p.X) && (y < p.Y) && (z < p.Z);
      if (p.upmode == 1) {  // row = coarse position c of class p: the fine voxel 2c + p
        x = 2 * x + (cls >> 2);
        y = 2 * y + ((cls >> 1) & 1);
        z = 2 * z + (cls & 1);
      }
      const int64_t v = (((int64_t)n * p.oX + x) * p.oY + y) * p.oZ + z;
      const int64_t off = v * p.out_C + p.out_cofs + n_tile * p.block_n;
      mbar_wait(tfull_bar(acc), acc_ph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)p.block_n;
      for (int c16 = 0; c16 < p.block_n / 16; ++c16) {
        uint32_t r[16];
        tmem_ld16(taddr + (uint32_t)c16 * 16u, r);
        tmem_ld_wait();
        if (valid) {
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(r[j]);
          if (p.bias != nullptr) {
            const float4* bp =
                reinterpret_cast<const float4*>(p.bias + n_tile * p.block_n + c16 * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b4 = __ldg(bp + j);
              f[4 * j] += b4.x;
              f[4 * j + 1] += b4.y;
              f[4 * j + 2] += b4.z;
              f[4 * j + 3] += b4.w;
            }
          }
          if (p.relu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
          }
          if (p.mask != nullptr) {
            const uint4* mp = reinterpret_cast<const uint4*>(p.mask + off + c16 * 16);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint4 mv = __ldg(mp + h);
              const __nv_bfloat162* mh = reinterpret_cast<const __nv_bfloat162*>(&mv);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 mf = __bfloat1622float2(mh[j]);
                if (!(mf.x > 0.f)) f[8 * h + 2 * j] = 0.f;
                if (!(mf.y > 0.f)) f[8 * h + 2 * j + 1] = 0.f;
              }
            }
          }
          uint4 o[2];
          __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(o);
#pragma unroll
          for (int j = 0; j < 8; ++j) oh[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
          uint4* op = reinterpret_cast<uint4*>(p.out + off + c16 * 16);
          op[0] = o[0];
          op[1] = o[1];
        }
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// wgrad kernel
// ---------------------------------------------------------------------------------------------
struct alignas(64) WgradParams {
  CUtensorMap tmX;   // input activation (5-D), box = (KC, bz, by, bx, 1)
  CUtensorMap tmDY;  // output gradient (5-D), box = (NC, bz, by, bx, 1)
  int KC, NC;        // channel chunk of X rows / dY sub-box
  int g;             // taps stacked per 128-row group = 128 / KC
  int ngroups;       // ceil(ntaps / g)
  int G;             // groups per CTA (accumulators resident in TMEM)
  int n_gsub;        // ceil(ngroups / G)
  int n_cchunks;     // Cin / KC
  int n_nblocks;     // Cout / NB
  int NB;            // Cout block (MMA N)
  int splits;        // split-K factor over voxel tiles
  int N, X, Y, Z;
  int bx, by, bz, tx, ty, tz;
  int m_tiles;
  int ksize, ntaps;
  int Ct, cofs, Cout;  // dW layout [Cout][ntaps][Ct], this source at channel offset cofs
  int stages;
  // upmode 1: weight gradient of the 64 class-combined taps of a decoder convolution over the COARSE tensor
  // (see FpropParams::upmode): X = coarse tensor, dY read with traversal stride 2 at 2c + p; a work item carries the
  // class p and accumulates its 8 taps; dW layout [Cout][64 = class*8 + j][Ct]. N, X, Y, Z are the coarse extents.
  int upmode;
  float* dw;
};

__global__ void __launch_bounds__(kThreadsTc, 1) conv3d_tc_wgrad_kernel(
    const __grid_constant__ WgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // smem: [stages] x 32 KB A slots (g tap tiles of 128 voxels x KC), then 2 dY buffers (128 x NB)
  const uint32_t a_slot = 32768u;
  const uint32_t dy_bytes = (uint32_t)kTileM * (uint32_t)p.NB * 2u;
  const uint32_t dy0 = smem0 + (uint32_t)p.stages * a_slot;
  const uint32_t bar0 = dy0 + 2u * dy_bytes;
  auto full_bar = [&](int s) { return bar0 + 8u * (uint32_t)s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (uint32_t)(p.stages + s); };
  auto dyfull_bar = [&](int b) { return bar0 + 8u * (uint32_t)(2 * p.stages + b); };
  auto dyempty_bar = [&](int b) { return bar0 + 8u * (uint32_t)(2 * p.stages + 2 + b); };
  const uint32_t done_bar = bar0 + 8u * (uint32_t)(2 * p.stages + 4);
  const uint32_t tmem_slot = bar0 + 8u * (uint32_t)(2 * p.stages + 5);

  uint32_t tmem_cols = 32;
  while (tmem_cols < (uint32_t)(p.G * p.NB)) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmX);
    prefetch_tmap(&p.tmDY);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < p.stages; ++s) {
        mbar_init(full_bar(s), 1);
        mbar_init(empty_bar(s), 1);
      }
      for (int b = 0; b < 2; ++b) {
        mbar_init(dyfull_bar(b), 1);
        mbar_init(dyempty_bar(b), 1);
      }
      mbar_init(done_bar, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  // work item decode: blockIdx.x = (((split * n_nblocks + nb) * n_cchunks + cc) * n_gsub + gs) [* 8 + class]
  int w = blockIdx.x;
  int cls = 0;
  if (p.upmode) {
    cls = w & 7;
    w >>= 3;
  }
  const int cpx = cls >> 2, cpy = (cls >> 1) & 1, cpz = cls & 1;
  const int gs = w % p.n_gsub;
  w /= p.n_gsub;
  const int cc = w % p.n_cchunks;
  w /= p.n_cchunks;
  const int nb = w % p.n_nblocks;
  const int split = w / p.n_nblocks;
  const int g_first = gs * p.G;
  const int g_count = min(p.G, p.ngroups - g_first);
  const int mt0 = (int)(((int64_t)p.m_tiles * split) / p.splits);
  const int mt1 = (int)(((int64_t)p.m_tiles * (split + 1)) / p.splits);
  const int kxy = kext_xy(p.ksize), kzz = kext_z(p.ksize);
  const int pad = kxy >> 1, padz = kzz >> 1;
  const uint32_t tap_tile_bytes = (uint32_t)kTileM * (uint32_t)p.KC * 2u;
  const uint32_t dy_sub_bytes = (uint32_t)kTileM * (uint32_t)p.NC * 2u;

  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);

  if (warp_u == 0) {
    // ===== TMA producer warp =====
    pdl_wait();
    pdl_launch_dependents();
    uint32_t stage = 0, ph = 0, vt = 0;
    for (int mt = mt0; mt < mt1; ++mt, ++vt) {
      int m = mt;
      const int iz = m % p.tz;
      m /= p.tz;
      const int iy = m % p.ty;
      m /= p.ty;
      const int ix = m % p.tx;
      const int n = m / p.tx;
      const int x0 = ix * p.bx, y0 = iy * p.by, z0 = iz * p.bz;
      const uint32_t b = vt & 1u, bph = (vt >> 1) & 1u;
      mbar_wait(dyempty_bar(b), bph ^ 1u);
      mbar_expect_tx_elect(dyfull_bar(b), dy_bytes);
      for (int j = 0; j < p.NB / p.NC; ++j)
        tma_load_5d_elect(dy0 + b * dy_bytes + (uint32_t)j * dy_sub_bytes, &p.tmDY, dyfull_bar(b),
                          nb * p.NB + j * p.NC, p.upmode ? 2 * z0 + cpz : z0, p.upmode ? 2 * y0 + cpy : y0,
                          p.upmode ? 2 * x0 + cpx : x0, n);
      for (int gi = 0; gi < g_count; ++gi) {
        mbar_wait(empty_bar(stage), ph ^ 1u);
        mbar_expect_tx_elect(full_bar(stage), (uint32_t)p.g * tap_tile_bytes);
        for (int t = 0; t < p.g; ++t) {
          const int tap = min((g_first + gi) * p.g + t, p.ntaps - 1);  // pad group with a repeat
          int dz = tap % kzz - padz;
          int dy = (tap / kzz) % kxy - pad;
          int dx = tap / (kzz * kxy) - pad;
          if (p.upmode) {  // tap = j of this class: coarse offset j - 1 + p per axis
            dx = (tap >> 2) - 1 + cpx;
            dy = ((tap >> 1) & 1) - 1 + cpy;
            dz = (tap & 1) - 1 + cpz;
          }
          tma_load_5d_elect(smem0 + stage * a_slot + (uint32_t)t * tap_tile_bytes, &p.tmX, full_bar(stage),
                            cc * p.KC, z0 + dz, y0 + dy, x0 + dx, n);
        }
        if (++stage == (uint32_t)p.stages) {
          stage = 0;
          ph ^= 1u;
        }
      }
    }
  } else if (warp_u == 1) {
    // ===== MMA warp =====
    const uint32_t idesc = make_idesc(kTileM, p.NB, 1, 1);
    const uint32_t a_row = (uint32_t)p.KC * 2u, b_row = (uint32_t)p.NC * 2u;
    const uint32_t a_sbo = 8u * a_row, b_sbo = 8u * b_row;
    const uint32_t a_hi = desc_hi(a_sbo, layout_code((int)a_row)), b_hi = desc_hi(b_sbo, layout_code((int)b_row));
    const uint32_t a_step = (2u * a_sbo) >> 4, b_step = (2u * b_sbo) >> 4;  // 16 voxels per MMA
    uint32_t stage = 0, ph = 0, vt = 0;
    for (int mt = mt0; mt < mt1; ++mt, ++vt) {
      const uint32_t b = vt & 1u, bph = (vt >> 1) & 1u;
      mbar_wait(dyfull_bar(b), bph);
      tc_fence_after();
      const uint32_t b_lo0 = desc_lo(dy0 + b * dy_bytes, dy_sub_bytes);
      for (int gi = 0; gi < g_count; ++gi) {
        mbar_wait(full_bar(stage), ph);
        tc_fence_after();
        uint32_t a_lo = desc_lo(smem0 + stage * a_slot, tap_tile_bytes);
        uint32_t b_lo = b_lo0;
        const uint32_t d_tmem = tmem_base + (uint32_t)(gi * p.NB);
#pragma unroll
        for (int ks = 0; ks < kTileM / 16; ++ks) {
          umma_bf16_lh_elect(d_tmem, a_lo, a_hi, b_lo, b_hi, idesc, (vt > 0 || ks > 0) ? 1u : 0u);
          a_lo += a_step;
          b_lo += b_step;
        }
        umma_commit_elect(empty_bar(stage));
        if (++stage == (uint32_t)p.stages) {
          stage = 0;
          ph ^= 1u;
        }
      }
      umma_commit_elect(dyempty_bar(b));
    }
    umma_commit_elect(done_bar);
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;     // (tap within group, channel within chunk)
    const int t_in_g = row / p.KC, ci = row % p.KC;
    mbar_wait(done_bar, 0);
    tc_fence_after();
    if (mt1 > mt0) {
      for (int gi = 0; gi < g_count; ++gi) {
        int tap = (g_first + gi) * p.g + t_in_g;
        const bool valid = tap < p.ntaps;
        int ntaps_out = p.ntaps;
        if (p.upmode) {
          tap += cls * 8;
          ntaps_out = 64;
        }
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(gi * p.NB);
        for (int c16 = 0; c16 < p.NB / 16; ++c16) {
          uint32_t r[16];
          tmem_ld16(taddr + (uint32_t)c16 * 16u, r);
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int co = nb * p.NB + c16 * 16 + j;
              atomicAdd(p.dw + ((int64_t)co * ntaps_out + tap) * p.Ct + p.cofs + cc * p.KC + ci,
                        __uint_as_float(r[j]));
            }
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side: TMA descriptors and launch configuration
// ---------------------------------------------------------------------------------------------
// 5-D map over a channels-last activation tensor [N][X][Y][Z][C] (bf16), box (cbox, bz, by, bx, 1)
int make_act_tmap(CUtensorMap* tm, const bf16* base, int N, int X, int Y, int Z, int C, int cbox,
                  int bz, int by, int bx, int stride = 1, int stride_z = 0) {
  EncodeTiledFn enc = encode_tiled();
  FM_CHECK(enc != nullptr, FM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)Z, (cuuint64_t)Y, (cuuint64_t)X, (cuuint64_t)N};
  cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)Z * C * 2, (cuuint64_t)Y * Z * C * 2,
                           (cuuint64_t)X * Y * Z * C * 2};
  // with a traversal stride the box is given in tensor elements and every stride-th element is loaded
  const cuuint32_t st = (cuuint32_t)stride, stz = (cuuint32_t)(stride_z > 0 ? stride_z : stride);
  cuuint32_t box[5] = {(cuuint32_t)cbox, (cuuint32_t)bz * stz, (cuuint32_t)by * st, (cuuint32_t)bx * st, 1};
  cuuint32_t estr[5] = {1, stz, st, st, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)base, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_row_bytes(cbox * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FM_CHECK(r == CUDA_SUCCESS, FM_ECUDA,
           "cuTensorMapEncodeTiled(act) failed: %d (N=%d %dx%dx%d C=%d box c=%d z=%d y=%d x=%d)", (int)r,
           N, X, Y, Z, C, cbox, bz, by, bx);
  return FM_OK;
}

// 3-D map over packed weights [Cout][taps][Ct] (bf16), box (kc, 1, nrows)
int make_w_tmap(CUtensorMap* tm, const bf16* base, int Cout, int taps, int Ct, int kc, int nrows) {
  EncodeTiledFn enc = encode_tiled();
  FM_CHECK(enc != nullptr, FM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {(cuuint64_t)Ct, (cuuint64_t)taps, (cuuint64_t)Cout};
  cuuint64_t strides[2] = {(cuuint64_t)Ct * 2, (cuuint64_t)taps * Ct * 2};
  cuuint32_t box[3] = {(cuuint32_t)kc, 1, (cuuint32_t)nrows};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void*)base, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_row_bytes(kc * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FM_CHECK(r == CUDA_SUCCESS, FM_ECUDA, "cuTensorMapEncodeTiled(weights) failed: %d (Cout=%d taps=%d Ct=%d)",
           (int)r, Cout, taps, Ct);
  return FM_OK;
}

int pow2_ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// 128-voxel tile box: z fastest, powers of two
void choose_box(int X, int Y, int Z, int* bx, int* by, int* bz) {
  int z = std::min(kTileM, pow2_ceil(Z));
  int y = std::min(kTileM / z, pow2_ceil(Y));
  int x = kTileM / (z * y);
  *bz = z;
  *by = y;
  *bx = x;
}

bool chan_ok(int C) { return C > 0 && C % 16 == 0 && (C <= 64 ? (C == 16 || C == 32 || C == 64) : C % 64 == 0); }
int chunk_of(int C) { return std::min(C, 64); }


}  // namespace

int conv_tc_supported(int C1, int C2, int Cout, int ksize) {
  if (!(ksize == 1 || ksize == 3 || ksize == 31)) return 0;
  if (!chan_ok(C1)) return 0;
  if (C2 != 0 && !chan_ok(C2)) return 0;
  if (!(Cout == 16 || Cout == 32 || Cout == 64 || (Cout >= 128 && Cout % 128 == 0))) return 0;
  return 1;
}

int k_conv3d_tc_fprop(fm_ctx* ctx, const bf16* x1, const bf16* x2, const bf16* w_packed,
                      const float* bias, bf16* y, const bf16* mask, int N, int X, int Y, int Z, int C1,
                      int C2, int Cout, int ksize, int relu, int out_C, int out_cofs, int stride, int Xin,
                      int Yin, int Zin) {
  FM_CHECK(stride == 1 || (stride == 2 && kext_xy(ksize) == 3 && C2 == 0), FM_EINVAL,
           "conv3d tc: stride %d unsupported", stride);
  const int stride_z = kext_z(ksize) == 1 ? 1 : stride;
  if (stride == 1) {
    Xin = X;
    Yin = Y;
    Zin = Z;
  }
  FM_CHECK(conv_tc_supported(C1, C2, Cout, ksize), FM_EINVAL,
           "conv3d tc: unsupported channels C1=%d C2=%d Cout=%d k=%d", C1, C2, Cout, ksize);
  FM_CHECK(out_C % 8 == 0 && out_cofs % 8 == 0, FM_EINVAL, "conv3d tc: output channel pitch/offset");
  FpropParams p;
  memset(&p, 0, sizeof(p));
  p.nsrc = C2 > 0 ? 2 : 1;
  p.N = N;
  p.X = X;
  p.Y = Y;
  p.Z = Z;
  choose_box(X, Y, Z, &p.bx, &p.by, &p.bz);
  p.tx = ceil_div(X, p.bx);
  p.ty = ceil_div(Y, p.by);
  p.tz = ceil_div(Z, p.bz);
  p.m_tiles = N * p.tx * p.ty * p.tz;
  p.block_n = std::min(Cout, 128);
  // small problems (the 8^3 level: 32 voxel tiles): at the widest N tile fewer than half of the SMs would get a CTA,
  // and each of those walks its 27 x Cin/64 pipeline stages at L2 latency. Narrower N tiles put 4x the SMs to work
  // (every N tile re-reads the A tiles from L2 - these layers are latency-bound, not bandwidth-bound).
  while (p.block_n > 32 && p.m_tiles * (Cout / p.block_n) * 2 <= ctx->num_sms) p.block_n /= 2;
  p.n_tiles = Cout / p.block_n;
  p.ksize = ksize;
  p.ntaps = kext_taps(ksize);
  p.out_C = out_C;
  p.out_cofs = out_cofs;
  p.relu = relu;
  p.bias = bias;
  p.out = y;
  p.mask = mask;
  p.stride = stride;
  p.stride_z = stride_z;
  p.upmode = 0;
  p.ntaps_s[0] = p.ntaps_s[1] = p.ntaps;
  p.oX = X;
  p.oY = Y;
  p.oZ = Z;
  {
    // TF 'SAME': pad_total = max((out-1)*stride + k - in, 0), pad_before = pad_total / 2
    auto pb = [&](int out, int in, int k, int st) { return std::max((out - 1) * st + k - in, 0) / 2; };
    p.pbx = pb(X, Xin, kext_xy(ksize), stride);
    p.pby = pb(Y, Yin, kext_xy(ksize), stride);
    p.pbz = pb(Z, Zin, kext_z(ksize), stride_z);
  }
  const int Ct = C1 + C2;
  const int Cs[2] = {C1, C2};
  const bf16* xs[2] = {x1, x2};
  int cofs = 0;
  for (int s = 0; s < p.nsrc; ++s) {
    p.KC[s] = chunk_of(Cs[s]);
    p.nchunks[s] = Cs[s] / p.KC[s];
    p.wcofs[s] = cofs;
    FM_TRY(make_act_tmap(&p.tmA[s], xs[s], N, Xin, Yin, Zin, Cs[s], p.KC[s], p.bz, p.by, p.bx, stride, stride_z));
    FM_TRY(make_w_tmap(&p.tmW[s], w_packed, Cout, p.ntaps, Ct, p.KC[s], p.block_n));
    cofs += Cs[s];
  }
  const uint32_t stage_bytes = kABytes + (uint32_t)p.block_n * 128u;
  int stages = (kMaxDynSmem - 2048) / (int)stage_bytes;
  stages = std::max(2, std::min(stages, 8));
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + 1024 /*align*/ + 256 /*barriers*/;
  static bool attr_set = false;
  if (!attr_set) {
    FM_CUDA(cudaFuncSetAttribute(conv3d_tc_fprop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 kMaxDynSmem));
    attr_set = true;
  }
  const int grid = std::min(p.m_tiles * p.n_tiles, ctx->num_sms);
  const double vox = (double)N * X * Y * Z;
  ProfScope prof(ctx, mask != nullptr || bias == nullptr ? "conv3d_tc_dgrad" : "conv3d_tc_fprop",
                 2.0 * p.ntaps * Ct * Cout * vox, vox * (Ct + Cout) * 2.0);
  FM_CUDA(launch_pdl(conv3d_tc_fprop_kernel, dim3(grid), dim3(kThreadsTc), smem, ctx->stream, p));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// ---------------------------------------------------------------------------------------------
// decoder convolutions at coarse resolution (see FpropParams::upmode)
// ---------------------------------------------------------------------------------------------
namespace {

int launch_tc_fprop(fm_ctx* ctx, FpropParams& p, const char* name, double flops, double bytes) {
  const uint32_t stage_bytes = kABytes + (uint32_t)p.block_n * 128u;
  int stages = (kMaxDynSmem - 2048) / (int)stage_bytes;
  stages = std::max(2, std::min(stages, 8));
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + 1024 /*align*/ + 256 /*barriers*/;
  static bool attr_set = false;
  if (!attr_set) {
    FM_CUDA(cudaFuncSetAttribute(conv3d_tc_fprop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem));
    attr_set = true;
  }
  const int grid = std::min(p.m_tiles * p.n_tiles, ctx->num_sms);
  ProfScope prof(ctx, name, flops, bytes);
  FM_CUDA(launch_pdl(conv3d_tc_fprop_kernel, dim3(grid), dim3(kThreadsTc), smem, ctx->stream, p));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// W'_p[j] = sum of the taps t with floor((p + t - 1) / 2) == j - 1 + p per axis (nearest-neighbour upsampling by 2)
__device__ __forceinline__ bool tap_in_class(int p, int j, int t) { return ((p + t + 1) >> 1) - 1 == j - 1 + p; }

// master [Cout][27][Ct] fp32 (up source = channels [0, Cc)) -> wf [Cout][64][Cc] and wd [Cc][64][Cout], bf16,
// tap index = class * 8 + j, class = (px*2 + py)*2 + pz, j = (jx*2 + jy)*2 + jz
__global__ void __launch_bounds__(256) repack_up_kernel(const float* __restrict__ params, const __grid_constant__ RepackUpTable tab) {
  FM_PDL_SYNC();
  int li = 0;
  while (li + 1 < tab.n && (int)blockIdx.x >= tab.d[li + 1].block0) ++li;
  const RepackUpDesc d = tab.d[li];
  const float* w = params + d.w_off;
  const int Cout = d.cout, Cc = d.cc, Ct = d.ct;
  const int64_t total = (int64_t)Cout * 64 * Cc;
  const int64_t g = (int64_t)(blockIdx.x - d.block0) * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int ci = (int)(g % Cc);
  const int pj = (int)((g / Cc) % 64);
  const int co = (int)(g / ((int64_t)Cc * 64));
  const int cls = pj >> 3, j = pj & 7;
  const int px = cls >> 2, py = (cls >> 1) & 1, pz = cls & 1;
  const int jx = j >> 2, jy = (j >> 1) & 1, jz = j & 1;
  float acc = 0.f;
  for (int tx = 0; tx < 3; ++tx) {
    if (!tap_in_class(px, jx, tx)) continue;
    for (int ty = 0; ty < 3; ++ty) {
      if (!tap_in_class(py, jy, ty)) continue;
      for (int tz = 0; tz < 3; ++tz) {
        if (!tap_in_class(pz, jz, tz)) continue;
        acc += w[((int64_t)co * 27 + (tx * 3 + ty) * 3 + tz) * Ct + ci];
      }
    }
  }
  const bf16 v = __float2bfloat16(acc);
  if (d.wf) d.wf[g] = v;
  if (d.wd) d.wd[((int64_t)ci * 64 + pj) * Cout + co] = v;
}

// dW[co][t][ci] += sum over the classes p of dW'_p[j(p, t)][co][ci]: the 64 class-tap gradients folded back onto the
// 27 taps of the master kernel (every tap belongs to exactly one j per class)
__global__ void __launch_bounds__(256) fold_up_wgrad_kernel(const float* __restrict__ dwu, float* __restrict__ dw,
                                                            int Cout, int Cc, int Ct) {
  FM_PDL_SYNC();
  const int64_t total = (int64_t)Cout * 27 * Cc;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int ci = (int)(g % Cc);
  const int t = (int)((g / Cc) % 27);
  const int co = (int)(g / ((int64_t)Cc * 27));
  const int tx = t / 9, ty = (t / 3) % 3, tz = t % 3;
  float acc = 0.f;
#pragma unroll
  for (int cls = 0; cls < 8; ++cls) {
    const int px = cls >> 2, py = (cls >> 1) & 1, pz = cls & 1;
    const int jx = ((px + tx + 1) >> 1) - px, jy = ((py + ty + 1) >> 1) - py, jz = ((pz + tz + 1) >> 1) - pz;
    acc += dwu[((int64_t)co * 64 + cls * 8 + (jx * 2 + jy) * 2 + jz) * Cc + ci];
  }
  dw[((int64_t)co * 27 + t) * Ct + ci] += acc;
}

}  // namespace

int conv_up_supported(int X, int Y, int Z, int Cc, int Cs, int Cout) {
  if (X % 2 || Y % 2 || Z % 2) return 0;
  if (!chan_ok(Cc) || !chan_ok(Cs) || !chan_ok(Cout)) return 0;
  if (!(Cout == 16 || Cout == 32 || Cout == 64 || (Cout >= 128 && Cout % 128 == 0))) return 0;
  if (!(Cc == 16 || Cc == 32 || Cc == 64 || (Cc >= 128 && Cc % 128 == 0))) return 0;  // N blocks of the dgrad
  return 1;
}

int k_repack_up_table(fm_ctx* ctx, const float* params, const RepackUpTable& tab) {
  if (tab.n == 0) return FM_OK;
  const RepackUpDesc& last = tab.d[tab.n - 1];
  const int blocks = last.block0 + (int)ceil_div64((int64_t)last.cout * 64 * last.cc, 256);
  double total = 0.0;
  for (int i = 0; i < tab.n; ++i) total += (double)tab.d[i].cout * 64 * tab.d[i].cc;
  ProfScope prof(ctx, "repack_up", 0.0, total * 12.0);
  FM_CUDA(launch_pdl(repack_up_kernel, dim3((unsigned)blocks), dim3(256), 0, ctx->stream, params, tab));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_repack_up(fm_ctx* ctx, const float* w_master, bf16* w_up_f, bf16* w_up_d, int Cout, int Cc, int Ct) {
  RepackUpTable tab;
  memset(&tab, 0, sizeof(tab));
  tab.n = 1;
  tab.d[0].w_off = 0;
  tab.d[0].wf = w_up_f;
  tab.d[0].wd = w_up_d;
  tab.d[0].cout = Cout;
  tab.d[0].cc = Cc;
  tab.d[0].ct = Ct;
  tab.d[0].block0 = 0;
  return k_repack_up_table(ctx, w_master, tab);
}

int k_fold_up_wgrad(fm_ctx* ctx, const float* dw_up, float* dw_master, int Cout, int Cc, int Ct) {
  const int64_t total = (int64_t)Cout * 27 * Cc;
  ProfScope prof(ctx, "fold_up_wgrad", 0.0, (double)total * 40.0);
  FM_CUDA(launch_pdl(fold_up_wgrad_kernel, dim3((unsigned)ceil_div64(total, 256)), dim3(256), 0, ctx->stream, dw_up,
                     dw_master, Cout, Cc, Ct));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

// y[fine] = act(conv3x3x3(concatenate([upsample2(coarse), skip])) + bias), fine extents X, Y, Z
int k_conv3d_up_fprop(fm_ctx* ctx, const bf16* coarse, const bf16* skip, const bf16* w_up, const bf16* w_packed,
                      const float* bias, bf16* y, int N, int X, int Y, int Z, int Cc, int Cs, int Cout, int relu) {
  FM_CHECK(conv_up_supported(X, Y, Z, Cc, Cs, Cout), FM_EINVAL, "conv3d up fprop: unsupported %dx%dx%d Cc=%d Cs=%d Cout=%d",
           X, Y, Z, Cc, Cs, Cout);
  FpropParams p;
  memset(&p, 0, sizeof(p));
  const int Xc = X / 2, Yc = Y / 2, Zc = Z / 2;
  p.nsrc = 2;
  p.N = N;
  p.X = Xc;
  p.Y = Yc;
  p.Z = Zc;
  p.oX = X;
  p.oY = Y;
  p.oZ = Z;
  choose_box(Xc, Yc, Zc, &p.bx, &p.by, &p.bz);
  p.tx = ceil_div(Xc, p.bx);
  p.ty = ceil_div(Yc, p.by);
  p.tz = ceil_div(Zc, p.bz);
  p.m_tiles = N * p.tx * p.ty * p.tz * 8;
  p.block_n = std::min(Cout, 128);
  p.n_tiles = Cout / p.block_n;
  p.ksize = 3;
  p.ntaps = 27;
  p.ntaps_s[0] = 8;
  p.ntaps_s[1] = 27;
  p.upmode = 1;
  p.out_C = Cout;
  p.out_cofs = 0;
  p.relu = relu;
  p.bias = bias;
  p.out = y;
  p.mask = nullptr;
  p.stride = 1;
  p.stride_z = 1;
  p.KC[0] = chunk_of(Cc);
  p.nchunks[0] = Cc / p.KC[0];
  p.wcofs[0] = 0;
  p.KC[1] = chunk_of(Cs);
  p.nchunks[1] = Cs / p.KC[1];
  p.wcofs[1] = Cc;
  FM_TRY(make_act_tmap(&p.tmA[0], coarse, N, Xc, Yc, Zc, Cc, p.KC[0], p.bz, p.by, p.bx));
  FM_TRY(make_w_tmap(&p.tmW[0], w_up, Cout, 64, Cc, p.KC[0], p.block_n));
  FM_TRY(make_act_tmap(&p.tmA[1], skip, N, X, Y, Z, Cs, p.KC[1], p.bz, p.by, p.bx, 2));
  FM_TRY(make_w_tmap(&p.tmW[1], w_packed, Cout, 27, Cc + Cs, p.KC[1], p.block_n));
  const double vox = (double)N * X * Y * Z;
  // algorithmic FLOPs of the reference layer (27 taps over every fine voxel); executed: 8 taps on the coarse source
  return launch_tc_fprop(ctx, p, "conv3d_up_fprop", 2.0 * 27 * (Cc + Cs) * Cout * vox,
                         vox * ((double)Cc / 8 + Cs + Cout) * 2.0);
}

// dcoarse = (gradient of the layer above w.r.t. the coarse tensor) [* ReLU mask]: dy fine [N,X,Y,Z,Cout]
int k_conv3d_up_dgrad(fm_ctx* ctx, const bf16* dy, const bf16* w_up_d, bf16* dcoarse, const bf16* mask, int N, int X,
                      int Y, int Z, int Cout, int Cc) {
  FM_CHECK(conv_up_supported(X, Y, Z, Cc, Cout, Cout), FM_EINVAL, "conv3d up dgrad: unsupported %dx%dx%d Cc=%d Cout=%d", X,
           Y, Z, Cc, Cout);
  FpropParams p;
  memset(&p, 0, sizeof(p));
  const int Xc = X / 2, Yc = Y / 2, Zc = Z / 2;
  p.nsrc = 1;
  p.N = N;
  p.X = p.oX = Xc;
  p.Y = p.oY = Yc;
  p.Z = p.oZ = Zc;
  choose_box(Xc, Yc, Zc, &p.bx, &p.by, &p.bz);
  p.tx = ceil_div(Xc, p.bx);
  p.ty = ceil_div(Yc, p.by);
  p.tz = ceil_div(Zc, p.bz);
  p.m_tiles = N * p.tx * p.ty * p.tz;
  p.block_n = std::min(Cc, 128);
  p.n_tiles = Cc / p.block_n;
  p.ksize = 3;
  p.ntaps = 64;
  p.ntaps_s[0] = 64;
  p.upmode = 2;
  p.out_C = Cc;
  p.out_cofs = 0;
  p.relu = 0;
  p.bias = nullptr;
  p.out = dcoarse;
  p.mask = mask;
  p.stride = 1;
  p.stride_z = 1;
  p.KC[0] = chunk_of(Cout);
  p.nchunks[0] = Cout / p.KC[0];
  p.wcofs[0] = 0;
  FM_TRY(make_act_tmap(&p.tmA[0], dy, N, X, Y, Z, Cout, p.KC[0], p.bz, p.by, p.bx, 2));
  FM_TRY(make_w_tmap(&p.tmW[0], w_up_d, Cc, 64, Cout, p.KC[0], p.block_n));
  const double vox = (double)N * X * Y * Z;
  // algorithmic: the fine-resolution dgrad towards the upsampled source (27 taps per fine voxel) + its 2^3 sum-pool
  return launch_tc_fprop(ctx, p, "conv3d_up_dgrad", 2.0 * 27 * Cc * Cout * vox, vox * ((double)Cc / 8 + Cout) * 2.0);
}

// dw_up [Cout][64][Cc] fp32 (zeroed by the caller) += class-combined weight gradients; fine extents X, Y, Z
int k_conv3d_up_wgrad(fm_ctx* ctx, const bf16* coarse, const bf16* dy, float* dw_up, int N, int X, int Y, int Z,
                      int Cc, int Cout) {
  FM_CHECK(conv_up_supported(X, Y, Z, Cc, Cout, Cout), FM_EINVAL, "conv3d up wgrad: unsupported %dx%dx%d Cc=%d Cout=%d", X,
           Y, Z, Cc, Cout);
  WgradParams p;
  memset(&p, 0, sizeof(p));
  const int Xc = X / 2, Yc = Y / 2, Zc = Z / 2;
  p.N = N;
  p.X = Xc;
  p.Y = Yc;
  p.Z = Zc;
  choose_box(Xc, Yc, Zc, &p.bx, &p.by, &p.bz);
  p.tx = ceil_div(Xc, p.bx);
  p.ty = ceil_div(Yc, p.by);
  p.tz = ceil_div(Zc, p.bz);
  p.m_tiles = N * p.tx * p.ty * p.tz;
  p.ksize = 3;
  p.ntaps = 8;
  p.upmode = 1;
  p.KC = chunk_of(Cc);
  p.n_cchunks = Cc / p.KC;
  p.g = kTileM / p.KC;
  p.ngroups = ceil_div(p.ntaps, p.g);
  p.NB = std::min(Cout, 128);
  p.NC = std::min(p.NB, 64);
  p.n_nblocks = Cout / p.NB;
  p.G = std::min(p.ngroups, 512 / p.NB);
  p.n_gsub = ceil_div(p.ngroups, p.G);
  p.Ct = Cc;
  p.cofs = 0;
  p.Cout = Cout;
  p.dw = dw_up;
  const int items = p.n_gsub * p.n_cchunks * p.n_nblocks * 8;
  int splits = std::max(1, (2 * ctx->num_sms) / items);
  splits = std::min(splits, p.m_tiles);
  p.splits = splits;
  FM_TRY(make_act_tmap(&p.tmX, coarse, N, Xc, Yc, Zc, Cc, p.KC, p.bz, p.by, p.bx));
  FM_TRY(make_act_tmap(&p.tmDY, dy, N, X, Y, Z, Cout, p.NC, p.bz, p.by, p.bx, 2));
  const uint32_t dy_bytes = (uint32_t)kTileM * (uint32_t)p.NB * 2u;
  int stages = (kMaxDynSmem - 2048 - 2 * (int)dy_bytes) / 32768;
  stages = std::max(2, std::min(stages, 5));
  p.stages = stages;
  const size_t smem = (size_t)stages * 32768 + 2 * dy_bytes + 1024 + 256;
  FM_CUDA(cudaFuncSetAttribute(conv3d_tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem));
  const double vox = (double)N * X * Y * Z;
  // algorithmic: the fine-resolution weight gradient over the upsampled source (27 taps per fine voxel)
  ProfScope prof(ctx, "conv3d_up_wgrad", 2.0 * 27 * Cc * Cout * vox, vox * ((double)Cc / 8 + Cout) * 2.0);
  FM_CUDA(launch_pdl(conv3d_tc_wgrad_kernel, dim3(items * splits), dim3(kThreadsTc), smem, ctx->stream, p));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_conv3d_tc_wgrad(fm_ctx* ctx, const bf16* x, const bf16* dy, float* dw_packed, int N, int X, int Y,
                      int Z, int Cin, int Cin_total, int cin_ofs, int Cout, int ksize) {
  FM_CHECK(conv_tc_supported(Cin, 0, Cout, ksize), FM_EINVAL,
           "conv3d tc wgrad: unsupported channels Cin=%d Cout=%d k=%d", Cin, Cout, ksize);
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.N = N;
  p.X = X;
  p.Y = Y;
  p.Z = Z;
  choose_box(X, Y, Z, &p.bx, &p.by, &p.bz);
  p.tx = ceil_div(X, p.bx);
  p.ty = ceil_div(Y, p.by);
  p.tz = ceil_div(Z, p.bz);
  p.m_tiles = N * p.tx * p.ty * p.tz;
  p.ksize = ksize;
  p.ntaps = kext_taps(ksize);
  p.KC = chunk_of(Cin);
  p.n_cchunks = Cin / p.KC;
  p.g = kTileM / p.KC;
  p.ngroups = ceil_div(p.ntaps, p.g);
  p.NB = std::min(Cout, 128);
  p.NC = std::min(p.NB, 64);
  p.n_nblocks = Cout / p.NB;
  p.G = std::min(p.ngroups, 512 / p.NB);
  p.n_gsub = ceil_div(p.ngroups, p.G);
  p.Ct = Cin_total;
  p.cofs = cin_ofs;
  p.Cout = Cout;
  p.dw = dw_packed;
  const int items = p.n_gsub * p.n_cchunks * p.n_nblocks;
  int splits = std::max(1, (2 * ctx->num_sms) / items);
  splits = std::min(splits, p.m_tiles);
  p.splits = splits;
  FM_TRY(make_act_tmap(&p.tmX, x, N, X, Y, Z, Cin, p.KC, p.bz, p.by, p.bx));
  FM_TRY(make_act_tmap(&p.tmDY, dy, N, X, Y, Z, Cout, p.NC, p.bz, p.by, p.bx));
  const uint32_t dy_bytes = (uint32_t)kTileM * (uint32_t)p.NB * 2u;
  int stages = (kMaxDynSmem - 2048 - 2 * (int)dy_bytes) / 32768;
  stages = std::max(2, std::min(stages, 5));
  p.stages = stages;
  const size_t smem = (size_t)stages * 32768 + 2 * dy_bytes + 1024 + 256;
  static bool attr_set = false;
  if (!attr_set) {
    FM_CUDA(cudaFuncSetAttribute(conv3d_tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 kMaxDynSmem));
    attr_set = true;
  }
  const double vox = (double)N * X * Y * Z;
  ProfScope prof(ctx, "conv3d_tc_wgrad", 2.0 * p.ntaps * Cin * Cout * vox, vox * (Cin + Cout) * 2.0);
  FM_CUDA(launch_pdl(conv3d_tc_wgrad_kernel, dim3(items * splits), dim3(kThreadsTc), smem, ctx->stream, p));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
