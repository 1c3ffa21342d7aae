// conv_wgrad_march.cu — plane-marching weight gradient of Conv3D 3x3x3 on tcgen05:
//
//     dW[kx,ky,kz][ci][co] = sum_v  X[v + (kx-1, ky-1, kz-1)][ci] * dY[v][co]
//
// GEMM view per CTA: M = (ky, ci) stacked to 128 rows, N = (kx, co) stacked to 96 columns, K = voxels.
// Both operands are MN-major (channels are contiguous in memory, voxels are the K axis).
//   * A CTA owns a 16 (y) x 8 (z) column of the volume and marches along x, exactly like the forward
//     marching kernel (conv_march.cu): per input plane it loads three z-shifted, y-haloed slabs of X
//     (19 x 8 rows x 32 channels) and one dY tile per output plane (128 rows x 32 channels).
//   * the three ky taps are the M-blocks of ONE UMMA A operand: block j starts 8 slab rows (= one swizzle
//     atom) after block j-1, which is expressed by the descriptor's leading-byte-offset == stride-byte-offset.
//     (M = 128 holds four 32-channel blocks; the fourth reads one more halo row and is discarded.)
//   * the three kx taps are the N-blocks of the B operand: the dY tiles of output planes xi-1, xi, xi+1 sit
//     in consecutive slots of a ring, leading-byte-offset = slot size.
//   * kz selects the slab copy; each copy has its own MMA-issuing warp and its own TMEM accumulator, which
//     stays resident for the CTA's whole lifetime (persistent CTA over many columns) and is flushed with
//     fp32 red.add once at the end.
// One CTA handles one (32 input channels x 32 output channels) pair; pairs are spread over the grid.
// Round 2: (1) three TMA producer warps (one per kz slab copy; warp 0 also feeds the dY ring) - a single producer
// walking 4 barrier waits + 4 TMA issues per plane was the pacing role; (2) the dY ring has two MIRROR slots (slots
// 8, 9 repeat 0, 1, loaded by a second TMA), so the three consecutive N blocks of a plane never wrap and every k-step
// is ONE MMA (the wrap used to split a quarter of them into an N = 64 and an N = 32 MMA that read A twice); (3) the
// bias gradient (column sums of dY) is folded in: the four epilogue warps, idle during the march, sum the dY tiles
// they find in shared memory - the separate bias_grad pass over every dY tensor is gone.
// TF autodiff gradient of Conv3D in create_convolution_block (fetal_net/model/unet3d/unet.py:102).
#include <algorithm>

#include "tc_ptx.cuh"

using namespace tcp;

namespace {

constexpr int kThreadsW = 320;  // warps 0-2 TMA (kz = 0,1,2; warp 0 also dY), warps 3-5 MMA issue (kz), warps 6-9 epilogue
constexpr int kProdW = 3, kMma0 = 3, kEpi0W = 6;
constexpr int kBY = 16, kBZ = 8;
constexpr int kCC = 32;                                   // channels per operand block (64 B rows, SWIZZLE_64B)
constexpr uint32_t kRow = kCC * 2;                        // 64 B
constexpr uint32_t kSbo = 8 * kRow;                       // 512 B: one y row of 8 voxels = one swizzle atom
constexpr uint32_t kXSlabRows = (kBY + 3) * kBZ;          // 19 y rows: 16 + halo + the discarded 4th block
constexpr uint32_t kXSlotBytes = 9728;                    // 19 y rows x 512 B: a multiple of the 512-byte swizzle period
constexpr uint32_t kDyTile = kBY * kBZ * kRow;            // 8192 B
constexpr int kDyRing = 8;
constexpr int kDyMirror = 2;                              // slots 8, 9 repeat slots 0, 1
constexpr int kNcols = 96;                                // (kx, co) columns per accumulator

struct alignas(64) WgMarchParams {
  CUtensorMap tmX;   // box (32, 8, 19, 1, 1)
  CUtensorMap tmDY;  // box (32, 8, 16, 1, 1)
  int N, X, Y, Z;
  int ny, nz;
  PlaneSplit split;      // how the (column, x) plane-tiles are dealt to the CTAs of a pair (common.cuh)
  int n_ci, n_co;      // 32-channel chunks of Cin (this source) and Cout
  int ctas_per_pair;   // grid = n_ci * n_co * ctas_per_pair
  int S3;              // X slab slots per kz ring
  uint32_t xslot;      // bytes between slab slots
  int kcx;             // input channels per CTA / per M block: 32 (SWIZZLE_64B) or 16 (SWIZZLE_32B, Cin = 16)
  int kcy;             // output channels per CTA / per N block: 32 (SWIZZLE_64B) or 16 (SWIZZLE_32B, Cout = 16)
  int Ct, cofs;        // dW layout [Cout][27][Ct], this source at channel offset cofs
  float* dw;
  float* db;           // bias gradient [Cout] (column sums of dY), or NULL
};

__global__ void __launch_bounds__(kThreadsW, 1) conv3d_wgrad_march_kernel(const __grid_constant__ WgMarchParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t x_base = smem0;                                        // 3 * S3 slab slots
  const uint32_t dy_base = x_base + 3u * (uint32_t)p.S3 * p.xslot;        // kDyRing tiles
  const uint32_t bar0 = dy_base + (uint32_t)(kDyRing + kDyMirror) * kDyTile;
  const int nx = 3 * p.S3;
  auto xfull_bar = [&](uint32_t s) { return bar0 + 8u * s; };
  auto xempty_bar = [&](uint32_t s) { return bar0 + 8u * ((uint32_t)nx + s); };
  auto dyfull_bar = [&](uint32_t s) { return bar0 + 8u * ((uint32_t)(2 * nx) + s); };
  auto dyempty_bar = [&](uint32_t s) { return bar0 + 8u * ((uint32_t)(2 * nx + kDyRing) + s); };
  const uint32_t zero_bar = bar0 + 8u * (uint32_t)(2 * nx + 2 * kDyRing);
  const uint32_t done_bar = zero_bar + 8u;
  const uint32_t tmem_slot = done_bar + 8u;
  constexpr uint32_t tmem_cols = 512;  // 3 accumulators x 96 columns, power of two

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tmX);
    prefetch_tmap(&p.tmDY);
  }
  const int pair = blockIdx.x / p.ctas_per_pair;
  const int rank = blockIdx.x % p.ctas_per_pair;
  const int cic = pair % p.n_ci, coc = pair / p.n_ci;
  const bool do_bias = p.db != nullptr && cic == 0;   // one ci chunk per co chunk sums dY
  if (warp == kMma0) {
    if (lane == 0) {
      for (int s = 0; s < nx; ++s) {
        mbar_init(xfull_bar(s), 1);
        mbar_init(xempty_bar(s), 1);
      }
      for (int s = 0; s < kDyRing; ++s) {
        mbar_init(dyfull_bar(s), 1);
        mbar_init(dyempty_bar(s), do_bias ? 7 : 3);  // three MMA warps (+ one arrival per bias-summing warp)
      }
      mbar_init(zero_bar, 128);
      mbar_init(done_bar, 3);
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
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);

  // k-th work unit of this CTA (see PlaneSplit in common.cuh)
  auto next_seg = [&](int& it, int& n, int& iy, int& iz, int& xa, int& xb) -> bool {
    int col;
    if (!plane_split_next(p.split, rank, p.ctas_per_pair, it, col, xa, xb)) return false;
    iz = col % p.nz;
    const int r = col / p.nz;
    iy = r % p.ny;
    n = r / p.ny;
    ++it;
    return true;
  };

  if (warp_u < kProdW) {
    // ===== TMA producers: warp kz loads the kz-shifted X slab of every plane; warp 0 also the dY tiles =====
    const int dz = warp_u;
    pdl_wait();  // x and dY come from the previous kernels in the stream
    if (dz == 0) pdl_launch_dependents();
    const uint32_t x_bytes = (uint32_t)(kBY + 128 / p.kcx - 1) * kBZ * (uint32_t)p.kcx * 2u;  // slab box bytes
    const uint32_t dy_bytes = (uint32_t)(kBY * kBZ) * (uint32_t)p.kcy * 2u;
    uint32_t sidx = 0, sph = 0;
    uint32_t dcount = 0;  // dY tiles issued so far (ring position)
    const uint32_t slot0 = (uint32_t)dz * (uint32_t)p.S3;
    for (int it = 0, n, iy, iz, xa, xb; next_seg(it, n, iy, iz, xa, xb);) {
      const int x_first = max(xa - 1, 0), x_last = min(xb, p.X - 1);
      int next_dy = xa;  // next output plane whose dY tile has to be loaded
      for (int xi = x_first; xi <= x_last; ++xi) {
        if (dz == 0) {
          const int need = min(xi + 1, xb - 1);  // dY tiles up to this output plane feed input plane xi
          for (; next_dy <= need; ++next_dy, ++dcount) {
            const uint32_t slot = dcount & (uint32_t)(kDyRing - 1);
            mbar_wait(dyempty_bar(slot), ((dcount >> 3) & 1u) ^ 1u);
            const bool mirror = slot < (uint32_t)kDyMirror;
            mbar_expect_tx_elect(dyfull_bar(slot), mirror ? 2u * dy_bytes : dy_bytes);
            tma_load_5d_elect(dy_base + slot * kDyTile, &p.tmDY, dyfull_bar(slot), coc * p.kcy, iz * kBZ, iy * kBY, next_dy, n);
            if (mirror)
              tma_load_5d_elect(dy_base + (slot + (uint32_t)kDyRing) * kDyTile, &p.tmDY, dyfull_bar(slot), coc * p.kcy,
                                iz * kBZ, iy * kBY, next_dy, n);
          }
        }
        const uint32_t stage = slot0 + sidx;
        mbar_wait(xempty_bar(stage), sph ^ 1u);
        mbar_expect_tx_elect(xfull_bar(stage), x_bytes);
        tma_load_5d_elect(x_base + stage * p.xslot, &p.tmX, xfull_bar(stage), cic * p.kcx, iz * kBZ + dz - 1, iy * kBY - 1, xi, n);
        if (++sidx == (uint32_t)p.S3) {
          sidx = 0;
          sph ^= 1u;
        }
      }
    }
  } else if (warp_u < kEpi0W) {
    // ===== MMA warps: warp kMma0 + kz issues the kz slab copy into its own accumulator =====
    const int dz = warp_u - kMma0;
    const uint32_t d_acc = tmem_base + (uint32_t)(dz * kNcols);
    const uint32_t ncy = (uint32_t)p.kcy;
    const uint32_t idesc1 = make_idesc(128, (int)ncy, 1, 1), idesc2 = make_idesc(128, 2 * (int)ncy, 1, 1),
                   idesc3 = make_idesc(128, 3 * (int)ncy, 1, 1);
    (void)idesc2;
    const uint32_t b_row = ncy * 2u, b_sbo = 8u * b_row;                     // dY operand: 64- or 32-byte rows
    const uint32_t hi32 = desc_hi(b_sbo, layout_code((int)b_row));
    const uint32_t kstep = (2u * b_sbo) >> 4;  // 16 voxels (two 8-row groups) per MMA, in 16-byte units
    const uint32_t a_row = (uint32_t)p.kcx * 2u, a_sbo = 8u * a_row;         // X operand: 64- or 32-byte rows
    const uint32_t a_hi32 = desc_hi(a_sbo, layout_code((int)a_row));
    const uint32_t a_kstep = (2u * a_sbo) >> 4;
    mbar_wait(zero_bar, 0);                   // accumulators zeroed by the epilogue warps
    tc_fence_after();
    uint32_t sidx = 0, sph = 0, dcount = 0, dwaited = 0;
    const uint32_t slot0 = (uint32_t)dz * (uint32_t)p.S3;
    for (int it = 0, n, iy, iz, xa, xb; next_seg(it, n, iy, iz, xa, xb);) {
      const int x_first = max(xa - 1, 0), x_last = min(xb, p.X - 1);
      for (int xi = x_first; xi <= x_last; ++xi) {
        const int lo = max(xa, xi - 1), hi = min(xb - 1, xi + 1);  // output planes paired with input plane xi
        const uint32_t j_lo = (uint32_t)(lo - (xi - 1));           // N block j <-> xo = xi - 1 + j <-> kx = 2 - j
        const uint32_t nblk = (uint32_t)(hi - lo + 1);
        const uint32_t seq_lo = dcount + (uint32_t)(lo - xa);      // ring sequence number of dY(lo)
        // wait (once per tile and warp) for the dY tiles up to output plane hi
        const uint32_t seq_need = dcount + (uint32_t)(hi - xa);
        for (; dwaited <= seq_need; ++dwaited)
          mbar_wait(dyfull_bar(dwaited & (uint32_t)(kDyRing - 1)), (dwaited >> 3) & 1u);
        const uint32_t stage = slot0 + sidx;
        mbar_wait(xfull_bar(stage), sph);
        tc_fence_after();
        // the <= 3 consecutive dY tiles never wrap: slots 8, 9 mirror slots 0, 1
        const uint32_t rs = seq_lo & (uint32_t)(kDyRing - 1);
        const uint32_t idA = nblk == 1 ? idesc1 : (nblk == 2 ? idesc2 : idesc3);
        uint32_t a_lo = desc_lo(x_base + stage * p.xslot, a_sbo);          // M blocks (ky) one atom apart
        uint32_t bA = desc_lo(dy_base + rs * kDyTile, kDyTile);           // N blocks (kx) one ring slot apart
        const uint32_t dA = d_acc + j_lo * ncy;
#pragma unroll
        for (int ks = 0; ks < (kBY * kBZ) / 16; ++ks) {
          umma_bf16_lh_elect(dA, a_lo, a_hi32, bA, hi32, idA, 1u);
          a_lo += a_kstep;
          bA += kstep;
        }
        umma_commit_elect(xempty_bar(stage));
        if (++sidx == (uint32_t)p.S3) {
          sidx = 0;
          sph ^= 1u;
        }
        // dY tiles this warp is done with: output plane xi-1 always, and the rest at the end of the item
        if (xi - 1 >= xa) umma_commit_elect(dyempty_bar((dcount + (uint32_t)(xi - 1 - xa)) & (uint32_t)(kDyRing - 1)));
        if (xi == x_last && xi <= xb - 1)
          umma_commit_elect(dyempty_bar((dcount + (uint32_t)(xi - xa)) & (uint32_t)(kDyRing - 1)));
      }
      dcount += (uint32_t)(xb - xa);
    }
    umma_commit_elect(done_bar);
  } else {
    // ===== epilogue warps: zero the accumulators, and flush them once at the end =====
    const int q = warp & 3;         // TMEM lane quarter of this warp (warp id mod 4)
    const int row = q * 32 + lane;  // (ky, ci) = (row / 32, row % 32); ky == 3 is the discarded block
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    for (int c16 = 0; c16 < 3 * kNcols / 16; ++c16) tmem_st16_zero(lane_base + (uint32_t)c16 * 16u);
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(zero_bar);
    if (do_bias) {
      // ===== bias gradient: column sums of the dY tiles as they pass through shared memory. Thread t owns the
      // 16-byte channel chunk c = t % CH of the rows r0 + k * (128 / CH); TMA wrote the rows swizzled (64-byte rows:
      // chunk ^= (row >> 1) & 3; 32-byte rows: chunk ^= (row >> 2) & 1). =====
      const int et = (warp - kEpi0W) * 32 + lane;
      const int CH = p.kcy / 8, RP = 128 / CH;
      const int c = et % CH, r0 = et / CH;
      const uint32_t rowb = (uint32_t)p.kcy * 2u;
      float acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.f;
      uint32_t dcount = 0;
      for (int it = 0, n, iy, iz, xa, xb; next_seg(it, n, iy, iz, xa, xb);) {
        for (int xo = xa; xo < xb; ++xo, ++dcount) {
          const uint32_t slot = dcount & (uint32_t)(kDyRing - 1);
          mbar_wait(dyfull_bar(slot), (dcount >> 3) & 1u);
          const uint32_t tile = dy_base + slot * kDyTile;
          for (int k = 0; k < CH; ++k) {
            const int r = r0 + k * RP;
            const int sw = CH == 4 ? ((r >> 1) & 3) : ((r >> 2) & 1);
            uint32_t v0, v1, v2, v3;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3)
                         : "r"(tile + (uint32_t)r * rowb + (uint32_t)((c ^ sw) * 16)));
            const uint32_t vv[4] = {v0, v1, v2, v3};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&vv[j]));
              acc[2 * j] += f.x;
              acc[2 * j + 1] += f.y;
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(dyempty_bar(slot));
        }
      }
      // lanes with the same chunk c (lane % CH) fold their sums, then one atomic per channel and warp
      for (int ofs = CH; ofs < 32; ofs <<= 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], ofs);
      }
      if (lane < CH) {
#pragma unroll
        for (int j = 0; j < 8; ++j) atomicAdd(p.db + coc * p.kcy + c * 8 + j, acc[j]);
      }
    }
  }

  // ===== flush: once every MMA has landed, ALL ten warps read the accumulators back - a warp reaches the TMEM lane
  // quarter (warp % 4), so quarters 0 and 1 are shared by three warps, quarters 2 and 3 by two, and each takes every
  // third / second 16-column group. (Measured: the flush is bound by the red.add throughput of L2, not by the warps
  // that issue it - 0.859 -> 0.853 ms over the 12 launches of a step.) =====
  {
    const int q = warp & 3, share = warp >> 2;
    const int nshare = (q + 8 < kThreadsW / 32) ? 3 : 2;
    const int row = q * 32 + lane;  // (ky, ci) = (row / kcx, row % kcx); ky == 3 is the discarded block
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
    mbar_wait(done_bar, 0);
    tc_fence_after();
    const int ky = row / p.kcx, ci = row % p.kcx;
    const int per = 3 * p.kcy / 16;  // 16-column groups per kz accumulator
    for (int g = share; g < 3 * per; g += nshare) {
      const int dz = g / per, c16 = g % per;
      uint32_t r[16];
      tmem_ld16(lane_base + (uint32_t)(dz * kNcols + c16 * 16), r);
      tmem_ld_wait();
      if (ky < 3) {
        const int col = c16 * 16;                      // kcy columns per kx block
        const int kx = 2 - col / p.kcy;
        const int tap = (kx * 3 + ky) * 3 + dz;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int co = coc * p.kcy + col % p.kcy + j;
          atomicAdd(p.dw + ((int64_t)co * 27 + tap) * p.Ct + p.cofs + cic * p.kcx + ci, __uint_as_float(r[j]));
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMma0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

int make_map(CUtensorMap* tm, const bf16* base, int N, int X, int Y, int Z, int C, int by, int cbox) {
  EncodeTiledFn enc = encode_tiled();
  FM_CHECK(enc != nullptr, FM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)Z, (cuuint64_t)Y, (cuuint64_t)X, (cuuint64_t)N};
  cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)Z * C * 2, (cuuint64_t)Y * Z * C * 2,
                           (cuuint64_t)X * Y * Z * C * 2};
  cuuint32_t box[5] = {(cuuint32_t)cbox, (cuuint32_t)kBZ, (cuuint32_t)by, 1, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)base, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_row_bytes(cbox * 2),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FM_CHECK(r == CUDA_SUCCESS, FM_ECUDA, "cuTensorMapEncodeTiled(wgrad march) failed: %d", (int)r);
  return FM_OK;
}

}  // namespace

int conv_wgrad_march_supported(int X, int Y, int Z, int Cin, int Cout, int ksize) {
  if (ksize != 3) return 0;
  if (Y % kBY != 0 || Z % kBZ != 0 || X < 2) return 0;
  if (!(Cin % kCC == 0 || Cin == 16) || !(Cout % kCC == 0 || Cout == 16)) return 0;
  return 1;
}

int k_conv3d_wgrad_march(fm_ctx* ctx, const bf16* x, const bf16* dy, float* dw_packed, int N, int X, int Y, int Z,
                         int Cin, int Cin_total, int cin_ofs, int Cout, float* db) {
  FM_CHECK(conv_wgrad_march_supported(X, Y, Z, Cin, Cout, 3), FM_EINVAL,
           "conv3d wgrad march: unsupported shape %dx%dx%d Cin=%d Cout=%d", X, Y, Z, Cin, Cout);
  WgMarchParams p;
  memset(&p, 0, sizeof(p));
  p.N = N;
  p.X = X;
  p.Y = Y;
  p.Z = Z;
  p.ny = Y / kBY;
  p.nz = Z / kBZ;
  p.kcx = (Cin % kCC == 0) ? kCC : 16;
  p.n_ci = Cin / p.kcx;
  p.kcy = (Cout % kCC == 0) ? kCC : 16;
  p.n_co = Cout / p.kcy;
  p.Ct = Cin_total;
  p.cofs = cin_ofs;
  p.dw = dw_packed;
  p.db = db;
  const int pairs = p.n_ci * p.n_co;
  const int cols = N * p.ny * p.nz;
  // CTAs per (ci, co) pair: at least 4 planes each; work units dealt as PlaneSplit describes (common.cuh)
  p.ctas_per_pair = std::max(1, std::min(ctx->num_sms / pairs, cols * X / 4));
  plane_split_setup(&p.split, cols, X, p.ctas_per_pair, 1.0);
  p.ctas_per_pair = std::min(p.ctas_per_pair, cols * p.split.nxc);
  FM_TRY(make_map(&p.tmX, x, N, X, Y, Z, Cin, kBY + 128 / p.kcx - 1, p.kcx));  // halo + discarded M blocks
  FM_TRY(make_map(&p.tmDY, dy, N, X, Y, Z, Cout, kBY, p.kcy));
  // five slab slots per kz ring, packed at the slab's own 9728 bytes (512-byte aligned: enough for SWIZZLE_64B / 32B,
  // whose pattern repeats every 512 / 256 bytes of shared-memory address)
  p.S3 = 5;
  p.xslot = kXSlotBytes;
  const size_t smem = (size_t)3 * p.S3 * p.xslot + (size_t)(kDyRing + kDyMirror) * kDyTile + 1024 + 512;
  static bool attr_set = false;
  if (!attr_set) {
    FM_CUDA(cudaFuncSetAttribute(conv3d_wgrad_march_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 kMaxDynSmem));
    attr_set = true;
  }
  const double vox = (double)N * X * Y * Z;
  ProfScope prof(ctx, "conv3d_wgrad_march", 2.0 * 27 * Cin * Cout * vox, vox * (Cin + Cout) * 2.0);
  FM_CUDA(launch_pdl(conv3d_wgrad_march_kernel, dim3(pairs * p.ctas_per_pair), dim3(kThreadsW), smem, ctx->stream, p));
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
