// conv_march.cu — "plane-marching" implicit-GEMM Conv3D 3x3x3 (fprop + dgrad) for layers whose whole filter bank fits
// in shared memory (the full-resolution layers that hold most of the U-Net's FLOPs).
//
// The per-tap kernel (conv_tc.cu) re-reads every activation tile 27x from L2 and, for Cout <= 64, is bound by the
// A-operand read from shared memory. This kernel removes both limits:
//
//   * a CTA owns a column of the volume: 16 (y) x 8 (z) output voxels = the 128 rows of one UMMA tile, and marches
//     along x. Per input plane it loads, once, three z-shifted y-haloed slabs (18 x 8 rows x KC channels, one TMA box
//     each; out-of-bounds rows zero-filled = 'same' padding). A dy shift is an 8-row (= one swizzle atom) offset of
//     the UMMA descriptor start address, a dz shift selects the slab copy, so all 9 (dy,dz) taps read the same
//     resident data.
//   * the three dx taps are stacked along N: one MMA with B = [W(dx=+1); W(dx=0); W(dx=-1)] (3*Cout rows) accumulates
//     plane xi into the TMEM accumulators of output planes xi-1, xi, xi+1 at once (a ring of accumulator blocks), so
//     each A byte read from shared memory feeds 3x the MMA work and every input plane is consumed exactly once.
//   * weights are loaded to shared memory once per CTA and stay resident for its whole lifetime.
//
// The issue path is shaped by what the round-1 ncu captures showed (profiles/README.md):
//
//   * the MMA-issuing warps were ISSUE bound (231 warp instructions per plane for 6 MMAs: per-plane recomputation
//     of descriptor constants, un-unrolled k loops, ring bookkeeping). Here Cout is a template parameter, every
//     per-source constant is hoisted out of the item loop, and a K chunk is issued by a fully unrolled
//     issue_chunk<NK>() (3 dy x NK MMAs, immediates only), about 70 instructions per plane.
//   * the epilogue spent a third of its time on the per-plane bias loads (LDG + long scoreboard); bias now lives in
//     registers for the CTA's lifetime, all TMEM loads of a plane are issued before one wait, and the accumulator
//     block is handed back (zeroed) before the bf16 conversion and the global stores.
//   * one accumulator ring shared by all issuing warps (the epilogue hands blocks back zeroed, every MMA
//     accumulates); the issue modes are described at the kernel.
//
// fprop: epilogue = bias + ReLU. dgrad: same kernel on dY with flipped/transposed weights, epilogue = ReLU mask of
// the producing block. Keras call site: Conv3D in create_convolution_block (fetal_net/model/unet3d/unet.py:102).
#include <algorithm>

#include "tc_ptx.cuh"

using namespace tcp;

namespace {

// Warp roles: warps 0-2 TMA producers (one per dz slab copy), warps 3-6 MMA issue (1, 3 or 4 of them active),
// warps 7.. epilogue: 4 warps for Cout = 16, 8 (two channel halves) from Cout = 32.
constexpr int kProdWarps = 3, kMmaWarps = 4, kEpi0 = kProdWarps + kMmaWarps;
__host__ __device__ constexpr int march2_epw(int cn) { return cn >= 32 ? 8 : 4; }
__host__ __device__ constexpr int march2_threads(int cn) { return 32 * (kEpi0 + march2_epw(cn)); }
constexpr int kBY = 16, kBZ = 8, kSlabRows = (kBY + 2) * kBZ;  // 144 rows per slab
constexpr uint32_t kSlot = kSlabRows * 128;                    // 18432 B (1024-aligned): slab slot at KC = 64
constexpr int kMaxRing2 = 16;

struct alignas(64) March2Params {
  CUtensorMap tmA[2];  // activations, box (KC, 8, 18, 1, 1)
  CUtensorMap tmW[2];  // march-packed weights, 2-D (KC, rows), box (KC, 3*Cn)
  int nsrc;
  int nchunks[2];
  int KC[2];
  uint32_t wofs[2];  // byte offset of the source's resident weights inside the W region
  int N, X, Y, Z;
  int ny, nz;
  PlaneSplit split;  // how the (column, x) plane-tiles are dealt to the CTAs (common.cuh)
  int R;       // accumulator ring blocks (power of two)
  int stages;  // slab slots, a multiple of 3 (one private ring per dz slab copy)
  int out_C, out_cofs, relu;
  uint32_t w_bytes;   // bytes the weight TMA loads deliver (mbarrier expect_tx)
  uint32_t w_region;  // shared-memory bytes reserved for them (1024-aligned per source)
  uint32_t slot;      // bytes per slab slot (1024-aligned)
  const float* bias;
  bf16* out;
  const bf16* mask;
};

// 3 dy taps x NK k-steps of one resident K chunk: A = slab (dy = +8 rows = +KC 16-byte units), B = the dx-stacked
// filter tile of (dz, dy); every MMA accumulates into the ring blocks at `col`.
template <int NK>
__device__ __forceinline__ void issue_chunk(uint32_t col, uint32_t a_lo, uint32_t b_lo, uint32_t hi32,
                                            uint32_t btile16, uint32_t idesc) {
#pragma unroll
  for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
    for (int k = 0; k < NK; ++k)
      umma_bf16_lh_elect(col, a_lo + (uint32_t)(dy * NK * 16 + 2 * k), hi32, b_lo + (uint32_t)dy * btile16 + 2u * (uint32_t)k,
                         hi32, idesc, 1u);
  }
}

__device__ __forceinline__ void issue_chunk_nk(int nk, uint32_t col, uint32_t a_lo, uint32_t b_lo, uint32_t hi32,
                                               uint32_t btile16, uint32_t idesc) {
  if (nk == 2)
    issue_chunk<2>(col, a_lo, b_lo, hi32, btile16, idesc);
  else if (nk == 4)
    issue_chunk<4>(col, a_lo, b_lo, hi32, btile16, idesc);
  else
    issue_chunk<1>(col, a_lo, b_lo, hi32, btile16, idesc);
}

// Issue modes (who sends the MMAs of an input plane to the tensor pipe):
//   0  one warp, every plane, dz = 0, 1, 2 in turn: fixed fp32 summation order (bit-reproducible).
//   1  three warps, warp w = slab copy dz = w of every plane (summation order follows their interleaving).
//   2  three warps take whole planes in turn (plane t -> warp t mod 3); a token (mbarrier) passes from the warp that
//      has issued plane t to the owner of plane t + 1, so the MMAs reach the pipe in the order of mode 0
//      (bit-reproducible) while barrier waits, descriptor arithmetic and commits of neighbouring planes overlap.
// (Unordered plane-owner variants - mode 2 without the token, three and four warps - were measured twice, with 4-deep and
// with 6- to 12-deep slab rings: no faster than mode 1 on any layer (profiles/README.md); they are not built.)
// In mode 2 an accumulator block receives MMAs of three different threads (planes b-1, b, b+1): every plane
// owner commits to the tfull barrier of each block it fed (tcgen05.commit tracks the executing thread's MMAs only),
// and the owner of the centre plane stands in for a neighbour plane that does not exist at the volume boundary.
template <int MODE, int CN>
__global__ void __launch_bounds__(march2_threads(CN), 1) conv3d_march2_kernel(const __grid_constant__ March2Params p) {
  constexpr int NMMA = MODE == 0 ? 1 : 3;
  constexpr bool PLANE_OWNERS = MODE >= 2;
  constexpr int EPW = march2_epw(CN);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t w_base = smem0;
  const uint32_t a_base = smem0 + p.w_region;
  const uint32_t bar0 = a_base + (uint32_t)p.stages * p.slot;
  const uint32_t nst = (uint32_t)p.stages;
  // barrier layout: full[stages] | empty[stages] | tfull[16] | tempty[16] | wfull | token[4] | tmem slot
  const uint32_t full0 = bar0, empty0 = bar0 + 8u * nst, tfull0 = bar0 + 16u * nst, tempty0 = tfull0 + 8u * kMaxRing2;
  const uint32_t wfull_bar = tempty0 + 8u * kMaxRing2;
  const uint32_t tok0 = wfull_bar + 8u;  // mode 2: one "your turn" barrier per issuing warp
  const uint32_t tmem_slot = tok0 + 32u;

  constexpr uint32_t Cn = (uint32_t)CN;
  const uint32_t R = (uint32_t)p.R;
  uint32_t tmem_cols = 32;
  while (tmem_cols < R * Cn) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.nsrc; ++s) {
      prefetch_tmap(&p.tmA[s]);
      prefetch_tmap(&p.tmW[s]);
    }
  }
  if (warp == kProdWarps) {
    if (lane == 0) {
      for (uint32_t s = 0; s < nst; ++s) {
        mbar_init(full0 + 8u * s, 1);
        mbar_init(empty0 + 8u * s, 1);
      }
      for (uint32_t b = 0; b < R; ++b) {
        // mode 0: the one issuing warp commits once per block. mode 1: one commit per dz warp. mode 2: one arrival
        // per contributing plane (b-1, b, b+1)
        mbar_init(tfull0 + 8u * b, MODE == 0 ? 1u : 3u);
        mbar_init(tempty0 + 8u * b, (uint32_t)EPW);  // one elected arrival per epilogue warp
      }
      mbar_init(wfull_bar, 1);
      for (uint32_t w = 0; w < 4; ++w) mbar_init(tok0 + 8u * w, 1);
      fence_barrier_init();
      if (MODE == 2) mbar_arrive(tok0);  // plane 0 may go at once
    }
    __syncwarp();
    tmem_alloc(tmem_slot, tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  // `item` = blockIdx.x + k * gridDim.x names the k-th work unit of this CTA (PlaneSplit in common.cuh).
  // Returns false past the last one.
  auto decode = [&](int item, int& n, int& iy, int& iz, int& xa, int& xb) -> bool {
    int col;
    if (!plane_split_next(p.split, (int)blockIdx.x, (int)gridDim.x, item / (int)gridDim.x, col, xa, xb)) return false;
    iz = col % p.nz;
    const int r = col / p.nz;
    iy = r % p.ny;
    n = r / p.ny;
    return true;
  };


  // make the values the producer / MMA warps compute on provably warp-uniform
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);
  const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
  const uint32_t S3 = nst / 3u;

  if (warp_u < kProdWarps) {
    // ===== producer warps (all lanes converged, one elected lane issues): warp dz feeds the ring of S3 slots of ITS
    //       z-shifted slab copy, one slab per (plane, source, chunk). Warp 0 first loads the resident filter bank. =====
    const int dz = warp_u;
    if (dz == 0) {
      mbar_expect_tx_elect(wfull_bar, p.w_bytes);
      for (int s = 0; s < p.nsrc; ++s) {
        const uint32_t tile = 3u * Cn * (uint32_t)p.KC[s] * 2u;
        for (int t = 0; t < p.nchunks[s] * 9; ++t)
          tma_load_2d_elect(w_base + p.wofs[s] + (uint32_t)t * tile, &p.tmW[s], wfull_bar, 0, t * 3 * CN);
      }
    }
    // the weights do not depend on the previous kernel in the stream; the activation slabs do
    pdl_wait();
    if (dz == 0) pdl_launch_dependents();
    uint32_t sidx = 0, sph = 0;
    const uint32_t ring0 = (uint32_t)dz * S3;
    const uint32_t bytes0 = (uint32_t)kSlabRows * (uint32_t)p.KC[0] * 2u;
    const uint32_t bytes1 = (uint32_t)kSlabRows * (uint32_t)p.KC[1] * 2u;
    const int nch0 = p.nchunks[0], nch1 = p.nsrc > 1 ? p.nchunks[1] : 0;
    const int kc0 = p.KC[0], kc1 = p.KC[1];
    for (int item = blockIdx.x, n, iy, iz, xa, xb; decode(item, n, iy, iz, xa, xb); item += gridDim.x) {
      const int x_first = max(xa - 1, 0), x_last = min(xb, p.X - 1);
      const int yc = iy * kBY - 1, zc = iz * kBZ - 1 + dz;
      for (int xi = x_first; xi <= x_last; ++xi) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const int nch = s == 0 ? nch0 : nch1;
          const uint32_t bytes = s == 0 ? bytes0 : bytes1;
          const int kc = s == 0 ? kc0 : kc1;
          for (int ch = 0; ch < nch; ++ch) {
            const uint32_t stage = ring0 + sidx;
            const uint32_t fb = full0 + 8u * stage;
            mbar_wait(empty0 + 8u * stage, sph ^ 1u);
            mbar_expect_tx_elect(fb, bytes);
            tma_load_5d_elect(a_base + stage * p.slot, &p.tmA[s], fb, ch * kc, zc, yc, xi, n);
            if (++sidx == S3) {
              sidx = 0;
              sph ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp_u < kEpi0) {
    // ===== MMA warps. All MMAs accumulate; the epilogue hands accumulator blocks back zeroed. =====
    const int mw = warp_u - kProdWarps;
    if (mw < NMMA) {
      const int dz_lo = (MODE == 1) ? mw : 0;
      constexpr int NDZ = (MODE == 1) ? 1 : 3;  // slab copies this warp walks per plane
      const uint32_t ring_mask = R - 1u;
      const uint32_t ring_shift = 31u - (uint32_t)__clz((int)R);
      constexpr uint32_t idesc1 = make_idesc(128, CN, 0, 0);
      constexpr uint32_t idesc2 = make_idesc(128, 2 * CN, 0, 0);
      constexpr uint32_t idesc3 = make_idesc(128, 3 * CN, 0, 0);
      // per-source constants (16-byte descriptor units)
      uint32_t hi32[2], btile16[2], blk16[2], bsrc[2];
      int nk[2], nch[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const uint32_t row_bytes = (uint32_t)p.KC[s] * 2u;
        hi32[s] = desc_hi(8u * row_bytes, layout_code((int)row_bytes));
        btile16[s] = (3u * Cn * row_bytes) >> 4;
        blk16[s] = (Cn * row_bytes) >> 4;
        bsrc[s] = desc_lo(w_base + p.wofs[s], 16u);
        nk[s] = p.KC[s] >> 4;
        nch[s] = s < p.nsrc ? p.nchunks[s] : 0;
      }
      const uint32_t a_lo0 = desc_lo(a_base, 16u);
      const uint32_t slot16 = p.slot >> 4;
      mbar_wait(wfull_bar, 0);
      tc_fence_after();
      // slab-ring positions. Modes 0 / 1: one (index, phase) per dz walked, advanced chunk by chunk. Plane owners: the
      // three dz rings move in lock step (CP chunks per plane each) and this warp holds every NMMA-th plane:
      // (sidx[0], sph[0]) is the position of ITS next plane's first chunk and jumps NMMA * CP positions per plane.
      uint32_t sidx[3] = {0u, 0u, 0u}, sph[3] = {0u, 0u, 0u};
      const uint32_t CP = (uint32_t)(nch[0] + nch[1]);
      uint32_t jump_idx = 0, jump_wrap = 0;  // (NMMA * CP) mod S3 and floor(NMMA * CP / S3) mod 2
      uint32_t turn = 0, tokph = 0;          // plane owners: planes until this warp's turn; mode 2: token parity
      if (PLANE_OWNERS) {
        const uint32_t pos = (uint32_t)mw * CP;
        sidx[0] = pos % S3;
        sph[0] = (pos / S3) & 1u;
        jump_idx = ((uint32_t)NMMA * CP) % S3;
        jump_wrap = (((uint32_t)NMMA * CP) / S3) & 1u;
        turn = (uint32_t)mw;
      }
      uint32_t ocount = 0;
      for (int item = blockIdx.x, n, iy, iz, xa, xb; decode(item, n, iy, iz, xa, xb); item += gridDim.x) {
        const int x_first = max(xa - 1, 0), x_last = min(xb, p.X - 1);
        for (int xi = x_first; xi <= x_last; ++xi) {
          if (PLANE_OWNERS) {
            if (turn != 0) {
              --turn;
              continue;
            }
            turn = NMMA - 1;
          }
          const int lo = max(xa, xi - 1), hi = min(xb - 1, xi + 1);  // output planes fed by plane xi
          const uint32_t j_lo = (uint32_t)(lo - (xi - 1));
          const uint32_t nblk = (uint32_t)(hi - lo + 1);
          const uint32_t seq_lo = ocount + (uint32_t)(lo - xa);
          const uint32_t rb_lo = seq_lo & ring_mask;
          // blocks FIRST touched by this plane must have been drained (and zeroed) by the epilogue (issue is in plane
          // order in every mode, so later planes find them checked)
          if (xi == x_first) {
            for (uint32_t j = 0; j < nblk; ++j) {
              const uint32_t seq = seq_lo + j;
              mbar_wait(tempty0 + 8u * (seq & ring_mask), (seq >> ring_shift) & 1u);
            }
          } else if (xi + 1 <= xb - 1) {
            const uint32_t seq = ocount + (uint32_t)(xi + 1 - xa);
            mbar_wait(tempty0 + 8u * (seq & ring_mask), (seq >> ring_shift) & 1u);
          }
          // the <= 3 consecutive ring blocks, split only where the ring wraps
          const uint32_t nA = min(nblk, R - rb_lo), nB = nblk - nA;
          const uint32_t colA = tmem_base + rb_lo * Cn, colB = tmem_base;
          const uint32_t idA = nA == 3 ? idesc3 : (nA == 2 ? idesc2 : idesc1);
          const uint32_t idB = nB == 2 ? idesc2 : idesc1;
          if (MODE == 2) {
            // what this plane needs first is checked BEFORE taking the token
            mbar_wait(full0 + 8u * sidx[0], sph[0]);
            mbar_wait(tok0 + 8u * (uint32_t)mw, tokph);
            tokph ^= 1u;
          }
          tc_fence_after();
#pragma unroll
          for (int dzi = 0; dzi < NDZ; ++dzi) {
            const int dz = dz_lo + dzi;
            uint32_t ci = sidx[PLANE_OWNERS ? 0 : dzi], cp = sph[PLANE_OWNERS ? 0 : dzi];
#pragma unroll
            for (int s = 0; s < 2; ++s) {
              const uint32_t b_s = bsrc[s] + (uint32_t)(dz * 3) * btile16[s] + j_lo * blk16[s];
              for (int ch = 0; ch < nch[s]; ++ch) {
                const uint32_t stage = (uint32_t)dz * S3 + ci;
                mbar_wait(full0 + 8u * stage, cp);
                tc_fence_after();
                const uint32_t a_lo = a_lo0 + stage * slot16;
                const uint32_t b_lo = b_s + (uint32_t)(ch * 9) * btile16[s];
                issue_chunk_nk(nk[s], colA, a_lo, b_lo, hi32[s], btile16[s], idA);
                if (nB) issue_chunk_nk(nk[s], colB, a_lo, b_lo + nA * blk16[s], hi32[s], btile16[s], idB);
                umma_commit_elect(empty0 + 8u * stage);
                if (++ci == S3) {
                  ci = 0;
                  cp ^= 1u;
                }
              }
            }
            if (!PLANE_OWNERS) {
              sidx[dzi] = ci;
              sph[dzi] = cp;
            }
          }
          if (PLANE_OWNERS) {
            // mode 2: every MMA of this plane is in the queue, the owner of the next plane may issue
            if (MODE == 2) mbar_arrive_elect(tok0 + 8u * (uint32_t)(mw == NMMA - 1 ? 0 : mw + 1));
            sidx[0] += jump_idx;
            uint32_t w = jump_wrap;
            if (sidx[0] >= S3) {
              sidx[0] -= S3;
              w ^= 1u;
            }
            sph[0] ^= w;
            // one arrival per block this plane fed; the owner of the centre plane also arrives for a neighbour plane
            // that does not exist (volume boundary), so that every block sees exactly three
            for (uint32_t j = 0; j < nblk; ++j) umma_commit_elect(tfull0 + 8u * ((seq_lo + j) & ring_mask));
            if (xi >= xa && xi <= xb - 1) {
              const uint32_t cb = tfull0 + 8u * ((ocount + (uint32_t)(xi - xa)) & ring_mask);
              if (xi - 1 < x_first) mbar_arrive_elect(cb);
              if (xi + 1 > x_last) mbar_arrive_elect(cb);
            }
          } else {
            // output planes completed by this input plane (mode 1: each dz warp contributes one arrival)
            if (xi - 1 >= xa) umma_commit_elect(tfull0 + 8u * ((ocount + (uint32_t)(xi - 1 - xa)) & ring_mask));
            if (xi == x_last && xi <= xb - 1) umma_commit_elect(tfull0 + 8u * ((ocount + (uint32_t)(xi - xa)) & ring_mask));
          }
        }
        ocount += (uint32_t)(xb - xa);
      }
    }
  } else {
    // ===== epilogue: EPW warps. Warp e works on TMEM lane quarter e & 3 (row = (y, z) of the 16 x 8 column) and, for
    //       Cout >= 32, on one half of the output channels (e >> 2). Per plane: wait for the loaded accumulator, hand
    //       the block back zeroed (one elected arrival per warp), convert, and START the TMEM load of the next plane
    //       before the global stores of this one - the round-1/early-round-2 captures showed this loop, not the tensor
    //       pipe, setting the pace (a plane took 1230 cycles with the MMAs switched off). =====
    constexpr int CW = CN / (EPW / 4);  // channels per epilogue warp
    constexpr int NCG = CW / 16;
    const int ew = warp - kEpi0;
    const int q = warp & 3, half = ew >> 2;  // a warp can only touch the TMEM lane quarter (warp id mod 4)
    const int row = q * 32 + lane;
    const int yl = row >> 3, zl = row & 7;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * CW);
    const uint32_t ring_mask = R - 1u;
    const uint32_t ring_shift = 31u - (uint32_t)__clz((int)R);
    // hand every accumulator block to the MMA warps zeroed (TMEM is not initialised by the allocation)
    for (uint32_t b = 0; b < R; ++b) {
#pragma unroll
      for (int c16 = 0; c16 < NCG; ++c16) tmem_st16_zero(lane_base + b * Cn + (uint32_t)(c16 * 16));
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty0 + 8u * b);
    }
    // bias stays in registers for the CTA's lifetime
    float bias_r[CW];
    if (p.bias != nullptr) {
#pragma unroll
      for (int j = 0; j < CW / 4; ++j) {
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + half * CW) + j);
        bias_r[4 * j] = b4.x;
        bias_r[4 * j + 1] = b4.y;
        bias_r[4 * j + 2] = b4.z;
        bias_r[4 * j + 3] = b4.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < CW; ++j) bias_r[j] = 0.f;
    }
    const bool relu = p.relu != 0;
    const bool has_mask = p.mask != nullptr;
    // iterator over this CTA's output planes (ring sequence number g counts them across items)
    int it_item = blockIdx.x, it_xo = 0, it_xb = 0;
    int64_t it_off = 0;
    const int64_t it_step = (int64_t)p.Y * p.Z * p.out_C;
    auto it_load = [&]() -> bool {
      int n, iy, iz, xa, xb;
      if (!decode(it_item, n, iy, iz, xa, xb)) return false;
      it_xo = xa;
      it_xb = xb;
      const int64_t v0 = (((int64_t)n * p.X + xa) * p.Y + (iy * kBY + yl)) * p.Z + (iz * kBZ + zl);
      it_off = v0 * p.out_C + p.out_cofs + half * CW;
      return true;
    };
    auto it_next = [&]() -> bool {
      if (++it_xo < it_xb) {
        it_off += it_step;
        return true;
      }
      it_item += gridDim.x;
      return it_load();
    };
    uint32_t r[NCG][16];
    constexpr bool kDeep = CN <= 32;  // Cout = 64 has no registers to spare for a second plane of mask
    uint4 mk[2 * NCG], mk1[kDeep ? 2 * NCG : 1];
    bool have = it_load();
    int64_t off = it_off;
    uint32_t g = 0;
    // dgrad: the ReLU mask of a plane is requested TWO planes ahead of its use (registers mk -> this plane, mk1 -> the
    // next one, mk2 in flight): one plane period (~0.8 us) did not cover the DRAM latency under load - the masked
    // 32 -> 32 launch at 64^3 took 141 us against 88 us for the same shape without a mask.
    if (have && has_mask) {
      const uint4* mp = reinterpret_cast<const uint4*>(p.mask + off);
#pragma unroll
      for (int h = 0; h < 2 * NCG; ++h) mk[h] = __ldg(mp + h);
    }
    bool have1 = false;
    int64_t off1 = 0;
    if constexpr (kDeep) {
      have1 = have && it_next();
      off1 = it_off;
      if (have1 && has_mask) {
        const uint4* mp = reinterpret_cast<const uint4*>(p.mask + off1);
#pragma unroll
        for (int h = 0; h < 2 * NCG; ++h) mk1[h] = __ldg(mp + h);
      }
    }
    if (have) {
      mbar_wait(tfull0, 0);
      tc_fence_after();
#pragma unroll
      for (int c16 = 0; c16 < NCG; ++c16) tmem_ld16(lane_base + (uint32_t)(c16 * 16), r[c16]);
    }
    while (have) {
      const bool have_next = kDeep ? have1 : it_next();
      const bool have2 = kDeep ? (have1 && it_next()) : have_next;  // the plane whose mask is requested now
      const int64_t off2 = it_off;
      uint4 mk2[2 * NCG];
      if (have2 && has_mask) {
        const uint4* mp = reinterpret_cast<const uint4*>(p.mask + off2);
#pragma unroll
        for (int h = 0; h < 2 * NCG; ++h) mk2[h] = __ldg(mp + h);
      }
      const uint32_t rb = g & ring_mask;
      const uint32_t taddr = lane_base + rb * Cn;
      tmem_ld_wait();
#pragma unroll
      for (int c16 = 0; c16 < NCG; ++c16) tmem_st16_zero(taddr + (uint32_t)(c16 * 16));
      uint4 o[NCG][2];
#pragma unroll
      for (int c16 = 0; c16 < NCG; ++c16) {
        float f[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(r[c16][j]) + bias_r[c16 * 16 + j];
        if (relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
        }
        if (has_mask) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint4 mv = mk[2 * c16 + h];
            const __nv_bfloat162* mh = reinterpret_cast<const __nv_bfloat162*>(&mv);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 mf = __bfloat1622float2(mh[j]);
              if (!(mf.x > 0.f)) f[8 * h + 2 * j] = 0.f;
              if (!(mf.y > 0.f)) f[8 * h + 2 * j + 1] = 0.f;
            }
          }
        }
        __nv_bfloat162* oh = reinterpret_cast<__nv_bfloat162*>(o[c16]);
#pragma unroll
        for (int j = 0; j < 8; ++j) oh[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
      }
      // the block is free (and zero) again: one arrival per warp
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty0 + 8u * rb);
      if (have_next) {
        const uint32_t g1 = g + 1u;
        mbar_wait(tfull0 + 8u * (g1 & ring_mask), (g1 >> ring_shift) & 1u);
        tc_fence_after();
        const uint32_t tnext = lane_base + (g1 & ring_mask) * Cn;
#pragma unroll
        for (int c16 = 0; c16 < NCG; ++c16) tmem_ld16(tnext + (uint32_t)(c16 * 16), r[c16]);
      }
#pragma unroll
      for (int c16 = 0; c16 < NCG; ++c16) {
        uint4* op = reinterpret_cast<uint4*>(p.out + off + c16 * 16);
        op[0] = o[c16][0];
        op[1] = o[c16][1];
      }
      if constexpr (kDeep) {
        off = off1;
        off1 = off2;
#pragma unroll
        for (int h = 0; h < 2 * NCG; ++h) {
          mk[h] = mk1[h];
          mk1[h] = mk2[h];
        }
        have = have1;
        have1 = have2;
      } else {
        off = off2;
#pragma unroll
        for (int h = 0; h < 2 * NCG; ++h) mk[h] = mk2[h];
        have = have_next;
      }
      ++g;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kProdWarps) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// march pack: Wm[chunk][dz][dy][kxr][n][kc] = P[n][tap(kx = 2 - kxr, ky = dy, kz = dz)][kofs + chunk*KC + kc]
__global__ void repack_march_kernel(const bf16* __restrict__ P, bf16* __restrict__ Wm, int Nrows, int Ktot,
                                    int kofs, int Cs, int KC) {
  const int64_t total = (int64_t)(Cs / KC) * 27 * Nrows * KC;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total) return;
  const int kc = (int)(g % KC);
  int64_t t = g / KC;
  const int n = (int)(t % Nrows);
  t /= Nrows;
  const int kxr = (int)(t % 3);
  t /= 3;
  const int dy = (int)(t % 3);
  t /= 3;
  const int dz = (int)(t % 3);
  const int ch = (int)(t / 3);
  const int tap = ((2 - kxr) * 3 + dy) * 3 + dz;
  Wm[g] = P[((int64_t)n * 27 + tap) * Ktot + kofs + ch * KC + kc];
}

bool chan_ok_m(int C) { return C == 16 || C == 32 || C == 64 || (C > 64 && C % 64 == 0); }

// resident filter bank: 27 taps * Cin * Cout * 2 B per source, each source region 1024-aligned
uint32_t march_w_region(int C1, int C2, int Cn) {
  const uint32_t a = ((uint32_t)27 * C1 * Cn * 2u + 1023u) & ~1023u;
  const uint32_t b = ((uint32_t)27 * C2 * Cn * 2u + 1023u) & ~1023u;
  return a + b;
}

template <int MODE, int CN>
int launch_march2(fm_ctx* ctx, const March2Params& p, size_t smem, int grid) {
  static bool attr_set = false;
  if (!attr_set) {
    FM_CUDA(cudaFuncSetAttribute(conv3d_march2_kernel<MODE, CN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 kMaxDynSmem));
    attr_set = true;
  }
  FM_CUDA(launch_pdl(conv3d_march2_kernel<MODE, CN>, dim3(grid), dim3(march2_threads(CN)), smem, ctx->stream, p));
  return FM_OK;
}

}  // namespace

// channels per source supported / whole filter bank + >= 3 slab stages fit in shared memory
int conv_march_supported(int X, int Y, int Z, int C1, int C2, int Cout, int ksize) {
  if (ksize != 3) return 0;
  if (Y % kBY != 0 || Z % kBZ != 0 || X < 2) return 0;
  if (!(Cout == 16 || Cout == 32 || Cout == 64)) return 0;
  if (!chan_ok_m(C1) || (C2 != 0 && !chan_ok_m(C2))) return 0;
  return (int64_t)march_w_region(C1, C2, Cout) + 3 * (int64_t)kSlot + 2048 <= kMaxDynSmem;
}

int64_t conv_march_pack_elems(int Cs, int Cout) { return (int64_t)27 * Cs * Cout; }

int conv_march_kc(int C1, int C2, int Cout, int Cs) {
  const int kc = std::min(Cs, 64);
  if (kc < 64) return kc;
  const int full_slots = (kMaxDynSmem - 2048 - (int)march_w_region(C1, C2, Cout)) / (int)kSlot;
  return full_slots < 6 ? 32 : 64;
}

// P: bf16 pack [Nrows][27][Ktot]; writes the march pack of channel range [kofs, kofs+Cs)
int k_repack_march(fm_ctx* ctx, const bf16* P, bf16* Wm, int Nrows, int Ktot, int kofs, int Cs, int KC) {
  const int64_t total = (int64_t)27 * Cs * Nrows;
  ProfScope prof(ctx, "repack_march", 0.0, (double)total * 4.0);
  repack_march_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(P, Wm, Nrows, Ktot, kofs, Cs, KC);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}

int k_conv3d_march(fm_ctx* ctx, const bf16* x1, const bf16* x2, const bf16* wm1, const bf16* wm2, const float* bias,
                   bf16* y, const bf16* mask, int N, int X, int Y, int Z, int C1, int C2, int Cout, int relu, int out_C,
                   int out_cofs, bool reproducible) {
  FM_CHECK(conv_march_supported(X, Y, Z, C1, C2, Cout, 3), FM_EINVAL,
           "conv3d march: unsupported shape %dx%dx%d C1=%d C2=%d Cout=%d", X, Y, Z, C1, C2, Cout);
  EncodeTiledFn enc = encode_tiled();
  FM_CHECK(enc != nullptr, FM_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  March2Params p;
  memset(&p, 0, sizeof(p));
  p.nsrc = C2 > 0 ? 2 : 1;
  p.N = N;
  p.X = X;
  p.Y = Y;
  p.Z = Z;
  p.ny = Y / kBY;
  p.nz = Z / kBZ;
  p.R = std::min(kMaxRing2, 512 / Cout);
  p.out_C = out_C;
  p.out_cofs = out_cofs;
  p.relu = relu;
  p.bias = bias;
  p.out = y;
  p.mask = mask;
  const int Cs[2] = {C1, C2};
  const bf16* xs[2] = {x1, x2};
  const bf16* wms[2] = {wm1, wm2};
  uint32_t wofs = 0, wbytes = 0;
  p.KC[1] = 16;  // harmless defaults for the unused second source
  for (int s = 0; s < p.nsrc; ++s) {
    const int KC = conv_march_kc(C1, C2, Cout, Cs[s]);
    p.KC[s] = KC;
    p.nchunks[s] = Cs[s] / KC;
    p.wofs[s] = wofs;
    wofs += ((uint32_t)27 * Cs[s] * Cout * 2u + 1023u) & ~1023u;
    wbytes += (uint32_t)27 * Cs[s] * Cout * 2u;
    {
      cuuint64_t dims[5] = {(cuuint64_t)Cs[s], (cuuint64_t)Z, (cuuint64_t)Y, (cuuint64_t)X, (cuuint64_t)N};
      cuuint64_t strides[4] = {(cuuint64_t)Cs[s] * 2, (cuuint64_t)Z * Cs[s] * 2, (cuuint64_t)Y * Z * Cs[s] * 2,
                               (cuuint64_t)X * Y * Z * Cs[s] * 2};
      cuuint32_t box[5] = {(cuuint32_t)KC, (cuuint32_t)kBZ, (cuuint32_t)(kBY + 2), 1, 1};
      cuuint32_t estr[5] = {1, 1, 1, 1, 1};
      CUresult r = enc(&p.tmA[s], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)xs[s], dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_row_bytes(KC * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      FM_CHECK(r == CUDA_SUCCESS, FM_ECUDA, "cuTensorMapEncodeTiled(march act) failed: %d", (int)r);
    }
    {
      const cuuint64_t rows = (cuuint64_t)p.nchunks[s] * 27 * Cout;
      cuuint64_t dims[2] = {(cuuint64_t)KC, rows};
      cuuint64_t strides[1] = {(cuuint64_t)KC * 2};
      cuuint32_t box[2] = {(cuuint32_t)KC, (cuuint32_t)(3 * Cout)};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = enc(&p.tmW[s], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)wms[s], dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_row_bytes(KC * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      FM_CHECK(r == CUDA_SUCCESS, FM_ECUDA, "cuTensorMapEncodeTiled(march weights) failed: %d", (int)r);
    }
  }
  p.w_bytes = wbytes;
  p.w_region = wofs;
  // slot = one slab at the widest K chunk in use (18 KB at KC = 64, 9 KB when every source runs at KC <= 32)
  p.slot = (uint32_t)kSlabRows * (uint32_t)std::max(p.KC[0], p.nsrc > 1 ? p.KC[1] : 0) * 2u;
  // slots start on a multiple of the swizzle period: 1 KB for 128-byte rows, 512 B (256 B) for 64- (32-) byte rows
  const uint32_t slot_align = std::max(p.KC[0], p.nsrc > 1 ? p.KC[1] : 0) >= 64 ? 1024u : 512u;
  p.slot = (p.slot + slot_align - 1u) & ~(slot_align - 1u);
  int stages = (kMaxDynSmem - 2048 - (int)wofs) / (int)p.slot;
  // three private rings (one per dz slab copy), as deep as shared memory allows: the slabs of a plane are requested a
  // ring-depth ahead of their MMAs, and four planes did not cover the TMA round trip. 36 = what the 1 KB barrier region
  // holds.
  stages = std::min(stages, 36) / 3 * 3;
  FM_CHECK(stages >= 3, FM_EINVAL, "conv3d march: filter bank leaves no room for the slab rings");
  p.stages = stages;
  const size_t smem = (size_t)wofs + (size_t)stages * p.slot + 2048;
  FM_CHECK(smem <= (size_t)kMaxDynSmem, FM_EINVAL, "conv3d march: %zu B of shared memory needed", smem);
  int grid = std::max(1, std::min(N * p.ny * p.nz * X / 4, ctx->num_sms));
  plane_split_setup(&p.split, N * p.ny * p.nz, X, grid, 1.4);
  grid = std::min(grid, N * p.ny * p.nz * p.split.nxc);
  const double vox = (double)N * X * Y * Z;
  ProfScope prof(ctx, mask != nullptr || bias == nullptr ? "conv3d_march_dgrad" : "conv3d_march_fprop",
                 2.0 * 27 * (C1 + C2) * Cout * vox, vox * (C1 + C2 + Cout) * 2.0);
  // issue mode (see the kernel): one issuing warp keeps up with the 96-cycle MMAs of Cout = 64 (mode 0); narrower
  // layers split the issue three ways, in a fixed order where the result has to be bit-reproducible (mode 2)
  int rc;
  if (Cout == 64)
    rc = launch_march2<0, 64>(ctx, p, smem, grid);
  else if (Cout == 32)
    rc = reproducible ? launch_march2<2, 32>(ctx, p, smem, grid) : launch_march2<1, 32>(ctx, p, smem, grid);
  else
    rc = reproducible ? launch_march2<2, 16>(ctx, p, smem, grid) : launch_march2<1, 16>(ctx, p, smem, grid);
  FM_TRY(rc);
  FM_LAUNCH_OK(ctx);
  return FM_OK;
}
