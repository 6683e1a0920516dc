// General convolution layers of the DRUNet denoiser as implicit GEMM on tcgen05 tensor cores (sm_100a):
//   CG_CONV3  3x3, stride 1, zero padding 1, C -> C      (the residual blocks at 128 / 256 / 512 channels)
//   CG_DOWN2  2x2, stride 2, no padding,     C -> 2C     (KAIR "strideconv" downsampling)
//   CG_UP2    2x2, stride 2 transposed,      C -> C/2    (KAIR "convtranspose" upsampling; one 1x1 GEMM with N = 4 C/2,
//                                                          (output quadrant (dy, dx), channel))
// Replaces the cuDNN fp32 convolutions behind deepinv.models.DRUNet.forward (constructed at sampling_images.py:136,
// called at restoration_algorithms.py:238); architecture restated in oracle/image_oracle.py (KAIR UNetRes).
//
// Unlike the 64-channel layers (conv_tc.cu), the weights of these layers (up to 9 x 512 x 512 bf16 = 4.7 MB) do not fit
// in shared memory, so both operands stream: for every (tap, 64-channel block) the TMA producer loads an A box
// (128 "tile pixels" x 64 channels; PX pixels x ROWS image rows, shifted by the tap, OOB zero fill = conv padding) and
// a B box (N_TILE output channels x 64) into a ring; one elected thread issues 4 K16 MMAs per box into a TMEM
// accumulator; 8 epilogue warps add the residual inputs, apply ReLU, convert to bf16 and store NHWC.
// Activations bf16 NHWC [B][H][W][C]; weights bf16 [tap][Cout][Cin].
#include <cuda_bf16.h>

#include <algorithm>
#include <utility>
#include <vector>

#include "common.cuh"
#include "conv_api.cuh"
#include "sm100.cuh"

namespace psgla {
using namespace sm100;

enum { CG_CONV3 = 0, CG_DOWN2 = 1, CG_UP2 = 2 };

constexpr int CG_EPI_WARPS = 8;
constexpr int CG_NACC = 2;

// The single-CTA kernel: N tiles of 64 columns, i.e. an output channel count that is an odd multiple of 64 (3x3 and stride-2
// convs); every wider N tile runs on the CTA pair below.
template <int N_TILE>
struct CgCfg {
  static constexpr int THREADS = 64 + 32 * CG_EPI_WARPS;
  static constexpr int A_BYTES = 128 * 128;     // 128 tile pixels x 64 channels bf16
  static constexpr int B_BYTES = N_TILE * 128;  // N_TILE output channels x 64 input channels bf16
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int NSTAGE = (196608 / STAGE_BYTES) > 8 ? 8 : (196608 / STAGE_BYTES);
  static constexpr int OFF_BAR = NSTAGE * STAGE_BYTES;
  static constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
  static constexpr int TMEM_COLS = (CG_NACC * N_TILE) < 32 ? 32 : CG_NACC * N_TILE;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of one CTA");
  static_assert((TMEM_COLS & (TMEM_COLS - 1)) == 0 && TMEM_COLS <= 512, "TMEM columns must be a power of two <= 512");
};

struct CgParams {
  int mode, taps, kblocks;
  int B, Hin, Win, Cin, Cout;
  int Hg, Wg;      // pixel grid the M tiles cover: the output grid (CONV3, DOWN2) or the input grid (UP2)
  int Hout, Wout;  // output tensor extent
  int PX, ROWS;    // tile = PX pixels x ROWS rows (PX * ROWS <= 128)
  int tiles_x, tiles_y, n_tiles_n, n_items;
  int reverse;  // pair kernels: walk the items back to front (alternates per layer, see conv_api.cuh)
  int relu;
  const __nv_bfloat16* res1;
  const __nv_bfloat16* res2;
  __nv_bfloat16* out;
};

struct CgItem {
  int b, y0, x0, n0;
};
__device__ __forceinline__ CgItem cg_decode(const CgParams& p, int item) {
  CgItem c;
  c.n0 = item % p.n_tiles_n;
  int t = item / p.n_tiles_n;
  const int tx = t % p.tiles_x;
  t /= p.tiles_x;
  const int ty = t % p.tiles_y;
  c.b = t / p.tiles_y;
  c.x0 = tx * p.PX;
  c.y0 = ty * p.ROWS;
  return c;
}

__device__ __forceinline__ uint32_t cg_pack(float a, float b, bool relu) {
  uint32_t d;
  if (relu)
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  else
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  return d;
}
__device__ __forceinline__ void cg_add_bf16x8(float (&f)[8], const uint4 r) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] += __uint_as_float(w[i] << 16);
    f[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
  }
}
// The gradient-step DRUNet's epilogues (conv_tc.cuh has the same two for the 64-channel kernel): ELU after the sum, and the
// backward's gate f *= elu'(z), with t = the bf16 ELU output the forward stored: 1 for t > 0, else t + 1 = exp(z).
__device__ __forceinline__ void cg_elu8(float (&f)[8]) {  // exp by MUFU, as elu8 in conv_tc.cuh explains
#pragma unroll
  for (int i = 0; i < 8; ++i) f[i] = f[i] > 0.f ? f[i] : __expf(f[i]) - 1.f;
}
__device__ __forceinline__ void cg_gate_bf16x8(float (&f)[8], const uint4 r) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float t0 = __uint_as_float(w[i] << 16), t1 = __uint_as_float(w[i] & 0xffff0000u);
    f[2 * i] *= t0 > 0.f ? 1.f : t0 + 1.f;
    f[2 * i + 1] *= t1 > 0.f ? 1.f : t1 + 1.f;
  }
}
enum { CG_EPI_SUM = 0, CG_EPI_ELU = 1, CG_EPI_GATE = 2 };

template <int N_TILE>
__global__ void __launch_bounds__((CgCfg<N_TILE>::THREADS), 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, const CgParams p) {
  using Cfg = CgCfg<N_TILE>;
  constexpr int NSTAGE = Cfg::NSTAGE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* empty = full + NSTAGE;
  uint64_t* tfull = empty + NSTAGE;
  uint64_t* tempty = tfull + CG_NACC;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(tempty + CG_NACC);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  griddep_launch_dependents();

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < CG_NACC; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 4);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_s, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  const int kiters = p.taps * p.kblocks;

  if (warp == 0) {
    if (lane == 0) {
      // ---------------------------------------------------------------- TMA producer
      tma_prefetch_desc(&map_a);
      tma_prefetch_desc(&map_w);
      griddep_wait();
      uint32_t L = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const CgItem c = cg_decode(p, item);
        for (int t = 0; t < p.taps; ++t) {
          for (int kb = 0; kb < p.kblocks; ++kb, ++L) {
            const uint32_t slot = L % NSTAGE;
            mbar_wait(&empty[slot], ((L / NSTAGE) & 1) ^ 1);
            uint8_t* sa = smem + slot * Cfg::STAGE_BYTES;
            uint8_t* sb = sa + Cfg::A_BYTES;
            mbar_expect_tx(&full[slot], (uint32_t)(p.PX * p.ROWS * 128 + Cfg::B_BYTES));
            if (p.mode == CG_CONV3) {
              tma_load_4d(sa, &map_a, &full[slot], kb * 64, c.x0 + (t % 3) - 1, c.y0 + (t / 3) - 1, c.b);
              tma_load_3d(sb, &map_w, &full[slot], kb * 64, c.n0 * N_TILE, t);
            } else {  // CG_DOWN2: input viewed as {C, 2 (dx), Win/2, 2 (dy), B * Hin/2}
              tma_load_5d(sa, &map_a, &full[slot], kb * 64, t & 1, c.x0, t >> 1, c.b * (p.Hin / 2) + c.y0);
              tma_load_3d(sb, &map_w, &full[slot], kb * 64, c.n0 * N_TILE, t);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer (warp-uniform, one elected lane)
    constexpr uint32_t idesc = make_idesc_bf16(128, N_TILE);
    constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (LAYOUT_SW128 << 29);
    const uint32_t smem_lo = (smem_u32(smem) >> 4) | 0x10000u;
    uint32_t L = 0, T = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++T) {
      const uint32_t acc = T % CG_NACC;
      mbar_wait(&tempty[acc], ((T / CG_NACC) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * N_TILE;
      for (int it = 0; it < kiters; ++it, ++L) {
        const uint32_t slot = L % NSTAGE;
        mbar_wait(&full[slot], (L / NSTAGE) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_lo = smem_lo + slot * (uint32_t)(Cfg::STAGE_BYTES >> 4);
          const uint32_t b_lo = a_lo + (uint32_t)(Cfg::A_BYTES >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(d_tmem, ((uint64_t)DESC_HI << 32) | (a_lo + k * 2), ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc,
                      (it | k) != 0);
          umma_commit(&empty[slot]);
          if (it == kiters - 1) umma_commit(&tfull[acc]);
        }
        __syncwarp();
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue: 2 groups x 4 warps
    const int ew = warp - 2;
    const int grp = ew >> 2;
    const int q4 = warp & 3;
    const int m = q4 * 32 + lane;  // tile pixel
    const int r = m / p.PX, px = m % p.PX;
    const bool relu = p.relu != 0;
    griddep_wait();
    uint32_t T = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++T) {
      if ((int)(T & 1) != grp) continue;
      const CgItem c = cg_decode(p, item);
      const uint32_t acc = T % CG_NACC;
      const int yg = c.y0 + r, xg = c.x0 + px;
      const bool valid = (m < p.PX * p.ROWS) && yg < p.Hg && xg < p.Wg;
      const size_t off = (((size_t)c.b * p.Hout + yg) * p.Wout + xg) * p.Cout + (size_t)c.n0 * N_TILE;
      mbar_wait(&tfull[acc], (T / CG_NACC) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * N_TILE;
#pragma unroll 1
      for (int ch = 0; ch < N_TILE / 32; ++ch) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + ch * 32, v);
        tmem_ld_wait();
        if (ch == N_TILE / 32 - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[acc]);
        }
        if (valid) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {  // 16-byte chunk = 8 channels
            float f[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[8 * j + i]);
            const size_t o = off + ch * 32 + j * 8;
            if (p.res1) cg_add_bf16x8(f, *reinterpret_cast<const uint4*>(p.res1 + o));
            if (p.res2) cg_add_bf16x8(f, *reinterpret_cast<const uint4*>(p.res2 + o));
            uint4 w;
            w.x = cg_pack(f[0], f[1], relu);
            w.y = cg_pack(f[2], f[3], relu);
            w.z = cg_pack(f[4], f[5], relu);
            w.w = cg_pack(f[6], f[7], relu);
            *reinterpret_cast<uint4*>(p.out + o) = w;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------ CTA-pair form
// With both operands streaming, a single CTA moves (A + B) bytes into shared memory and (A + B) bytes out of it per
// k-iteration: 64 KB per 256 MMA cycles at N = 128, 96 KB per 512 at N = 256 -- 250 / 187 B per clock against a 128 B/clk
// port, which is where the measured 0.51 / 0.68 of the tensor peak come from.  cta_group::2 halves the B half of that: two
// CTAs (one TPC) run one M = 256 MMA per K-step on two different pixel tiles, each streaming only N_TILE / 2 rows of
// the weights.  Both producers signal the LEADER's "stage full" barrier (cp.async.bulk.tensor.cta_group::2), the leader
// issues, and one multicast tcgen05.commit frees the stage in both CTAs.
// Items: item = ((m_tile_pair * n_tiles_n + n_tile) * 2 + rank), so the two CTAs of a cluster share the n tile and walk
// the same (tap, k-block) sequence on M tiles 2 i and 2 i + 1; an odd M-tile count is padded with a tile at b = B, whose
// loads are out of bounds (zero fill) and whose stores are masked.
//
// REUSE (3x3 layers whose rows are at least 128 pixels wide, tile = 128 pixels of one row): a stage holds ONE input-row box
// of 130 pixels (halo left and right) and the weights of the three taps of that row (dx = 0, 1, 2, one 3-D box), and serves
// 12 MMAs whose A descriptors start dx rows into the box -- a third of the activation traffic from L2 per MMA.  Without it
// the 128-channel layers (4 MMAs of 64 cycles per 16 KB A box) sit at 0.65 of the tensor peak on L2 -> SM bandwidth.
//
// WRES (128 -> 128 channels, REUSE geometry): the layer's weights stay RESIDENT in shared memory -- this CTA's 64 output
// channels x 128 input channels x 9 taps = 144 KB, loaded once per launch before the wait on the previous layer -- and the
// ring carries activations only.  With streamed weights an item pulls 147 KB of weights and 100 KB of activations per CTA
// through L2 -> SM (5 GB per layer at 64 chains of 160 x 240: the layer ran at 1 410 TFLOP/s where the 256-channel layers,
// twice the MMA work per byte, reach 1 530, and a residual input cost its full read time on top, 514 -> 637 us).
template <int N_TILE, bool REUSE, bool WRES = false>
struct CgCfg2 {
  static_assert(!WRES || (REUSE && N_TILE == 128), "resident weights: the 128-channel 3x3 layers only");
  static constexpr int THREADS = 64 + 32 * CG_EPI_WARPS;
  static constexpr int A_BOX_BYTES = REUSE ? 130 * 128 : 128 * 128;
  static constexpr int A_BYTES = REUSE ? 17 * 1024 : 128 * 128;
  static constexpr int TAP_BYTES = (N_TILE / 2) * 128;          // this CTA's half of the N tile, one tap
  static constexpr int B_BYTES = WRES ? 0 : (REUSE ? 3 : 1) * TAP_BYTES;
  static constexpr int W_KBLOCKS = 2;                            // WRES: Cin = 128
  static constexpr int W_BYTES = WRES ? 9 * W_KBLOCKS * TAP_BYTES : 0;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int NSTAGE = ((225280 - W_BYTES) / STAGE_BYTES) > 8 ? 8 : ((225280 - W_BYTES) / STAGE_BYTES);
  static constexpr int OFF_W = NSTAGE * STAGE_BYTES;
  static constexpr int OFF_BAR = OFF_W + W_BYTES;
  static constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
  static constexpr int TMEM_COLS = CG_NACC * N_TILE;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of one CTA");
  static_assert((TMEM_COLS & (TMEM_COLS - 1)) == 0 && TMEM_COLS <= 512 && TMEM_COLS >= 32, "TMEM columns");
};

__device__ __forceinline__ CgItem cg_decode2(const CgParams& p, int item) {
  if (p.reverse) item = p.n_items - 1 - item;  // items 2i, 2i+1 swap ranks and stay one pair
  CgItem c;
  const int rank = item & 1;
  const int t = item >> 1;
  int mt = 2 * (t / p.n_tiles_n) + rank;
  c.n0 = t % p.n_tiles_n;
  const int tx = mt % p.tiles_x;
  mt /= p.tiles_x;
  const int ty = mt % p.tiles_y;
  c.b = mt / p.tiles_y;  // == p.B for the padding tile
  c.x0 = tx * p.PX;
  c.y0 = ty * p.ROWS;
  return c;
}

// RES2: a second residual tensor (U-Net skip, one layer per scale) is prefetched like the first; its own instantiation,
// so that its 64 extra registers do not weigh on the other layers.  EPI: CG_EPI_SUM (residual adds, optional ReLU),
// CG_EPI_ELU (ELU instead of ReLU) or CG_EPI_GATE (res1 is a stored ELU output t; multiply by elu'(t) instead of adding it),
// the last two for the gradient-step DRUNet in instantiations of their own.
template <int N_TILE, bool REUSE, bool RES2, bool WRES = false, int EPI = CG_EPI_SUM>
__global__ void __launch_bounds__((CgCfg2<N_TILE, REUSE, WRES>::THREADS), 1)
conv_gemm2_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, const CgParams p) {
  using Cfg = CgCfg2<N_TILE, REUSE, WRES>;
  constexpr int NSTAGE = Cfg::NSTAGE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);  // leader: both CTAs' boxes of the stage landed
  uint64_t* empty = full + NSTAGE;                                    // both (multicast): the stage's MMAs completed
  uint64_t* tfull = empty + NSTAGE;                                   // both (multicast): accumulator complete
  uint64_t* tempty = tfull + CG_NACC;                                 // leader: both epilogues drained the stage
  uint64_t* done = tempty + CG_NACC;                                  // both (multicast): all MMAs of the launch completed
  uint64_t* wbar = done + 1;                                          // WRES, local: this CTA's half of the weights landed
  uint64_t* wready = wbar + 1;                                        // WRES, leader: the peer's half landed
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(wready + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  griddep_launch_dependents();

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < CG_NACC; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 8);
    }
    mbar_init(done, 1);
    mbar_init(wbar, 1);
    mbar_init(wready, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc2(tmem_ptr_s, Cfg::TMEM_COLS);
    tmem_relinquish2();
  }
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  const int kiters = (REUSE ? 3 : p.taps) * p.kblocks;

  if (warp == 0) {
    if (lane == 0) {
      // ---------------------------------------------------------------- TMA producer (both CTAs)
      tma_prefetch_desc(&map_a);
      tma_prefetch_desc(&map_w);
      const uint32_t full_c = mapa_shared(smem_u32(full), 0);
      const uint32_t stage_tx = 2u * (uint32_t)((REUSE ? Cfg::A_BOX_BYTES : p.PX * p.ROWS * 128) + Cfg::B_BYTES);
      const int nrow0 = (int)rank * (N_TILE / 2);
      if (WRES) {  // the whole layer's weights for this CTA's output channels: box (dy, kb) = taps 3 dy .. 3 dy + 2, 64 input channels
        mbar_expect_tx(wbar, (uint32_t)Cfg::W_BYTES);
        for (int dy = 0; dy < 3; ++dy)
          for (int kb = 0; kb < Cfg::W_KBLOCKS; ++kb)
            tma_load_3d(smem + Cfg::OFF_W + (dy * Cfg::W_KBLOCKS + kb) * 3 * Cfg::TAP_BYTES, &map_w, wbar, kb * 64, nrow0, dy * 3);
        if (rank != 0) {
          mbar_wait(wbar, 0);
          mbar_arrive_cluster(mapa_shared(smem_u32(wready), 0));
        }
      }
      griddep_wait();
      uint32_t L = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const CgItem c = cg_decode2(p, item);
        if (WRES) {
          for (int dy = 0; dy < 3; ++dy) {
            for (int kb = 0; kb < Cfg::W_KBLOCKS; ++kb, ++L) {
              const uint32_t slot = L % NSTAGE;
              mbar_wait(&empty[slot], ((L / NSTAGE) & 1) ^ 1);
              if (rank == 0) mbar_expect_tx(&full[slot], 2u * (uint32_t)Cfg::A_BOX_BYTES);
              tma_load_4d_2sm(smem + slot * Cfg::STAGE_BYTES, &map_a, full_c + slot * 8u, kb * 64, c.x0 - 1, c.y0 + dy - 1, c.b);
            }
          }
          continue;
        }
        if (REUSE) {
          for (int dy = 0; dy < 3; ++dy) {
            for (int kb = 0; kb < p.kblocks; ++kb, ++L) {
              const uint32_t slot = L % NSTAGE;
              mbar_wait(&empty[slot], ((L / NSTAGE) & 1) ^ 1);
              uint8_t* sa = smem + slot * Cfg::STAGE_BYTES;
              const uint32_t bar = full_c + slot * 8u;
              if (rank == 0) mbar_expect_tx(&full[slot], stage_tx);
              tma_load_4d_2sm(sa, &map_a, bar, kb * 64, c.x0 - 1, c.y0 + dy - 1, c.b);                 // 130 pixels of one row
              tma_load_3d_2sm(sa + Cfg::A_BYTES, &map_w, bar, kb * 64, c.n0 * N_TILE + nrow0, dy * 3);  // taps 3 dy .. 3 dy + 2
            }
          }
          continue;
        }
        for (int t = 0; t < p.taps; ++t) {
          for (int kb = 0; kb < p.kblocks; ++kb, ++L) {
            const uint32_t slot = L % NSTAGE;
            mbar_wait(&empty[slot], ((L / NSTAGE) & 1) ^ 1);
            uint8_t* sa = smem + slot * Cfg::STAGE_BYTES;
            uint8_t* sb = sa + Cfg::A_BYTES;
            const uint32_t bar = full_c + slot * 8u;
            if (rank == 0) mbar_expect_tx(&full[slot], stage_tx);
            if (p.mode == CG_CONV3) {
              tma_load_4d_2sm(sa, &map_a, bar, kb * 64, c.x0 + (t % 3) - 1, c.y0 + (t / 3) - 1, c.b);
              tma_load_3d_2sm(sb, &map_w, bar, kb * 64, c.n0 * N_TILE + nrow0, t);
            } else if (p.mode == CG_DOWN2) {
              tma_load_5d_2sm(sa, &map_a, bar, kb * 64, t & 1, c.x0, t >> 1, c.b * (p.Hin / 2) + c.y0);
              tma_load_3d_2sm(sb, &map_w, bar, kb * 64, c.n0 * N_TILE + nrow0, t);
            } else {  // CG_UP2: the weights are one [4 Cout][Cin] tap
              tma_load_4d_2sm(sa, &map_a, bar, kb * 64, c.x0, c.y0, c.b);
              tma_load_3d_2sm(sb, &map_w, bar, kb * 64, c.n0 * N_TILE + nrow0, 0);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ---------------------------------------------------------------- MMA issuer of the pair
      constexpr uint32_t idesc = make_idesc_bf16(256, N_TILE);
      constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (LAYOUT_SW128 << 29);
      const uint32_t smem_lo = (smem_u32(smem) >> 4) | 0x10000u;
      if (WRES) {
        mbar_wait(wbar, 0);
        mbar_wait_cluster(wready, 0);
        tc_fence_after();
      }
      uint32_t L = 0, T = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++T) {
        const uint32_t acc = T % CG_NACC;
        mbar_wait(&tempty[acc], ((T / CG_NACC) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * N_TILE;
        for (int it = 0; it < kiters; ++it, ++L) {
          const uint32_t slot = L % NSTAGE;
          mbar_wait(&full[slot], (L / NSTAGE) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t a_lo = smem_lo + slot * (uint32_t)(Cfg::STAGE_BYTES >> 4);
            const uint32_t b_lo = WRES ? smem_lo + (uint32_t)((Cfg::OFF_W + it * 3 * Cfg::TAP_BYTES) >> 4)  // it = dy * 2 + kb
                                       : a_lo + (uint32_t)(Cfg::A_BYTES >> 4);
            if (REUSE) {
#pragma unroll
              for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                for (int k = 0; k < 4; ++k)  // A: the row box read from pixel dx on (whole 128-byte rows keep the swizzle phase)
                  umma_bf16_ss2(d_tmem, ((uint64_t)DESC_HI << 32) | (a_lo + (uint32_t)(dx * 8 + k * 2)),
                                ((uint64_t)DESC_HI << 32) | (b_lo + (uint32_t)(dx * (Cfg::TAP_BYTES >> 4) + k * 2)), idesc,
                                (it | dx | k) != 0);
            } else {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_bf16_ss2(d_tmem, ((uint64_t)DESC_HI << 32) | (a_lo + k * 2), ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc,
                              (it | k) != 0);
            }
            umma_commit2(&empty[slot], 3);
            if (it == kiters - 1) umma_commit2(&tfull[acc], 3);
          }
          __syncwarp();
        }
      }
      if (elect_one()) umma_commit2(done, 3);
      __syncwarp();
    }
    mbar_wait(done, 0);
  } else {
    // ---------------------------------------------------------------- epilogue: 2 groups x 4 warps (each CTA its own M tile)
    // A thread owns one pixel: N_TILE consecutive channels of the output (and of the residual inputs).  The first residual
    // tensor is fetched into registers BEFORE the accumulator is awaited (the item's MMAs take thousands of cycles, the
    // loads a few hundred), 128 channels at a time; for N_TILE = 256 the registers of a finished 32-channel chunk are
    // refilled with the chunk 128 channels further on while the remaining chunks are processed.
    const int ew = warp - 2;
    const int grp = ew >> 2;
    const int q4 = warp & 3;
    const int m = q4 * 32 + lane;
    const int r = m / p.PX, px = m % p.PX;
    const bool relu = p.relu != 0;
    const uint32_t tempty_c = mapa_shared(smem_u32(tempty), 0);
    constexpr int NB = N_TILE / 128;  // batches of 128 channels
    griddep_wait();
    uint32_t T = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++T) {
      if ((int)(T & 1) != grp) continue;
      const CgItem c = cg_decode2(p, item);
      const uint32_t acc = T % CG_NACC;
      const int yg = c.y0 + r, xg = c.x0 + px;
      const bool valid = (m < p.PX * p.ROWS) && yg < p.Hg && xg < p.Wg && c.b < p.B;
      int yo = yg, xo = xg;
      if (p.mode == CG_UP2) {
        yo = 2 * yg;
        xo = 2 * xg;
      }
      const size_t off = (((size_t)c.b * p.Hout + yo) * p.Wout + xo) * p.Cout + (size_t)c.n0 * N_TILE;
      // transposed conv: the N axis is (quadrant, channel), a 32-column chunk lies in one quadrant
      const bool upm = p.mode == CG_UP2;
      auto chunk_off = [&](int ch) -> size_t {
        if (!upm) return off + (size_t)(ch * 32);
        const int n = c.n0 * N_TILE + ch * 32;
        const int q = n / p.Cout, cc = n - q * p.Cout;
        return (((size_t)c.b * p.Hout + 2 * yg + (q >> 1)) * p.Wout + 2 * xg + (q & 1)) * p.Cout + cc;
      };
      const bool has_res = valid && p.res1 != nullptr;
      const bool has_res2 = RES2 && valid && p.res2 != nullptr;
      uint4 rr[16], rr2[RES2 ? 16 : 1];
      if (has_res) {
#pragma unroll
        for (int j = 0; j < 16; j += 2) ldg256(p.res1 + off + j * 8, rr[j], rr[j + 1]);
      }
      if (RES2 && has_res2) {
#pragma unroll
        for (int j = 0; j < 16; j += 2) ldg256(p.res2 + off + j * 8, rr2[RES2 ? j : 0], rr2[RES2 ? j + 1 : 0]);
      }
      mbar_wait(&tfull[acc], (T / CG_NACC) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * N_TILE;
#pragma unroll
      for (int hb = 0; hb < NB; ++hb) {
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          const int ch = hb * 4 + c4;  // 32-channel chunk
          uint32_t v[32];
          tmem_ld_32x32b_x32(taddr + ch * 32, v);
          tmem_ld_wait();
          if (ch == N_TILE / 32 - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(tempty_c + acc * 8u);
          }
          const size_t choff = chunk_off(ch);
          if (valid) {
#pragma unroll
            for (int j2 = 0; j2 < 2; ++j2) {  // 32 bytes = 16 channels per access
              uint4 w[2];
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const int j = 2 * j2 + h;
                float f[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[8 * j + i]);
                if (EPI == CG_EPI_GATE) {
                  if (has_res) cg_gate_bf16x8(f, rr[c4 * 4 + j]);
                } else if (has_res) {
                  cg_add_bf16x8(f, rr[c4 * 4 + j]);
                }
                if (RES2 && has_res2) cg_add_bf16x8(f, rr2[RES2 ? c4 * 4 + j : 0]);
                if (EPI == CG_EPI_ELU) cg_elu8(f);
                w[h].x = cg_pack(f[0], f[1], relu);
                w[h].y = cg_pack(f[2], f[3], relu);
                w[h].z = cg_pack(f[4], f[5], relu);
                w[h].w = cg_pack(f[6], f[7], relu);
              }
              const size_t o = choff + j2 * 16;
              if (hb + 1 < NB) {
                if (has_res) ldg256(p.res1 + o + 128, rr[c4 * 4 + 2 * j2], rr[c4 * 4 + 2 * j2 + 1]);
                if (RES2 && has_res2) ldg256(p.res2 + o + 128, rr2[RES2 ? c4 * 4 + 2 * j2 : 0], rr2[RES2 ? c4 * 4 + 2 * j2 + 1 : 0]);
              }
              stg256(p.out + o, w[0], w[1]);
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  cluster_sync();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------ host side
static int cg_encode(CUtensorMap* map, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                     const cuuint32_t* box) {
  PFN_tensorMapEncodeTiled enc = get_tensor_map_encoder();
  if (!enc) return set_error(PSGLA_E_NODEVICE, "cuTensorMapEncodeTiled driver entry point not available");
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(PSGLA_E_BADARG, "cuTensorMapEncodeTiled (rank %d) failed with CUresult %d", rank, (int)r);
  return PSGLA_OK;
}

struct CgMapKey {
  const void* ptr;
  int a, b, c, d, e, f;
  bool operator==(const CgMapKey& o) const {
    return ptr == o.ptr && a == o.a && b == o.b && c == o.c && d == o.d && e == o.e && f == o.f;
  }
};
static int cg_cached_map(CUtensorMap* map, const CgMapKey& key, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                         const cuuint32_t* box) {
  static thread_local std::vector<std::pair<CgMapKey, CUtensorMap>> cache;
  for (const auto& e : cache)
    if (e.first == key) {
      *map = e.second;
      return PSGLA_OK;
    }
  int rc = cg_encode(map, key.ptr, rank, dims, strides, box);
  if (rc) return rc;
  if (cache.size() >= 256) cache.erase(cache.begin());
  cache.emplace_back(key, *map);
  return PSGLA_OK;
}

template <int N_TILE>
static int cg_launch(const CUtensorMap& ma, const CUtensorMap& mw, const CgParams& p, cudaStream_t st) {
  using Cfg = CgCfg<N_TILE>;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (!(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(conv_gemm_kernel<N_TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  const int grid = p.n_items < num_sms() ? p.n_items : num_sms();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(Cfg::THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv_gemm_kernel<N_TILE>, ma, mw, p));
  return PSGLA_OK;
}

template <int N_TILE, bool REUSE, bool RES2, bool WRES = false, int EPI = CG_EPI_SUM>
static int cg_launch2_t(const CUtensorMap& ma, const CUtensorMap& mw, CgParams p, cudaStream_t st) {
  using Cfg = CgCfg2<N_TILE, REUSE, WRES>;
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3(Cfg::THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  static std::atomic<int> max_clusters_dev[kMaxDevices];  // per device: co-resident CTA pairs; 0 = not asked yet (also: the function attribute is unset)
  std::atomic<int>& mc_slot = max_clusters_dev[current_device() % kMaxDevices];
  int max_clusters = mc_slot.load(std::memory_order_acquire);
  if (!max_clusters) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(conv_gemm2_kernel<N_TILE, REUSE, RES2, WRES, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    cfg.gridDim = dim3((unsigned)(num_sms() & ~1));
    int n = 0;
    PSGLA_CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, conv_gemm2_kernel<N_TILE, REUSE, RES2, WRES, EPI>, &cfg));
    max_clusters = n > 0 ? std::min(n, num_sms() / 2) : num_sms() / 2;
    mc_slot.store(max_clusters, std::memory_order_release);
  }
  const int m_tiles = p.B * p.tiles_y * p.tiles_x;
  const int pairs = ((m_tiles + 1) / 2) * p.n_tiles_n;
  p.n_items = 2 * pairs;
  cfg.gridDim = dim3((unsigned)(2 * std::min(pairs, max_clusters)));
  PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv_gemm2_kernel<N_TILE, REUSE, RES2, WRES, EPI>, ma, mw, p));
  return PSGLA_OK;
}

template <int N_TILE, bool REUSE, bool WRES = false>
static int cg_launch2(const CUtensorMap& ma, const CUtensorMap& mw, const CgParams& p, cudaStream_t st, int act) {
  if (act == ACT_ELU) return cg_launch2_t<N_TILE, REUSE, false, WRES, CG_EPI_ELU>(ma, mw, p, st);
  if (act == ACT_GATE) return cg_launch2_t<N_TILE, REUSE, false, WRES, CG_EPI_GATE>(ma, mw, p, st);
  return p.res2 ? cg_launch2_t<N_TILE, REUSE, true, WRES>(ma, mw, p, st) : cg_launch2_t<N_TILE, REUSE, false, WRES>(ma, mw, p, st);
}

// One layer.  in: bf16 NHWC [B][Hin][Win][Cin]; w: bf16 [taps][Cout][Cin]; out: bf16 NHWC (CONV3: same extent, DOWN2:
// half, UP2: double); res1 / res2: optional tensors of the output's shape added before the optional ReLU.  act: ConvAct;
// ACT_ELU and ACT_GATE (res1 = the gate's ELU output, no res2) run on the 3x3 CTA-pair kernels only.
int conv_gemm_layer(int mode, int B, int Hin, int Win, int Cin, int Cout, const void* w, const void* in, const void* res1,
                    const void* res2, void* out, int act, cudaStream_t st) {
  PSGLA_REQUIRE(mode >= CG_CONV3 && mode <= CG_UP2, "conv_gemm_layer: unknown mode %d", mode);
  PSGLA_REQUIRE(B > 0 && Hin > 0 && Win > 0 && Cin >= 64 && Cin % 64 == 0 && Cout >= 64 && Cout % 64 == 0,
                "conv_gemm_layer: channels must be multiples of 64 (got %d -> %d), extents positive", Cin, Cout);
  PSGLA_REQUIRE(w && in && out, "conv_gemm_layer: null pointer");
  PSGLA_REQUIRE(((uintptr_t)out | (uintptr_t)res1 | (uintptr_t)res2) % 32 == 0 && (uintptr_t)in % 16 == 0 && (uintptr_t)w % 16 == 0,
                "conv_gemm_layer: out / residual tensors must be 32-byte aligned, in / weights 16-byte aligned");
  PSGLA_REQUIRE(mode != CG_DOWN2 || (Hin % 2 == 0 && Win % 2 == 0), "stride-2 conv needs even extents (got %d x %d)", Hin, Win);
  PSGLA_REQUIRE(act == ACT_NONE || act == ACT_RELU || (mode == CG_CONV3 && Cout % 128 == 0 && !res2 && (act == ACT_ELU ? !res1 : act == ACT_GATE && res1)),
                "conv_gemm_layer: the ELU / gate epilogues are for 3x3 layers of 128k channels (ELU: no residual; gate: res1 only)");
  CgParams p{};
  p.mode = mode;
  p.taps = mode == CG_CONV3 ? 9 : (mode == CG_DOWN2 ? 4 : 1);
  p.kblocks = Cin / 64;
  p.B = B, p.Hin = Hin, p.Win = Win, p.Cin = Cin, p.Cout = Cout;
  p.Hg = mode == CG_DOWN2 ? Hin / 2 : Hin;
  p.Wg = mode == CG_DOWN2 ? Win / 2 : Win;
  p.Hout = mode == CG_UP2 ? 2 * Hin : p.Hg;
  p.Wout = mode == CG_UP2 ? 2 * Win : p.Wg;
  p.PX = std::min(p.Wg, 128);
  p.ROWS = std::max(1, std::min(128 / p.PX, p.Hg));
  p.tiles_x = (p.Wg + p.PX - 1) / p.PX;
  p.tiles_y = (p.Hg + p.ROWS - 1) / p.ROWS;
  // The transposed conv is ONE GEMM with N = 4 Cout -- the weights [quadrant][Cout][Cin] are a [4 Cout][Cin] matrix as they
  // lie, the epilogue scatters column n to quadrant n / Cout -- so an A tile is loaded once instead of once per quadrant, and
  // the 128 -> 64 layer gets 256-column tiles on the CTA pair.
  const int n_cols = mode == CG_UP2 ? 4 * Cout : Cout;
  // The widest N tile that divides the output columns.  Tiles of 128 and 256 columns run on the CTA-pair kernel (a single
  // CTA reaches only 0.51 / 0.68 of the tensor peak, see above); 64-column tiles, i.e. Cout an odd multiple of 64 in a 3x3 or
  // stride-2 conv (4 Cout is always a multiple of 256), on the single-CTA kernel.
  const int n_tile = n_cols % 256 == 0 ? 256 : (n_cols % 128 == 0 ? 128 : 64);
  const bool pair = n_tile >= 128;
  // one 130-pixel row box for the three horizontal taps (CgCfg2<., true>): 3x3 layers with rows of >= 128 pixels
  const bool reuse = pair && mode == CG_CONV3 && p.PX == 128 && p.ROWS == 1;
  p.reverse = pair ? next_layer_direction() : 0;
  p.n_tiles_n = n_cols / n_tile;
  p.n_items = B * p.tiles_y * p.tiles_x * p.n_tiles_n;
  p.relu = act == ACT_RELU;
  p.res1 = (const __nv_bfloat16*)res1;
  p.res2 = (const __nv_bfloat16*)res2;
  p.out = (__nv_bfloat16*)out;

  CUtensorMap ma, mw;
  int rc;
  if (mode == CG_DOWN2) {
    const cuuint64_t dims[5] = {(cuuint64_t)Cin, 2, (cuuint64_t)(Win / 2), 2, (cuuint64_t)B * (Hin / 2)};
    const cuuint64_t strides[4] = {(cuuint64_t)Cin * 2, (cuuint64_t)Cin * 4, (cuuint64_t)Win * Cin * 2, (cuuint64_t)Win * Cin * 4};
    const cuuint32_t box[5] = {64, 1, (cuuint32_t)p.PX, 1, (cuuint32_t)p.ROWS};
    rc = cg_cached_map(&ma, CgMapKey{in, 5, B, Hin, Win, Cin, p.PX * 1000 + p.ROWS}, 5, dims, strides, box);
  } else {
    const cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)Win, (cuuint64_t)Hin, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Win * Cin * 2, (cuuint64_t)Hin * Win * Cin * 2};
    const int box_px = reuse ? 130 : p.PX;
    const cuuint32_t box[4] = {64, (cuuint32_t)box_px, (cuuint32_t)p.ROWS, 1};
    rc = cg_cached_map(&ma, CgMapKey{in, 4, B, Hin, Win, Cin, box_px * 1000 + p.ROWS}, 4, dims, strides, box);
  }
  if (rc) return rc;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)Cin, (cuuint64_t)n_cols, (cuuint64_t)p.taps};
    const cuuint64_t strides[2] = {(cuuint64_t)Cin * 2, (cuuint64_t)n_cols * Cin * 2};
    const int box_n = pair ? n_tile / 2 : n_tile;  // a CTA of a pair streams half of the N tile
    const cuuint32_t box[3] = {64, (cuuint32_t)box_n, reuse ? 3u : 1u};
    rc = cg_cached_map(&mw, CgMapKey{w, 3, Cin, n_cols, p.taps, box_n, reuse ? 3 : 1}, 3, dims, strides, box);
  }
  if (rc) return rc;
  // resident weights for the 128 -> 128 channel layers (CgCfg2<128, true, true>)
  if (reuse && Cin == 128 && Cout == 128) return cg_launch2<128, true, true>(ma, mw, p, st, act);
  if (reuse) return n_tile == 256 ? cg_launch2<256, true>(ma, mw, p, st, act) : cg_launch2<128, true>(ma, mw, p, st, act);
  if (pair) return n_tile == 256 ? cg_launch2<256, false>(ma, mw, p, st, act) : cg_launch2<128, false>(ma, mw, p, st, act);
  return cg_launch<64>(ma, mw, p, st);
}

}  // namespace psgla

using namespace psgla;

extern "C" int psgla_convg_layer(int mode, int B, int Hin, int Win, int Cin, int Cout, const void* w_dev, const void* in_dev,
                                 const void* res1_dev, const void* res2_dev, void* out_dev, int relu, void* stream) {
  return conv_gemm_layer(mode, B, Hin, Win, Cin, Cout, w_dev, in_dev, res1_dev, res2_dev, out_dev, relu ? ACT_RELU : ACT_NONE,
                         (cudaStream_t)stream);
}
