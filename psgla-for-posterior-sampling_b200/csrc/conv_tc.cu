// 3x3 convolution layers with shared-memory-resident weights as implicit GEMM on tcgen05 tensor cores (sm_100a),
// activations bf16 NHWC, fp32 accumulate: all of DnCNN and the 64-channel full-resolution layers of DRUNet.
//
// Replaces the cuDNN fp32 convolutions behind `denoiser.forward` (restoration_algorithms.py:238,
// sampling_images.py:156; architecture: deepinv.models.DnCNN / DRUNet, see oracle/image_oracle.py).
//
// GEMM view per 128-pixel output row segment:  D[128 x NOUT] = sum over 9 taps  A_tap[128 x CIN] * W_tap[NOUT x CIN]^T.
// A work item is a (chain, 128-pixel strip, block of R rows); every input row (130 pixels = 128 + halo, TMA out-of-bounds
// zero fill = the convolution's padding) is loaded ONCE and serves the three output rows around it.  One kernel per layer role:
//   conv3x3_kernel<16,64>          the first layer (3 or 1, padded to 16, -> 64 channels).  SS form: A_tap = window into the
//                                  shared-memory row ring (tap dx = descriptor start + dx rows, tap dy = ring slot).
//   conv3x3_ts_kernel<16,C>        the last layer (64 -> C = 3 or 1, padded to 16, fused Langevin post / next pre epilogue).  TS form:
//                                  four loader warps copy each row into TENSOR MEMORY three times (shifted by dx) and the MMAs
//                                  take A from there (N/2 instead of 32 + N/4 cycles per MMA at N = 64).
//   conv3x3_ts2_kernel<NOUT,RES>   the hidden layers: a CTA PAIR (cta_group::2, M = 256) on two adjacent strips, weights split
//                                  32 / 32 output channels between the two shared memories; RES = 0 plain (no residual code in
//                                  the epilogue at all), 1 = residual input by TMA, 2 = and a second one (U-Net skip tensor).
//   (conv_fused2.cu: two hidden layers per launch when the work is a single wave of pairs.)
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc), [warps 2..5 = loaders (TS forms)], 8 epilogue warps
// in two groups (TMEM -> bias / residual / ReLU -> bf16 -> swizzled staging box -> TMA store; or the fused Langevin step,
// restoration_algorithms.py:238-262, for the last layer).  Consecutive layers walk their items in opposite directions
// (ConvParams::reverse) so that each starts on what the previous one left in L2.  DESIGN.md section 4 has the measurements.
#include <cuda_bf16.h>

#include <algorithm>
#include <cstring>
#include <mutex>
#include <utility>
#include <vector>

#include "conv_tc.cuh"

namespace psgla {

using namespace sm100;

// ------------------------------------------------------------------------------------------------ SS kernel (A from smem)
template <int CIN, int NOUT>
__global__ void __launch_bounds__(CONV_THREADS, 1)
conv3x3_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_out, const ConvParams p) {
  using Cfg = ConvCfg<CIN, NOUT>;
  constexpr int NSTAGE = Cfg::NSTAGE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_w = smem;
  uint8_t* ring = smem + Cfg::OFF_RING;
  float* bias_s = reinterpret_cast<float*>(smem + Cfg::OFF_BIAS);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* empty = full + NSTAGE;
  uint64_t* tfull = empty + NSTAGE;
  uint64_t* tempty = tfull + NACC;
  uint64_t* wbar = tempty + NACC;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(wbar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // Programmatic dependent launch: let the next layer's CTAs start their prologue as ours retire; everything below that
  // touches memory written by an earlier kernel sits behind griddep_wait().
  griddep_launch_dependents();

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < NACC; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 4);  // one elected arrive per warp of the group that drains this stage
    }
    mbar_init(wbar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_s, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + NOUT) bias_s[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  if (warp == 0) {
    if (lane == 0) {
      // ---------------------------------------------------------------- TMA producer
      tma_prefetch_desc(&tmap);
      mbar_expect_tx(wbar, Cfg::W_BYTES);
      bulk_load(smem_w, p.weights, Cfg::W_BYTES, wbar);  // weights are constant across launches: no dependency wait
      griddep_wait();
      uint32_t L = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const ItemCoord c = decode_item(p, item);
        for (int y = c.ylo; y <= c.yhi; ++y, ++L) {
          const uint32_t slot = L % NSTAGE, use = L / NSTAGE;
          mbar_wait(&empty[slot], (use & 1) ^ 1);
          mbar_expect_tx(&full[slot], Cfg::BOX_BYTES);
          tma_load_4d(ring + slot * Cfg::SLOT_BYTES, &tmap, &full[slot], 0, c.x0 - 1, y, c.b);
        }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    // The whole warp walks the (warp-uniform) control flow so that barrier addresses and descriptors live in uniform
    // registers; one elected lane issues the tcgen05 instructions.  Descriptors differ only in their 14-bit start
    // address field, so each MMA costs two integer adds.
    constexpr uint32_t idesc = make_idesc_bf16(TILE_M, NOUT);
    constexpr uint32_t DESC_HI = (Cfg::SBO >> 4) | (1u << 14) | (Cfg::LAYOUT << 29);  // SBO | version 1 | swizzle mode
    const uint32_t ring_lo = (smem_u32(ring) >> 4) | 0x10000u;                         // start address >> 4 | LBO = 1
    const uint32_t w_lo = (smem_u32(smem_w) >> 4) | 0x10000u;
    mbar_wait(wbar, 0);
    tc_fence_after();
    uint32_t L0 = 0, T = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const ItemCoord c = decode_item(p, item);
      int waited = 0;
      const int ylast = c.y0 + c.rcur - 1;
      for (int y = c.y0; y <= ylast; ++y, ++T) {
        const int need = min(y + 1, c.yhi) - c.ylo + 1;
        while (waited < need) {
          const uint32_t q = L0 + waited;
          mbar_wait(&full[q % NSTAGE], (q / NSTAGE) & 1);
          ++waited;
        }
        const uint32_t acc = T % NACC;
        mbar_wait(&tempty[acc], ((T / NACC) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * NOUT;
        if (elect_one()) {
          uint32_t accumulate = 0;
#pragma unroll
          for (int dy = 0; dy < 3; ++dy) {
            const int yy = y + dy - 1;
            if (yy < 0 || yy >= p.H) continue;
            const uint32_t q = L0 + (uint32_t)(yy - c.ylo);
            const uint32_t a_lo = ring_lo + (q % NSTAGE) * (uint32_t)(Cfg::SLOT_BYTES >> 4);
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
              // tap (dy, dx): the A operand is the input row shifted by dx pixels.  The swizzle pattern is anchored at
              // absolute 1024-byte boundaries, so shifting the start address by whole 128-byte rows needs no
              // base-offset correction (verified by psgla_selftest_umma).
#pragma unroll
              for (int k = 0; k < Cfg::KSTEPS; ++k) {
                const uint32_t al = a_lo + (uint32_t)((dx * Cfg::ROW_BYTES + k * 32) >> 4);
                const uint32_t bl = w_lo + (uint32_t)(((dy * 3 + dx) * Cfg::TAP_BYTES + k * 32) >> 4);
                umma_bf16(d_tmem, ((uint64_t)DESC_HI << 32) | al, ((uint64_t)DESC_HI << 32) | bl, idesc, accumulate);
                accumulate = 1;
              }
            }
          }
          umma_commit(&tfull[acc]);
          if (y - 1 >= c.ylo) umma_commit(&empty[(L0 + (uint32_t)(y - 1 - c.ylo)) % NSTAGE]);
          if (y == ylast)
            for (int yy = y; yy <= c.yhi; ++yy) umma_commit(&empty[(L0 + (uint32_t)(yy - c.ylo)) % NSTAGE]);
        }
        __syncwarp();
      }
      L0 += (uint32_t)(c.yhi - c.ylo + 1);
    }
  } else {
    // ------------------------------------------------------------------ epilogue: 2 groups x 4 warps
    const int ew = warp - 2;
    epilogue_hidden<NOUT, NACC>(p, &tmap_out, smem + Cfg::OFF_STAGE + ew * Cfg::STAGE_BYTES, bias_s, tfull, tempty, tmem_base,
                                ew >> 2, warp & 3, lane);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int NOUT, int C>  // C: image channels of the fused post, 3 or 1
__global__ void __launch_bounds__(TS_THREADS, 1)
conv3x3_ts_kernel(const __grid_constant__ CUtensorMap tmap, const ConvParams p) {
  using Cfg = ConvTsCfg<NOUT>;
  constexpr int NST = Cfg::NSTAGE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_w = smem;
  uint8_t* ring = smem + Cfg::OFF_RING;
  float* bias_s = reinterpret_cast<float*>(smem + Cfg::OFF_BIAS);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);  // TMA landed a row in the staging ring
  uint64_t* empty = full + NST;                                 // loaders have copied it out
  uint64_t* afull = empty + NST;                                // the row's three shifted copies are in TMEM
  uint64_t* aempty = afull + TS_NA;                                   // every MMA reading them has completed
  uint64_t* tfull = aempty + TS_NA;
  uint64_t* tempty = tfull + TS_NACC;
  uint64_t* wbar = tempty + TS_NACC;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(wbar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  griddep_launch_dependents();

  if (threadIdx.x == 0) {
    for (int i = 0; i < NST; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 4);
    }
    for (int i = 0; i < TS_NA; ++i) {
      mbar_init(&afull[i], 4);
      mbar_init(&aempty[i], 1);
    }
    for (int i = 0; i < TS_NACC; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 4);
    }
    mbar_init(wbar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_s, 512);
    tmem_relinquish();
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + NOUT) bias_s[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  if (warp == 0) {
    if (lane == 0) {
      // ---------------------------------------------------------------- TMA producer
      tma_prefetch_desc(&tmap);
      mbar_expect_tx(wbar, Cfg::W_BYTES);
      bulk_load(smem_w, p.weights, Cfg::W_BYTES, wbar);
      griddep_wait();
      uint32_t L = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const ItemCoord c = decode_item(p, item);
        for (int y = c.ylo; y <= c.yhi; ++y, ++L) {
          const uint32_t slot = L % NST;
          mbar_wait(&empty[slot], ((L / NST) & 1) ^ 1);
          mbar_expect_tx(&full[slot], Cfg::BOX_BYTES);
          tma_load_4d(ring + slot * Cfg::SLOT_BYTES, &tmap, &full[slot], 0, c.x0 - 1, y, c.b);
        }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer (warp-uniform, one elected lane)
    constexpr uint32_t idesc = make_idesc_bf16(TILE_M, NOUT);
    constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (LAYOUT_SW128 << 29);
    const uint32_t w_lo = (smem_u32(smem_w) >> 4) | 0x10000u;
    mbar_wait(wbar, 0);
    tc_fence_after();
    uint32_t L0 = 0, T = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const ItemCoord c = decode_item(p, item);
      int waited = 0;
      const int ylast = c.y0 + c.rcur - 1;
      for (int y = c.y0; y <= ylast; ++y, ++T) {
        const int need = min(y + 1, c.yhi) - c.ylo + 1;
        while (waited < need) {
          const uint32_t q = L0 + waited;
          mbar_wait(&afull[q % TS_NA], (q / TS_NA) & 1);
          ++waited;
        }
        const uint32_t acc = T % TS_NACC;
        mbar_wait(&tempty[acc], ((T / TS_NACC) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * NOUT;
        if (elect_one()) {
          uint32_t accumulate = 0;
#pragma unroll
          for (int dy = 0; dy < 3; ++dy) {
            const int yy = y + dy - 1;
            if (yy < 0 || yy >= p.H) continue;
            const uint32_t q = L0 + (uint32_t)(yy - c.ylo);
            const uint32_t a_t = tmem_base + TS_A_COL0 + (q % TS_NA) * 96u;
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t bl = w_lo + (uint32_t)(((dy * 3 + dx) * Cfg::TAP_BYTES + k * 32) >> 4);
                umma_bf16_ts(d_tmem, a_t + dx * 32 + k * 8, ((uint64_t)DESC_HI << 32) | bl, idesc, accumulate);
                accumulate = 1;
              }
            }
            // input row y - 1 is dead once its 12 MMAs (dy = 0) retire: free its TMEM slot now, two thirds of a row before
            // the accumulator completes, so that the loaders run a full row ahead
            if (dy == 0 && y - 1 >= c.ylo) umma_commit(&aempty[(L0 + (uint32_t)(y - 1 - c.ylo)) % TS_NA]);
          }
          umma_commit(&tfull[acc]);
          if (y == ylast)
            for (int yy = y; yy <= c.yhi; ++yy) umma_commit(&aempty[(L0 + (uint32_t)(yy - c.ylo)) % TS_NA]);
        }
        __syncwarp();
      }
      L0 += (uint32_t)(c.yhi - c.ylo + 1);
    }
  } else if (warp < 6) {
    // ---------------------------------------------------------------- loaders: staging ring -> registers -> TMEM
    const int q4 = warp & 3;
    const int m = q4 * 32 + lane;  // TMEM lane = pixel of the 128-pixel strip; box row m + dx is pixel x0 - 1 + m + dx
    const uint32_t ring_addr = smem_u32(ring);
    const uint32_t lane_taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + TS_A_COL0;
    uint32_t L = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const ItemCoord c = decode_item(p, item);
      for (int y = c.ylo; y <= c.yhi; ++y, ++L) {
        const uint32_t slot = L % NST, as = L % TS_NA;
        mbar_wait(&full[slot], (L / NST) & 1);
        mbar_wait(&aempty[as], ((L / TS_NA) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tile = ring_addr + slot * Cfg::SLOT_BYTES;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          uint32_t v[32];
          ld_swizzled_row128(tile, m + dx, v);
          tmem_st_32x32b_x32(lane_taddr + as * 96u + dx * 32u, v);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&empty[slot]);
          mbar_arrive(&afull[as]);
        }
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue: 2 groups x 4 warps
    const int ew = warp - 6;
    epilogue_post<NOUT, TS_NACC, C>(p, bias_s, tfull, tempty, tmem_base, ew >> 2, warp & 3, lane);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------ CTA-pair TS kernel
// The TS kernel above is bound by the shared-memory port, not the tensor pipe: per 128-pixel output row a CTA moves 72 KB
// of B operand (36 MMAs x 2 KB of weights) next to the loaders', the TMA ring's and the epilogue's traffic.  cta_group::2
// halves the dominant term: two CTAs on the SM pair of one TPC run ONE M = 256 MMA per (tap, K-step) -- 128 pixels (TMEM
// lanes) in each CTA, the 64 output channels' weights split 32 / 32 between the two shared memories -- so every CTA reads
// 1 KB instead of 2 KB of B per MMA and keeps only half of the layer's weights (36 KB).
// The pair works on the two strips (2 sp, 2 sp + 1) of the same chain and row block, so every row count is identical in
// both CTAs; the strip count is padded to even (a strip beyond the image loads zeros and stores nothing).
// Roles per CTA as in the TS kernel; only the leader's warp 1 issues MMAs.  Barriers the leader's issuer waits on (afull,
// tempty, wready) live in the leader and collect arrivals from both CTAs; barriers it signals (aempty, tfull, done) are
// arrived in both CTAs by one multicast tcgen05.commit.
constexpr int TS2_NSTAGE = 6;

template <int NOUT>
struct ConvTs2Cfg {
  static constexpr int ROW_BYTES = 128;
  static constexpr int BOX_BYTES = BOX_W * ROW_BYTES;
  static constexpr int SLOT_BYTES = round_up_c(BOX_BYTES, 1024);
  static constexpr int TAP_BYTES_FULL = NOUT * ROW_BYTES;       // one tap of the packed layer (all output channels)
  static constexpr int TAP_BYTES = (NOUT / 2) * ROW_BYTES;      // this CTA's half
  static constexpr int W_BYTES = 9 * TAP_BYTES;
  static constexpr int OFF_RING = round_up_c(W_BYTES, 1024);
  static constexpr int STAGE_BUFS = 2;
  static constexpr int STAGE_BYTES = STAGE_BUFS * 32 * NOUT * 2;
  static constexpr int OFF_STAGE = OFF_RING + TS2_NSTAGE * SLOT_BYTES;
  static constexpr int OFF_BIAS = OFF_STAGE + EPI_WARPS * STAGE_BYTES;
  static constexpr int OFF_BAR = OFF_BIAS + 256;
  static constexpr int BAR_BYTES = 512;
  static constexpr int SMEM_BYTES = OFF_BAR + BAR_BYTES + 1024;
  static_assert(TS_NACC * NOUT <= TS_A_COL0 && TS_A_COL0 + TS_NA * 96 <= 512, "TMEM plan does not fit 512 columns");
  static_assert((2 * TS2_NSTAGE + 2 * TS_NA + 2 * TS_NACC + 3 + 2 * EPI_WARPS) * 8 + 4 <= BAR_BYTES, "barrier block overflows");
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of one CTA");
};

// RES: the layer has a residual input and fetches it by TMA (epilogue_hidden_tmares), RES = 2: and a second one (the U-Net
// skip tensor, per-thread loads); separate instantiations so that the plain layers (all of DnCNN) keep their own register
// allocation and code (sharing one kernel cost them 5 %, ncu), and the single-residual layers theirs.  The gradient-step
// DRUNet adds two more: TS_GATE (the TMA-fetched tensor is an ELU output t and the sum is multiplied by elu'(t)) and TS_ELU
// (no residual, ELU instead of ReLU).
constexpr int TS_GATE = 3, TS_ELU = 4;
template <int NOUT, int RES>
__global__ void __launch_bounds__(TS_THREADS, 1)
conv3x3_ts2_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_out,
                   const __grid_constant__ CUtensorMap tmap_res, const ConvParams p) {
  using Cfg = ConvTs2Cfg<NOUT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_w = smem;
  uint8_t* ring = smem + Cfg::OFF_RING;
  float* bias_s = reinterpret_cast<float*>(smem + Cfg::OFF_BIAS);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);  // local: TMA landed a row in the staging ring
  uint64_t* empty = full + TS2_NSTAGE;                                // local: loaders have copied it out
  uint64_t* afull = empty + TS2_NSTAGE;                               // leader: both CTAs' copies of the row are in TMEM
  uint64_t* aempty = afull + TS_NA;                                   // both (multicast): MMAs reading them completed
  uint64_t* tfull = aempty + TS_NA;                                   // both (multicast): accumulator stage complete
  uint64_t* tempty = tfull + TS_NACC;                                 // leader: both CTAs' epilogues drained the stage
  uint64_t* wbar = tempty + TS_NACC;                                  // local: this CTA's half of the weights landed
  uint64_t* wready = wbar + 1;                                        // leader: the peer's half landed
  uint64_t* done = wready + 1;                                        // both (multicast): every MMA of the launch completed
  uint64_t* rbar = done + 1;                                          // local: residual boxes (two per epilogue warp) landed
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(rbar + 2 * EPI_WARPS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  griddep_launch_dependents();

  if (threadIdx.x == 0) {
    for (int i = 0; i < TS2_NSTAGE; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 4);
    }
    for (int i = 0; i < TS_NA; ++i) {
      mbar_init(&afull[i], 8);
      mbar_init(&aempty[i], 1);
    }
    for (int i = 0; i < TS_NACC; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 8);
    }
    mbar_init(wbar, 1);
    mbar_init(wready, 1);
    mbar_init(done, 1);
    if (RES && RES != TS_ELU)
      for (int i = 0; i < 2 * EPI_WARPS; ++i) mbar_init(&rbar[i], 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc2(tmem_ptr_s, 512);
    tmem_relinquish2();
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + NOUT) bias_s[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
  tc_fence_before();
  cluster_sync();  // barriers of both CTAs are initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t afull_c = mapa_shared(smem_u32(afull), 0);
  const uint32_t tempty_c = mapa_shared(smem_u32(tempty), 0);

  if (warp == 0) {
    if (lane == 0) {
      // ---------------------------------------------------------------- TMA producer
      tma_prefetch_desc(&tmap);
      mbar_expect_tx(wbar, Cfg::W_BYTES);
      for (int t = 0; t < 9; ++t)
        bulk_load(smem_w + t * Cfg::TAP_BYTES, p.weights + (size_t)t * Cfg::TAP_BYTES_FULL + rank * Cfg::TAP_BYTES,
                  Cfg::TAP_BYTES, wbar);
      if (rank != 0) {
        mbar_wait(wbar, 0);
        mbar_arrive_cluster(mapa_shared(smem_u32(wready), 0));
      }
      griddep_wait();
      uint32_t L = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const ItemCoord c = decode_item(p, item);
        for (int y = c.ylo; y <= c.yhi; ++y, ++L) {
          const uint32_t slot = L % TS2_NSTAGE;
          mbar_wait(&empty[slot], ((L / TS2_NSTAGE) & 1) ^ 1);
          mbar_expect_tx(&full[slot], Cfg::BOX_BYTES);
          tma_load_4d(ring + slot * Cfg::SLOT_BYTES, &tmap, &full[slot], 0, c.x0 - 1, y, c.b);
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ---------------------------------------------------------------- MMA issuer of the pair
      constexpr uint32_t idesc = make_idesc_bf16(2 * TILE_M, NOUT);
      constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (LAYOUT_SW128 << 29);
      const uint32_t w_lo = (smem_u32(smem_w) >> 4) | 0x10000u;
      mbar_wait(wbar, 0);
      mbar_wait_cluster(wready, 0);
      tc_fence_after();
      // ONE thread runs the whole issue loop, barrier waits included: the tensor pipe's queue is shallow, so whatever the
      // issuing thread executes between two MMAs beyond a few dozen cycles is a bubble in the pipe (a warp-uniform wait /
      // elect / syncwarp boundary per row cost ~160 cycles: conv_fused2.cu has the measurement).  A source row is awaited
      // right before the first 12 MMAs that read it.
      if (elect_one()) {
        uint32_t L0 = 0, T = 0;
#pragma unroll 1
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
          const ItemCoord c = decode_item(p, item);
          int waited = 0;
          const int ylast = c.y0 + c.rcur - 1;
#pragma unroll 1
          for (int y = c.y0; y <= ylast; ++y, ++T) {
            const uint32_t acc = T % TS_NACC;
            mbar_wait_spin(&tempty[acc], ((T / TS_NACC) & 1) ^ 1);
            const uint32_t d_tmem = tmem_base + acc * NOUT;
            uint32_t accumulate = 0;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
              const int yy = y + dy - 1;
              if (yy < 0 || yy >= p.H) continue;
              const int rel = yy - c.ylo;
              const uint32_t q = L0 + (uint32_t)rel;
              if (rel == waited) {
                mbar_wait_spin(&afull[q % TS_NA], (q / TS_NA) & 1);
                ++waited;
              }
              tc_fence_after();
              const uint32_t a_t = tmem_base + TS_A_COL0 + (q % TS_NA) * 96u;
#pragma unroll
              for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t bl = w_lo + (uint32_t)(((dy * 3 + dx) * Cfg::TAP_BYTES + k * 32) >> 4);
                  umma_bf16_ts2(d_tmem, a_t + dx * 32 + k * 8, ((uint64_t)DESC_HI << 32) | bl, idesc, accumulate | (uint32_t)(dx | k));
                }
              }
              accumulate = 1;
              if ((dy == 0 && y - 1 >= c.ylo) || y == ylast) umma_commit2(&aempty[q % TS_NA], 3);
            }
            umma_commit2(&tfull[acc], 3);
          }
          L0 += (uint32_t)(c.yhi - c.ylo + 1);
        }
        umma_commit2(done, 3);
      }
      __syncwarp();
    }
    mbar_wait(done, 0);  // both CTAs: no MMA still reads this CTA's shared / tensor memory, no commit is still in flight
  } else if (warp < 6) {
    // ---------------------------------------------------------------- loaders: staging ring -> registers -> TMEM
    const int q4 = warp & 3;
    const int m = q4 * 32 + lane;
    const uint32_t ring_addr = smem_u32(ring);
    const uint32_t lane_taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + TS_A_COL0;
    uint32_t L = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const ItemCoord c = decode_item(p, item);
      for (int y = c.ylo; y <= c.yhi; ++y, ++L) {
        const uint32_t slot = L % TS2_NSTAGE, as = L % TS_NA;
        mbar_wait(&full[slot], (L / TS2_NSTAGE) & 1);
        mbar_wait(&aempty[as], ((L / TS_NA) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tile = ring_addr + slot * Cfg::SLOT_BYTES;
        // (reading the three shifted rows into registers before the TMEM slot is awaited was tried: 113 -> 122 us per layer,
        // 96 live registers per loader thread and shared-memory reads bunched against the operand fetch)
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          uint32_t v[32];
          ld_swizzled_row128(tile, m + dx, v);
          tmem_st_32x32b_x32(lane_taddr + as * 96u + dx * 32u, v);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&empty[slot]);
          mbar_arrive_remote(afull_c + as * 8u);
        }
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue: 2 groups x 4 warps
    const int ew = warp - 6;
    if (RES && RES != TS_ELU)
      epilogue_hidden_tmares<NOUT, TS_NACC, RES == 2, RES == TS_GATE>(p, &tmap_out, &tmap_res,
                                            smem + Cfg::OFF_STAGE + ew * Cfg::STAGE_BYTES,
                                            rbar + 2 * ew, bias_s, tfull, tempty, tmem_base, ew >> 2, warp & 3, lane, tempty_c);
    else
      epilogue_hidden<NOUT, TS_NACC, RES == TS_ELU>(p, &tmap_out, smem + Cfg::OFF_STAGE + ew * Cfg::STAGE_BYTES, bias_s, tfull,
                                                    tempty, tmem_base, ew >> 2, warp & 3, lane, tempty_c);
  }
  tc_fence_before();
  cluster_sync();  // neither CTA may exit (or free tensor memory) while its partner can still signal or read it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------ host side
PFN_tensorMapEncodeTiled get_tensor_map_encoder() {
  static PFN_tensorMapEncodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tensorMapEncodeTiled>(ptr);
  });
  return fn;
}

// Activation tensor maps (bf16 NHWC, dims {C, W, H, B}).  box_w = BOX_W: input rows with halo (OOB zero fill = the
// convolution's zero padding); box_w = 32: one epilogue warp's output box.  Encoding costs microseconds on the host,
// so the few (pointer, shape) combinations of a run are cached per thread.
struct MapKey {
  const void* ptr;
  int B, H, W, C, box_w;
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && B == o.B && H == o.H && W == o.W && C == o.C && box_w == o.box_w;
  }
};
int get_act_tensor_map(CUtensorMap* map, const void* ptr, int B, int H, int W, int C, int box_w) {
  static thread_local std::vector<std::pair<MapKey, CUtensorMap>> cache;
  const MapKey key{ptr, B, H, W, C, box_w};
  for (const auto& e : cache)
    if (e.first == key) {
      *map = e.second;
      return PSGLA_OK;
    }
  PFN_tensorMapEncodeTiled enc = get_tensor_map_encoder();
  if (!enc) return set_error(PSGLA_E_NODEVICE, "cuTensorMapEncodeTiled driver entry point not available");
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  const cuuint32_t box[4] = {(cuuint32_t)C, (cuuint32_t)box_w, 1, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUtensorMapSwizzle sw = (C == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(PSGLA_E_BADARG, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  if (cache.size() >= 64) cache.erase(cache.begin());
  cache.emplace_back(key, *map);
  return PSGLA_OK;
}

// Work items = (chain, 128-pixel strip, block of R output rows), dealt round-robin to one persistent CTA per SM.
// R trades the 2 halo rows an item re-reads against the tail when items do not divide by the CTA count:
// pick the R that minimises (items per CTA) * (R + 1).
static void plan_items(ConvParams* p) {
  p->strips = (p->W + TILE_M - 1) / TILE_M;
  const int sms = num_sms();
  int best = 1;
  long long best_cost = -1;
  const int cands[] = {32, 16, 8, 4, 2, 1};
  for (int R : cands) {
    const long long items = (long long)p->B * p->strips * ((p->H + R - 1) / R);
    const long long cost = ((items + sms - 1) / sms) * (std::min(R, p->H) + 1);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = R;
    }
  }
  const char* e = getenv("PSGLA_CONV_ROWS");
  if (e && atoi(e) > 0) best = atoi(e);
  p->R = best;
  p->row_blocks = (p->H + best - 1) / best;
  p->n_items = p->B * p->strips * p->row_blocks;
}

// The first layer: bf16 NHWC16 input (3 channels padded to 16) -> bf16 NHWC 64-channel output
static int launch_first(const void* in, void* out_bf16, ConvParams p, cudaStream_t st) {
  using Cfg = ConvCfg<16, 64>;
  CUtensorMap map, map_out;
  int rc = get_act_tensor_map(&map, in, p.B, p.H, p.W, 16, BOX_W);
  if (rc) return rc;
  rc = get_act_tensor_map(&map_out, out_bf16, p.B, p.H, p.W, 64, 32);
  if (rc) return rc;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (!(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(conv3x3_kernel<16, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        Cfg::SMEM_BYTES));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  plan_items(&p);
  const int grid = p.n_items < num_sms() ? p.n_items : num_sms();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(CONV_THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // pairs with griddepcontrol.* in the kernel
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv3x3_kernel<16, 64>, map, map_out, p));
  return PSGLA_OK;
}

// The last layer: bf16 NHWC 64-channel input -> the fused Langevin post epilogue (fp32 NCHW outputs of C channels named in p)
template <int C>
static int launch_last_t(const void* in, ConvParams p, cudaStream_t st) {
  using Cfg = ConvTsCfg<16>;
  CUtensorMap map;
  int rc = get_act_tensor_map(&map, in, p.B, p.H, p.W, 64, BOX_W);
  if (rc) return rc;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (!(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(conv3x3_ts_kernel<16, C>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        Cfg::SMEM_BYTES));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  plan_items(&p);
  const int grid = p.n_items < num_sms() ? p.n_items : num_sms();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(TS_THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv3x3_ts_kernel<16, C>, map, p));
  return PSGLA_OK;
}
static int launch_last(const void* in, const ConvParams& p, int channels, cudaStream_t st) {
  return channels == 1 ? launch_last_t<1>(in, p, st) : launch_last_t<3>(in, p, st);
}

// Work items of the pair kernel: (chain, row block, strip) with the strip count padded to even and the strip index
// fastest, so that items 2i and 2i + 1 -- the two CTAs of a cluster -- share chain and rows.
static void plan_items_pair(ConvParams* p, int n_clusters) {
  p->strips = ((p->W + TILE_M - 1) / TILE_M + 1) & ~1;
  int best = 1;
  long long best_cost = -1;
  const int cands[] = {32, 16, 8, 4, 2, 1};
  for (int R : cands) {
    const long long pairs = (long long)p->B * (p->strips / 2) * ((p->H + R - 1) / R);
    const long long cost = ((pairs + n_clusters - 1) / n_clusters) * (std::min(R, p->H) + 1);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = R;
    }
  }
  const char* e = getenv("PSGLA_CONV_ROWS");
  if (e && atoi(e) > 0) best = atoi(e);
  p->R = best;
  p->row_blocks = (p->H + best - 1) / best;
  p->n_items = p->B * p->strips * p->row_blocks;
}

template <int NOUT, int RES>
static int launch_conv_ts2_t(const void* in, void* out_bf16, ConvParams p, cudaStream_t st) {
  using Cfg = ConvTs2Cfg<NOUT>;
  CUtensorMap map, map_out;
  int rc = get_act_tensor_map(&map, in, p.B, p.H, p.W, 64, BOX_W);
  if (rc) return rc;
  rc = get_act_tensor_map(&map_out, out_bf16, p.B, p.H, p.W, NOUT, 32);
  if (rc) return rc;
  CUtensorMap map_res = map_out;  // unused without a residual input
  if (p.res1) {
    rc = get_act_tensor_map(&map_res, p.res1, p.B, p.H, p.W, NOUT, 32);
    if (rc) return rc;
  }
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3(TS_THREADS);
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
  static std::atomic<int> max_clusters_dev[kMaxDevices];  // per device: CTA pairs it holds at once (one CTA per SM); 0 = not asked yet
  std::atomic<int>& mc_slot = max_clusters_dev[current_device() % kMaxDevices];
  int max_clusters = mc_slot.load(std::memory_order_acquire);
  if (!max_clusters) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(conv3x3_ts2_kernel<NOUT, RES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        Cfg::SMEM_BYTES));
    cfg.gridDim = dim3((unsigned)(num_sms() & ~1));
    int n = 0;
    PSGLA_CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, conv3x3_ts2_kernel<NOUT, RES>, &cfg));
    max_clusters = n > 0 ? std::min(n, num_sms() / 2) : num_sms() / 2;
    mc_slot.store(max_clusters, std::memory_order_release);
    if (getenv("PSGLA_VERBOSE")) fprintf(stderr, "psgla_b200: conv3x3_ts2_kernel: %d co-resident CTA pairs (occupancy query %d)\n", max_clusters, n);
  }
  plan_items_pair(&p, max_clusters);
  const int pairs = p.n_items / 2;
  cfg.gridDim = dim3((unsigned)(2 * std::min(pairs, max_clusters)));
  if (getenv("PSGLA_VERBOSE")) fprintf(stderr, "psgla_b200: pair conv B=%d H=%d W=%d: R=%d items=%d grid=%u\n", p.B, p.H, p.W, p.R, p.n_items, cfg.gridDim.x);
  PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv3x3_ts2_kernel<NOUT, RES>, map, map_out, map_res, p));
  return PSGLA_OK;
}

// The hidden 64 -> 64 channel layers, with up to two residual inputs, or (act ACT_ELU / ACT_GATE) the gradient-step DRUNet's
// ELU and gate epilogues
static int launch_hidden64(const void* in, void* out, const ConvParams& p, cudaStream_t st, int act = ACT_NONE) {
  if (act == ACT_ELU) return launch_conv_ts2_t<64, TS_ELU>(in, out, p, st);
  if (act == ACT_GATE) return launch_conv_ts2_t<64, TS_GATE>(in, out, p, st);
  if (!p.res1) return launch_conv_ts2_t<64, 0>(in, out, p, st);
  return p.res2 ? launch_conv_ts2_t<64, 2>(in, out, p, st) : launch_conv_ts2_t<64, 1>(in, out, p, st);
}

// ---- packed weight layout: per layer [weights (9 taps, swizzled) | bias fp32], each layer 1024 B aligned
struct LayerInfo {
  int cin, nout;  // padded
  size_t w_off, b_off;
};
static LayerInfo layer_info(int depth, int layer) {
  LayerInfo li{};
  size_t off = 0;
  for (int l = 0; l <= layer; ++l) {
    const int cin = (l == 0) ? 16 : 64;
    const int nout = (l == depth - 1) ? 16 : 64;
    li.cin = cin;
    li.nout = nout;
    li.w_off = off;
    const size_t wbytes = (size_t)9 * nout * cin * 2;
    li.b_off = off + wbytes;
    off = (li.b_off + (size_t)nout * 4 + 1023) / 1024 * 1024;
  }
  return li;
}
static size_t packed_bytes(int depth) {
  LayerInfo li = layer_info(depth, depth - 1);
  return (li.b_off + (size_t)li.nout * 4 + 1023) / 1024 * 1024;
}

static inline uint16_t f32_to_bf16_rn(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);  // NaN
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

void pack_conv3x3_swizzled(const float* w, int nout_real, int cin_real, int nout_pad, int cin_pad, uint8_t* dst);

}  // namespace psgla

using namespace psgla;

extern "C" size_t psgla_dncnn_packed_bytes(int depth) { return depth >= 2 ? packed_bytes(depth) : 0; }

extern "C" int psgla_dncnn_pack_weights(int depth, const float* const* weights_host, const float* const* biases_host,
                                        void* packed_dev, void* stream) {
  return psgla_dncnn_pack_weights_ch(depth, 3, weights_host, biases_host, packed_dev, stream);
}

// Image channel k of a C-channel network (C = 3 or 1) is K slot k of the first layer and N slot k of the last: the denoiser
// input is NHWC16 with the image from slot 0 whatever C (the DRUNet head's noise-level channel: dru_pack_layer).
extern "C" int psgla_dncnn_pack_weights_ch(int depth, int channels, const float* const* weights_host,
                                           const float* const* biases_host, void* packed_dev, void* stream) {
  PSGLA_REQUIRE(depth >= 2 && weights_host && packed_dev, "psgla_dncnn_pack_weights: bad argument");
  PSGLA_REQUIRE(channels == 3 || channels == 1, "psgla_dncnn_pack_weights_ch: channels must be 3 or 1 (got %d)", channels);
  std::vector<uint8_t> host(packed_bytes(depth), 0);
  for (int l = 0; l < depth; ++l) {
    const LayerInfo li = layer_info(depth, l);
    const int cin_real = (l == 0) ? channels : 64;
    const int nout_real = (l == depth - 1) ? channels : 64;
    const float* w = weights_host[l];  // OIHW [nout_real][cin_real][3][3]
    PSGLA_REQUIRE(w != nullptr, "layer %d: null weight pointer", l);
    pack_conv3x3_swizzled(w, nout_real, cin_real, li.nout, li.cin, host.data() + li.w_off);
    if (biases_host && biases_host[l])
      std::memcpy(&host[li.b_off], biases_host[l], (size_t)nout_real * 4);
  }
  PSGLA_CUDA_TRY(cudaMemcpyAsync(packed_dev, host.data(), host.size(), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  PSGLA_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));  // `host` dies at return
  return PSGLA_OK;
}

extern "C" size_t psgla_dncnn_workspace_bytes(psgla_img_shape s) {
  // two ping-pong activation buffers, each rounded up to 1 KB
  return 2 * (((size_t)s.B * s.H * s.W * 64 * 2 + 1023) / 1024 * 1024);
}

static int check_shape(const psgla_img_shape& s) {
  PSGLA_REQUIRE(s.B > 0 && s.H > 0 && s.W > 0 && (s.C == 3 || s.C == 1),
                "image shape must be [B>0][C = 1 or 3][H>0][W>0], got [%d][%d][%d][%d]", s.B, s.C, s.H, s.W);
  return PSGLA_OK;
}

static ConvParams base_params(const psgla_img_shape& s, const uint8_t* packed, const LayerInfo& li) {
  ConvParams p{};
  p.B = s.B;
  p.H = s.H;
  p.W = s.W;
  p.weights = packed + li.w_off;
  p.bias = reinterpret_cast<const float*>(packed + li.b_off);
  return p;
}

// The last layer (64 -> C) with the Langevin post (and optionally the next iteration's pre) in its epilogue.
static int last_layer_post(int depth, const uint8_t* packed, const psgla_img_shape& shape, const void* hidden, const float* base_dev,
                           const psgla_post_params* post, float* x_out_dev, float* sample_dev, float* mean_dev,
                           float* mean2_dev, const psgla_next_pre* next, cudaStream_t st) {
  const LayerInfo li = layer_info(depth, depth - 1);
  ConvParams p = base_params(shape, packed, li);
  p.base = base_dev;
  p.x_out = x_out_dev;
  p.sample = sample_dev;
  p.mean = mean_dev;
  p.mean2 = mean2_dev;
  p.gain = post->gain;
  p.base_scale = 1.0f;  // DnCNN is a residual denoiser: X+ = base + gain * R
  p.w_old = post->w_old;
  p.w_new = post->w_new;
  p.reverse = (depth - 1) & 1;
  int rc = set_next_pre(&p, next, shape.C);
  if (rc) return rc;
  return launch_last(hidden, p, shape.C, st);
}

extern "C" int psgla_conv3x3_layer(const void* packed_dev, int depth, int layer, psgla_img_shape shape,
                                   const void* in_dev, void* out_dev, int relu, void* stream) {
  PSGLA_REQUIRE(packed_dev && in_dev && out_dev && depth >= 2 && layer >= 0 && layer < depth,
                "psgla_conv3x3_layer: bad argument");
  int rc = check_shape(shape);
  if (rc) return rc;
  const LayerInfo li = layer_info(depth, layer);
  ConvParams p = base_params(shape, (const uint8_t*)packed_dev, li);
  p.relu = relu;
  cudaStream_t st = (cudaStream_t)stream;
  if (layer == depth - 1) {  // raw conv + bias -> fp32 NCHW
    p.x_out = (float*)out_dev;
    return launch_last(in_dev, p, shape.C, st);
  }
  return layer == 0 ? launch_first(in_dev, out_dev, p, st) : launch_hidden64(in_dev, out_dev, p, st);
}

extern "C" int psgla_dncnn_residual_post(int depth, const void* packed_dev, psgla_img_shape shape,
                                         const void* den_in_dev, void* workspace_dev, size_t workspace_bytes,
                                         const float* base_dev, const psgla_post_params* post, float* x_out_dev,
                                         float* sample_dev, float* mean_dev, float* mean2_dev, void* stream) {
  return psgla_dncnn_residual_post_next(depth, packed_dev, shape, den_in_dev, workspace_dev, workspace_bytes, base_dev, post,
                                        x_out_dev, sample_dev, mean_dev, mean2_dev, nullptr, stream);
}

extern "C" int psgla_dncnn_residual_post_next(int depth, const void* packed_dev, psgla_img_shape shape,
                                              const void* den_in_dev, void* workspace_dev, size_t workspace_bytes,
                                              const float* base_dev, const psgla_post_params* post, float* x_out_dev,
                                              float* sample_dev, float* mean_dev, float* mean2_dev,
                                              const psgla_next_pre* next, void* stream) {
  PSGLA_REQUIRE(packed_dev && den_in_dev && workspace_dev && post && x_out_dev && depth >= 2,
                "psgla_dncnn_residual_post: bad argument");
  {
    const int rcn = check_next_pre(next, shape);
    if (rcn) return rcn;
  }
  PSGLA_REQUIRE((mean_dev == nullptr) == (mean2_dev == nullptr), "mean and mean2 must be given together");
  int rc = check_shape(shape);
  if (rc) return rc;
  if (workspace_bytes < psgla_dncnn_workspace_bytes(shape))
    return set_error(PSGLA_E_WORKSPACE, "workspace of %zu bytes is smaller than the %zu needed", workspace_bytes,
                     psgla_dncnn_workspace_bytes(shape));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t half = ((size_t)shape.B * shape.H * shape.W * 64 * 2 + 1023) / 1024 * 1024;
  uint8_t* ws[2] = {(uint8_t*)workspace_dev, (uint8_t*)workspace_dev + half};
  const uint8_t* packed = (const uint8_t*)packed_dev;
  const void* cur = den_in_dev;
  int wsel = 0;  // the buffer the next layer writes
  for (int l = 0; l < depth - 1; ++l) {
    const LayerInfo li = layer_info(depth, l);
    if (l >= 1 && l + 1 < depth - 1) {
      // few chains: two hidden layers per launch (conv_fused2.cu), the intermediate rows never leave the SM pair
      const LayerInfo l2 = layer_info(depth, l + 1);
      int fused = 0;
      rc = conv64_hidden_fused2(cur, ws[wsel], packed + li.w_off, reinterpret_cast<const float*>(packed + li.b_off),
                                packed + l2.w_off, reinterpret_cast<const float*>(packed + l2.b_off), shape.B, shape.H, shape.W,
                                &fused, st);
      if (rc) return rc;
      if (fused) {
        cur = ws[wsel];
        wsel ^= 1;
        ++l;
        continue;
      }
    }
    ConvParams pl = base_params(shape, packed, li);
    pl.relu = 1;
    pl.reverse = l & 1;
    rc = (l == 0) ? launch_first(cur, ws[wsel], pl, st) : launch_hidden64(cur, ws[wsel], pl, st);
    if (rc) return rc;
    cur = ws[wsel];
    wsel ^= 1;
  }
  return last_layer_post(depth, packed, shape, cur, base_dev, post, x_out_dev, sample_dev, mean_dev, mean2_dev, next, st);
}

extern "C" int psgla_dncnn_last_layer_post_next(int depth, const void* packed_dev, psgla_img_shape shape,
                                                const void* hidden_dev, const float* base_dev,
                                                const psgla_post_params* post, float* x_out_dev, float* sample_dev,
                                                float* mean_dev, float* mean2_dev, const psgla_next_pre* next, void* stream) {
  PSGLA_REQUIRE(packed_dev && hidden_dev && base_dev && post && x_out_dev && depth >= 2,
                "psgla_dncnn_last_layer_post_next: bad argument");
  PSGLA_REQUIRE((mean_dev == nullptr) == (mean2_dev == nullptr), "mean and mean2 must be given together");
  int rc = check_next_pre(next, shape);
  if (rc) return rc;
  rc = check_shape(shape);
  if (rc) return rc;
  return last_layer_post(depth, (const uint8_t*)packed_dev, shape, hidden_dev, base_dev, post, x_out_dev, sample_dev, mean_dev,
                         mean2_dev, next, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ internal API (drunet.cu)
namespace psgla {

// fp32 OIHW [nout_real][cin_real][3][3] -> bf16 [tap][nout_pad][cin_pad], 128B- (cin_pad = 64) or 32B- (16) swizzled as the
// resident-weight kernels expect; dst must be zero-initialised (padding rows / channels stay zero).
void pack_conv3x3_swizzled(const float* w, int nout_real, int cin_real, int nout_pad, int cin_pad, uint8_t* dst) {
  const int row_bytes = cin_pad * 2;
  for (int tap = 0; tap < 9; ++tap)
    for (int n = 0; n < nout_real; ++n)
      for (int k = 0; k < cin_real; ++k) {
        const float val = w[((size_t)n * cin_real + k) * 9 + tap];
        const int kbyte = k * 2;
        int chunk = kbyte >> 4;
        chunk ^= (row_bytes == 128) ? (n & 7) : ((n >> 2) & 1);
        const size_t phys = (size_t)tap * nout_pad * row_bytes + (size_t)n * row_bytes + chunk * 16 + (kbyte & 15);
        const uint16_t h = f32_to_bf16_rn(val);
        std::memcpy(dst + phys, &h, 2);
      }
}

int next_layer_direction() {
  static thread_local int dir = 0;
  dir ^= 1;
  return dir;
}

int conv64_hidden(const void* in, void* out, const uint8_t* w, const float* bias, int B, int H, int W, int act,
                  const void* res1, const void* res2, cudaStream_t st) {
  ConvParams p{};
  p.B = B, p.H = H, p.W = W;
  p.reverse = next_layer_direction();
  p.weights = w;
  p.bias = bias;
  p.relu = act == ACT_RELU;
  p.res1 = (const __nv_bfloat16*)res1;
  p.res2 = (const __nv_bfloat16*)res2;
  return launch_hidden64(in, out, p, st, act);
}

int conv_first16(const void* in16, void* out, const uint8_t* w, const float* bias, int B, int H, int W, int relu,
                 cudaStream_t st) {
  ConvParams p{};
  p.B = B, p.H = H, p.W = W;
  p.weights = w;
  p.bias = bias;
  p.relu = relu;
  return launch_first(in16, out, p, st);
}

int check_next_pre(const psgla_next_pre* next, const psgla_img_shape& s) {
  if (!next) return PSGLA_OK;
  PSGLA_REQUIRE(next->pre && next->mask_dev && next->y_dev && next->base_dev && next->den_in_dev,
                "psgla_next_pre: null pointer");
  PSGLA_REQUIRE((next->mask_B == 1 || next->mask_B == s.B) && (next->y_B == 1 || next->y_B == s.B),
                "psgla_next_pre: mask_B / y_B must be 1 or B");
  PreArgs a;
  return fill_pre(next->pre, &a);
}

int set_next_pre(ConvParams* p, const psgla_next_pre* next, int channels) {
  p->nx_enable = 0;
  if (!next) return PSGLA_OK;
  int rc = fill_pre(next->pre, &p->nx);
  if (rc) return rc;
  p->nx.chw = (long long)channels * p->H * p->W;
  p->nx_enable = 1;
  p->nx_mask = next->mask_dev;
  p->nx_y = next->y_dev;
  p->nx_mask_B = next->mask_B;
  p->nx_y_B = next->y_B;
  p->nx_base = next->base_dev;
  p->nx_den_in = (__nv_bfloat16*)next->den_in_dev;
  return PSGLA_OK;
}

int conv_last_post(const void* in, const uint8_t* w, const float* bias, int B, int C, int H, int W, const float* base,
                   float base_scale, float gain, float w_old, float w_new, float* x_out, float* sample, float* mean,
                   float* mean2, const psgla_next_pre* next, cudaStream_t st) {
  ConvParams p{};
  p.B = B, p.H = H, p.W = W;
  p.weights = w;
  p.bias = bias;
  p.base = base;
  p.base_scale = base_scale;
  p.gain = gain;
  p.w_old = w_old;
  p.w_new = w_new;
  p.x_out = x_out;
  p.sample = sample;
  p.mean = mean;
  p.mean2 = mean2;
  int rc = set_next_pre(&p, next, C);
  if (rc) return rc;
  return launch_last(in, p, C, st);
}

}  // namespace psgla
