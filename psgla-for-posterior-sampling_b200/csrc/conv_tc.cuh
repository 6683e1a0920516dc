// Shared device code of the resident-weight 3x3 convolution kernels (conv_tc.cu: one kernel per layer role; conv_fused2.cu:
// two hidden layers per launch): configurations, the parameter block, work-item decoding, the epilogues.
#pragma once
#include <cuda_bf16.h>

#include <cstdint>

#include "common.cuh"
#include "conv_api.cuh"
#include "langevin.cuh"
#include "sm100.cuh"

namespace psgla {

using namespace sm100;

constexpr int TILE_M = 128;
constexpr int BOX_W = TILE_M + 2;
constexpr int NACC = 4;       // TMEM accumulator stages; stage s is drained by epilogue group s & 1
constexpr int EPI_WARPS = 8;  // two groups of four warps (one warp per TMEM lane quarter)
constexpr int CONV_THREADS = 64 + 32 * EPI_WARPS;

constexpr int round_up_c(int v, int a) { return (v + a - 1) / a * a; }

// f[0..7] += eight bf16 values packed in a 16-byte vector
__device__ __forceinline__ void add_bf16x8(float (&f)[8], const uint4 r) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] += __uint_as_float(w[i] << 16);
    f[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
  }
}
// ELU (alpha = 1) in place: z for z > 0, exp(z) - 1 otherwise (the gradient-step DRUNet's block activation).  exp by the
// MUFU approximation: its ~1e-7 absolute error near 0 is far below the bf16 output's rounding and the conv's own error bound;
// expm1f, inlined per element, made the forward's ELU layers slower than the whole backward.
__device__ __forceinline__ void elu8(float (&f)[8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) f[i] = f[i] > 0.f ? f[i] : __expf(f[i]) - 1.f;
}
// f *= elu'(z) with t = bf16 ELU(z) as the forward stored it: elu'(z) = 1 for t > 0, else exp(z) = t + 1.  The backward of a
// residual block's activation, so that no pre-activation has to be kept.
__device__ __forceinline__ void gate_bf16x8(float (&f)[8], const uint4 r) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float t0 = __uint_as_float(w[i] << 16), t1 = __uint_as_float(w[i] & 0xffff0000u);
    f[2 * i] *= t0 > 0.f ? 1.f : t0 + 1.f;
    f[2 * i + 1] *= t1 > 0.f ? 1.f : t1 + 1.f;
  }
}

// The 8 biases of 16-byte output chunk j.  The epilogues fetch them ONE CHUNK AHEAD with explicit shared-space loads: through a
// generic pointer they compile to LD.E, and placed after the previous chunk's staging store (a "memory"-clobbering asm
// statement keeps program order) every chunk paid a long-scoreboard round trip -- the first layer, whose epilogue is its
// critical path, ran at 1 240 cycles per row (profiles/r02_first_last_layer_full.txt).
struct BiasPair {
  float4 b0, b1;
};
__device__ __forceinline__ BiasPair load_bias_pair(uint32_t bias_saddr, int j) {
  BiasPair r;
  r.b0 = ld_shared_f4_nc(bias_saddr + 32u * (uint32_t)j);
  r.b1 = ld_shared_f4_nc(bias_saddr + 32u * (uint32_t)j + 16u);
  return r;
}

// The SS kernel (A from shared memory), i.e. the first layer: 16 (3 padded) input channels, 64 output channels
template <int CIN, int NOUT>
struct ConvCfg {
  static_assert(CIN == 16, "ring depth, swizzle and staging are sized for the 16-channel rows of the first layer");
  static constexpr int ROW_BYTES = CIN * 2;
  static constexpr int BOX_BYTES = BOX_W * ROW_BYTES;
  static constexpr int SLOT_BYTES = round_up_c(BOX_BYTES, 1024);
  static constexpr uint32_t LAYOUT = LAYOUT_SW32;
  static constexpr uint32_t SBO = 8 * ROW_BYTES;
  static constexpr int KSTEPS = CIN / 16;
  static constexpr int TAP_BYTES = NOUT * ROW_BYTES;
  static constexpr int W_BYTES = 9 * TAP_BYTES;
  static constexpr int OFF_RING = round_up_c(W_BYTES, 1024);
  // Ring depth.  A slot stays occupied for three output rows, so NSTAGE - 3 rows are in flight ahead of the MMAs; the
  // 16-channel first layer consumes a row in ~430 cycles against ~2 us of TMA latency from HBM and needs a deep ring
  // (6 slots: 1 560 cycles per row measured), its rows are only 5 KB.
  static constexpr int NSTAGE = 20;
  // two 32-pixel output boxes per epilogue warp: the warp fills one while the TMA store of the previous row still reads
  // the other
  static constexpr int STAGE_BUFS = 2;
  static constexpr int STAGE_BYTES = STAGE_BUFS * 32 * NOUT * 2;
  static constexpr int OFF_STAGE = OFF_RING + NSTAGE * SLOT_BYTES;
  static constexpr int OFF_BIAS = OFF_STAGE + EPI_WARPS * STAGE_BYTES;
  static constexpr int OFF_BAR = OFF_BIAS + 256;
  static constexpr int BAR_BYTES = 512;
  static_assert((2 * NSTAGE + 2 * NACC + 1) * 8 + 4 <= BAR_BYTES, "barrier block overflows");
  static constexpr int SMEM_BYTES = OFF_BAR + BAR_BYTES + 1024;  // + slack to align the dynamic base to 1024
  static constexpr int TMEM_COLS = (NACC * NOUT) < 32 ? 32 : NACC * NOUT;
  static_assert((TMEM_COLS & (TMEM_COLS - 1)) == 0 && TMEM_COLS <= 512, "TMEM columns must be a power of two <= 512");
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of one CTA");
};

struct ConvParams {
  int B, H, W;
  int R, strips, row_blocks, n_items;
  int reverse;  // walk the work items back to front (see decode_item)
  const uint8_t* weights;  // 9 taps, swizzled
  const float* bias;       // NOUT floats
  int relu;
  // hidden layers: optional bf16 NHWC tensors of the output's shape added before the ReLU (DRUNet residual / skip adds)
  const __nv_bfloat16* res1;
  const __nv_bfloat16* res2;
  // last layer
  const float* base;
  float* x_out;
  float* sample;
  float* mean;
  float* mean2;
  float gain, base_scale, w_old, w_new;
  // last layer, optional: the "pre" step of the NEXT iteration applied to the iterate this epilogue produces (inpainting):
  // nx_base = langevin_base(X+), nx_den_in = bf16 NHWC16 of it (PSGLA) or of X+ (PnP-ULA); nx_base may alias base.
  int nx_enable;
  PreArgs nx;
  const float* nx_mask;
  const float* nx_y;
  int nx_mask_B, nx_y_B;
  float* nx_base;
  __nv_bfloat16* nx_den_in;
};

int set_next_pre(ConvParams* p, const psgla_next_pre* next, int channels);  // host: fills the nx_* fields (conv_tc.cu)

struct ItemCoord {
  int b, y0, rcur, x0, ylo, yhi;
};
// Items are dealt to the persistent CTAs in index order, so a layer finishes with the END of the activation tensor freshly
// written -- and a 268 MB tensor (32 chains of 256 x 256 x 64 bf16) leaves roughly its last third in the 126 MB L2.  Consecutive
// layers therefore walk the items in opposite directions (reverse = layer parity): each layer starts on what the previous one
// wrote last and reads it from L2 instead of HBM.  (In the pair kernel items 2i and 2i + 1 swap ranks under the reversal and
// still share chain and rows.)
__device__ __forceinline__ ItemCoord decode_item(const ConvParams& p, int item) {
  if (p.reverse) item = p.n_items - 1 - item;
  ItemCoord c;
  const int sx = item % p.strips;
  const int t = item / p.strips;
  const int ry = t % p.row_blocks;
  c.b = t / p.row_blocks;
  c.y0 = ry * p.R;
  c.rcur = min(p.R, p.H - c.y0);
  c.x0 = sx * TILE_M;
  c.ylo = max(c.y0 - 1, 0);
  c.yhi = min(c.y0 + c.rcur, p.H - 1);
  return c;
}

// relu(a), relu(b) (or a, b) rounded to nearest-even bf16 and packed {lo = a, hi = b}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b, bool relu) {
  uint32_t d;
  if (relu)
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  else
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  return d;
}

// ------------------------------------------------------------------------------------------------ epilogues
// Eight epilogue warps form two groups of four (one warp per TMEM lane quarter q4); group g drains the output rows
// with T % 2 == g, where T counts the CTA's output rows in issue order and accumulator stage = T % NACC_.

// Hidden layers without a residual input: TMEM -> +bias -> ReLU -> bf16 -> 128B-swizzled staging box in shared memory -> one
// TMA store of 32 pixels x NOUT channels per warp and row (clipped at the image edge by the tensor map).  The warp alternates
// between two staging boxes, so a row is staged while the previous row's TMA store is still reading its box (the store's
// read latency otherwise serialises with the warp's work on every row).
// ELU: apply ELU instead of the optional ReLU (gradient-step DRUNet forward, its own instantiation).
template <int NOUT, int NACC_, bool ELU = false>
__device__ __forceinline__ void epilogue_hidden(const ConvParams& p, const CUtensorMap* tmap_out, uint8_t* stage,
                                                const float* bias_s, uint64_t* tfull, uint64_t* tempty,
                                                uint32_t tmem_base, int grp, int q4, int lane, uint32_t tempty_cluster = 0) {
  // tempty_cluster != 0 (CTA-pair kernel): the accumulator-free barriers live in the leader CTA, at this cluster address.
  // T: the CTA's running output-row counter (accumulator stage and mbarrier phase).
  uint32_t nrow = 0, T = 0;
  const uint32_t bias_sa = smem_u32(bias_s);
  const bool relu = p.relu != 0;
  if (lane == 0) tma_prefetch_desc(tmap_out);
  for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
    const ItemCoord c = decode_item(p, item);
    const int xw = c.x0 + q4 * 32;  // first pixel of this warp's 32-pixel box
    for (int y = c.y0; y < c.y0 + c.rcur; ++y, ++T) {
      if ((int)(T & 1) != grp) continue;
      const uint32_t acc = T % NACC_;
      mbar_wait(&tfull[acc], (T / NACC_) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * NOUT;
      uint32_t v[NOUT];
#pragma unroll
      for (int h = 0; h < NOUT / 32; ++h) tmem_ld_32x32b_x32(taddr + h * 32, *reinterpret_cast<uint32_t(*)[32]>(&v[h * 32]));
      tmem_ld_wait();
      tc_fence_before();
      // the staging box of the previous row must have been read by its TMA store before it is overwritten
      uint8_t* stage_cur = stage + (nrow & 1u) * (32 * NOUT * 2);
      const uint32_t stage_row = smem_u32(stage_cur) + lane * (NOUT * 2);
      ++nrow;
      if (lane == 0) {
        bulk_wait_group_read1();
        if (tempty_cluster)
          mbar_arrive_remote(tempty_cluster + acc * 8u);
        else
          mbar_arrive(&tempty[acc]);
      }
      __syncwarp();
      BiasPair bp = load_bias_pair(bias_sa, 0);
#pragma unroll
      for (int j = 0; j < NOUT / 8; ++j) {  // 16-byte chunk j = channels 8j..8j+7
        const float4 b0 = bp.b0, b1 = bp.b1;
        if (j + 1 < NOUT / 8) bp = load_bias_pair(bias_sa, j + 1);
        float f[8] = {__uint_as_float(v[8 * j + 0]) + b0.x, __uint_as_float(v[8 * j + 1]) + b0.y,
                      __uint_as_float(v[8 * j + 2]) + b0.z, __uint_as_float(v[8 * j + 3]) + b0.w,
                      __uint_as_float(v[8 * j + 4]) + b1.x, __uint_as_float(v[8 * j + 5]) + b1.y,
                      __uint_as_float(v[8 * j + 6]) + b1.z, __uint_as_float(v[8 * j + 7]) + b1.w};
        if (ELU) elu8(f);
        uint4 o;
        o.x = pack_bf16x2(f[0], f[1], relu);
        o.y = pack_bf16x2(f[2], f[3], relu);
        o.z = pack_bf16x2(f[4], f[5], relu);
        o.w = pack_bf16x2(f[6], f[7], relu);
        st_shared_v4(stage_row + ((uint32_t)(j ^ (lane & 7)) << 4), o);  // 128B swizzle: chunk ^= row & 7
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        if (xw < p.W) tma_store_4d(tmap_out, stage_cur, 0, xw, y, c.b);
        bulk_commit_group();  // also when nothing was stored: wait_group.read 1 counts one group per row
      }
    }
  }
  // Before the CTA exits its stores must have READ their staging boxes; their writes are complete and visible when the grid
  // completes, which is what a dependent launch's griddepcontrol.wait awaits.
  if (lane == 0) bulk_wait_group_read0();
}

// The same with the first residual tensor fetched by TMA (pair kernel, DRUNet's 64-channel residual blocks).  At 64 chains of
// 320 x 480 the layer moves 3.8 GB and is HBM-bound (580 us at the measured copy bandwidth against 540 us of MMAs); per-thread
// 16-byte loads of the residual reached only ~4 TB/s in total (950 us per layer, ncu).  Here lane 0 loads the warp's
// 32-pixel residual box of its NEXT row straight into the staging box that row will use (the two boxes alternate), one row
// ahead; the lanes then read-modify-write the box in shared memory and the TMA store ships it.  Box ownership: the load for
// row n + 1 into box b' is issued after cp.async.bulk.wait_group.read 1, i.e. once the store of row n - 1 has finished
// reading b'; generic writes precede the store by fence.proxy.async as before.
// GATE (gradient-step DRUNet backward, its own instantiation, no RES2): the box holds a stored ELU output t and the sum is
// multiplied by elu'(t) instead of added to it.
template <int NOUT, int NACC_, bool RES2, bool GATE = false>
__device__ __forceinline__ void epilogue_hidden_tmares(const ConvParams& p, const CUtensorMap* tmap_out,
                                                       const CUtensorMap* tmap_res, uint8_t* stage, uint64_t* rbar,
                                                       const float* bias_s, uint64_t* tfull, uint64_t* tempty,
                                                       uint32_t tmem_base, int grp, int q4, int lane, uint32_t tempty_cluster) {
  constexpr uint32_t BOX = 32 * NOUT * 2;
  struct Iter {
    int item, y, yend;
    uint32_t T;
    ItemCoord c;
    bool done;
  };
  auto step = [&](Iter& r) {
    ++r.y;
    ++r.T;
    if (r.y >= r.yend) {
      r.item += gridDim.x;
      if (r.item >= p.n_items) {
        r.done = true;
      } else {
        r.c = decode_item(p, r.item);
        r.y = r.c.y0;
        r.yend = r.c.y0 + r.c.rcur;
      }
    }
  };
  auto settle = [&](Iter& r) {
    while (!r.done && (int)(r.T & 1) != grp) step(r);
  };
  auto issue = [&](const Iter& r, uint32_t box) {  // lane 0: residual box of row r -> staging box `box`
    const int xw = r.c.x0 + q4 * 32;
    if (xw < p.W) {
      mbar_expect_tx(&rbar[box], BOX);
      tma_load_4d(stage + box * BOX, tmap_res, &rbar[box], 0, xw, r.y, r.c.b);
    }
  };
  const uint32_t bias_sa = smem_u32(bias_s);
  const bool relu = p.relu != 0;
  if (lane == 0) {
    tma_prefetch_desc(tmap_out);
    tma_prefetch_desc(tmap_res);
  }
  griddep_wait();  // the residual tensor was written by an earlier kernel
  Iter it;
  it.item = blockIdx.x;
  it.T = 0;
  it.done = it.item >= p.n_items;
  if (!it.done) {
    it.c = decode_item(p, it.item);
    it.y = it.c.y0;
    it.yend = it.c.y0 + it.c.rcur;
  }
  settle(it);
  uint32_t n = 0, cnt[2] = {0, 0};
  if (!it.done && lane == 0) issue(it, 0);
  while (!it.done) {
    Iter nxt = it;
    step(nxt);
    settle(nxt);
    const ItemCoord& c = it.c;
    const int y = it.y;
    const uint32_t T = it.T;
    const uint32_t box = n & 1u;
    const int xw = c.x0 + q4 * 32;
    const bool row_has = xw < p.W;
    const uint32_t acc = T % NACC_;
    // second residual tensor (U-Net skip, one layer per scale, its own instantiation): per-thread loads, issued before the
    // accumulator is awaited
    const bool has_res2 = RES2 && xw + lane < p.W;
    const size_t roff = (((size_t)c.b * p.H + y) * p.W + (xw + lane)) * NOUT;
    uint4 rr2[RES2 ? NOUT / 8 : 1];
    if (RES2 && has_res2) {  // 32 bytes per lane and access: full sectors (16-byte accesses cost this layer 1 266 instead of ~1 000 us)
#pragma unroll
      for (int j = 0; j < NOUT / 8; j += 2) ldg256(p.res2 + roff + 8 * j, rr2[RES2 ? j : 0], rr2[RES2 ? j + 1 : 0]);
    }
    // This row's residual box landed a row ago: all of it goes into registers in one batch, ahead of the wait for the
    // accumulator.  (Chunk by chunk inside the loop below -- load, add, pack, store to the same address -- every chunk paid a
    // shared-memory round trip behind the previous chunk's store, and the epilogue warps, not HBM or the tensor pipe, bound
    // the layer: 885 -> 738 us at 64 chains of 320 x 480, profiles/r02_drunet_conv64_full.txt.  With the second residual's 32
    // registers live as well the batch is two halves inside the loop: all three vectors at once spill, 1 750 us.)
    uint8_t* stage_cur = stage + box * BOX;
    const uint32_t stage_row = smem_u32(stage_cur) + lane * (NOUT * 2);
    constexpr int RB = RES2 ? NOUT / 16 : NOUT / 8;  // chunks per batch
    uint4 rr[RB];
    if (row_has) {
      mbar_wait(&rbar[box], cnt[box] & 1u);  // (pixels beyond W: zero fill)
      ++cnt[box];
      if (!RES2) {
#pragma unroll
        for (int j = 0; j < NOUT / 8; ++j) rr[j] = ld_shared_v4_nc(stage_row + ((uint32_t)(j ^ (lane & 7)) << 4));  // 128B swizzle
      }
    }
    mbar_wait(&tfull[acc], (T / NACC_) & 1);
    tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * NOUT;
    uint32_t v[NOUT];
#pragma unroll
    for (int h = 0; h < NOUT / 32; ++h) tmem_ld_32x32b_x32(taddr + h * 32, *reinterpret_cast<uint32_t(*)[32]>(&v[h * 32]));
    tmem_ld_wait();
    tc_fence_before();
    if (lane == 0) {
      if (tempty_cluster)
        mbar_arrive_remote(tempty_cluster + acc * 8u);
      else
        mbar_arrive(&tempty[acc]);
    }
    BiasPair bp = load_bias_pair(bias_sa, 0);
#pragma unroll
    for (int j = 0; j < NOUT / 8; ++j) {
      const float4 b0 = bp.b0, b1 = bp.b1;
      if (j + 1 < NOUT / 8) bp = load_bias_pair(bias_sa, j + 1);
      float f[8] = {__uint_as_float(v[8 * j + 0]) + b0.x, __uint_as_float(v[8 * j + 1]) + b0.y,
                    __uint_as_float(v[8 * j + 2]) + b0.z, __uint_as_float(v[8 * j + 3]) + b0.w,
                    __uint_as_float(v[8 * j + 4]) + b1.x, __uint_as_float(v[8 * j + 5]) + b1.y,
                    __uint_as_float(v[8 * j + 6]) + b1.z, __uint_as_float(v[8 * j + 7]) + b1.w};
      if (RES2 && row_has && j % RB == 0) {
#pragma unroll
        for (int i = 0; i < RB; ++i) rr[i] = ld_shared_v4_nc(stage_row + ((uint32_t)((j + i) ^ (lane & 7)) << 4));
      }
      if (GATE) {
        if (row_has) gate_bf16x8(f, rr[j % RB]);
      } else if (row_has) {
        add_bf16x8(f, rr[j % RB]);
      }
      if (RES2 && has_res2) add_bf16x8(f, rr2[RES2 ? j : 0]);
      uint4 o;
      o.x = pack_bf16x2(f[0], f[1], relu);
      o.y = pack_bf16x2(f[2], f[3], relu);
      o.z = pack_bf16x2(f[4], f[5], relu);
      o.w = pack_bf16x2(f[6], f[7], relu);
      st_shared_v4_nc(stage_row + ((uint32_t)(j ^ (lane & 7)) << 4), o);
    }
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
      if (row_has) tma_store_4d(tmap_out, stage_cur, 0, xw, y, c.b);
      bulk_commit_group();
      if (!nxt.done) {
        bulk_wait_group_read1();  // the store of the previous row no longer reads the other box
        issue(nxt, box ^ 1u);
      }
    }
    __syncwarp();  // no lane touches the other box before lane 0 has seen it released
    ++n;
    it = nxt;
  }
  if (lane == 0) bulk_wait_group_read0();  // see epilogue_hidden
}

// Last layer: the fused Langevin "post" step, fp32 NCHW (restoration_algorithms.py:238-262 / :115-135), optionally followed
// by the next iteration's "pre" on the fresh iterate.
// The layer is HBM-bound (128 B of activations in, ~70-140 B of fp32 state in and out per pixel) and its MMAs take only a few
// hundred cycles per row, so nothing hides a DRAM round trip behind them: the epilogue therefore walks ITS rows with a
// one-row-ahead register prefetch of everything it reads from global memory, and draws the row's noise before it waits
// for the accumulator.  C: image channels, 3 (colour) or 1 (grayscale: output column 0 of the accumulator; the element index
// within a chain is c H W + pixel either way, so channel 0 draws the same noise at C = 1 and C = 3).
struct PostRowIter {
  int item, y, yend;
  uint32_t T;
  ItemCoord c;
  bool done;
};
template <int C>
struct PostRowData {
  float bse[C], m1[C], m2[C], nmask[C], nobs[C];
};

template <int NOUT, int NACC_, int C>
__device__ __forceinline__ void epilogue_post(const ConvParams& p, const float* bias_s, uint64_t* tfull, uint64_t* tempty,
                                              uint32_t tmem_base, int grp, int q4, int lane) {
  griddep_wait();  // base / running moments were written by earlier kernels
  const size_t plane = (size_t)p.H * p.W;
  auto step = [&](PostRowIter& r) {
    ++r.y;
    ++r.T;
    if (r.y >= r.yend) {
      r.item += gridDim.x;
      if (r.item >= p.n_items) {
        r.done = true;
      } else {
        r.c = decode_item(p, r.item);
        r.y = r.c.y0;
        r.yend = r.c.y0 + r.c.rcur;
      }
    }
  };
  auto settle = [&](PostRowIter& r) {  // forward to the next row this epilogue group drains
    while (!r.done && (int)(r.T & 1) != grp) step(r);
  };
  auto fetch = [&](const PostRowIter& r, PostRowData<C>& d) {
    const int x = r.c.x0 + q4 * 32 + lane;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) d.bse[ch] = d.m1[ch] = d.m2[ch] = d.nmask[ch] = d.nobs[ch] = 0.f;
    if (r.done || x >= p.W) return;
    const size_t e0 = (size_t)r.y * p.W + x;
    const size_t idx0 = ((size_t)r.c.b * C) * plane + e0;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) {
      if (p.base) d.bse[ch] = p.base[idx0 + ch * plane];
      if (p.mean) {
        d.m1[ch] = p.mean[idx0 + ch * plane];
        d.m2[ch] = p.mean2[idx0 + ch * plane];
      }
    }
    if (p.nx_enable) {
      const size_t mi = ((size_t)(p.nx_mask_B > 1 ? r.c.b : 0) * C) * plane + e0;
      const size_t yi = ((size_t)(p.nx_y_B > 1 ? r.c.b : 0) * C) * plane + e0;
#pragma unroll
      for (int ch = 0; ch < C; ++ch) {
        d.nmask[ch] = p.nx_mask[mi + ch * plane];
        d.nobs[ch] = p.nx_y[yi + ch * plane];
      }
    }
  };

  PostRowIter it;
  it.item = blockIdx.x;
  it.T = 0;
  it.done = it.item >= p.n_items;
  if (!it.done) {
    it.c = decode_item(p, it.item);
    it.y = it.c.y0;
    it.yend = it.c.y0 + it.c.rcur;
  }
  settle(it);
  PostRowData<C> cur;
  fetch(it, cur);
  while (!it.done) {
    PostRowIter nxt = it;
    step(nxt);
    settle(nxt);
    PostRowData<C> nd;
    fetch(nxt, nd);  // in flight while this row is processed
    const ItemCoord& c = it.c;
    const int y = it.y;
    const uint32_t T = it.T;
    const int x = c.x0 + q4 * 32 + lane;
    const bool valid = x < p.W;
    const size_t idx0 = ((size_t)c.b * C) * plane + (size_t)y * p.W + x;
    float z[C];
#pragma unroll
    for (int ch = 0; ch < C; ++ch) z[ch] = 0.f;
    if (p.nx_enable) {
      if (p.nx.noise_mode == PSGLA_NOISE_PHILOX && (p.W & 3) == 0) {
        // Library stream: one Philox call serves four consecutive elements, and lanes 4k .. 4k+3 hold four consecutive
        // pixels (x0, the warp offset and W are multiples of 4).  Lane 4k + ch draws channel ch's quad, the four lanes
        // exchange components by shuffle: one Philox call per lane instead of three.  Grayscale: lane 4k draws the quad
        // of its four pixels and shares it.
        const int sub = lane & 3;
        float z4[4] = {0.f, 0.f, 0.f, 0.f};
        if (sub < C && x - sub < p.W)
          draw_quad(p.nx, c.b, (uint32_t)((size_t)sub * plane + (size_t)y * p.W + (size_t)(x - sub)), z4);
#pragma unroll
        for (int ch = 0; ch < C; ++ch) {
          const int src = (lane & ~3) + ch;
          const float t0 = __shfl_sync(0xffffffffu, z4[0], src), t1 = __shfl_sync(0xffffffffu, z4[1], src);
          const float t2 = __shfl_sync(0xffffffffu, z4[2], src), t3 = __shfl_sync(0xffffffffu, z4[3], src);
          z[ch] = sub == 0 ? t0 : (sub == 1 ? t1 : (sub == 2 ? t2 : t3));
        }
      } else if (valid) {
#pragma unroll
        for (int ch = 0; ch < C; ++ch) z[ch] = draw_at(p.nx, c.b, (uint32_t)((size_t)ch * plane + (size_t)y * p.W + x));
      }
    }
    const uint32_t acc = T % NACC_;
    mbar_wait(&tfull[acc], (T / NACC_) & 1);
    tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * NOUT;
    uint32_t v[16];
    tmem_ld_32x32b_x16(taddr, v);
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&tempty[acc]);
    if (valid) {
      float xnew[C];
#pragma unroll
      for (int ch = 0; ch < C; ++ch) {
        const size_t idx = idx0 + ch * plane;
        const float r = __uint_as_float(v[ch]) + bias_s[ch];
        const float xn = p.base ? fmaf(p.gain, r, p.base_scale * cur.bse[ch]) : r;
        xnew[ch] = xn;
        p.x_out[idx] = xn;
        if (p.sample) p.sample[idx] = xn;
        if (p.mean) {
          // three rounded fp32 operations each, as the reference's eager ops (restoration_algorithms.py:257-258)
          p.mean[idx] = __fadd_rn(__fmul_rn(p.w_old, cur.m1[ch]), __fmul_rn(p.w_new, xn));
          p.mean2[idx] = __fadd_rn(__fmul_rn(p.w_old, cur.m2[ch]), __fmul_rn(p.w_new, __fmul_rn(xn, xn)));
        }
      }
      if (p.nx_enable) {
        // the next iteration's Langevin "pre" on the fresh iterate: same arithmetic and the same noise element as
        // pre_inpaint_kernel (img_elementwise.cu), so fused and unfused runs agree bit for bit
        float din[C];
#pragma unroll
        for (int ch = 0; ch < C; ++ch) {
          const float bv = langevin_base(p.nx, xnew[ch], cur.nmask[ch] * (xnew[ch] - cur.nobs[ch]), z[ch]);
          p.nx_base[idx0 + ch * plane] = bv;
          din[ch] = (p.nx.alg == PSGLA_ALG_PNPULA) ? xnew[ch] : bv;
        }
        store_nhwc16(p.nx_den_in + (((size_t)c.b * plane) + (size_t)y * p.W + x) * 16, din[0], C > 1 ? din[1 % C] : 0.f,
                     C > 2 ? din[2 % C] : 0.f, p.nx.den_in_c3);
      }
    }
    it = nxt;
    cur = nd;
  }
}

// ------------------------------------------------------------------------------------------------ TS kernel (A from TMEM)
// Measured on B200 (psgla_selftest_mma_rate): an M128 x N64 x K16 bf16 MMA takes 72 cycles with both operands in shared
// memory (the 4 KB A fetch is exposed) but 41 cycles with A in tensor memory (floor 32).  For the 64-input-channel layers
// four "loader" warps therefore copy every input row from the TMA ring into TMEM three times, shifted by dx = 0, 1, 2
// pixels (TMEM lanes are pixels and cannot be shifted by the MMA), and the MMAs read A from there:
//   TMEM columns [0, NACC_TS * NOUT)            accumulators (one stage per epilogue group)
//                [128 + s*96 + dx*32 + k*8 ...)  A ring: slot s = input row mod 4, shift dx, K-step k (8 columns = 16 bf16)
// Warps: 0 TMA producer, 1 MMA issuer, 2-5 loaders (TMEM lane quarter = warp & 3), 6-13 epilogue (two groups).
constexpr int TS_NA = 4;       // input rows resident in TMEM
constexpr int TS_NACC = 2;
constexpr int TS_A_COL0 = 128;
constexpr int TS_THREADS = 64 + 128 + 32 * EPI_WARPS;

// The single-CTA TS kernel, i.e. the last layer: 64 input channels, 16 (3 or 1 padded) output channels, fused Langevin epilogue
template <int NOUT>
struct ConvTsCfg {
  static_assert(NOUT == 16, "ring depth and shared-memory plan are sized for the last layer");
  static constexpr int ROW_BYTES = 128;
  static constexpr int BOX_BYTES = BOX_W * ROW_BYTES;
  static constexpr int SLOT_BYTES = round_up_c(BOX_BYTES, 1024);
  static constexpr int TAP_BYTES = NOUT * ROW_BYTES;
  static constexpr int W_BYTES = 9 * TAP_BYTES;
  static constexpr int OFF_RING = round_up_c(W_BYTES, 1024);
  // staging ring depth: the last layer (N = 16: 9 x 4 MMAs of ~9 cycles per row, no output staging) outruns a 4-slot
  // ring by far and has the shared memory for a deep one
  static constexpr int NSTAGE = 10;
  static constexpr int OFF_BIAS = OFF_RING + NSTAGE * SLOT_BYTES;
  static constexpr int OFF_BAR = OFF_BIAS + 256;
  static constexpr int BAR_BYTES = 512;
  static_assert((2 * NSTAGE + 2 * TS_NA + 2 * TS_NACC + 3) * 8 + 4 <= BAR_BYTES, "barrier block overflows");
  static constexpr int SMEM_BYTES = OFF_BAR + BAR_BYTES + 1024;
  static_assert(TS_NACC * NOUT <= TS_A_COL0 && TS_A_COL0 + TS_NA * 96 <= 512, "TMEM plan does not fit 512 columns");
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of one CTA");
};

// host helper defined in conv_tc.cu
int get_act_tensor_map(CUtensorMap* map, const void* ptr, int B, int H, int W, int C, int box_w);
// conv_fused2.cu: two hidden layers (both conv + bias + ReLU) in one launch when the shape is a single wave of CTA pairs
// (few chains); *applicable = 0 and nothing launched otherwise
int conv64_hidden_fused2(const void* in, void* out, const uint8_t* w1, const float* b1, const uint8_t* w2, const float* b2, int B,
                         int H, int W, int* applicable, cudaStream_t st);

}  // namespace psgla
