// Two consecutive 64 -> 64 channel 3x3 layers (conv + bias + ReLU, twice) in ONE launch, for runs of few chains: the
// reference's own run shape is ONE chain of one 256 x 256 image (sampling_images.py:351, restoration_algorithms.py:238), and
// there a hidden layer of DnCNN is ~2.4 us of MMAs inside ~9 us of latency (first TMA loads, three rows through the loader
// warps before the first MMA, the last row's epilogue, its store, the kernel boundary).  Fusing two layers pays that latency
// once per two layers at the price of recomputing a one-row halo of the intermediate layer.
//
// Geometry: as conv3x3_ts2_kernel (conv_tc.cu) -- a CTA pair (cta_group::2, M = 256) on the two 128-pixel strips of one block of
// R output rows, A operand through tensor memory, each layer's weights split 32 / 32 output channels between the two CTAs --
// but ONE work item per pair (grid = items, a single wave) and two phases:
//   phase 1: layer l for rows y0 - 1 .. y0 + R (clipped to the image), epilogue -> bf16 -> the MID ring in shared memory, in
//            the very layout a TMA row box has (130 pixels x 128 B, 16-byte chunk j of box row r at j ^ (r & 7)); the one
//            pixel a strip needs from its neighbour (box row 0 / 129) is written into the PEER's ring by st.async
//            (shared::cluster, completes transaction bytes on the peer's "row ready" mbarrier, so no fence is needed);
//   phase 2: layer l + 1 for rows y0 .. y0 + R - 1, the loader warps reading the mid ring instead of the TMA ring; the epilogue
//            stores straight from registers (one pixel = 128 contiguous bytes per lane).
// The intermediate activations are rounded to bf16 exactly as when they travel through global memory, so the result is
// bit-identical to two conv3x3_ts2_kernel launches (tests/test_image_gpu.py::test_fused_layer_pairs_equal_single_layers).
// Limits: W <= 256 (the pair holds whole rows, so every halo pixel is on chip) and a single wave of pairs; everything else
// keeps the per-layer kernels.  PSGLA_CONV_FUSE2=0 disables the path: bench.py times the single-chain iteration with one
// hidden layer per launch beside the fused one, and tests compare the two bit for bit.
#include <cuda_bf16.h>

#include <algorithm>
#include <atomic>
#include <utility>
#include <vector>

#include "conv_tc.cuh"

namespace psgla {

using namespace sm100;

constexpr int F2_NSTAGE = 3;  // TMA staging slots (the loaders empty a slot within a fraction of a row's MMA time)
constexpr int F2_MAXR = 4;
constexpr int F2_MID = F2_MAXR + 2;  // intermediate rows kept on chip

struct ConvF2Cfg {
  static constexpr int ROW_BYTES = 128;
  static constexpr int BOX_BYTES = BOX_W * ROW_BYTES;
  static constexpr int SLOT_BYTES = round_up_c(BOX_BYTES, 1024);
  static constexpr int TAP_BYTES_FULL = 64 * ROW_BYTES;
  static constexpr int TAP_BYTES = 32 * ROW_BYTES;  // this CTA's half of the output channels
  static constexpr int W_BYTES = 9 * TAP_BYTES;     // one layer
  static constexpr int OFF_RING = 2 * W_BYTES;
  static constexpr int OFF_MID = OFF_RING + F2_NSTAGE * SLOT_BYTES;
  static constexpr int MID_SLOT = BOX_BYTES;  // read and written by ld / st.shared only: no 1 KB alignment needed
  static constexpr int OFF_BIAS = OFF_MID + F2_MID * MID_SLOT;
  static constexpr int OFF_BAR = OFF_BIAS + 512;
  static constexpr int BAR_BYTES = 512;
  static constexpr int SMEM_BYTES = OFF_BAR + BAR_BYTES + 1024;
  static_assert(OFF_RING % 1024 == 0 && W_BYTES % 1024 == 0, "UMMA / TMA operands need 1 KB aligned bases");
  static_assert((2 * F2_NSTAGE + 2 * TS_NA + 2 * TS_NACC + 5 + F2_MID) * 8 + 4 <= BAR_BYTES, "barrier block overflows");
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared memory of one CTA");
};

struct F2Params {
  const uint8_t* weights2;  // second layer: 9 taps, swizzled, all 64 output channels (as ConvParams::weights)
  const float* bias2;
  __nv_bfloat16* out;  // bf16 NHWC [B][H][W][64]
};

// 16 bytes into the shared memory of another CTA of the cluster; the bytes count as a transaction on that CTA's mbarrier
__device__ __forceinline__ void st_async_v4(uint32_t cluster_addr, const uint4& v, uint32_t mbar_cluster_addr) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(cluster_addr),
               "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(mbar_cluster_addr)
               : "memory");
}

__global__ void __launch_bounds__(TS_THREADS, 1)
conv3x3_fused2_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_w1,
                      const __grid_constant__ CUtensorMap tmap_w2, const ConvParams p, const F2Params f) {
  using Cfg = ConvF2Cfg;
  constexpr int NOUT = 64;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_w = smem;  // layer l at 0, layer l + 1 at W_BYTES
  uint8_t* ring = smem + Cfg::OFF_RING;
  uint8_t* mid = smem + Cfg::OFF_MID;
  float* bias_s = reinterpret_cast<float*>(smem + Cfg::OFF_BIAS);    // [0, 64) layer l, [64, 128) layer l + 1
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);  // local: TMA landed an input row
  uint64_t* empty = full + F2_NSTAGE;                                 // local: loaders have copied it out
  uint64_t* afull = empty + F2_NSTAGE;                                // leader: both CTAs' copies of the row are in TMEM
  uint64_t* aempty = afull + TS_NA;                                   // both (multicast): MMAs reading them completed
  uint64_t* tfull = aempty + TS_NA;                                   // both (multicast): accumulator stage complete
  uint64_t* tempty = tfull + TS_NACC;                                 // leader: both CTAs' epilogues drained the stage
  uint64_t* wbar = tempty + TS_NACC;                                  // local: this CTA's halves of both layers' weights landed
  uint64_t* wready = wbar + 1;                                        // leader: the peer's landed
  uint64_t* done = wready + 1;                                        // both (multicast): every MMA of the launch completed
  uint64_t* wbar2 = done + 1;                                         // local: the second layer's weights landed
  uint64_t* wready2 = wbar2 + 1;                                      // leader: the peer's second layer landed
  uint64_t* mfull = wready2 + 1;                                         // local: an intermediate row is complete (4 warps + 128 B from the peer)
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(mfull + F2_MID);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  griddep_launch_dependents();

  // the pair's work item: output rows [y0, y0 + rcur), intermediate rows [m_lo, m_hi], input rows [i_lo, i_hi]
  const ItemCoord c = decode_item(p, blockIdx.x);
  const int m_lo = c.ylo, m_hi = c.yhi;
  const int i_lo = max(m_lo - 1, 0), i_hi = min(m_hi + 1, p.H - 1);
  const int n_in = i_hi - i_lo + 1, n_mid = m_hi - m_lo + 1;

  // The prologue sits on every launch's critical path (one short item per CTA), so whatever can start before the cluster
  // barrier does: the producer initialises its own "row landed" barriers, waits for the previous grid and issues the first
  // rows' loads; warp 1's lane 0 does the same for the weights; the other barriers are initialised one per thread.
  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&tmap_w1);
      tma_prefetch_desc(&tmap);
      for (int i = 0; i < F2_NSTAGE; ++i) mbar_init(&full[i], 1);
      mbar_init(wbar, 1);
      fence_barrier_init();
      fence_proxy_async();
      // The weights (this CTA's 32 output channels of each layer) are constant across launches: no dependency wait.  The SM's
      // TMA queue is served in order and a bulk copy takes ~100 cycles to issue, so: the first layer's weights from here, while
      // the previous grid drains, ahead of the input rows (the first MMA needs both); the second layer's behind the rows
      // (warp 1, after the cluster barrier).
      mbar_expect_tx(wbar, Cfg::W_BYTES);
      tma_load_3d(smem_w, &tmap_w1, wbar, 0, (int)rank * 32, 0);  // one box: 9 taps x this CTA's 32 rows x 128 B, as they lie
      griddep_wait();
      for (int q = 0; q < min(n_in, F2_NSTAGE); ++q) {
        mbar_expect_tx(&full[q], Cfg::BOX_BYTES);
        tma_load_4d(ring + q * Cfg::SLOT_BYTES, &tmap, &full[q], 0, c.x0 - 1, i_lo + q, c.b);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    tmem_alloc2(tmem_ptr_s, 512);
    tmem_relinquish2();
    if (lane == 0) {
      tma_prefetch_desc(&tmap_w2);
      mbar_init(wbar2, 1);
      mbar_init(wready, 1);
      mbar_init(wready2, 1);
      mbar_init(done, 1);
      fence_barrier_init();
      fence_proxy_async();
    }
    __syncwarp();
  } else {
    // empty (4: the loader warps), afull (8: the loader warps of both CTAs), aempty, tfull (1), tempty (8), mfull (4: one
    // epilogue group, + 128 B from the peer)
    constexpr int N0 = F2_NSTAGE, N1 = N0 + TS_NA, N2 = N1 + TS_NA, N3 = N2 + TS_NACC, N4 = N3 + TS_NACC, N5 = N4 + F2_MID;
    const int i = threadIdx.x - 64;
    if (i < N5) {
      uint64_t* bar = i < N0 ? &empty[i] : i < N1 ? &afull[i - N0] : i < N2 ? &aempty[i - N1] : i < N3 ? &tfull[i - N2]
                      : i < N4 ? &tempty[i - N3] : &mfull[i - N4];
      const uint32_t count = i < N0 ? 4u : i < N1 ? 8u : i < N3 ? 1u : i < N4 ? 8u : 4u;
      mbar_init(bar, count);
      fence_barrier_init();
    }
  }
  tc_fence_before();
  __syncthreads();        // this CTA: barriers, the TMEM base address
  cluster_sync_relaxed();  // the pair: both CTAs' barriers exist before any remote arrive / store / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t afull_c = mapa_shared(smem_u32(afull), 0);
  const uint32_t tempty_c = mapa_shared(smem_u32(tempty), 0);

  // One loader pass: row q of the sequence (input rows, then intermediate rows) from its ring into TMEM slot q % 4, three times,
  // shifted by dx = 0, 1, 2 pixels; run by four warps that cover the four TMEM lane quarters.  A pass is ~500 cycles of
  // shared-memory reads and TMEM stores plus four mbarrier operations of ~90 cycles, and passes of one warp set are serial; so
  // where rows wait in line on the critical path -- the first three rows of the launch, the rows the second layer starts
  // with -- the epilogue groups, idle at those moments, each take one (helper_row) and the passes run side by side.
  auto loader_pass = [&](int q, int q4, int lane_) {
    const int m = q4 * 32 + lane_;
    const uint32_t lane_taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + TS_A_COL0;
    const uint32_t as = (uint32_t)q % TS_NA;
    uint32_t tile;
    uint32_t slot = 0;
    if (q < n_in) {
      slot = (uint32_t)q % F2_NSTAGE;
      mbar_wait(&full[slot], ((uint32_t)q / F2_NSTAGE) & 1);
      tile = smem_u32(ring) + slot * Cfg::SLOT_BYTES;
    } else {
      mbar_wait(&mfull[q - n_in], 0);
      tile = smem_u32(mid) + (uint32_t)(q - n_in) * Cfg::MID_SLOT;
    }
    mbar_wait(&aempty[as], (((uint32_t)q / TS_NA) & 1) ^ 1);
    tc_fence_after();
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
      uint32_t v[32];
      ld_swizzled_row128(tile, m + dx, v);
      tmem_st_32x32b_x32(lane_taddr + as * 96u + dx * 32u, v);
    }
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane_ == 0) {
      if (q < n_in) mbar_arrive(&empty[slot]);
      mbar_arrive_remote(afull_c + as * 8u);
    }
  };
  // rows taken by an epilogue group: input rows 1 and 2 (groups 0 and 1, before their first accumulator), and the third
  // intermediate row (the group that is NOT draining the last intermediate row's accumulator; it also owns the second layer's
  // first output row, which cannot start before that pass anyway)
  auto helper_row = [&](int q) { return ((q == 1 || q == 2) && q < n_in) || (n_mid > 2 && q == n_in + 2); };

  if (warp == 0) {
    if (lane == 0) {
      // ---------------------------------------------------------------- TMA producer: the rows beyond the first three
      for (int q = F2_NSTAGE; q < n_in; ++q) {
        const uint32_t slot = (uint32_t)q % F2_NSTAGE;
        mbar_wait(&empty[slot], (((uint32_t)q / F2_NSTAGE) & 1) ^ 1);
        mbar_expect_tx(&full[slot], Cfg::BOX_BYTES);
        tma_load_4d(ring + slot * Cfg::SLOT_BYTES, &tmap, &full[slot], 0, c.x0 - 1, i_lo + q, c.b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      mbar_expect_tx(wbar2, Cfg::W_BYTES);
      tma_load_3d(smem_w + Cfg::W_BYTES, &tmap_w2, wbar2, 0, (int)rank * 32, 0);
      if (rank != 0) {  // tell the leader (behind the cluster barrier: its barrier exists), once per layer
        mbar_wait(wbar, 0);
        mbar_arrive_cluster(mapa_shared(smem_u32(wready), 0));
        mbar_wait(wbar2, 0);
        mbar_arrive_cluster(mapa_shared(smem_u32(wready2), 0));
      }
    }
    __syncwarp();
    if (rank == 0) {
      // ---------------------------------------------------------------- MMA issuer of the pair
      // Rows enter tensor memory in ONE sequence q = 0 .. n_in + n_mid - 1 (input rows, then intermediate rows), slot q % 4.
      constexpr uint32_t idesc = make_idesc_bf16(2 * TILE_M, NOUT);
      constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (LAYOUT_SW128 << 29);
      const uint32_t w_lo = (smem_u32(smem_w) >> 4) | 0x10000u;
      mbar_wait(wbar, 0);
      mbar_wait_cluster(wready, 0);
      tc_fence_after();
      // ONE thread runs the whole issue loop, barrier waits included.  The tensor pipe's queue is shallow: whatever the issuing
      // thread executes between two MMAs beyond a few dozen cycles is a bubble in the pipe (measured with clock64 stamps, commit
      // e803185: one warp-uniform wait / elect / syncwarp boundary per dy group cost 180 cycles per 384 cycles of MMAs), so the
      // loop carries nothing but try_waits that pass at once in steady state, address adds and the MMAs.
      if (elect_one()) {
        uint32_t T = 0;
        int waited = 0;
#pragma unroll 1
        for (int ph = 0; ph < 2; ++ph) {
          // phase ph: output rows [o_lo, o_hi] of the phase from source rows [s_lo, s_hi], which sit at sequence q0 + (row - s_lo)
          const int o_lo = ph ? c.y0 : m_lo, o_hi = ph ? c.y0 + c.rcur - 1 : m_hi;
          const int s_lo = ph ? m_lo : i_lo;
          const int q0 = ph ? n_in : 0;
          const uint32_t wl = w_lo + (uint32_t)(ph * (Cfg::W_BYTES >> 4));
          if (ph) {  // the second layer's weights: both CTAs' halves (they landed long ago)
            mbar_wait_spin(wbar2, 0);
            mbar_wait_cluster(wready2, 0);
          }
#pragma unroll 1
          for (int y = o_lo; y <= o_hi; ++y, ++T) {
            const uint32_t acc = T % TS_NACC;
            mbar_wait_spin(&tempty[acc], ((T / TS_NACC) & 1) ^ 1);
            const uint32_t d_tmem = tmem_base + acc * NOUT;
            uint32_t accumulate = 0;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
              const int yy = y + dy - 1;
              if (yy < 0 || yy >= p.H) continue;  // the layer's zero padding above / below the image
              // a source row is awaited right before the first 12 MMAs that read it: at the start of a phase the MMAs of the
              // first rows run while the loader warps are still copying the next one
              const int q = q0 + yy - s_lo;
              if (q == waited) {
                mbar_wait_spin(&afull[(uint32_t)q % TS_NA], ((uint32_t)q / TS_NA) & 1);
                ++waited;
              }
              tc_fence_after();
              const uint32_t a_t = tmem_base + TS_A_COL0 + ((uint32_t)q % TS_NA) * 96u;
#pragma unroll
              for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t bl = wl + (uint32_t)(((dy * 3 + dx) * Cfg::TAP_BYTES + k * 32) >> 4);
                  umma_bf16_ts2(d_tmem, a_t + dx * 32 + k * 8, ((uint64_t)DESC_HI << 32) | bl, idesc, accumulate | (uint32_t)(dx | k));
                }
              }
              accumulate = 1;
              // source row y - 1 is dead once these 12 MMAs retire; after the phase's last output row so are the others
              if ((dy == 0 && y - 1 >= s_lo) || y == o_hi) umma_commit2(&aempty[(uint32_t)q % TS_NA], 3);
            }
            umma_commit2(&tfull[acc], 3);
          }
        }
        umma_commit2(done, 3);
      }
      __syncwarp();
    }
    mbar_wait(done, 0);
    // both CTAs: no MMA still reads this CTA's shared / tensor memory, no commit is still in flight
  } else if (warp < 6) {
    // ---------------------------------------------------------------- loaders: TMA ring / mid ring -> registers -> TMEM
    const int n_rows = n_in + n_mid;
    for (int q = 0; q < n_rows; ++q)
      if (!helper_row(q)) loader_pass(q, warp & 3, lane);
  } else {
    // ---------------------------------------------------------------- epilogue: 2 groups x 4 warps
    const int ew = warp - 6;
    const int grp = ew >> 2, q4 = warp & 3;
    {
      const int i = ew * 32 + lane;
      if (i < 2 * NOUT) bias_s[i] = i < NOUT ? p.bias[i] : f.bias2[i - NOUT];
      asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");  // the eight epilogue warps only
    }
    if (1 + grp < n_in) loader_pass(1 + grp, q4, lane);
    // phase 1: layer l -> the mid ring (this CTA's 128 pixels, plus its edge pixel into the peer's ring)
    {
      const int mpx = q4 * 32 + lane;       // pixel of the strip
      const uint32_t r = (uint32_t)mpx + 1u;  // its box row
      const bool inside = c.x0 + mpx < p.W;
      const bool relu = p.relu != 0;
      const float4* bias4 = reinterpret_cast<const float4*>(bias_s);
      const uint32_t mid_addr = smem_u32(mid);
      const uint32_t peer = rank ^ 1u;
      const uint32_t peer_mid = mapa_shared(mid_addr, peer);
      const uint32_t peer_mfull = mapa_shared(smem_u32(mfull), peer);
      const bool edge = rank == 0 ? (mpx == TILE_M - 1) : (mpx == 0);
      // the intermediate layer's zero padding left of strip 0 (box row 0) / right of strip 1 (box row 129): written by the lane
      // whose own pixel is next to it, ahead of the same "row ready" arrive
      const bool pad = rank == 0 ? (mpx == 0) : (mpx == TILE_M - 1);
      const uint32_t r_pad = rank == 0 ? 0u : (uint32_t)(BOX_W - 1);
      const uint32_t r_peer = rank == 0 ? 0u : (uint32_t)(BOX_W - 1);  // where the peer's box holds that pixel
      for (int t = 0; t < n_mid; ++t) {
        if ((t & 1) != grp) continue;
        const uint32_t acc = (uint32_t)t % TS_NACC;
        mbar_wait(&tfull[acc], ((uint32_t)t / TS_NACC) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * NOUT;
        uint32_t v[NOUT];
#pragma unroll
        for (int h = 0; h < NOUT / 32; ++h) tmem_ld_32x32b_x32(taddr + h * 32, *reinterpret_cast<uint32_t(*)[32]>(&v[h * 32]));
        tmem_ld_wait();
        tc_fence_before();
        if (lane == 0) mbar_arrive_remote(tempty_c + acc * 8u);
        const uint32_t row_addr = mid_addr + (uint32_t)t * Cfg::MID_SLOT + r * 128u;
        const uint32_t peer_row = peer_mid + (uint32_t)t * Cfg::MID_SLOT + r_peer * 128u;
#pragma unroll
        for (int j = 0; j < NOUT / 8; ++j) {
          const float4 b0 = bias4[2 * j], b1 = bias4[2 * j + 1];
          uint4 o;
          o.x = pack_bf16x2(__uint_as_float(v[8 * j + 0]) + b0.x, __uint_as_float(v[8 * j + 1]) + b0.y, relu);
          o.y = pack_bf16x2(__uint_as_float(v[8 * j + 2]) + b0.z, __uint_as_float(v[8 * j + 3]) + b0.w, relu);
          o.z = pack_bf16x2(__uint_as_float(v[8 * j + 4]) + b1.x, __uint_as_float(v[8 * j + 5]) + b1.y, relu);
          o.w = pack_bf16x2(__uint_as_float(v[8 * j + 6]) + b1.z, __uint_as_float(v[8 * j + 7]) + b1.w, relu);
          if (!inside) o = make_uint4(0u, 0u, 0u, 0u);  // beyond the image: the next layer's zero padding
          st_shared_v4(row_addr + ((uint32_t)(j ^ (int)(r & 7u)) << 4), o);
          if (edge) st_async_v4(peer_row + ((uint32_t)(j ^ (int)(r_peer & 7u)) << 4), o, peer_mfull + (uint32_t)t * 8u);
          if (pad) st_shared_v4(mid_addr + (uint32_t)t * Cfg::MID_SLOT + r_pad * 128u + ((uint32_t)j << 4), make_uint4(0u, 0u, 0u, 0u));
        }
        __syncwarp();
        if (lane == 0) {
          if (q4 == 0)
            mbar_expect_tx(&mfull[t], 128);  // arrive + the peer's edge pixel
          else
            mbar_arrive(&mfull[t]);
        }
      }
    }
    if (n_mid > 2 && grp == (n_mid & 1)) loader_pass(n_in + 2, q4, lane);
    // phase 2: layer l + 1 -> registers -> global memory, one pixel (128 contiguous bytes) per lane.  No staging box and no TMA
    // store here: with one item per CTA nothing overlaps the store's shared-memory round trip, and plain stores let the CTA
    // retire as soon as they are issued (they are complete when the grid is, which is what the next launch waits for).
    {
      const int x = c.x0 + q4 * 32 + lane;
      const bool relu = p.relu != 0;
      const float4* bias4 = reinterpret_cast<const float4*>(bias_s + NOUT);
      uint32_t T = (uint32_t)n_mid;  // accumulator stages and phases continue after the intermediate rows
      for (int y = c.y0; y < c.y0 + c.rcur; ++y, ++T) {
        if ((int)(T & 1) != grp) continue;
        const uint32_t acc = T % TS_NACC;
        mbar_wait(&tfull[acc], (T / TS_NACC) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + acc * NOUT;
        uint32_t v[NOUT];
#pragma unroll
        for (int h = 0; h < NOUT / 32; ++h) tmem_ld_32x32b_x32(taddr + h * 32, *reinterpret_cast<uint32_t(*)[32]>(&v[h * 32]));
        tmem_ld_wait();
        tc_fence_before();
        if (lane == 0) mbar_arrive_remote(tempty_c + acc * 8u);
        __nv_bfloat16* dst = f.out + (((size_t)c.b * p.H + y) * p.W + x) * NOUT;
#pragma unroll
        for (int j = 0; j < NOUT / 8; j += 2) {
          uint4 o[2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float4 b0 = bias4[2 * (j + h)], b1 = bias4[2 * (j + h) + 1];
            const int e = 8 * (j + h);
            o[h].x = pack_bf16x2(__uint_as_float(v[e + 0]) + b0.x, __uint_as_float(v[e + 1]) + b0.y, relu);
            o[h].y = pack_bf16x2(__uint_as_float(v[e + 2]) + b0.z, __uint_as_float(v[e + 3]) + b0.w, relu);
            o[h].z = pack_bf16x2(__uint_as_float(v[e + 4]) + b1.x, __uint_as_float(v[e + 5]) + b1.y, relu);
            o[h].w = pack_bf16x2(__uint_as_float(v[e + 6]) + b1.z, __uint_as_float(v[e + 7]) + b1.w, relu);
          }
          if (x < p.W) stg256(dst + 8 * j, o[0], o[1]);
        }
      }
    }
  }
  tc_fence_before();
  cluster_sync_relaxed();
  // neither CTA may exit (or free tensor memory) while its partner can still signal, read or write it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, 512);
  }
}

// A layer's packed weights [9 taps][64 output channels][64 input channels] bf16 (pre-swizzled rows of 128 B) as a 3-D tensor,
// box = 9 taps x 32 rows x 128 B without swizzle: one TMA instruction lands a CTA's half of the layer in shared memory as the
// bytes lie (nine 4 KB bulk copies take ~900 cycles to issue and, measured, ~2 000 cycles longer to complete).
static int get_weight_tensor_map(CUtensorMap* map, const void* ptr) {
  static thread_local std::vector<std::pair<const void*, CUtensorMap>> cache;
  for (const auto& e : cache)
    if (e.first == ptr) {
      *map = e.second;
      return PSGLA_OK;
    }
  PFN_tensorMapEncodeTiled enc = get_tensor_map_encoder();
  if (!enc) return set_error(PSGLA_E_NODEVICE, "cuTensorMapEncodeTiled driver entry point not available");
  const cuuint64_t dims[3] = {64, 64, 9};
  const cuuint64_t strides[2] = {128, 64 * 128};
  const cuuint32_t box[3] = {64, 32, 9};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(PSGLA_E_BADARG, "cuTensorMapEncodeTiled (weights) failed with CUresult %d", (int)r);
  if (cache.size() >= 128) cache.erase(cache.begin());
  cache.emplace_back(ptr, *map);
  return PSGLA_OK;
}

// R for which the fused kernel runs (0 = not applicable): the smallest block height whose pairs form a single wave.
static int fused2_rows(int B, int H, int W, int max_clusters) {
  if (W > 2 * TILE_M) return 0;
  const int cands[] = {1, 2, 4};
  for (int R : cands)
    if ((long long)B * ((H + R - 1) / R) <= max_clusters) return R;
  return 0;
}

static int fused2_clusters(int* out) {
  static std::atomic<int> max_clusters_dev[kMaxDevices];  // per device: co-resident CTA pairs; 0 = not asked yet
  std::atomic<int>& slot = max_clusters_dev[current_device() % kMaxDevices];
  int mc = slot.load(std::memory_order_acquire);
  if (!mc) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(conv3x3_fused2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvF2Cfg::SMEM_BYTES));
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(TS_THREADS);
    cfg.dynamicSmemBytes = ConvF2Cfg::SMEM_BYTES;
    cfg.gridDim = dim3((unsigned)(num_sms() & ~1));
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    PSGLA_CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, conv3x3_fused2_kernel, &cfg));
    mc = n > 0 ? std::min(n, num_sms() / 2) : num_sms() / 2;
    slot.store(mc, std::memory_order_release);
  }
  *out = mc;
  return PSGLA_OK;
}

// PSGLA_CONV_FUSE2=0: per-layer launches everywhere (read per call: bench.py and tests switch it inside one process)
static bool fused2_enabled() {
  const char* e = getenv("PSGLA_CONV_FUSE2");
  return !(e && e[0] == '0');
}

// *applicable = 0 and nothing launched when the shape does not qualify; otherwise layers (w1, b1) and (w2, b2), both with ReLU,
// are applied to `in` and the result lands in `out` (which must not alias `in`).
int conv64_hidden_fused2(const void* in, void* out, const uint8_t* w1, const float* b1, const uint8_t* w2, const float* b2, int B,
                         int H, int W, int* applicable, cudaStream_t st) {
  *applicable = 0;
  if (!fused2_enabled()) return PSGLA_OK;
  int max_clusters = 0;
  int rc = fused2_clusters(&max_clusters);
  if (rc) return rc;
  const int R = fused2_rows(B, H, W, max_clusters);
  if (!R) return PSGLA_OK;
  ConvParams p{};
  p.B = B, p.H = H, p.W = W;
  p.weights = w1;
  p.bias = b1;
  p.relu = 1;
  p.R = R;
  p.strips = 2;
  p.row_blocks = (H + R - 1) / R;
  p.n_items = B * 2 * p.row_blocks;
  const F2Params f{w2, b2, (__nv_bfloat16*)out};
  CUtensorMap map, map_w1, map_w2;
  rc = get_act_tensor_map(&map, in, B, H, W, 64, BOX_W);
  if (rc) return rc;
  rc = get_weight_tensor_map(&map_w1, w1);
  if (rc) return rc;
  rc = get_weight_tensor_map(&map_w2, w2);
  if (rc) return rc;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)p.n_items);
  cfg.blockDim = dim3(TS_THREADS);
  cfg.dynamicSmemBytes = ConvF2Cfg::SMEM_BYTES;
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
  PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv3x3_fused2_kernel, map, map_w1, map_w2, p, f));
  *applicable = 1;
  return PSGLA_OK;
}

}  // namespace psgla
