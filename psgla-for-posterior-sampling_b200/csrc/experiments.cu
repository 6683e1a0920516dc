// Development probes of the tcgen05 path, kept OUT of the production kernels' files: the UMMA descriptor / TMEM self-tests
// the gpu tests run (tests/test_image_gpu.py::test_umma_descriptor_selftest), the CTA-pair (cta_group::2) self-test, and
// the MMA issue-rate probes whose measurements DESIGN.md section 4 quotes (profiles/r01b_mma_rate.txt,
// profiles/r01e_mma_rate.txt).  Nothing here is on a sampler's path.
#include <atomic>

#include "common.cuh"
#include "sm100.cuh"

namespace psgla {
using namespace sm100;
}  // namespace psgla

using namespace psgla;

// ------------------------------------------------------------------------------------------------ descriptor self-test
namespace psgla {
__global__ void __launch_bounds__(128, 1)
selftest_umma_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                     float* __restrict__ d, int row_shift, int mode) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sa = smem;                // 136 rows x 128 B = 17408 B
  uint8_t* sb = smem + 18 * 1024;    // 64 rows x 128 B
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 28 * 1024);
  uint32_t* tptr = reinterpret_cast<uint32_t*>(bar + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tptr, 128);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tptr;
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar[0], 136 * 128 + 64 * 128);
    tma_load_2d(sa, &map_a, &bar[0], 0, 0);
    tma_load_2d(sb, &map_b, &bar[0], 0, 0);
  }
  if (mode == 2) {
    // A through tensor memory: every thread copies its (shifted) row into TMEM columns [64, 96), then TS MMAs
    mbar_wait(&bar[0], 0);
    uint32_t v[32];
    ld_swizzled_row128(smem_u32(sa), (int)threadIdx.x + row_shift, v);
    tmem_st_32x32b_x32(tbase + ((uint32_t)(warp * 32) << 16) + 64, v);
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) {
      tc_fence_after();
      constexpr uint32_t idesc = make_idesc_bf16(128, 64);
      for (int k = 0; k < 4; ++k)
        umma_bf16_ts(tbase, tbase + 64 + k * 8, make_smem_desc(smem_u32(sb) + k * 32, 1024, LAYOUT_SW128, 0), idesc, k > 0);
      umma_commit(&bar[1]);
    }
  } else if (threadIdx.x == 0) {
    mbar_wait(&bar[0], 0);
    tc_fence_after();
    const uint32_t a0 = smem_u32(sa) + row_shift * 128, b0 = smem_u32(sb);
    constexpr uint32_t idesc = make_idesc_bf16(128, 64);
    for (int k = 0; k < 4; ++k)
      umma_bf16(tbase, make_smem_desc(a0 + k * 32, 1024, LAYOUT_SW128, 0),
                make_smem_desc(b0 + k * 32, 1024, LAYOUT_SW128, 0), idesc, k > 0);
    umma_commit(&bar[1]);
  }
  mbar_wait(&bar[1], 0);
  tc_fence_after();
  for (int half = 0; half < 2; ++half) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(tbase + ((uint32_t)(warp * 32) << 16) + half * 32, v);
    tmem_ld_wait();
    for (int j = 0; j < 32; ++j) d[(size_t)(warp * 32 + lane) * 64 + half * 32 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tbase, 128);
  }
}
}  // namespace psgla

extern "C" int psgla_selftest_umma(const void* a_dev, const void* b_dev, float* d_dev, int row_shift, int mode,
                                   void* stream) {
  PSGLA_REQUIRE(a_dev && b_dev && d_dev && row_shift >= 0 && row_shift <= 8 && (mode == 0 || mode == 2),
                "psgla_selftest_umma: bad argument");
  PFN_tensorMapEncodeTiled enc = get_tensor_map_encoder();
  if (!enc) return set_error(PSGLA_E_NODEVICE, "cuTensorMapEncodeTiled driver entry point not available");
  CUtensorMap ma, mb;
  const cuuint32_t estr[2] = {1, 1};
  {
    const cuuint64_t dims[2] = {64, 136};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {64, 136};
    CUresult r = enc(&ma, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(a_dev), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(PSGLA_E_BADARG, "tensor map A: CUresult %d", (int)r);
  }
  {
    const cuuint64_t dims[2] = {64, 64};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {64, 64};
    CUresult r = enc(&mb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(b_dev), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(PSGLA_E_BADARG, "tensor map B: CUresult %d", (int)r);
  }
  const int smem = 30 * 1024;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (!(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(selftest_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  selftest_umma_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(ma, mb, d_dev, row_shift, mode);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

// ------------------------------------------------------------------------------------------------ CTA-pair self-test
// D[256 x 64] = A[256 x 64] B[64 x 64]^T with one cta_group::2 MMA chain: CTA r of the pair holds A rows [128 r, 128 r + 128)
// in tensor memory (copied there by its own threads) and B rows [32 r, 32 r + 32) in shared memory; the leader issues,
// both read their 128 accumulator lanes back.  Pins down the operand split, the multicast commit and the remote arrive
// the conv kernel relies on.  mode 0: A from TMEM (TS); mode 1: A from shared memory (SS).
namespace psgla {
__global__ void __launch_bounds__(128, 1)
selftest_umma2_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                      float* __restrict__ d, int mode) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sa = smem;                // 128 rows x 128 B
  uint8_t* sb = smem + 16 * 1024;    // 32 rows x 128 B
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 20 * 1024);  // 0: TMA landed, 1: MMAs done, 2 (leader): operands ready
  uint32_t* tptr = reinterpret_cast<uint32_t*>(bar + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  if (threadIdx.x == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    mbar_init(&bar[2], 2);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc2(tptr, 128);
    tmem_relinquish2();
  }
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tbase = *tptr;
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar[0], 128 * 128 + 32 * 128);
    tma_load_2d(sa, &map_a, &bar[0], 0, (int)rank * 128);
    tma_load_2d(sb, &map_b, &bar[0], 0, (int)rank * 32);
  }
  mbar_wait(&bar[0], 0);
  if (mode == 0) {
    uint32_t v[32];
    ld_swizzled_row128(smem_u32(sa), (int)threadIdx.x, v);
    tmem_st_32x32b_x32(tbase + ((uint32_t)(warp * 32) << 16) + 64, v);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&bar[2]), 0));  // this CTA's operands are in place
  if (rank == 0 && warp == 0) {
    mbar_wait_cluster(&bar[2], 0);
    tc_fence_after();
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(256, 64);
      for (int k = 0; k < 4; ++k) {
        const uint64_t bd = make_smem_desc(smem_u32(sb) + k * 32, 1024, LAYOUT_SW128, 0);
        if (mode == 0)
          umma_bf16_ts2(tbase, tbase + 64 + k * 8, bd, idesc, k > 0);
        else
          umma_bf16_ss2(tbase, make_smem_desc(smem_u32(sa) + k * 32, 1024, LAYOUT_SW128, 0), bd, idesc, k > 0);
      }
      umma_commit2(&bar[1], 3);
    }
    __syncwarp();
  }
  mbar_wait(&bar[1], 0);
  tc_fence_after();
  for (int half = 0; half < 2; ++half) {
    uint32_t v[32];
    tmem_ld_32x32b_x32(tbase + ((uint32_t)(warp * 32) << 16) + half * 32, v);
    tmem_ld_wait();
    for (int j = 0; j < 32; ++j)
      d[(size_t)(rank * 128 + warp * 32 + lane) * 64 + half * 32 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before();
  cluster_sync();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc2(tbase, 128);
  }
}
}  // namespace psgla

extern "C" int psgla_selftest_umma2(const void* a_dev, const void* b_dev, float* d_dev, int mode, void* stream) {
  PSGLA_REQUIRE(a_dev && b_dev && d_dev && mode >= 0 && mode <= 1, "psgla_selftest_umma2: bad argument");
  PFN_tensorMapEncodeTiled enc = get_tensor_map_encoder();
  if (!enc) return set_error(PSGLA_E_NODEVICE, "cuTensorMapEncodeTiled driver entry point not available");
  CUtensorMap ma, mb;
  const cuuint32_t estr[2] = {1, 1};
  const cuuint64_t strides[1] = {128};
  {
    const cuuint64_t dims[2] = {64, 256};
    const cuuint32_t box[2] = {64, 128};
    CUresult r = enc(&ma, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(a_dev), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(PSGLA_E_BADARG, "tensor map A: CUresult %d", (int)r);
  }
  {
    const cuuint64_t dims[2] = {64, 64};
    const cuuint32_t box[2] = {64, 32};
    CUresult r = enc(&mb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(b_dev), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(PSGLA_E_BADARG, "tensor map B: CUresult %d", (int)r);
  }
  const int smem = 22 * 1024;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2);
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, selftest_umma2_kernel, ma, mb, d_dev, mode));
  return PSGLA_OK;
}

// ------------------------------------------------------------------------------------------------ MMA rate probe
namespace psgla {
// One CTA per block issues `iters` x 4 K-steps of M128 x N x K16 bf16 MMAs back to back on zeroed operands and reports
// the cycles one MMA took.  mode 0: A and B from shared memory (SS); 1: SS with the A start address shifted by one
// 128-byte row (the conv kernel's dx tap shift); 2: A from tensor memory (TS).
template <int mode>  // compile-time so that the issue loop is nothing but the MMAs
__global__ void __launch_bounds__(128, 1) mma_rate_kernel(int n, int iters, long long* __restrict__ cycles) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sa = smem;                 // 136 rows x 128 B
  uint8_t* sb = smem + 18 * 1024;     // 256 rows x 128 B
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 52 * 1024);
  uint32_t* tptr = reinterpret_cast<uint32_t*>(bar + 16);
  for (int i = threadIdx.x; i < 52 * 1024 / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    mbar_init(bar + 8, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tptr, 512);
    tmem_relinquish();
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tptr;
  if (warp == 0) {
    const uint32_t idesc = make_idesc_bf16(128, n);
    constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (LAYOUT_SW128 << 29);
    const uint32_t a_lo = ((smem_u32(sa) + (mode == 1 ? 128u : 0u)) >> 4) | 0x10000u;
    const uint32_t b_lo = (smem_u32(sb) >> 4) | 0x10000u;
    long long t0 = 0, t1 = 0;
    if (elect_one()) {
      t0 = clock64();
      for (int it = 0; it < (mode >= 5 ? 0 : iters); ++it) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (mode == 2)
            umma_bf16_ts(tbase, tbase + 256 + k * 8, ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc, 1);
          else if (mode >= 5)
            ;  // handled below
          else if (mode == 3)  // TS, consecutive MMAs alternate between two accumulators (no back-to-back dependency)
            umma_bf16_ts(tbase + ((it * 4 + k) & 1) * 128, tbase + 256 + k * 8, ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc, 1);
          else if (mode == 4)  // SS, alternating accumulators
            umma_bf16(tbase + ((it * 4 + k) & 1) * 128, ((uint64_t)DESC_HI << 32) | (a_lo + k * 2),
                      ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc, 1);
          else
            umma_bf16(tbase, ((uint64_t)DESC_HI << 32) | (a_lo + k * 2), ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc, 1);
        }
      }
      if (mode >= 5) {
        // the conv kernel's issue pattern: per "row" 9 taps x 4 K-steps into one of two accumulators, first MMA overwrites,
        // B walks the 72 KB weight array (8 KB per tap), A walks a 4-slot ring of 96 columns; one commit per row.
        // mode 5: commit to a second barrier every row; mode 6: no per-row commit; mode 7: as 5 with A always at slot 0
        for (int it = 0; it < iters; ++it) {
          const uint32_t d = tbase + (it & 1) * 64;
          uint32_t accumulate = 0;
#pragma unroll
          for (int dy = 0; dy < 3; ++dy) {
            const uint32_t a_t = tbase + 128 + (mode == 7 ? 0u : (uint32_t)((it + dy) & 3) * 96u);
#pragma unroll
            for (int dx = 0; dx < 3; ++dx)
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t bl = b_lo + (uint32_t)((((dy * 3 + dx) * 8192) % 32768 + k * 32) >> 4);
                umma_bf16_ts(d, a_t + dx * 32 + k * 8, ((uint64_t)DESC_HI << 32) | bl, idesc, accumulate);
                accumulate = 1;
              }
          }
          if (mode != 6) umma_commit(bar + 8);  // a dummy barrier nobody waits on (initialised below)
        }
      }
      umma_commit(bar);
    }
    __syncwarp();
    mbar_wait(bar, 0);
    t1 = clock64();
    if (elect_one()) cycles[blockIdx.x] = t0 ? (t1 - t0) : 0;
    // only the elected lane took t0
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tbase, 512);
  }
}
}  // namespace psgla

namespace psgla {
// The same probe for a CTA pair: the leader issues `iters` x 4 K-steps of M256 x N x K16 MMAs (cta_group::2) on zeroed
// operands, A from tensor memory (mode 0) or shared memory (mode 1), B split between the two shared memories.
template <int mode>
__global__ void __launch_bounds__(128, 1) mma_rate2_kernel(int n, int iters, long long* __restrict__ cycles) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sa = smem;                 // 128 rows x 128 B
  uint8_t* sb = smem + 18 * 1024;     // up to 128 rows x 128 B (this CTA's half of N)
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 52 * 1024);
  uint32_t* tptr = reinterpret_cast<uint32_t*>(bar + 16);
  for (int i = threadIdx.x; i < 52 * 1024 / 16; i += blockDim.x) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  const int warp = threadIdx.x >> 5;
  const uint32_t rank = cluster_ctarank();
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc2(tptr, 512);
    tmem_relinquish2();
  }
  fence_proxy_async();
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tbase = *tptr;
  if (warp == 0) {
    long long t0 = 0, t1 = 0;
    if (rank == 0 && elect_one()) {
      const uint32_t idesc = make_idesc_bf16(256, n);
      constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (LAYOUT_SW128 << 29);
      const uint32_t a_lo = (smem_u32(sa) >> 4) | 0x10000u;
      const uint32_t b_lo = (smem_u32(sb) >> 4) | 0x10000u;
      t0 = clock64();
      for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (mode == 0)
            umma_bf16_ts2(tbase, tbase + 256 + k * 8, ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc, 1);
          else
            umma_bf16_ss2(tbase, ((uint64_t)DESC_HI << 32) | (a_lo + k * 2), ((uint64_t)DESC_HI << 32) | (b_lo + k * 2), idesc, 1);
        }
      }
      umma_commit2(bar, 3);
    }
    __syncwarp();
    mbar_wait(bar, 0);
    t1 = clock64();
    if (rank == 0 && elect_one()) cycles[blockIdx.x >> 1] = t0 ? (t1 - t0) : 0;
  }
  tc_fence_before();
  cluster_sync();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc2(tbase, 512);
  }
}
}  // namespace psgla

extern "C" int psgla_selftest_mma_rate2(int mode, int n, int iters, int n_pairs, long long* cycles_dev, void* stream) {
  PSGLA_REQUIRE(cycles_dev && mode >= 0 && mode <= 1 && n >= 32 && n <= 256 && n % 32 == 0 && iters > 0 && n_pairs > 0,
                "psgla_selftest_mma_rate2: bad argument");
  const int smem = 54 * 1024;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (!(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate2_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * n_pairs));
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (mode == 0)
    PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, mma_rate2_kernel<0>, n, iters, cycles_dev));
  else
    PSGLA_CUDA_TRY(cudaLaunchKernelEx(&cfg, mma_rate2_kernel<1>, n, iters, cycles_dev));
  return PSGLA_OK;
}

extern "C" int psgla_selftest_mma_rate(int mode, int n, int iters, int grid, long long* cycles_dev, void* stream) {
  PSGLA_REQUIRE(cycles_dev && mode >= 0 && mode <= 7 && n >= 16 && n <= 256 && n % 16 == 0 && iters > 0 && grid > 0,
                "psgla_selftest_mma_rate: bad argument");
  PSGLA_REQUIRE(mode < 3 || n <= 128, "alternating-accumulator modes need n <= 128");
  const int smem = 54 * 1024;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (!(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(mma_rate_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  cudaStream_t st = (cudaStream_t)stream;
  switch (mode) {
    case 0: mma_rate_kernel<0><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
    case 1: mma_rate_kernel<1><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
    case 2: mma_rate_kernel<2><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
    case 3: mma_rate_kernel<3><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
    case 5: mma_rate_kernel<5><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
    case 6: mma_rate_kernel<6><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
    case 7: mma_rate_kernel<7><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
    default: mma_rate_kernel<4><<<grid, 128, smem, st>>>(n, iters, cycles_dev); break;
  }
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}
