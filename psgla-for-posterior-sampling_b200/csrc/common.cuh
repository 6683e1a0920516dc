// Shared device/host helpers of libpsgla_b200: error plumbing, Philox4x32-10, Box-Muller.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>

#include "../../include/psgla_b200.h"

namespace psgla {

// ---------------------------------------------------------------- errors (thread-local message, int codes)
char* last_error_buffer();
int set_error(int code, const char* fmt, ...);

#define PSGLA_CUDA_TRY(expr)                                                                      \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess)                                                                        \
      return ::psgla::set_error((int)_e, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                __FILE__, __LINE__);                                              \
  } while (0)

#define PSGLA_REQUIRE(cond, ...)                                         \
  do {                                                                   \
    if (!(cond)) return ::psgla::set_error(PSGLA_E_BADARG, __VA_ARGS__); \
  } while (0)

// Per-device caches: the library may be driven on several GPUs from one process (the Python layer takes device=...), so
// nothing that depends on the device is cached process-wide.
constexpr int kMaxDevices = 64;
inline int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev;
}
inline int num_sms() {
  static std::atomic<int> cached[kMaxDevices];
  const int dev = current_device();
  int v = (dev >= 0 && dev < kMaxDevices) ? cached[dev].load(std::memory_order_relaxed) : 0;
  if (!v) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    if (v <= 0) v = 148;
    if (dev >= 0 && dev < kMaxDevices) cached[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}
// ---------------------------------------------------------------- Philox4x32-10 (Salmon et al. 2011)
// counter = (c0, c1, c2, c3), key = (seed_lo, seed_hi).  Library convention:
//   2D   : c0,c1 = (global step >> 1) as 64 bit, c2,c3 = global chain id
//   image: c0 = element index / 4, c1 = iteration, c2,c3 = global chain id
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3,
                                                       uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    // one 32 x 32 -> 64 bit product per multiplier (IMAD.WIDE.U32 on the device), round keys are compile-time offsets
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ (k0 + (uint32_t)i * 0x9E3779B9u);
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ (k1 + (uint32_t)i * 0xBB67AE85u);
    c0 = n0;
    c1 = (uint32_t)p1;
    c2 = n2;
    c3 = (uint32_t)p0;
  }
}

// The ten round keys (k0 + i W0, k1 + i W1) of a seed, computed once on the host and passed as a kernel parameter: in the
// kernels they are then constant-bank operands of the round's XOR instead of 20 integer adds per Philox call.
struct PhiloxKeys {
  uint32_t k[20];
};
inline PhiloxKeys philox_round_keys(uint64_t seed) {
  PhiloxKeys r;
  for (int i = 0; i < 10; ++i) {
    r.k[2 * i] = (uint32_t)seed + (uint32_t)i * 0x9E3779B9u;
    r.k[2 * i + 1] = (uint32_t)(seed >> 32) + (uint32_t)i * 0xBB67AE85u;
  }
  return r;
}
// Rounds FIRST .. 9 of the keyed form: a caller that has computed the first rounds itself (gmm2d_lean_kernel, whose first
// two rounds are mostly launch or thread constants) finishes the call here.
template <int FIRST = 0>
__device__ __forceinline__ void philox4x32_10_keyed(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3,
                                                    const PhiloxKeys& keys) {
#pragma unroll
  for (int i = FIRST; i < 10; ++i) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ keys.k[2 * i];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ keys.k[2 * i + 1];
    c0 = n0;
    c1 = (uint32_t)p1;
    c2 = n2;
    c3 = (uint32_t)p0;
  }
}

// Two uniform 32-bit words -> two independent N(0,1) (Box-Muller).  u1 in (0,1], theta = 2 pi u2.
// Fast-math intrinsics on purpose: MUFU.LG2 / MUFU.RSQ-or-SQRT / MUFU.SIN / MUFU.COS; absolute error ~1e-6, far
// below the Monte-Carlo resolution of any statistic the samplers feed (tests/test_gmm2d_gpu.py checks moments).
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
  const float u1 = fmaf((float)a, 2.3283064365386963e-10f, 1.1641532182693481e-10f);  // (a + 0.5) / 2^32
  // theta = 2 pi (b + 0.5) / 2^32 in one FMA (the 2 pi is folded into the constants: one multiply less per pair)
  const float theta = fmaf((float)b, 1.4629180792671596e-9f, 7.314590396335798e-10f);
  // sqrt(-2 ln u1) = sqrt(-2 ln2 log2 u1).  u1 >= 2^-33 is never subnormal and the radicand is >= 0, so the bare MUFU.LG2 /
  // MUFU.SQRT (.ftz forms) need none of the range fix-ups the library wrappers add.
  float lg, r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(u1));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * lg));
  float s, c;
  __sincosf(theta, &s, &c);
  z0 = r * c;
  z1 = r * s;
}

__device__ __forceinline__ void philox_normal4(uint64_t seed, uint64_t subsequence, uint32_t ctr_lo, uint32_t ctr_hi,
                                               float& z0, float& z1, float& z2, float& z3) {
  uint32_t c0 = ctr_lo, c1 = ctr_hi, c2 = (uint32_t)subsequence, c3 = (uint32_t)(subsequence >> 32);
  philox4x32_10(c0, c1, c2, c3, (uint32_t)seed, (uint32_t)(seed >> 32));
  box_muller(c0, c1, z0, z1);
  box_muller(c2, c3, z2, z3);
}

__device__ __forceinline__ void philox_normal4_keyed(const PhiloxKeys& keys, uint64_t subsequence, uint32_t ctr_lo,
                                                     uint32_t ctr_hi, float& z0, float& z1, float& z2, float& z3) {
  uint32_t c0 = ctr_lo, c1 = ctr_hi, c2 = (uint32_t)subsequence, c3 = (uint32_t)(subsequence >> 32);
  philox4x32_10_keyed(c0, c1, c2, c3, keys);
  box_muller(c0, c1, z0, z1);
  box_muller(c2, c3, z2, z3);
}

}  // namespace psgla
