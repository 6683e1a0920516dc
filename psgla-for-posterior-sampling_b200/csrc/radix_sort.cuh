// Segmented LSD radix sort of 32-bit keys on the device, shared by the sliced-W2 metric (gmm2d_metric.cu: keys only) and the
// large-S convergence diagnostics (mcmc_diag_large.cu: keys with a 32-bit payload, the split position).
//
//   P segments of n keys each, [P][n]; 4 passes of 8 bits, each:
//     histogram (per tile of 4096 keys) -> exclusive scan over [digit][tile] -> stable scatter, in which each warp owns a
//     contiguous slice of the tile and ranks equal digits with __match_any_sync
//   Offsets within a segment are 32-bit: n < 2^32.  One grid row per segment: P <= 65 535.
//   The sort is stable, so equal keys keep their input order (and the payload with them).
#pragma once
#include "common.cuh"

namespace psgla {

constexpr int RS_TILE = 4096;  // keys per CTA per pass: 8 warps x 16 rounds x 32 lanes
constexpr int RS_ROUNDS = RS_TILE / 256;
constexpr int RS_MAX_SEGMENTS = 65535;

// order-preserving map float -> uint32 (-0 sorts just below +0; NaN above +inf or below -inf by sign)
__device__ __forceinline__ uint32_t float_to_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
  return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xFFFFFFFFu));
}

inline int radix_tiles(long long n) { return (int)((n + RS_TILE - 1) / RS_TILE); }
// bytes of the histogram buffer for P segments of n keys
inline size_t radix_hist_bytes(long long n, int P) { return (size_t)P * 256 * (size_t)radix_tiles(n) * 4; }

static __global__ void __launch_bounds__(256)
radix_hist_kernel(const uint32_t* __restrict__ keys, long long n, int shift, int nb, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int p = blockIdx.y;
  const long long t0 = (long long)blockIdx.x * RS_TILE;
  const uint32_t* k = keys + (long long)p * n;
#pragma unroll 4
  for (int r = 0; r < RS_ROUNDS; ++r) {
    const long long i = t0 + r * 256 + threadIdx.x;
    if (i < n) atomicAdd(&h[(k[i] >> shift) & 255u], 1u);
  }
  __syncthreads();
  hist[((long long)p * 256 + threadIdx.x) * nb + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of one segment's [256 digits][nb tiles] counts (digit-major = the order keys land in)
static __global__ void __launch_bounds__(1024)
radix_scan_kernel(uint32_t* __restrict__ hist, int nb) {
  __shared__ uint32_t part[1024];
  const long long L = 256LL * nb;
  uint32_t* h = hist + (long long)blockIdx.x * L;
  const long long per = (L + 1023) / 1024;
  const long long a = threadIdx.x * per, b = (a + per < L) ? a + per : L;
  uint32_t s = 0;
  for (long long i = a; i < b; ++i) s += h[i];
  part[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {  // Hillis-Steele inclusive scan of the 1024 partial sums
    const uint32_t v = threadIdx.x >= off ? part[threadIdx.x - off] : 0u;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  uint32_t run = part[threadIdx.x] - s;
  for (long long i = a; i < b; ++i) {
    const uint32_t c = h[i];
    h[i] = run;
    run += c;
  }
}

// PAYLOAD: pay_in / pay_out [P][n] move with their keys; otherwise they are not touched (and may be null).
template <bool PAYLOAD>
__global__ void __launch_bounds__(256)
radix_scatter_kernel(const uint32_t* __restrict__ keys_in, uint32_t* __restrict__ keys_out, const uint32_t* __restrict__ pay_in,
                     uint32_t* __restrict__ pay_out, long long n, int shift, int nb, const uint32_t* __restrict__ hist) {
  __shared__ uint32_t wh[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = threadIdx.x; j < 8 * 256; j += 256) (&wh[0][0])[j] = 0;
  __syncthreads();
  const int p = blockIdx.y;
  const uint32_t* kin = keys_in + (long long)p * n;
  uint32_t* kout = keys_out + (long long)p * n;
  const long long w0 = (long long)blockIdx.x * RS_TILE + (long long)warp * (RS_TILE / 8);  // this warp's contiguous slice
  uint32_t mine[RS_ROUNDS];
#pragma unroll
  for (int r = 0; r < RS_ROUNDS; ++r) {
    const long long i = w0 + r * 32 + lane;
    mine[r] = i < n ? kin[i] : 0u;
    if (i < n) atomicAdd(&wh[warp][(mine[r] >> shift) & 255u], 1u);
  }
  __syncthreads();
  {  // digit d: global base of this tile, then the warps' slices in order
    const int d = threadIdx.x;
    uint32_t run = hist[((long long)p * 256 + d) * nb + blockIdx.x];
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const uint32_t c = wh[w][d];
      wh[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < RS_ROUNDS; ++r) {
    const long long i = w0 + r * 32 + lane;
    const bool valid = i < n;
    const uint32_t d = valid ? ((mine[r] >> shift) & 255u) : 256u;  // invalid lanes form their own group
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
    uint32_t base = 0;
    if (valid) base = wh[warp][d];
    __syncwarp();
    if (valid) {
      kout[base + rank] = mine[r];
      if (PAYLOAD) pay_out[(long long)p * n + base + rank] = pay_in[(long long)p * n + i];
      if (rank == 0) wh[warp][d] = base + __popc(peers);
    }
    __syncwarp();
  }
}

// Sorts P segments of n keys in a (and, when pa is not null, the payload in pa with them).  b / pb are scratch of the same
// size, hist radix_hist_bytes(n, P) bytes.  After the 4 (even) passes the result is back in a / pa.
inline void radix_sort_segments(uint32_t* a, uint32_t* b, uint32_t* pa, uint32_t* pb, long long n, int P, uint32_t* hist,
                                cudaStream_t st) {
  const int nb = radix_tiles(n);
  for (int pass = 0; pass < 4; ++pass) {
    radix_hist_kernel<<<dim3(nb, P), 256, 0, st>>>(a, n, pass * 8, nb, hist);
    radix_scan_kernel<<<P, 1024, 0, st>>>(hist, nb);
    if (pa)
      radix_scatter_kernel<true><<<dim3(nb, P), 256, 0, st>>>(a, b, pa, pb, n, pass * 8, nb, hist);
    else
      radix_scatter_kernel<false><<<dim3(nb, P), 256, 0, st>>>(a, b, nullptr, nullptr, n, pass * 8, nb, hist);
    uint32_t* t = a;
    a = b;
    b = t;
    t = pa;
    pa = pb;
    pb = t;
  }
}

}  // namespace psgla
