// Convergence diagnostics of multi-chain runs, per element, on the device: rank-normalised split-R-hat and bulk / tail ESS
// (Vehtari, Gelman, Simpson, Carpenter, Buerkner 2021), as arviz's rhat(method="rank"), ess(method="bulk") and
// ess(method="tail") define them; tests/mcmc_reference.py is the float64 restatement the kernel is tested against.
//
// Input: the sampler's own sample buffer, fp32 [N][M][E] (draw, chain, element), read in place.  Each chain is split into
// two halves of N' = N / 2 draws (odd N: the middle draw is dropped), S = 2 M N' values per element.
//
// One CTA per element, everything in shared memory:
//   srt[P]  the S split draws sorted (bitonic, P = S rounded up to a power of two, +inf padded);
//   xv[S]   the same draws in split-chain order (chain c = half * M + m, then draw);
//   ser[S]  the series being analysed: z of the draws, z of the folded draws |x - median|, the indicators x <= q05 / q95;
//           for odd N it first holds the M middle draws, sorted, for the median and quantiles of all N M draws;
// Ranks come from binary searches in srt (ties get the average rank), the fold's ranks from binary searches on either side
// of the median (|x - med| is monotone there).  z = Phi^-1((r - 3/8) / (S + 1/4)) depends only on 2r and S: a table of 2S + 1
// fp32 values (AS241 in fp64, rounded) is built once per call in the workspace.  Chain moments are fp64; autocovariances
// are fp64 sums of products of the centred fp32 series, one Geyer pair of lags per pass, and the lag loop stops where Geyer's initial positive
// sequence stops (arviz's _ess, the adjustment after the last pair included).
//
// The order of every sum is fixed by the thread and warp layout, which depends on N and M only: results are bit-identical
// across calls and do not depend on E or on the other elements of the launch.
#include <cmath>
#include <cstring>

#include "mcmc_diag.cuh"

namespace psgla {

constexpr int DG_THREADS = 1024;
constexpr int DG_WARPS = DG_THREADS / 32;
constexpr size_t DG_TABLE_OFFSET = 256;  // workspace: stage cycle counters, then the z table

// table[k] = Phi^-1((k / 2 - 3/8) / (S + 1/4)), k = 2r for the (half-)integer average rank r in [1, S]
__global__ void mcmc_z_table_kernel(int S, float* __restrict__ table) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > 2 * S) return;
  table[k] = k < 1 ? 0.f : rank_z(k, S);
}

struct DiagShared {
  double part[DG_WARPS][3];
  double sum[3];
  double med, q05, q95;
  int r0;  // first sorted position at or above the median
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sums of three values, in a fixed order; every thread gets the totals.
__device__ void block_sum3(double& a, double& b, double& c, DiagShared& sh) {
  a = warp_sum(a), b = warp_sum(b), c = warp_sum(c);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) sh.part[warp][0] = a, sh.part[warp][1] = b, sh.part[warp][2] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s0 = 0, s1 = 0, s2 = 0;
    for (int w = 0; w < DG_WARPS; ++w) s0 += sh.part[w][0], s1 += sh.part[w][1], s2 += sh.part[w][2];
    sh.sum[0] = s0, sh.sum[1] = s1, sh.sum[2] = s2;
  }
  __syncthreads();
  a = sh.sum[0], b = sh.sum[1], c = sh.sum[2];
}

__device__ void bitonic_sort(float* a, int P) {
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < (P >> 1); i += DG_THREADS) {
        const int lo = 2 * i - (i & (j - 1)), hi = lo + j;
        const float x = a[lo], y = a[hi];
        if ((x > y) == ((lo & k) == 0)) a[lo] = y, a[hi] = x;
      }
      __syncthreads();
    }
}

__device__ __forceinline__ int lower_bound(const float* a, int n, float v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (a[m] < v) lo = m + 1; else hi = m;
  }
  return lo;
}
__device__ __forceinline__ int upper_bound(const float* a, int n, float v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (a[m] <= v) lo = m + 1; else hi = m;
  }
  return lo;
}

// chain index of flat position j of a chain-major [n_chains][n] array, without an integer division
__device__ __forceinline__ int chain_of(int j, int n, float inv_n) {
  int c = (int)((float)j * inv_n);
  if (c * n > j) --c;
  else if ((c + 1) * n <= j) ++c;
  return c;
}

struct SeriesStats {
  double rhat, ess;
};

// Split-R-hat and (want_ess) ESS of the series ser [Mp][n] (centred in place).  W == 0: both NaN.
__device__ SeriesStats series_stats(float* ser, int Mp, int n, bool want_ess, DiagShared& sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double sm = 0, sm2 = 0, sv = 0;
  for (int c = warp; c < Mp; c += DG_WARPS) {
    float* x = ser + (size_t)c * n;
    double s = 0;
    for (int i = lane; i < n; i += 32) s += x[i];
    const double m = warp_sum(s) / n;
    double q = 0;
    for (int i = lane; i < n; i += 32) {
      const double d = x[i] - m;
      q += d * d;
      x[i] = (float)d;
    }
    q = warp_sum(q);
    if (lane == 0) sm += m, sm2 += m * m, sv += q / (n - 1);
  }
  block_sum3(sm, sm2, sv, sh);
  const double W = sv / Mp, mbar = sm / Mp;
  const double B = n * (sm2 - Mp * mbar * mbar) / (Mp - 1);
  const double vp = (n - 1.0) / n * W + B / n;
  SeriesStats r{NAN, NAN};
  if (!(W > 0)) return r;
  r.rhat = sqrt(vp / W);
  if (!want_ess) return r;

  const int S = Mp * n;
  const float inv_n = 1.f / n;
  const double norm = 1.0 / ((double)n * Mp);
  // mean over chains of the lag-t autocovariances (divisor n), for lags t, t + 1, t + 2
  auto acov3 = [&](int t, double& a0, double& a1, double& a2) {
    a0 = a1 = a2 = 0;
    for (int j = threadIdx.x; j < S; j += DG_THREADS) {
      const int i = j - chain_of(j, n, inv_n) * n;
      const double v = ser[j];
      if (i + t < n) a0 += v * ser[j + t];
      if (i + t + 1 < n) a1 += v * ser[j + t + 1];
      if (i + t + 2 < n) a2 += v * ser[j + t + 2];
    }
    block_sum3(a0, a1, a2, sh);
    a0 *= norm, a1 *= norm, a2 *= norm;
  };
  double a1, a2, a3;
  acov3(1, a1, a2, a3);
  // Geyer's initial positive / monotone sequence (mcmc_diag.cuh); a2 / a3 of the first pass serve the first pair.
  Geyer g = geyer_start(W, vp, a1);
  while (geyer_running(g, n)) {
    if (g.t > 1) {
      double unused;
      acov3(g.t + 1, a2, a3, unused);
    }
    geyer_step(g, a2, a3);
  }
  r.ess = geyer_ess(g, S);
  return r;
}

// grid: one CTA per element.  cycles: [4] SM cycles summed over CTAs: load; sort, median and quantiles; ranks (binary searches
// and the z table); chain moments and autocovariances.
__global__ void __launch_bounds__(DG_THREADS, 1)
mcmc_diag_kernel(const float* __restrict__ draws, int N, int M, long long E, const float* __restrict__ table,
                 float* __restrict__ rhat_out, float* __restrict__ ess_bulk_out, float* __restrict__ ess_tail_out,
                 unsigned long long* __restrict__ cycles) {
  extern __shared__ float smem[];
  __shared__ DiagShared sh;
  const int n = N / 2, Mp = 2 * M, S = Mp * n, odd_n = N & 1;
  int P = 1;
  while (P < S) P <<= 1;
  float* srt = smem;
  float* xv = srt + P;
  float* ser = xv + S;
  const long long e = blockIdx.x;
  const long long t0 = clock64();

  const float inv_n = 1.f / n;
  bool bad = false;
  for (int j = threadIdx.x; j < S; j += DG_THREADS) {
    const int c = chain_of(j, n, inv_n), i = j - c * n;
    const int m = c < M ? c : c - M, draw = c < M ? i : N - n + i;
    const float v = draws[((long long)draw * M + m) * E + e];
    bad |= isnan(v);
    xv[j] = srt[j] = v;
  }
  for (int j = S + threadIdx.x; j < P; j += DG_THREADS) srt[j] = INFINITY;
  int Pm = 0;  // odd N: the middle draws, sorted, +inf padded to a power of two
  if (odd_n) {
    Pm = 1;
    while (Pm < M) Pm <<= 1;
    for (int m = threadIdx.x; m < Pm; m += DG_THREADS) {
      const float v = m < M ? draws[((long long)(N / 2) * M + m) * E + e] : INFINITY;
      bad |= isnan(v);
      ser[m] = v;
    }
  }
  if (__syncthreads_or(bad)) {  // arviz: NaN anywhere in the draws gives NaN
    if (threadIdx.x == 0) rhat_out[e] = ess_bulk_out[e] = ess_tail_out[e] = NAN;
    return;
  }
  const long long t1 = clock64();

  bitonic_sort(srt, P);
  if (odd_n) bitonic_sort(ser, Pm);
  if (threadIdx.x == 0) {  // median and quantiles of all N M draws
    const int nm = odd_n ? M : 0, tot = S + nm;
    const double lo = kth_of_union(srt, S, ser, nm, (tot - 1) / 2);
    sh.med = (tot & 1) ? lo : (lo + kth_of_union(srt, S, ser, nm, tot / 2)) * 0.5;
    sh.q05 = quantile_linear(srt, S, ser, nm, 0.05);
    sh.q95 = quantile_linear(srt, S, ser, nm, 0.95);
    int a = 0, b = S;
    while (a < b) {
      const int mid = (a + b) >> 1;
      if ((double)srt[mid] < sh.med) a = mid + 1; else b = mid;
    }
    sh.r0 = a;
  }
  __syncthreads();
  const long long t_sort = clock64() - t1;
  const double med = sh.med;
  const int r0 = sh.r0;

  // bulk: z of the average ranks
  for (int j = threadIdx.x; j < S; j += DG_THREADS) {
    const float v = xv[j];
    ser[j] = __ldg(table + lower_bound(srt, S, v) + 1 + upper_bound(srt, S, v));
  }
  __syncthreads();
  long long t_rank = clock64() - t1 - t_sort;
  long long t2 = clock64();
  const SeriesStats bulk = series_stats(ser, Mp, n, true, sh);
  long long t_mom = clock64() - t2;

  // tail R-hat: z of the ranks of |x - median|.  Right of the median (positions >= r0) the fold grows with the position, left
  // of it the fold shrinks: the count of folds below / at d is two binary searches per side.
  t2 = clock64();
  for (int j = threadIdx.x; j < S; j += DG_THREADS) {
    const double d = fabs((double)xv[j] - med);
    int a = r0, b = S;  // right: first position with fold >= d
    while (a < b) {
      const int mid = (a + b) >> 1;
      if ((double)srt[mid] - med < d) a = mid + 1; else b = mid;
    }
    int less = a - r0;
    b = S;  // right: first position with fold > d
    while (a < b) {
      const int mid = (a + b) >> 1;
      if ((double)srt[mid] - med <= d) a = mid + 1; else b = mid;
    }
    int le = a - r0;
    a = 0, b = r0;  // left: first position with fold <= d
    while (a < b) {
      const int mid = (a + b) >> 1;
      if (med - (double)srt[mid] > d) a = mid + 1; else b = mid;
    }
    le += r0 - a;
    b = r0;  // left: first position with fold < d
    while (a < b) {
      const int mid = (a + b) >> 1;
      if (med - (double)srt[mid] >= d) a = mid + 1; else b = mid;
    }
    less += r0 - a;
    ser[j] = __ldg(table + less + 1 + le);
  }
  __syncthreads();
  t_rank += clock64() - t2;
  t2 = clock64();
  const SeriesStats tail = series_stats(ser, Mp, n, false, sh);

  // tail ESS: the indicator series of the 5 % and 95 % quantiles (not rank-normalised)
  SeriesStats q[2];
  for (int h = 0; h < 2; ++h) {
    const double qv = h ? sh.q95 : sh.q05;
    for (int j = threadIdx.x; j < S; j += DG_THREADS) ser[j] = (double)xv[j] <= qv ? 1.f : 0.f;
    __syncthreads();
    q[h] = series_stats(ser, Mp, n, true, sh);
  }
  t_mom += clock64() - t2;

  if (threadIdx.x == 0) {
    rhat_out[e] = (isnan(bulk.rhat) || isnan(tail.rhat)) ? NAN : (float)fmax(bulk.rhat, tail.rhat);
    ess_bulk_out[e] = (float)bulk.ess;
    ess_tail_out[e] = (isnan(q[0].ess) || isnan(q[1].ess)) ? NAN : (float)fmin(q[0].ess, q[1].ess);
    atomicAdd(cycles + 0, (unsigned long long)(t1 - t0));
    atomicAdd(cycles + 1, (unsigned long long)t_sort);
    atomicAdd(cycles + 2, (unsigned long long)t_rank);
    atomicAdd(cycles + 3, (unsigned long long)t_mom);
  }
}

inline long long diag_size(int64_t n_draws, int64_t n_chains) {  // S, or -1 when out of range
  if (n_draws < 4 || n_chains < 1 || n_chains > PSGLA_MCMC_MAX_DRAWS || n_draws / 2 > PSGLA_MCMC_MAX_DRAWS) return -1;
  return 2 * n_chains * (n_draws / 2);
}

}  // namespace psgla

using namespace psgla;

extern "C" size_t psgla_mcmc_diag_workspace_bytes(int64_t n_draws, int64_t n_chains) {
  const long long S = diag_size(n_draws, n_chains);
  if (S < 0 || S > PSGLA_MCMC_MAX_DRAWS) return 0;
  return DG_TABLE_OFFSET + (((size_t)(2 * S + 1) * sizeof(float) + 255) & ~(size_t)255);
}

extern "C" int psgla_mcmc_diag(const float* draws_dev, int64_t n_draws, int64_t n_chains, int64_t n_elem, void* ws_dev,
                               size_t ws_bytes, float* rhat_dev, float* ess_bulk_dev, float* ess_tail_dev, void* stream) {
  PSGLA_REQUIRE(draws_dev && ws_dev && rhat_dev && ess_bulk_dev && ess_tail_dev, "psgla_mcmc_diag: null pointer");
  PSGLA_REQUIRE(n_draws >= 4, "psgla_mcmc_diag: n_draws = %lld; split chains need at least 4 draws", (long long)n_draws);
  PSGLA_REQUIRE(n_chains >= 1, "psgla_mcmc_diag: n_chains = %lld must be >= 1", (long long)n_chains);
  PSGLA_REQUIRE(n_elem >= 1 && n_elem <= 0x7fffffffLL, "psgla_mcmc_diag: n_elem = %lld out of range", (long long)n_elem);
  const long long S = diag_size(n_draws, n_chains);
  PSGLA_REQUIRE(S >= 0 && S <= PSGLA_MCMC_MAX_DRAWS,
                "psgla_mcmc_diag: %lld chains x %lld draws give more than %d split draws per element (S = 2 M floor(N/2)); "
                "store fewer draws (a larger thinning n_inter) or diagnose fewer chains",
                (long long)n_chains, (long long)n_draws, PSGLA_MCMC_MAX_DRAWS);
  if (ws_bytes < psgla_mcmc_diag_workspace_bytes(n_draws, n_chains))
    return set_error(PSGLA_E_WORKSPACE, "psgla_mcmc_diag: workspace of %zu bytes is smaller than the %zu needed", ws_bytes,
                     psgla_mcmc_diag_workspace_bytes(n_draws, n_chains));
  const int N = (int)n_draws, M = (int)n_chains, Si = (int)S;
  int P = 1;
  while (P < Si) P <<= 1;
  const size_t smem = ((size_t)P + 2 * (size_t)Si) * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  float* table = (float*)((char*)ws_dev + DG_TABLE_OFFSET);
  PSGLA_CUDA_TRY(cudaFuncSetAttribute(mcmc_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  PSGLA_CUDA_TRY(cudaMemsetAsync(ws_dev, 0, DG_TABLE_OFFSET, st));
  mcmc_z_table_kernel<<<(2 * Si + 1 + 255) / 256, 256, 0, st>>>(Si, table);
  PSGLA_CUDA_TRY(cudaGetLastError());
  mcmc_diag_kernel<<<(unsigned)n_elem, DG_THREADS, smem, st>>>(draws_dev, N, M, (long long)n_elem, table, rhat_dev,
                                                                ess_bulk_dev, ess_tail_dev, (unsigned long long*)ws_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}
