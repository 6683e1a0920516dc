// Convergence diagnostics for any number of split draws per element, device-wide: the same rank-normalised split-R-hat and
// bulk / tail ESS as mcmc_diag.cu (tests/mcmc_reference.py is the float64 restatement both are tested against), for
// S = 2 M floor(N / 2) up to 2^31 - 1 instead of the 16 384 one element's shared memory holds.  The use cases are the 2D
// chain populations (10^6 chains x hundreds of draws, [N][M][2]) and image runs thinned as the reference thins them.
//
// Input: fp32 [N][M][E] (draw, chain, element), read in place.  Elements are processed in groups of
// G = min(E, max(1, floor(2^28 / S)), 65 535); per group, all stream-ordered, the host never waits:
//   gather   the split draws of G elements into [G][S] split-chain order (chain c = half * M + m, then draw) as sortable keys
//            with their split position as payload, through a 32 x 32 shared-memory transpose; NaN elements are flagged.
//            Odd N: the M middle draws [G][M] too.
//   sort     segmented LSD radix sort (radix_sort.cuh, the one the sliced-W2 metric uses), keys with payload; the middle draws
//            keys only.  Then per element (one thread): median and 5 % / 95 % quantiles of all N M draws (numpy's, over the
//            union of the two sorted arrays) and the first sorted position at or above the median.
//   ranks    one thread per sorted position: the tie run around it (binary searches only where a neighbour is equal) gives
//            the average rank, z = Phi^-1((r - 3/8) / (S + 1/4)) by AS241 in fp64 rounded to fp32 (the small path's table
//            value), scattered to the split position through the payload.  Folded ranks: the count of folds |x - median|
//            below / at a position's fold on either side of the median, by binary search in the sorted array (the fold
//            grows with the position right of the median and shrinks left of it, compared in fp64): no second sort.
//   moments  fp64 per split chain (one CTA per chain, the series centred in place), then W, B, var+ and R-hat per element.
//   lags     autocovariances in rounds of B_r = 32 * 2^r lags (at most 2^22): per tile of the element's series one thread
//            per lag sums fp64 products over the tile, the tiles are summed in order per lag, and one thread per element
//            advances Geyer's recurrence (mcmc_diag.cuh) over the round's lags and marks the element done.  Later rounds
//            skip done elements; the launch count is O(log n') and the work at most twice what the last element needs.
// Series: bulk z (R-hat, ESS), folded z (R-hat), the indicators x <= q05 and x <= q95 (ESS), one after the other in one
// buffer.
//
// Every sum runs in an order fixed by N and M only (tiles, chunk lengths and block sizes are functions of S and n'): results
// are bit-identical across calls and do not depend on E, on the group an element lands in, or on the other elements.
#include "mcmc_large.cuh"

namespace psgla {

// one thread per element: median and quantiles of all N M draws, and the first sorted position at or above the median
__global__ void lg_quantiles_kernel(const float* __restrict__ srt, long long S, const float* __restrict__ mid, int nm, int G,
                                    LgElem* __restrict__ el) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G || el[g].nan) return;
  const float* a = srt + g * S;
  const float* b = nm ? mid + (long long)g * nm : nullptr;
  const long long tot = S + nm;
  const double lo = kth_of_union(a, S, b, nm, (tot - 1) / 2);
  const double med = (tot & 1) ? lo : (lo + kth_of_union(a, S, b, nm, tot / 2)) * 0.5;
  LgElem& e = el[g];
  e.med = med;
  e.q05 = quantile_linear(a, S, b, nm, 0.05);
  e.q95 = quantile_linear(a, S, b, nm, 0.95);
  long long x = 0, y = S;
  while (x < y) {
    const long long m = (x + y) >> 1;
    if ((double)a[m] < med) x = m + 1; else y = m;
  }
  e.r0 = x;
}

// bulk: z of the average rank of every sorted position, to its split position
__global__ void lg_rank_kernel(const float* __restrict__ srt, const uint32_t* __restrict__ pay, long long S, long long total,
                               const LgElem* __restrict__ el, float* __restrict__ ser) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= total) return;
  const long long g = k / S, p = k - g * S;
  if (el[g].nan) return;
  const float* a = srt + g * S;
  const float v = a[p];
  long long lo = p, hi = p + 1;
  if (p > 0 && a[p - 1] == v) {  // first position of the tie run
    long long x = 0, y = p - 1;
    while (x < y) {
      const long long m = (x + y) >> 1;
      if (a[m] < v) x = m + 1; else y = m;
    }
    lo = x;
  }
  if (p + 1 < S && a[p + 1] == v) {  // one past its last position
    long long x = p + 2, y = S;
    while (x < y) {
      const long long m = (x + y) >> 1;
      if (a[m] <= v) x = m + 1; else y = m;
    }
    hi = x;
  }
  ser[g * S + pay[k]] = rank_z(lo + 1 + hi, S);
}

// folded: z of the average rank of |x - median| (fp64) among the folds of both sides of the median
__global__ void lg_fold_rank_kernel(const float* __restrict__ srt, const uint32_t* __restrict__ pay, long long S,
                                    long long total, const LgElem* __restrict__ el, float* __restrict__ ser) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= total) return;
  const long long g = k / S, p = k - g * S;
  const LgElem& e = el[g];
  if (e.nan) return;
  const float* s = srt + g * S;
  const double med = e.med;
  const long long r0 = e.r0;
  const double d = fabs((double)s[p] - med);
  long long a = r0, b = S;  // right: first position with fold >= d
  while (a < b) {
    const long long m = (a + b) >> 1;
    if ((double)s[m] - med < d) a = m + 1; else b = m;
  }
  long long less = a - r0;
  b = S;  // right: first position with fold > d
  while (a < b) {
    const long long m = (a + b) >> 1;
    if ((double)s[m] - med <= d) a = m + 1; else b = m;
  }
  long long le = a - r0;
  a = 0, b = r0;  // left: first position with fold <= d
  while (a < b) {
    const long long m = (a + b) >> 1;
    if (med - (double)s[m] > d) a = m + 1; else b = m;
  }
  le += r0 - a;
  b = r0;  // left: first position with fold < d
  while (a < b) {
    const long long m = (a + b) >> 1;
    if (med - (double)s[m] >= d) a = m + 1; else b = m;
  }
  less += r0 - a;
  ser[g * S + pay[k]] = rank_z(less + 1 + le, S);
}

// tail: the indicator x <= q (h = 0: q05, 1: q95), not rank-normalised
__global__ void lg_indicator_kernel(const float* __restrict__ srt, const uint32_t* __restrict__ pay, long long S,
                                    long long total, const LgElem* __restrict__ el, int h, float* __restrict__ ser) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= total) return;
  const long long g = k / S;
  if (el[g].nan) return;
  const double q = h ? el[g].q95 : el[g].q05;
  ser[g * S + pay[k]] = (double)srt[k] <= q ? 1.f : 0.f;
}

__global__ void lg_output_kernel(const LgElem* __restrict__ el, int G, long long e0, float* __restrict__ rhat,
                                 float* __restrict__ ess_bulk, float* __restrict__ ess_tail) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const LgElem& e = el[g];
  const long long o = e0 + g;
  if (e.nan) {  // arviz: NaN anywhere in the draws gives NaN
    rhat[o] = ess_bulk[o] = ess_tail[o] = NAN;
    return;
  }
  rhat[o] = (isnan(e.rhat[0]) || isnan(e.rhat[1])) ? NAN : (float)fmax(e.rhat[0], e.rhat[1]);
  ess_bulk[o] = (float)e.ess[0];
  ess_tail[o] = (isnan(e.ess[1]) || isnan(e.ess[2])) ? NAN : (float)fmin(e.ess[1], e.ess[2]);
}

}  // namespace psgla

using namespace psgla;

extern "C" size_t psgla_mcmc_diag_large_workspace_bytes(int64_t n_draws, int64_t n_chains, int64_t n_elem) {
  LgLayout l;
  return lg_layout(n_draws, n_chains, n_elem, l) ? l.total : 0;
}

extern "C" int psgla_mcmc_diag_large(const float* draws_dev, int64_t n_draws, int64_t n_chains, int64_t n_elem, void* ws_dev,
                                     size_t ws_bytes, float* rhat_dev, float* ess_bulk_dev, float* ess_tail_dev,
                                     void* stream) {
  PSGLA_REQUIRE(draws_dev && ws_dev && rhat_dev && ess_bulk_dev && ess_tail_dev, "psgla_mcmc_diag_large: null pointer");
  PSGLA_REQUIRE(n_draws >= 4, "psgla_mcmc_diag_large: n_draws = %lld; split chains need at least 4 draws",
                (long long)n_draws);
  PSGLA_REQUIRE(n_chains >= 1, "psgla_mcmc_diag_large: n_chains = %lld must be >= 1", (long long)n_chains);
  PSGLA_REQUIRE(n_elem >= 1 && n_elem <= 0x7fffffffLL, "psgla_mcmc_diag_large: n_elem = %lld out of range",
                (long long)n_elem);
  LgLayout l;
  static thread_local LgRounds R;
  PSGLA_REQUIRE(lg_layout(n_draws, n_chains, n_elem, l, &R),
                "psgla_mcmc_diag_large: %lld chains x %lld draws give more than 2^31 - 1 split draws per element "
                "(S = 2 M floor(N/2)); n_draws or n_chains is out of range",
                (long long)n_chains, (long long)n_draws);
  if (ws_bytes < l.total)
    return set_error(PSGLA_E_WORKSPACE, "psgla_mcmc_diag_large: workspace of %zu bytes is smaller than the %zu needed",
                     ws_bytes, l.total);
  PSGLA_REQUIRE(((uintptr_t)ws_dev & 255) == 0, "psgla_mcmc_diag_large: workspace must be 256-byte aligned");

  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)ws_dev;
  unsigned long long* head = (unsigned long long*)ws;
  uint32_t* keys_a = (uint32_t*)(ws + l.keys_a);
  uint32_t* keys_b = (uint32_t*)(ws + l.keys_b);
  uint32_t* pay_a = (uint32_t*)(ws + l.pay_a);
  uint32_t* pay_b = (uint32_t*)(ws + l.pay_b);
  uint32_t* hist = (uint32_t*)(ws + l.hist);
  uint32_t* mid_a = (uint32_t*)(ws + l.mid_a);
  uint32_t* mid_b = (uint32_t*)(ws + l.mid_b);
  LgElem* el = (LgElem*)(ws + l.elem);
  double* cst = (double*)(ws + l.chain);
  double* acov = (double*)(ws + l.acov);
  double* part = (double*)(ws + l.part);
  const float* srt = (const float*)keys_a;  // the sorted draws, after the in-place conversion
  float* ser = (float*)keys_b;              // the sort's scratch holds the series afterwards

  const int N = (int)n_draws, M = (int)n_chains, n = l.n, Mp = l.Mp;
  const long long S = l.S, E = n_elem;
  const int mom_threads = n > 1024 ? 256 : 32;

  PSGLA_CUDA_TRY(cudaMemsetAsync(head, 0, 256, st));
  lg_stamp_kernel<<<1, 1, 0, st>>>(head, -1);
  for (long long e0 = 0; e0 < E; e0 += l.G) {
    const int G = (int)std::min<long long>(l.G, E - e0);
    const long long total = (long long)G * S;
    PSGLA_CUDA_TRY(cudaMemsetAsync(el, 0, (size_t)G * sizeof(LgElem), st));
    lg_gather_kernel<<<dim3(blocks_of(S, 32), blocks_of(G, 32)), dim3(32, 8), 0, st>>>(
        draws_dev, N, M, E, e0, G, S, n, keys_a, pay_a, el);
    if (l.odd)
      lg_gather_middle_kernel<<<blocks_of((long long)G * M, 256), 256, 0, st>>>(draws_dev, N, M, E, e0, G, mid_a, el);
    lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_GATHER);

    radix_sort_segments(keys_a, keys_b, pay_a, pay_b, S, G, hist, st);
    lg_keys_to_float_kernel<<<blocks_of(total, 256), 256, 0, st>>>(keys_a, total);
    if (l.odd) {
      radix_sort_segments(mid_a, mid_b, nullptr, nullptr, M, G, hist, st);
      lg_keys_to_float_kernel<<<blocks_of((long long)G * M, 256), 256, 0, st>>>(mid_a, (long long)G * M);
    }
    lg_quantiles_kernel<<<blocks_of(G, 128), 128, 0, st>>>(srt, S, (const float*)mid_a, l.odd ? M : 0, G, el);
    PSGLA_CUDA_TRY(cudaGetLastError());
    lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_SORT);

    // series 0 bulk z, 1 folded z, 2 x <= q05, 3 x <= q95
    for (int series = 0; series < 4; ++series) {
      if (series == 0)
        lg_rank_kernel<<<blocks_of(total, 256), 256, 0, st>>>(srt, pay_a, S, total, el, ser);
      else if (series == 1)
        lg_fold_rank_kernel<<<blocks_of(total, 256), 256, 0, st>>>(srt, pay_a, S, total, el, ser);
      else
        lg_indicator_kernel<<<blocks_of(total, 256), 256, 0, st>>>(srt, pay_a, S, total, el, series - 2, ser);
      lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_RANK);
      lg_chain_moments_kernel<<<(unsigned)((long long)G * Mp), mom_threads, 0, st>>>(ser, n, cst);
      lg_element_moments_kernel<<<G, 256, 0, st>>>(cst, Mp, n, el, series);
      PSGLA_CUDA_TRY(cudaGetLastError());
      lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_MOMENTS);
      if (series == 1) continue;  // folded: R-hat only
      lg_launch_lag_rounds(R, l, G, ser, el, part, acov, series == 0 ? 0 : series - 1, head, st);
      PSGLA_CUDA_TRY(cudaGetLastError());
    }
    lg_output_kernel<<<blocks_of(G, 128), 128, 0, st>>>(el, G, e0, rhat_dev, ess_bulk_dev, ess_tail_dev);
    PSGLA_CUDA_TRY(cudaGetLastError());
  }
  return PSGLA_OK;
}
