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
#include <cmath>
#include <cstring>

#include "mcmc_diag.cuh"
#include "radix_sort.cuh"

namespace psgla {

constexpr long long LG_MAX_S = 0x7fffffffLL;
constexpr long long LG_GROUP_DRAWS = 1LL << 28;  // split draws per group (G S <= 2^28 unless one element is larger)
constexpr int LG_LAG_BLOCK = 256;                // lags per CTA of the lag kernel
constexpr int LG_CHUNK = 2048;                   // series values staged per pass of the lag kernel
constexpr int LG_MAX_ROUNDS = 512;
constexpr int LG_MAX_LAGS = 1 << 22;  // lags per round

// workspace head, uint64 words
enum { LGH_GATHER, LGH_SORT, LGH_RANK, LGH_MOMENTS, LGH_LAGS, LGH_ROUNDS_RUN, LGH_ROUNDS_LAUNCHED, LGH_LAST, LGH_ACTIVE };

struct LgElem {
  double med, q05, q95;
  long long r0;       // first sorted position at or above the median
  double rhat[2];     // bulk, folded
  double ess[3];      // bulk, x <= q05, x <= q95
  Geyer geyer;        // the series in progress
  double W, vp;
  int nan, done;
};

struct LgRounds {
  int n;
  int lag0[LG_MAX_ROUNDS], lags[LG_MAX_ROUNDS];
  long long tile[LG_MAX_ROUNDS];
};

// The lag rounds an element whose recurrence runs to the end needs; every running element advances in step, so this is the
// plan for all of them.  Round r computes the lags [lag0, lag0 + lags) of which Geyer's steps take pairs (t + 1, t + 2).
static void lag_rounds(int n, LgRounds& R) {
  R.n = 0;
  int next = 1, t = 1;
  for (int r = 0; r < LG_MAX_ROUNDS; ++r) {
    const long long want = 32LL << (r < 20 ? r : 20);
    const int B = (int)std::min<long long>(std::min<long long>(want, LG_MAX_LAGS), (long long)n - next);
    if (B < 1) break;
    R.lag0[R.n] = next, R.lags[R.n] = B, R.tile[R.n] = std::max<long long>(4096, 16LL * B);
    ++R.n;
    const int end = next + B - 1;
    while (t < n - 3 && t + 2 <= end) t += 2;
    if (!(t < n - 3)) break;
    next = t + 1;
  }
}

struct LgLayout {
  long long S, G;
  int n, Mp, odd;
  size_t keys_a, keys_b, pay_a, pay_b, hist, mid_a, mid_b, elem, chain, acov, part, total;
  int max_lags;
};

static size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

// false when out of range
static bool lg_layout(int64_t N, int64_t M, int64_t E, LgLayout& l, LgRounds* R = nullptr) {
  if (N < 4 || M < 1 || E < 1 || E > 0x7fffffffLL) return false;
  const long long n = N / 2;
  if (M > LG_MAX_S / (2 * n)) return false;
  l.S = 2 * M * n;
  l.n = (int)n, l.Mp = (int)(2 * M), l.odd = (int)(N & 1);
  l.G = std::min<long long>(std::min<long long>(E, std::max<long long>(1, LG_GROUP_DRAWS / l.S)), RS_MAX_SEGMENTS);
  LgRounds local;
  LgRounds& r = R ? *R : local;
  lag_rounds(l.n, r);
  size_t part = 0;
  l.max_lags = 1;
  for (int i = 0; i < r.n; ++i) {
    const long long tiles = (l.S + r.tile[i] - 1) / r.tile[i];
    part = std::max(part, (size_t)(tiles * r.lags[i]));
    l.max_lags = std::max(l.max_lags, r.lags[i]);
  }
  const size_t P = (size_t)(l.G * l.S);
  size_t o = 256;
  l.keys_a = o, o += al256(P * 4);
  l.keys_b = o, o += al256(P * 4);
  l.pay_a = o, o += al256(P * 4);
  l.pay_b = o, o += al256(P * 4);
  l.hist = o, o += al256(radix_hist_bytes(l.S, (int)l.G));
  l.mid_a = o, o += l.odd ? al256((size_t)l.G * M * 4) : 0;
  l.mid_b = o, o += l.odd ? al256((size_t)l.G * M * 4) : 0;
  l.elem = o, o += al256((size_t)l.G * sizeof(LgElem));
  l.chain = o, o += al256((size_t)l.G * l.Mp * 2 * sizeof(double));
  l.acov = o, o += al256((size_t)l.G * l.max_lags * sizeof(double));
  l.part = o, o += al256((size_t)l.G * part * sizeof(double));
  l.total = o;
  return true;
}

// ------------------------------------------------------------------------------------------------------------- kernels
__device__ __forceinline__ double lg_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum in a fixed order (lanes by butterfly, then the warps in order); every thread gets the total.
__device__ double lg_block_sum(double v, double* part /* [32] shared */) {
  v = lg_warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) part[warp] = v;
  __syncthreads();
  double s = 0;
  for (int w = 0; w < nw; ++w) s += part[w];
  return s;
}

__global__ void lg_stamp_kernel(unsigned long long* head, int stage) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  if (stage >= 0) head[stage] += t - head[LGH_LAST];
  if (stage == LGH_LAGS) {
    head[LGH_ROUNDS_LAUNCHED] += 1;
    head[LGH_ROUNDS_RUN] += head[LGH_ACTIVE];
    head[LGH_ACTIVE] = 0;
  }
  head[LGH_LAST] = t;
}

// grid (ceil(S / 32), ceil(G / 32)), block (32, 8): [draw][chain][element] tile -> [element][split position] keys
__global__ void __launch_bounds__(256)
lg_gather_kernel(const float* __restrict__ draws, int N, int M, long long E, long long e0, int G, long long S, int n,
                 uint32_t* __restrict__ keys, uint32_t* __restrict__ pay, LgElem* __restrict__ el) {
  __shared__ float tile[32][33];
  const long long p0 = (long long)blockIdx.x * 32;
  const int g0 = blockIdx.y * 32, tx = threadIdx.x, ty = threadIdx.y;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const long long p = p0 + ty + 8 * r;
    const int g = g0 + tx;
    float v = 0.f;
    if (p < S && g < G) {
      const long long c = p / n, i = p - c * n;
      const long long m = c < M ? c : c - M, draw = c < M ? i : N - n + i;
      v = draws[(draw * M + m) * E + e0 + g];
    }
    tile[ty + 8 * r][tx] = v;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int g = g0 + ty + 8 * r;
    const long long p = p0 + tx;
    if (p < S && g < G) {
      const float v = tile[tx][ty + 8 * r];
      keys[g * S + p] = float_to_key(v);
      pay[g * S + p] = (uint32_t)p;
      if (isnan(v)) el[g].nan = 1;
    }
  }
}

// odd N: the middle draws [G][M]
__global__ void lg_gather_middle_kernel(const float* __restrict__ draws, int N, int M, long long E, long long e0, int G,
                                        uint32_t* __restrict__ keys, LgElem* __restrict__ el) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= (long long)G * M) return;
  const long long m = k / G, g = k - m * G;
  const float v = draws[((long long)(N / 2) * M + m) * E + e0 + g];
  keys[g * M + m] = float_to_key(v);
  if (isnan(v)) el[g].nan = 1;
}

__global__ void lg_keys_to_float_kernel(uint32_t* __restrict__ k, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) k[i] = __float_as_uint(key_to_float(k[i]));
}

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

// one CTA per split chain: fp64 mean and variance (divisor n - 1); the chain is centred in place (fp32)
__global__ void lg_chain_moments_kernel(float* __restrict__ ser, int n, double* __restrict__ cst) {
  __shared__ double part[32];
  float* x = ser + (long long)blockIdx.x * n;
  double s = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += x[i];
  const double m = lg_block_sum(s, part) / n;
  double q = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double d = x[i] - m;
    q += d * d;
    x[i] = (float)d;
  }
  q = lg_block_sum(q, part);
  if (threadIdx.x == 0) cst[2 * (long long)blockIdx.x] = m, cst[2 * (long long)blockIdx.x + 1] = q / (n - 1);
}

// one CTA per element: W, B, var+ and R-hat of the series; elements with NaN draws or W = 0 are done (NaN) at once
__global__ void __launch_bounds__(256)
lg_element_moments_kernel(const double* __restrict__ cst, int Mp, int n, LgElem* __restrict__ el, int series) {
  __shared__ double part[32];
  const double* c = cst + 2LL * blockIdx.x * Mp;
  double sm = 0, sm2 = 0, sv = 0;
  for (int k = threadIdx.x; k < Mp; k += blockDim.x) {
    const double m = c[2 * k];
    sm += m, sm2 += m * m, sv += c[2 * k + 1];
  }
  sm = lg_block_sum(sm, part);
  sm2 = lg_block_sum(sm2, part);
  sv = lg_block_sum(sv, part);
  if (threadIdx.x) return;
  LgElem& e = el[blockIdx.x];
  const double W = sv / Mp, mbar = sm / Mp;
  const double B = n * (sm2 - Mp * mbar * mbar) / (Mp - 1);
  const double vp = (n - 1.0) / n * W + B / n;
  const bool ok = !e.nan && W > 0;
  if (series < 2) e.rhat[series] = ok ? sqrt(vp / W) : NAN;
  const int s = series == 0 ? 0 : series - 1;  // ESS slot of series 0, 2, 3
  e.W = W, e.vp = vp;
  e.done = !ok;
  if (series != 1) e.ess[s] = NAN;
}

// grid (G * tiles, ceil(lags / 256)), block min(lags, 256): part[g][tile][l] = sum over the tile's positions j of
// ser[j] ser[j + lag0 + l], for pairs within one split chain
__global__ void __launch_bounds__(LG_LAG_BLOCK)
lg_lag_kernel(const float* __restrict__ ser, long long S, int n, const LgElem* __restrict__ el, int lag0, int lags,
              long long tile_len, int tiles, double* __restrict__ part) {
  __shared__ float sa[LG_CHUNK], sb[LG_CHUNK + LG_LAG_BLOCK];
  const int g = blockIdx.x / tiles, tile = blockIdx.x - g * tiles;
  if (el[g].done) return;
  const int l = blockIdx.y * LG_LAG_BLOCK + threadIdx.x;
  const long long lb = lag0 + (long long)blockIdx.y * LG_LAG_BLOCK;  // this CTA's first lag
  const int lim = n - (lag0 + l);                                     // a product stays in its chain while i < lim
  const float* x = ser + g * S;
  const long long j0 = tile * tile_len, j1 = min(S, j0 + tile_len);
  double acc = 0;
  for (long long c0 = j0; c0 < j1; c0 += LG_CHUNK) {
    const int len = (int)min((long long)LG_CHUNK, j1 - c0);
    __syncthreads();
    for (int k = threadIdx.x; k < LG_CHUNK; k += blockDim.x) sa[k] = k < len ? x[c0 + k] : 0.f;
    for (int k = threadIdx.x; k < LG_CHUNK + LG_LAG_BLOCK; k += blockDim.x) {
      const long long q = c0 + lb + k;
      sb[k] = q < S ? x[q] : 0.f;
    }
    __syncthreads();
    if (l < lags && lim > 0) {
      int i = (int)(c0 % n);
      for (int k = 0; k < len; ++k) {
        if (i < lim) acc = fma((double)sa[k], (double)sb[k + threadIdx.x], acc);
        if (++i == n) i = 0;
      }
    }
  }
  if (l < lags) part[((long long)g * tiles + tile) * lags + l] = acc;
}

// grid (G, ceil(lags / 256)): acov[g][l] = norm * sum over tiles in order
__global__ void __launch_bounds__(256)
lg_acov_kernel(const double* __restrict__ part, int tiles, int lags, const LgElem* __restrict__ el, double norm,
               int max_lags, double* __restrict__ acov) {
  const int g = blockIdx.x, l = blockIdx.y * 256 + threadIdx.x;
  if (l >= lags || el[g].done) return;
  const double* p = part + (long long)g * tiles * lags + l;
  double s = 0;
  for (int t = 0; t < tiles; ++t) s += p[(long long)t * lags];
  acov[(long long)g * max_lags + l] = s * norm;
}

// one thread per element: Geyer's steps over the round's lags [lag0, lag0 + lags)
__global__ void lg_geyer_kernel(LgElem* __restrict__ el, int G, const double* __restrict__ acov, int max_lags, int n,
                                int lag0, int lags, long long S, int slot, unsigned long long* __restrict__ head) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  LgElem& e = el[g];
  if (e.done) return;
  head[LGH_ACTIVE] = 1;
  const double* a = acov + (long long)g * max_lags;  // a[t - lag0] = acov at lag t
  Geyer gy = lag0 == 1 ? geyer_start(e.W, e.vp, a[0]) : e.geyer;
  const int end = lag0 + lags - 1;
  while (geyer_running(gy, n) && gy.t + 2 <= end) geyer_step(gy, a[gy.t + 1 - lag0], a[gy.t + 2 - lag0]);
  e.geyer = gy;
  if (!geyer_running(gy, n)) {
    e.done = 1;
    e.ess[slot] = geyer_ess(gy, S);
  }
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

static unsigned blocks_of(long long total, int threads) { return (unsigned)((total + threads - 1) / threads); }

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
  const double norm = 1.0 / ((double)n * Mp);

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
      const int slot = series == 0 ? 0 : series - 1;
      for (int r = 0; r < R.n; ++r) {
        const int lags = R.lags[r], tiles = (int)((S + R.tile[r] - 1) / R.tile[r]);
        lg_lag_kernel<<<dim3((unsigned)((long long)G * tiles), blocks_of(lags, LG_LAG_BLOCK)),
                        std::min(lags, LG_LAG_BLOCK), 0, st>>>(ser, S, n, el, R.lag0[r], lags, R.tile[r], tiles, part);
        lg_acov_kernel<<<dim3(G, blocks_of(lags, 256)), 256, 0, st>>>(part, tiles, lags, el, norm, l.max_lags, acov);
        lg_geyer_kernel<<<blocks_of(G, 128), 128, 0, st>>>(el, G, acov, l.max_lags, n, R.lag0[r], lags, S, slot, head);
        lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_LAGS);
      }
      PSGLA_CUDA_TRY(cudaGetLastError());
    }
    lg_output_kernel<<<blocks_of(G, 128), 128, 0, st>>>(el, G, e0, rhat_dev, ess_bulk_dev, ess_tail_dev);
    PSGLA_CUDA_TRY(cudaGetLastError());
  }
  return PSGLA_OK;
}
