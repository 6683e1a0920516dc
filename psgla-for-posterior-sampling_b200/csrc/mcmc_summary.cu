// Posterior summary of every element of a multi-chain run, device-wide, as arviz's published functions define it
// (tests/mcmc_summary_reference.py restates them in float64): mean and sd of all N M draws, the ESS of the raw draws and
// its MCSE sd / sqrt(ESS), numpy's linear quantiles with the ESS of the indicator x <= q and arviz's Beta-interval MCSE of
// each, and the highest-density interval.  Input and groups as mcmc_diag_large.cu, on its engine (mcmc_large.cuh); per group
// of G elements, all stream-ordered:
//   gather, sort   the split draws with their split position as payload and the middle draws of odd N, radix-sorted; odd N:
//                  merged into one sorted union of K = S + M draws (the position of a split draw is its index plus the middle
//                  draws below it, of a middle draw its index plus the split draws at or below it: binary searches).  Then
//                  per element (one thread) the quantile of every p.
//   series         the raw draws (scattered to split positions through the payload), then one indicator x <= q_p per p; each
//                  through the engine's fp64 chain / element moments and lag rounds of Geyer's recurrence, its ESS copied
//                  to the element's slot.  After the raw series' chain moments, mean and sd of all K draws (one CTA per
//                  element) from the split chains' fp64 means and variances plus the middle draws.
//   hdi            k = floor(hdi_prob K): one thread per window of the sorted union, width a[i + k] - a[i] in fp64, 8 windows
//                  per thread, a (width, index) arg-min per CTA in np.argmin's order (the first NaN width, from infinite
//                  draws, else the first smallest, ties to the smaller index), then one CTA per element over the CTA partials
//                  (the arg-min is exact, so any order gives the same index).
//   finish         one thread per (element, p): Beta(ess p + 1, ess (1 - p) + 1) quantiles at 0.1586553 and 0.8413447 in
//                  fp64 (beta_ppf below), then the outputs.
// Every sum runs in an order fixed by N, M and the probabilities only: results are bit-identical across calls and do not
// depend on E, on the group an element lands in, or on the other elements.
#include "mcmc_large.cuh"

namespace psgla {

constexpr int SM_MAX_PROBS = 8;       // PSGLA_MCMC_MAX_PROBS
constexpr int SM_HDI_THREADS = 256;
constexpr int SM_HDI_WIN = 8 * SM_HDI_THREADS;  // windows per CTA of the HDI scan

// workspace head: the engine's words, then these stages
// (the merge of odd N, the incomplete-beta evaluations of beta_ppf, their continued-fraction terms, and the most terms one
// (element, p) thread ran, the finishing stage's critical path)
enum { SMH_HDI = LGH_ACTIVE + 1, SMH_FINISH, SMH_MERGE, SMH_BETA_EVALS, SMH_CF_TERMS, SMH_CF_MAX };

struct SmProbs {
  double p[SM_MAX_PROBS];
};

struct SmStat {
  double mean, sd, hdi_lo, hdi_hi;
};

struct HdiMin {
  double w;
  long long i;
};

struct SmLayout {
  LgLayout lg;
  long long K;  // all draws per element: S plus the middle draws of odd N
  int P, hblk;
  size_t q, ess, st, hpart, uni, total;
};

static bool sm_layout(int64_t N, int64_t M, int64_t E, int P, SmLayout& s, LgRounds* R = nullptr) {
  if (P < 1 || P > SM_MAX_PROBS || !lg_layout(N, M, E, s.lg, R)) return false;
  const long long G = s.lg.G;
  s.P = P;
  s.K = s.lg.S + (s.lg.odd ? M : 0);
  s.hblk = (int)((s.K + SM_HDI_WIN - 1) / SM_HDI_WIN);
  size_t o = s.lg.total;
  s.q = o, o += al256((size_t)G * P * sizeof(double));
  s.ess = o, o += al256((size_t)G * (P + 1) * sizeof(double));
  s.st = o, o += al256((size_t)G * sizeof(SmStat));
  s.hpart = o, o += al256((size_t)G * s.hblk * sizeof(HdiMin));
  s.uni = o, o += s.lg.odd ? al256((size_t)(G * s.K) * 4) : 0;
  s.total = o;
  return true;
}

// ------------------------------------------------------------------------------------------- regularised incomplete beta
// z -> lgamma(z) - ((z - 1/2) log z - z + log(2 pi) / 2): Stirling's series, 5 terms (error below 2e-14 for z >= 10)
static __device__ double stirling_tail(double z) {
  const double r = 1.0 / z, r2 = r * r;
  return r * (1.0 / 12 - r2 * (1.0 / 360 - r2 * (1.0 / 1260 - r2 * (1.0 / 1680 - r2 * (1.0 / 1188)))));
}

// log(x^a (1 - x)^b / B(a, b)).  For a, b >= 10 around x0 = a / (a + b): a log x + b log(1 - x) - log B(a, b) is a sum of
// terms of size (a + b) log 2 whose result is O(log(a + b)), so it is written as a log1p(d / x0) + b log1p(-d / y0) plus
// log(x0^a y0^b / B(a, b)) from Stirling's series, in which the large terms cancel analytically: fp64 keeps ~1e-11 absolute
// at a + b = 1e9, where lgamma alone loses 1e-6.
static __device__ double beta_log_front(double a, double b, double x) {
  if (fmin(a, b) >= 10.0) {
    const double s = a + b, x0 = a / s, y0 = b / s, d = x - x0;
    return a * log1p(d / x0) + b * log1p(-d / y0) + 0.5 * log(a / s * b) - 0.91893853320467274178 -
           (stirling_tail(a) + stirling_tail(b) - stirling_tail(s));
  }
  return a * log(x) + b * log1p(-x) - (lgamma(a) + lgamma(b) - lgamma(a + b));
}

// the continued fraction of I_x(a, b) by modified Lentz (Numerical Recipes' betacf), for x < (a + 1) / (a + b + 2)
static __device__ double beta_cf(double a, double b, double x, int maxit, long long* terms) {
  const double tiny = 1e-300, qab = a + b, qap = a + 1.0, qam = a - 1.0;
  double c = 1.0, d = 1.0 - qab * x / qap;
  if (fabs(d) < tiny) d = tiny;
  d = 1.0 / d;
  double h = d;
  int m = 1;
  for (; m <= maxit; ++m) {
    const double m2 = 2.0 * m;
    double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
    d = 1.0 + aa * d;
    if (fabs(d) < tiny) d = tiny;
    c = 1.0 + aa / c;
    if (fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    h *= d * c;
    aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
    d = 1.0 + aa * d;
    if (fabs(d) < tiny) d = tiny;
    c = 1.0 + aa / c;
    if (fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    const double del = d * c;
    h *= del;
    if (fabs(del - 1.0) < 1e-16) break;
  }
  *terms += m < maxit ? m : maxit;
  return h;
}

// I_x(a, b), and the density x^(a-1) (1 - x)^(b-1) / B(a, b) in *dens; the fraction runs on the side of the mean where it
// converges, I_x(a, b) = 1 - I_(1-x)(b, a) beyond it
static __device__ double beta_inc(double a, double b, double x, int maxit, double* dens, long long* terms) {
  const double front = exp(beta_log_front(a, b, x));
  *dens = front / (x * (1.0 - x));
  if (x < (a + 1.0) / (a + b + 2.0)) return front * beta_cf(a, b, x, maxit, terms) / a;
  return 1.0 - front * beta_cf(b, a, 1.0 - x, maxit, terms) / b;
}

// Beta(a, b) quantile at t: Newton from the normal approximation, safeguarded by the bracket [lo, hi] the signs of
// I_x - t maintain (a step leaving it bisects), until a step moves x by at most 1e-13.  The fraction needs
// O(sqrt(max(a, b))) terms near the mean: it is cut at 64 + 8 sqrt(max(a, b)) (2.5e5 at a = 1e9, which the 2D populations
// reach), and Newton at 100 steps (bisection alone reaches 1e-13 in 44).
static __device__ double beta_ppf(double a, double b, double t, int* evals, long long* terms) {
  const int maxit = 64 + (int)(8.0 * sqrt(fmax(a, b)));
  const double s = a + b;
  double lo = 0.0, hi = 1.0, x = a / s + ppnd16(t) * sqrt(a * b / (s * s * (s + 1.0)));
  if (!(x > 0.0 && x < 1.0)) x = 0.5;
  for (int it = 0; it < 100; ++it) {
    double dens;
    const double f = beta_inc(a, b, x, maxit, &dens, terms) - t;
    ++*evals;
    if (f < 0) lo = x; else hi = x;
    double nx = x - f / dens;
    if (!(nx > lo && nx < hi)) nx = 0.5 * (lo + hi);
    const double dx = fabs(nx - x);
    x = nx;
    if (dx <= 1e-13) break;
  }
  return x;
}

// ----------------------------------------------------------------------------------------------------------------- kernels
// odd N: the sorted split draws [G][S] and middle draws [G][M] merged into the sorted union [G][K]
__global__ void sm_merge_kernel(const float* __restrict__ srt, long long S, const float* __restrict__ mid, int M, int G,
                                const LgElem* __restrict__ el, float* __restrict__ uni) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x, na = (long long)G * S, K = S + M;
  if (k >= na + (long long)G * M) return;
  if (k < na) {
    const long long g = k / S, i = k - g * S;
    if (el[g].nan) return;
    const float v = srt[k], *b = mid + g * M;
    int x = 0, y = M;  // middle draws below v
    while (x < y) {
      const int m = (x + y) >> 1;
      if (b[m] < v) x = m + 1; else y = m;
    }
    uni[g * K + i + x] = v;
  } else {
    const long long g = (k - na) / M, j = (k - na) - g * M;
    if (el[g].nan) return;
    const float v = mid[k - na], *a = srt + g * S;
    long long x = 0, y = S;  // split draws at or below v
    while (x < y) {
      const long long m = (x + y) >> 1;
      if (a[m] <= v) x = m + 1; else y = m;
    }
    uni[g * K + x + j] = v;
  }
}

// one thread per element: numpy's linear quantile of every p over the sorted union
__global__ void sm_quantiles_kernel(const float* __restrict__ uni, long long K, int G, SmProbs pr, int P,
                                    const LgElem* __restrict__ el, double* __restrict__ q) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G || el[g].nan) return;
  for (int h = 0; h < P; ++h) q[g * P + h] = quantile_linear(uni + g * K, K, nullptr, 0, pr.p[h]);
}

// series h < 0: the raw draws; h >= 0: the indicator x <= q_h; to the split positions
__global__ void sm_series_kernel(const float* __restrict__ srt, const uint32_t* __restrict__ pay, long long S, long long total,
                                 const LgElem* __restrict__ el, const double* __restrict__ q, int P, int h,
                                 float* __restrict__ ser) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= total) return;
  const long long g = k / S;
  if (el[g].nan) return;
  const float v = srt[k];
  ser[g * S + pay[k]] = h < 0 ? v : ((double)v <= q[g * P + h] ? 1.f : 0.f);
}

// one CTA per element, after the raw series' chain moments: mean and sd (divisor K - 1) of all K draws in fp64,
// sum (x - mean)^2 = sum over split chains of (n - 1) var_c + n (mean_c - mean)^2, plus the middle draws
__global__ void __launch_bounds__(256)
sm_mean_sd_kernel(const double* __restrict__ cst, int Mp, int n, const float* __restrict__ mid, int nm, SmStat* __restrict__ st) {
  __shared__ double part[32];
  const double* c = cst + 2LL * blockIdx.x * Mp;
  const float* b = mid + (long long)blockIdx.x * nm;
  double s = 0, sm = 0;
  for (int k = threadIdx.x; k < Mp; k += blockDim.x) s += c[2 * k];
  for (int j = threadIdx.x; j < nm; j += blockDim.x) sm += b[j];
  s = lg_block_sum(s, part);
  sm = lg_block_sum(sm, part);
  const double K = (double)n * Mp + nm, mean = ((double)n * s + sm) / K;
  double q = 0;
  for (int k = threadIdx.x; k < Mp; k += blockDim.x) {
    const double d = c[2 * k] - mean;
    q += (n - 1.0) * c[2 * k + 1] + n * d * d;
  }
  for (int j = threadIdx.x; j < nm; j += blockDim.x) {
    const double d = b[j] - mean;
    q += d * d;
  }
  q = lg_block_sum(q, part);
  if (threadIdx.x == 0) st[blockIdx.x].mean = mean, st[blockIdx.x].sd = sqrt(q / (K - 1.0));
}

// the engine leaves a series' ESS in el[g].ess[0]; the summary keeps one slot per series
__global__ void sm_take_ess_kernel(const LgElem* __restrict__ el, int G, double* __restrict__ ess, int slots, int slot) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < G) ess[g * slots + slot] = el[g].ess[0];
}

// np.argmin's order over the widths: the first NaN (inf - inf, from infinite draws) if any, else the first smallest width,
// +inf included; i < 0 marks "no window yet"
__device__ __forceinline__ HdiMin hdi_min(HdiMin x, HdiMin y) {
  if (y.i < 0) return x;
  if (x.i < 0) return y;
  const bool xn = isnan(x.w), yn = isnan(y.w);
  if (xn || yn) return (xn && yn) ? (y.i < x.i ? y : x) : (xn ? x : y);
  return (y.w < x.w || (y.w == x.w && y.i < x.i)) ? y : x;
}

// CTA-wide (width, index) arg-min; thread 0 gets it
__device__ HdiMin hdi_block_min(HdiMin v, HdiMin* part /* [32] shared */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    HdiMin u;
    u.w = __shfl_xor_sync(0xffffffffu, v.w, o);
    u.i = __shfl_xor_sync(0xffffffffu, v.i, o);
    v = hdi_min(v, u);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) part[warp] = v;
  __syncthreads();
  for (int w = 0; w < nw; ++w) v = hdi_min(v, part[w]);
  return v;
}

// grid (windows / SM_HDI_WIN, G): the narrowest of the CTA's windows [a_i, a_(i+k)], i < nw = K - k
__global__ void __launch_bounds__(SM_HDI_THREADS)
sm_hdi_kernel(const float* __restrict__ uni, long long K, long long kh, long long nw, const LgElem* __restrict__ el,
              HdiMin* __restrict__ part) {
  __shared__ HdiMin sp[32];
  const int g = blockIdx.y;
  if (el[g].nan) return;
  const float* a = uni + g * K;
  HdiMin best{0.0, -1};
#pragma unroll
  for (int r = 0; r < SM_HDI_WIN / SM_HDI_THREADS; ++r) {
    const long long i = (long long)blockIdx.x * SM_HDI_WIN + r * SM_HDI_THREADS + threadIdx.x;
    if (i < nw) best = hdi_min(best, HdiMin{(double)a[i + kh] - (double)a[i], i});
  }
  best = hdi_block_min(best, sp);
  if (threadIdx.x == 0) part[(long long)g * gridDim.x + blockIdx.x] = best;
}

// one CTA per element: the arg-min over the scan's CTA partials, and the interval
__global__ void __launch_bounds__(256)
sm_hdi_pick_kernel(const HdiMin* __restrict__ part, int nblk, const float* __restrict__ uni, long long K, long long kh,
                   const LgElem* __restrict__ el, SmStat* __restrict__ st) {
  __shared__ HdiMin sp[32];
  const int g = blockIdx.x;
  if (el[g].nan) return;
  HdiMin best{0.0, -1};  // every CTA of the scan had a window: the result is one of them
  for (int b = threadIdx.x; b < nblk; b += blockDim.x) best = hdi_min(best, part[(long long)g * nblk + b]);
  best = hdi_block_min(best, sp);
  if (threadIdx.x == 0) {
    st[g].hdi_lo = uni[g * K + best.i];
    st[g].hdi_hi = uni[g * K + best.i + kh];
  }
}

struct SmOut {
  float *mean, *sd, *mcse_mean, *ess_mean, *q, *mcse_q, *ess_q, *hdi_lo, *hdi_hi;  // q, mcse_q, ess_q: [P][E]
};

// one thread per (element, p): arviz's _mcse_quantile, and for p = 0 the element's other outputs
__global__ void sm_finish_kernel(const LgElem* __restrict__ el, const SmStat* __restrict__ st, const double* __restrict__ q,
                                 const double* __restrict__ ess, const float* __restrict__ uni, long long K, int G, SmProbs pr,
                                 int P, long long E, long long e0, SmOut out, unsigned long long* __restrict__ head) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= G * P) return;
  const int g = k / P, h = k - g * P;
  const long long o = e0 + g, oh = h * E + o;
  if (el[g].nan) {  // arviz: NaN anywhere in the draws gives NaN
    out.q[oh] = out.mcse_q[oh] = out.ess_q[oh] = NAN;
    if (h == 0) out.mean[o] = out.sd[o] = out.mcse_mean[o] = out.ess_mean[o] = out.hdi_lo[o] = out.hdi_hi[o] = NAN;
    return;
  }
  const double e = ess[g * (P + 1) + 1 + h], p = pr.p[h];
  double mcse = NAN;
  if (!isnan(e)) {
    int evals = 0;
    long long terms = 0;
    const double lo = beta_ppf(e * p + 1.0, e * (1.0 - p) + 1.0, 0.1586553, &evals, &terms);
    const double hi = beta_ppf(e * p + 1.0, e * (1.0 - p) + 1.0, 0.8413447, &evals, &terms);
    atomicAdd(head + SMH_BETA_EVALS, (unsigned long long)evals);
    atomicAdd(head + SMH_CF_TERMS, (unsigned long long)terms);
    atomicMax(head + SMH_CF_MAX, (unsigned long long)terms);
    const long long i1 = (long long)rint(fmax(lo * K - 1.0, 0.0));
    long long i2 = (long long)rint(fmin(hi * K - 1.0, K - 1.0));
    if (i2 < 0) i2 += K;  // hi < 0.5 / K (a tiny p at an ESS above ~3.7 K): arviz indexes numpy's a[-1], the largest draw
    mcse = ((double)uni[g * K + i2] - (double)uni[g * K + i1]) / 2.0;
  }
  out.q[oh] = (float)q[g * P + h];
  out.ess_q[oh] = (float)e;
  out.mcse_q[oh] = (float)mcse;
  if (h) return;
  const SmStat& s = st[g];
  const double em = ess[g * (P + 1)];
  out.mean[o] = (float)s.mean;
  out.sd[o] = (float)s.sd;
  out.ess_mean[o] = (float)em;
  out.mcse_mean[o] = (float)(s.sd / sqrt(em));
  out.hdi_lo[o] = (float)s.hdi_lo;
  out.hdi_hi[o] = (float)s.hdi_hi;
}

}  // namespace psgla

using namespace psgla;

extern "C" size_t psgla_mcmc_summary_workspace_bytes(int64_t n_draws, int64_t n_chains, int64_t n_elem, int n_probs) {
  SmLayout s;
  return sm_layout(n_draws, n_chains, n_elem, n_probs, s) ? s.total : 0;
}

extern "C" int psgla_mcmc_summary(const float* draws_dev, int64_t n_draws, int64_t n_chains, int64_t n_elem,
                                  const double* probs_host, int n_probs, double hdi_prob, void* ws_dev, size_t ws_bytes,
                                  float* mean_dev, float* sd_dev, float* mcse_mean_dev, float* ess_mean_dev,
                                  float* quantiles_dev, float* mcse_quantiles_dev, float* ess_quantiles_dev,
                                  float* hdi_low_dev, float* hdi_high_dev, void* stream) {
  PSGLA_REQUIRE(draws_dev && probs_host && ws_dev && mean_dev && sd_dev && mcse_mean_dev && ess_mean_dev && quantiles_dev &&
                    mcse_quantiles_dev && ess_quantiles_dev && hdi_low_dev && hdi_high_dev,
                "psgla_mcmc_summary: null pointer");
  PSGLA_REQUIRE(n_draws >= 4, "psgla_mcmc_summary: n_draws = %lld; split chains need at least 4 draws", (long long)n_draws);
  PSGLA_REQUIRE(n_chains >= 1, "psgla_mcmc_summary: n_chains = %lld must be >= 1", (long long)n_chains);
  PSGLA_REQUIRE(n_elem >= 1 && n_elem <= 0x7fffffffLL, "psgla_mcmc_summary: n_elem = %lld out of range", (long long)n_elem);
  PSGLA_REQUIRE(n_probs >= 1 && n_probs <= SM_MAX_PROBS, "psgla_mcmc_summary: n_probs = %d must be in 1..%d", n_probs,
                SM_MAX_PROBS);
  SmProbs pr;
  for (int h = 0; h < n_probs; ++h) {
    PSGLA_REQUIRE(std::isfinite(probs_host[h]) && probs_host[h] > 0.0 && probs_host[h] < 1.0,
                  "psgla_mcmc_summary: probs[%d] = %g must be in (0, 1)", h, probs_host[h]);
    pr.p[h] = probs_host[h];
  }
  for (int h = n_probs; h < SM_MAX_PROBS; ++h) pr.p[h] = 0.0;
  PSGLA_REQUIRE(std::isfinite(hdi_prob) && hdi_prob > 0.0 && hdi_prob < 1.0,
                "psgla_mcmc_summary: hdi_prob = %g must be in (0, 1)", hdi_prob);
  SmLayout s;
  static thread_local LgRounds R;
  PSGLA_REQUIRE(sm_layout(n_draws, n_chains, n_elem, n_probs, s, &R),
                "psgla_mcmc_summary: %lld chains x %lld draws give more than 2^31 - 1 split draws per element "
                "(S = 2 M floor(N/2)); n_draws or n_chains is out of range",
                (long long)n_chains, (long long)n_draws);
  if (ws_bytes < s.total)
    return set_error(PSGLA_E_WORKSPACE, "psgla_mcmc_summary: workspace of %zu bytes is smaller than the %zu needed", ws_bytes,
                     s.total);
  PSGLA_REQUIRE(((uintptr_t)ws_dev & 255) == 0, "psgla_mcmc_summary: workspace must be 256-byte aligned");

  const LgLayout& l = s.lg;
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
  double* qv = (double*)(ws + s.q);
  double* ess = (double*)(ws + s.ess);
  SmStat* stat = (SmStat*)(ws + s.st);
  HdiMin* hpart = (HdiMin*)(ws + s.hpart);
  const float* srt = (const float*)keys_a;                     // the sorted split draws, after the in-place conversion
  const float* uni = l.odd ? (const float*)(ws + s.uni) : srt;  // the sorted union of all K draws
  float* ser = (float*)keys_b;                                 // the sort's scratch holds the series afterwards

  const int N = (int)n_draws, M = (int)n_chains, n = l.n, Mp = l.Mp, P = n_probs, nm = l.odd ? M : 0;
  const long long S = l.S, E = n_elem, K = s.K;
  const long long kh = (long long)floor(hdi_prob * (double)K), nw = K - kh;
  const int hblk = (int)((nw + SM_HDI_WIN - 1) / SM_HDI_WIN);
  const int mom_threads = n > 1024 ? 256 : 32;
  const SmOut out{mean_dev, sd_dev, mcse_mean_dev, ess_mean_dev, quantiles_dev, mcse_quantiles_dev, ess_quantiles_dev,
                  hdi_low_dev, hdi_high_dev};

  PSGLA_CUDA_TRY(cudaMemsetAsync(head, 0, 256, st));
  lg_stamp_kernel<<<1, 1, 0, st>>>(head, -1);
  for (long long e0 = 0; e0 < E; e0 += l.G) {
    const int G = (int)std::min<long long>(l.G, E - e0);
    const long long total = (long long)G * S;
    PSGLA_CUDA_TRY(cudaMemsetAsync(el, 0, (size_t)G * sizeof(LgElem), st));
    lg_gather_kernel<<<dim3(blocks_of(S, 32), blocks_of(G, 32)), dim3(32, 8), 0, st>>>(draws_dev, N, M, E, e0, G, S, n,
                                                                                       keys_a, pay_a, el);
    if (l.odd) lg_gather_middle_kernel<<<blocks_of((long long)G * M, 256), 256, 0, st>>>(draws_dev, N, M, E, e0, G, mid_a, el);
    lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_GATHER);

    radix_sort_segments(keys_a, keys_b, pay_a, pay_b, S, G, hist, st);
    lg_keys_to_float_kernel<<<blocks_of(total, 256), 256, 0, st>>>(keys_a, total);
    if (l.odd) {
      radix_sort_segments(mid_a, mid_b, nullptr, nullptr, M, G, hist, st);
      lg_keys_to_float_kernel<<<blocks_of((long long)G * M, 256), 256, 0, st>>>(mid_a, (long long)G * M);
      lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_SORT);
      sm_merge_kernel<<<blocks_of((long long)G * K, 256), 256, 0, st>>>(srt, S, (const float*)mid_a, M, G, el,
                                                                         (float*)(ws + s.uni));
      lg_stamp_kernel<<<1, 1, 0, st>>>(head, SMH_MERGE);
    }
    sm_quantiles_kernel<<<blocks_of(G, 128), 128, 0, st>>>(uni, K, G, pr, P, el, qv);
    PSGLA_CUDA_TRY(cudaGetLastError());
    lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_SORT);

    // series -1: the raw draws; h >= 0: x <= q_h
    for (int h = -1; h < P; ++h) {
      sm_series_kernel<<<blocks_of(total, 256), 256, 0, st>>>(srt, pay_a, S, total, el, qv, P, h, ser);
      lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_RANK);
      lg_chain_moments_kernel<<<(unsigned)((long long)G * Mp), mom_threads, 0, st>>>(ser, n, cst);
      lg_element_moments_kernel<<<G, 256, 0, st>>>(cst, Mp, n, el, 0);
      if (h < 0) sm_mean_sd_kernel<<<G, 256, 0, st>>>(cst, Mp, n, (const float*)mid_a, nm, stat);
      PSGLA_CUDA_TRY(cudaGetLastError());
      lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_MOMENTS);
      lg_launch_lag_rounds(R, l, G, ser, el, part, acov, 0, head, st);
      sm_take_ess_kernel<<<blocks_of(G, 128), 128, 0, st>>>(el, G, ess, P + 1, h + 1);
      PSGLA_CUDA_TRY(cudaGetLastError());
    }

    sm_hdi_kernel<<<dim3(hblk, G), SM_HDI_THREADS, 0, st>>>(uni, K, kh, nw, el, hpart);
    sm_hdi_pick_kernel<<<G, 256, 0, st>>>(hpart, hblk, uni, K, kh, el, stat);
    PSGLA_CUDA_TRY(cudaGetLastError());
    lg_stamp_kernel<<<1, 1, 0, st>>>(head, SMH_HDI);
    sm_finish_kernel<<<blocks_of((long long)G * P, 64), 64, 0, st>>>(el, stat, qv, ess, uni, K, G, pr, P, E, e0, out,
                                                                        head);
    PSGLA_CUDA_TRY(cudaGetLastError());
    lg_stamp_kernel<<<1, 1, 0, st>>>(head, SMH_FINISH);
  }
  return PSGLA_OK;
}
