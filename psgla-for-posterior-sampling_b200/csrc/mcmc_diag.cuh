// Device helpers shared by the two convergence-diagnostic paths (mcmc_diag.cu: one CTA per element in shared memory;
// mcmc_diag_large.cu: device-wide, for any S): the normal quantile, numpy's median / quantile of the union of two sorted
// arrays, and Geyer's initial-positive / monotone recurrence as arviz's _ess runs it.
#pragma once
#include <cmath>

#include "common.cuh"

namespace psgla {

// Wichura's AS241 (PPND16): the standard normal quantile to about 1e-16 relative.
static __device__ __forceinline__ double ppnd16(double p) {
  const double q = p - 0.5;
  if (fabs(q) <= 0.425) {
    const double r = 0.180625 - q * q;
    const double num = (((((((2509.0809287301226727 * r + 33430.575583588128105) * r + 67265.770927008700853) * r +
                            45921.953931549871457) * r + 13731.693765509461125) * r + 1971.5909503065514427) * r +
                         133.14166789178437745) * r + 3.387132872796366608);
    const double den = (((((((5226.495278852545925 * r + 28729.085735721942674) * r + 39307.89580009271061) * r +
                            21213.794301586595867) * r + 5394.1960214247511077) * r + 687.1870074920579083) * r +
                         42.313330701600911252) * r + 1.0);
    return q * num / den;
  }
  double r = sqrt(-log(q < 0 ? p : 1.0 - p));
  double num, den;
  if (r <= 5.0) {
    r -= 1.6;
    num = (((((((7.7454501427834140764e-4 * r + 0.0227238449892691845833) * r + 0.24178072517745061177) * r +
               1.27045825245236838258) * r + 3.64784832476320460504) * r + 5.7694972214606914055) * r +
            4.6303378461565452959) * r + 1.42343711074968357734);
    den = (((((((1.05075007164441684324e-9 * r + 5.475938084995344946e-4) * r + 0.0151986665636164571966) * r +
               0.14810397642748007459) * r + 0.68976733498510000455) * r + 1.6763848301838038494) * r +
            2.05319162663775882187) * r + 1.0);
  } else {
    r -= 5.0;
    num = (((((((2.01033439929228813265e-7 * r + 2.71155556874348757815e-5) * r + 0.0012426609473880784386) * r +
               0.026532189526576123093) * r + 0.29656057182850489123) * r + 1.7848265399172913358) * r +
            5.4637849111641143699) * r + 6.6579046435011037772);
    den = (((((((2.04426310338993978564e-15 * r + 1.4215117583164458887e-7) * r + 1.8463183175100546818e-5) * r +
               7.868691311456132591e-4) * r + 0.0148753612908506148525) * r + 0.13692988092273580531) * r +
            0.59983220655588793769) * r + 1.0);
  }
  return q < 0 ? -num / den : num / den;
}

// Normal score of the (half-)integer average rank r = k / 2 among S values: Phi^-1((r - 3/8) / (S + 1/4)), rounded to fp32.
static __device__ __forceinline__ float rank_z(long long k, long long S) {
  return (float)ppnd16((0.5 * (double)k - 0.375) / ((double)S + 0.25));
}

// k-th smallest (0-based) of the union of the sorted arrays a[na] and b[nb]
static __device__ double kth_of_union(const float* a, long long na, const float* b, long long nb, long long k) {
  long long lo = k + 1 - nb > 0 ? k + 1 - nb : 0, hi = k + 1 < na ? k + 1 : na;  // i = how many of the k + 1 smallest from a
  while (lo < hi) {
    const long long i = (lo + hi) >> 1, j = k + 1 - i;
    if (j > 0 && i < na && b[j - 1] > a[i]) lo = i + 1; else hi = i;
  }
  const long long i = lo, j = k + 1 - lo;
  const double x = i > 0 ? (double)a[i - 1] : -INFINITY, y = j > 0 ? (double)b[j - 1] : -INFINITY;
  return fmax(x, y);
}

// numpy's quantile, method "linear": virtual index (n - 1) q, then numpy's _lerp
static __device__ double quantile_linear(const float* a, long long na, const float* b, long long nb, double q) {
  const double h = (double)(na + nb - 1) * q, f = floor(h), t = h - f;
  const long long k = (long long)f;
  const double lo = kth_of_union(a, na, b, nb, k);
  const double hi = k + 1 < na + nb ? kth_of_union(a, na, b, nb, k + 1) : lo;
  const double d = hi - lo;
  return t >= 0.5 ? hi - d * (1.0 - t) : lo + d * t;
}

// Geyer's initial positive sequence P_k = rho_2k + rho_2k+1 (rho_0 = 1) made monotone by a running minimum, with
// rho_t = 1 - (W - acov_t) / var+, acov_t the mean over split chains of the lag-t autocovariances (divisor n).  The steps and
// the term added after the loop are arviz's _ess step for step:
//   Geyer g = geyer_start(W, vp, acov_1);
//   while (geyer_running(g, n)) geyer_step(g, acov_{g.t + 1}, acov_{g.t + 2});
//   ess = geyer_ess(g, S);
struct Geyer {
  double W, vp, even, odd, p_adj, sum_p;
  int t;
};

static __device__ __forceinline__ Geyer geyer_start(double W, double vp, double a1) {
  Geyer g;
  g.W = W, g.vp = vp, g.even = 1.0, g.odd = 1.0 - (W - a1) / vp;
  g.p_adj = g.even + g.odd, g.sum_p = 0.0, g.t = 1;
  return g;
}
static __device__ __forceinline__ bool geyer_running(const Geyer& g, int n) { return g.t < n - 3 && g.even + g.odd > 0.0; }
static __device__ __forceinline__ void geyer_step(Geyer& g, double a_even, double a_odd) {
  g.sum_p += g.p_adj;
  g.even = 1.0 - (g.W - a_even) / g.vp;
  g.odd = 1.0 - (g.W - a_odd) / g.vp;
  g.p_adj = fmin(g.even + g.odd, g.p_adj);
  g.t += 2;
}
static __device__ __forceinline__ double geyer_ess(const Geyer& g, long long S) {
  const double last = (g.even > 0.0 || g.even + g.odd >= 0.0) ? g.even : 0.0;
  const double tau = fmax(-1.0 + 2.0 * g.sum_p + last, 1.0 / log10((double)S));
  return (double)S / tau;
}

}  // namespace psgla
