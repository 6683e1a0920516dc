// The device-wide engine of the convergence diagnostics for any number of split draws per element, shared by
// mcmc_diag_large.cu (split-R-hat, bulk / tail ESS) and mcmc_summary.cu (MCSE, quantiles, HDI): the group layout of the
// workspace, the gather into split-chain order, fp64 chain / element moments of a series and the lag rounds of Geyer's
// recurrence.  mcmc_diag_large.cu describes the stages.
#pragma once
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
static __device__ double lg_block_sum(double v, double* part /* [32] shared */) {
  v = lg_warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) part[warp] = v;
  __syncthreads();
  double s = 0;
  for (int w = 0; w < nw; ++w) s += part[w];
  return s;
}

static __global__ void lg_stamp_kernel(unsigned long long* head, int stage) {
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
static __global__ void __launch_bounds__(256)
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
static __global__ void lg_gather_middle_kernel(const float* __restrict__ draws, int N, int M, long long E, long long e0, int G,
                                        uint32_t* __restrict__ keys, LgElem* __restrict__ el) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= (long long)G * M) return;
  const long long m = k / G, g = k - m * G;
  const float v = draws[((long long)(N / 2) * M + m) * E + e0 + g];
  keys[g * M + m] = float_to_key(v);
  if (isnan(v)) el[g].nan = 1;
}

static __global__ void lg_keys_to_float_kernel(uint32_t* __restrict__ k, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) k[i] = __float_as_uint(key_to_float(k[i]));
}

// one CTA per split chain: fp64 mean and variance (divisor n - 1); the chain is centred in place (fp32)
static __global__ void lg_chain_moments_kernel(float* __restrict__ ser, int n, double* __restrict__ cst) {
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
static __global__ void __launch_bounds__(256)
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
static __global__ void __launch_bounds__(LG_LAG_BLOCK)
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
static __global__ void __launch_bounds__(256)
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
static __global__ void lg_geyer_kernel(LgElem* __restrict__ el, int G, const double* __restrict__ acov, int max_lags, int n,
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

static unsigned blocks_of(long long total, int threads) { return (unsigned)((total + threads - 1) / threads); }

// The lag rounds R of the series ser [G][S] for the elements not done; an element's ESS goes to el[g].ess[slot] when its
// recurrence stops (NaN, from lg_element_moments_kernel, for an element done before).
static void lg_launch_lag_rounds(const LgRounds& R, const LgLayout& l, int G, const float* ser, LgElem* el, double* part,
                                 double* acov, int slot, unsigned long long* head, cudaStream_t st) {
  const long long S = l.S;
  const double norm = 1.0 / ((double)l.n * l.Mp);
  for (int r = 0; r < R.n; ++r) {
    const int lags = R.lags[r], tiles = (int)((S + R.tile[r] - 1) / R.tile[r]);
    lg_lag_kernel<<<dim3((unsigned)((long long)G * tiles), blocks_of(lags, LG_LAG_BLOCK)), std::min(lags, LG_LAG_BLOCK), 0,
                    st>>>(ser, S, l.n, el, R.lag0[r], lags, R.tile[r], tiles, part);
    lg_acov_kernel<<<dim3(G, blocks_of(lags, 256)), 256, 0, st>>>(part, tiles, lags, el, norm, l.max_lags, acov);
    lg_geyer_kernel<<<blocks_of(G, 128), 128, 0, st>>>(el, G, acov, l.max_lags, l.n, R.lag0[r], lags, S, slot, head);
    lg_stamp_kernel<<<1, 1, 0, st>>>(head, LGH_LAGS);
  }
}

}  // namespace psgla
