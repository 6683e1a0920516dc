// 2D Gaussian-mixture posterior sampling: PSGLA (SnoPnP_ULA) and PnP-ULA as one register-resident kernel.
//
// Replaces the Python loops sampling_2D.py:21-45 / :48-72, the data-fidelity score sampling_2D.py:30-31 and the
// closed-form MMSE denoiser utils_2D.py:209-233 of the reference.  One thread owns CPT chains for all n_steps:
// state, Philox counter and step constants live in registers / the constant bank; HBM sees x_0 once, the final
// state once, and (optionally) a thinned trajectory.  Bound: FP32 + MUFU issue, not memory (DESIGN.md, "2D kernel").
//
// Algebra (all folding done on the host in double, see fold_problem):
//   score(x) = A^T (y - A x) / sigma^2 = bb - G x
//   tau      = sqrt(eps)           (the reference feeds sqrt(epsilon) where a variance belongs, utils_2D.py:223-226;
//                                   PSGLA calls the denoiser with eps = delta, sampling_2D.py:63)
//   D(v)     = sum_i w_i(v) (M_i v + b_i),  w = softmax_i( kappa_i - 1/2 (v-mu_i)^T S_i (v-mu_i) )
//              S_i = (tau I + Sigma_i)^-1, kappa_i = log pi_i - 1/2 log det(tau I + Sigma_i),
//              M_i = (I/tau + Sigma_i^-1)^-1 / tau, b_i = (I/tau + Sigma_i^-1)^-1 Sigma_i^-1 mu_i
//   PSGLA  : x+ = D(P x + q + cn z),            P = I - (delta/alpha) G, q = (delta/alpha) bb, cn = sqrt(2 delta)
//   PnP-ULA: x+ = P x + q + cn z + cp D(x),     P = (1 - cp) I - delta G, q = delta bb, cp = alpha delta / eps
// The reference evaluates the softmax with plain exp() and can hit 0/0 far from every mode; here the logits are
// carried in log2 units and normalised (r == 2: a single sigmoid of the logit *difference*, which is itself a
// quadratic in v; r > 2: online log-sum-exp over the components held in shared memory).
#include <algorithm>
#include <cmath>
#include <cstring>

#include "common.cuh"

namespace psgla {

constexpr int RMAX = PSGLA_GMM_MAX_COMPONENTS;

// gmm2d_lean_kernel's geometry: 4 Philox counter blocks (8 steps) per round, 64-thread blocks, 16 of them resident per SM.
constexpr int LEAN_NB = 4, LEAN_BLOCK = 64, LEAN_MINB = 16;

// Philox's launch-uniform words of gmm2d_lean_kernel's counter blocks after round 2 (see the kernel), one entry per round:
// component b of each vector belongs to counter pair pair0 + r LEAN_NB + b.  Passed BY VALUE as a kernel parameter, so each
// launch (and each stream: several cells may run at once) carries its own table, read through the uniform datapath.  12 B per
// counter pair; kernel parameters may take 32 764 B, of which the kernel's other parameters take less than 256.
struct LeanPairWords {
  struct Round {
    uint4 ua, ub, uc;
  } r[(32764 - 256) / (3 * 16)];  // 677 rounds (5 416 steps) per launch
};
constexpr int LEAN_TAB_ROUNDS = sizeof(LeanPairWords) / sizeof(LeanPairWords::Round);
static_assert(LEAN_NB == 4, "one uint4 per LEAN_NB counter pairs");

template <typename T>
struct Gmm2dConsts {
  T P[4], q[2];
  T cn, cp;
  // r == 2 fast path: t(v) = l_1(v) - l_0(v) in log2 units, D = m_1 + sigmoid * (m_0 - m_1)
  T tq[6];
  T M1[4], b1[2], dM[4], db[2];
  int r;
};

template <typename T>
struct Gmm2dComponents {  // general-r path, staged into shared memory
  T mu[RMAX][2];
  T s[RMAX][3];  // 1/2 log2(e) S00, log2(e) S01, 1/2 log2(e) S11
  T kappa2[RMAX];
  T M[RMAX][4];
  T b[RMAX][2];
};

// ------------------------------------------------------------------------------------------------ math helpers
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ double fast_exp2(double x) { return exp2(x); }
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ double fast_rcp(double x) { return 1.0 / x; }
__device__ __forceinline__ float fma_(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_(double a, double b, double c) { return fma(a, b, c); }

template <typename T>
struct Vec2;
template <>
struct Vec2<float> {
  using type = float2;
};
template <>
struct Vec2<double> {
  using type = double2;
};

// D(v) for r == 2: everything comes from the constant bank as FFMA operands.
template <typename T>
__device__ __forceinline__ void denoise_r2(const Gmm2dConsts<T>& c, T v0, T v1, T& d0, T& d1) {
  const T t = fma_(v0, fma_(c.tq[3], v0, fma_(c.tq[4], v1, c.tq[1])), fma_(v1, fma_(c.tq[5], v1, c.tq[2]), c.tq[0]));
  const T w0 = fast_rcp(T(1) + fast_exp2(t));  // weight of component 0
  const T m0 = fma_(c.M1[0], v0, fma_(c.M1[1], v1, c.b1[0]));
  const T m1 = fma_(c.M1[2], v0, fma_(c.M1[3], v1, c.b1[1]));
  const T e0 = fma_(c.dM[0], v0, fma_(c.dM[1], v1, c.db[0]));
  const T e1 = fma_(c.dM[2], v0, fma_(c.dM[3], v1, c.db[1]));
  d0 = fma_(w0, e0, m0);
  d1 = fma_(w0, e1, m1);
}

// D(v) for general r: online log-sum-exp over components in shared memory (broadcast LDS).
template <typename T>
__device__ __forceinline__ void denoise_general(const Gmm2dComponents<T>* __restrict__ k, int r, T v0, T v1, T& d0,
                                                T& d1) {
  T mx = -INFINITY, den = 0, a0 = 0, a1 = 0;
  for (int i = 0; i < r; ++i) {
    const T e0 = v0 - k->mu[i][0], e1 = v1 - k->mu[i][1];
    const T l = k->kappa2[i] - fma_(k->s[i][0] * e0, e0, fma_(k->s[i][1] * e0, e1, k->s[i][2] * e1 * e1));
    const T m0 = fma_(k->M[i][0], v0, fma_(k->M[i][1], v1, k->b[i][0]));
    const T m1 = fma_(k->M[i][2], v0, fma_(k->M[i][3], v1, k->b[i][1]));
    const T nmx = l > mx ? l : mx;
    const T scale = fast_exp2(mx - nmx);  // exp2(-inf) = 0 on the first component
    const T w = fast_exp2(l - nmx);
    den = fma_(den, scale, w);
    a0 = fma_(a0, scale, w * m0);
    a1 = fma_(a1, scale, w * m1);
    mx = nmx;
  }
  const T inv = T(1) / den;
  d0 = a0 * inv;
  d1 = a1 * inv;
}

template <typename T, int ALG, bool R2>
__device__ __forceinline__ void langevin_step(const Gmm2dConsts<T>& c, const Gmm2dComponents<T>* __restrict__ comps,
                                              T& x0, T& x1, T z0, T z1) {
  const T l0 = fma_(c.P[0], x0, fma_(c.P[1], x1, fma_(c.cn, z0, c.q[0])));
  const T l1 = fma_(c.P[2], x0, fma_(c.P[3], x1, fma_(c.cn, z1, c.q[1])));
  const T v0 = (ALG == PSGLA_ALG_PSGLA) ? l0 : x0;
  const T v1 = (ALG == PSGLA_ALG_PSGLA) ? l1 : x1;
  T d0, d1;
  if (R2)
    denoise_r2(c, v0, v1, d0, d1);
  else
    denoise_general(comps, c.r, v0, v1, d0, d1);
  if (ALG == PSGLA_ALG_PSGLA) {
    x0 = d0;
    x1 = d1;
  } else {
    x0 = fma_(c.cp, d0, l0);
    x1 = fma_(c.cp, d1, l1);
  }
}

// ------------------------------------------------------------------------------------------------ packed fp32 pairs
// sm_100 issues two fp32 FMAs per lane as ONE instruction (FFMA2, PTX fma.rn.f32x2).  The lean kernel is issue-bound, so it
// runs the Box-Muller arithmetic of two Philox counter blocks as pairs: each 64-bit register holds the same quantity of both
// blocks and costs one instruction instead of two.  The operations and their order per value are those of box_muller
// (common.cuh): results are bit-identical to the scalar path.
typedef unsigned long long pk2;  // {lo, hi}
__device__ __forceinline__ pk2 pk(float lo, float hi) {
  pk2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpk(pk2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ pk2 fma2(pk2 a, pk2 b, pk2 c) {
  pk2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ pk2 mul2(pk2 a, pk2 b) {
  pk2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// box_muller (common.cuh) on the same word of two counter blocks at once: (a, b) of block A and of block B.
__device__ __forceinline__ void box_muller_pk(uint32_t aA, uint32_t bA, uint32_t aB, uint32_t bB, pk2& z0, pk2& z1) {
  const pk2 u1 = fma2(pk((float)aA, (float)aB), pk(2.3283064365386963e-10f, 2.3283064365386963e-10f),
                      pk(1.1641532182693481e-10f, 1.1641532182693481e-10f));
  const pk2 th = fma2(pk((float)bA, (float)bB), pk(1.4629180792671596e-9f, 1.4629180792671596e-9f),
                      pk(7.314590396335798e-10f, 7.314590396335798e-10f));
  float ua, ub, la, lb, ra, rb, ta, tb;
  unpk(u1, ua, ub);
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(la) : "f"(ua));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lb) : "f"(ub));
  unpk(mul2(pk(la, lb), pk(-1.3862943611198906f, -1.3862943611198906f)), ua, ub);
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(ra) : "f"(ua));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rb) : "f"(ub));
  unpk(th, ta, tb);
  float sa, ca, sb, cb;
  __sincosf(ta, &sa, &ca);
  __sincosf(tb, &sb, &cb);
  const pk2 r = pk(ra, rb);
  z0 = mul2(r, pk(ca, cb));
  z1 = mul2(r, pk(sa, sb));
}

// ------------------------------------------------------------------------------------------------ the kernel
// Chain j of thread g is chain index g + j * (gridDim.x * blockDim.x): every global access is coalesced.
// Philox mode draws NB counter blocks (= 2 NB steps) of every owned chain at once: the 10-round integer pipeline of the NB x CPT
// independent blocks is where the instruction-level parallelism comes from, so a thread that owns ONE chain (small populations,
// and the 1-warp blocks of the dynamically scheduled launch) still keeps the pipes busy between the dependent Langevin steps.
template <typename T, int ALG, bool R2, int CPT, int NB, int BLOCK>
__global__ void __launch_bounds__(BLOCK, (sizeof(T) == 4 && R2) ? 1024 / BLOCK : 1)
gmm2d_kernel(const Gmm2dConsts<T> c, const Gmm2dComponents<T>* __restrict__ comps_gmem, T* __restrict__ x,
             long long n_chains, long long chain_lo, long long n_launch, unsigned long long chain_id0, long long n_steps,
             long long step0, const PhiloxKeys keys, const T* __restrict__ noise, T* __restrict__ traj, long long thin) {
  // This launch owns chains [chain_lo, chain_lo + n_launch) of the call's n_chains (the stride of noise / traj rows).
  using V2 = typename Vec2<T>::type;
  __shared__ Gmm2dComponents<T> comps_smem;
  const Gmm2dComponents<T>* comps = nullptr;
  if (!R2) {
    const int nwords = sizeof(Gmm2dComponents<T>) / 4;
    for (int i = threadIdx.x; i < nwords; i += blockDim.x)
      reinterpret_cast<uint32_t*>(&comps_smem)[i] = reinterpret_cast<const uint32_t*>(comps_gmem)[i];
    __syncthreads();
    comps = &comps_smem;
  }
  const long long nthreads = (long long)gridDim.x * blockDim.x;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;

  T x0[CPT], x1[CPT];
  bool live[CPT];
#pragma unroll
  for (int j = 0; j < CPT; ++j) {
    const long long ch = chain_lo + g + j * nthreads;
    live[j] = g + j * nthreads < n_launch;
    V2 v = live[j] ? reinterpret_cast<const V2*>(x)[ch] : V2{0, 0};
    x0[j] = v.x;
    x1[j] = v.y;
  }

  long long keep_in = thin;  // steps until the next trajectory row
  long long row = 0;
  auto after_step = [&](void) {
    if (traj != nullptr) {
      if (--keep_in == 0) {
        keep_in = thin;
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
          const long long ch = chain_lo + g + j * nthreads;
          if (live[j]) reinterpret_cast<V2*>(traj)[row * n_chains + ch] = V2{x0[j], x1[j]};
        }
        ++row;
      }
    }
  };

  if (noise != nullptr) {
    // replay: the caller's N(0,1) draws (the reference's np.random.randn(2) per step, sampling_2D.py:35,62)
    for (long long k = 0; k < n_steps; ++k) {
#pragma unroll
      for (int j = 0; j < CPT; ++j) {
        const long long ch = chain_lo + g + j * nthreads;
        if (live[j]) {
          const V2 z = reinterpret_cast<const V2*>(noise)[k * n_chains + ch];
          langevin_step<T, ALG, R2>(c, comps, x0[j], x1[j], z.x, z.y);
        }
      }
      after_step();
    }
  } else {
    long long t = step0;
    const long long t_end = step0 + n_steps;
    unsigned long long sub[CPT];
#pragma unroll
    for (int j = 0; j < CPT; ++j) sub[j] = chain_id0 + (unsigned long long)(chain_lo + g + j * nthreads);
    // one counter block = the normals of steps 2 * pair and 2 * pair + 1; `first` / `second`: which of the two are taken
    auto one_block = [&](bool first, bool second) {
      float z[CPT][4];
      const unsigned long long pair = (unsigned long long)t >> 1;
#pragma unroll
      for (int j = 0; j < CPT; ++j)
        philox_normal4_keyed(keys, sub[j], (uint32_t)pair, (uint32_t)(pair >> 32), z[j][0], z[j][1], z[j][2], z[j][3]);
      if (first) {
#pragma unroll
        for (int j = 0; j < CPT; ++j) langevin_step<T, ALG, R2>(c, comps, x0[j], x1[j], T(z[j][0]), T(z[j][1]));
        after_step();
        ++t;
      }
      if (second) {
#pragma unroll
        for (int j = 0; j < CPT; ++j) langevin_step<T, ALG, R2>(c, comps, x0[j], x1[j], T(z[j][2]), T(z[j][3]));
        after_step();
        ++t;
      }
    };
    if (t < t_end && (t & 1)) one_block(false, true);  // a segment that starts on the second half of a counter block
    while (t + 2 * NB <= t_end) {
      float z[NB][CPT][4];
      const unsigned long long pair = (unsigned long long)t >> 1;
#pragma unroll
      for (int b = 0; b < NB; ++b)
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
          const unsigned long long pr = pair + b;
          philox_normal4_keyed(keys, sub[j], (uint32_t)pr, (uint32_t)(pr >> 32), z[b][j][0], z[b][j][1], z[b][j][2], z[b][j][3]);
        }
#pragma unroll
      for (int b = 0; b < NB; ++b) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
#pragma unroll
          for (int j = 0; j < CPT; ++j)
            langevin_step<T, ALG, R2>(c, comps, x0[j], x1[j], T(z[b][j][2 * h]), T(z[b][j][2 * h + 1]));
          after_step();
        }
      }
      t += 2 * NB;
    }
    while (t < t_end) one_block(true, t + 1 < t_end);  // fewer than 2 NB steps left
  }

#pragma unroll
  for (int j = 0; j < CPT; ++j) {
    const long long ch = chain_lo + g + j * nthreads;
    if (live[j]) reinterpret_cast<V2*>(x)[ch] = V2{x0[j], x1[j]};
  }
}

// Structure of the folded constants.  The kernel is bound by the FMA pipe (scripts/pipe_rates.py: an FFMA costs the pipe 1
// cycle per warp, each of Philox's ten IMAD.WIDE.U32 pairs 4), so FMAs whose coefficient is exactly zero are worth removing:
//   STRUCT 1: P diagonal (A^T A diagonal -- every cell of the reference's experiment has A = I, sampling_2D.py:84);
//   STRUCT 2: additionally M_i, M_0 - M_1 diagonal and no v0 v1 term in the logit (isotropic / axis-aligned covariances: the
//             "symetric_gaussians" and "disymmetric_gaussians" priors, utils_2D.py:28-33): 15 FP32 instructions per step
//             instead of 24.
// fma(0, a, b) == b for finite a, so dropping those terms leaves every result bit-identical to the general path.
template <int ALG, int STRUCT>
__device__ __forceinline__ void langevin_step_s(const Gmm2dConsts<float>& c, float& x0, float& x1, float z0, float z1) {
  float l0, l1;
  if (STRUCT >= 1) {
    l0 = fmaf(c.P[0], x0, fmaf(c.cn, z0, c.q[0]));
    l1 = fmaf(c.P[3], x1, fmaf(c.cn, z1, c.q[1]));
  } else {
    l0 = fmaf(c.P[0], x0, fmaf(c.P[1], x1, fmaf(c.cn, z0, c.q[0])));
    l1 = fmaf(c.P[2], x0, fmaf(c.P[3], x1, fmaf(c.cn, z1, c.q[1])));
  }
  const float v0 = (ALG == PSGLA_ALG_PSGLA) ? l0 : x0;
  const float v1 = (ALG == PSGLA_ALG_PSGLA) ? l1 : x1;
  float d0, d1;
  if (STRUCT >= 2) {
    const float t = fmaf(v0, fmaf(c.tq[3], v0, c.tq[1]), fmaf(v1, fmaf(c.tq[5], v1, c.tq[2]), c.tq[0]));
    const float w0 = fast_rcp(1.0f + fast_exp2(t));
    const float m0 = fmaf(c.M1[0], v0, c.b1[0]);
    const float m1 = fmaf(c.M1[3], v1, c.b1[1]);
    const float e0 = fmaf(c.dM[0], v0, c.db[0]);
    const float e1 = fmaf(c.dM[3], v1, c.db[1]);
    d0 = fmaf(w0, e0, m0);
    d1 = fmaf(w0, e1, m1);
  } else {
    denoise_r2(c, v0, v1, d0, d1);
  }
  if (ALG == PSGLA_ALG_PSGLA) {
    x0 = d0;
    x1 = d1;
  } else {
    x0 = fmaf(c.cp, d0, l0);
    x1 = fmaf(c.cp, d1, l1);
  }
}

static int constants_structure(const Gmm2dConsts<float>& c) {
  if (c.P[1] != 0.0f || c.P[2] != 0.0f) return 0;
  if (c.M1[1] != 0.0f || c.M1[2] != 0.0f || c.dM[1] != 0.0f || c.dM[2] != 0.0f || c.tq[4] != 0.0f) return 1;
  return 2;
}

// ------------------------------------------------------------------------------------------------ the lean kernel
// fp32, r == 2, in-kernel Philox, no trajectory: the throughput path and nothing else, so that it fits a register budget
// that keeps more warps resident than the general kernel's 64 registers allow (the general kernel spends ~20 registers on
// 64-bit bookkeeping of the optional replay / trajectory paths).  One chain per thread; each round draws LEAN_NB counter
// blocks (2 LEAN_NB steps), with the Box-Muller arithmetic of two blocks packed into FFMA2 / FMUL2.  Same Philox counters,
// same arithmetic per chain as gmm2d_kernel: bit-identical results.
template <int ALG, int STRUCT>
__global__ void __launch_bounds__(LEAN_BLOCK, LEAN_MINB)
gmm2d_lean_kernel(const Gmm2dConsts<float> c, float2* __restrict__ x, unsigned n_launch, uint32_t sub0_lo, uint32_t pair0_hi,
                  int n_rounds, const PhiloxKeys keys, const LeanPairWords tab) {
  static_assert(LEAN_NB % 2 == 0, "Box-Muller packs counter blocks in pairs");
  const unsigned g = blockIdx.x * LEAN_BLOCK + threadIdx.x;
  if (g >= n_launch) return;
  float2 v = x[g];
  float x0 = v.x, x1 = v.y;
  // The launch's chain ids share their high word s_hi, and so do its counter pairs (launch_lean_body splits where they would
  // not), so Philox's counter words c1 = pair >> 32 and c3 = s_hi are launch constants and its first two rounds are thread
  // constants (T) and values that depend only on the counter pair and the launch (U):
  //   round 1: c0' = hi(M1 s_lo) ^ c1 ^ k0 (T), c1' = lo(M1 s_lo) (T), c2' = hi(M0 pair) ^ s_hi ^ k1 (U), c3' = lo(M0 pair) (U)
  //   round 2: M0 c0' (T) and M1 c2' (U)
  // The host computes the U words after round 2 (ua = hi(M1 c2') ^ k2, ub = lo(M1 c2'), uc = c3' ^ k3) into `tab`, so per
  // thread and per counter block rounds 1-2 cost no IMAD.WIDE.U32 and two LOP3: 16 per block, the floor for rounds 3-10.  Same
  // words as philox4x32_10_keyed from round 0, i.e. bit-identical draws.
  const uint32_t s_lo = sub0_lo + g;
  const uint64_t t1 = (uint64_t)0xCD9E8D57u * s_lo;               // round 1, chain word
  const uint32_t t1_lo = (uint32_t)t1;
  const uint64_t t2 = (uint64_t)0xD2511F53u * ((uint32_t)(t1 >> 32) ^ pair0_hi ^ keys.k[0]);  // round 2, first product
  const uint32_t t2_hi = (uint32_t)(t2 >> 32), t2_lo = (uint32_t)t2;
  for (int r = 0; r < n_rounds; ++r) {
    const uint4 ua = tab.r[r].ua, ub = tab.r[r].ub, uc = tab.r[r].uc;
    const uint32_t wa[LEAN_NB] = {ua.x, ua.y, ua.z, ua.w}, wb[LEAN_NB] = {ub.x, ub.y, ub.z, ub.w},
                   wc[LEAN_NB] = {uc.x, uc.y, uc.z, uc.w};
    uint32_t w[LEAN_NB][4];  // Philox4x32-10 of counter blocks pair0 + r LEAN_NB .. + LEAN_NB - 1
#pragma unroll
    for (int b = 0; b < LEAN_NB; ++b) {
      w[b][0] = wa[b] ^ t1_lo;
      w[b][1] = wb[b];
      w[b][2] = t2_hi ^ wc[b];
      w[b][3] = t2_lo;
      philox4x32_10_keyed<2>(w[b][0], w[b][1], w[b][2], w[b][3], keys);
    }
    float z[LEAN_NB][4];
#pragma unroll
    for (int b = 0; b < LEAN_NB; b += 2) {
      pk2 q0, q1, q2, q3;
      box_muller_pk(w[b][0], w[b][1], w[b + 1][0], w[b + 1][1], q0, q1);
      box_muller_pk(w[b][2], w[b][3], w[b + 1][2], w[b + 1][3], q2, q3);
      unpk(q0, z[b][0], z[b + 1][0]);
      unpk(q1, z[b][1], z[b + 1][1]);
      unpk(q2, z[b][2], z[b + 1][2]);
      unpk(q3, z[b][3], z[b + 1][3]);
    }
#pragma unroll
    for (int b = 0; b < LEAN_NB; ++b) {
      langevin_step_s<ALG, STRUCT>(c, x0, x1, z[b][0], z[b][1]);
      langevin_step_s<ALG, STRUCT>(c, x0, x1, z[b][2], z[b][3]);
    }
  }
  x[g] = float2{x0, x1};
}

template <typename T, bool R2>
__global__ void gmm2d_denoise_kernel(const Gmm2dConsts<T> c, const Gmm2dComponents<T>* __restrict__ comps_gmem,
                                     const T* __restrict__ x, T* __restrict__ out, long long n) {
  using V2 = typename Vec2<T>::type;
  __shared__ Gmm2dComponents<T> comps_smem;
  const int nwords = sizeof(Gmm2dComponents<T>) / 4;
  for (int i = threadIdx.x; i < nwords; i += blockDim.x)
    reinterpret_cast<uint32_t*>(&comps_smem)[i] = reinterpret_cast<const uint32_t*>(comps_gmem)[i];
  __syncthreads();
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  const V2 v = reinterpret_cast<const V2*>(x)[g];
  T d0, d1;
  if (R2)
    denoise_r2(c, v.x, v.y, d0, d1);
  else
    denoise_general(&comps_smem, c.r, v.x, v.y, d0, d1);
  reinterpret_cast<V2*>(out)[g] = V2{d0, d1};
}

__global__ void gmm2d_noise_kernel(float* __restrict__ out, long long n_chains, unsigned long long chain_id0,
                                   long long n_steps, long long step0, unsigned long long seed) {
  const long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= n_chains) return;
  for (long long k = 0; k < n_steps; ++k) {
    const unsigned long long t = (unsigned long long)(step0 + k), pair = t >> 1;
    float z0, z1, z2, z3;
    philox_normal4(seed, chain_id0 + (unsigned long long)ch, (uint32_t)pair, (uint32_t)(pair >> 32), z0, z1, z2, z3);
    reinterpret_cast<float2*>(out)[k * n_chains + ch] = (t & 1) ? float2{z2, z3} : float2{z0, z1};
  }
}

// ------------------------------------------------------------------------------------------------ host folding
struct Mat2 {
  double a, b, c, d;  // [[a b][c d]]
};
static inline Mat2 inv2(const Mat2& m) {
  const double det = m.a * m.d - m.b * m.c;
  return {m.d / det, -m.b / det, -m.c / det, m.a / det};
}
static inline double det2(const Mat2& m) { return m.a * m.d - m.b * m.c; }

struct Folded {
  Gmm2dConsts<double> c;
  Gmm2dComponents<double> k;
};

static int fold_problem(const psgla_gmm2d_problem* p, double eps, bool linear_part, Folded* out) {
  const int r = p->n_components;
  if (r < 1 || r > RMAX) return set_error(PSGLA_E_UNSUPPORTED, "n_components=%d outside 1..%d", r, RMAX);
  if (!(eps > 0)) return set_error(PSGLA_E_BADARG, "denoiser level must be > 0 (got %g)", eps);
  std::memset(out, 0, sizeof(*out));
  const double LOG2E = 1.4426950408889634;
  const double tau = std::sqrt(eps);
  Gmm2dConsts<double>& c = out->c;
  Gmm2dComponents<double>& k = out->k;
  c.r = r;
  double lq[RMAX][6];
  for (int i = 0; i < r; ++i) {
    const Mat2 Sig{p->Sigma[i][0], p->Sigma[i][1], p->Sigma[i][2], p->Sigma[i][3]};
    if (!(det2(Sig) > 0) || !(Sig.a > 0) || !(p->pi[i] > 0))
      return set_error(PSGLA_E_BADARG, "component %d: Sigma must be SPD and pi > 0", i);
    const Mat2 Sinv = inv2(Sig);
    const Mat2 St = inv2({tau + Sig.a, Sig.b, Sig.c, tau + Sig.d});
    const double kappa = std::log(p->pi[i]) - 0.5 * std::log(det2({tau + Sig.a, Sig.b, Sig.c, tau + Sig.d}));
    const Mat2 Pm = inv2({1.0 / tau + Sinv.a, Sinv.b, Sinv.c, 1.0 / tau + Sinv.d});
    const double m0 = p->mu[i][0], m1 = p->mu[i][1];
    const double sm0 = Sinv.a * m0 + Sinv.b * m1, sm1 = Sinv.c * m0 + Sinv.d * m1;
    k.mu[i][0] = m0;
    k.mu[i][1] = m1;
    k.s[i][0] = 0.5 * LOG2E * St.a;
    k.s[i][1] = 0.5 * LOG2E * (St.b + St.c);
    k.s[i][2] = 0.5 * LOG2E * St.d;
    k.kappa2[i] = kappa * LOG2E;
    k.M[i][0] = Pm.a / tau;
    k.M[i][1] = Pm.b / tau;
    k.M[i][2] = Pm.c / tau;
    k.M[i][3] = Pm.d / tau;
    k.b[i][0] = Pm.a * sm0 + Pm.b * sm1;
    k.b[i][1] = Pm.c * sm0 + Pm.d * sm1;
    // l_i(v) = lq0 + lq1 v0 + lq2 v1 + lq3 v0^2 + lq4 v0 v1 + lq5 v1^2
    const double s00 = k.s[i][0], s01 = k.s[i][1], s11 = k.s[i][2];
    lq[i][0] = k.kappa2[i] - (s00 * m0 * m0 + s01 * m0 * m1 + s11 * m1 * m1);
    lq[i][1] = 2 * s00 * m0 + s01 * m1;
    lq[i][2] = 2 * s11 * m1 + s01 * m0;
    lq[i][3] = -s00;
    lq[i][4] = -s01;
    lq[i][5] = -s11;
  }
  if (r == 2) {
    for (int j = 0; j < 6; ++j) c.tq[j] = lq[1][j] - lq[0][j];
    for (int j = 0; j < 4; ++j) {
      c.M1[j] = k.M[1][j];
      c.dM[j] = k.M[0][j] - k.M[1][j];
    }
    for (int j = 0; j < 2; ++j) {
      c.b1[j] = k.b[1][j];
      c.db[j] = k.b[0][j] - k.b[1][j];
    }
  }
  if (linear_part) {
    if (!(p->delta > 0) || !(p->sigma != 0) || !(p->alpha != 0))
      return set_error(PSGLA_E_BADARG, "delta must be > 0, sigma and alpha non-zero");
    const double s2 = p->sigma * p->sigma;
    const double* A = p->A;
    const Mat2 G{(A[0] * A[0] + A[2] * A[2]) / s2, (A[0] * A[1] + A[2] * A[3]) / s2, (A[1] * A[0] + A[3] * A[2]) / s2,
                 (A[1] * A[1] + A[3] * A[3]) / s2};
    const double bb0 = (A[0] * p->y[0] + A[2] * p->y[1]) / s2, bb1 = (A[1] * p->y[0] + A[3] * p->y[1]) / s2;
    c.cn = std::sqrt(2 * p->delta);
    if (p->alg == PSGLA_ALG_PSGLA) {
      const double cs = p->delta / p->alpha;
      c.P[0] = 1 - cs * G.a;
      c.P[1] = -cs * G.b;
      c.P[2] = -cs * G.c;
      c.P[3] = 1 - cs * G.d;
      c.q[0] = cs * bb0;
      c.q[1] = cs * bb1;
      c.cp = 0;
    } else if (p->alg == PSGLA_ALG_PNPULA) {
      c.cp = p->alpha * p->delta / p->epsilon;
      c.P[0] = 1 - c.cp - p->delta * G.a;
      c.P[1] = -p->delta * G.b;
      c.P[2] = -p->delta * G.c;
      c.P[3] = 1 - c.cp - p->delta * G.d;
      c.q[0] = p->delta * bb0;
      c.q[1] = p->delta * bb1;
    } else {
      return set_error(PSGLA_E_BADARG, "alg=%d is neither PSGLA_ALG_PSGLA nor PSGLA_ALG_PNPULA", p->alg);
    }
  }
  return PSGLA_OK;
}

template <typename T>
static void narrow(const Folded& f, Gmm2dConsts<T>* c, Gmm2dComponents<T>* k) {
  // Gmm2dConsts<double> is all doubles followed by one int: copy field by field
  for (int i = 0; i < 4; ++i) c->P[i] = (T)f.c.P[i];
  for (int i = 0; i < 2; ++i) c->q[i] = (T)f.c.q[i];
  c->cn = (T)f.c.cn;
  c->cp = (T)f.c.cp;
  for (int i = 0; i < 6; ++i) c->tq[i] = (T)f.c.tq[i];
  for (int i = 0; i < 4; ++i) {
    c->M1[i] = (T)f.c.M1[i];
    c->dM[i] = (T)f.c.dM[i];
  }
  for (int i = 0; i < 2; ++i) {
    c->b1[i] = (T)f.c.b1[i];
    c->db[i] = (T)f.c.db[i];
  }
  c->r = f.c.r;
  for (int i = 0; i < RMAX; ++i) {
    for (int j = 0; j < 2; ++j) k->mu[i][j] = (T)f.k.mu[i][j];
    for (int j = 0; j < 3; ++j) k->s[i][j] = (T)f.k.s[i][j];
    k->kappa2[i] = (T)f.k.kappa2[i];
    for (int j = 0; j < 4; ++j) k->M[i][j] = (T)f.k.M[i][j];
    for (int j = 0; j < 2; ++j) k->b[i][j] = (T)f.k.b[i][j];
  }
}

// Per-stream-ordered staging of the general-r component table: a small device buffer per call, freed stream-ordered.
template <typename T>
static int upload_components(const Gmm2dComponents<T>& k, cudaStream_t st, Gmm2dComponents<T>** dev) {
  PSGLA_CUDA_TRY(cudaMallocAsync((void**)dev, sizeof(k), st));
  PSGLA_CUDA_TRY(cudaMemcpyAsync(*dev, &k, sizeof(k), cudaMemcpyHostToDevice, st));
  return PSGLA_OK;
}

// Launch policy.  The kernel is issue-bound and its warps do identical work, but the SM's warp arbiter is not fair: of the
// warps resident on a scheduler some finish long before others (ncu: 5.4 of 8 warps active on average over a launch whose
// grid is exactly one resident wave), and what they leave behind is an under-filled tail.  So the fp32, r == 2 Philox path,
// the throughput path, runs all its chains in each launch (one per LEAN_TAB_ROUNDS rounds, launch_lean_body) as small blocks,
// many more blocks than fit: the hardware block scheduler back-fills every slot a finished warp frees, so all SMs stay full
// until the population is exhausted and the tail is one short block.
// The other paths (fp64, replay, r != 2: parity paths, not throughput paths) keep the round-1 policy: occupancy-sized waves.
struct Launch {  // everything a launch needs besides its chain range
  const void* c;
  const void* kdev;
  void* x;
  long long n_chains;
  unsigned long long chain_id0;
  long long n_steps, step0;
  PhiloxKeys keys;
  const void* noise;
  void* traj;
  long long thin;
  cudaStream_t st;
};

template <typename T, int ALG, bool R2, int CPT, int NB, int BLOCK>
static void launch_one(const Launch& a, long long lo, long long n_launch) {
  const long long threads = (n_launch + CPT - 1) / CPT;
  const unsigned grid = (unsigned)((threads + BLOCK - 1) / BLOCK);
  gmm2d_kernel<T, ALG, R2, CPT, NB, BLOCK><<<grid, BLOCK, 0, a.st>>>(
      *(const Gmm2dConsts<T>*)a.c, (const Gmm2dComponents<T>*)a.kdev, (T*)a.x, a.n_chains, lo, n_launch, a.chain_id0,
      a.n_steps, a.step0, a.keys, (const T*)a.noise, (T*)a.traj, a.thin);
}

// Threads that one wave of the full-wave kernel, gmm2d_kernel<T, ALG, R2, 4, 1, 128>, holds on the device.
template <typename T, int ALG, bool R2>
static int resident_threads(long long* threads) {
  int per_sm = 0;
  PSGLA_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gmm2d_kernel<T, ALG, R2, 4, 1, 128>, 128, 0));
  *threads = (long long)num_sms() * (per_sm > 0 ? per_sm : 8) * 128;
  return PSGLA_OK;
}

// Full waves of 4 chains per resident thread, then one remainder wave of as few chains per thread (1..4) as still fit in one
// wave.
template <typename T, int ALG, bool R2>
static int launch_waves(const Launch& a, int* launches) {
  long long resident = 0;
  const int rc = resident_threads<T, ALG, R2>(&resident);
  if (rc) return rc;
  for (long long lo = 0; lo < a.n_chains; ++*launches) {
    const long long n = std::min(a.n_chains - lo, 4 * resident);
    const long long cpt = (n + resident - 1) / resident;
    if (cpt == 1)
      launch_one<T, ALG, R2, 1, 1, 128>(a, lo, n);
    else if (cpt == 2)
      launch_one<T, ALG, R2, 2, 1, 128>(a, lo, n);
    else if (cpt == 3)
      launch_one<T, ALG, R2, 3, 1, 128>(a, lo, n);
    else
      launch_one<T, ALG, R2, 4, 1, 128>(a, lo, n);
    lo += n;
  }
  return PSGLA_OK;
}

// Philox words of a counter block after round 2 that depend only on the counter pair and the chain id's high word (the U
// words of gmm2d_lean_kernel), with the kernel's arithmetic.
static void lean_pair_words(const PhiloxKeys& keys, uint32_t pair_lo, uint32_t sub_hi, uint32_t* ua, uint32_t* ub,
                            uint32_t* uc) {
  const uint64_t u1 = (uint64_t)0xD2511F53u * pair_lo;                                      // round 1, pair word
  const uint64_t u2 = (uint64_t)0xCD9E8D57u * ((uint32_t)(u1 >> 32) ^ sub_hi ^ keys.k[1]);  // round 2, second product
  *ua = (uint32_t)(u2 >> 32) ^ keys.k[2];
  *ub = (uint32_t)u2;
  *uc = (uint32_t)u1 ^ keys.k[3];
}

template <int ALG, int STRUCT>
static void launch_lean(const Launch& a, long long lo, long long n, long long n_rounds, unsigned long long pair0) {
  static thread_local LeanPairWords tab;  // copied into the launch's parameters at the launch
  const unsigned long long sub0 = a.chain_id0 + (unsigned long long)lo;
  for (long long r = 0; r < n_rounds; ++r) {
    uint32_t ua[LEAN_NB], ub[LEAN_NB], uc[LEAN_NB];
    for (int b = 0; b < LEAN_NB; ++b)
      lean_pair_words(a.keys, (uint32_t)pair0 + (uint32_t)(r * LEAN_NB + b), (uint32_t)(sub0 >> 32), &ua[b], &ub[b], &uc[b]);
    tab.r[r] = {{ua[0], ua[1], ua[2], ua[3]}, {ub[0], ub[1], ub[2], ub[3]}, {uc[0], uc[1], uc[2], uc[3]}};
  }
  gmm2d_lean_kernel<ALG, STRUCT><<<(unsigned)((n + LEAN_BLOCK - 1) / LEAN_BLOCK), LEAN_BLOCK, 0, a.st>>>(
      *(const Gmm2dConsts<float>*)a.c, (float2*)a.x + lo, (unsigned)n, (uint32_t)sub0, (uint32_t)(pair0 >> 32), (int)n_rounds,
      a.keys, tab);
}

// The lean kernel on chains [lo, lo + n) (one high word of the chain id) for `rounds` rounds from counter pair pair0, in
// launches within which the pair's high word does not change either (gmm2d_lean_kernel takes both as launch constants) and
// of at most LEAN_TAB_ROUNDS rounds (what its table of pair words holds).  A round whose LEAN_NB pairs straddle a multiple of
// 2^32 goes to the general kernel.  Returns the number of launches.
template <int ALG, int STRUCT>
static int launch_lean_body(const Launch& a, long long lo, long long n, unsigned long long pair0, long long rounds) {
  int launches = 0;
  for (; rounds > 0; ++launches) {
    const unsigned long long next = ((pair0 >> 32) + 1) << 32;  // the first pair with the next high word
    const long long fit =
        (long long)std::min<unsigned long long>({(next - pair0) / LEAN_NB, (unsigned long long)rounds, LEAN_TAB_ROUNDS});
    if (fit > 0) {
      launch_lean<ALG, STRUCT>(a, lo, n, fit, pair0);
      pair0 += (unsigned long long)fit * LEAN_NB, rounds -= fit;
    } else {
      Launch b = a;
      b.step0 = (long long)(pair0 << 1), b.n_steps = 2 * LEAN_NB;
      launch_one<float, ALG, true, 1, 1, 128>(b, lo, n);
      pair0 += LEAN_NB, --rounds;
    }
  }
  return launches;
}

// fp32, r == 2, in-kernel Philox; returns the number of launches.  With a trajectory: one launch of 1-warp blocks of the
// general kernel (the lean kernel keeps no trajectory).  Without: the lean kernel on the whole rounds of 2 LEAN_NB steps that
// start on an even step, in chunks of at most 2^30 chains that do not cross a multiple of 2^32 in the global chain id; the
// general kernel takes the lead step of an odd step0 and the steps after the last whole round.
template <int ALG>
static int launch_philox_r2(const Launch& a) {
  if (a.traj != nullptr) {
    launch_one<float, ALG, true, 1, 4, 32>(a, 0, a.n_chains);
    return 1;
  }
  const int structure = constants_structure(*(const Gmm2dConsts<float>*)a.c);
  const long long lead = std::min(a.step0 & 1, a.n_steps);
  const long long rounds = (a.n_steps - lead) / (2 * LEAN_NB), body = rounds * 2 * LEAN_NB;
  const unsigned long long pair0 = (unsigned long long)(a.step0 + lead) >> 1;
  int launches = 0;
  if (lead) {
    Launch b = a;
    b.n_steps = lead;
    launch_one<float, ALG, true, 1, 1, 128>(b, 0, a.n_chains);
    ++launches;
  }
  for (long long lo = 0, n = 0; lo < a.n_chains && rounds > 0; lo += n) {
    const unsigned long long id = a.chain_id0 + (unsigned long long)lo, next = ((id >> 32) + 1) << 32;
    n = (long long)std::min({(unsigned long long)(a.n_chains - lo), 1ull << 30, next - id});
    if (structure == 2)
      launches += launch_lean_body<ALG, 2>(a, lo, n, pair0, rounds);
    else if (structure == 1)
      launches += launch_lean_body<ALG, 1>(a, lo, n, pair0, rounds);
    else
      launches += launch_lean_body<ALG, 0>(a, lo, n, pair0, rounds);
  }
  if (lead + body < a.n_steps) {
    Launch b = a;
    b.step0 = a.step0 + lead + body;
    b.n_steps = a.n_steps - lead - body;
    launch_one<float, ALG, true, 1, 1, 128>(b, 0, a.n_chains);
    ++launches;
  }
  return launches;
}

static thread_local int g_last_launches = 0;  // launches of this thread's most recent psgla_gmm2d_run (bench bookkeeping)

template <typename T, int ALG, bool R2>
static int launch_run(const Folded& f, T* x, long long n_chains, unsigned long long chain_id0, long long n_steps,
                      long long step0, unsigned long long seed, const T* noise, T* traj, long long thin,
                      cudaStream_t st) {
  Gmm2dConsts<T> c;
  static thread_local Gmm2dComponents<T> k;  // pageable source of the async copy must outlive the call: keep it TLS
  narrow<T>(f, &c, &k);
  Gmm2dComponents<T>* kdev = nullptr;
  if (!R2) {
    int rc = upload_components<T>(k, st, &kdev);
    if (rc) return rc;
  }
  const Launch a{&c, kdev, x, n_chains, chain_id0, n_steps, step0, philox_round_keys(seed), noise, traj, thin, st};
  int launches = 0, rc = PSGLA_OK;
  if (sizeof(T) == 4 && R2 && noise == nullptr)
    launches = launch_philox_r2<ALG>(a);
  else
    rc = launch_waves<T, ALG, R2>(a, &launches);
  if (rc) return rc;
  g_last_launches = launches;
  PSGLA_CUDA_TRY(cudaGetLastError());
  if (kdev) PSGLA_CUDA_TRY(cudaFreeAsync(kdev, st));
  return PSGLA_OK;
}

template <typename T>
static int dispatch_run(const psgla_gmm2d_problem* p, const Folded& f, void* x, long long n_chains,
                        unsigned long long chain_id0, long long n_steps, long long step0, unsigned long long seed,
                        const void* noise, void* traj, long long thin, cudaStream_t st) {
  const bool r2 = p->n_components == 2;
  T* xx = (T*)x;
  const T* nz = (const T*)noise;
  T* tj = (T*)traj;
  if (p->alg == PSGLA_ALG_PSGLA)
    return r2 ? launch_run<T, PSGLA_ALG_PSGLA, true>(f, xx, n_chains, chain_id0, n_steps, step0, seed, nz, tj, thin, st)
              : launch_run<T, PSGLA_ALG_PSGLA, false>(f, xx, n_chains, chain_id0, n_steps, step0, seed, nz, tj, thin, st);
  return r2 ? launch_run<T, PSGLA_ALG_PNPULA, true>(f, xx, n_chains, chain_id0, n_steps, step0, seed, nz, tj, thin, st)
            : launch_run<T, PSGLA_ALG_PNPULA, false>(f, xx, n_chains, chain_id0, n_steps, step0, seed, nz, tj, thin, st);
}

}  // namespace psgla

using namespace psgla;

extern "C" int psgla_gmm2d_run(const psgla_gmm2d_problem* problem, int precision, void* x_dev, int64_t n_chains,
                               int64_t chain_id0, int64_t n_steps, int64_t step0, uint64_t seed,
                               const void* noise_dev, void* traj_dev, int64_t thin, void* stream) {
  PSGLA_REQUIRE(problem != nullptr && x_dev != nullptr, "psgla_gmm2d_run: null problem or state pointer");
  PSGLA_REQUIRE(precision == 0 || precision == 1, "precision must be 0 (fp32) or 1 (fp64), got %d", precision);
  PSGLA_REQUIRE(n_chains > 0 && n_steps >= 0 && step0 >= 0 && chain_id0 >= 0, "negative size or offset");
  PSGLA_REQUIRE(traj_dev == nullptr || thin >= 1, "thin must be >= 1 when a trajectory buffer is given");
  if (n_steps == 0) return PSGLA_OK;
  Folded f;
  const double eps = problem->alg == PSGLA_ALG_PSGLA ? problem->delta : problem->epsilon;
  int rc = fold_problem(problem, eps, true, &f);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == 0)
    return dispatch_run<float>(problem, f, x_dev, n_chains, (unsigned long long)chain_id0, n_steps, step0, seed,
                               noise_dev, traj_dev, thin, st);
  return dispatch_run<double>(problem, f, x_dev, n_chains, (unsigned long long)chain_id0, n_steps, step0, seed,
                              noise_dev, traj_dev, thin, st);
}

template <typename T>
static int denoise_impl(const psgla_gmm2d_problem* p, const Folded& f, const void* x, void* out, long long n,
                        cudaStream_t st) {
  Gmm2dConsts<T> c;
  static thread_local Gmm2dComponents<T> k;
  narrow<T>(f, &c, &k);
  Gmm2dComponents<T>* kdev = nullptr;
  int rc = upload_components<T>(k, st, &kdev);
  if (rc) return rc;
  const int block = 128;
  const unsigned grid = (unsigned)((n + block - 1) / block);
  if (p->n_components == 2)
    gmm2d_denoise_kernel<T, true><<<grid, block, 0, st>>>(c, kdev, (const T*)x, (T*)out, n);
  else
    gmm2d_denoise_kernel<T, false><<<grid, block, 0, st>>>(c, kdev, (const T*)x, (T*)out, n);
  PSGLA_CUDA_TRY(cudaGetLastError());
  PSGLA_CUDA_TRY(cudaFreeAsync(kdev, st));
  return PSGLA_OK;
}

extern "C" int psgla_gmm2d_denoise(const psgla_gmm2d_problem* problem, double epsilon, int precision,
                                   const void* x_dev, void* out_dev, int64_t n, void* stream) {
  PSGLA_REQUIRE(problem != nullptr && x_dev != nullptr && out_dev != nullptr, "psgla_gmm2d_denoise: null pointer");
  PSGLA_REQUIRE(precision == 0 || precision == 1, "precision must be 0 (fp32) or 1 (fp64), got %d", precision);
  PSGLA_REQUIRE(n >= 0, "negative size");
  if (n == 0) return PSGLA_OK;
  Folded f;
  int rc = fold_problem(problem, epsilon, false, &f);
  if (rc) return rc;
  return precision == 0 ? denoise_impl<float>(problem, f, x_dev, out_dev, n, (cudaStream_t)stream)
                        : denoise_impl<double>(problem, f, x_dev, out_dev, n, (cudaStream_t)stream);
}

extern "C" int psgla_gmm2d_last_launches(void) { return g_last_launches; }

extern "C" int psgla_gmm2d_noise(float* out_dev, int64_t n_chains, int64_t chain_id0, int64_t n_steps, int64_t step0,
                                 uint64_t seed, void* stream) {
  PSGLA_REQUIRE(out_dev != nullptr && n_chains > 0 && n_steps >= 0 && step0 >= 0 && chain_id0 >= 0,
                "psgla_gmm2d_noise: bad argument");
  if (n_steps == 0) return PSGLA_OK;
  const int block = 128;
  gmm2d_noise_kernel<<<(unsigned)((n_chains + block - 1) / block), block, 0, (cudaStream_t)stream>>>(
      out_dev, n_chains, (unsigned long long)chain_id0, n_steps, step0, seed);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}
