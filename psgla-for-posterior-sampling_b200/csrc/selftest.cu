// Measured FP32 issue peak: the denominator of the 2D chain kernel's roofline (MEASURED_PEAKS.json, written by the driver,
// holds a copy bandwidth and a cuBLAS bf16 figure but no FP32 one).  Every thread runs `iters` rounds of 8 independent
// dependent-FMA chains -- nothing but FFMA (mode 0) or the packed FFMA2 (mode 1) issues in the loop.
#include "common.cuh"

namespace psgla {

template <int MODE>
__global__ void __launch_bounds__(256) fp32_rate_kernel(int iters, float seed, float* __restrict__ out) {
  const float a = 1.0f + seed * 1e-7f, b = seed * 1e-3f;
  if (MODE == 0) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = seed + (float)(threadIdx.x + j);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], a, b);
    }
    float s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[j];
    if (s == 123.456f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;  // keeps the loop alive, never true in practice
  } else {
    unsigned long long v[8], aa, bb;
    asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a));
    asm("mov.b64 %0, {%1, %1};" : "=l"(bb) : "f"(b));
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float x = seed + (float)(threadIdx.x + j);
      asm("mov.b64 %0, {%1, %2};" : "=l"(v[j]) : "f"(x), "f"(x + 0.5f));
    }
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int j = 0; j < 8; ++j) asm("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(v[j]) : "l"(aa), "l"(bb));
    }
    float s = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float lo, hi;
      asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v[j]));
      s += lo + hi;
    }
    if (s == 123.456f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  }
}


// The FP64-pipe form of a Philox round product's high word (modes 12-14 and 200 + NF): for a = the double with bit pattern
// {lo word x, hi word 0x43380000} (= 1.5 2^52 + x), fma.rm(a, M 2^-32, 1.5 2^52 - 1.5 2^20 M) = 1.5 2^52 + floor(x M / 2^32)
// exactly, so the result's low word is mulhi(x, M) and its high word 0x43380000 again (M = 0xD2511F53 here).
__device__ __forceinline__ uint64_t pair_of(uint32_t lo, uint32_t hi) {
  uint64_t a;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(lo), "r"(hi));
  return a;
}
__device__ __forceinline__ uint32_t pair_lo(uint64_t a) {
  uint32_t lo;
  asm("mov.b64 {%0, _}, %1;" : "=r"(lo) : "l"(a));
  return lo;
}
__device__ __forceinline__ uint32_t pair_hi(uint64_t a) {
  uint32_t hi;
  asm("mov.b64 {_, %0}, %1;" : "=r"(hi) : "l"(a));
  return hi;
}
__device__ __forceinline__ uint64_t mulhi_fp64(uint64_t a) {
  uint64_t t;
  asm volatile("fma.rm.f64 %0, %1, 0d3FEA4A23EA600000, 0d4311219440E00000;" : "=l"(t) : "l"(a));
  return t;
}

// One round product in that form: the low word x * m by IMAD, the high word by DFMA.RM, and a LOP3 that consumes the high word
// and writes the next input into the pair's low register.
__device__ __forceinline__ uint64_t fp64_round_product(uint64_t a, unsigned m) {
  unsigned lo;
  asm volatile("mul.lo.u32 %0, %1, %2;" : "=r"(lo) : "r"(pair_lo(a)), "r"(m));
  const uint64_t t = mulhi_fp64(a);
  unsigned n;
  asm volatile("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(n) : "r"(pair_lo(t)), "r"(lo), "r"(m));
  return pair_of(n, pair_hi(t));
}

// Issue-rate probe of single instruction classes (what bounds the chain kernel's Philox + Box-Muller + sigmoid mix):
// every thread runs iters x 32 instructions of ONE class in 8 independent dependency chains.
//   0 IMAD.WIDE.U32 (mul.wide.u32, the Philox round multiply)   1 IMAD.HI.U32 (mul.hi.u32)   2 IMAD (mul.lo.u32)
//   3 LOP3 (3-input xor)   4 MUFU.EX2   5 I2FP.F32.U32   6 FFMA   7 MUFU.SIN   8 IMAD.WIDE + FFMA interleaved 1:1
//   9 MUFU.EX2 + IMAD.WIDE 1:1   10 MUFU.EX2 + 4 FFMA
//   11 / 100 + NF: the chain kernel's per-step MIX as independent chains (6 MUFU, 9 IMAD.WIDE, NF FFMA, 10 LOP3, 2 I2FP per
//      "step", 4 steps per loop round; NF = 19 for mode 11, else 21 / 23 / 26 / 28 / 30 = the FP32 pipe slots per step of the six
//      (algorithm, constants-structure) specialisations of gmm2d_lean_kernel): what the SM sustains for this instruction mix
//      when no instruction waits for another -- the measured ceiling the chain kernel is held against
//   12 DFMA.RM (fma.rm.f64, the high word of a Philox round product on the FP64 pipe, below)   13 IMAD + DFMA.RM + LOP3: that
//   form of one round product (low word, high word, the XOR that consumes it) -- set against mode 0
//   14 DFMA.RM + FFMA 1:1
//   200 + NF: the chain-step MIX with the FP64-pipe multiply (6 MUFU, 9 IMAD, 9 DFMA.RM, 2 MOV, NF FFMA, 10 LOP3, 2 I2FP)
template <int MODE, int NF = 19>
__global__ void __launch_bounds__(256) pipe_rate_kernel(int iters, unsigned seed, unsigned* __restrict__ out) {
  unsigned v[8];
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    v[j] = seed * 2654435761u + threadIdx.x * 40503u + j;
    f[j] = (float)(v[j] & 1023) * 1e-3f;
  }
  uint64_t d[8];  // modes 12-14, 20: {x, 0x43380000} pairs
#pragma unroll
  for (int j = 0; j < 8; ++j) d[j] = pair_of(v[j], 0x43380000u);
  const unsigned m = 0xD2511F53u + seed;
  const float a = 1.0f + seed * 1e-7f, b = seed * 1e-3f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (MODE == 0) {
          unsigned long long p;
          asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(v[j]), "r"(m));
          v[j] = (unsigned)(p >> 32) + (unsigned)p;  // IADD on the ALU pipe keeps both halves live
        } else if (MODE == 1) {
          asm volatile("mul.hi.u32 %0, %0, %1;" : "+r"(v[j]) : "r"(m));
        } else if (MODE == 2) {
          asm volatile("mul.lo.u32 %0, %0, %1;" : "+r"(v[j]) : "r"(m));
        } else if (MODE == 3) {
          asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(v[j]) : "r"(m), "r"(v[(j + 1) & 7]));
        } else if (MODE == 4) {
          asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(f[j]));
        } else if (MODE == 5) {
          asm volatile("cvt.rn.f32.u32 %0, %1;" : "=f"(f[j]) : "r"(v[j]));
          v[j] = __float_as_uint(f[j]);
        } else if (MODE == 6) {
          f[j] = fmaf(f[j], a, b);
        } else if (MODE == 7) {
          asm volatile("sin.approx.ftz.f32 %0, %0;" : "+f"(f[j]));
        } else if (MODE == 8) {
          unsigned long long p;
          asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(v[j]), "r"(m));
          v[j] = (unsigned)(p >> 32) ^ (unsigned)p;
          f[j] = fmaf(f[j], a, b);
        } else if (MODE == 9) {
          unsigned long long p;
          asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(v[j]), "r"(m));
          v[j] = (unsigned)(p >> 32) ^ (unsigned)p;
          asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(f[j]));
        } else if (MODE == 10) {
          asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(f[j]));
          float g = f[(j + 1) & 7];
          g = fmaf(g, a, b), g = fmaf(g, a, b), g = fmaf(g, a, b), g = fmaf(g, a, b);
          f[(j + 1) & 7] = g;
        } else if (MODE == 12) {
          d[j] = mulhi_fp64(d[j]);
        } else if (MODE == 13) {
          d[j] = fp64_round_product(d[j], m);
        } else if (MODE == 14) {
          d[j] = mulhi_fp64(d[j]);
          f[j] = fmaf(f[j], a, b);
        }
      }
    if (MODE == 11) {
      float e[6];  // MUFU chains
      unsigned w[3];
#pragma unroll
      for (int q = 0; q < 6; ++q) e[q] = f[q];
#pragma unroll
      for (int q = 0; q < 3; ++q) w[q] = v[q];
#pragma unroll
      for (int st = 0; st < 4; ++st) {  // 4 "steps"
#pragma unroll
        for (int q = 0; q < 6; ++q) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(e[q]));
#pragma unroll
        for (int q = 0; q < 9; ++q) {
          unsigned long long p;
          asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(w[q % 3]), "r"(m));
          asm volatile("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(w[q % 3]) : "r"((unsigned)(p >> 32)), "r"((unsigned)p), "r"(m));
        }
#pragma unroll
        for (int q = 0; q < NF; ++q) asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(f[6 + (q & 1)]) : "f"(a), "f"(b));
        float c0, c1;
        asm volatile("cvt.rn.f32.u32 %0, %1;" : "=f"(c0) : "r"(w[0]));
        asm volatile("cvt.rn.f32.u32 %0, %1;" : "=f"(c1) : "r"(w[1]));
        asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(v[7]) : "r"(__float_as_uint(c0)), "r"(__float_as_uint(c1)));  // the 10th LOP3
      }
#pragma unroll
      for (int q = 0; q < 6; ++q) f[q] = e[q];
#pragma unroll
      for (int q = 0; q < 3; ++q) v[q] = w[q];
    }
    if (MODE == 20) {  // as mode 11, each IMAD.WIDE.U32 + LOP3 replaced by IMAD + DFMA.RM + LOP3, plus the kernel's ~2 MOV
      float e[6];
#pragma unroll
      for (int q = 0; q < 6; ++q) e[q] = f[q];
#pragma unroll
      for (int st = 0; st < 4; ++st) {
#pragma unroll
        for (int q = 0; q < 6; ++q) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(e[q]));
#pragma unroll
        for (int q = 0; q < 9; ++q) d[q % 3] = fp64_round_product(d[q % 3], m);
#pragma unroll
        for (int q = 0; q < 2; ++q) asm volatile("mov.b32 %0, %1;" : "=r"(v[4 + q]) : "r"(v[3 + q]));
#pragma unroll
        for (int q = 0; q < NF; ++q) asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(f[6 + (q & 1)]) : "f"(a), "f"(b));
        float c0, c1;
        asm volatile("cvt.rn.f32.u32 %0, %1;" : "=f"(c0) : "r"(pair_lo(d[0])));
        asm volatile("cvt.rn.f32.u32 %0, %1;" : "=f"(c1) : "r"(pair_lo(d[1])));
        asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(v[7]) : "r"(__float_as_uint(c0)), "r"(__float_as_uint(c1)));
      }
#pragma unroll
      for (int q = 0; q < 6; ++q) f[q] = e[q];
    }
  }
  unsigned s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += v[j] + __float_as_uint(f[j]) + pair_lo(d[j]);
  if (s == 0x12345678u) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace psgla

using namespace psgla;

extern "C" int psgla_selftest_fp32_rate(int mode, int iters, int blocks_per_sm, float* out_dev, double* flop_out,
                                        void* stream) {
  PSGLA_REQUIRE((mode == 0 || mode == 1) && iters > 0 && blocks_per_sm > 0 && blocks_per_sm <= 8 && out_dev != nullptr,
                "psgla_selftest_fp32_rate: bad argument");
  const int grid = num_sms() * blocks_per_sm;
  if (mode == 0)
    fp32_rate_kernel<0><<<grid, 256, 0, (cudaStream_t)stream>>>(iters, 0.25f, out_dev);
  else
    fp32_rate_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(iters, 0.25f, out_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  if (flop_out) *flop_out = (double)grid * 256.0 * (double)iters * 32.0 * 2.0 * (mode == 1 ? 2.0 : 1.0);
  return PSGLA_OK;
}

extern "C" int psgla_selftest_pipe_rate(int mode, int iters, int blocks_per_sm, void* out_dev, double* ops_out, void* stream) {
  const bool mix_nf = mode % 100 == 21 || mode % 100 == 23 || mode % 100 == 26 || mode % 100 == 28 || mode % 100 == 30;
  PSGLA_REQUIRE(((mode >= 0 && mode <= 14) || ((mode / 100 == 1 || mode / 100 == 2) && mix_nf)) && iters > 0 && blocks_per_sm > 0 && blocks_per_sm <= 8 && out_dev != nullptr,
                "psgla_selftest_pipe_rate: bad argument");
  const int grid = num_sms() * blocks_per_sm;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned* o = (unsigned*)out_dev;
  switch (mode) {
    case 0: pipe_rate_kernel<0><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 1: pipe_rate_kernel<1><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 2: pipe_rate_kernel<2><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 3: pipe_rate_kernel<3><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 4: pipe_rate_kernel<4><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 5: pipe_rate_kernel<5><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 6: pipe_rate_kernel<6><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 7: pipe_rate_kernel<7><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 8: pipe_rate_kernel<8><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 9: pipe_rate_kernel<9><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 10: pipe_rate_kernel<10><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 121: pipe_rate_kernel<11, 21><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 123: pipe_rate_kernel<11, 23><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 126: pipe_rate_kernel<11, 26><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 128: pipe_rate_kernel<11, 28><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 130: pipe_rate_kernel<11, 30><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 11: pipe_rate_kernel<11><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 12: pipe_rate_kernel<12><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 13: pipe_rate_kernel<13><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 14: pipe_rate_kernel<14><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 221: pipe_rate_kernel<20, 21><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 223: pipe_rate_kernel<20, 23><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 226: pipe_rate_kernel<20, 26><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    case 228: pipe_rate_kernel<20, 28><<<grid, 256, 0, st>>>(iters, 3u, o); break;
    default: pipe_rate_kernel<20, 30><<<grid, 256, 0, st>>>(iters, 3u, o); break;
  }
  PSGLA_CUDA_TRY(cudaGetLastError());
  // thread-level instructions of the probed class; mix modes (11, 100 + NF, 200 + NF): thread-level "steps" (4 per loop round)
  const bool mix = mode == 11 || mode >= 100;
  if (ops_out) *ops_out = (double)grid * 256.0 * (double)iters * (mix ? 4.0 : 32.0);
  return PSGLA_OK;
}

