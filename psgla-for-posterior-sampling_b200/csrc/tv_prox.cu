// Total-variation proximal operator (deepinv's TVDenoiser, the prior of the reference's PSGLA-TV runs,
// sampling_images.py:139-140,181-184) fused with the Langevin post of the samplers.
//
// One cooperative launch runs a whole prox call for B chains: over-relaxed Chambolle-Pock on
//   argmin_x 1/2 ||x - y||^2 + ths sum_{c,p} ||grad x_{c,p}||_2
// with fp32 state and arithmetic, then X+ = gain * D + base_scale * y, thinning and the running moments.
//
// Layout and barriers
//   * every chain's [3][H][W] is cut into TV_TH x TV_TW tiles of one channel plane; the tile layout depends on (H, W) only.
//     Work items (chain, tile) are dealt round-robin over the CTAs.
//   * one grid-wide barrier per CP iteration.  Iteration k reads state copy k % 2 and writes copy (k + 1) % 2 (copy 0 is the
//     caller's state buffer, copy 1 lives in the workspace), so a CTA that reads its neighbours' border values never races
//     with their writes.  x is recomputed on a one-pixel bottom / right halo: u at p needs x at p, p + down, p + right, and x
//     needs u2 at p, p - up, p - left.
//   * convergence: each tile writes fp64 partial sums of ||x_prev - x2||^2 and ||x2 + 1e-12||^2 to part[k % 2][chain][tile].
//     After the barrier one CTA per chain reduces them in an order fixed by the tile count alone (so the decision does not
//     depend on B, the chain's batch position or the grid size) and records the chain's iteration count in stat[k % 2][chain]
//     once it meets the criterion (or reaches n_it_max).  Every other CTA reads that record one barrier later, so all CTAs take
//     the same "skip this chain" and "all chains done" decisions and execute the same number of barriers.  A chain that stops
//     after n iterations is computed once more (into copy (n + 1) % 2, never read); its result stays in copy n % 2.
//   * final pass: x2 / u2 of copy 1 are copied to the caller's state where n is odd, then the post.
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace psgla {
namespace {

constexpr int TV_TH = 16, TV_TW = 32, TV_THREADS = 256;

struct TvArgs {
  int B, H, W, tiles_x, tiles_plane, tiles_chain;
  float ths, tau, rho, sigma, one_plus_tau;
  double crit;
  int n_it_max, restart;
  const float* y;
  float* x2[2];  // [B][3][H][W]
  float* u2[2];  // [B][3][H][W][2]
  double* part;  // [2][B][tiles_chain][2]
  int* stat;     // [2][B]: 0 while the chain runs, else its iteration count
  float gain, base_scale, w_old, w_new;
  float* x_out;
  float* sample;
  float* mean;
  float* mean2;
  int* iters;
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(TV_THREADS, 6) tv_prox_post_kernel(TvArgs a) {
  cg::grid_group grid = cg::this_grid();
  __shared__ float us0[TV_TH + 2][TV_TW + 2], us1[TV_TH + 2][TV_TW + 2];  // u2 on rows r0-1 .. r0+TH, cols c0-1 .. c0+TW
  __shared__ float xbar[TV_TH + 1][TV_TW + 1];                           // 2x - x2 on the tile + bottom / right halo
  __shared__ float ys[TV_TH + 1][TV_TW + 1], x2s[TV_TH + 1][TV_TW + 1];
  __shared__ float xs[TV_TH][TV_TW];
  __shared__ double red[2][TV_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long plane = (long long)a.H * a.W, chain = 3 * plane;
  const int n_items = a.B * a.tiles_chain;
  int k = 0;
  for (;; ++k) {
    const int* seen = a.stat + ((k - 1) & 1) * a.B;  // written before the previous barrier
    if (k >= 2) {
      int all = 1;
      for (int b0 = 0; b0 < a.B; b0 += TV_THREADS) all &= __syncthreads_and(b0 + tid >= a.B || seen[b0 + tid] != 0);
      if (all) break;
    }
    if (k >= 1 && warp == 0) {  // reducer of chains blockIdx.x, blockIdx.x + gridDim.x, ...: records iteration k - 1's verdict
      for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        int n = k >= 2 ? seen[b] : 0;
        if (n == 0) {
          const double* pp = a.part + ((size_t)((k - 1) & 1) * a.B + b) * a.tiles_chain * 2;
          double sa = 0.0, sb = 0.0;
          for (int t = lane; t < a.tiles_chain; t += 32) sa += pp[2 * t], sb += pp[2 * t + 1];
          sa = warp_sum(sa);
          sb = warp_sum(sb);
          const bool conv = k - 1 > 1 && sqrt(sa) / sqrt(sb) < a.crit;
          if (conv || k == a.n_it_max) n = k;
        }
        if (lane == 0) a.stat[(k & 1) * a.B + b] = n;
      }
    }
    if (k < a.n_it_max) {
      const bool virt = a.restart && k == 0;  // first iteration of a restart: x2 = y, u2 = 0
      const float* sx = a.x2[k & 1];
      const float* su = a.u2[k & 1];
      float* dx = a.x2[(k + 1) & 1];
      float* du = a.u2[(k + 1) & 1];
      for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
        const int b = w / a.tiles_chain, t = w - b * a.tiles_chain;
        if (k >= 2 && seen[b] != 0) continue;  // frozen (uniform over the CTA)
        const int c = t / a.tiles_plane, tp = t - c * a.tiles_plane;
        const int r0 = (tp / a.tiles_x) * TV_TH, c0 = (tp % a.tiles_x) * TV_TW;
        const long long base = (long long)b * chain + c * plane;
        // every global read of the item in one round trip: u2 on the tile + one-pixel ring, x2 and y on the tile + bottom /
        // right halo
        for (int i = tid; i < (TV_TH + 2) * (TV_TW + 2); i += TV_THREADS) {
          const int rr = i / (TV_TW + 2), cc = i - rr * (TV_TW + 2), gr = r0 - 1 + rr, gc = c0 - 1 + cc;
          float v0 = 0.f, v1 = 0.f;
          if (!virt && gr >= 0 && gr < a.H && gc >= 0 && gc < a.W) {
            const long long e = base + (long long)gr * a.W + gc;
            v0 = su[2 * e];
            v1 = su[2 * e + 1];
          }
          us0[rr][cc] = v0;
          us1[rr][cc] = v1;
        }
        for (int i = tid; i < (TV_TH + 1) * (TV_TW + 1); i += TV_THREADS) {
          const int rr = i / (TV_TW + 1), cc = i - rr * (TV_TW + 1), gr = r0 + rr, gc = c0 + cc;
          float yv = 0.f, x2v = 0.f;
          if (gr < a.H && gc < a.W) {
            const long long e = base + (long long)gr * a.W + gc;
            yv = a.y[e];
            x2v = virt ? yv : sx[e];
          }
          ys[rr][cc] = yv;
          x2s[rr][cc] = x2v;
        }
        __syncthreads();
        for (int i = tid; i < (TV_TH + 1) * (TV_TW + 1); i += TV_THREADS) {
          const int rr = i / (TV_TW + 1), cc = i - rr * (TV_TW + 1), gr = r0 + rr, gc = c0 + cc;
          float xb = 0.f;
          if (gr < a.H && gc < a.W) {
            const float x2v = x2s[rr][cc];
            float d = 0.f;  // (grad^T u2) at (gr, gc)
            if (gr < a.H - 1) d -= us0[rr + 1][cc + 1];
            if (gr >= 1) d += us0[rr][cc + 1];
            if (gc < a.W - 1) d -= us1[rr + 1][cc + 1];
            if (gc >= 1) d += us1[rr + 1][cc];
            const float x = (x2v - a.tau * d + a.tau * ys[rr][cc]) / a.one_plus_tau;
            xb = 2.f * x - x2v;
            if (rr < TV_TH && cc < TV_TW) xs[rr][cc] = x;
          }
          xbar[rr][cc] = xb;
        }
        __syncthreads();
        double pa = 0.0, pb = 0.0;
        for (int i = tid; i < TV_TH * TV_TW; i += TV_THREADS) {
          const int rr = i / TV_TW, cc = i - rr * TV_TW, gr = r0 + rr, gc = c0 + cc;
          if (gr >= a.H || gc >= a.W) continue;
          const long long e = base + (long long)gr * a.W + gc;
          const float xb = xbar[rr][cc];
          const float g0 = gr < a.H - 1 ? xbar[rr + 1][cc] - xb : 0.f;
          const float g1 = gc < a.W - 1 ? xbar[rr][cc + 1] - xb : 0.f;
          const float u0o = us0[rr + 1][cc + 1], u1o = us1[rr + 1][cc + 1];
          float u0 = u0o + a.sigma * g0, u1 = u1o + a.sigma * g1;
          const float f = fmaxf(sqrtf(u0 * u0 + u1 * u1) / a.ths, 1.f);
          u0 = u0 / f;
          u1 = u1 / f;
          const float x2o = x2s[rr][cc];
          const float x2n = x2o + a.rho * (xs[rr][cc] - x2o);
          dx[e] = x2n;
          du[2 * e] = u0o + a.rho * (u0 - u0o);
          du[2 * e + 1] = u1o + a.rho * (u1 - u1o);
          const double dd = (double)(x2o - x2n), nn = (double)(x2n + 1e-12f);
          pa += dd * dd;
          pb += nn * nn;
        }
        pa = warp_sum(pa);
        pb = warp_sum(pb);
        if (lane == 0) red[0][warp] = pa, red[1][warp] = pb;
        __syncthreads();
        if (tid == 0) {
          double sa = 0.0, sb = 0.0;
          for (int i = 0; i < TV_THREADS / 32; ++i) sa += red[0][i], sb += red[1][i];
          double* pp = a.part + ((size_t)(k & 1) * a.B + b) * a.tiles_chain * 2 + 2 * t;
          pp[0] = sa;
          pp[1] = sb;
        }
        __syncthreads();  // shared tiles are reused by the next item
      }
    }
    grid.sync();
  }
  // final pass: chain b's result is copy n % 2 of its state, n = its iteration count
  const int* fin = a.stat + ((k - 1) & 1) * a.B;
  const long long total = (long long)a.B * chain;
  for (long long e = (long long)blockIdx.x * TV_THREADS + tid; e < total; e += (long long)gridDim.x * TV_THREADS) {
    const int b = (int)(e / chain), n = fin[b];
    const float d = a.x2[n & 1][e];
    if (n & 1) {
      a.x2[0][e] = d;
      a.u2[0][2 * e] = a.u2[1][2 * e];
      a.u2[0][2 * e + 1] = a.u2[1][2 * e + 1];
    }
    const float xn = fmaf(a.gain, d, a.base_scale * a.y[e]);  // the DRUNet epilogue's post (conv_tc.cuh)
    a.x_out[e] = xn;
    if (a.sample) a.sample[e] = xn;
    if (a.mean) {
      // three rounded fp32 operations each, as the reference's eager ops (restoration_algorithms.py:257-258)
      a.mean[e] = __fadd_rn(__fmul_rn(a.w_old, a.mean[e]), __fmul_rn(a.w_new, xn));
      a.mean2[e] = __fadd_rn(__fmul_rn(a.w_old, a.mean2[e]), __fmul_rn(a.w_new, __fmul_rn(xn, xn)));
    }
    if (a.iters && e - (long long)b * chain == 0) a.iters[b] = n;
  }
}

struct TvLayout {
  size_t n;             // elements of x2 = B * 3 * H * W
  size_t x2, u2, part, stat, total;  // workspace byte offsets
  int tiles_x, tiles_plane, tiles_chain;
};

bool tv_shape_ok(const psgla_img_shape& s) {
  return s.C == 3 && s.B >= 1 && s.H >= 1 && s.W >= 1 && (long long)s.B * 3 * s.H * s.W < (1LL << 40);
}

TvLayout tv_layout(const psgla_img_shape& s) {
  TvLayout L;
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  L.n = (size_t)s.B * 3 * s.H * s.W;
  L.tiles_x = (s.W + TV_TW - 1) / TV_TW;
  L.tiles_plane = L.tiles_x * ((s.H + TV_TH - 1) / TV_TH);
  L.tiles_chain = 3 * L.tiles_plane;
  L.x2 = 0;
  L.u2 = up(L.x2 + 4 * L.n);
  L.part = up(L.u2 + 8 * L.n);
  L.stat = up(L.part + (size_t)2 * s.B * L.tiles_chain * 2 * sizeof(double));
  L.total = up(L.stat + (size_t)2 * s.B * sizeof(int));
  return L;
}

}  // namespace
}  // namespace psgla

using namespace psgla;

extern "C" size_t psgla_tv_state_bytes(psgla_img_shape s) {
  return tv_shape_ok(s) ? (size_t)s.B * 3 * s.H * s.W * 12 : 0;
}

extern "C" size_t psgla_tv_workspace_bytes(psgla_img_shape s) { return tv_shape_ok(s) ? tv_layout(s).total : 0; }

extern "C" int psgla_tv_prox_post(const psgla_tv_params* tv, psgla_img_shape s, const float* y_dev, void* state_dev,
                                  size_t state_bytes, void* workspace_dev, size_t workspace_bytes,
                                  const psgla_post_params* post, float* x_out_dev, float* sample_dev, float* mean_dev,
                                  float* mean2_dev, int32_t* iters_dev, void* stream) {
  PSGLA_REQUIRE(tv && post && y_dev && state_dev && workspace_dev && x_out_dev, "psgla_tv_prox_post: null pointer");
  PSGLA_REQUIRE(!mean_dev == !mean2_dev, "psgla_tv_prox_post: mean_dev and mean2_dev go together");
  PSGLA_REQUIRE(tv_shape_ok(s), "image shape must be [B>0][3][H>0][W>0], got [%d][%d][%d][%d]", s.B, s.C, s.H, s.W);
  PSGLA_REQUIRE(tv->ths > 0.f && tv->ths <= 3.4e38f, "ths must be > 0 (got %g)", (double)tv->ths);
  PSGLA_REQUIRE(tv->tau > 0.f && tv->tau <= 3.4e38f, "tau must be > 0 (got %g)", (double)tv->tau);
  PSGLA_REQUIRE(tv->rho > 0.f && tv->rho < 2.f, "rho must be in (0, 2) (got %g)", (double)tv->rho);
  PSGLA_REQUIRE(tv->crit >= 0.f && tv->crit <= 3.4e38f, "crit must be >= 0 (got %g)", (double)tv->crit);
  PSGLA_REQUIRE(tv->n_it_max >= 1, "n_it_max must be >= 1 (got %d)", tv->n_it_max);
  PSGLA_REQUIRE(tv->restart == 0 || tv->restart == 1, "restart must be 0 or 1 (got %d)", tv->restart);
  const TvLayout L = tv_layout(s);
  if (state_bytes < 12 * L.n)
    return set_error(PSGLA_E_WORKSPACE, "state buffer holds %zu bytes, needs %zu", state_bytes, 12 * L.n);
  if (workspace_bytes < L.total)
    return set_error(PSGLA_E_WORKSPACE, "workspace holds %zu bytes, needs %zu", workspace_bytes, L.total);

  TvArgs a;
  a.B = s.B, a.H = s.H, a.W = s.W;
  a.tiles_x = L.tiles_x, a.tiles_plane = L.tiles_plane, a.tiles_chain = L.tiles_chain;
  a.ths = tv->ths, a.tau = tv->tau, a.rho = tv->rho;
  a.sigma = (float)(1.0 / (double)tv->tau / 8.0);  // deepinv: sigma = 1 / tau / 8
  a.one_plus_tau = (float)(1.0 + (double)tv->tau);
  a.crit = tv->crit, a.n_it_max = tv->n_it_max, a.restart = tv->restart;
  a.y = y_dev;
  char* st = (char*)state_dev;
  char* ws = (char*)workspace_dev;
  a.x2[0] = (float*)st, a.u2[0] = (float*)(st + 4 * L.n);
  a.x2[1] = (float*)(ws + L.x2), a.u2[1] = (float*)(ws + L.u2);
  a.part = (double*)(ws + L.part);
  a.stat = (int*)(ws + L.stat);
  a.gain = post->gain, a.base_scale = post->base_scale, a.w_old = post->w_old, a.w_new = post->w_new;
  a.x_out = x_out_dev, a.sample = sample_dev, a.mean = mean_dev, a.mean2 = mean2_dev, a.iters = iters_dev;

  int per_sm = 0;
  PSGLA_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tv_prox_post_kernel, TV_THREADS, 0));
  if (per_sm < 1) return set_error(PSGLA_E_UNSUPPORTED, "tv_prox_post_kernel cannot be resident on this device");
  // co-resident by construction: the cooperative launch fails instead of hanging if this were too many
  const long long items = (long long)s.B * L.tiles_chain;
  const int grid = (int)std::min<long long>((long long)per_sm * num_sms(), items);
  void* args[] = {&a};
  PSGLA_CUDA_TRY(cudaLaunchCooperativeKernel((const void*)tv_prox_post_kernel, dim3(grid), dim3(TV_THREADS), args, 0,
                                             (cudaStream_t)stream));
  return PSGLA_OK;
}
