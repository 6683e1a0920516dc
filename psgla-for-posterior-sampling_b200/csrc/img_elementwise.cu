// HBM-bound stages of the image samplers: the Langevin "pre" step (data-fidelity gradient + noise) for inpainting and
// deblurring, the circular separable blur as a shared-memory staged stencil, Philox noise, layout conversion.
//
// Reference arithmetic replaced here:
//   inpainting data_grad  -mask (x - y) / sigma^2                         sampling_images.py:295
//   deblurring data_grad  -A^T(A x - y) / sigma^2, A = circular blur      sampling_images.py:329-338
//   PSGLA   Y = X + (delta/lambd) grad + sqrt(2) s Z                      restoration_algorithms.py:232-236
//   PnP-ULA X + delta (-(X - proj)/lambd + grad) + sqrt(2 delta) Z        restoration_algorithms.py:104-115
// (the denoiser term of either update is added by the last conv layer's epilogue, csrc/conv_tc.cu).
#include <cuda_bf16.h>

#include <cstring>

#include "common.cuh"
#include "langevin.cuh"

namespace psgla {

// ------------------------------------------------------------------------------------------------ inpainting pre
// One thread = 4 consecutive pixels of one row (all C channels) when W % 4 == 0, else 1 pixel.  C = 3 (colour) or 1
// (grayscale): the element index within a chain is e = c H W + pixel either way, so channel 0 draws the same noise.
template <int VEC, int C>
__global__ void __launch_bounds__(256)
pre_inpaint_kernel(PreArgs a, int B, int H, int W, const float* __restrict__ x, const float* __restrict__ mask,
                   int mask_B, const float* __restrict__ y, int y_B, const float* __restrict__ noise,
                   float* __restrict__ base, __nv_bfloat16* __restrict__ den_in) {
  const long long plane = (long long)H * W;
  const long long groups_per_chain = plane / VEC;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= groups_per_chain * B) return;
  const int b = (int)(g / groups_per_chain);
  const long long pix = (g % groups_per_chain) * VEC;  // first pixel (row-major) of this thread
  float outv[C][VEC];
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const long long e = c * plane + pix;  // element index inside the chain
    const long long gi = ((long long)b * C) * plane + e;
    const long long mi = ((long long)(mask_B > 1 ? b : 0) * C) * plane + e;
    const long long yi = ((long long)(y_B > 1 ? b : 0) * C) * plane + e;
    float xv[VEC], mv[VEC], yv[VEC], zv[VEC];
    if (VEC == 4) {
      const float4 t0 = *reinterpret_cast<const float4*>(x + gi);
      const float4 t1 = *reinterpret_cast<const float4*>(mask + mi);
      const float4 t2 = *reinterpret_cast<const float4*>(y + yi);
      xv[0] = t0.x, xv[1 % VEC] = t0.y, xv[2 % VEC] = t0.z, xv[3 % VEC] = t0.w;
      mv[0] = t1.x, mv[1 % VEC] = t1.y, mv[2 % VEC] = t1.z, mv[3 % VEC] = t1.w;
      yv[0] = t2.x, yv[1 % VEC] = t2.y, yv[2 % VEC] = t2.z, yv[3 % VEC] = t2.w;
      if (noise) {
        const float4 t3 = *reinterpret_cast<const float4*>(noise + gi);
        zv[0] = t3.x, zv[1 % VEC] = t3.y, zv[2 % VEC] = t3.z, zv[3 % VEC] = t3.w;
      } else {
        float z4[4];
        draw_quad(a, b, (uint32_t)e, z4);
#pragma unroll
        for (int j = 0; j < VEC; ++j) zv[j] = z4[j];
      }
    } else {
      xv[0] = x[gi];
      mv[0] = mask[mi];
      yv[0] = y[yi];
      zv[0] = noise ? noise[gi] : draw_at(a, b, (uint32_t)e);
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) outv[c][j] = langevin_base(a, xv[j], mv[j] * (xv[j] - yv[j]), zv[j]);
    if (VEC == 4)
      *reinterpret_cast<float4*>(base + gi) = make_float4(outv[c][0], outv[c][1 % VEC], outv[c][2 % VEC], outv[c][3 % VEC]);
    else
      base[gi] = outv[c][0];
    if (a.alg == PSGLA_ALG_PNPULA) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) outv[c][j] = xv[j];  // the denoiser sees X, not the partial update
    }
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j)
    store_nhwc16(den_in + ((long long)b * plane + pix + j) * 16, outv[0][j], C > 1 ? outv[1 % C][j] : 0.f,
                 C > 2 ? outv[2 % C][j] : 0.f, a.den_in_c3);
}

// ------------------------------------------------------------------------------------------------ blur / deblur pre
// Tile 32 x 32 pixels of one chain, 256 threads, each thread owns 4 consecutive pixels of a tile row.
// Shared memory: two float planes of (32 + 4l)^2.  Separable circular blur with taps h[2l+1]:
//   pass 1/2: r = A x - y on tile + l halo (from x on tile + 2l halo);  pass 3/4: g = A^T r on the tile (A^T = A: the
//   taps are symmetric by construction, sampling_images.py:306-314).
constexpr int BT = 32;
constexpr int MAX_L = 16;
// The taps travel BY VALUE in the kernel arguments (they then sit in the constant bank as FMA operands): a __constant__
// symbol would be one array per device, shared -- and raced on -- by every stream and host thread that blurs with other taps.
struct Taps {
  float v[2 * MAX_L + 1];
};

// i mod n for i in [-n, 2n) by one conditional correction; the general case (tiny images, halo wider than the image)
// falls back to the remainder.
__device__ __forceinline__ int wrap(int i, int n) {
  if (i < 0) i += n;
  if (i >= n) i -= n;
  if (i < 0 || i >= n) {
    i %= n;
    if (i < 0) i += n;
  }
  return i;
}

// All loops below are (row = warp, warp + 8, ...; column = lane, lane + 32, ...): no integer division in the hot path.
template <bool FULL, int C>  // FULL: Langevin pre; else: out = A x.  C: image channels (3 or 1)
__global__ void __launch_bounds__(256)
blur_kernel(PreArgs a, const Taps c_taps_arg, int B, int H, int W, int l, const float* __restrict__ x, const float* __restrict__ y, int y_B,
            const float* __restrict__ noise, float* __restrict__ out, __nv_bfloat16* __restrict__ den_in) {
  extern __shared__ float sm[];
  const int halo = FULL ? 2 * l : l;
  const int SW = BT + 2 * halo;  // staged width/height
  float* s0 = sm;
  float* s1 = sm + SW * SW;
  const int tiles_x = (W + BT - 1) / BT;
  const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
  const int b = blockIdx.y;
  const int x0 = tx * BT, y0 = ty * BT;
  const long long plane = (long long)H * W;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int prow = tid >> 3, pcol = (tid & 7) * 4;  // this thread's 4 pixels inside the tile
  const int nt = 2 * l + 1;
  const int w1 = SW - 2 * l, h1 = SW - 2 * l;  // extent after one pass of A
  float res[C][4];
  float xin[C][4];

#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float* xp = x + ((long long)b * C + c) * plane;
    __syncthreads();
    for (int r = warp; r < SW; r += 8) {
      const float* row = xp + (long long)wrap(y0 - halo + r, H) * W;
      for (int cc = lane; cc < SW; cc += 32) s0[r * SW + cc] = row[wrap(x0 - halo + cc, W)];
    }
    __syncthreads();
    // horizontal pass of A: s1[r][cc], cc in [0, w1)  <->  column x0 - halo + l + cc
    for (int r = warp; r < SW; r += 8)
      for (int cc = lane; cc < w1; cc += 32) {
        const float* src = s0 + r * SW + cc;
        float acc = 0.f;
        for (int t = 0; t < nt; ++t) acc = fmaf(c_taps_arg.v[t], src[t], acc);
        s1[r * SW + cc] = acc;
      }
    __syncthreads();
    // vertical pass of A (minus the observation for the Langevin step): s0[r][cc], r in [0, h1)
    const float* yp = FULL ? y + ((long long)(y_B > 1 ? b : 0) * C + c) * plane : nullptr;
    for (int r = warp; r < h1; r += 8) {
      const long long yrow = FULL ? (long long)wrap(y0 - l + r, H) * W : 0;
      for (int cc = lane; cc < w1; cc += 32) {
        const float* src = s1 + r * SW + cc;
        float acc = 0.f;
        for (int t = 0; t < nt; ++t) acc = fmaf(c_taps_arg.v[t], src[t * SW], acc);
        if (FULL) acc -= yp[yrow + wrap(x0 - l + cc, W)];
        s0[r * SW + cc] = acc;
      }
    }
    __syncthreads();
    if (!FULL) {
      // s0 holds A x on the tile (halo == l  =>  h1 == w1 == BT)
      const int gy = y0 + prow;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int gx = x0 + pcol + j;
        if (gy < H && gx < W) out[((long long)b * C + c) * plane + (long long)gy * W + gx] = s0[prow * SW + pcol + j];
      }
      continue;
    }
    // A^T r: horizontal then vertical on the (BT + 2l)^2 residual in s0 (A^T = A, the taps are symmetric)
    for (int r = warp; r < h1; r += 8) {
      const float* src = s0 + r * SW + lane;  // BT == 32 columns: one per lane
      float acc = 0.f;
      for (int t = 0; t < nt; ++t) acc = fmaf(c_taps_arg.v[t], src[t], acc);
      s1[r * SW + lane] = acc;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float* src = s1 + prow * SW + pcol + j;
      float acc = 0.f;
      for (int t = 0; t < nt; ++t) acc = fmaf(c_taps_arg.v[t], src[t * SW], acc);
      res[c][j] = acc;
    }
  }
  if (!FULL) return;

  const int gy = y0 + prow;
  if (gy >= H) return;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const long long rowoff = ((long long)b * C + c) * plane + (long long)gy * W;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gx = x0 + pcol + j;
      if (gx >= W) continue;
      const float xv = x[rowoff + gx];
      const long long e = (long long)c * plane + (long long)gy * W + gx;
      const float z = noise ? noise[rowoff + gx] : draw_at(a, b, (uint32_t)e);
      const float bv = langevin_base(a, xv, res[c][j], z);
      out[rowoff + gx] = bv;
      xin[c][j] = (a.alg == PSGLA_ALG_PNPULA) ? xv : bv;
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int gx = x0 + pcol + j;
    if (gx < W)
      store_nhwc16(den_in + ((long long)b * plane + (long long)gy * W + gx) * 16, xin[0][j], C > 1 ? xin[1 % C][j] : 0.f,
                   C > 2 ? xin[2 % C][j] : 0.f, a.den_in_c3);
  }
}

// ---- fast path: even half-width L known at compile time.
// Profiling showed the stencil is instruction-bound, not bandwidth-bound, so the kernel is written to spend its
// instructions on FMAs: wrap-around indices are hoisted out of the staging loops, every pass is register-tiled (one task
// = 4 consecutive outputs along the filtered direction from 4 + 2L staged values: three 16-byte shared-memory loads for
// 36 FMAs at L = 4), taps sit in registers, tile extents are compile-time, and the result is handed to row-quad owners
// through shared memory so that one Philox call serves 4 pixels.
template <bool FULL, int L>
struct BlurCfg {
  static constexpr int HALO = FULL ? 2 * L : L;
  static constexpr int SW = BT + 2 * HALO;  // staged extent of x
  static constexpr int W1 = SW - 2 * L;     // extent after one pass of A (= BT when !FULL)
  static constexpr size_t SMEM = (size_t)(2 * SW * SW + (FULL ? W1 * W1 : 0)) * sizeof(float);
};

template <bool FULL, int L, int C>
__global__ void __launch_bounds__(256, 3)
blur_kernel_t(PreArgs a, const Taps c_taps_arg, int B, int H, int W, const float* __restrict__ x, const float* __restrict__ y, int y_B,
              const float* __restrict__ noise, float* __restrict__ out, __nv_bfloat16* __restrict__ den_in) {
  using Cfg = BlurCfg<FULL, L>;
  constexpr int HALO = Cfg::HALO, SW = Cfg::SW, W1 = Cfg::W1;
  constexpr int NT = 2 * L + 1;
  constexpr int G1 = W1 / 4;  // 4-wide groups per row / per column after the first pass
  static_assert(L % 2 == 0, "the vectorised passes need an even half-width (W1 % 4 == 0)");
  static_assert(SW <= 96, "two column iterations per lane cover the staged row only up to 64 + 32");
  extern __shared__ float sm[];
  float* s0 = sm;                // [SW][SW]  x with halo, then the residual A x - y, then the result A^T(A x - y)
  float* s1 = sm + SW * SW;      // [SW][SW]  scratch between the passes
  float* sy = s1 + SW * SW;      // [W1][W1]  y on the residual's extent
  const int tiles_x = (W + BT - 1) / BT;
  const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
  const int b = blockIdx.y;
  const int x0 = tx * BT, y0 = ty * BT;
  const long long plane = (long long)H * W;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int prow = tid >> 3, pcol = (tid & 7) * 4;  // final owner: row prow, columns pcol..pcol+3 of the tile
  float h[NT];
#pragma unroll
  for (int t = 0; t < NT; ++t) h[t] = c_taps_arg.v[t];
  // wrapped global columns of this lane's staged columns (lane, lane + 32, lane + 64)
  int gxs[3], gys[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    gxs[i] = wrap(x0 - HALO + lane + 32 * i, W);
    gys[i] = wrap(x0 - L + lane + 32 * i, W);
  }
  float res[C][4], xc[C][4];
  // Global -> register staging of one channel's tile: every load of the channel is issued before the first dependent
  // store (an in-order warp otherwise pays one DRAM round trip per staged row), and channel c + 1 is fetched while
  // channel c runs its four passes.
  constexpr int XR = (SW + 7) / 8, YR = (W1 + 7) / 8;        // staged rows per warp
  constexpr int XI = (SW + 31) / 32, YI = (W1 + 31) / 32;    // staged columns per lane
  float xv[XR][XI], yv[FULL ? YR : 1][FULL ? YI : 1];
  auto fetch = [&](int c) {
    const float* xp = x + ((long long)b * C + c) * plane;
#pragma unroll
    for (int k = 0; k < XR; ++k) {
      const int r = warp + 8 * k;
      const float* row = xp + (long long)wrap(y0 - HALO + min(r, SW - 1), H) * W;
#pragma unroll
      for (int i = 0; i < XI; ++i) xv[k][i] = (r < SW && lane + 32 * i < SW) ? row[gxs[i]] : 0.f;
    }
    if (FULL) {
      const float* yp = y + ((long long)(y_B > 1 ? b : 0) * C + c) * plane;
#pragma unroll
      for (int k = 0; k < YR; ++k) {
        const int r = warp + 8 * k;
        const float* row = yp + (long long)wrap(y0 - L + min(r, W1 - 1), H) * W;
#pragma unroll
        for (int i = 0; i < YI; ++i) yv[k][i] = (r < W1 && lane + 32 * i < W1) ? row[gys[i]] : 0.f;
      }
    }
  };
  fetch(0);

#pragma unroll
  for (int c = 0; c < C; ++c) {
    __syncthreads();  // previous channel's readers of s0 / s1 are done
#pragma unroll
    for (int k = 0; k < XR; ++k) {
      const int r = warp + 8 * k;
#pragma unroll
      for (int i = 0; i < XI; ++i)
        if (r < SW && lane + 32 * i < SW) s0[r * SW + lane + 32 * i] = xv[k][i];
    }
    if (FULL) {
#pragma unroll
      for (int k = 0; k < YR; ++k) {
        const int r = warp + 8 * k;
#pragma unroll
        for (int i = 0; i < YI; ++i)
          if (r < W1 && lane + 32 * i < W1) sy[r * W1 + lane + 32 * i] = yv[k][i];
      }
    }
    if (c < C - 1) fetch(c + 1);
    __syncthreads();
    {
      const float4 v = *reinterpret_cast<const float4*>(s0 + (HALO + prow) * SW + HALO + pcol);  // x at the owned pixels
      xc[c][0] = v.x, xc[c][1] = v.y, xc[c][2] = v.z, xc[c][3] = v.w;
    }
    // horizontal pass of A: s1[r][0..W1)
    for (int task = tid; task < SW * G1; task += 256) {
      const int r = task / G1, g = task - r * G1;
      const float4* src4 = reinterpret_cast<const float4*>(s0 + r * SW + 4 * g);
      float in[4 + 2 * L];
#pragma unroll
      for (int q = 0; q < (4 + 2 * L) / 4; ++q) {
        const float4 v = src4[q];
        in[4 * q] = v.x, in[4 * q + 1] = v.y, in[4 * q + 2] = v.z, in[4 * q + 3] = v.w;
      }
      float o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < NT; ++t) acc = fmaf(h[t], in[k + t], acc);
        o[k] = acc;
      }
      *reinterpret_cast<float4*>(s1 + r * SW + 4 * g) = make_float4(o[0], o[1], o[2], o[3]);
    }
    __syncthreads();
    if (FULL) {
      // vertical pass of A minus the observation: residual on W1 x W1 into s0
      for (int task = tid; task < G1 * W1; task += 256) {
        const int g = task / W1, cc = task - g * W1;
        const float* src = s1 + (4 * g) * SW + cc;
        float in[4 + 2 * L];
#pragma unroll
        for (int j = 0; j < 4 + 2 * L; ++j) in[j] = src[j * SW];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float acc = 0.f;
#pragma unroll
          for (int t = 0; t < NT; ++t) acc = fmaf(h[t], in[k + t], acc);
          s0[(4 * g + k) * SW + cc] = acc - sy[(4 * g + k) * W1 + cc];
        }
      }
      __syncthreads();
      // A^T (= A): horizontal on W1 rows x BT columns
      for (int task = tid; task < W1 * (BT / 4); task += 256) {
        const int r = task / (BT / 4), g = task - r * (BT / 4);
        const float4* src4 = reinterpret_cast<const float4*>(s0 + r * SW + 4 * g);
        float in[4 + 2 * L];
#pragma unroll
        for (int q = 0; q < (4 + 2 * L) / 4; ++q) {
          const float4 v = src4[q];
          in[4 * q] = v.x, in[4 * q + 1] = v.y, in[4 * q + 2] = v.z, in[4 * q + 3] = v.w;
        }
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float acc = 0.f;
#pragma unroll
          for (int t = 0; t < NT; ++t) acc = fmaf(h[t], in[k + t], acc);
          o[k] = acc;
        }
        *reinterpret_cast<float4*>(s1 + r * SW + 4 * g) = make_float4(o[0], o[1], o[2], o[3]);
      }
      __syncthreads();
    }
    // last vertical pass (column lane, rows 4 warp .. 4 warp + 3), handed to the row-quad owners through s0
    {
      const float* src = s1 + (warp * 4) * SW + lane;
      float in[4 + 2 * L];
#pragma unroll
      for (int j = 0; j < 4 + 2 * L; ++j) in[j] = src[j * SW];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < NT; ++t) acc = fmaf(h[t], in[k + t], acc);
        s0[(warp * 4 + k) * SW + lane] = acc;
      }
    }
    __syncthreads();
    {
      const float4 v = *reinterpret_cast<const float4*>(s0 + prow * SW + pcol);
      res[c][0] = v.x, res[c][1] = v.y, res[c][2] = v.z, res[c][3] = v.w;
    }
  }

  const int gy = y0 + prow;
  if (gy >= H) return;
  const int gx0 = x0 + pcol;
  if (gx0 >= W) return;
  const bool full_quad = gx0 + 3 < W;
  float xin[C][4];
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const long long e0 = (long long)c * plane + (long long)gy * W + gx0;  // element index inside the chain
    const long long gi0 = (long long)b * C * plane + e0;
    if (!FULL) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (gx0 + j < W) out[gi0 + j] = res[c][j];
      continue;
    }
    float z[4];
    if (noise) {
#pragma unroll
      for (int j = 0; j < 4; ++j) z[j] = (gx0 + j < W) ? noise[gi0 + j] : 0.f;
    } else if ((e0 & 3) == 0) {
      draw_quad(a, b, (uint32_t)e0, z);  // one call, 4 pixels
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) z[j] = draw_at(a, b, (uint32_t)(e0 + j));
    }
    float bv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      bv[j] = langevin_base(a, xc[c][j], res[c][j], z[j]);
      xin[c][j] = (a.alg == PSGLA_ALG_PNPULA) ? xc[c][j] : bv[j];
    }
    if (full_quad && (gi0 & 3) == 0) {
      *reinterpret_cast<float4*>(out + gi0) = make_float4(bv[0], bv[1], bv[2], bv[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (gx0 + j < W) out[gi0 + j] = bv[j];
    }
  }
  if (FULL) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (gx0 + j < W)
        store_nhwc16(den_in + ((long long)b * plane + (long long)gy * W + gx0 + j) * 16, xin[0][j], C > 1 ? xin[1 % C][j] : 0.f,
                     C > 2 ? xin[2 % C][j] : 0.f, a.den_in_c3);
  }
}


// ------------------------------------------------------------------------------------------------ deblur pre, A^T A form
// A and A^T are the same symmetric separable circular operator (sampling_images.py:306-330; flip(h_) == h_ bit for bit), so
//   A^T(A x - y) = (A^T A) x - A^T y,   A^T A separable with the 1-D taps k = h * h (4l + 1 of them),
// and A^T y does not change during a run: the caller blurs y once (psgla_img_blur) and hands it in.  What is left per
// iteration is ONE horizontal and ONE vertical (4l + 1)-tap pass over x, done here as a row-streaming filter:
//   * a block of 192 threads owns a strip of 256 columns (the whole row of a 256-wide image: no horizontal halo) of all three
//     channels and walks RH + 4l input rows top to bottom; thread (channel, quad q) owns 4 consecutive columns;
//   * input rows arrive through a 4-deep cp.async ring in shared memory (wrap-around indices precomputed per thread);
//   * the horizontal pass is register-tiled (4 outputs from 4 + 4l staged values: five 16-byte shared loads for 68 FMAs);
//   * the vertical pass never touches shared memory: each thread keeps the last 4l + 1 horizontally filtered rows of its 4
//     columns in registers (the row loop is unrolled by 4l + 1 so that the ring is statically indexed);
//   * the Langevin step, the noise draw and the fp32 base store happen in the thread that owns the pixel; the bf16 NHWC16
//     denoiser input needs the three channels of a pixel together and is written one row late by the channel-0 threads from
//     a double-buffered shared-memory row;
//   * grayscale (C = 1): the three thread groups that take the three channels of a colour image take three bands of RH rows
//     of the one channel instead (a block covers 3 RH rows), so the block stays full; each thread stores its own pixels'
//     denoiser input.
// Per pixel-channel: 2 (4l + 1) FMAs against the 4-pass kernel's ~50 at l = 4 -- but what the 4-pass kernel really lost its
// time on was five block-wide barriers per channel-tile and a 2.25x read amplification; here it is two barriers per ROW and
// (RH + 4l) / RH.  Results differ from the two-pass-of-A formulation by fp32 rounding only (tests: 2e-5 relative).
constexpr int ATA_THREADS = 192;
constexpr int ATA_COLS = 256;   // strip width: 64 quads of 4 columns
constexpr int ATA_AHEAD = 3;    // input rows in flight beyond the one being filtered
struct Taps2 {
  float v[4 * 4 + 1];  // k = h * h for l <= 4
};
template <int K2>
struct AtaCfg {
  static constexpr int NT = 2 * K2 + 1;            // taps of A^T A
  static constexpr int SROW = ATA_COLS + 2 * K2;   // staged columns per channel
  static constexpr int ROWSET = 3 * SROW;          // floats of one staged row (3 channels)
  static constexpr int NBUF = K2 + ATA_AHEAD + 1;  // x ring: rows r - K2 (the centre of the output row) .. r + ATA_AHEAD
  static constexpr int NABUF = ATA_AHEAD + 1;      // A^T y ring
  static constexpr size_t SMEM = (size_t)(NBUF * ROWSET + NABUF * 3 * ATA_COLS + 2 * 3 * ATA_COLS) * sizeof(float);
};

// Phase P of the vertical window: the newest horizontally filtered row goes to slot P, the output row is the tap-weighted
// sum of slots P + 1, P + 2, ... (mod NT) = rows r - 2 K2 .. r.  One instantiation per phase keeps the window in registers
// with static indices; the row loop itself is NOT unrolled (an unrolled body per phase is ~5 KB of code per row step, 17 of
// them thrash the instruction cache: 2.3 us per row step measured).
template <int P, int NT>
__device__ __forceinline__ void ata_vpass(float (&hring)[NT][4], const float (&o)[4], const Taps2& k, bool emit, float (&g)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) hring[P][j] = o[j];
  if (emit) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float acc = 0.f;
#pragma unroll
      for (int t = 0; t < NT; ++t) acc = fmaf(k.v[t], hring[(P + 1 + t) % NT][j], acc);
      g[j] = acc;
    }
  }
}

// Two blocks per SM (156 registers).  A 96-register build with three resident blocks spills part of the window: 86 us
// instead of 58 (measured with scripts/blur_sweep.py, removed; commit 409bc30 is the last that contains it).
template <int K2, int C>  // K2 = 2 l: half-width of A^T A;  C: image channels (3 or 1)
__global__ void __launch_bounds__(ATA_THREADS, 2)
deblur_ata_kernel(PreArgs a, const Taps2 k, int B, int H, int W, int RH, const float* __restrict__ x,
                  const float* __restrict__ aty, int aty_B, const float* __restrict__ noise, float* __restrict__ out,
                  __nv_bfloat16* __restrict__ den_in) {
  using Cfg = AtaCfg<K2>;
  constexpr int NT = Cfg::NT, SROW = Cfg::SROW, ROWSET = Cfg::ROWSET, NBUF = Cfg::NBUF, NABUF = Cfg::NABUF;
  constexpr int NE = (ROWSET + ATA_THREADS - 1) / ATA_THREADS;
  extern __shared__ __align__(16) float ata_sm[];
  float* ring = ata_sm;                          // [NBUF][ROWSET]
  float* aring = ring + NBUF * ROWSET;           // [NABUF][3][ATA_COLS]: every thread stages and reads its own 4 floats
  float* xin_s = aring + NABUF * 3 * ATA_COLS;   // [2][3][ATA_COLS]
  const int tid = threadIdx.x;
  const int ch = tid >> 6, q = tid & 63;  // ch: the thread group's channel (C = 3) or row band (C = 1)
  const int b = blockIdx.z;
  const int x0 = blockIdx.x * ATA_COLS, y0 = blockIdx.y * RH * (3 / C);
  const int yb = C == 3 ? y0 : y0 + ch * RH;  // first output row of this thread group
  const int rh = min(RH, H - y0);        // output rows of this block (C = 1: of its first band, the longest)
  const int rhb = min(RH, H - yb);       // output rows of this thread group's band (C = 1)
  const int nrows = rh + 2 * K2;         // input rows it walks
  const long long plane = (long long)H * W;
  const float* xb = x + (long long)b * C * plane;
  const float* ab = aty + (long long)(aty_B > 1 ? b : 0) * C * plane + (long long)(C == 3 ? ch : 0) * plane;
  const int gx0 = x0 + 4 * q;
  const bool vec_ok = (W % 4 == 0) && gx0 + 3 < W;
  // this thread's staged elements: e = tid + 192 i  ->  (channel, staged column); global offset without the row term.
  // When W and the halo are multiples of 4, a staged quad of columns is one aligned, unwrapped quad in global memory:
  // 16-byte copies, (3 SROW / 4) / 192 = 2 per thread instead of 5 four-byte ones.
  constexpr int NQ = (ROWSET / 4 + ATA_THREADS - 1) / ATA_THREADS;
  const bool vstage = (K2 % 4 == 0) && (W % 4 == 0);
  unsigned goff[NE];
  int grow[NE];  // C = 1: the staged element's band, as its first input row minus K2
#pragma unroll
  for (int i = 0; i < NE; ++i) {
    const int e = vstage ? 4 * (tid + ATA_THREADS * i) : tid + ATA_THREADS * i;  // first element of the quad / the element
    const int c = e / SROW, col = e - c * SROW;
    goff[i] = (e < ROWSET) ? (unsigned)((long long)(C == 3 ? c : 0) * plane + wrap(x0 - K2 + col, W)) : 0u;
    grow[i] = y0 + c * RH - K2;
  }
  // One commit group per input row r: the row itself and the A^T y values of the output row it completes (r - 2 K2).
  auto stage = [&](int r) {
    if (r < nrows) {
      const long long rowoff = (long long)wrap(y0 - K2 + r, H) * W;
      float* dst = ring + (r % NBUF) * ROWSET;
      if (vstage) {
#pragma unroll
        for (int i = 0; i < NQ; ++i) {
          const int e = 4 * (tid + ATA_THREADS * i);
          if (e < ROWSET) {
            const unsigned saddr = (unsigned)__cvta_generic_to_shared(dst + e);
            const long long ro = C == 3 ? rowoff : (long long)wrap(grow[i] + r, H) * W;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(xb + ro + goff[i]) : "memory");
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < NE; ++i) {
          const int e = tid + ATA_THREADS * i;
          if (e < ROWSET) {
            const unsigned saddr = (unsigned)__cvta_generic_to_shared(dst + e);
            const long long ro = C == 3 ? rowoff : (long long)wrap(grow[i] + r, H) * W;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr), "l"(xb + ro + goff[i]) : "memory");
          }
        }
      }
      const int orow = r - 2 * K2;
      if (orow >= 0 && gx0 < W && (C == 3 || orow < rhb)) {
        const float* src = ab + (long long)(yb + orow) * W + gx0;
        float* adst = aring + ((orow % NABUF) * 3 + ch) * ATA_COLS + 4 * q;
        const unsigned saddr = (unsigned)__cvta_generic_to_shared(adst);
        if (vec_ok) {
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(src) : "memory");
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (gx0 + j < W) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr + 4 * j), "l"(src + j) : "memory");
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
#pragma unroll
  for (int r = 0; r < ATA_AHEAD; ++r) stage(r);

  float hring[NT][4];  // horizontally filtered rows r - 2 K2 .. r of this thread's 4 columns
#pragma unroll
  for (int t = 0; t < NT; ++t)
#pragma unroll
    for (int j = 0; j < 4; ++j) hring[t][j] = 0.f;

  // den_in of output row `orow` (tile-local), written by the channel-0 threads once all three channels are in xin_s (C = 3)
  auto flush_den_in = [&](int orow) {
    if (ch == 0 && gx0 < W) {
      const int gy = y0 + orow;
      const float* xs = xin_s + (orow & 1) * 3 * ATA_COLS + 4 * q;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (gx0 + j < W)
          store_nhwc16(den_in + ((long long)b * plane + (long long)gy * W + gx0 + j) * 16, xs[j], xs[ATA_COLS + j],
                       xs[2 * ATA_COLS + j], a.den_in_c3);
    }
  };

  int ph = 0;
  for (int r = 0; r < nrows; ++r) {
    asm volatile("cp.async.wait_group %0;" ::"n"(ATA_AHEAD - 1) : "memory");  // this thread's part of row r has landed
    __syncthreads();           // row r is visible to all; every thread has finished iteration r - 1
    stage(r + ATA_AHEAD);      // into the slot of row r - K2 - 1, whose last reader was iteration r - 1 (the centre row)
    if (C == 3 && r > 2 * K2) flush_den_in(r - 2 * K2 - 1);  // the previous output row's xin_s is complete
    // ---- horizontal pass on row r
    float o[4];
    {
      const float4* src4 = reinterpret_cast<const float4*>(ring + (r % NBUF) * ROWSET + ch * SROW + 4 * q);
      float in[4 + 2 * K2];
#pragma unroll
      for (int v = 0; v < (4 + 2 * K2) / 4; ++v) {
        const float4 t = src4[v];
        in[4 * v] = t.x, in[4 * v + 1] = t.y, in[4 * v + 2] = t.z, in[4 * v + 3] = t.w;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < NT; ++t) acc = fmaf(k.v[t], in[j + t], acc);
        o[j] = acc;
      }
    }
    // ---- vertical pass (window in registers, one code path per phase) for output row r - 2 K2
    const bool emit = r >= 2 * K2;
    float g[4] = {0.f, 0.f, 0.f, 0.f};
    switch (ph) {
#define PSGLA_ATA_CASE(P_)                                        \
  case P_:                                                        \
    if constexpr (P_ < NT) ata_vpass<P_, NT>(hring, o, k, emit, g); \
    break;
      PSGLA_ATA_CASE(0) PSGLA_ATA_CASE(1) PSGLA_ATA_CASE(2) PSGLA_ATA_CASE(3) PSGLA_ATA_CASE(4) PSGLA_ATA_CASE(5)
      PSGLA_ATA_CASE(6) PSGLA_ATA_CASE(7) PSGLA_ATA_CASE(8) PSGLA_ATA_CASE(9) PSGLA_ATA_CASE(10) PSGLA_ATA_CASE(11)
      PSGLA_ATA_CASE(12) PSGLA_ATA_CASE(13) PSGLA_ATA_CASE(14) PSGLA_ATA_CASE(15) PSGLA_ATA_CASE(16)
#undef PSGLA_ATA_CASE
      default: break;
    }
    if (++ph == NT) ph = 0;
    // ---- Langevin step
    if (emit) {
      const int orow = r - 2 * K2;
      const int gy = yb + orow;
      float xin[4] = {0.f, 0.f, 0.f, 0.f};
      if (gx0 < W && (C == 3 || orow < rhb)) {
        const long long e0 = (long long)(C == 3 ? ch : 0) * plane + (long long)gy * W + gx0;  // element index inside the chain
        const long long gi0 = (long long)b * C * plane + e0;
        float xv[4], av[4], z[4];
        const float* xc = ring + ((r - K2) % NBUF) * ROWSET + ch * SROW + K2 + 4 * q;  // the output row itself, still staged
        const float* ac = aring + ((orow % NABUF) * 3 + ch) * ATA_COLS + 4 * q;
#pragma unroll
        for (int j = 0; j < 4; ++j) xv[j] = xc[j], av[j] = ac[j];
        if (noise) {
#pragma unroll
          for (int j = 0; j < 4; ++j) z[j] = (gx0 + j < W) ? noise[gi0 + j] : 0.f;
        } else if ((e0 & 3) == 0) {
          draw_quad(a, b, (uint32_t)e0, z);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) z[j] = draw_at(a, b, (uint32_t)(e0 + j));
        }
        float bv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          bv[j] = langevin_base(a, xv[j], g[j] - av[j], z[j]);
          xin[j] = (a.alg == PSGLA_ALG_PNPULA) ? xv[j] : bv[j];
        }
        if (vec_ok) {
          *reinterpret_cast<float4*>(out + gi0) = make_float4(bv[0], bv[1], bv[2], bv[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (gx0 + j < W) out[gi0 + j] = bv[j];
        }
        if (C == 1) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (gx0 + j < W) store_nhwc16(den_in + ((long long)b * plane + (long long)gy * W + gx0 + j) * 16, xin[j], 0.f, 0.f, a.den_in_c3);
        }
      }
      if (C == 3)
        *reinterpret_cast<float4*>(xin_s + ((orow & 1) * 3 + ch) * ATA_COLS + 4 * q) = make_float4(xin[0], xin[1], xin[2], xin[3]);
    }
  }
  if (C == 3) {
    __syncthreads();
    flush_den_in(rh - 1);
  }
}

__global__ void __launch_bounds__(256)
noise_kernel(int B, long long chw, unsigned long long seed, long long chain_id0, unsigned int iteration,
             float* __restrict__ out) {
  const long long quads = (chw + 3) / 4;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= quads * B) return;
  const int b = (int)(g / quads);
  const long long q = g % quads;
  float z[4];
  normal_quad(seed, (unsigned long long)(chain_id0 + b), iteration, (uint32_t)q, z);
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (q * 4 + j < chw) out[(long long)b * chw + q * 4 + j] = z[j];
}

__global__ void __launch_bounds__(256)
noise_torch_cuda_kernel(long long numel, unsigned long long seed, unsigned long long offset, unsigned int T,
                        float* __restrict__ out) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < numel) out[g] = torch_cuda_normal_at(seed, offset, T, (uint64_t)g);
}

template <int C>
__global__ void __launch_bounds__(256)
to_nhwc16_kernel(int B, int H, int W, const float* __restrict__ x, float c3, __nv_bfloat16* __restrict__ out) {
  const long long plane = (long long)H * W;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= plane * B) return;
  const long long b = g / plane, pix = g % plane;
  const float* xp = x + b * C * plane + pix;
  store_nhwc16(out + g * 16, xp[0], C > 1 ? xp[plane] : 0.f, C > 2 ? xp[2 * plane] : 0.f, c3);
}

// Replication padding of a bf16 NHWC16 image batch in place: pixels with y >= H or x >= W (the pad a U-Net needs to reach a
// multiple of 8) copy the nearest valid pixel -- KAIR's test_pad (ReplicationPad2d on the bottom / right).
__global__ void __launch_bounds__(256)
pad_replicate_nhwc16_kernel(int B, int Hp, int Wp, int H, int W, __nv_bfloat16* __restrict__ img) {
  const int n_pad_per_chain = Hp * Wp - H * W;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (long long)n_pad_per_chain * B) return;
  const int b = (int)(g / n_pad_per_chain);
  int k = (int)(g % n_pad_per_chain);
  int y, x;
  if (k < H * (Wp - W)) {  // right band of the valid rows
    y = k / (Wp - W);
    x = W + k % (Wp - W);
  } else {                 // bottom band, full padded width
    k -= H * (Wp - W);
    y = H + k / Wp;
    x = k % Wp;
  }
  const int ys = min(y, H - 1), xs = min(x, W - 1);
  const uint4* src = reinterpret_cast<const uint4*>(img + (((long long)b * Hp + ys) * Wp + xs) * 16);
  uint4* dst = reinterpret_cast<uint4*>(img + (((long long)b * Hp + y) * Wp + x) * 16);
  dst[0] = src[0];
  dst[1] = src[1];
}

int fill_pre(const psgla_pre_params* p, PreArgs* a) {
  PSGLA_REQUIRE(p != nullptr, "null psgla_pre_params");
  PSGLA_REQUIRE(p->alg == PSGLA_ALG_PSGLA || p->alg == PSGLA_ALG_PNPULA, "alg=%d is not a PSGLA_ALG_* value", p->alg);
  PSGLA_REQUIRE(p->iteration >= 0 && p->iteration <= 0xffffffffLL && p->chain_id0 >= 0, "iteration / chain id out of range");
  a->alg = p->alg;
  a->gain_data = p->gain_data;
  a->noise_scale = p->noise_scale;
  a->proj_gain = p->proj_gain;
  a->c_min = p->c_min;
  a->c_max = p->c_max;
  a->x_gain = p->x_gain;
  a->den_in_c3 = p->den_in_c3;
  a->seed = p->seed;
  a->chain_id0 = p->chain_id0;
  a->iteration = (unsigned int)p->iteration;
  PSGLA_REQUIRE(p->noise_mode == PSGLA_NOISE_PHILOX || p->noise_mode == PSGLA_NOISE_TORCH_CUDA,
                "noise_mode=%d is not a PSGLA_NOISE_* value", p->noise_mode);
  PSGLA_REQUIRE(p->noise_mode != PSGLA_NOISE_TORCH_CUDA || (p->torch_threads >= 256 && p->torch_threads % 256 == 0 &&
                                                            p->torch_offset % 4 == 0),
                "PSGLA_NOISE_TORCH_CUDA needs torch_threads (a multiple of 256) and torch_offset (a multiple of 4) from "
                "psgla_torch_cuda_randn_policy");
  a->noise_mode = p->noise_mode;
  a->torch_threads = p->torch_threads;
  a->torch_offset = p->torch_offset;
  a->chw = 0;  // set by the caller once the shape is checked
  return PSGLA_OK;
}

// C = 3 (colour) or 1 (grayscale): the kernels take the channel count as a template parameter
static int check_img(const psgla_img_shape& s) {
  PSGLA_REQUIRE(s.B > 0 && s.H > 0 && s.W > 0 && (s.C == 3 || s.C == 1),
                "image shape must be [B>0][C = 1 or 3][H>0][W>0], got [%d][%d][%d][%d]", s.B, s.C, s.H, s.W);
  PSGLA_REQUIRE((long long)s.C * s.H * s.W < (1LL << 32), "one chain must have fewer than 2^32 elements");
  return PSGLA_OK;
}

static int make_taps(const float* h1d_host, int l, Taps* t) {
  PSGLA_REQUIRE(h1d_host != nullptr && l >= 0 && l <= MAX_L, "blur half-width l must be in 0..%d (got %d)", MAX_L, l);
  std::memset(t, 0, sizeof(*t));
  std::memcpy(t->v, h1d_host, sizeof(float) * (2 * l + 1));
  return PSGLA_OK;
}

}  // namespace psgla

using namespace psgla;

extern "C" int psgla_img_pre_inpaint(const psgla_pre_params* p, psgla_img_shape s, const float* x_dev,
                                     const float* mask_dev, int mask_B, const float* y_dev, int y_B,
                                     const float* noise_dev, float* base_dev, void* den_in_dev, void* stream) {
  PreArgs a;
  int rc = fill_pre(p, &a);
  if (rc) return rc;
  rc = check_img(s);
  if (rc) return rc;
  PSGLA_REQUIRE(x_dev && mask_dev && y_dev && base_dev && den_in_dev, "psgla_img_pre_inpaint: null pointer");
  PSGLA_REQUIRE((mask_B == 1 || mask_B == s.B) && (y_B == 1 || y_B == s.B), "mask_B / y_B must be 1 or B");
  const long long plane = (long long)s.H * s.W;
  a.chw = s.C * plane;
  cudaStream_t st = (cudaStream_t)stream;
  const int vec = plane % 4 == 0 ? 4 : 1;
  const long long n = plane / vec * s.B;
  auto kern = vec == 4 ? (s.C == 3 ? pre_inpaint_kernel<4, 3> : pre_inpaint_kernel<4, 1>)
                       : (s.C == 3 ? pre_inpaint_kernel<1, 3> : pre_inpaint_kernel<1, 1>);
  kern<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a, s.B, s.H, s.W, x_dev, mask_dev, mask_B, y_dev, y_B, noise_dev, base_dev,
                                                    (__nv_bfloat16*)den_in_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

template <bool FULL, int L, int C>
static int launch_blur_t(const PreArgs& a, const Taps& taps, psgla_img_shape s, const float* x, const float* y, int y_B,
                         const float* noise, float* out, void* den_in, cudaStream_t st) {
  constexpr size_t smem = BlurCfg<FULL, L>::SMEM;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (smem > 48 * 1024 && !(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(blur_kernel_t<FULL, L, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  const int tiles = ((s.W + BT - 1) / BT) * ((s.H + BT - 1) / BT);
  blur_kernel_t<FULL, L, C><<<dim3(tiles, s.B), 256, smem, st>>>(a, taps, s.B, s.H, s.W, x, y, y_B, noise, out, (__nv_bfloat16*)den_in);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

template <bool FULL, int C>
static int launch_blur(const PreArgs& a, const Taps& taps, psgla_img_shape s, int l, const float* x, const float* y, int y_B,
                       const float* noise, float* out, void* den_in, cudaStream_t st) {
  switch (l) {  // compile-time even half-widths (the reference's default is l = 4); anything else takes the generic kernel
    case 2: return launch_blur_t<FULL, 2, C>(a, taps, s, x, y, y_B, noise, out, den_in, st);
    case 4: return launch_blur_t<FULL, 4, C>(a, taps, s, x, y, y_B, noise, out, den_in, st);
    case 6: return launch_blur_t<FULL, 6, C>(a, taps, s, x, y, y_B, noise, out, den_in, st);
    case 8: return launch_blur_t<FULL, 8, C>(a, taps, s, x, y, y_B, noise, out, den_in, st);
    default: break;
  }
  const int halo = FULL ? 2 * l : l;
  const int SW = BT + 2 * halo;
  const size_t smem = (size_t)2 * SW * SW * sizeof(float);
  if (smem > 48 * 1024)  // a per-device attribute of the function, cheap to set: no process-wide cache
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(blur_kernel<FULL, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles = ((s.W + BT - 1) / BT) * ((s.H + BT - 1) / BT);
  blur_kernel<FULL, C><<<dim3(tiles, s.B), 256, smem, st>>>(a, taps, s.B, s.H, s.W, l, x, y, y_B, noise, out,
                                                        (__nv_bfloat16*)den_in);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

extern "C" int psgla_img_pre_deblur(const psgla_pre_params* p, psgla_img_shape s, const float* x_dev,
                                    const float* h1d_host, int l, const float* y_dev, int y_B, const float* noise_dev,
                                    float* base_dev, void* den_in_dev, void* stream) {
  PreArgs a;
  int rc = fill_pre(p, &a);
  if (rc) return rc;
  rc = check_img(s);
  if (rc) return rc;
  PSGLA_REQUIRE(x_dev && y_dev && base_dev && den_in_dev, "psgla_img_pre_deblur: null pointer");
  PSGLA_REQUIRE(x_dev != base_dev, "psgla_img_pre_deblur: base must not alias x (the stencil reads neighbours)");
  PSGLA_REQUIRE(y_B == 1 || y_B == s.B, "y_B must be 1 or B");
  a.chw = (long long)s.C * s.H * s.W;
  Taps taps;
  rc = make_taps(h1d_host, l, &taps);
  if (rc) return rc;
  return (s.C == 3 ? launch_blur<true, 3> : launch_blur<true, 1>)(a, taps, s, l, x_dev, y_dev, y_B, noise_dev, base_dev,
                                                                  den_in_dev, (cudaStream_t)stream);
}

// k = h * h (full 1-D convolution, 4 l + 1 taps) in double, rounded once.
static void ata_taps(const float* h, int l, Taps2* k) {
  std::memset(k, 0, sizeof(*k));
  const int n = 2 * l + 1;
  for (int i = 0; i < 2 * n - 1; ++i) {
    double acc = 0;
    for (int j = 0; j < n; ++j)
      if (i - j >= 0 && i - j < n) acc += (double)h[j] * (double)h[i - j];
    k->v[i] = (float)acc;
  }
}

template <int K2, int C>
static int launch_ata(const PreArgs& a, const Taps2& k, psgla_img_shape s, const float* x, const float* aty, int aty_B,
                      const float* noise, float* out, void* den_in, cudaStream_t st) {
  // rows per block: two blocks are resident per SM (registers) and hide each other's latencies, so the launch takes about
  // ceil(blocks / (2 SMs)) rounds of RH + 2 K2 row steps (measured at 32 chains of 256 x 256, l = 4: RH = 8 / 16 / 32 / 64 / 128
  // -> 83 / 66 / 59 / 82 / 152 us; the four-pass kernel 84 us).  A grayscale block covers `bands` = 3 bands of RH rows in the
  // same RH + 2 K2 row steps, so the cost model holds for it with three times the rows per block.
  const int bands = 3 / C;
  const int strips = (s.W + ATA_COLS - 1) / ATA_COLS, sms = 2 * num_sms();
  int best_rh = 16;
  long long best = -1;
  for (int rh = 8; rh <= 128; rh *= 2) {
    const long long blocks = (long long)strips * ((s.H + bands * rh - 1) / (bands * rh)) * s.B;
    const long long cost = ((blocks + sms - 1) / sms) * (rh + 2 * K2);
    if (best < 0 || cost < best) best = cost, best_rh = rh;
  }
  const int row_blocks = (s.H + bands * best_rh - 1) / (bands * best_rh);
  PSGLA_REQUIRE(s.B <= 65535 && row_blocks <= 65535, "too many chains / rows for one launch");
  constexpr size_t smem = AtaCfg<K2>::SMEM;
  static std::atomic<unsigned long long> attr_done{0};  // bit d: opted in on device d (a per-device function attribute)
  const unsigned long long dev_bit = 1ull << (current_device() & 63);
  if (smem > 48 * 1024 && !(attr_done.load(std::memory_order_acquire) & dev_bit)) {
    PSGLA_CUDA_TRY(cudaFuncSetAttribute(deblur_ata_kernel<K2, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done.fetch_or(dev_bit, std::memory_order_release);
  }
  deblur_ata_kernel<K2, C><<<dim3(strips, row_blocks, s.B), ATA_THREADS, smem, st>>>(
      a, k, s.B, s.H, s.W, best_rh, x, aty, aty_B, noise, out, (__nv_bfloat16*)den_in);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

extern "C" int psgla_img_pre_deblur_ata(const psgla_pre_params* p, psgla_img_shape s, const float* x_dev,
                                        const float* h1d_host, int l, const float* aty_dev, int aty_B,
                                        const float* noise_dev, float* base_dev, void* den_in_dev, void* stream) {
  PreArgs a;
  int rc = fill_pre(p, &a);
  if (rc) return rc;
  rc = check_img(s);
  if (rc) return rc;
  PSGLA_REQUIRE(x_dev && aty_dev && base_dev && den_in_dev && h1d_host, "psgla_img_pre_deblur_ata: null pointer");
  PSGLA_REQUIRE(x_dev != base_dev, "psgla_img_pre_deblur_ata: base must not alias x (the stencil reads neighbours)");
  PSGLA_REQUIRE(aty_B == 1 || aty_B == s.B, "aty_B must be 1 or B");
  PSGLA_REQUIRE(l >= 1 && l <= 4, "psgla_img_pre_deblur_ata serves half-widths 1..4 (got %d); use psgla_img_pre_deblur", l);
  a.chw = (long long)s.C * s.H * s.W;
  Taps2 k;
  ata_taps(h1d_host, l, &k);
  cudaStream_t st = (cudaStream_t)stream;
  const bool gray = s.C == 1;
  switch (l) {
    case 1: return (gray ? launch_ata<2, 1> : launch_ata<2, 3>)(a, k, s, x_dev, aty_dev, aty_B, noise_dev, base_dev, den_in_dev, st);
    case 2: return (gray ? launch_ata<4, 1> : launch_ata<4, 3>)(a, k, s, x_dev, aty_dev, aty_B, noise_dev, base_dev, den_in_dev, st);
    case 3: return (gray ? launch_ata<6, 1> : launch_ata<6, 3>)(a, k, s, x_dev, aty_dev, aty_B, noise_dev, base_dev, den_in_dev, st);
    default: return (gray ? launch_ata<8, 1> : launch_ata<8, 3>)(a, k, s, x_dev, aty_dev, aty_B, noise_dev, base_dev, den_in_dev, st);
  }
}

extern "C" int psgla_img_blur(psgla_img_shape s, const float* x_dev, const float* h1d_host, int l, float* out_dev,
                              void* stream) {
  int rc = check_img(s);
  if (rc) return rc;
  PSGLA_REQUIRE(x_dev && out_dev && x_dev != out_dev, "psgla_img_blur: null or aliased pointer");
  Taps taps;
  rc = make_taps(h1d_host, l, &taps);
  if (rc) return rc;
  PreArgs a{};
  return (s.C == 3 ? launch_blur<false, 3> : launch_blur<false, 1>)(a, taps, s, l, x_dev, nullptr, 1, nullptr, out_dev, nullptr,
                                                                    (cudaStream_t)stream);
}

extern "C" int psgla_img_noise(psgla_img_shape s, uint64_t seed, int64_t chain_id0, int64_t iteration, float* out_dev,
                               void* stream) {
  int rc = check_img(s);
  if (rc) return rc;
  PSGLA_REQUIRE(out_dev && iteration >= 0 && iteration <= 0xffffffffLL && chain_id0 >= 0, "psgla_img_noise: bad argument");
  const long long chw = (long long)s.C * s.H * s.W;
  const long long n = (chw + 3) / 4 * s.B;
  noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(s.B, chw, seed, chain_id0,
                                                                             (unsigned int)iteration, out_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

extern "C" int psgla_torch_cuda_randn_policy(int64_t numel, int sm_count, int max_threads_per_sm, uint32_t* threads,
                                             uint64_t* offset_step) {
  PSGLA_REQUIRE(numel > 0 && threads && offset_step, "psgla_torch_cuda_randn_policy: bad argument");
  if (sm_count <= 0) {
    int dev = 0;
    PSGLA_CUDA_TRY(cudaGetDevice(&dev));
    PSGLA_CUDA_TRY(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev));
    PSGLA_CUDA_TRY(cudaDeviceGetAttribute(&max_threads_per_sm, cudaDevAttrMaxThreadsPerMultiProcessor, dev));
  }
  PSGLA_REQUIRE(max_threads_per_sm >= 256, "max_threads_per_sm must be >= 256");
  // ATen/native/cuda/DistributionTemplates.h calc_execution_policy: block 256, unroll 4 (one curand_normal4 per stride)
  const uint64_t block = 256, unroll = 4;
  uint64_t grid = ((uint64_t)numel + block - 1) / block;
  const uint64_t cap = (uint64_t)sm_count * (uint64_t)(max_threads_per_sm / 256);
  if (grid > cap) grid = cap;
  PSGLA_REQUIRE(grid * block < (1ull << 32), "launch too large");
  *threads = (uint32_t)(grid * block);
  *offset_step = (((uint64_t)numel - 1) / (block * grid * unroll) + 1) * 4;
  return PSGLA_OK;
}

extern "C" int psgla_img_noise_torch_cuda(int64_t numel, uint64_t seed, uint64_t offset, uint32_t threads, float* out_dev,
                                          void* stream) {
  PSGLA_REQUIRE(out_dev && numel > 0 && threads >= 256 && threads % 256 == 0 && offset % 4 == 0,
                "psgla_img_noise_torch_cuda: bad argument");
  noise_torch_cuda_kernel<<<(unsigned)((numel + 255) / 256), 256, 0, (cudaStream_t)stream>>>(numel, seed, offset, threads,
                                                                                            out_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

extern "C" int psgla_img_pad_replicate_nhwc16(psgla_img_shape padded, int H, int W, void* img_dev, void* stream) {
  int rc = check_img(padded);
  if (rc) return rc;
  PSGLA_REQUIRE(img_dev && H >= 1 && W >= 1 && H <= padded.H && W <= padded.W, "psgla_img_pad_replicate_nhwc16: bad argument");
  const long long n = ((long long)padded.H * padded.W - (long long)H * W) * padded.B;
  if (n == 0) return PSGLA_OK;
  pad_replicate_nhwc16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(padded.B, padded.H, padded.W, H, W,
                                                                                            (__nv_bfloat16*)img_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

extern "C" int psgla_img_to_nhwc16(psgla_img_shape s, const float* x_dev, float c3, void* out_dev, void* stream) {
  int rc = check_img(s);
  if (rc) return rc;
  PSGLA_REQUIRE(x_dev && out_dev, "psgla_img_to_nhwc16: null pointer");
  const long long n = (long long)s.H * s.W * s.B;
  (s.C == 3 ? to_nhwc16_kernel<3> : to_nhwc16_kernel<1>)<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      s.B, s.H, s.W, x_dev, c3, (__nv_bfloat16*)out_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}
