// Gradient-step DRUNet denoiser (deepinv.models.GSDRUNet as the reference's image driver builds it, sampling_images.py:129-140;
// Prox-DRUNet is the same network from another checkpoint):
//   N   = KAIR UNetRes with nc = [64, 128, 256, 512], nb = 2 residual blocks x -> x + conv(elu(conv(x))) per stage, no biases,
//         the noise-level map of sigma as fourth input channel (tests/gs_reference.py restates it)
//   g   = 1/2 ||x - N(x)||^2,   grad g(x) = v - J^T v  with v = x - N(x)  (the sigma channel's gradient is dropped)
//   D   = x - alpha grad g(x)
//
// One call runs N's 36 layers, one element-wise kernel and the 36 layers of J^T v.  The backward is the U-Net walked in
// reverse, every layer the adjoint of a forward layer and run by the kernel of a forward layer of the same shape:
//   3x3 "same" conv     -> 3x3 conv with transposed channels and flipped taps (the head's adjoint is tail-shaped and vice versa)
//   2x2 stride-2 conv   -> 2x2 stride-2 transposed conv, the same weight tensor read as [cin][cout][2][2]
//   2x2 transposed conv -> 2x2 stride-2 conv, the same weight tensor read as OIHW
// A residual block x + c2(elu(c1 x)) has the backward g -> g + c1^T(elu'(z) * c2^T g): c2^T runs the gate epilogue (its input
// t = elu(z) is the bf16 tensor the forward stored) and c1^T adds g as res1.  A U-Net skip x_s + ... becomes a held gradient
// tensor, added as res2 where the gradient of the encoder feature x_s is produced (the first block's c1^T of that stage).
// The element-wise kernel forms v (bf16 NHWC16, the first backward layer's input) and base' = base_scale base +
// gain (x - alpha v); the last backward layer's fused post then writes X+ = base' + (gain alpha) J^T v = base_scale base + gain D(x).
#include <cmath>
#include <cstring>
#include <vector>

#include <cuda_bf16.h>

#include "common.cuh"
#include "conv_api.cuh"

namespace psgla {

constexpr int GS_LAYERS = 36;  // per direction
constexpr int GS_ELU = 14;     // residual blocks, each keeps its ELU output for the backward

struct GsLayer {
  DruKind kind;
  int cin, cout;
  int scale;  // the layer's input is (H >> scale) x (W >> scale)
  int act;    // ConvAct: ACT_ELU (forward c1), ACT_GATE (backward c2^T), else ACT_NONE
  int nres;   // residual inputs: 1 = res1, 2 = res1 and res2 (as in drunet.cu)
  int src;    // the state-dict weight tensor it is packed from
  size_t w_off, bytes;
};

// [0, 36): the forward in state-dict order (m_head, m_down1.{0,1}.res.{0,2}, m_down1.2, ..., m_body.*, m_up3.0,
// m_up3.{1,2}.res.{0,2}, ..., m_tail); [36, 72): backward layer b = the adjoint of forward layer 35 - b.
static const std::vector<GsLayer>& gs_plan() {
  static std::vector<GsLayer> plan;
  if (!plan.empty()) return plan;
  std::vector<GsLayer> v;
  std::vector<int> bres2;  // forward c1 layers whose adjoint also adds a held skip gradient
  const int nc[4] = {64, 128, 256, 512};
  auto add = [&](DruKind k, int cin, int cout, int scale, int act, int nres) {
    v.push_back({k, cin, cout, scale, act, nres, (int)v.size(), 0, 0});
  };
  // two residual blocks; `skip`: the last adds the U-Net skip; `grad_skip`: the input is a skip feature x_s
  auto blocks = [&](int s, bool skip, bool grad_skip) {
    for (int i = 0; i < 4; ++i) {
      if (i == 0 && grad_skip) bres2.push_back((int)v.size());
      add(s == 0 ? DRU_C64 : DRU_GEMM3, nc[s], nc[s], s, i % 2 == 0 ? ACT_ELU : ACT_NONE,
          i % 2 == 0 ? 0 : (skip && i == 3 ? 2 : 1));
    }
  };
  add(DRU_HEAD, 4, 64, 0, ACT_NONE, 0);
  for (int s = 0; s < 3; ++s) {
    blocks(s, false, true);
    add(DRU_DOWN, nc[s], nc[s + 1], s, ACT_NONE, 0);
  }
  blocks(3, true, true);
  for (int s = 2; s >= 0; --s) {
    add(DRU_UP, nc[s + 1], nc[s], s + 1, ACT_NONE, 0);
    blocks(s, true, false);
  }
  add(DRU_TAIL, 64, 3, 0, ACT_NONE, 0);
  for (int b = 0; b < GS_LAYERS; ++b) {
    const GsLayer F = v[GS_LAYERS - 1 - b];
    GsLayer A = F;
    A.cin = F.cout;
    A.cout = F.cin;
    A.act = ACT_NONE;
    A.nres = 0;
    switch (F.kind) {
      case DRU_HEAD: A.kind = DRU_TAIL, A.cout = 3; break;  // the sigma channel's gradient is dropped
      case DRU_TAIL: A.kind = DRU_HEAD; break;
      case DRU_DOWN: A.kind = DRU_UP, A.scale = F.scale + 1; break;
      case DRU_UP: A.kind = DRU_DOWN, A.scale = F.scale - 1; break;
      default:
        if (F.act == ACT_ELU) {
          A.nres = 1;
          for (int l : bres2)
            if (l == F.src) A.nres = 2;
        } else {
          A.act = ACT_GATE;
        }
    }
    v.push_back(A);
  }
  size_t off = 0;
  for (auto& L : v) {
    L.bytes = dru_layer_bytes(L.kind, L.cin, L.cout);
    L.w_off = off;
    off += L.bytes;
  }
  plan.swap(v);
  return plan;
}

static size_t gs_align(size_t n) { return (n + 1023) / 1024 * 1024; }

struct GsBuffers {
  uint8_t* buf[4][4];  // [scale][4]: forward ping-pong (slot 0: the skip feature x_s), then backward (slot 0: the skip gradient)
  uint8_t* elu[GS_ELU];
  float* n_out;        // N(x), fp32 NCHW
  float* base2;        // base', fp32 NCHW
  uint8_t* v16;        // v, bf16 NHWC16
};

static int gs_elu_scale(int k) {  // forward order: encoder 0, 1, 2, body, decoder 2, 1, 0 -- two blocks each
  const int stage = k / 2;
  return stage <= 3 ? stage : 6 - stage;
}

static size_t gs_layout(int B, int H, int W, uint8_t* base, GsBuffers* b) {
  size_t off = 0;
  auto take = [&](size_t n) {
    uint8_t* p = base ? base + off : nullptr;
    off += gs_align(n);
    return p;
  };
  const size_t px = (size_t)B * H * W;
  for (int s = 0; s < 4; ++s)
    for (int j = 0; j < 4; ++j) {
      uint8_t* p = take(px / ((size_t)1 << (2 * s)) * (64 << s) * 2);
      if (b) b->buf[s][j] = p;
    }
  for (int k = 0; k < GS_ELU; ++k) {
    const int s = gs_elu_scale(k);
    uint8_t* p = take(px / ((size_t)1 << (2 * s)) * (64 << s) * 2);
    if (b) b->elu[k] = p;
  }
  uint8_t* n_out = take(px * 3 * 4);
  uint8_t* base2 = take(px * 3 * 4);
  uint8_t* v16 = take(px * 16 * 2);
  if (b) {
    b->n_out = (float*)n_out;
    b->base2 = (float*)base2;
    b->v16 = v16;
  }
  return off + 1024;  // + alignment slack of the caller's pointer
}

struct GsPost {  // the fused post of the last layer of a direction; base == NULL: x_out = the raw fp32 NCHW conv
  const float* base;
  float base_scale, gain, w_old, w_new;
  float* x_out;
  float* sample;
  float* mean;
  float* mean2;
  const psgla_next_pre* next;
};

// Plan layer l (0..71) with its inputs: res1 / res2 residual adds, gate = the stored ELU output of ACT_GATE layers.
static int gs_layer(const uint8_t* packed, int l, int B, int H, int W, const void* in, const void* res1, const void* res2,
                    const void* gate, void* out, const GsPost& post, cudaStream_t st) {
  const GsLayer& L = gs_plan()[l];
  const uint8_t* w = packed + L.w_off;
  const int h = H >> L.scale, wd = W >> L.scale;
  if (L.act == ACT_GATE) res1 = gate;
  auto bias = [&](int nout_pad, int cin_pad) { return reinterpret_cast<const float*>(w + (size_t)9 * nout_pad * cin_pad * 2); };
  switch (L.kind) {
    case DRU_HEAD: return conv_first16(in, out, w, bias(64, 16), B, H, W, 0, st);
    case DRU_C64: return conv64_hidden(in, out, w, bias(64, 64), B, h, wd, L.act, res1, res2, st);
    case DRU_GEMM3: return conv_gemm_layer(0, B, h, wd, L.cin, L.cout, w, in, res1, res2, out, L.act, st);
    case DRU_DOWN: return conv_gemm_layer(1, B, h, wd, L.cin, L.cout, w, in, nullptr, nullptr, out, ACT_NONE, st);
    case DRU_UP: return conv_gemm_layer(2, B, h, wd, L.cin, L.cout, w, in, nullptr, nullptr, out, ACT_NONE, st);
    case DRU_TAIL:
      return conv_last_post(in, w, bias(16, 64), B, 3, H, W, post.base, post.base_scale, post.gain, post.w_old, post.w_new,
                            post.x_out, post.sample, post.mean, post.mean2, post.next, st);
  }
  return set_error(PSGLA_E_BADARG, "GSDRUNet layer %d: unknown kind", l);
}

// v = x - N as bf16 NHWC16 (channels 3..15 zero) and base' = base_scale base + gain (x - alpha v), per pixel.
__global__ void __launch_bounds__(256)
gs_cotangent_kernel(int B, int HW, const float* __restrict__ x, const float* __restrict__ base, const float* __restrict__ n_out,
                    float alpha, float base_scale, float gain, __nv_bfloat16* __restrict__ v16, float* __restrict__ base2) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (long long)B * HW) return;
  const long long b = g / HW, pix = g % HW;
  __align__(16) __nv_bfloat16 o[16];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const long long i = (b * 3 + c) * HW + pix;
    const float xv = x[i];
    const float vv = xv - n_out[i];
    o[c] = __float2bfloat16_rn(vv);
    base2[i] = base_scale * base[i] + gain * (xv - alpha * vv);
  }
#pragma unroll
  for (int c = 3; c < 16; ++c) o[c] = __float2bfloat16_rn(0.f);
  uint4* dst = reinterpret_cast<uint4*>(v16 + g * 16);
  dst[0] = reinterpret_cast<const uint4*>(o)[0];
  dst[1] = reinterpret_cast<const uint4*>(o)[1];
}

static int gs_check_shape(const psgla_img_shape& shape) {
  PSGLA_REQUIRE(shape.B > 0 && shape.C == 3 && shape.H > 0 && shape.W > 0, "image shape must be [B>0][3][H>0][W>0]");
  PSGLA_REQUIRE(shape.H % 8 == 0 && shape.W % 8 == 0, "GSDRUNet needs H and W to be multiples of 8 (got %d x %d): the "
                "gradient through a padded input is not implemented", shape.H, shape.W);
  return PSGLA_OK;
}

// transposed channels, flipped taps: wt[i][o][8 - t] = w[o][i][t]  (OIHW 3x3)
static std::vector<float> gs_adjoint3x3(const float* w, int cout, int cin) {
  std::vector<float> wt((size_t)cin * cout * 9);
  for (int o = 0; o < cout; ++o)
    for (int i = 0; i < cin; ++i)
      for (int t = 0; t < 9; ++t) wt[((size_t)i * cout + o) * 9 + (8 - t)] = w[((size_t)o * cin + i) * 9 + t];
  return wt;
}

}  // namespace psgla

using namespace psgla;

extern "C" int psgla_gsdrunet_num_weights(void) { return GS_LAYERS; }

extern "C" size_t psgla_gsdrunet_packed_bytes(void) {
  const auto& plan = gs_plan();
  return plan.back().w_off + plan.back().bytes;
}

extern "C" int psgla_gsdrunet_pack_weights(const float* const* weights_host, void* packed_dev, void* stream) {
  PSGLA_REQUIRE(weights_host && packed_dev, "psgla_gsdrunet_pack_weights: null pointer");
  const auto& plan = gs_plan();
  for (int l = 0; l < GS_LAYERS; ++l) PSGLA_REQUIRE(weights_host[l] != nullptr, "GSDRUNet weight tensor %d is null", l);
  std::vector<uint8_t> host(psgla_gsdrunet_packed_bytes(), 0);
  for (int l = 0; l < 2 * GS_LAYERS; ++l) {
    const GsLayer& L = plan[l];
    const float* w = weights_host[L.src];
    uint8_t* dst = host.data() + L.w_off;
    if (l < GS_LAYERS) {
      dru_pack_layer(L.kind, w, L.cin, L.cout, dst);
      continue;
    }
    const GsLayer& F = plan[L.src];
    switch (L.kind) {
      case DRU_DOWN:  // adjoint of the transposed conv: its [cin][cout][2][2] weight read as OIHW [L.cout][L.cin]
      case DRU_UP:    // adjoint of the stride-2 conv: its OIHW [cout][cin] weight read as [L.cin][L.cout][2][2]
        dru_pack_layer(L.kind, w, L.cin, L.cout, dst);
        break;
      default: {  // 3x3: transpose and flip; the head's adjoint keeps the three image channels (the sigma channel is dropped)
        // (for the head, wt is [4][64][3][3] and the packer reads its first L.cout = 3 rows)
        const std::vector<float> wt = gs_adjoint3x3(w, F.cout, F.cin);
        dru_pack_layer(L.kind, wt.data(), L.cin, L.cout, dst);
      }
    }
  }
  PSGLA_CUDA_TRY(cudaMemcpyAsync(packed_dev, host.data(), host.size(), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  PSGLA_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));  // `host` dies at return
  return PSGLA_OK;
}

extern "C" size_t psgla_gsdrunet_workspace_bytes(psgla_img_shape s) {
  if (s.B <= 0 || s.H <= 0 || s.W <= 0) return 0;
  return gs_layout(s.B, s.H, s.W, nullptr, nullptr);
}

extern "C" int psgla_gsdrunet_denoise_post_next(const void* packed_dev, psgla_img_shape shape, const void* den_in_dev,
                                                const float* x_dev, void* workspace_dev, size_t workspace_bytes,
                                                const float* base_dev, float alpha, const psgla_post_params* post,
                                                float* x_out_dev, float* sample_dev, float* mean_dev, float* mean2_dev,
                                                const psgla_next_pre* next, void* stream) {
  PSGLA_REQUIRE(packed_dev && den_in_dev && workspace_dev && base_dev && post && x_out_dev,
                "psgla_gsdrunet_denoise_post_next: null pointer");
  PSGLA_REQUIRE(std::isfinite(alpha), "psgla_gsdrunet_denoise_post_next: alpha must be finite");
  {
    const int rcn = check_next_pre(next, shape);
    if (rcn) return rcn;
  }
  PSGLA_REQUIRE((mean_dev == nullptr) == (mean2_dev == nullptr), "mean and mean2 must be given together");
  {
    const int rcs = gs_check_shape(shape);
    if (rcs) return rcs;
  }
  const int B = shape.B, H = shape.H, W = shape.W;
  const size_t need = psgla_gsdrunet_workspace_bytes(shape);
  if (workspace_bytes < need)
    return set_error(PSGLA_E_WORKSPACE, "workspace of %zu bytes is smaller than the %zu needed", workspace_bytes, need);
  if (!x_dev) x_dev = base_dev;
  cudaStream_t st = (cudaStream_t)stream;
  const uint8_t* packed = (const uint8_t*)packed_dev;
  GsBuffers bufs;
  gs_layout(B, H, W, (uint8_t*)(((uintptr_t)workspace_dev + 1023) & ~(uintptr_t)1023), &bufs);
  int li = 0, ei = 0, rc = 0;
  const GsPost raw_post{};
  auto run = [&](const void* in, const void* res1, const void* res2, const void* gate, void* out) {
    if (!rc) rc = gs_layer(packed, li, B, H, W, in, res1, res2, gate, out, raw_post, st);
    ++li;
  };
  // a free buffer of scale s in slots 1..3 (slot 0 holds the skip feature, later the skip gradient)
  auto other = [&](int s, const uint8_t* a, const uint8_t* b) -> uint8_t* {
    for (int j = 1; j < 4; ++j)
      if (bufs.buf[s][j] != a && bufs.buf[s][j] != b) return bufs.buf[s][j];
    return nullptr;
  };
  // ---- forward: N(x)
  auto blocks = [&](int s, uint8_t* cur, const uint8_t* skip) -> uint8_t* {
    for (int blk = 0; blk < 2 && !rc; ++blk) {
      uint8_t* t = bufs.elu[ei++];
      uint8_t* nxt = other(s, cur, nullptr);
      run(cur, nullptr, nullptr, nullptr, t);
      run(t, cur, blk == 1 ? skip : nullptr, nullptr, nxt);
      cur = nxt;
    }
    return cur;
  };
  run(den_in_dev, nullptr, nullptr, nullptr, bufs.buf[0][0]);  // head: x1
  uint8_t* cur = bufs.buf[0][0];
  for (int s = 0; s < 3; ++s) {
    cur = blocks(s, cur, nullptr);
    run(cur, nullptr, nullptr, nullptr, bufs.buf[s + 1][0]);
    cur = bufs.buf[s + 1][0];
  }
  cur = blocks(3, cur, bufs.buf[3][0]);
  for (int s = 2; s >= 0; --s) {
    run(cur, nullptr, nullptr, nullptr, bufs.buf[s][1]);
    cur = blocks(s, bufs.buf[s][1], bufs.buf[s][0]);
  }
  if (!rc) {
    GsPost tail{};
    tail.x_out = bufs.n_out;
    rc = gs_layer(packed, li++, B, H, W, cur, nullptr, nullptr, nullptr, nullptr, tail, st);
  }
  if (rc) return rc;
  // ---- v = x - N, base'
  {
    const long long n = (long long)B * H * W;
    gs_cotangent_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(B, H * W, x_dev, base_dev, bufs.n_out, alpha, post->base_scale,
                                                                      post->gain, (__nv_bfloat16*)bufs.v16, bufs.base2);
    PSGLA_CUDA_TRY(cudaGetLastError());
  }
  // ---- backward: J^T v
  auto bblocks = [&](int s, uint8_t* g, const uint8_t* skip_grad) -> uint8_t* {
    for (int blk = 1; blk >= 0 && !rc; --blk) {
      const uint8_t* t = bufs.elu[--ei];
      uint8_t* tmp = other(s, g, nullptr);
      uint8_t* nxt = other(s, g, tmp);
      run(g, nullptr, nullptr, t, tmp);                              // c2^T, gated by elu'(t)
      run(tmp, g, blk == 0 ? skip_grad : nullptr, nullptr, nxt);     // c1^T + the block's residual (+ the skip's gradient)
      g = nxt;
    }
    return g;
  };
  run(bufs.v16, nullptr, nullptr, nullptr, bufs.buf[0][0]);  // tail^T: the skip gradient of scale 0
  uint8_t* g = bufs.buf[0][0];
  for (int s = 0; s < 3; ++s) {  // decoder, from the top
    g = bblocks(s, g, nullptr);
    run(g, nullptr, nullptr, nullptr, bufs.buf[s + 1][0]);  // up^T: the skip gradient of scale s + 1
    g = bufs.buf[s + 1][0];
  }
  g = bblocks(3, g, bufs.buf[3][0]);  // body; x4's gradient also takes the skip's
  for (int s = 2; s >= 0; --s) {      // encoder
    run(g, nullptr, nullptr, nullptr, bufs.buf[s][1]);  // down^T
    g = bblocks(s, bufs.buf[s][1], bufs.buf[s][0]);
  }
  if (rc) return rc;
  // head^T + fused post: X+ = base' + gain alpha J^T v
  GsPost fin{bufs.base2, 1.0f, post->gain * alpha, post->w_old, post->w_new, x_out_dev, sample_dev, mean_dev, mean2_dev, next};
  return gs_layer(packed, li, B, H, W, g, nullptr, nullptr, nullptr, nullptr, fin, st);
}

extern "C" int psgla_gsdrunet_layer(const void* packed_dev, psgla_img_shape shape, int backward, int layer, const void* in_dev,
                                    const void* res1_dev, const void* res2_dev, const void* gate_dev, void* out_dev,
                                    void* stream) {
  PSGLA_REQUIRE(backward == 0 || backward == 1, "psgla_gsdrunet_layer: backward must be 0 or 1");
  PSGLA_REQUIRE(layer >= 0 && layer < GS_LAYERS, "psgla_gsdrunet_layer: layer %d is not in 0..%d", layer, GS_LAYERS - 1);
  PSGLA_REQUIRE(packed_dev && in_dev && out_dev, "psgla_gsdrunet_layer: null pointer");
  const int rc = gs_check_shape(shape);
  if (rc) return rc;
  const int l = backward * GS_LAYERS + layer;
  const GsLayer& L = gs_plan()[l];
  PSGLA_REQUIRE((res1_dev != nullptr) == (L.nres >= 1) && (res2_dev != nullptr) == (L.nres >= 2) &&
                    (gate_dev != nullptr) == (L.act == ACT_GATE),
                "psgla_gsdrunet_layer: %s layer %d takes %d residual input(s) and %s gate, got res1 %s, res2 %s, gate %s",
                backward ? "backward" : "forward", layer, L.nres, L.act == ACT_GATE ? "a" : "no", res1_dev ? "set" : "null",
                res2_dev ? "set" : "null", gate_dev ? "set" : "null");
  GsPost raw{};
  raw.x_out = (float*)out_dev;
  return gs_layer((const uint8_t*)packed_dev, l, shape.B, shape.H, shape.W, in_dev, res1_dev, res2_dev, gate_dev, out_dev, raw,
                  (cudaStream_t)stream);
}
