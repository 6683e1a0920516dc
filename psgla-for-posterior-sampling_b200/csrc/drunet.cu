// DRUNet denoiser (deepinv.models.DRUNet as constructed at sampling_images.py:136 and called at
// restoration_algorithms.py:238 / sampling_images.py:156): KAIR UNetRes with nc = [64, 128, 256, 512], nb = 4 residual
// blocks per stage, stride-2 2x2 convs down, 2x2 transposed convs up, no biases, ReLU; the input is the image plus a
// constant noise-level channel and the output is the denoised image (architecture restated in oracle/image_oracle.py).
//
// Colour (C = 3) or grayscale (C = 1) images: the head takes C + 1 channels, the tail gives C.
//
// Layer schedule (68 launches): head 4->64 (first-layer SS kernel on the NHWC16 input, channel 3 = sigma), the 16
// full-resolution 64-channel convs on the weight-resident TS kernel (conv_tc.cu), every other layer on the streamed
// implicit-GEMM kernel (conv_gemm.cu); residual and U-Net skip additions are folded into the epilogue of the conv that
// produces the sum; the 64->3 tail runs the fused Langevin "post" epilogue.
#include <cstring>
#include <vector>

#include "common.cuh"
#include "conv_api.cuh"

namespace psgla {

struct DruLayer {
  DruKind kind;
  int cin, cout;
  int scale;  // the layer's input is (H >> scale) x (W >> scale)
  int relu;   // ReLU after the sum
  int nres;   // residual inputs added before the ReLU: 1 = the block input (second conv of a residual block), 2 = and the U-Net skip
  size_t w_off, bytes;
};

size_t dru_layer_bytes(DruKind k, int cin, int cout) {
  size_t b = 0;
  switch (k) {
    case DRU_HEAD: b = (size_t)9 * 64 * 16 * 2 + 64 * 4; break;   // swizzled weights + (zero) bias
    case DRU_C64: b = (size_t)9 * 64 * 64 * 2 + 64 * 4; break;
    case DRU_TAIL: b = (size_t)9 * 16 * 64 * 2 + 16 * 4; break;
    case DRU_GEMM3: b = (size_t)9 * cout * cin * 2; break;
    case DRU_DOWN:
    case DRU_UP: b = (size_t)4 * cout * cin * 2; break;
  }
  return (b + 1023) / 1024 * 1024;
}

// The 64 weight tensors in state-dict order: m_head, m_down1.{0..3}.res.{0,2}, m_down1.4, m_down2..., m_down3...,
// m_body.{0..3}.res.{0,2}, m_up3.0, m_up3.{1..4}.res.{0,2}, m_up2..., m_up1..., m_tail.
static const std::vector<DruLayer>& dru_plan() {
  static std::vector<DruLayer> plan;
  if (!plan.empty()) return plan;
  std::vector<DruLayer> v;
  size_t off = 0;
  auto add = [&](DruKind k, int cin, int cout, int scale, int relu, int nres) {
    const size_t b = dru_layer_bytes(k, cin, cout);
    v.push_back({k, cin, cout, scale, relu, nres, off, b});
    off += b;
  };
  const int nc[4] = {64, 128, 256, 512};
  // four residual blocks x -> x + conv(relu(conv(x))); with `skip`, the last one also adds the U-Net skip connection
  auto blocks = [&](int s, bool skip) {
    for (int i = 0; i < 8; ++i)
      add(s == 0 ? DRU_C64 : DRU_GEMM3, nc[s], nc[s], s, i % 2 == 0, i % 2 == 0 ? 0 : (skip && i == 7 ? 2 : 1));
  };
  add(DRU_HEAD, 4, 64, 0, 0, 0);
  for (int s = 0; s < 3; ++s) {  // encoder
    blocks(s, false);
    add(DRU_DOWN, nc[s], nc[s + 1], s, 0, 0);
  }
  blocks(3, true);  // body, + x4
  for (int s = 2; s >= 0; --s) {  // decoder, + x3 / x2 / x1
    add(DRU_UP, nc[s + 1], nc[s], s + 1, 0, 0);
    blocks(s, true);
  }
  add(DRU_TAIL, 64, 3, 0, 0, 0);  // (colour; psgla_drunet_pack_weights_ch packs head and tail for the channel count)
  plan.swap(v);
  return plan;
}

static inline uint16_t dru_bf16(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

void dru_pack_layer(DruKind kind, const float* w, int cin, int cout, uint8_t* dst) {
  switch (kind) {
    case DRU_HEAD: {
      // The NHWC16 denoiser input holds the image from slot 0 and the noise level in slot 3 whatever the channel count, so a
      // grayscale head [64][2] (image, sigma) is packed as the colour head [64][4] with input channels 1 and 2 zero.  Every
      // other cin is packed as it stands (colour: 4; the gradient-step DRUNet's adjoint of the tail: 3).
      if (cin != 2) {
        pack_conv3x3_swizzled(w, 64, cin, 64, 16, dst);
        break;
      }
      std::vector<float> w4((size_t)64 * 4 * 9, 0.f);
      for (int n = 0; n < 64; ++n)
        for (int t = 0; t < 9; ++t) {
          w4[((size_t)n * 4 + 0) * 9 + t] = w[((size_t)n * 2 + 0) * 9 + t];
          w4[((size_t)n * 4 + 3) * 9 + t] = w[((size_t)n * 2 + 1) * 9 + t];
        }
      pack_conv3x3_swizzled(w4.data(), 64, 4, 64, 16, dst);
      break;
    }
    case DRU_C64: pack_conv3x3_swizzled(w, 64, 64, 64, 64, dst); break;
    case DRU_TAIL: pack_conv3x3_swizzled(w, cout, 64, 16, 64, dst); break;
    case DRU_GEMM3:  // OIHW [cout][cin][3][3] -> [tap][cout][cin]
    case DRU_DOWN: {  // OIHW [cout][cin][2][2] -> [tap][cout][cin]
      const int taps = kind == DRU_GEMM3 ? 9 : 4;
      uint16_t* d = reinterpret_cast<uint16_t*>(dst);
      for (int n = 0; n < cout; ++n)
        for (int k = 0; k < cin; ++k)
          for (int t = 0; t < taps; ++t)
            d[((size_t)t * cout + n) * cin + k] = dru_bf16(w[((size_t)n * cin + k) * taps + t]);
      break;
    }
    case DRU_UP: {  // ConvTranspose2d weight [cin][cout][2][2] -> [quadrant][cout][cin]
      uint16_t* d = reinterpret_cast<uint16_t*>(dst);
      for (int k = 0; k < cin; ++k)
        for (int n = 0; n < cout; ++n)
          for (int t = 0; t < 4; ++t)
            d[((size_t)t * cout + n) * cin + k] = dru_bf16(w[((size_t)k * cout + n) * 4 + t]);
      break;
    }
  }
}

struct DruBuffers {
  uint8_t* buf[4][4];  // [scale][P, A, B, C]
};
static size_t dru_scale_bytes(int B, int H, int W, int s) {
  const size_t n = (size_t)B * (H >> s) * (W >> s) * (64 << s) * 2;
  return (n + 1023) / 1024 * 1024;
}
static size_t dru_workspace_bytes(int B, int H, int W) {
  size_t t = 0;
  for (int s = 0; s < 4; ++s) t += 4 * dru_scale_bytes(B, H, W, s);
  return t + 1024;
}

// What the tail does with its conv output: the fused Langevin post (the network) or nothing (base == NULL: x_out = the raw
// fp32 NCHW conv, psgla_drunet_layer).
struct DruPost {
  const float* base;
  float base_scale, gain, w_old, w_new;
  float* x_out;
  float* sample;
  float* mean;
  float* mean2;
  const psgla_next_pre* next;
};

// Layer l of the plan as the network runs it: the kernel its kind selects, its ReLU, and its residual inputs (res1 = the block
// input, res2 = the U-Net skip; null where the plan has none).  in / out / res are bf16 NHWC except the head's input (NHWC16)
// and the tail's output, which goes through `post`.
static int dru_layer(const uint8_t* packed, int l, int B, int C, int H, int W, const void* in, const void* res1, const void* res2,
                     void* out, const DruPost& post, cudaStream_t st) {
  const DruLayer& L = dru_plan()[l];
  const uint8_t* w = packed + L.w_off;
  const int h = H >> L.scale, wd = W >> L.scale;
  auto bias = [&](int nout_pad, int cin_pad) { return reinterpret_cast<const float*>(w + (size_t)9 * nout_pad * cin_pad * 2); };
  switch (L.kind) {
    case DRU_HEAD: return conv_first16(in, out, w, bias(64, 16), B, H, W, L.relu, st);
    case DRU_C64: return conv64_hidden(in, out, w, bias(64, 64), B, h, wd, L.relu, res1, res2, st);
    case DRU_GEMM3: return conv_gemm_layer(0, B, h, wd, L.cin, L.cout, w, in, res1, res2, out, L.relu, st);
    case DRU_DOWN: return conv_gemm_layer(1, B, h, wd, L.cin, L.cout, w, in, res1, res2, out, L.relu, st);
    case DRU_UP: return conv_gemm_layer(2, B, h, wd, L.cin, L.cout, w, in, res1, res2, out, L.relu, st);
    case DRU_TAIL:
      return conv_last_post(in, w, bias(16, 64), B, C, H, W, post.base, post.base_scale, post.gain, post.w_old, post.w_new,
                            post.x_out, post.sample, post.mean, post.mean2, post.next, st);
  }
  return set_error(PSGLA_E_BADARG, "DRUNet layer %d: unknown kind", l);
}

static int dru_check_shape(const psgla_img_shape& shape) {
  PSGLA_REQUIRE(shape.B > 0 && (shape.C == 3 || shape.C == 1) && shape.H > 0 && shape.W > 0,
                "image shape must be [B>0][C = 1 or 3][H>0][W>0]");
  PSGLA_REQUIRE(shape.H % 8 == 0 && shape.W % 8 == 0, "DRUNet needs H and W to be multiples of 8 (got %d x %d): crop or pad "
                "the image (the reference's deepinv pads internally by an unverifiable rule)", shape.H, shape.W);
  return PSGLA_OK;
}

}  // namespace psgla

using namespace psgla;

extern "C" int psgla_drunet_num_weights(void) { return (int)dru_plan().size(); }

extern "C" size_t psgla_drunet_packed_bytes(void) {
  const auto& plan = dru_plan();
  return plan.back().w_off + plan.back().bytes;
}

extern "C" int psgla_drunet_pack_weights(const float* const* weights_host, void* packed_dev, void* stream) {
  return psgla_drunet_pack_weights_ch(3, weights_host, packed_dev, stream);
}

extern "C" int psgla_drunet_pack_weights_ch(int channels, const float* const* weights_host, void* packed_dev, void* stream) {
  PSGLA_REQUIRE(weights_host && packed_dev, "psgla_drunet_pack_weights: null pointer");
  PSGLA_REQUIRE(channels == 3 || channels == 1, "psgla_drunet_pack_weights_ch: channels must be 3 or 1 (got %d)", channels);
  const auto& plan = dru_plan();
  std::vector<uint8_t> host(psgla_drunet_packed_bytes(), 0);
  for (size_t l = 0; l < plan.size(); ++l) {
    const DruLayer& L = plan[l];
    const float* w = weights_host[l];
    PSGLA_REQUIRE(w != nullptr, "DRUNet weight tensor %zu is null", l);
    const int cin = L.kind == DRU_HEAD ? channels + 1 : L.cin, cout = L.kind == DRU_TAIL ? channels : L.cout;
    dru_pack_layer(L.kind, w, cin, cout, host.data() + L.w_off);
  }
  PSGLA_CUDA_TRY(cudaMemcpyAsync(packed_dev, host.data(), host.size(), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  PSGLA_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));  // `host` dies at return
  return PSGLA_OK;
}

extern "C" size_t psgla_drunet_workspace_bytes(psgla_img_shape s) { return dru_workspace_bytes(s.B, s.H, s.W); }

extern "C" int psgla_drunet_denoise_post(const void* packed_dev, psgla_img_shape shape, const void* den_in_dev,
                                         void* workspace_dev, size_t workspace_bytes, const float* base_dev,
                                         const psgla_post_params* post, float* x_out_dev, float* sample_dev,
                                         float* mean_dev, float* mean2_dev, void* stream) {
  return psgla_drunet_denoise_post_next(packed_dev, shape, den_in_dev, workspace_dev, workspace_bytes, base_dev, post, x_out_dev,
                                        sample_dev, mean_dev, mean2_dev, nullptr, stream);
}

extern "C" int psgla_drunet_denoise_post_next(const void* packed_dev, psgla_img_shape shape, const void* den_in_dev,
                                              void* workspace_dev, size_t workspace_bytes, const float* base_dev,
                                              const psgla_post_params* post, float* x_out_dev, float* sample_dev,
                                              float* mean_dev, float* mean2_dev, const psgla_next_pre* next, void* stream) {
  PSGLA_REQUIRE(packed_dev && den_in_dev && workspace_dev && post && x_out_dev, "psgla_drunet_denoise_post: null pointer");
  {
    const int rcn = check_next_pre(next, shape);
    if (rcn) return rcn;
  }
  PSGLA_REQUIRE((mean_dev == nullptr) == (mean2_dev == nullptr), "mean and mean2 must be given together");
  {
    const int rcs = dru_check_shape(shape);
    if (rcs) return rcs;
  }
  const int B = shape.B, H = shape.H, W = shape.W;
  if (workspace_bytes < dru_workspace_bytes(B, H, W))
    return set_error(PSGLA_E_WORKSPACE, "workspace of %zu bytes is smaller than the %zu needed", workspace_bytes,
                     dru_workspace_bytes(B, H, W));
  cudaStream_t st = (cudaStream_t)stream;
  const uint8_t* packed = (const uint8_t*)packed_dev;
  DruBuffers bufs;
  {
    uint8_t* pp = (uint8_t*)(((uintptr_t)workspace_dev + 1023) & ~(uintptr_t)1023);
    for (int s = 0; s < 4; ++s)
      for (int j = 0; j < 4; ++j) {
        bufs.buf[s][j] = pp;
        pp += dru_scale_bytes(B, H, W, s);
      }
  }
  int li = 0;
  int rc = 0;
  const DruPost no_post{};
  auto run = [&](const void* in, const void* res1, const void* res2, void* out) {
    if (!rc) rc = dru_layer(packed, li, B, shape.C, H, W, in, res1, res2, out, no_post, st);
    ++li;
  };
  // four residual blocks at scale s starting from `cur`; the last block also adds `skip` (U-Net skip connection)
  auto resblocks = [&](int s, uint8_t* cur, const uint8_t* skip) -> uint8_t* {
    for (int blk = 0; blk < 4 && !rc; ++blk) {
      uint8_t* scratch[2];
      int n = 0;
      for (int j = 1; j < 4 && n < 2; ++j)
        if (bufs.buf[s][j] != cur) scratch[n++] = bufs.buf[s][j];
      uint8_t* tmp = scratch[0];
      uint8_t* nxt = scratch[1];
      run(cur, nullptr, nullptr, tmp);
      run(tmp, cur, blk == 3 ? skip : nullptr, nxt);
      cur = nxt;
    }
    return cur;
  };

  run(den_in_dev, nullptr, nullptr, bufs.buf[0][0]);  // head: x1
  uint8_t* cur = bufs.buf[0][0];
  for (int s = 0; s < 3; ++s) {  // encoder
    cur = resblocks(s, cur, nullptr);
    run(cur, nullptr, nullptr, bufs.buf[s + 1][0]);
    cur = bufs.buf[s + 1][0];
  }
  cur = resblocks(3, cur, bufs.buf[3][0]);  // body, + x4
  for (int s = 2; s >= 0; --s) {  // decoder
    run(cur, nullptr, nullptr, bufs.buf[s][1]);
    cur = resblocks(s, bufs.buf[s][1], bufs.buf[s][0]);  // + x3 / x2 / x1
  }
  if (rc) return rc;
  // tail + fused Langevin post:  X+ = base_scale * base + gain * D
  const DruPost tail{base_dev,  post->base_scale, post->gain, post->w_old, post->w_new,
                     x_out_dev, sample_dev,       mean_dev,   mean2_dev,   next};
  return dru_layer(packed, li, B, shape.C, H, W, cur, nullptr, nullptr, nullptr, tail, st);
}

extern "C" int psgla_drunet_layer(const void* packed_dev, psgla_img_shape shape, int layer, const void* in_dev,
                                  const void* res1_dev, const void* res2_dev, void* out_dev, void* stream) {
  const auto& plan = dru_plan();
  PSGLA_REQUIRE(layer >= 0 && layer < (int)plan.size(), "psgla_drunet_layer: layer %d is not in 0..%d", layer,
                (int)plan.size() - 1);
  PSGLA_REQUIRE(packed_dev && in_dev && out_dev, "psgla_drunet_layer: null pointer");
  const int rc = dru_check_shape(shape);
  if (rc) return rc;
  const DruLayer& L = plan[layer];
  PSGLA_REQUIRE((res1_dev != nullptr) == (L.nres >= 1) && (res2_dev != nullptr) == (L.nres >= 2),
                "psgla_drunet_layer: layer %d takes %d residual input(s) (res1 = block input, res2 = U-Net skip), got res1 %s, "
                "res2 %s", layer, L.nres, res1_dev ? "set" : "null", res2_dev ? "set" : "null");
  DruPost raw{};
  raw.x_out = (float*)out_dev;
  return dru_layer((const uint8_t*)packed_dev, layer, shape.B, shape.C, shape.H, shape.W, in_dev, res1_dev, res2_dev, out_dev, raw,
                   (cudaStream_t)stream);
}
