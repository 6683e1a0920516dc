// Internal entry points shared by the denoiser drivers (conv_tc.cu, conv_gemm.cu, drunet.cu); not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/psgla_b200.h"

namespace psgla {

// validates a psgla_next_pre (inpainting "pre" of the next iteration, fused into the last layer's epilogue)
int check_next_pre(const psgla_next_pre* next, const psgla_img_shape& shape);

// Direction in which the next layer of a denoiser walks its work items: consecutive layers alternate, so that each starts on
// the part of its input the previous layer wrote last (still in L2).
int next_layer_direction();

// What a hidden layer's epilogue applies after the sum (the `relu` / `act` arguments below): ACT_NONE, ACT_RELU, ACT_ELU
// (gradient-step DRUNet forward), or ACT_GATE: res1 is a stored ELU output t and the conv is multiplied by elu'(t) instead of
// added to it (its backward).
enum ConvAct { ACT_NONE = 0, ACT_RELU = 1, ACT_ELU = 2, ACT_GATE = 3 };

// conv_tc.cu -- layers whose weights stay resident in shared memory
void pack_conv3x3_swizzled(const float* w, int nout_real, int cin_real, int nout_pad, int cin_pad, uint8_t* dst);
int conv64_hidden(const void* in, void* out, const uint8_t* w, const float* bias, int B, int H, int W, int act,
                  const void* res1, const void* res2, cudaStream_t st);
int conv_first16(const void* in16, void* out, const uint8_t* w, const float* bias, int B, int H, int W, int relu,
                 cudaStream_t st);
// the last layer (64 -> C = 3 or 1 image channels) and the fused post
int conv_last_post(const void* in, const uint8_t* w, const float* bias, int B, int C, int H, int W, const float* base,
                   float base_scale, float gain, float w_old, float w_new, float* x_out, float* sample, float* mean,
                   float* mean2, const psgla_next_pre* next, cudaStream_t st);

// drunet.cu -- the U-Net layer kinds (which kernel runs a layer) and their packed weights, shared with gsdrunet.cu
enum DruKind { DRU_HEAD, DRU_C64, DRU_GEMM3, DRU_DOWN, DRU_UP, DRU_TAIL };
size_t dru_layer_bytes(DruKind k, int cin, int cout);
// fp32 torch-layout weight -> the kind's packed layout: HEAD / C64 / TAIL OIHW 3x3 (HEAD: cin <= 16 real input channels; cin = 2
// is the grayscale DRUNet head (image, noise level), whose noise level goes to K slot 3 as the colour head's does; TAIL: cout <= 16 real outputs), GEMM3
// / DOWN OIHW, UP ConvTranspose2d [cin][cout][2][2].  dst zero-initialised.
void dru_pack_layer(DruKind kind, const float* w, int cin, int cout, uint8_t* dst);

// conv_gemm.cu -- layers with streamed weights (mode: 0 conv3x3, 1 2x2 stride-2 down, 2 2x2 transposed up)
int conv_gemm_layer(int mode, int B, int Hin, int Win, int Cin, int Cout, const void* w, const void* in, const void* res1,
                    const void* res2, void* out, int act, cudaStream_t st);

}  // namespace psgla
