/*
 * psgla_b200.h -- C ABI of the B200-native PSGLA / PnP-ULA hot path (libpsgla_b200.so).
 *
 * The reference (Marien-RENAUD/PSGLA-for-posterior-sampling) has no FFI layer: its boundary is the
 * Python call signatures of the samplers plus four opaque callables (SURVEY.md section 8b).  Each entry point below
 * names the reference lines whose arithmetic it replaces.  Python binds these with ctypes
 * (psgla-for-posterior-sampling_b200/_lib.py); INTEGRATION.md shows the stub a maintainer of the reference adds.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  "dev" pointers are CUDA device pointers owned by the caller
 *     (torch allocates inputs, outputs and workspace); the library never frees caller memory.
 *   - every call is stream-ordered on `stream` (a cudaStream_t passed as void*), asynchronous, re-entrant.
 *   - return value: 0 = ok; >0 = cudaError_t; <0 = PSGLA_E_* below.  psgla_last_error() gives a thread-local message.
 *   - image tensors are fp32 NCHW [B][C][H][W] ("chains" = B; C = 3 colour, or 1 grayscale where an entry says so);
 *     denoiser activations are bf16 NHWC, library-internal.
 *   - noise: in-kernel Philox4x32-10 keyed by (seed; subsequence = global chain id; counter = step / element), or,
 *     when a replay pointer is given, the caller's N(0,1) draws (the reference's np.random.randn / torch.randn).
 */
#ifndef PSGLA_B200_H
#define PSGLA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define PSGLA_ABI_VERSION 5

enum {
  PSGLA_OK = 0,
  PSGLA_E_BADARG = -1,      /* null pointer, size out of range, unsupported option */
  PSGLA_E_UNSUPPORTED = -2, /* valid request this build cannot serve (e.g. r > PSGLA_GMM_MAX_COMPONENTS) */
  PSGLA_E_NODEVICE = -3,    /* no sm_100 device / driver entry point missing */
  PSGLA_E_WORKSPACE = -4    /* workspace too small */
};

const char* psgla_last_error(void);
int psgla_abi_version(void);
/* sizeof() of the structs below as the library was compiled (0: psgla_gmm2d_problem, 1: psgla_img_shape, 2: psgla_pre_params,
 * 3: psgla_post_params, 4: psgla_next_pre, 5: psgla_tv_params; -1 otherwise) -- lets a binding verify its struct layout. */
int psgla_struct_size(int which);
/* Philox4x32-10 (Salmon et al., SC'11) block function as the kernels use it: counter[4], key[2] -> out[4].  Host code,
 * no GPU needed; the tests pin it to the Random123 known-answer vectors. */
void psgla_philox4x32_10(const uint32_t* counter, const uint32_t* key, uint32_t* out);
/* compute capability of the current device as major*10+minor (100 on B200); <0 on error. */
int psgla_device_arch(void);

/* ------------------------------------------------------------------------------------------------------------
 * 2D Gaussian-mixture posterior sampling: replaces the Python loops of sampling_2D.py:21-45 (PnP_ULA) and
 * sampling_2D.py:48-72 (SnoPnP_ULA = PSGLA) together with the closed-form MMSE denoiser utils_2D.py:209-233 and the
 * data-fidelity score sampling_2D.py:30-31.  One thread owns one chain for all n_steps; nothing but the final state
 * (and optional thinned trajectory) touches HBM.
 * ---------------------------------------------------------------------------------------------------------- */
#define PSGLA_GMM_MAX_COMPONENTS 16
#define PSGLA_ALG_PSGLA 0   /* x+ = D(x + (delta/alpha) score(x) + sqrt(2 delta) z, delta)            sampling_2D.py:63 */
#define PSGLA_ALG_PNPULA 1  /* x+ = x + delta score(x) + alpha delta/eps (D(x,eps)-x) + sqrt(2 delta) z  sampling_2D.py:36 */

typedef struct psgla_gmm2d_problem {
  int32_t alg;          /* PSGLA_ALG_* */
  int32_t n_components; /* r, 1..PSGLA_GMM_MAX_COMPONENTS */
  double delta;         /* step size */
  double alpha;         /* regularisation / relaxation parameter */
  double epsilon;       /* denoiser level for PnP-ULA (PSGLA uses delta, sampling_2D.py:63) */
  double sigma;         /* score = A^T (y - A x) / sigma^2                      sampling_2D.py:31 */
  double A[4];          /* row-major 2x2 */
  double y[2];
  double mu[PSGLA_GMM_MAX_COMPONENTS][2];
  double Sigma[PSGLA_GMM_MAX_COMPONENTS][4]; /* row-major 2x2, SPD */
  double pi[PSGLA_GMM_MAX_COMPONENTS];
} psgla_gmm2d_problem;

/* Runs n_steps Langevin steps on n_chains chains.
 *   precision   0: fp32 state and arithmetic (throughput path); 1: fp64 (parity path vs the float64 reference).
 *   x_dev       [n_chains][2] of float/double: in = current state (x_0), out = state after n_steps.
 *   chain_id0   global id of x_dev[0] (Philox subsequence), so results do not depend on how chains are sharded.
 *   step0       global index of the first step (Philox counter), so a run may be split into segments.
 *   noise_dev   NULL (Philox) or [n_steps][n_chains][2] standard normals of the same precision (replay).
 *   traj_dev    NULL or [n_steps/thin][n_chains][2]: state after every global step t with (t+1) % thin == 0.
 */
int psgla_gmm2d_run(const psgla_gmm2d_problem* problem, int precision, void* x_dev, int64_t n_chains,
                    int64_t chain_id0, int64_t n_steps, int64_t step0, uint64_t seed, const void* noise_dev,
                    void* traj_dev, int64_t thin, void* stream);

/* How many kernel launches the most recent psgla_gmm2d_run issued (the population is cut into occupancy-sized waves:
 * full waves of 4 chains per thread plus one remainder wave).  Bookkeeping for benchmarks. */
int psgla_gmm2d_last_launches(void);

/* The denoiser alone on n points (utils_2D.py:219-232, log-sum-exp form): out = D(x, epsilon). */
int psgla_gmm2d_denoise(const psgla_gmm2d_problem* problem, double epsilon, int precision, const void* x_dev,
                        void* out_dev, int64_t n, void* stream);

/* Standard normals from the library's Philox stream, exactly the draws psgla_gmm2d_run consumes for
 * (chain_id0.., step0..): out_dev [n_steps][n_chains][2] fp32.  Test / replay aid. */
int psgla_gmm2d_noise(float* out_dev, int64_t n_chains, int64_t chain_id0, int64_t n_steps, int64_t step0,
                      uint64_t seed, void* stream);

/* Sliced Wasserstein-2 distance between a chain population and a reference sample of the same size, on the device
 * (sampling_2D.py:168-170 `ot.sliced.sliced_wasserstein_distance`, and the "metric every k steps" of :38-39,65-66 for a
 * population resident in HBM): sqrt( mean_p mean_i (sort_i(theta_p . x_i) - sort_i(theta_p . ref_i))^2 ).
 *   theta_host        [n_proj][2] unit directions (host floats), n_proj <= 128
 *   ws_dev / ws_bytes caller-owned scratch of psgla_gmm2d_sw2_workspace_bytes(n, n_proj) bytes, 256-byte aligned
 * psgla_gmm2d_sorted_projections writes the sorted projections [n_proj][n] fp32 (done once for the reference sample);
 * psgla_gmm2d_sliced_w2 projects + sorts x_dev and writes the distance to *out_dev (a device double; no host sync). */
size_t psgla_gmm2d_sw2_workspace_bytes(int64_t n, int n_proj);
int psgla_gmm2d_sorted_projections(const void* x_dev, int precision, int64_t n, const float* theta_host, int n_proj,
                                   float* out_sorted_dev, void* ws_dev, size_t ws_bytes, void* stream);
int psgla_gmm2d_sliced_w2(const void* x_dev, int precision, int64_t n, const float* theta_host, int n_proj,
                          const float* ref_sorted_dev, void* ws_dev, size_t ws_bytes, double* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Image inverse problems.  One "iteration" of psgla (restoration_algorithms.py:232-238) or pnpula (:104-115) on a
 * batch of B independent chains of shape [C][H][W] is
 *     pre   : data-fidelity gradient (+ projection term for PnP-ULA) + noise  -> base (fp32) and the denoiser input
 *     dncnn : 20 conv3x3 layers (tcgen05 implicit GEMM, bf16 in / fp32 accumulate)
 *     post  : fused into the last conv's epilogue: X+ = base + gain * (out_conv(h) + bias), thinning, E[X], E[X^2]
 * ---------------------------------------------------------------------------------------------------------- */

typedef struct psgla_img_shape {
  int32_t B, C, H, W; /* chains, channels, rows, cols */
} psgla_img_shape;
/* Channels: the pre kernels, psgla_img_blur, psgla_img_noise, psgla_img_to_nhwc16, psgla_img_pad_replicate_nhwc16,
 * psgla_img_psnr_ssim, psgla_dncnn_*, psgla_conv3x3_layer and psgla_drunet_* take C = 3 (colour) or C = 1 (grayscale); the
 * TV prox and the gradient-step DRUNet take C = 3 only.  Any other C is rejected before any CUDA call.  The element index
 * within a chain is c H W + pixel for both, so channel 0 of a colour chain and a grayscale chain draw the same Philox noise. */

/* Inpainting "pre" (sampling_images.py:295 data_grad; restoration_algorithms.py:236 / :110-115):
 *   PSGLA  : base = X + gain_data * (-mask (X - y)) + noise_scale * Z        (gain_data = (delta/lambd)/sigma^2)
 *            den_in = bf16(base)
 *   PnP-ULA: base = X + delta * (-(X - clamp(X,cmin,cmax))/lambd) + gain_data * (-mask (X - y)) + noise_scale * Z
 *            den_in = bf16(X)                                              (gain_data = delta/sigma^2)
 * mask_dev, y_dev: [1 or B][C][H][W] fp32 (mask_B / y_B say which; 1 = shared by all chains).
 * noise_dev: NULL (Philox: subsequence = chain_id0 + b, counter = (iteration, element)) or [B][C][H][W] fp32.
 * den_in_dev: bf16 NHWC [B][H][W][16] -- the padded input of the first conv layer: the C image channels from slot 0, slot 3 =
 * den_in_c3, every other slot zero (grayscale: (v, 0, 0, den_in_c3, 0, ...)). */
typedef struct psgla_pre_params {
  int32_t alg;        /* PSGLA_ALG_* */
  float gain_data;    /* multiplies -mask (X - y) resp. -A^T(A X - y) */
  float noise_scale;  /* sqrt(2) s  resp.  sqrt(2 delta) */
  float proj_gain;    /* PnP-ULA: delta / lambd; PSGLA: 0 */
  float c_min, c_max; /* PnP-ULA projection box, restoration_algorithms.py:38 defaults -1, 2 */
  float x_gain;       /* base += x_gain * X: PnP-ULA with a non-residual denoiser (DRUNet) needs -delta*alpha/s2 here
                         because alpha (D(X) - X)/s2 is no longer a pure function of the network output; else 0 */
  float den_in_c3;    /* value written to channel 3 of den_in: the DRUNet noise-level map (sigma); 0 for DnCNN */
  uint64_t seed;
  int64_t chain_id0;
  int64_t iteration;
  /* Which N(0,1) stream the kernel generates when noise_dev is NULL:
   *   PSGLA_NOISE_PHILOX     the library's own (subsequence = chain_id0 + b, counter = (iteration, element / 4));
   *   PSGLA_NOISE_TORCH_CUDA the stream of torch.randn((B,C,H,W), generator=Generator("cuda").manual_seed(seed)) -- what
   *                          the reference draws each iteration (restoration_algorithms.py:104,232) -- bit for bit:
   *                          torch_offset = the generator's Philox offset before that call and torch_threads = the
   *                          thread count of torch's launch, both from psgla_torch_cuda_randn_policy(). */
  int32_t noise_mode;
  uint32_t torch_threads;
  uint64_t torch_offset;
} psgla_pre_params;

enum { PSGLA_NOISE_PHILOX = 0, PSGLA_NOISE_TORCH_CUDA = 1 };

/* Launch policy of torch's CUDA randn for a float tensor of numel elements (ATen DistributionTemplates.h
 * calc_execution_policy, block 256, unroll 4) on a device with sm_count SMs and max_threads_per_sm resident threads:
 * *threads = 256 * grid, *offset_step = how far one call advances the generator's Philox offset.  Iteration i of a sampler
 * that draws once per iteration therefore uses torch_offset = i * offset_step.  Host code, no GPU needed;
 * sm_count <= 0 asks the current device. */
int psgla_torch_cuda_randn_policy(int64_t numel, int sm_count, int max_threads_per_sm, uint32_t* threads,
                                  uint64_t* offset_step);
/* out_dev[0..numel) = that torch.randn call's values (seed, offset as above).  Test / replay aid. */
int psgla_img_noise_torch_cuda(int64_t numel, uint64_t seed, uint64_t offset, uint32_t threads, float* out_dev,
                               void* stream);

int psgla_img_pre_inpaint(const psgla_pre_params* p, psgla_img_shape shape, const float* x_dev, const float* mask_dev,
                          int mask_B, const float* y_dev, int y_B, const float* noise_dev, float* base_dev,
                          void* den_in_dev, void* stream);

/* Deblurring "pre" (sampling_images.py:329-338): data_grad = -A^T(A x - y)/sigma^2 with A = AT = separable circular
 * blur with taps h1d[2l+1] (float, host pointer; symmetric by construction, sampling_images.py:306-314).
 * The blur is a shared-memory staged stencil: tile + 2l halo, wrap-around indexing. */
int psgla_img_pre_deblur(const psgla_pre_params* p, psgla_img_shape shape, const float* x_dev, const float* h1d_host,
                         int l, const float* y_dev, int y_B, const float* noise_dev, float* base_dev,
                         void* den_in_dev, void* stream);
/* The same step in its A^T A form: A^T(A x - y) = (A^T A) x - A^T y.  A^T A is the separable circular (4l+1)-tap stencil with
 * taps h * h, and aty_dev = A^T y = psgla_img_blur(y) is computed ONCE per run by the caller ([1 or B][C][H][W] fp32): one
 * horizontal and one vertical pass over x per iteration, done as a row-streaming filter (vertical window in registers).  Same
 * results as psgla_img_pre_deblur up to fp32 rounding (2e-5 relative in the tests).  Half-widths l = 1..4. */
int psgla_img_pre_deblur_ata(const psgla_pre_params* p, psgla_img_shape shape, const float* x_dev, const float* h1d_host,
                             int l, const float* aty_dev, int aty_B, const float* noise_dev, float* base_dev,
                             void* den_in_dev, void* stream);
/* y = A x alone (builds the observation, sampling_images.py:335). */
int psgla_img_blur(psgla_img_shape shape, const float* x_dev, const float* h1d_host, int l, float* out_dev,
                   void* stream);

/* Fills out_dev [B][C][H][W] with the N(0,1) draws the "pre" kernels consume for (seed, chain_id0, iteration). */
int psgla_img_noise(psgla_img_shape shape, uint64_t seed, int64_t chain_id0, int64_t iteration, float* out_dev,
                    void* stream);

/* DnCNN (deepinv.models.DnCNN as constructed at sampling_images.py:130; called restoration_algorithms.py:238 and
 * sampling_images.py:156): depth conv3x3 layers, nf = 64 features, bias, ReLU, residual.
 * psgla_dncnn_pack_weights converts the fp32 OIHW state-dict tensors (host pointers, in layer order:
 * in_conv, conv_list[0..depth-3], out_conv) into the library's device layout (bf16, tap-major, K-major, 128B-swizzled
 * as the tcgen05 B operand wants it) inside packed_dev (psgla_dncnn_packed_bytes(depth) bytes).
 * psgla_dncnn_pack_weights_ch packs a network of `channels` = 3 or 1 image channels (in_conv [64][channels][3][3], out_conv
 * [channels][64][3][3]); psgla_dncnn_pack_weights is it with 3.  The packed size does not depend on the channel count, but a
 * packed buffer must be used with shapes of the channel count it was packed for. */
size_t psgla_dncnn_packed_bytes(int depth);
int psgla_dncnn_pack_weights(int depth, const float* const* weights_host, const float* const* biases_host,
                             void* packed_dev, void* stream);
int psgla_dncnn_pack_weights_ch(int depth, int channels, const float* const* weights_host, const float* const* biases_host,
                                void* packed_dev, void* stream);
/* Bytes of activation workspace for B chains of H x W (two ping-pong bf16 NHWC [B][H][W][64] buffers). */
size_t psgla_dncnn_workspace_bytes(psgla_img_shape shape);

/* "post" parameters, applied in the last layer's epilogue:
 *   X+ = base + gain * (out_conv(h) + bias)      PSGLA: gain = alpha (restoration_algorithms.py:238, D(Y) - Y = residual)
 *                                                PnP-ULA: gain = delta * alpha / s2 (sampling_images.py:157, :115)
 *   if sample_dev: sample = X+                   thinning, restoration_algorithms.py:118-121 / :241-244
 *   if mean_dev  : mean = w_old * mean + w_new * X+ ; mean2 = w_old * mean2 + w_new * X+^2   (:128-135 / :255-262,
 *                  three rounded fp32 operations each, like the reference's eager ops) */
typedef struct psgla_post_params {
  float gain;
  float base_scale;   /* DRUNet path only: X+ = base_scale * base + gain * D(den_in)  (PSGLA: 1 - alpha, alpha);
                         the DnCNN path is residual (X+ = base + gain * R) and ignores it */
  float w_old, w_new; /* iter_mmse/(iter_mmse+1), 1/(iter_mmse+1) as float */
} psgla_post_params;

/* One full denoiser application + post:  x_out = post(base, DnCNN residual of den_in).
 * den_in_dev as written by a "pre" call; x_out_dev may alias the X the pre call read. */
int psgla_dncnn_residual_post(int depth, const void* packed_dev, psgla_img_shape shape, const void* den_in_dev,
                              void* workspace_dev, size_t workspace_bytes, const float* base_dev,
                              const psgla_post_params* post, float* x_out_dev, float* sample_dev, float* mean_dev,
                              float* mean2_dev, void* stream);

/* The same with the NEXT iteration's inpainting "pre" fused into the epilogue: the thread that has just produced X+ for a
 * pixel also evaluates psgla_img_pre_inpaint's arithmetic on it (same noise element, bit-identical results) and writes the
 * next base and denoiser input, so that a sampler iteration is the conv launches alone.  next == NULL: plain post.
 * base_dev / den_in_dev of `next` may be this call's base_dev / den_in_dev (in place: every element is read before it is
 * rewritten by the same thread, and den_in was consumed by the first layer). */
typedef struct psgla_next_pre {
  const psgla_pre_params* pre; /* parameters of iteration i + 1 (its `iteration`, torch_offset, ...) */
  const float* mask_dev;       /* [1 or B][C][H][W] */
  const float* y_dev;
  int32_t mask_B, y_B;
  float* base_dev;             /* out: [B][C][H][W] fp32 */
  void* den_in_dev;            /* out: bf16 NHWC [B][H][W][16] */
} psgla_next_pre;
int psgla_dncnn_residual_post_next(int depth, const void* packed_dev, psgla_img_shape shape, const void* den_in_dev,
                                   void* workspace_dev, size_t workspace_bytes, const float* base_dev,
                                   const psgla_post_params* post, float* x_out_dev, float* sample_dev, float* mean_dev,
                                   float* mean2_dev, const psgla_next_pre* next, void* stream);

/* The last layer of that chain alone (64 -> C channels + the fused post / next pre): hidden_dev = bf16 NHWC [B][H][W][64], the
 * output of layer depth - 2.  What psgla_dncnn_residual_post_next launches last; exposed so that the fused epilogue can be
 * timed (bench.py's HBM roofline of this stage) and tested on its own. */
int psgla_dncnn_last_layer_post_next(int depth, const void* packed_dev, psgla_img_shape shape, const void* hidden_dev,
                                     const float* base_dev, const psgla_post_params* post, float* x_out_dev,
                                     float* sample_dev, float* mean_dev, float* mean2_dev, const psgla_next_pre* next,
                                     void* stream);

/* Single conv3x3 layers, exposed for parity tests against torch.nn.functional.conv2d.
 *   cin_pad: 16 (first layer, channels C..15 zero) or 64.   in_dev: bf16 NHWC [B][H][W][cin_pad].
 *   out_dev: bf16 NHWC [B][H][W][64], ReLU applied if relu != 0; the last layer: the raw conv as fp32 NCHW [B][C][H][W].
 *   layer: index into the packed weights. */
int psgla_conv3x3_layer(const void* packed_dev, int depth, int layer, psgla_img_shape shape, const void* in_dev,
                        void* out_dev, int relu, void* stream);

/* Layout helper: fp32 NCHW [B][C][H][W] -> bf16 NHWC [B][H][W][16]: the C channels from slot 0, slot 3 = c3 (the DRUNet
 * noise-level map, 0 for DnCNN), every other slot zero. */
int psgla_img_to_nhwc16(psgla_img_shape shape, const float* x_dev, float c3, void* out_dev, void* stream);

/* In-place replication padding of a bf16 NHWC16 batch [B][padded.H][padded.W][16]: pixels with y >= H or x >= W copy the nearest
 * valid pixel (KAIR's test_pad, what the DRUNet of the reference -- deepinv.models.DRUNet, sampling_images.py:136 -- applies to
 * inputs whose sides are not multiples of 8).  The samplers call it on the denoiser input before every DRUNet application of a
 * problem that was padded to multiples of 8. */
int psgla_img_pad_replicate_nhwc16(psgla_img_shape padded, int H, int W, void* img_dev, void* stream);

/* Total-variation denoiser (deepinv.models.TVDenoiser, sampling_images.py:139-140; the PSGLA-TV runs of :181-184): the prox
 *   D(y) = argmin_x 1/2 ||x - y||^2 + ths * sum_{c,p} ||(grad x)_{c,p}||_2     (isotropic per channel and pixel)
 * by over-relaxed Chambolle-Pock, tau, rho, sigma = 1 / (8 tau), iterated until ||x_prev - x2|| / ||x2 + 1e-12|| < crit after
 * the third iteration or n_it_max iterations.  The norms run per chain, so a chain's result does not depend on the other
 * chains of the batch.  fp32 state and arithmetic; one cooperative launch per call, fused with the post:
 *   x_out = post->base_scale * y + post->gain * D(y), thinning and moments as in psgla_dncnn_residual_post.
 * state_dev (psgla_tv_state_bytes): x2 fp32 [B][3][H][W], then u2 fp32 [B][3][H][W][2]; restart = 0 continues from it (warm
 * start), restart = 1 starts from x2 = y, u2 = 0.  On return it holds each chain's final x2 / u2.
 * workspace_dev (psgla_tv_workspace_bytes): the second ping-pong copy of the state, per-tile partial sums, per-chain counters.
 * x_out_dev may alias y_dev; state_dev may not.  iters_dev: NULL or int32 [B], each chain's CP iteration count.
 * Any H, W >= 1. */
typedef struct psgla_tv_params {
  float ths, tau, rho, crit;   /* ths > 0; tau > 0; 0 < rho < 2; crit >= 0 (0: run n_it_max) */
  int32_t n_it_max;            /* >= 1 */
  int32_t restart;             /* 1: x2 = y, u2 = 0 first; 0: continue from state_dev */
} psgla_tv_params;             /* psgla_struct_size(5) */
size_t psgla_tv_state_bytes(psgla_img_shape shape);      /* x2 fp32 [B][3][H][W], then u2 fp32 [B][3][H][W][2]; 0: bad shape */
size_t psgla_tv_workspace_bytes(psgla_img_shape shape);  /* ping-pong copy, tile partials, counters; 0: bad shape */
int psgla_tv_prox_post(const psgla_tv_params* tv, psgla_img_shape shape, const float* y_dev, void* state_dev,
                       size_t state_bytes, void* workspace_dev, size_t workspace_bytes, const psgla_post_params* post,
                       float* x_out_dev, float* sample_dev, float* mean_dev, float* mean2_dev, int32_t* iters_dev,
                       void* stream);

/* Convergence diagnostics of a multi-chain run, per element (csrc/mcmc_diag.cu): rank-normalised split-R-hat and bulk / tail
 * ESS (Vehtari et al. 2021), as arviz's rhat(method="rank"), ess(method="bulk"), ess(method="tail") define them.
 *   draws_dev   fp32 [n_draws][n_chains][n_elem]: the samplers' own sample buffer ([n_samples][B][C][H][W]), read in place.
 *   rhat_dev, ess_bulk_dev, ess_tail_dev   fp32 [n_elem].  R-hat = max(bulk, folded-tail) split-R-hat; tail ESS = the smaller
 *               ESS of the indicators x <= q05, x <= q95.  An element with NaN draws, or whose split chains are each constant
 *               in a series (W = 0), gets NaN for the statistics of that series.
 * Each chain is split into two halves (odd n_draws: the middle draw is dropped), so an element has S = 2 n_chains
 * floor(n_draws / 2) split draws; n_draws >= 4, n_chains >= 1 and S <= PSGLA_MCMC_MAX_DRAWS (one element's draws are sorted
 * in shared memory).  A longer run is diagnosed after thinning it further (a larger n_inter) or on fewer chains.
 * ws_dev: psgla_mcmc_diag_workspace_bytes(n_draws, n_chains) bytes (0: out of range), 256-byte aligned.  On return its first
 * four uint64 hold the SM cycles the call spent, summed over elements, in: loading the draws; sorting them (with the median
 * and quantiles); ranking and normal scores; chain moments and autocovariances.  Deterministic: an element's results do not
 * depend on n_elem or on the other elements. */
#define PSGLA_MCMC_MAX_DRAWS 16384
size_t psgla_mcmc_diag_workspace_bytes(int64_t n_draws, int64_t n_chains);
int psgla_mcmc_diag(const float* draws_dev, int64_t n_draws, int64_t n_chains, int64_t n_elem, void* ws_dev, size_t ws_bytes,
                    float* rhat_dev, float* ess_bulk_dev, float* ess_tail_dev, void* stream);

/* tcgen05 descriptor self-test (development aid): runs a 128 x 64 x 64 GEMM tile whose A operand starts `row_shift`
 * rows into a 128B-swizzled shared-memory buffer.  mode 0: A from shared memory, shift = descriptor start address;
 * mode 2: A copied to tensor memory.
 * a_dev: bf16 [136][64], b_dev: bf16 [64][64] (N x K), d_dev: fp32 [128][64]. */
int psgla_selftest_umma(const void* a_dev, const void* b_dev, float* d_dev, int row_shift, int mode, void* stream);
/* CTA-pair (cta_group::2) self-test: D[256][64] = A[256][64] B[64][64]^T by one pair of CTAs, A rows split 128 / 128 over
 * the two CTAs' tensor memories (mode 0) or shared memories (mode 1), B rows split 32 / 32 over their shared memories. */
int psgla_selftest_umma2(const void* a_dev, const void* b_dev, float* d_dev, int mode, void* stream);

/* PSNR and SSIM of n = shape.B images [n][C][H][W] (fp32) against one reference image [C][H][W], on the device: the
 * per-sample metric loop of sampling_images.py:373-384 and the MMSE curves of :411-433 without copying samples to the host.
 * skimage 0.24 definitions as the reference calls them: PSNR = 10 log10(R^2 / MSE); SSIM = 7x7 uniform window, sample
 * covariance, K1 = 0.01, K2 = 0.03, mean over the interior and the channels (channel_axis=2).  Either output may be NULL.
 * workspace: psgla_img_metrics_workspace_bytes(n) bytes. */
size_t psgla_img_metrics_workspace_bytes(int n);
int psgla_img_psnr_ssim(psgla_img_shape shape, const float* stack_dev, const float* ref_dev, float data_range,
                        void* workspace_dev, size_t workspace_bytes, float* psnr_out_dev, float* ssim_out_dev, void* stream);

/* DRUNet (deepinv.models.DRUNet(in_channels=C, out_channels=C), sampling_images.py:136; KAIR UNetRes nc = 64/128/256/512,
 * nb = 4, no biases).  weights_host: psgla_drunet_num_weights() = 64 fp32 tensors in state-dict order (m_head, m_down1.*,
 * m_down2.*, m_down3.*, m_body.*, m_up3.*, m_up2.*, m_up1.*, m_tail; torch layouts).  den_in_dev: bf16 NHWC16 as written by a
 * "pre" call with den_in_c3 = sigma.  H and W must be multiples of 8.
 * psgla_drunet_denoise_post: X+ = post->base_scale * base + post->gain * DRUNet(den_in), thinning and moments as above.
 * psgla_drunet_pack_weights_ch packs a network of `channels` = 3 or 1 image channels: m_head [64][channels + 1][3][3] (the
 * noise level last, as deepinv appends it), m_tail [channels][64][3][3]; psgla_drunet_pack_weights is it with 3.  The packed
 * size does not depend on the channel count, but a packed buffer must be used with shapes of the channel count it was
 * packed for. */
int psgla_drunet_num_weights(void);
size_t psgla_drunet_packed_bytes(void);
int psgla_drunet_pack_weights(const float* const* weights_host, void* packed_dev, void* stream);
int psgla_drunet_pack_weights_ch(int channels, const float* const* weights_host, void* packed_dev, void* stream);
size_t psgla_drunet_workspace_bytes(psgla_img_shape shape);
int psgla_drunet_denoise_post(const void* packed_dev, psgla_img_shape shape, const void* den_in_dev, void* workspace_dev,
                              size_t workspace_bytes, const float* base_dev, const psgla_post_params* post,
                              float* x_out_dev, float* sample_dev, float* mean_dev, float* mean2_dev, void* stream);
int psgla_drunet_denoise_post_next(const void* packed_dev, psgla_img_shape shape, const void* den_in_dev, void* workspace_dev,
                                   size_t workspace_bytes, const float* base_dev, const psgla_post_params* post,
                                   float* x_out_dev, float* sample_dev, float* mean_dev, float* mean2_dev,
                                   const psgla_next_pre* next, void* stream);
/* One layer of that network, exposed for parity tests like psgla_conv3x3_layer: exactly the kernel, ReLU and residual adds
 * psgla_drunet_denoise_post runs for it.  layer: 0..63 in the state-dict order above; shape: the network's image shape (H, W
 * multiples of 8); the layer works at its own scale of it.  in_dev: bf16 NHWC16 (layer 0, channel 3 = sigma) or bf16 NHWC.
 * out_dev: bf16 NHWC, or for layer 63 the raw conv as fp32 NCHW [B][C][H][W].  res1_dev (the residual block's input) must
 * be given exactly for the second conv of a residual block, res2_dev (the U-Net skip) exactly for the last such conv of the
 * body and of each decoder stage; both are bf16 NHWC of the output's shape. */
int psgla_drunet_layer(const void* packed_dev, psgla_img_shape shape, int layer, const void* in_dev, const void* res1_dev,
                       const void* res2_dev, void* out_dev, void* stream);

/* Gradient-step DRUNet (deepinv.models.GSDRUNet(alpha, in_channels=3, out_channels=3, nb=2, nc=[64,128,256,512],
 * act_mode="E"), sampling_images.py:129-140; Prox-DRUNet is the same network from another checkpoint):
 *   N = KAIR UNetRes with nb = 2 residual blocks x + conv(elu(conv(x))) per stage, no biases, sigma map as fourth input channel
 *   D(x) = x - alpha (v - J^T v),  v = x - N(x),  J^T v = the vector-Jacobian product of N at x (sigma's gradient dropped).
 * weights_host: psgla_gsdrunet_num_weights() = 36 fp32 tensors in state-dict order (m_head, m_down1.{0,1}.res.{0,2}, m_down1.2,
 * m_down2.*, m_down3.*, m_body.{0,1}.res.{0,2}, m_up3.0, m_up3.{1,2}.res.{0,2}, m_up2.*, m_up1.*, m_tail; torch layouts); the
 * packed buffer holds them for the forward and, repacked as adjoints, for the backward.  H and W must be multiples of 8.
 * psgla_gsdrunet_denoise_post_next: X+ = post->base_scale * base + post->gain * D(x), thinning, moments and the optional next
 * pre as in psgla_drunet_denoise_post_next.  den_in_dev: bf16 NHWC16 of x with channel 3 = sigma (a "pre" call's output);
 * x_dev: x itself, fp32 [B][3][H][W], or NULL when x is base_dev (PSGLA; PnP-ULA and RED evaluate D at the chain state X,
 * which may be x_out_dev).  alpha: finite.  One call is 72 conv launches and one element-wise launch; the workspace holds
 * the forward activations, the 14 ELU outputs the backward's gates read and the four held skip gradients (~2 KB per pixel). */
int psgla_gsdrunet_num_weights(void);
size_t psgla_gsdrunet_packed_bytes(void);
int psgla_gsdrunet_pack_weights(const float* const* weights_host, void* packed_dev, void* stream);
size_t psgla_gsdrunet_workspace_bytes(psgla_img_shape shape); /* 0: bad shape */
int psgla_gsdrunet_denoise_post_next(const void* packed_dev, psgla_img_shape shape, const void* den_in_dev, const float* x_dev,
                                     void* workspace_dev, size_t workspace_bytes, const float* base_dev, float alpha,
                                     const psgla_post_params* post, float* x_out_dev, float* sample_dev, float* mean_dev,
                                     float* mean2_dev, const psgla_next_pre* next, void* stream);
/* One layer of that call, for tests: backward = 0: forward layer 0..35 (state-dict order); backward = 1: backward layer b =
 * the adjoint of forward layer 35 - b.  in_dev: bf16 NHWC16 (forward 0, channel 3 = sigma; backward 0, the cotangent in
 * channels 0..2) or bf16 NHWC; out_dev: bf16 NHWC, or the raw conv as fp32 NCHW [B][3][H][W] for forward 35 and backward 35.
 * res1_dev / res2_dev exactly where the layer adds them (forward: as psgla_drunet_layer; backward: res1 = the gradient of
 * the block's output on each first conv's adjoint, res2 = the held skip gradient on the first block's of the body and of
 * each encoder stage); gate_dev exactly for the adjoint of each block's second conv: the forward's ELU output of that block,
 * the conv is multiplied by elu'(z) (1 where gate > 0, else gate + 1).  All bf16 NHWC of the output's shape. */
int psgla_gsdrunet_layer(const void* packed_dev, psgla_img_shape shape, int backward, int layer, const void* in_dev,
                         const void* res1_dev, const void* res2_dev, const void* gate_dev, void* out_dev, void* stream);

/* One general convolution layer of the DRUNet denoiser (deepinv.models.DRUNet, sampling_images.py:136) as implicit GEMM:
 *   mode 0: 3x3 stride 1 zero-pad 1 (Cin -> Cout); 1: 2x2 stride 2 (downsampling); 2: 2x2 stride 2 transposed (upsampling).
 * in_dev bf16 NHWC [B][Hin][Win][Cin]; w_dev bf16 [taps][Cout][Cin] (taps = 9 / 4 / 4, tap = ky * kw + kx);
 * out_dev bf16 NHWC of extent Hin x Win / Hin/2 x Win/2 / 2Hin x 2Win; res1_dev / res2_dev: optional tensors of the
 * output's shape that are added before the optional ReLU.  Channels are multiples of 64; no bias (DRUNet has none). */
int psgla_convg_layer(int mode, int B, int Hin, int Win, int Cin, int Cout, const void* w_dev, const void* in_dev,
                      const void* res1_dev, const void* res2_dev, void* out_dev, int relu, void* stream);

/* tcgen05 issue-rate probe (development aid): every one of `grid` CTAs issues iters x 4 MMAs of shape M128 x n x K16
 * (bf16, zeroed operands) back to back and writes the elapsed SM cycles to cycles_dev[block].
 * mode 0: A and B from shared memory; 1: same with the A start address shifted by one 128-byte row; 2: A from TMEM;
 * 3 / 4: as 2 / 0 with consecutive MMAs alternating between two accumulators (n <= 128). */
int psgla_selftest_mma_rate(int mode, int n, int iters, int grid, long long* cycles_dev, void* stream);
/* The same for a CTA pair: M256 x n x K16 MMAs (cta_group::2), mode 0: A from tensor memory, 1: from shared memory;
 * cycles_dev[n_pairs] = cycles the leader of each pair took for iters x 4 MMAs. */
int psgla_selftest_mma_rate2(int mode, int n, int iters, int n_pairs, long long* cycles_dev, void* stream);

/* FP32 issue-rate probe: the measured denominator of the 2D chain kernel's roofline.  num_sms x blocks_per_sm blocks of 256
 * threads each run iters x 32 dependent-chain FMAs per thread (8 independent chains), mode 0: FFMA, mode 1: the packed FFMA2
 * (fma.rn.f32x2).  out_dev: scratch of num_sms x blocks_per_sm x 256 floats (never written in practice); *flop_out (host) =
 * flop the launch performs, so TFLOP/s = *flop_out / (CUDA-event time). */
int psgla_selftest_fp32_rate(int mode, int iters, int blocks_per_sm, float* out_dev, double* flop_out, void* stream);
/* The same for single instruction classes of the chain kernel's mix (csrc/selftest.cu lists the modes: 0 IMAD.WIDE.U32, 1
 * IMAD.HI.U32, 2 IMAD, 3 LOP3, 4 MUFU.EX2, 5 I2FP, 6 FFMA, 7 MUFU.SIN, 8 IMAD.WIDE + FFMA 1:1, 9 MUFU + IMAD.WIDE 1:1, 10 MUFU + 4
 * FFMA, 11 and 100 + NF (NF = 21, 23, 26, 28, 30): the chain kernel's whole per-step instruction mix with NF FP32 instructions as
 * independent chains, 12 DFMA.RM, 13 IMAD + DFMA.RM + LOP3, 14 DFMA.RM + FFMA 1:1, 200 + NF: the mix with the Philox round
 * products' high words as DFMA.RM on the FP64 pipe); *ops_out = thread-level instructions of the probed class the launch executes (modes 8-10: of the
 * first-named class; mix modes: thread-level "steps"). */
int psgla_selftest_pipe_rate(int mode, int iters, int blocks_per_sm, void* out_dev, double* ops_out, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* PSGLA_B200_H */
