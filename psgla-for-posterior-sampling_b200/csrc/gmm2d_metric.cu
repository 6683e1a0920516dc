// Sliced Wasserstein-2 distance between the current chain population and a posterior sample, on the device
// (sampling_2D.py:168-170 `ot.sliced.sliced_wasserstein_distance(..., p=2)`; SURVEY.md section 8 row f4: the metric "every
// k steps" of sampling_2D.py:38-39,65-66 for a population that never leaves HBM).
//
//   project   : keys[p][i] = sortable(theta_p . x_i)                       (one read of the state, P coalesced writes)
//   sort      : per projection, LSD radix sort of the 32-bit keys, 4 passes of 8 bits (radix_sort.cuh, keys only):
//                 histogram (per tile of 4096 keys) -> exclusive scan over [digit][tile] -> stable scatter, in which each
//                 warp owns a contiguous slice of the tile and ranks equal digits with __match_any_sync
//   reduce    : sum_p sum_i (sorted_x[p][i] - sorted_ref[p][i])^2 in double -> sqrt(mean)
// HBM-bound: 4 passes x (2 reads + 1 write) x 4 B per key; at P = 50, n = 10^6 that is 2.4 GB per evaluation.
#include "radix_sort.cuh"

namespace psgla {

constexpr int SW_MAX_PROJ = 128;

struct Thetas {
  float t[SW_MAX_PROJ][2];
};

template <typename T>
__global__ void __launch_bounds__(256)
sw_project_kernel(const T* __restrict__ x, long long n, int P, Thetas th, uint32_t* __restrict__ keys) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x0 = (float)x[2 * i], x1 = (float)x[2 * i + 1];
  for (int p = 0; p < P; ++p) keys[(long long)p * n + i] = float_to_key(fmaf(th.t[p][0], x0, th.t[p][1] * x1));
}

__global__ void __launch_bounds__(256)
sw_keys_to_float_kernel(const uint32_t* __restrict__ keys, long long total, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) out[i] = key_to_float(keys[i]);
}

__global__ void __launch_bounds__(256)
sw_diff_kernel(const uint32_t* __restrict__ keys, const float* __restrict__ ref, long long total, double* __restrict__ acc) {
  double s = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const float d = key_to_float(keys[i]) - ref[i];
    s += (double)d * (double)d;
  }
  for (int off = 16; off; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
  __shared__ double ws[8];
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += ws[w];
    atomicAdd(acc, t);
  }
}

__global__ void sw_finalize_kernel(const double* acc, double denom, double* out) { *out = sqrt(*acc / denom); }

struct SwLayout {
  size_t keys_a, keys_b, hist, acc, total;
  int nb;
};
static SwLayout sw_layout(long long n, int P) {
  SwLayout l;
  l.nb = radix_tiles(n);
  const size_t kb = ((size_t)P * (size_t)n * 4 + 255) & ~(size_t)255;
  l.keys_a = 0;
  l.keys_b = kb;
  l.hist = 2 * kb;
  const size_t hb = ((size_t)P * 256 * (size_t)l.nb * 4 + 255) & ~(size_t)255;
  l.acc = l.hist + hb;
  l.total = l.acc + 256;
  return l;
}

// project + sort; returns the buffer (inside ws) that holds the sorted keys [P][n]
static int sw_sorted_keys(const void* x_dev, int precision, long long n, const float* theta_host, int P, void* ws,
                          size_t ws_bytes, cudaStream_t st, uint32_t** sorted) {
  PSGLA_REQUIRE(x_dev && theta_host && ws, "sliced W2: null pointer");
  PSGLA_REQUIRE(precision == 0 || precision == 1, "precision must be 0 (fp32) or 1 (fp64)");
  PSGLA_REQUIRE(n > 0 && n < (1LL << 31) && P > 0 && P <= SW_MAX_PROJ, "sliced W2: n must be in 1..2^31-1 and n_proj in 1..%d",
                SW_MAX_PROJ);
  const SwLayout l = sw_layout(n, P);
  if (ws_bytes < l.total) return set_error(PSGLA_E_WORKSPACE, "sliced W2 workspace: need %zu bytes, got %zu", l.total, ws_bytes);
  PSGLA_REQUIRE(((uintptr_t)ws & 255) == 0, "sliced W2 workspace must be 256-byte aligned");
  Thetas th;
  for (int p = 0; p < P; ++p) th.t[p][0] = theta_host[2 * p], th.t[p][1] = theta_host[2 * p + 1];
  uint32_t* a = reinterpret_cast<uint32_t*>((char*)ws + l.keys_a);
  uint32_t* b = reinterpret_cast<uint32_t*>((char*)ws + l.keys_b);
  uint32_t* hist = reinterpret_cast<uint32_t*>((char*)ws + l.hist);
  const unsigned gb = (unsigned)((n + 255) / 256);
  if (precision == 0)
    sw_project_kernel<float><<<gb, 256, 0, st>>>((const float*)x_dev, n, P, th, a);
  else
    sw_project_kernel<double><<<gb, 256, 0, st>>>((const double*)x_dev, n, P, th, a);
  radix_sort_segments(a, b, nullptr, nullptr, n, P, hist, st);
  PSGLA_CUDA_TRY(cudaGetLastError());
  *sorted = a;  // after an even number of passes the result is back in the first buffer
  return PSGLA_OK;
}

}  // namespace psgla

using namespace psgla;

extern "C" size_t psgla_gmm2d_sw2_workspace_bytes(int64_t n, int n_proj) {
  if (n <= 0 || n_proj <= 0 || n_proj > SW_MAX_PROJ) return 0;
  return sw_layout(n, n_proj).total;
}

extern "C" int psgla_gmm2d_sorted_projections(const void* x_dev, int precision, int64_t n, const float* theta_host,
                                              int n_proj, float* out_sorted_dev, void* ws_dev, size_t ws_bytes,
                                              void* stream) {
  PSGLA_REQUIRE(out_sorted_dev != nullptr, "psgla_gmm2d_sorted_projections: null output");
  uint32_t* sorted = nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = sw_sorted_keys(x_dev, precision, n, theta_host, n_proj, ws_dev, ws_bytes, st, &sorted);
  if (rc) return rc;
  const long long total = (long long)n * n_proj;
  sw_keys_to_float_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(sorted, total, out_sorted_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}

extern "C" int psgla_gmm2d_sliced_w2(const void* x_dev, int precision, int64_t n, const float* theta_host, int n_proj,
                                     const float* ref_sorted_dev, void* ws_dev, size_t ws_bytes, double* out_dev,
                                     void* stream) {
  PSGLA_REQUIRE(ref_sorted_dev && out_dev, "psgla_gmm2d_sliced_w2: null pointer");
  uint32_t* sorted = nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = sw_sorted_keys(x_dev, precision, n, theta_host, n_proj, ws_dev, ws_bytes, st, &sorted);
  if (rc) return rc;
  double* acc = reinterpret_cast<double*>((char*)ws_dev + sw_layout(n, n_proj).acc);
  PSGLA_CUDA_TRY(cudaMemsetAsync(acc, 0, sizeof(double), st));
  const long long total = (long long)n * n_proj;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  sw_diff_kernel<<<(unsigned)blocks, 256, 0, st>>>(sorted, ref_sorted_dev, total, acc);
  sw_finalize_kernel<<<1, 1, 0, st>>>(acc, (double)total, out_dev);
  PSGLA_CUDA_TRY(cudaGetLastError());
  return PSGLA_OK;
}
