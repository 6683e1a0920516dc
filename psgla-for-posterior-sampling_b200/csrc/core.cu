// Error plumbing and library-level queries of libpsgla_b200.
#include "common.cuh"

namespace psgla {

char* last_error_buffer() {
  static thread_local char buf[512] = {0};
  return buf;
}

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(last_error_buffer(), 512, fmt, ap);
  va_end(ap);
  return code;
}

}  // namespace psgla

extern "C" const char* psgla_last_error(void) { return psgla::last_error_buffer(); }

extern "C" int psgla_abi_version(void) { return PSGLA_ABI_VERSION; }

extern "C" int psgla_device_arch(void) {
  int dev = 0, major = 0, minor = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return psgla::set_error(PSGLA_E_NODEVICE, "no CUDA device");
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev) != cudaSuccess)
    return psgla::set_error(PSGLA_E_NODEVICE, "cannot query compute capability");
  return major * 10 + minor;
}

// sizeof() of the ABI structs as this library was compiled, for binding self-checks (0: gmm2d_problem, 1: img_shape,
// 2: pre_params, 3: post_params, 4: next_pre, 5: tv_params).
extern "C" int psgla_struct_size(int which) {
  switch (which) {
    case 0: return (int)sizeof(psgla_gmm2d_problem);
    case 1: return (int)sizeof(psgla_img_shape);
    case 2: return (int)sizeof(psgla_pre_params);
    case 3: return (int)sizeof(psgla_post_params);
    case 4: return (int)sizeof(psgla_next_pre);
    case 5: return (int)sizeof(psgla_tv_params);
    default: return -1;
  }
}

// Philox4x32-10 on the host, the same function the kernels inline: known-answer tests bind this.
extern "C" void psgla_philox4x32_10(const uint32_t* counter, const uint32_t* key, uint32_t* out) {
  uint32_t c0 = counter[0], c1 = counter[1], c2 = counter[2], c3 = counter[3];
  psgla::philox4x32_10(c0, c1, c2, c3, key[0], key[1]);
  out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}
