// common.cuh -- shared device helpers of the sm_100a backend.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>

namespace hifgpu {

// ---- error handling: CUDA failures become exceptions inside the library and are
// turned into LhfStatus + message at the C boundary (capi.cu) -------------------
struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

inline void cuda_check(cudaError_t e, const char *what, const char *file, int line) {
  if (e != cudaSuccess) {
    throw CudaError(std::string(what) + " failed: " + cudaGetErrorString(e) + " (" + file + ":" +
                    std::to_string(line) + ")");
  }
}
#define HIF_CUDA(call) ::hifgpu::cuda_check((call), #call, __FILE__, __LINE__)
#define HIF_KERNEL_CHECK() ::hifgpu::cuda_check(cudaGetLastError(), "kernel launch", __FILE__, __LINE__)

constexpr int kNumSMs = 148;  // B200

// ---- readiness-tagged values ---------------------------------------------------
// A value produced by a sync-free sweep carries its own ready flag in the least
// significant mantissa bit: a consumer polls ONE 8-byte word that delivers both the
// data and "it has been written during this apply".  Every tagged buffer is written
// exactly once per apply, so the stale content always carries the other parity and no
// reset pass over the buffers is needed between applies.  Cost: <= 1 ulp per stored
// intermediate (2.2e-16 relative), far inside the 1e-12 parity budget.
__device__ __forceinline__ unsigned long long tag_set(double v, unsigned parity) {
  return (static_cast<unsigned long long>(__double_as_longlong(v)) & ~1ull) | parity;
}
__device__ __forceinline__ bool tag_ready(unsigned long long bits, unsigned parity) {
  return ((static_cast<unsigned>(bits) ^ parity) & 1u) == 0u;  // 32-bit: the 64-bit compare cost two more instructions per poll
}
__device__ __forceinline__ double tag_value(unsigned long long bits) {
  return __longlong_as_double(static_cast<long long>(bits));
}
// host twin of tag_set for the emulations of the sweeps (wsweep.cu, stream.cu): the value a consumer
// of the tagged word computes with
inline double tag_set_host(double v, unsigned parity) {
  unsigned long long b;
  std::memcpy(&b, &v, 8);
  b = (b & ~1ull) | parity;
  std::memcpy(&v, &b, 8);
  return v;
}

// polling load: must observe other SMs' stores -> L2 (never a stale L1 line)
__device__ __forceinline__ unsigned long long ld_poll(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_publish(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// streaming read-only loads for factor data (touched once per sweep)
__device__ __forceinline__ double ldg_stream(const double *p) { return __ldg(p); }
__device__ __forceinline__ int ldg_stream(const int *p) { return __ldg(p); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// a spin that exceeds this many polls flags an error instead of hanging the GPU
constexpr unsigned kSpinLimit = 1u << 26;

}  // namespace hifgpu
