// Shared helpers for the sscvae sm_100a kernels (error plumbing, small device utilities).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cstdlib>
#include <cstring>

typedef __nv_bfloat16 bf16;

namespace sscvae {

// ---- error plumbing: no exceptions cross the C ABI (SURVEY §8b) -------------------------------
void set_error(const char* fmt, ...);
const char* get_error();

#define SSCVAE_ERR_BAD_ARG (-1)
#define SSCVAE_ERR_WORKSPACE (-2)
#define SSCVAE_ERR_UNSUPPORTED (-3)
#define SSCVAE_ERR_DRIVER (-4)

#define CUDA_TRY(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      sscvae::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return (int)_e;                                                                      \
    }                                                                                      \
  } while (0)

#define TRY(expr)                 \
  do {                            \
    int _r = (expr);              \
    if (_r != 0) return _r;       \
  } while (0)

#define REQUIRE(cond, ...)                 \
  do {                                     \
    if (!(cond)) {                         \
      sscvae::set_error(__VA_ARGS__);      \
      return SSCVAE_ERR_BAD_ARG;           \
    }                                      \
  } while (0)

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
static inline size_t round_up_sz(size_t x, size_t m) { return (x + m - 1) / m * m; }
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ---- device utilities ---------------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// 8 bf16 <-> 16-byte vector
struct __align__(16) bf16x8 { __nv_bfloat162 v[4]; };

__device__ __forceinline__ bf16x8 ld_bf16x8(const bf16* p) { return *reinterpret_cast<const bf16x8*>(p); }
__device__ __forceinline__ void st_bf16x8(bf16* p, const bf16x8& v) { *reinterpret_cast<bf16x8*>(p) = v; }

}  // namespace sscvae
