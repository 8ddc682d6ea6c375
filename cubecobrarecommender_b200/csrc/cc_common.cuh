// Shared helpers for the cubecobra_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cubecobra_b200.h"

namespace cc {

// ---- error convention: int return, message kept per host thread -------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define CC_CHECK_CUDA(expr)                                                     \
  do {                                                                          \
    cudaError_t _e = (expr);                                                    \
    if (_e != cudaSuccess) return cc::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define CC_CHECK_LAUNCH()                                                          \
  do {                                                                             \
    cudaError_t _e = cudaPeekAtLastError();                                        \
    if (_e != cudaSuccess) return cc::cuda_fail(_e, "launch", __FILE__, __LINE__); \
  } while (0)

#define CC_REQUIRE(cond, ...)        \
  do {                               \
    if (!(cond)) {                   \
      cc::set_error(__VA_ARGS__);    \
      return CC_ERR_ARGUMENT;        \
    }                                \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// NVTX range around every C-ABI entry point that enqueues work (header-only NVTX v3: a no-op unless a tool such as
// Nsight Systems / ncu --nvtx injects itself), so a timeline shows which host call a kernel belongs to.
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};
#define CC_NVTX(name) cc::NvtxRange cc_nvtx_range_(name)

int sm_count();

template <typename T>
__host__ __device__ constexpr T ceil_div(T a, T b) { return (a + b - 1) / b; }

// ---- device helpers ---------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// round-to-nearest fp32 -> tf32 (the tensor core's kind::tf32 truncates the low 13 mantissa bits, which
// biases every product towards zero; operands are rounded once, where they are produced)
__device__ __forceinline__ float rn_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// the same rounding (nearest, ties away from zero) as two integer operations: add half a tf32 ulp to the
// magnitude bits, clear the 13 low bits (cvt.rna.tf32.f32 expands to more, with Inf/NaN handling the gradients
// and activations rounded in the GEMM epilogues never need)
__device__ __forceinline__ float rn_tf32_bits(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

// sigmoid of a logit as the recommenders report it (reference ml_recommend.py:78-80 reads float32 sigmoid
// outputs); ONE definition, so the fused select and the standalone sigmoid pass give identical bits
__device__ __forceinline__ float sigmoid_f32(float z) { return 1.f / (1.f + expf(-z)); }

// streaming 128-bit loads that do not pollute L1 (data is read once per CTA)
__device__ __forceinline__ uint4 ld_nc_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ld_nc_f4(const void* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ double2 ld_nc_d2(const void* p) {
  double2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
  return r;
}
// ---- the recommender's total order on (score, index): every select and the target-rank kernel ----------
template <typename T> struct KeyOf;
template <> struct KeyOf<float> {
  using U = uint32_t; using K = unsigned long long; static constexpr int BITS = 64;
  __device__ static U ord(float v) { v += 0.0f; U b = __float_as_uint(v); return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u); }
};
template <> struct KeyOf<double> {
  using U = unsigned long long; using K = unsigned __int128; static constexpr int BITS = 96;
  __device__ static U ord(double v) {
    v += 0.0; U b = (U)__double_as_longlong(v);
    return b ^ ((b >> 63) ? 0xffffffffffffffffull : 0x8000000000000000ull);
  }
};

// composite key: (orderable score, tie word); all keys of one cube are distinct, so the
// n-th largest is unique and {key >= it} has exactly n members.
//   descending: larger score first, ties -> larger index first  (argsort(stable)[::-1])
//   ascending : smaller score first, ties -> smaller index first (argsort(stable))
template <typename T>
__device__ __forceinline__ typename KeyOf<T>::K make_key(T v, uint32_t idx, int descending) {
  using KO = KeyOf<T>;
  typename KO::U u = KO::ord(v);
  uint32_t t = idx;
  if (!descending) { u = ~u; t = ~idx; }
  return (typename KO::K(u) << 32) | typename KO::K(t);
}

// a bound on the RAW value such that no element whose key is >= thr fails `pass`: the threshold's own score, or --
// fused sigmoid -- its logit.  The logit is evaluated in float32 (one thread computes it while the CTA waits, and a
// double-precision log costs that thread several hundred cycles).  The probability is first moved 2e-6 relative to the
// safe side (16-33 float32 ulps: covers the <= 3 ulp error of sigmoid_f32 = 1 / (1 + expf(-z)) with IEEE division, and
// keeps 1 - p >= 2e-6); the float32 logit of the moved probability is then moved by a bound on its own evaluation error:
// 1e-5 (1 + |L|) for the quotient and logf (~80 ulps of L) plus 2.5e-7 / (1 - p) for the rounding of p next to 1 (half
// an ulp of p is 3e-8 of the 1 - p it is subtracted from).  A constant slack of 0.08 (round 1) was safe but let EVERY
// element of a row whose logits lie within 0.08 of each other (an untrained model) into the survivor buffer, sending
// the cube through the overflow path; the slack here is 1e-5 for logits near 0 and grows to 0.125 only where the sigmoid
// saturates.  A looser bound only lets a few more elements into the survivor buffer; it never loses one (checked densely
// against float32 sigmoid on the host, tests/test_rowselect_model.py).
__device__ __forceinline__ float rs_logit_slack(float logit, float one_minus_p) {
  return 1e-5f * (1.f + fabsf(logit)) + 2.5e-7f / one_minus_p;
}
template <bool SIGMOID>
__device__ __forceinline__ float rs_raw_bound(unsigned long long thr, int descending) {
  if (thr == 0ull) return descending ? -INFINITY : INFINITY;
  uint32_t u = (uint32_t)(thr >> 32);
  if (!descending) u = ~u;
  const float pthr = __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
  if (!SIGMOID) return pthr;
  if (descending) {
    const float pm = pthr * (1.f - 2e-6f) - 1e-37f;
    if (pm <= 0.f) return -INFINITY;
    const float l = logf(pm / (1.f - pm));
    return l - rs_logit_slack(l, 1.f - pm);
  }
  const float pp = pthr * (1.f + 2e-6f) + 1e-37f;
  if (pp >= 1.f) return INFINITY;
  const float l = logf(pp / (1.f - pp));
  return l + rs_logit_slack(l, 1.f - pp);
}
// the float64 counterpart (no sigmoid): the threshold key's own double, decoded from its 64-bit score word
__device__ __forceinline__ double rs_raw_bound_f64(unsigned __int128 thr, int descending) {
  if (thr == 0) return descending ? -INFINITY : INFINITY;
  unsigned long long u = (unsigned long long)(thr >> 32);
  if (!descending) u = ~u;
  return __longlong_as_double((long long)((u & 0x8000000000000000ull) ? (u ^ 0x8000000000000000ull) : ~u));
}
#endif

}  // namespace cc
