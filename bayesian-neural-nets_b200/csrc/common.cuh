// Shared device/host helpers for liblbbnn (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

#include "../../include/lbbnn.h"

namespace lbbnn {

// ---- error plumbing (C-ABI returns int, message via lbbnn_last_error) -------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define LBBNN_REQUIRE(cond, ...)                                  \
  do {                                                            \
    if (!(cond)) {                                                \
      ::lbbnn::set_error(__VA_ARGS__);                            \
      return LBBNN_ERR_INVALID;                                   \
    }                                                             \
  } while (0)

#define LBBNN_CUDA(call)                                                           \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      ::lbbnn::set_error("%s failed: %s", #call, cudaGetErrorString(e__));         \
      return LBBNN_ERR_CUDA;                                                       \
    }                                                                              \
  } while (0)

int sm_count();

// ---- scalar math of the variational parameters ------------------------------------------------
// sigma = log1p(exp(rho)) with no threshold, alpha = 1/(1+exp(-lambda)): the reference's own
// formulations (LBBNN-GP-MF-LRT.py:80-82,167), so fp32 rounding follows the same path.
__device__ __forceinline__ float sigma_of(float rho) { return log1pf(expf(rho)); }
__device__ __forceinline__ float alpha_of(float lam) { return 1.0f / (1.0f + expf(-lam)); }

// x = hi + lo with hi representable in TF32 (round to nearest on the 13 dropped mantissa bits); lo = x - hi is exact
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  const uint32_t u = __float_as_uint(x);
  hi = __uint_as_float((u + 0x1000u) & 0xFFFFE000u);
  lo = x - hi;
}
// d sigma / d rho = e^rho / (1 + e^rho)
__device__ __forceinline__ float dsigma_drho(float rho) {
  float e = expf(rho);
  return e / (1.0f + e);
}

struct Moments { float m, v; };
// M = alpha*mu (*z for MNF), V = sigma^2 alpha^2 (reference) or alpha(sigma^2+(1-alpha)mu^2) (exact)
__device__ __forceinline__ Moments weight_moments(float mu, float sigma, float alpha, int var_mode) {
  Moments r;
  r.m = mu * alpha;
  r.v = (var_mode == LBBNN_VAR_REFERENCE) ? (sigma * sigma) * (alpha * alpha)
                                          : alpha * (sigma * sigma + (1.0f - alpha) * mu * mu);
  return r;
}

// KL contribution of one weight (LRT:189-192; with MNF's z folded in as mu*z, MNF:230-233)
__device__ __forceinline__ float kl_weight_elem(float mu_z, float sigma, float alpha, const lbbnn_priors& p) {
  float d = mu_z - p.mu;
  float slab = logf(p.sigma / sigma) - 0.5f + logf(alpha / p.alpha) +
               (sigma * sigma + d * d) / (2.0f * p.sigma * p.sigma);
  float om = 1.0f - alpha;
  return alpha * slab + om * logf(om / (1.0f - p.alpha));
}
// KL contribution of one bias (LRT:185-186)
__device__ __forceinline__ float kl_bias_elem(float mu, float sigma, const lbbnn_priors& p) {
  float d = mu - p.bias_mu;
  return logf(p.bias_sigma / sigma) - 0.5f + (sigma * sigma + d * d) / (2.0f * p.bias_sigma * p.bias_sigma);
}

// ---- reductions ------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum; result valid in thread 0.  `scratch` holds >= 32 T's.  Deterministic order.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  T r = T(0);
  if (warp == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? scratch[lane] : T(0);
    r = warp_sum(r);
  }
  return r;
}

// ---- Philox4x32-10 + Box-Muller --------------------------------------------------------------------
// One call yields 4 words for counter (idx, stream) under key seed.  Element i of a tensor uses
// idx = i/4, word i%4, so any kernel that walks the tensor 4 elements at a time reproduces the same
// values as lbbnn_philox_export.
struct Philox4 { uint32_t x, y, z, w; };

__device__ __forceinline__ Philox4 philox4x32_10(uint64_t seed, uint64_t stream, uint64_t idx) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  uint32_t c0 = (uint32_t)idx, c1 = (uint32_t)(idx >> 32), c2 = (uint32_t)stream, c3 = (uint32_t)(stream >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return Philox4{c0, c1, c2, c3};
}

// uniform in (0,1): 24 random bits, never 0 or 1
__device__ __forceinline__ float u01(uint32_t w) { return ((float)(w >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// Box-Muller on the special-function unit: log and sin / cos through MUFU (__logf, __sincosf: absolute error 2^-21 on
// the angle range (-pi, pi) used here) -- the accurate logf / sincospif cost ~90 of the ~250 instructions of a quad of
// draws and made every sampling kernel issue-bound.  lbbnn_philox_normal exports exactly these values, so the oracle's
// noise and the fused kernels' noise stay identical.
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint64_t stream, uint64_t idx, float out[4]) {
  Philox4 p = philox4x32_10(seed, stream, idx);
  float r0 = sqrtf(-2.0f * __logf(u01(p.x))), r1 = sqrtf(-2.0f * __logf(u01(p.z)));
  float s0, c0, s1, c1;
  __sincosf(6.28318530717958647692f * (u01(p.y) - 0.5f), &s0, &c0);
  __sincosf(6.28318530717958647692f * (u01(p.w) - 0.5f), &s1, &c1);
  out[0] = r0 * c0; out[1] = r0 * s0; out[2] = r1 * c1; out[3] = r1 * s1;
}
__device__ __forceinline__ void philox_uniform4(uint64_t seed, uint64_t stream, uint64_t idx, float out[4]) {
  Philox4 p = philox4x32_10(seed, stream, idx);
  out[0] = u01(p.x); out[1] = u01(p.y); out[2] = u01(p.z); out[3] = u01(p.w);
}
// single element (odd shapes): recomputes the group, picks the lane
__device__ __forceinline__ float philox_normal1(uint64_t seed, uint64_t stream, uint64_t elem) {
  float n[4];
  philox_normal4(seed, stream, elem >> 2, n);
  return n[elem & 3];
}
__device__ __forceinline__ float philox_uniform1(uint64_t seed, uint64_t stream, uint64_t elem) {
  float n[4];
  philox_uniform4(seed, stream, elem >> 2, n);
  return n[elem & 3];
}

// eps source: injected tensor or native Philox (device view of lbbnn_noise)
struct Noise {
  const float* ptr;   // non-null: injected, indexed like the output tensor
  uint64_t seed, stream;
  const int64_t* step_dev;
  uint64_t step_stride;
  // resolve the per-replay stream once per thread
  __device__ __forceinline__ void resolve() {
    if (step_dev) stream += (uint64_t)(*step_dev) * step_stride;
    step_dev = nullptr;
  }
};
inline Noise make_noise(const lbbnn_noise* n) {
  Noise r{nullptr, 0, 0, nullptr, 0};
  if (n) { r.ptr = n->eps; r.seed = n->seed; r.stream = n->stream_id; r.step_dev = n->step_dev; r.step_stride = n->step_stride; }
  return r;
}

__host__ __device__ __forceinline__ int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// NVSwitch multicast (NVLS) access through a multicast address: ld_reduce returns the sum over every rank's copy (the
// reduction happens in the switch), st writes the value to every rank's copy.
__device__ __forceinline__ float4 mc_ld_reduce4(const float* p) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ void mc_st4(float* p, const float v[4]) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3])
               : "memory");
}
__device__ __forceinline__ float mc_ld_reduce1(const float* p) {
  float r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.f32 %0, [%1];" : "=f"(r) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ void mc_st1(float* p, float v) {
  asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

}  // namespace lbbnn
