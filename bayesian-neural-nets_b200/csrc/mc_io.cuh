// Quad-wise loads / stores and TF32 splits shared by the elementwise kernels of the posterior-predictive loops
// (csrc/lrt_predict.cu, csrc/vd_predict.cu): one thread handles four consecutive elements of an n-element buffer, as float4
// when `vec` (the caller checked sizes and alignment), element by element at the ragged end.
#pragma once
#include "common.cuh"

namespace lbbnn {
namespace mc_io {

constexpr int kThreads = 256;

__device__ __forceinline__ void load4(const float* __restrict__ p, int64_t e0, int64_t n, bool vec, float out[4]) {
  if (vec && e0 + 3 < n) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p + e0));
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = (e0 + j < n) ? __ldg(p + e0 + j) : 0.f;
  }
}

__device__ __forceinline__ void store4(float* __restrict__ p, int64_t e0, int64_t n, bool vec, const float v[4]) {
  if (vec && e0 + 3 < n) {
    *reinterpret_cast<float4*>(p + e0) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < n) p[e0 + j] = v[j];
  }
}

// hi / lo of four values into two (n)-element buffers at e0
__device__ __forceinline__ void store_split4(float* __restrict__ hi, float* __restrict__ lo, int64_t e0, int64_t n, bool vec,
                                             const float v[4]) {
  float h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) tf32_split(v[j], h[j], l[j]);
  store4(hi, e0, n, vec, h);
  store4(lo, e0, n, vec, l);
}

inline int64_t grid_for(int64_t quads) {
  int64_t blocks = ceil_div(quads, kThreads);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  return blocks < 1 ? 1 : blocks;
}

}  // namespace mc_io
}  // namespace lbbnn
