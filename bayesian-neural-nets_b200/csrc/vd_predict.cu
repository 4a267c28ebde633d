// Elementwise halves of the variational-dropout posterior-predictive loop (the evaluation branch of run_epoch, VD:148-157)
// on the tensor cores.
//
// The VD forward of a stacked batch of n MC samples is two plain linear layers, E = A theta and S = A^2 theta^2; theta does
// not depend on the sample, so each is ONE 3xTF32 tensor-core GEMM of n * B rows (lbbnn_tc_linear_tf32x3, zero bias).  That
// GEMM reads its weights K-major, (out, in), while theta is (in, out):
//   vd_tc_prepare     hi / lo of theta^T and of (theta .* theta)^T, squared in fp32 while staging (as csrc/vd.cu does), in
//                     one tiled transpose pass -- once per predictor run(), from the current theta
//   vd_mc_epilogue    act = E + sqrtf(S alpha[col]) zeta_s [relu] (the forward epilogue of csrc/vd.cu, alpha kept there
//                     rather than folded into the weights) for the n samples, and the operands of the next tensor-core
//                     layer: hi / lo of act and of act^2.  With shared E and S (stride 0) it is also the CUDA-core layer-1
//                     expansion of the moments lbbnn_vd_fwd_ex(FLAG_MOMENTS) computes once per test batch.
// Native noise is drawn exactly as lbbnn_vd_fwd_ex draws it (stream_id + s * group_stride, element row * m + col).
#include "mc_io.cuh"

namespace lbbnn {
namespace {

using namespace mc_io;

struct VdEpiArgs {
  const float *E, *S;
  int64_t es, ss;              // per-sample strides of E / S in floats (0 = shared by all samples)
  const float* alpha;
  int64_t B, N;
  int n_samples, relu;
  Noise noise;
  uint64_t group_stride;
  float* act;                  // (n, B, N) or NULL
  float *a_hi, *a_lo, *sq_hi, *sq_lo;
};

// One thread = four consecutive elements of one sample (flat index inside the sample: b * N + col).
__global__ void __launch_bounds__(kThreads) vd_mc_epilogue_kernel(const VdEpiArgs a) {
  Noise nz = a.noise;
  nz.resolve();
  const int64_t total = a.B * a.N, nq = ceil_div(total, 4);
  const bool vec = (total % 4 == 0) && aligned16(a.E) && aligned16(a.S) && a.es % 4 == 0 && a.ss % 4 == 0 &&
                   (a.act == nullptr || aligned16(a.act)) && (nz.ptr == nullptr || aligned16(nz.ptr)) &&
                   (a.a_hi == nullptr || (aligned16(a.a_hi) && aligned16(a.a_lo))) &&
                   (a.sq_hi == nullptr || (aligned16(a.sq_hi) && aligned16(a.sq_lo)));
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq * a.n_samples; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i / nq);
    const int64_t q = i - (int64_t)s * nq, e0 = q * 4, so = (int64_t)s * total;
    float v[4], sv[4], z[4];
    load4(a.E + (int64_t)s * a.es, e0, total, vec, v);
    load4(a.S + (int64_t)s * a.ss, e0, total, vec, sv);
    if (nz.ptr) load4(nz.ptr + so, e0, total, vec, z);
    else if (total % 4 == 0) philox_normal4(nz.seed, nz.stream + (uint64_t)s * a.group_stride, (uint64_t)q, z);
    else {
#pragma unroll
      for (int j = 0; j < 4; ++j) z[j] = philox_normal1(nz.seed, nz.stream + (uint64_t)s * a.group_stride, (uint64_t)(e0 + j));
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t col = (e0 + j < total) ? (e0 + j) % a.N : 0;
      const float delta = sv[j] * __ldg(a.alpha + col);      // the expressions of csrc/vd.cu's forward epilogue
      const float sd = sqrtf(delta);
      float o = v[j] + sd * z[j];
      v[j] = a.relu ? fmaxf(o, 0.f) : o;
    }
    if (a.act) store4(a.act + so, e0, total, vec, v);
    if (a.a_hi) store_split4(a.a_hi + so, a.a_lo + so, e0, total, vec, v);
    if (a.sq_hi) {
      float sq[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) sq[j] = v[j] * v[j];
      store_split4(a.sq_hi + so, a.sq_lo + so, e0, total, vec, sq);
    }
  }
}

constexpr int kT = 32;           // transpose tile; 32 x 8 threads, 4 rows each

// theta (n, m) -> hi / lo of theta^T and of (theta^2)^T, both (m, n)
__global__ void __launch_bounds__(kT * 8) vd_tc_prepare_kernel(const float* __restrict__ theta, int64_t n, int64_t m,
                                                               float* __restrict__ t_hi, float* __restrict__ t_lo,
                                                               float* __restrict__ sq_hi, float* __restrict__ sq_lo) {
  __shared__ float tile[kT][kT + 1];
  const int tx = threadIdx.x % kT, ty = threadIdx.x / kT;
  const int64_t r0 = (int64_t)blockIdx.y * kT, c0 = (int64_t)blockIdx.x * kT;       // rows of theta (in), columns (out)
#pragma unroll
  for (int k = 0; k < kT; k += 8) {
    const int64_t r = r0 + ty + k, c = c0 + tx;
    tile[ty + k][tx] = (r < n && c < m) ? __ldg(theta + r * m + c) : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kT; k += 8) {
    const int64_t c = c0 + ty + k, r = r0 + tx;                                     // output row c (out), column r (in)
    if (c < m && r < n) {
      const float v = tile[tx][ty + k];
      float h, l;
      tf32_split(v, h, l);
      t_hi[c * n + r] = h;
      t_lo[c * n + r] = l;
      tf32_split(v * v, h, l);
      sq_hi[c * n + r] = h;
      sq_lo[c * n + r] = l;
    }
  }
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" int lbbnn_vd_mc_epilogue(const float* E, int64_t e_sample_stride, const float* S, int64_t s_sample_stride,
                                    const float* alpha, int64_t batch, int64_t out_features, int n_samples,
                                    const lbbnn_noise* noise, uint64_t noise_group_stride, int flags, float* act, float* a_hi,
                                    float* a_lo, float* sq_hi, float* sq_lo, lbbnn_stream s) {
  LBBNN_REQUIRE(E && S && alpha && noise && batch > 0 && out_features > 0 && n_samples > 0, "bad argument");
  LBBNN_REQUIRE(e_sample_stride >= 0 && s_sample_stride >= 0, "negative sample stride");
  LBBNN_REQUIRE(act || a_hi || sq_hi, "no output requested");
  LBBNN_REQUIRE((a_hi == nullptr) == (a_lo == nullptr) && (sq_hi == nullptr) == (sq_lo == nullptr), "hi / lo outputs come in pairs");
  VdEpiArgs a;
  a.E = E; a.S = S; a.es = e_sample_stride; a.ss = s_sample_stride; a.alpha = alpha;
  a.B = batch; a.N = out_features; a.n_samples = n_samples; a.relu = (flags & LBBNN_FLAG_RELU) ? 1 : 0;
  a.noise = make_noise(noise); a.group_stride = noise_group_stride;
  a.act = act; a.a_hi = a_hi; a.a_lo = a_lo; a.sq_hi = sq_hi; a.sq_lo = sq_lo;
  const int64_t quads = ceil_div(batch * out_features, 4) * n_samples;
  vd_mc_epilogue_kernel<<<(unsigned)grid_for(quads), kThreads, 0, (cudaStream_t)s>>>(a);
  return check_launch("vd_mc_epilogue");
}

extern "C" int lbbnn_vd_tc_prepare(const float* theta, int64_t n, int64_t m, float* t_hi, float* t_lo, float* sq_hi, float* sq_lo,
                                   lbbnn_stream s) {
  LBBNN_REQUIRE(theta && t_hi && t_lo && sq_hi && sq_lo && n > 0 && m > 0, "bad argument");
  LBBNN_REQUIRE(ceil_div(n, kT) < 65536, "in_features %lld too large", (long long)n);
  dim3 grid((unsigned)ceil_div(m, kT), (unsigned)ceil_div(n, kT));
  vd_tc_prepare_kernel<<<grid, kT * 8, 0, (cudaStream_t)s>>>(theta, n, m, t_hi, t_lo, sq_hi, sq_lo);
  return check_launch("vd_tc_prepare");
}
