// Elementwise halves of the LRT / MNF posterior-predictive loop (test_ensemble, LRT:239-265 / MNF:287-318) on the tensor cores.
//
// The LRT forward of a stacked batch of n MC samples splits into two plain linear layers, E = A_E M^T (M = alpha mu) and
// S = A_S V^T (V = alpha^2 sigma^2): M and V do not depend on the sample, so each is ONE 3xTF32 tensor-core GEMM of n * B
// rows (lbbnn_tc_linear_tf32x3, no bias).  The kernels here sit around those two calls:
//   lrt_mc_epilogue   act = E + b_mu + sqrt(S + sigma_b^2) eps_s [relu] (the fp32 forward epilogue, LRT:172-175) for the n
//                     samples, and the operands of the next tensor-core layer: hi / lo of act .* rowscale_s (its mean
//                     product; rowscale = the next MNF layer's z) and of act^2 (its variance product, squared in fp32)
//   tf32_split_rows   hi / lo of x .* rowscale_s and / or of x^2: the test input of layer 1, or the fp32 activations of a
//                     CUDA-core layer that feeds a tensor-core one
// Native noise is drawn exactly as lbbnn_lrt_f32_fwd_ex / lbbnn_lrt_sample_expand draw it (stream_id + s * group_stride,
// element row * out + col), so both paths see the same eps.
#include "mc_io.cuh"

namespace lbbnn {
namespace {

using namespace mc_io;

struct McEpiArgs {
  const float *E, *S;
  int64_t es, ss;              // per-sample strides of E / S in floats (0 = shared by all samples)
  const float *bias_mu, *bias_rho;
  int64_t B, N;
  int n_samples, sample, relu;
  Noise noise;
  uint64_t group_stride;
  float* act;                  // (n, B, N) or NULL
  const float* rowscale;       // (n, N) or NULL
  float *m_hi, *m_lo, *v_hi, *v_lo;
};

// One thread = four consecutive elements of one sample (flat index inside the sample: b * N + n).
__global__ void __launch_bounds__(kThreads) lrt_mc_epilogue_kernel(const McEpiArgs a) {
  Noise nz = a.noise;
  nz.resolve();
  const int64_t total = a.B * a.N, nq = ceil_div(total, 4);
  const bool vec = (total % 4 == 0) && aligned16(a.E) && a.es % 4 == 0 && (!a.sample || (aligned16(a.S) && a.ss % 4 == 0)) &&
                   (a.act == nullptr || aligned16(a.act)) && (nz.ptr == nullptr || aligned16(nz.ptr)) &&
                   (a.m_hi == nullptr || (aligned16(a.m_hi) && aligned16(a.m_lo))) &&
                   (a.v_hi == nullptr || (aligned16(a.v_hi) && aligned16(a.v_lo)));
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq * a.n_samples; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i / nq);
    const int64_t q = i - (int64_t)s * nq, e0 = q * 4, so = (int64_t)s * total;
    float v[4], sv[4], ep[4];
    load4(a.E + (int64_t)s * a.es, e0, total, vec, v);
    if (a.sample) {
      load4(a.S + (int64_t)s * a.ss, e0, total, vec, sv);
      if (nz.ptr) load4(nz.ptr + so, e0, total, vec, ep);
      else if (total % 4 == 0) philox_normal4(nz.seed, nz.stream + (uint64_t)s * a.group_stride, (uint64_t)q, ep);
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j) ep[j] = philox_normal1(nz.seed, nz.stream + (uint64_t)s * a.group_stride, (uint64_t)(e0 + j));
      }
    }
    float zr[4] = {1.f, 1.f, 1.f, 1.f};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t n = (e0 + j < total) ? (e0 + j) % a.N : 0;
      float o = v[j] + __ldg(a.bias_mu + n);
      if (a.sample) {                           // the fp32 forward epilogue's expressions (LRT:172-175)
        const float sb = sigma_of(__ldg(a.bias_rho + n));
        const float sd = sqrtf(sv[j] + sb * sb);
        o = fmaf(sd, ep[j], o);
      }
      v[j] = a.relu ? fmaxf(o, 0.f) : o;
      if (a.rowscale) zr[j] = __ldg(a.rowscale + (int64_t)s * a.N + n);
    }
    if (a.act) store4(a.act + so, e0, total, vec, v);
    if (a.m_hi) {
      float m[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) m[j] = a.rowscale ? v[j] * zr[j] : v[j];
      store_split4(a.m_hi + so, a.m_lo + so, e0, total, vec, m);
    }
    if (a.v_hi) {
      float sq[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) sq[j] = v[j] * v[j];
      store_split4(a.v_hi + so, a.v_lo + so, e0, total, vec, sq);
    }
  }
}

struct SplitRowsArgs {
  const float* x;
  int64_t xs, rows, cols;
  int n_samples;
  const float* rowscale;
  float *hi, *lo, *sq_hi, *sq_lo;
};

__global__ void __launch_bounds__(kThreads) tf32_split_rows_kernel(const SplitRowsArgs a) {
  const int64_t total = a.rows * a.cols, nq = ceil_div(total, 4);
  const bool vec = (total % 4 == 0) && aligned16(a.x) && a.xs % 4 == 0 && (a.hi == nullptr || (aligned16(a.hi) && aligned16(a.lo))) &&
                   (a.sq_hi == nullptr || (aligned16(a.sq_hi) && aligned16(a.sq_lo)));
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nq * a.n_samples; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i / nq);
    const int64_t e0 = (i - (int64_t)s * nq) * 4, so = (int64_t)s * total;
    float v[4];
    load4(a.x + (int64_t)s * a.xs, e0, total, vec, v);
    if (a.hi) {
      float m[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        m[j] = (a.rowscale && e0 + j < total) ? v[j] * __ldg(a.rowscale + (int64_t)s * a.cols + (e0 + j) % a.cols) : v[j];
      store_split4(a.hi + so, a.lo + so, e0, total, vec, m);
    }
    if (a.sq_hi) {
      float sq[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) sq[j] = v[j] * v[j];
      store_split4(a.sq_hi + so, a.sq_lo + so, e0, total, vec, sq);
    }
  }
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" int lbbnn_lrt_mc_epilogue(const float* E, int64_t e_sample_stride, const float* S, int64_t s_sample_stride,
                                     const float* bias_mu, const float* bias_rho, int64_t batch, int64_t out_features,
                                     int n_samples, const lbbnn_noise* noise, uint64_t noise_group_stride, int flags,
                                     float* act, const float* rowscale, float* m_hi, float* m_lo, float* v_hi, float* v_lo,
                                     lbbnn_stream s) {
  const bool sample = flags & LBBNN_FLAG_SAMPLE;
  LBBNN_REQUIRE(E && bias_mu && batch > 0 && out_features > 0 && n_samples > 0, "bad argument");
  LBBNN_REQUIRE(!sample || (S && bias_rho && noise), "the sample branch needs S, bias_rho and noise");
  LBBNN_REQUIRE(e_sample_stride >= 0 && s_sample_stride >= 0, "negative sample stride");
  LBBNN_REQUIRE(act || m_hi || v_hi, "no output requested");
  LBBNN_REQUIRE((m_hi == nullptr) == (m_lo == nullptr) && (v_hi == nullptr) == (v_lo == nullptr), "hi / lo outputs come in pairs");
  LBBNN_REQUIRE(rowscale == nullptr || m_hi, "rowscale scales the mean-product operand only");
  McEpiArgs a;
  a.E = E; a.S = S; a.es = e_sample_stride; a.ss = s_sample_stride; a.bias_mu = bias_mu; a.bias_rho = bias_rho;
  a.B = batch; a.N = out_features; a.n_samples = n_samples; a.sample = sample ? 1 : 0;
  a.relu = (flags & LBBNN_FLAG_RELU) ? 1 : 0;
  a.noise = make_noise(noise); a.group_stride = noise_group_stride;
  a.act = act; a.rowscale = rowscale; a.m_hi = m_hi; a.m_lo = m_lo; a.v_hi = v_hi; a.v_lo = v_lo;
  const int64_t quads = ceil_div(batch * out_features, 4) * n_samples;
  lrt_mc_epilogue_kernel<<<(unsigned)grid_for(quads), kThreads, 0, (cudaStream_t)s>>>(a);
  return check_launch("lrt_mc_epilogue");
}

extern "C" int lbbnn_tf32_split_rows(const float* x, int64_t x_sample_stride, int64_t rows, int64_t cols, int n_samples,
                                     const float* rowscale, float* hi, float* lo, float* sq_hi, float* sq_lo, lbbnn_stream s) {
  LBBNN_REQUIRE(x && rows > 0 && cols > 0 && n_samples > 0 && x_sample_stride >= 0, "bad argument");
  LBBNN_REQUIRE(hi || sq_hi, "no output requested");
  LBBNN_REQUIRE((hi == nullptr) == (lo == nullptr) && (sq_hi == nullptr) == (sq_lo == nullptr), "hi / lo outputs come in pairs");
  LBBNN_REQUIRE(rowscale == nullptr || hi, "rowscale scales the hi / lo output only");
  SplitRowsArgs a;
  a.x = x; a.xs = x_sample_stride; a.rows = rows; a.cols = cols; a.n_samples = n_samples; a.rowscale = rowscale;
  a.hi = hi; a.lo = lo; a.sq_hi = sq_hi; a.sq_lo = sq_lo;
  const int64_t quads = ceil_div(rows * cols, 4) * n_samples;
  tf32_split_rows_kernel<<<(unsigned)grid_for(quads), kThreads, 0, (cudaStream_t)s>>>(a);
  return check_launch("tf32_split_rows");
}
