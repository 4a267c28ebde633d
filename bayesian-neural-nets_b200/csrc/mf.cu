// Mean-field (full weight sampling) path: LBBNN-GP-MF.py:74-255 (sim-study variant MFsim:173-244).
//
//   mf_gamma      gamma.rsample(): hard Bernoulli mask [u < alpha] (MF:113) or the relaxed-Bernoulli
//                 reparameterisation at temperature T (MF:115), and its backward to lambda
//   mf_sample     w = gamma (mu + sigma eps)  (MF:232-233; medimean / joint-mean variants MF:237-242) and,
//                 in the same pass over the weights, the five element sums that the log-prior and
//                 log-variational-posterior are built from (MF:247-251):
//                   s0 = sum g            (GaussGamma: multiplies the (a,b,tau) constant, MF:148)
//                   s1 = sum w^2          (GaussGamma: -tau w^2)
//                   s2 = sum lgamma(1+pb-g) - lgamma(2-g)      (BetaBinomial, MF:167-173; the other seven
//                                          lgamma terms do not depend on the element or cancel)
//                   s3 = sum log(gamma N(w; mu, sigma) + (1-gamma) + 1e-8)     (full_log_prob, MF:99-101)
//                   s4 = sum g log(alpha+1e-8) + (1-g) log(1-alpha+1e-8)      (Bernoulli.log_prob, MF:122-128)
//   mf_sample_bwd autograd of the above: (dL/dw, dL/ds0..4) -> dmu, drho, dlambda, dgamma, dpb
// All vectorised (float4) and coalesced; reductions are two-stage with a fixed order (deterministic).
#include "mf_math.cuh"

#include <cstdlib>

namespace lbbnn {
namespace {

constexpr int kThreads = 256;
constexpr int kLpWidthDefault = 2;   // see lp_width(): same-box A/B 0.2734 (4) / 0.2641 (2) / 0.2644 (1) ms per MF step

__device__ __forceinline__ void ldq(const float* __restrict__ p, int64_t e0, int64_t n, bool vec, float out[4]) {
  if (vec && e0 + 3 < n) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p + e0));
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = (e0 + j < n) ? __ldg(p + e0 + j) : 0.f;
  }
}
__device__ __forceinline__ void stq(float* __restrict__ p, int64_t e0, int64_t n, bool vec, const float v[4]) {
  if (vec && e0 + 3 < n) {
    *reinterpret_cast<float4*>(p + e0) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < n) p[e0 + j] = v[j];
  }
}

// W consecutive elements per thread (W = 4: one Philox group per thread; 2 / 1: two / four threads share a group and each
// recomputes it -- more warps in flight for the latency-bound log-probability kernels, ncu: 24 % warps active at W = 4)
template <int W>
__device__ __forceinline__ void ldw(const float* __restrict__ p, int64_t e0, int64_t n, bool vec, float (&out)[W]) {
  if constexpr (W == 4) {
    ldq(p, e0, n, vec, out);
  } else if constexpr (W == 2) {
    if (vec && e0 + 1 < n) {
      const float2 v = __ldg(reinterpret_cast<const float2*>(p + e0));
      out[0] = v.x; out[1] = v.y;
    } else {
      out[0] = e0 < n ? __ldg(p + e0) : 0.f;
      out[1] = e0 + 1 < n ? __ldg(p + e0 + 1) : 0.f;
    }
  } else {
    out[0] = e0 < n ? __ldg(p + e0) : 0.f;
  }
}
template <int W>
__device__ __forceinline__ void stw(float* __restrict__ p, int64_t e0, int64_t n, bool vec, const float (&v)[W]) {
  if constexpr (W == 4) {
    stq(p, e0, n, vec, v);
  } else if constexpr (W == 2) {
    if (vec && e0 + 1 < n) {
      *reinterpret_cast<float2*>(p + e0) = make_float2(v[0], v[1]);
    } else {
      if (e0 < n) p[e0] = v[0];
      if (e0 + 1 < n) p[e0 + 1] = v[1];
    }
  } else {
    if (e0 < n) p[e0] = v[0];
  }
}
// this thread's W values of a Philox group of four (sub = first element's position in the group)
template <int W>
__device__ __forceinline__ void pickw(const float (&g4)[4], int sub, float (&out)[W]) {
  if constexpr (W == 4) {
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = g4[j];
  } else if constexpr (W == 2) {
    out[0] = sub ? g4[2] : g4[0];
    out[1] = sub ? g4[3] : g4[1];
  } else {
    out[0] = sub == 0 ? g4[0] : (sub == 1 ? g4[1] : (sub == 2 ? g4[2] : g4[3]));
  }
}

// ---- gamma.rsample ----------------------------------------------------------------------------------
struct GammaArgs {
  const float *lam, *alpha_in;  // one of them: alpha = sigmoid(lam) or the given tensor
  Noise u;
  int64_t n;
  int exact;
  float inv_t;
  float* gamma;
};

__global__ void __launch_bounds__(kThreads) mf_gamma_kernel(const GammaArgs a) {
  Noise nz = a.u;
  nz.resolve();
  const float* src = a.lam ? a.lam : a.alpha_in;
  const bool vec = (a.n % 4 == 0) && aligned16(src) && aligned16(a.gamma) && (nz.ptr == nullptr || aligned16(nz.ptr));
  const int64_t nq = ceil_div(a.n, 4);
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = q * 4;
    float s[4], u[4], g[4];
    ldq(src, e0, a.n, vec, s);
    if (nz.ptr) ldq(nz.ptr, e0, a.n, vec, u);
    else philox_uniform4(nz.seed, nz.stream, (uint64_t)q, u);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float al = a.lam ? alpha_of(s[j]) : s[j];
      g[j] = a.exact ? (u[j] < al ? 1.0f : 0.0f) : relaxed_bernoulli(al, u[j], a.inv_t);
    }
    stq(a.gamma, e0, a.n, vec, g);
  }
}

// d gamma / d lambda for the relaxed draw: gamma(1-gamma)/T * (1/p + 1/(1-p)) * alpha(1-alpha), zero where clipped
__global__ void __launch_bounds__(kThreads) mf_gamma_bwd_kernel(const float* __restrict__ lam, const float* __restrict__ alpha_in,
                                                                const float* __restrict__ gamma, const float* __restrict__ dgamma,
                                                                int64_t n, float inv_t, float* __restrict__ dout) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float al = lam ? alpha_of(lam[i]) : alpha_in[i];
    dout[i] = relaxed_bernoulli_bwd(dgamma[i], gamma[i], al, inv_t, lam != nullptr);
  }
}

// ---- weight sampling + log-prob sums ------------------------------------------------------------------
// The last block to arrive sums the per-block partials [gridDim.x][width] in sum_partials_kernel's order (thread-strided, then
// block_sum) and returns true to thread 0 with the totals in out[]; every other block returns false.  The ticket is reset.
template <int WIDTH>
__device__ __forceinline__ bool last_block_totals(const double* __restrict__ part, unsigned int* ticket, double* red,
                                                  double (&out)[WIDTH]) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return false;
  __threadfence();
#pragma unroll
  for (int k = 0; k < WIDTH; ++k) {
    double acc = 0.0;
    for (unsigned i = threadIdx.x; i < gridDim.x; i += blockDim.x) acc += __ldcg(part + (int64_t)i * WIDTH + k);
    out[k] = block_sum(acc, red);
  }
  if (threadIdx.x == 0) *ticket = 0u;
  return threadIdx.x == 0;
}

struct SampleArgs {
  const float *mu, *rho, *lam, *gamma, *alpha_stale, *pb;
  Noise eps;
  int64_t n;
  int mode;        // LBBNN_MF_SAMPLE / MEDIMEAN / JOINTMEAN
  int want_lp;     // compute the five sums
  int lp_on_ws;    // sim-study: log-probs at the unmasked ws
  int exact_b, exact_wp, exact_gp;   // round(gamma.detach()) inside Bernoulli / GaussGamma / BetaBinomial log_prob
  float* w;
  double* part;    // [gridDim.x][5]
  // optional: the last block to arrive (ticket) closes the five sums itself -- same order as sum_partials_kernel -- instead of
  // a second launch; the ticket is zero on entry and is left zero
  unsigned int* ticket;
  float* sums;
  // optional, for the Monte-Carlo predictive loop: draw the hard mask inside ([u < alpha], no gamma tensor)
  int native_gamma;
  Noise gu;
  // optional: sample the bias vector in the same launch (block 0): bias = b_mu + sigma_b eps_b  (MF:234)
  const float *bias_mu, *bias_rho;
  Noise eb;
  int64_t n_bias;
  float* bias_out;
};

template <int W>
__global__ void __launch_bounds__(kThreads) mf_sample_kernel(const SampleArgs a) {
  __shared__ double red[32];
  Noise nz = a.eps, gu = a.gu;
  nz.resolve();
  gu.resolve();
  if (a.bias_out && blockIdx.x == 0) {
    Noise eb = a.eb;
    eb.resolve();
    for (int64_t i = threadIdx.x; i < a.n_bias; i += blockDim.x) {
      const float e = eb.ptr ? eb.ptr[i] : philox_normal1(eb.seed, eb.stream, (uint64_t)i);
      a.bias_out[i] = fmaf(sigma_of(__ldg(a.bias_rho + i)), e, __ldg(a.bias_mu + i));
    }
  }
  const bool vec = (a.n % 4 == 0) && aligned16(a.mu) && aligned16(a.rho) && aligned16(a.lam) && aligned16(a.w) &&
                   (a.gamma == nullptr || aligned16(a.gamma)) && (a.alpha_stale == nullptr || aligned16(a.alpha_stale)) &&
                   (nz.ptr == nullptr || aligned16(nz.ptr));
  const float pb = a.want_lp ? __ldg(a.pb) : 1.0f;
  const int64_t nth = ceil_div(a.n, (int64_t)W);
  float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nth; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = t * W;
    const uint64_t q = (uint64_t)(e0 >> 2);      // Philox group of the elements, as in the one-group-per-thread form
    const int sub = (int)(e0 & 3);
    float mu[W], rho[W], lam[W], ga[W], ep[W], w[W];
#pragma unroll
    for (int j = 0; j < W; ++j) ga[j] = ep[j] = rho[j] = lam[j] = 0.f;
    ldw<W>(a.mu, e0, a.n, vec, mu);
    if (a.mode == LBBNN_MF_SAMPLE || a.want_lp) ldw<W>(a.rho, e0, a.n, vec, rho);
    if (a.want_lp || a.native_gamma || (a.mode == LBBNN_MF_JOINTMEAN && a.alpha_stale == nullptr)) ldw<W>(a.lam, e0, a.n, vec, lam);
    if (a.mode == LBBNN_MF_JOINTMEAN) {
      if (a.alpha_stale) ldw<W>(a.alpha_stale, e0, a.n, vec, ga);
    } else if (a.native_gamma) {
      float u4[4], u[W];
      philox_uniform4(gu.seed, gu.stream, q, u4);
      pickw<W>(u4, sub, u);
#pragma unroll
      for (int j = 0; j < W; ++j) ga[j] = u[j] < alpha_of(lam[j]) ? 1.0f : 0.0f;
    } else {
      ldw<W>(a.gamma, e0, a.n, vec, ga);
    }
    if (a.mode == LBBNN_MF_SAMPLE) {
      if (nz.ptr) {
        ldw<W>(nz.ptr, e0, a.n, vec, ep);
      } else {
        float n4[4];
        philox_normal4(nz.seed, nz.stream, q, n4);
        pickw<W>(n4, sub, ep);
      }
    }
#pragma unroll
    for (int j = 0; j < W; ++j) {
      w[j] = 0.f;
      if (e0 + j >= a.n) continue;
      float ws = mu[j];
      float sg = 0.f;
      if (a.mode == LBBNN_MF_SAMPLE) { sg = sigma_of(rho[j]); ws = fmaf(sg, ep[j], mu[j]); }
      float g = ga[j];
      if (a.mode == LBBNN_MF_JOINTMEAN && a.alpha_stale == nullptr) g = alpha_of(lam[j]);
      w[j] = g * ws;
      if (a.want_lp) {
        if (a.mode != LBBNN_MF_SAMPLE) sg = sigma_of(rho[j]);
        const float al = alpha_of(lam[j]);
        mf_lp_terms(g, a.lp_on_ws ? ws : w[j], mu[j], sg, al, pb, a.exact_b, a.exact_wp, a.exact_gp, s);
      }
    }
    stw<W>(a.w, e0, a.n, vec, w);
  }
  if (a.want_lp) {
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const double t = block_sum((double)s[k], red);
      if (threadIdx.x == 0) a.part[(int64_t)blockIdx.x * 5 + k] = t;
    }
    if (a.ticket) {
      double tot[5];
      if (last_block_totals<5>(a.part, a.ticket, red, tot)) {
#pragma unroll
        for (int k = 0; k < 5; ++k) a.sums[k] = (float)tot[k];
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads) sum_partials_kernel(const double* __restrict__ part, int nblocks, int width,
                                                                float* __restrict__ out) {
  __shared__ double red[32];
  for (int k = 0; k < width; ++k) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += blockDim.x) acc += part[(int64_t)i * width + k];
    const double t = block_sum(acc, red);
    if (threadIdx.x == 0) out[k] = (float)t;
  }
}

struct SampleBwdArgs {
  const float *mu, *rho, *lam, *gamma, *pb, *dw, *c;   // c: dL/ds0..4 (device, 5 floats)
  Noise eps;
  int64_t n;
  int lp_on_ws, exact_b, exact_wp, exact_gp, want_dgamma;
  float *dmu, *drho, *dlam, *dgamma;
  double* part;   // [gridDim.x][1]: sum psi(1+pb-g) (for dpb)
  unsigned int* ticket;   // optional, as in SampleArgs: the last block writes dpb = c[2] * sum of the partials
  float* dpb;
};


template <int W>
__global__ void __launch_bounds__(kThreads) mf_sample_bwd_kernel(const SampleBwdArgs a) {
  __shared__ double red[32];
  Noise nz = a.eps;
  nz.resolve();
  const bool vec = (a.n % 4 == 0) && aligned16(a.mu) && aligned16(a.rho) && aligned16(a.lam) && aligned16(a.gamma) &&
                   (a.dw == nullptr || aligned16(a.dw)) && aligned16(a.dmu) && aligned16(a.drho) && aligned16(a.dlam) &&
                   (a.dgamma == nullptr || aligned16(a.dgamma)) && (nz.ptr == nullptr || aligned16(nz.ptr));
  float c[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  if (a.c) {
#pragma unroll
    for (int k = 0; k < 5; ++k) c[k] = __ldg(a.c + k);
  }
  const float pb = __ldg(a.pb);
  const int64_t nth = ceil_div(a.n, (int64_t)W);
  float psisum = 0.f;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nth; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = t * W;
    const uint64_t q = (uint64_t)(e0 >> 2);
    const int sub = (int)(e0 & 3);
    float mu[W], rho[W], lam[W], ga[W], ep[W], dw[W], gm[W], gr[W], gl[W], gg[W];
#pragma unroll
    for (int j = 0; j < W; ++j) dw[j] = 0.f;
    ldw<W>(a.mu, e0, a.n, vec, mu);
    ldw<W>(a.rho, e0, a.n, vec, rho);
    ldw<W>(a.lam, e0, a.n, vec, lam);
    ldw<W>(a.gamma, e0, a.n, vec, ga);
    if (a.dw) ldw<W>(a.dw, e0, a.n, vec, dw);
    if (nz.ptr) {
      ldw<W>(nz.ptr, e0, a.n, vec, ep);
    } else {
      float n4[4];
      philox_normal4(nz.seed, nz.stream, q, n4);
      pickw<W>(n4, sub, ep);
    }
#pragma unroll
    for (int j = 0; j < W; ++j) {
      gm[j] = gr[j] = gl[j] = gg[j] = 0.f;
      if (e0 + j >= a.n) continue;
      const MfElemGrad e = mf_lp_terms_bwd(c, mu[j], rho[j], lam[j], ga[j], ep[j], dw[j], pb, a.lp_on_ws, a.exact_b,
                                           a.exact_wp, a.exact_gp);
      psisum += e.psi;
      gm[j] = e.dmu;
      gr[j] = e.drho;
      gl[j] = e.dlam;
      gg[j] = e.dgamma;
    }
    stw<W>(a.dmu, e0, a.n, vec, gm);
    stw<W>(a.drho, e0, a.n, vec, gr);
    stw<W>(a.dlam, e0, a.n, vec, gl);
    if (a.want_dgamma) stw<W>(a.dgamma, e0, a.n, vec, gg);
  }
  const double t = block_sum((double)psisum, red);
  if (threadIdx.x == 0) a.part[blockIdx.x] = t;
  if (a.ticket) {
    double tot[1];
    if (last_block_totals<1>(a.part, a.ticket, red, tot)) *a.dpb = (float)tot[0] * (a.c ? a.c[2] : 0.f);   // = sum_partials + scale_scalar
  }
}

// Monte-Carlo predictive accumulators (test_ensemble, MF:367-406): per input row add log_softmax(logits) and
// the row-normalised expit(log_softmax) of this weight sample; fp64 so the result does not depend on how the
// samples are split across GPUs.  One warp per row; also bumps the sample counter (Philox stream key).
__global__ void __launch_bounds__(kThreads) mc_accumulate_kernel(const float* __restrict__ logits, int64_t B, int64_t C,
                                                                 double* __restrict__ sum_logp, double* __restrict__ sum_prob,
                                                                 int64_t* counter) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  if (b < B) {
    const float* row = logits + b * C;
    float mx = -INFINITY;
    for (int64_t c = lane; c < C; c += 32) mx = fmaxf(mx, row[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.f;
    for (int64_t c = lane; c < C; c += 32) se += expf(row[c] - mx);
    se = warp_sum(se);
    const float lse = mx + logf(se);
    float ps = 0.f;
    for (int64_t c = lane; c < C; c += 32) ps += 1.0f / (1.0f + expf(-(row[c] - lse)));
    ps = warp_sum(ps);
    for (int64_t c = lane; c < C; c += 32) {
      const float lp = row[c] - lse;
      sum_logp[b * C + c] += (double)lp;
      sum_prob[b * C + c] += (double)((1.0f / (1.0f + expf(-lp))) / ps);
    }
  }
  if (counter && blockIdx.x == 0 && threadIdx.x == 0) *counter += 1;
}

__global__ void scale_scalar_kernel(float* v, const float* c, int k) { *v *= c ? c[k] : 0.f; }

int64_t ew_blocks(int64_t n) {
  int64_t b = ceil_div(ceil_div(n, 4), kThreads);
  const int64_t cap = 8LL * sm_count();
  return b < 1 ? 1 : (b > cap ? cap : b);
}
// weights per thread of the log-probability kernels (mf_sample with log-probs, mf_sample_bwd): LBBNN_MF_SPLIT = 4 | 2 | 1
int lp_width() {
  static int w = 0;
  if (!w) {
    const char* e = getenv("LBBNN_MF_SPLIT");
    const int v = e ? atoi(e) : kLpWidthDefault;
    w = (v == 1 || v == 2 || v == 4) ? v : kLpWidthDefault;
  }
  return w;
}
int64_t lp_blocks(int64_t n, int width) {
  int64_t b = ceil_div(ceil_div(n, (int64_t)width), kThreads);
  const int64_t cap = 8LL * sm_count();
  return b < 1 ? 1 : (b > cap ? cap : b);
}

// ---- the scalar tail of the MF layer's log-probabilities (MF:148-150, 167-173, 246-251) as one forward and one backward kernel ----
// Given the five sums s[0..4] of lbbnn_mf_sample_fwd, the Gamma draws tau_w (1) and tau_b (out) and the hyper-parameters:
//   bias      = bias_mu + sigma_b eps_b                  (sample branch; bias_mu otherwise)
//   c_w       = a log b + (a - 1/2) tau_w - b tau_w - lgamma(a) - log sqrt(2 pi)
//   log_prior = [s0 c_w - tau_w s1 + (n - s0) + n 1e-8]                                        GaussGamma on the weights
//             + sum_i [ba_i log bb_i + (ba_i - 1/2) tau_b_i - bb_i tau_b_i - lgamma(ba_i) - log sqrt(2 pi) - tau_b_i bias_i^2 + 1e-8]
//             + s2 + n (lgamma(pa + pb) - lgamma(1 + pa + pb) - lgamma(pa) - lgamma(pb))        BetaBinomial
//   log_q     = s3 + s4 + sum_i [-log sqrt(2 pi) - log sigma_b_i - (bias_i - bias_mu_i)^2 / (2 sigma_b_i^2)]
// (the reference's own expressions, term for term: ~70 elementwise / reduction launches per layer forward and ~140 backward
// in the eager formulation, on (1,) and (out,) tensors).  One block: out <= a few thousand.
struct PriorArgs {
  const float *s, *a, *b, *tau_w, *pa, *pb;                 // (5), (1) each
  const float *ba, *bb, *tau_b, *bias_mu, *bias_rho;        // (out) each
  Noise eps;                                                // eps_b: injected (out) or Philox
  int out, sample;                                          // sample: bias is drawn (training / sample=True)
  float n;                                                  // number of weights
  float *bias, *eps_out;                                    // (out) each; eps_out keeps the draw for the backward
  float* lp;                                                // [log_prior, log_q]
};

__global__ void __launch_bounds__(kThreads) mf_prior_fwd_kernel(PriorArgs a) {
  __shared__ float red[32];
  a.eps.resolve();
  float gb = 0.f, lq = 0.f;
  for (int i = threadIdx.x; i < a.out; i += kThreads) {
    const float mu = __ldg(a.bias_mu + i), sb = sigma_of(__ldg(a.bias_rho + i));
    float e = 0.f;
    if (a.sample) e = a.eps.ptr ? __ldg(a.eps.ptr + i) : philox_normal1(a.eps.seed, a.eps.stream, (uint64_t)i);
    const float bias = a.sample ? mu + sb * e : mu;
    a.bias[i] = bias;
    a.eps_out[i] = e;
    mf_bias_lp_terms(bias, mu, sb, __ldg(a.ba + i), __ldg(a.bb + i), __ldg(a.tau_b + i), gb, lq);
  }
  gb = block_sum(gb, red);
  lq = block_sum(lq, red);
  if (threadIdx.x == 0) {
    a.lp[0] = mf_log_prior(a.s, gb, a.a[0], a.b[0], a.tau_w[0], a.pa[0], a.pb[0], a.n);
    a.lp[1] = a.s[3] + a.s[4] + lq;
  }
}

struct PriorBwdArgs {
  const float *s, *a, *b, *tau_w, *pa, *pb, *ba, *bb, *tau_b, *bias_mu, *bias_rho, *bias, *eps;
  const float *g_lp, *g_lq, *g_bias;                        // d loss / d log_prior, d log_q (device scalars), d bias (out) or NULL
  int out, sample;
  float n;
  float* d_scalar;                                          // [ds0..ds4, da, db, dtau_w, dpa, dpb]
  float *d_ba, *d_bb, *d_tau_b, *d_bias_mu, *d_bias_rho;    // (out) each
  // optional: the precisions were drawn outside autograd as tau = g / b; their partial derivatives wrt (a, b) -- (1,) for the
  // weights' tau, (out) for the biases' -- fold the gradient that reaches tau into da, db here
  const float *tw_da, *tw_db, *tb_da, *tb_db;
};

__global__ void __launch_bounds__(kThreads) mf_prior_bwd_kernel(const PriorBwdArgs a) {
  const float gp = a.g_lp ? __ldg(a.g_lp) : 0.f, gq = a.g_lq ? __ldg(a.g_lq) : 0.f;
  for (int i = threadIdx.x; i < a.out; i += kThreads) {
    const MfBiasGrad g = mf_bias_lp_terms_bwd(gp, gq, a.g_bias ? __ldg(a.g_bias + i) : 0.f, __ldg(a.bias_mu + i),
                                              __ldg(a.bias_rho + i), __ldg(a.bias + i), __ldg(a.eps + i), __ldg(a.ba + i),
                                              __ldg(a.bb + i), __ldg(a.tau_b + i), a.sample, a.tb_da != nullptr,
                                              a.tb_da ? __ldg(a.tb_da + i) : 0.f, a.tb_da ? __ldg(a.tb_db + i) : 0.f);
    a.d_ba[i] = g.dba;
    a.d_bb[i] = g.dbb;
    a.d_tau_b[i] = g.dtb;
    a.d_bias_mu[i] = g.dmu;
    a.d_bias_rho[i] = g.drho;
  }
  if (threadIdx.x == 0) {
    mf_log_prior_bwd(gp, gq, a.s[0], a.s[1], a.a[0], a.b[0], a.tau_w[0], a.pa[0], a.pb[0], a.n, a.tw_da != nullptr,
                     a.tw_da ? a.tw_da[0] : 0.f, a.tw_da ? a.tw_db[0] : 0.f, a.d_scalar);
  }
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" size_t lbbnn_mf_workspace_bytes(int64_t n) { return n > 0 ? (size_t)lp_blocks(n, 1) * 5 * sizeof(double) + 256 : 0; }

extern "C" int lbbnn_mf_gamma_sample(const float* lambdal, const float* alpha, int64_t n, const lbbnn_noise* u, int exact,
                                     float temperature, float* gamma, lbbnn_stream s) {
  LBBNN_REQUIRE((lambdal != nullptr) != (alpha != nullptr), "give exactly one of lambdal / alpha");
  LBBNN_REQUIRE(gamma && n > 0 && temperature > 0.f, "bad argument");
  GammaArgs a;
  a.lam = lambdal; a.alpha_in = alpha; a.u = make_noise(u); a.n = n; a.exact = exact; a.inv_t = 1.0f / temperature; a.gamma = gamma;
  mf_gamma_kernel<<<(unsigned)ew_blocks(n), kThreads, 0, (cudaStream_t)s>>>(a);
  return check_launch("mf_gamma");
}

extern "C" int lbbnn_mf_gamma_sample_bwd(const float* lambdal, const float* alpha, const float* gamma, const float* dgamma,
                                         int64_t n, float temperature, float* dout, lbbnn_stream s) {
  LBBNN_REQUIRE((lambdal != nullptr) != (alpha != nullptr), "give exactly one of lambdal / alpha");
  LBBNN_REQUIRE(gamma && dgamma && dout && n > 0, "bad argument");
  int64_t blocks = ceil_div(n, kThreads);
  if (blocks > 8LL * sm_count()) blocks = 8LL * sm_count();
  mf_gamma_bwd_kernel<<<(unsigned)blocks, kThreads, 0, (cudaStream_t)s>>>(lambdal, alpha, gamma, dgamma, n, 1.0f / temperature, dout);
  return check_launch("mf_gamma_bwd");
}

static int mf_sample_launch(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                            const float* alpha_stale, const float* pb, int64_t n, const lbbnn_noise* eps, int mode, int flags,
                            float* w, float* sums, void* ws, size_t ws_bytes, const lbbnn_noise* gamma_u,
                            const float* bias_mu, const float* bias_rho, const lbbnn_noise* eps_b, int64_t n_bias,
                            float* bias_out, lbbnn_stream s, unsigned int* ticket = nullptr) {
  LBBNN_REQUIRE(mu && rho && lambdal && w && n > 0, "NULL argument");
  LBBNN_REQUIRE(mode == LBBNN_MF_JOINTMEAN || gamma || gamma_u, "gamma (tensor or native draw) required");
  LBBNN_REQUIRE(!bias_out || (bias_mu && bias_rho && n_bias > 0), "bias sampling needs bias_mu/bias_rho");
  const bool lp = flags & LBBNN_MF_FLAG_LOGPROBS;
  LBBNN_REQUIRE(!lp || (sums && pb && ws && ws_bytes >= lbbnn_mf_workspace_bytes(n)), "log-probs need sums, pb and workspace");
  SampleArgs a;
  a.mu = mu; a.rho = rho; a.lam = lambdal; a.gamma = gamma; a.alpha_stale = alpha_stale; a.pb = pb;
  a.eps = make_noise(eps); a.n = n; a.mode = mode; a.want_lp = lp ? 1 : 0;
  a.lp_on_ws = (flags & LBBNN_MF_FLAG_LP_ON_WS) ? 1 : 0;
  a.exact_b = (flags & LBBNN_MF_FLAG_EXACT_GAMMA) ? 1 : 0;
  a.exact_wp = (flags & LBBNN_MF_FLAG_EXACT_WPRIOR) ? 1 : 0;
  a.exact_gp = (flags & LBBNN_MF_FLAG_EXACT_GPRIOR) ? 1 : 0;
  a.w = w; a.part = (double*)ws;
  a.native_gamma = (gamma == nullptr && gamma_u != nullptr && mode != LBBNN_MF_JOINTMEAN) ? 1 : 0;
  a.gu = make_noise(gamma_u);
  a.bias_mu = bias_mu; a.bias_rho = bias_rho; a.eb = make_noise(eps_b); a.n_bias = n_bias; a.bias_out = bias_out;
  a.ticket = lp ? ticket : nullptr; a.sums = sums;
  const int width = lp ? lp_width() : 4;        // without log-probs the kernel is a light elementwise pass: one group per thread
  const unsigned blocks = (unsigned)lp_blocks(n, width);
  if (width == 1) mf_sample_kernel<1><<<blocks, kThreads, 0, (cudaStream_t)s>>>(a);
  else if (width == 2) mf_sample_kernel<2><<<blocks, kThreads, 0, (cudaStream_t)s>>>(a);
  else mf_sample_kernel<4><<<blocks, kThreads, 0, (cudaStream_t)s>>>(a);
  if (int rc = check_launch("mf_sample")) return rc;
  if (lp && !ticket) {
    sum_partials_kernel<<<1, kThreads, 0, (cudaStream_t)s>>>((const double*)ws, (int)blocks, 5, sums);
    return check_launch("mf_sum_partials");
  }
  return LBBNN_OK;
}

extern "C" int lbbnn_mf_sample_fwd(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                                   const float* alpha_stale, const float* pb, int64_t n, const lbbnn_noise* eps, int mode,
                                   int flags, float* w, float* sums, void* ws, size_t ws_bytes, lbbnn_stream s) {
  return mf_sample_launch(mu, rho, lambdal, gamma, alpha_stale, pb, n, eps, mode, flags, w, sums, ws, ws_bytes, nullptr,
                          nullptr, nullptr, nullptr, 0, nullptr, s);
}

extern "C" int lbbnn_mf_sample_fwd_ticket(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                                          const float* alpha_stale, const float* pb, int64_t n, const lbbnn_noise* eps, int mode,
                                          int flags, float* w, float* sums, void* ws, size_t ws_bytes, unsigned int* ticket,
                                          lbbnn_stream s) {
  LBBNN_REQUIRE(ticket, "NULL ticket");
  return mf_sample_launch(mu, rho, lambdal, gamma, alpha_stale, pb, n, eps, mode, flags, w, sums, ws, ws_bytes, nullptr,
                          nullptr, nullptr, nullptr, 0, nullptr, s, ticket);
}

// one launch per layer of the Monte-Carlo predictive loop: hard mask drawn natively, weights and bias sampled
extern "C" int lbbnn_mf_sample_predict(const lbbnn_layer* L, const lbbnn_noise* gamma_u, const lbbnn_noise* eps_w,
                                       const lbbnn_noise* eps_b, float* w, float* bias, lbbnn_stream s) {
  LBBNN_REQUIRE(L && gamma_u && w && bias, "NULL argument");
  return mf_sample_launch(L->weight_mu, L->weight_rho, L->lambdal, nullptr, nullptr, nullptr, L->in_features * L->out_features,
                          eps_w, LBBNN_MF_SAMPLE, 0, w, nullptr, nullptr, 0, gamma_u, L->bias_mu, L->bias_rho, eps_b,
                          L->out_features, bias, s);
}

extern "C" int lbbnn_mc_accumulate(const float* logits, int64_t batch, int64_t classes, double* sum_logp, double* sum_prob,
                                   int64_t* counter, lbbnn_stream s) {
  LBBNN_REQUIRE(logits && sum_logp && sum_prob && batch > 0 && classes > 0, "NULL argument");
  mc_accumulate_kernel<<<(unsigned)ceil_div(batch, kThreads / 32), kThreads, 0, (cudaStream_t)s>>>(logits, batch, classes,
                                                                                                 sum_logp, sum_prob, counter);
  return check_launch("mc_accumulate");
}

extern "C" int lbbnn_mf_sample_bwd(const float* mu, const float* rho, const float* lambdal, const float* gamma, const float* pb,
                                   int64_t n, const lbbnn_noise* eps, int flags, const float* dw, const float* dsums,
                                   float* dmu, float* drho, float* dlambdal, float* dgamma, float* dpb, void* ws,
                                   size_t ws_bytes, lbbnn_stream s) {
  return lbbnn_mf_sample_bwd_ticket(mu, rho, lambdal, gamma, pb, n, eps, flags, dw, dsums, dmu, drho, dlambdal, dgamma, dpb, ws,
                                    ws_bytes, nullptr, s);
}

extern "C" int lbbnn_mf_sample_bwd_ticket(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                                          const float* pb, int64_t n, const lbbnn_noise* eps, int flags, const float* dw,
                                          const float* dsums, float* dmu, float* drho, float* dlambdal, float* dgamma, float* dpb,
                                          void* ws, size_t ws_bytes, unsigned int* ticket, lbbnn_stream s) {
  LBBNN_REQUIRE(mu && rho && lambdal && gamma && pb && dmu && drho && dlambdal && dpb && n > 0, "NULL argument");
  LBBNN_REQUIRE(ws && ws_bytes >= lbbnn_mf_workspace_bytes(n), "workspace too small");
  SampleBwdArgs a;
  a.mu = mu; a.rho = rho; a.lam = lambdal; a.gamma = gamma; a.pb = pb; a.dw = dw; a.c = dsums;
  a.eps = make_noise(eps); a.n = n;
  a.lp_on_ws = (flags & LBBNN_MF_FLAG_LP_ON_WS) ? 1 : 0;
  a.exact_b = (flags & LBBNN_MF_FLAG_EXACT_GAMMA) ? 1 : 0;
  a.exact_wp = (flags & LBBNN_MF_FLAG_EXACT_WPRIOR) ? 1 : 0;
  a.exact_gp = (flags & LBBNN_MF_FLAG_EXACT_GPRIOR) ? 1 : 0;
  a.want_dgamma = dgamma ? 1 : 0;
  a.dmu = dmu; a.drho = drho; a.dlam = dlambdal; a.dgamma = dgamma; a.part = (double*)ws;
  a.ticket = ticket; a.dpb = dpb;
  const int width = lp_width();
  const unsigned blocks = (unsigned)lp_blocks(n, width);
  if (width == 1) mf_sample_bwd_kernel<1><<<blocks, kThreads, 0, (cudaStream_t)s>>>(a);
  else if (width == 2) mf_sample_bwd_kernel<2><<<blocks, kThreads, 0, (cudaStream_t)s>>>(a);
  else mf_sample_bwd_kernel<4><<<blocks, kThreads, 0, (cudaStream_t)s>>>(a);
  if (int rc = check_launch("mf_sample_bwd")) return rc;
  if (ticket) return LBBNN_OK;          // the last block has written dpb = dL/ds2 * sum psi(1+pb-g)
  sum_partials_kernel<<<1, kThreads, 0, (cudaStream_t)s>>>((const double*)ws, (int)blocks, 1, dpb);
  if (int rc = check_launch("mf_sum_partials")) return rc;
  scale_scalar_kernel<<<1, 1, 0, (cudaStream_t)s>>>(dpb, dsums, 2);   // dpb = dL/ds2 * sum psi(1+pb-g)
  return check_launch("mf_scale");
}

extern "C" int lbbnn_mf_prior_fwd(const float* sums5, const float* a, const float* b, const float* tau_w, const float* pa,
                                  const float* pb, const float* bias_a, const float* bias_b, const float* tau_b,
                                  const float* bias_mu, const float* bias_rho, const lbbnn_noise* eps_b, int sample_bias,
                                  int64_t out_features, double n_weights, float* bias, float* eps_out, float* logprobs2,
                                  lbbnn_stream s) {
  LBBNN_REQUIRE(sums5 && a && b && tau_w && pa && pb && bias_a && bias_b && tau_b && bias_mu && bias_rho && bias && eps_out &&
                    logprobs2, "NULL argument");
  LBBNN_REQUIRE(out_features > 0 && out_features < (1LL << 24), "bad shape");
  LBBNN_REQUIRE(!sample_bias || eps_b, "the sampled bias needs its noise source");
  PriorArgs p;
  p.s = sums5; p.a = a; p.b = b; p.tau_w = tau_w; p.pa = pa; p.pb = pb; p.ba = bias_a; p.bb = bias_b; p.tau_b = tau_b;
  p.bias_mu = bias_mu; p.bias_rho = bias_rho; p.eps = make_noise(eps_b); p.out = (int)out_features; p.sample = sample_bias ? 1 : 0;
  p.n = (float)n_weights; p.bias = bias; p.eps_out = eps_out; p.lp = logprobs2;
  mf_prior_fwd_kernel<<<1, kThreads, 0, (cudaStream_t)s>>>(p);
  return check_launch("mf_prior_fwd");
}

extern "C" int lbbnn_mf_prior_bwd(const float* sums5, const float* a, const float* b, const float* tau_w, const float* pa,
                                  const float* pb, const float* bias_a, const float* bias_b, const float* tau_b,
                                  const float* bias_mu, const float* bias_rho, const float* bias, const float* eps,
                                  int sample_bias, int64_t out_features, double n_weights, const float* g_log_prior,
                                  const float* g_log_q, const float* g_bias, float* d_scalars10, float* d_bias_a, float* d_bias_b,
                                  float* d_tau_b, float* d_bias_mu, float* d_bias_rho, lbbnn_stream s) {
  return lbbnn_mf_prior_bwd_tau(sums5, a, b, tau_w, pa, pb, bias_a, bias_b, tau_b, bias_mu, bias_rho, bias, eps, sample_bias,
                                out_features, n_weights, g_log_prior, g_log_q, g_bias, nullptr, nullptr, nullptr, nullptr,
                                d_scalars10, d_bias_a, d_bias_b, d_tau_b, d_bias_mu, d_bias_rho, s);
}

extern "C" int lbbnn_mf_prior_bwd_tau(const float* sums5, const float* a, const float* b, const float* tau_w, const float* pa,
                                      const float* pb, const float* bias_a, const float* bias_b, const float* tau_b,
                                      const float* bias_mu, const float* bias_rho, const float* bias, const float* eps,
                                      int sample_bias, int64_t out_features, double n_weights, const float* g_log_prior,
                                      const float* g_log_q, const float* g_bias, const float* dtau_w_da, const float* dtau_w_db,
                                      const float* dtau_b_da, const float* dtau_b_db, float* d_scalars10, float* d_bias_a,
                                      float* d_bias_b, float* d_tau_b, float* d_bias_mu, float* d_bias_rho, lbbnn_stream s) {
  LBBNN_REQUIRE((dtau_w_da == nullptr) == (dtau_w_db == nullptr) && (dtau_b_da == nullptr) == (dtau_b_db == nullptr),
                "the derivative factors of a precision come in pairs");
  LBBNN_REQUIRE(sums5 && a && b && tau_w && pa && pb && bias_a && bias_b && tau_b && bias_mu && bias_rho && bias && eps,
                "NULL argument");
  LBBNN_REQUIRE(d_scalars10 && d_bias_a && d_bias_b && d_tau_b && d_bias_mu && d_bias_rho, "NULL output");
  LBBNN_REQUIRE(out_features > 0 && out_features < (1LL << 24), "bad shape");
  PriorBwdArgs p;
  p.s = sums5; p.a = a; p.b = b; p.tau_w = tau_w; p.pa = pa; p.pb = pb; p.ba = bias_a; p.bb = bias_b; p.tau_b = tau_b;
  p.bias_mu = bias_mu; p.bias_rho = bias_rho; p.bias = bias; p.eps = eps; p.g_lp = g_log_prior; p.g_lq = g_log_q; p.g_bias = g_bias;
  p.out = (int)out_features; p.sample = sample_bias ? 1 : 0; p.n = (float)n_weights;
  p.d_scalar = d_scalars10; p.d_ba = d_bias_a; p.d_bb = d_bias_b; p.d_tau_b = d_tau_b; p.d_bias_mu = d_bias_mu; p.d_bias_rho = d_bias_rho;
  p.tw_da = dtau_w_da; p.tw_db = dtau_w_db; p.tb_da = dtau_b_da; p.tb_db = dtau_b_db;
  mf_prior_bwd_kernel<<<1, kThreads, 0, (cudaStream_t)s>>>(p);
  return check_launch("mf_prior_bwd");
}
