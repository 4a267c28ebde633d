// The simulation study of LBBNN-GP-MFsim_study.py:344-429 in one launch: R independent repetitions of the 20 -> 1 mean-field
// logistic regression (SimStudyNetwork.sample_elbo, MFsim:272-300, SAMPLES = 1) trained with per-tensor SGD (MFsim:359-374)
// for any number of epochs.  The repetitions share nothing but read-only data, so each is one CTA that keeps its parameters in
// registers for the whole run: no grid barrier, no host round trip, no launch per step.
//
// Layout of a step (two __syncthreads):
//   A  warp 0, lane i = weight i (in <= 32): noise, gamma, w = gamma (mu + sigma eps), the five log-probability element terms
//      (warp sums), bias, both Gamma precisions and the log prior / log q scalars (every lane of warp 0 holds them)
//   B  all threads, one batch row at a time: logit = x w + bias, sigmoid, BCE and its gradient, dW / db / nll partials
//      in registers, then a fixed-order reduction (shuffle tree per warp, warps in order) through shared memory
//   C  warp 0: the backward of A through the shared per-element math (mf_math.cuh) and the SGD update
// 128 threads: a minibatch of the study has 400 rows of 20 features, ~3 rows per thread; more warps shorten B but lengthen the
// per-warp reduction and the barrier of every step, fewer leave B as the longest phase.
#include "mf_math.cuh"

namespace lbbnn {
namespace {

constexpr int kSimThreads = 128;
constexpr int kSimWarps = kSimThreads / 32;
constexpr int kSimMaxIn = LBBNN_MFSIM_MAX_IN;
constexpr int kGammaMaxAttempts = 64;

// Philox stream of one kind of draw of one step of one replica: replica < 2^24 in bits 40.., step < 2^36 in bits 4..39
enum { kDrawU = 0, kDrawEpsW = 1, kDrawEpsB = 2, kDrawTau = 3 };
__device__ __forceinline__ uint64_t sim_stream(int64_t replica, int64_t step, int kind) {
  return ((uint64_t)replica << 40) | ((uint64_t)step << 4) | (uint64_t)kind;
}

// Standard Gamma(a) draw, Marsaglia & Tsang (2000): attempt k of draw `sub` reads the Philox group idx = sub << 32 | k of
// (seed, stream): words x, y -> one normal (Box-Muller), z -> the acceptance uniform.  a < 1 draws Gamma(a + 1) and boosts it
// by U^(1/a) with U = word w of attempt 0.  The value depends on (a, seed, stream, sub) only.
__device__ float philox_std_gamma(float a, uint64_t seed, uint64_t stream, uint32_t sub) {
  if (!(a > 0.f) || isinf(a)) return NAN;
  const bool boost = a < 1.0f;
  const float d = (boost ? a + 1.0f : a) - 1.0f / 3.0f, c = 1.0f / sqrtf(9.0f * d);
  float ub = 1.0f;
  for (uint32_t k = 0; k < kGammaMaxAttempts; ++k) {   // each attempt accepts with probability > 0.95
    const Philox4 p = philox4x32_10(seed, stream, ((uint64_t)sub << 32) | k);
    if (k == 0) ub = u01(p.w);
    const float x = sqrtf(-2.0f * logf(u01(p.x))) * cospif(2.0f * u01(p.y));
    float v = 1.0f + c * x;
    if (v <= 0.f) continue;
    v = v * v * v;
    const float u = u01(p.z), x2 = x * x;
    if (u < 1.0f - 0.0331f * x2 * x2 || logf(u) < 0.5f * x2 + d * (1.0f - v + logf(v)))
      return boost ? d * v * powf(ub, 1.0f / a) : d * v;
  }
  return NAN;
}

// d g / d a of a standard Gamma(a) draw g (implicit reparameterisation): ATen's standard_gamma_grad_one
// (ATen/native/Distributions.h) in fp32, the function torch._standard_gamma_grad evaluates on the GPU
__device__ float standard_gamma_grad(float alpha, float x) {
  if (x < 0.8f) {                                  // Taylor series for small x
    float numer = 1.f, denom = alpha;
    float series1 = numer / denom, series2 = numer / (denom * denom);
    for (int i = 1; i <= 5; ++i) {
      numer *= -x / (float)i;
      denom += 1.f;
      series1 += numer / denom;
      series2 += numer / (denom * denom);
    }
    const float pow_x_alpha = powf(x, alpha);
    const float gamma_pdf = powf(x, alpha - 1.f) * expf(-x);
    const float gamma_cdf = pow_x_alpha * series1;
    const float gamma_cdf_alpha = (logf(x) - digammaf(alpha)) * gamma_cdf - pow_x_alpha * series2;
    const float result = -gamma_cdf_alpha / gamma_pdf;
    return isnan(result) ? 0.f : result;
  }
  if (alpha > 8.0f) {                              // Rice saddle point expansion for large alpha
    if (0.9f * alpha <= x && x <= 1.1f * alpha) {
      const float numer_1 = 1 + 24 * alpha * (1 + 12 * alpha);
      const float numer_2 = 1440 * (alpha * alpha) + 6 * x * (53 - 120 * x) - 65 * x * x / alpha + alpha * (107 + 3600 * x);
      const float denom = 1244160 * (alpha * alpha) * (alpha * alpha);
      return numer_1 * numer_2 / denom;
    }
    const float denom = sqrtf(8 * alpha);
    const float term2 = denom / (alpha - x);
    const float term3 = powf(x - alpha - alpha * logf(x / alpha), -1.5f);
    const float term23 = (x < alpha) ? term2 - term3 : term2 + term3;
    const float term1 = logf(x / alpha) * term23 - sqrtf(2 / alpha) * (alpha + x) / ((alpha - x) * (alpha - x));
    const float stirling = 1 + 1 / (12 * alpha) * (1 + 1 / (24 * alpha));
    const float numer = x * term1;
    return -stirling * numer / denom;
  }
  // bivariate rational approximation
  const float u = logf(x / alpha), v = logf(alpha);
  const float coef_uv[3][8] = {
      {0.16009398f, -0.094634809f, 0.025146376f, -0.0030648343f, 1.f, 0.32668115f, 0.10406089f, 0.0014179084f},
      {0.53487893f, 0.1298071f, 0.065735949f, -0.0015649758f, 0.16639465f, 0.020070113f, -0.0035938915f, -0.00058392623f},
      {0.040121004f, -0.0065914022f, -0.0026286047f, -0.0013441777f, 0.017050642f, -0.0021309326f, 0.00085092367f,
       -1.5247877e-07f},
  };
  float coef_v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) coef_v[i] = coef_uv[0][i] + u * (coef_uv[1][i] + u * coef_uv[2][i]);
  const float p = coef_v[0] + v * (coef_v[1] + v * (coef_v[2] + v * coef_v[3]));
  const float q = coef_v[4] + v * (coef_v[5] + v * (coef_v[6] + v * coef_v[7]));
  return expf(p / q);
}

// tau = Gamma(a, b).rsample() from the standard draw g, clamped at tiny in value only, and its partial derivatives
// (BayesianLinear._tau_draw): d tau / d a = standard_gamma_grad(a, g) / b, d tau / d b = -g / b^2
struct Tau { float tau, da, db; };
__device__ __forceinline__ Tau tau_draw(float a, float b, float g) {
  const float rb = 1.0f / b, raw = g * rb;
  return Tau{fmaxf(raw, kTiny), standard_gamma_grad(a, g) * rb, -raw * rb};
}

__device__ __forceinline__ float pick4(const float (&v)[4], int i) { return i == 0 ? v[0] : (i == 1 ? v[1] : (i == 2 ? v[2] : v[3])); }

// packed parameter row: weight_mu, weight_rho, lambdal (in each), then the eight scalars
enum { kBiasMu = 0, kBiasRho, kWa, kWb, kBa, kBb, kPa, kPb, kNScalars };

__global__ void __launch_bounds__(kSimThreads) mfsim_train_kernel(const lbbnn_mfsim d, int epochs) {
  __shared__ float w_s[kSimMaxIn];
  __shared__ float bias_s;
  __shared__ float red[kSimWarps][kSimMaxIn + 2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int in = (int)d.in_features;
  const int64_t B = d.batch, nb = d.rows / d.batch, steps = (int64_t)epochs * nb;
  const float inv_t = 1.0f / d.temperature;
  const int exact_b = (d.flags & LBBNN_MF_FLAG_EXACT_GAMMA) ? 1 : 0;
  const int exact_wp = (d.flags & LBBNN_MF_FLAG_EXACT_WPRIOR) ? 1 : 0;
  const int exact_gp = (d.flags & LBBNN_MF_FLAG_EXACT_GPRIOR) ? 1 : 0;
  const bool injected = d.eps_w != nullptr;
  const bool gamma_grad = d.gamma == nullptr && !exact_b;     // relaxed draw: the gradient reaches lambda through gamma
  const float gq = 1.0f / d.num_batches, gp = -gq;           // loss = nll + (log q - log prior) / num_batches
  const bool el = warp == 0 && lane < in;

  for (int64_t r = blockIdx.x; r < d.replicas; r += gridDim.x) {
    float* prm = d.params + r * d.param_stride;
    const float* X = d.x + r * d.x_stride;
    const float* Y = d.y + r * d.y_stride;
    // warp 0 holds the parameters for the whole run: weight `lane`, and the scalars on every lane
    float mu = 0.f, rho = 0.f, lam = 0.f, sc[kNScalars];
    int64_t step0 = 0;
    if (warp == 0) {
      if (el) { mu = prm[lane]; rho = prm[in + lane]; lam = prm[2 * in + lane]; }
#pragma unroll
      for (int k = 0; k < kNScalars; ++k) sc[k] = prm[3 * in + k];
      step0 = d.step[r];
    }
    for (int64_t s = 0; s < steps; ++s) {
      // ---- A: draws, weights, log-probabilities (warp 0) ----
      float ep = 0.f, u = 0.5f, g = 0.f, eb = 0.f, g0w = 0.f, g0b = 0.f, lp = 0.f, lq = 0.f, bias = 0.f, sums[5];
      Tau tw{}, tb{};
      if (warp == 0) {
        const int64_t o = r * steps + s;
        if (injected) {
          if (el) {
            ep = __ldg(d.eps_w + o * in + lane);
            if (d.gamma) g = __ldg(d.gamma + o * in + lane);
            else if (d.u) u = __ldg(d.u + o * in + lane);
          }
          eb = __ldg(d.eps_b + o); g0w = __ldg(d.g0_w + o); g0b = __ldg(d.g0_b + o);
        } else {
          const int64_t gs = step0 + s;
          float v4[4];     // element `lane` of the stream, as philox_uniform1 / philox_normal1 (selects, not a local array)
          philox_uniform4(d.seed, sim_stream(r, gs, kDrawU), (uint64_t)(lane >> 2), v4);
          u = pick4(v4, lane & 3);
          philox_normal4(d.seed, sim_stream(r, gs, kDrawEpsW), (uint64_t)(lane >> 2), v4);
          ep = pick4(v4, lane & 3);
          eb = philox_normal1(d.seed, sim_stream(r, gs, kDrawEpsB), 0);
          g0w = philox_std_gamma(sc[kWa], d.seed, sim_stream(r, gs, kDrawTau), 0);
          g0b = philox_std_gamma(sc[kBa], d.seed, sim_stream(r, gs, kDrawTau), 1);
        }
        const float al = alpha_of(lam), sg = sigma_of(rho);
        if (d.gamma == nullptr) g = exact_b ? (u < al ? 1.0f : 0.0f) : relaxed_bernoulli(al, u, inv_t);
        const float ws = fmaf(sg, ep, mu);
#pragma unroll
        for (int k = 0; k < 5; ++k) sums[k] = 0.f;
        if (el) {
          w_s[lane] = g * ws;
          mf_lp_terms(g, ws, mu, sg, al, sc[kPb], exact_b, exact_wp, exact_gp, sums);   // at the unmasked ws (MFsim:233,237)
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) sums[k] = warp_sum(sums[k]);
        const float sb = sigma_of(sc[kBiasRho]);
        bias = sc[kBiasMu] + sb * eb;
        tw = tau_draw(sc[kWa], sc[kWb], g0w);
        tb = tau_draw(sc[kBa], sc[kBb], g0b);
        float gb = 0.f, lqb = 0.f;
        mf_bias_lp_terms(bias, sc[kBiasMu], sb, sc[kBa], sc[kBb], tb.tau, gb, lqb);
        lp = mf_log_prior(sums, gb, sc[kWa], sc[kWb], tw.tau, sc[kPa], sc[kPb], (float)in);
        lq = sums[3] + sums[4] + lqb;
        if (lane == 0) bias_s = bias;
      }
      __syncthreads();

      // ---- B: logits, sigmoid, BCE (torch's formulas) and the batch sums of the backward (all threads) ----
      const int64_t k = s % nb;
      const float* Xb = X + k * B * in;
      const float* Yb = Y + k * B;
      float acc[kSimMaxIn], nll = 0.f, dbl = 0.f;
#pragma unroll
      for (int f = 0; f < kSimMaxIn; ++f) acc[f] = 0.f;
      for (int64_t j = threadIdx.x; j < B; j += kSimThreads) {
        const float* xr = Xb + j * in;
        float xv[kSimMaxIn];
        float z = 0.f;
#pragma unroll
        for (int f = 0; f < kSimMaxIn; ++f) {
          xv[f] = f < in ? __ldg(xr + f) : 0.f;
          if (f < in) z = fmaf(xv[f], w_s[f], z);
        }
        z += bias_s;
        const float p = 1.0f / (1.0f + expf(-z));
        const float y = __ldg(Yb + j);
        // binary_cross_entropy: log terms clamped at -100; backward (p - y) / max(p (1 - p), 1e-12), then sigmoid's p (1 - p)
        const float li = fmaxf(logf(p), -100.f), l1 = fmaxf(log1pf(-p), -100.f);
        nll += (y - 1.0f) * l1 - y * li;
        const float dp = (p - y) / fmaxf((1.0f - p) * p, 1e-12f);
        const float dz = dp * (1.0f - p) * p;
        dbl += dz;
#pragma unroll
        for (int f = 0; f < kSimMaxIn; ++f)
          if (f < in) acc[f] = fmaf(dz, xv[f], acc[f]);
      }
#pragma unroll
      for (int f = 0; f < kSimMaxIn; ++f) {
        if (f < in) {
          const float v = warp_sum(acc[f]);
          if (lane == 0) red[warp][f] = v;
        }
      }
      nll = warp_sum(nll);
      dbl = warp_sum(dbl);
      if (lane == 0) { red[warp][kSimMaxIn] = nll; red[warp][kSimMaxIn + 1] = dbl; }
      __syncthreads();

      // ---- C: backward and SGD (warp 0) ----
      if (warp == 0) {
        float dW = 0.f, nll_t = 0.f, db_lin = 0.f;
#pragma unroll
        for (int q = 0; q < kSimWarps; ++q) {
          if (el) dW += red[q][lane];
          nll_t += red[q][kSimMaxIn];
          db_lin += red[q][kSimMaxIn + 1];
        }
        float dsc[10];
        mf_log_prior_bwd(gp, gq, sums[0], sums[1], sc[kWa], sc[kWb], tw.tau, sc[kPa], sc[kPb], (float)in, 1, tw.da, tw.db, dsc);
        const MfElemGrad e = mf_lp_terms_bwd(dsc, mu, rho, lam, g, ep, dW, sc[kPb], 1, exact_b, exact_wp, exact_gp);
        float dlam = e.dlam;
        if (gamma_grad) dlam += relaxed_bernoulli_bwd(e.dgamma, g, alpha_of(lam), inv_t, true);
        const float psis = warp_sum(el ? e.psi : 0.f);
        const MfBiasGrad bg = mf_bias_lp_terms_bwd(gp, gq, db_lin, sc[kBiasMu], sc[kBiasRho], bias, eb, sc[kBa], sc[kBb],
                                                   tb.tau, 1, 1, tb.da, tb.db);
        float gs[kNScalars];
        gs[kBiasMu] = bg.dmu; gs[kBiasRho] = bg.drho; gs[kWa] = dsc[5]; gs[kWb] = dsc[6];
        gs[kBa] = bg.dba; gs[kBb] = bg.dbb; gs[kPa] = dsc[8]; gs[kPb] = dsc[9] + psis * dsc[2];
        if (d.grads && s == steps - 1) {
          float* gr = d.grads + r * d.param_stride;
          if (el) { gr[lane] = e.dmu; gr[in + lane] = e.drho; gr[2 * in + lane] = dlam; }
          if (lane == 0) {
#pragma unroll
            for (int q = 0; q < kNScalars; ++q) gr[3 * in + q] = gs[q];
          }
        }
        if (lane == 0) {
          float* st = d.stats + (r * steps + s) * 4;
          st[0] = nll_t + (lq - lp) / d.num_batches;
          st[1] = nll_t;
          st[2] = lp;
          st[3] = lq;
        }
        if (el) {
          mu = fmaf(-d.lr[0], e.dmu, mu);
          rho = fmaf(-d.lr[1], e.drho, rho);
          lam = fmaf(-d.lr[2], dlam, lam);
        }
#pragma unroll
        for (int q = 0; q < kNScalars; ++q) sc[q] = fmaf(-d.lr[3 + q], gs[q], sc[q]);
      }
    }
    if (warp == 0) {
      if (el) { prm[lane] = mu; prm[in + lane] = rho; prm[2 * in + lane] = lam; }
      if (lane == 0) {
#pragma unroll
        for (int q = 0; q < kNScalars; ++q) prm[3 * in + q] = sc[q];
        d.step[r] = step0 + steps;
      }
    }
  }
}

__global__ void std_gamma_kernel(float a, int64_t n, uint64_t seed, uint64_t stream, float* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = philox_std_gamma(a, seed, stream, (uint32_t)i);
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" int lbbnn_mfsim_train_f32(const lbbnn_mfsim* d, int epochs, lbbnn_stream s) {
  LBBNN_REQUIRE(d, "NULL descriptor");
  LBBNN_REQUIRE(epochs >= 1, "epochs must be >= 1, got %d", epochs);
  LBBNN_REQUIRE(d->replicas >= 1 && d->replicas < (1LL << 24), "replicas must be in [1, 2^24), got %lld", (long long)d->replicas);
  LBBNN_REQUIRE(d->in_features >= 1 && d->in_features <= LBBNN_MFSIM_MAX_IN,
                "in_features must be in [1, %d] (one warp holds the weights), got %lld", LBBNN_MFSIM_MAX_IN,
                (long long)d->in_features);
  LBBNN_REQUIRE(d->batch >= 1 && d->rows >= d->batch && d->rows % d->batch == 0,
                "rows (%lld) must be a positive multiple of the batch size (%lld)", (long long)d->rows, (long long)d->batch);
  LBBNN_REQUIRE(d->params && d->x && d->y && d->step && d->stats, "NULL params, x, y, step or stats");
  LBBNN_REQUIRE(d->param_stride >= 3 * d->in_features + 8, "param_stride too small");
  LBBNN_REQUIRE(d->x_stride == 0 || d->x_stride == d->rows * d->in_features, "x_stride must be 0 (shared) or rows * in_features");
  LBBNN_REQUIRE(d->y_stride == 0 || d->y_stride == d->rows, "y_stride must be 0 (shared) or rows");
  LBBNN_REQUIRE(d->temperature > 0.f && d->num_batches > 0.f, "temperature and num_batches must be positive");
  const bool inj = d->eps_w != nullptr;
  LBBNN_REQUIRE((d->eps_b != nullptr) == inj && (d->g0_w != nullptr) == inj && (d->g0_b != nullptr) == inj,
                "injected noise: give all of eps_w, eps_b, g0_w, g0_b or none");
  LBBNN_REQUIRE(inj ? ((d->u != nullptr) != (d->gamma != nullptr)) : (!d->u && !d->gamma),
                "injected noise takes exactly one of u / gamma; native noise neither");
  LBBNN_REQUIRE((d->flags & ~(LBBNN_MF_FLAG_EXACT_GAMMA | LBBNN_MF_FLAG_EXACT_WPRIOR | LBBNN_MF_FLAG_EXACT_GPRIOR)) == 0,
                "flags: only the three EXACT flags apply");
  const int64_t cap = 16LL * sm_count();
  const unsigned grid = (unsigned)(d->replicas < cap ? d->replicas : cap);
  mfsim_train_kernel<<<grid, kSimThreads, 0, (cudaStream_t)s>>>(*d, epochs);
  return check_launch("mfsim_train");
}

extern "C" int lbbnn_philox_std_gamma(float a, int64_t n, uint64_t seed, uint64_t stream_id, float* out, lbbnn_stream s) {
  LBBNN_REQUIRE(out && n > 0 && n <= (1LL << 32), "bad argument");
  LBBNN_REQUIRE(a > 0.f && a < INFINITY, "the shape a must be positive and finite");
  int64_t blocks = ceil_div(n, 256);
  if (blocks > 8LL * sm_count()) blocks = 8LL * sm_count();
  std_gamma_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(a, n, seed, stream_id, out);
  return check_launch("philox_std_gamma");
}
