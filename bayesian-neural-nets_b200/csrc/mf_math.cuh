// Per-element math of the mean-field layer (LBBNN-GP-MF.py:74-255, sim-study variant MFsim:173-244), shared by the
// layer kernels (mf.cu) and the one-launch simulation-study trainer (mf_sim.cu).  The expressions are the reference's,
// term for term; both callers inline them, so the fp32 rounding is the same wherever they run.
#pragma once
#include "common.cuh"

namespace lbbnn {

constexpr float kLogSqrt2Pi = 0.91893853320467274178f;
constexpr float kEps = 1.1920928955078125e-07f;   // torch.finfo(float32).eps
constexpr float kTiny = 1.1754943508222875e-38f;  // torch.finfo(float32).tiny

// digamma for x > 0: recurrence up to x >= 6, then the asymptotic series
__device__ __forceinline__ float digammaf(float x) {
  float r = 0.f;
  while (x < 6.0f) { r -= 1.0f / x; x += 1.0f; }
  const float f = 1.0f / (x * x);
  return r + logf(x) - 0.5f / x - f * (1.0f / 12.0f - f * (1.0f / 120.0f - f * (1.0f / 252.0f - f * (1.0f / 240.0f - f / 132.0f))));
}

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

// torch RelaxedBernoulli(probs = al, T).rsample() for the uniform u: clamp_probs, logistic noise, / T, clipped sigmoid (MF:115)
__device__ __forceinline__ float relaxed_bernoulli(float al, float u, float inv_t) {
  const float p = clampf(al, kEps, 1.0f - kEps), uu = clampf(u, kEps, 1.0f - kEps);
  const float logits = (logf(uu) - log1pf(-uu) + logf(p) - log1pf(-p)) * inv_t;
  return clampf(1.0f / (1.0f + expf(-logits)), kTiny, 1.0f - kEps);
}

// d gamma / d alpha of the relaxed draw applied to dgamma: gamma(1-gamma)/T * (1/p + 1/(1-p)), zero where a clamp is active;
// from_lambda: times d alpha / d lambda = alpha(1-alpha) (alpha = sigmoid(lambda) formed inside the kernel)
__device__ __forceinline__ float relaxed_bernoulli_bwd(float dgamma, float g, float al, float inv_t, bool from_lambda) {
  float d = 0.f;
  if (g > kTiny && g < 1.0f - kEps && al > kEps && al < 1.0f - kEps) {
    d = dgamma * g * (1.0f - g) * inv_t * (1.0f / al + 1.0f / (1.0f - al));
    if (from_lambda) d *= al * (1.0f - al);
  }
  return d;
}

// One weight's terms of the five log-probability sums (MF:99-101, 122-128, 140-151, 162-173):
//   s0 += g, s1 += wl^2, s2 += lgamma(1+pb-g) - lgamma(2-g), s3 += log(g N(wl; mu, sg) + (1-g) + 1e-8),
//   s4 += g log(al+1e-8) + (1-g) log(1-al+1e-8)
// with g rounded where the matching `.exact` flag is set; wl is w (MF) or the unmasked ws (MFsim:233,237).
__device__ __forceinline__ void mf_lp_terms(float g, float wl, float mu, float sg, float al, float pb, int exact_b,
                                            int exact_wp, int exact_gp, float s[5]) {
  const float gr = rintf(g);
  const float g_wp = exact_wp ? gr : g, g_gp = exact_gp ? gr : g, g_b = exact_b ? gr : g;
  s[0] += g_wp;
  s[1] += wl * wl;
  s[2] += lgammaf(1.0f + pb - g_gp) - lgammaf(2.0f - g_gp);
  const float dlt = wl - mu;
  const float logn = -kLogSqrt2Pi - logf(sg) - (dlt * dlt) / (2.0f * sg * sg);
  s[3] += logf(g * expf(logn) + (1.0f - g) + 1e-8f);
  s[4] += g_b * logf(al + 1e-8f) + (1.0f - g_b) * logf(1.0f - al + 1e-8f);
}

// Gradients of one weight: autograd of ws = mu + sigma(rho) eps, w = g ws and of mf_lp_terms, given dL/dw and
// c = dL/ds0..4.  Outputs dmu, drho, dlambda (through alpha in s4), dgamma and psi(1+pb-g) (the weight's share of dpb / c2).
struct MfElemGrad { float dmu, drho, dlam, dgamma, psi; };

__device__ __forceinline__ MfElemGrad mf_lp_terms_bwd(const float c[5], float mu, float rho, float lam, float g, float ep,
                                                      float dw, float pb, int lp_on_ws, int exact_b, int exact_wp,
                                                      int exact_gp) {
  const float sg = sigma_of(rho), al = alpha_of(lam);
  const float ws = fmaf(sg, ep, mu), w = g * ws, wl = lp_on_ws ? ws : w;
  const float grd = rintf(g);
  const float g_gp = exact_gp ? grd : g, g_b = exact_b ? grd : g;
  const float dlt = wl - mu, inv_s2 = 1.0f / (sg * sg);
  const float logn = -kLogSqrt2Pi - logf(sg) - (dlt * dlt) * 0.5f * inv_s2;
  const float p = expf(logn), D = g * p + (1.0f - g) + 1e-8f, r = g * p / D;
  const float dwl = c[1] * 2.0f * wl - c[3] * r * dlt * inv_s2;          // direct dL/d(wl)
  const float dmu_dir = c[3] * r * dlt * inv_s2;
  const float dsg_dir = c[3] * r * (dlt * dlt * inv_s2 / sg - 1.0f / sg);
  const float psi = digammaf(1.0f + pb - g_gp);
  float dg_dir = c[3] * (p - 1.0f) / D;
  if (!exact_wp) dg_dir += c[0];
  if (!exact_gp) dg_dir += c[2] * (digammaf(2.0f - g_gp) - psi);
  if (!exact_b) dg_dir += c[4] * (logf(al + 1e-8f) - logf(1.0f - al + 1e-8f));
  const float dal = c[4] * (g_b / (al + 1e-8f) - (1.0f - g_b) / (1.0f - al + 1e-8f));
  const float dw_tot = dw + (lp_on_ws ? 0.f : dwl);
  const float dws = g * dw_tot + (lp_on_ws ? dwl : 0.f);
  MfElemGrad o;
  o.dmu = dws + dmu_dir;
  o.drho = (ep * dws + dsg_dir) * dsigma_drho(rho);
  o.dlam = dal * al * (1.0f - al);
  o.dgamma = ws * dw_tot + dg_dir;
  o.psi = psi;
  return o;
}

// log N-Gamma constant of GaussGamma.log_prob (MF:148): a log b + (a - 1/2) tau - b tau - lgamma(a) - log sqrt(2 pi)
__device__ __forceinline__ float gauss_gamma_const(float a, float b, float tau) {
  return a * logf(b) + (a - 0.5f) * tau - b * tau - lgammaf(a) - kLogSqrt2Pi;
}

// One bias's log-prior (GaussGamma with gamma = 1) and log-q (Gaussian) terms (MF:246-251)
__device__ __forceinline__ void mf_bias_lp_terms(float bias, float mu, float sb, float ba, float bb, float tb, float& gb,
                                                 float& lq) {
  const float cb = gauss_gamma_const(ba, bb, tb);
  gb += cb - tb * bias * bias + 1e-8f;
  const float d = bias - mu;
  lq += -kLogSqrt2Pi - logf(sb) - (d * d) / (2.0f * sb * sb);
}

// Gradients of one bias's terms: gp = dL/d log_prior, gq = dL/d log_q, gbias = dL/d bias from the linear layer; tb_da / tb_db
// (NULL-able as has_tau_grads = 0) fold the precision's own derivative wrt (ba, bb) in.
struct MfBiasGrad { float dba, dbb, dtb, dmu, drho; };

__device__ __forceinline__ MfBiasGrad mf_bias_lp_terms_bwd(float gp, float gq, float gbias, float mu, float rho, float bias,
                                                           float e, float ba, float bb, float tb, int sample, int has_tau_grads,
                                                           float tb_da, float tb_db) {
  const float sb = sigma_of(rho), d = bias - mu;
  const float dtb = gp * ((ba - 0.5f) - bb - bias * bias);
  float dba = gp * (logf(bb) + tb - digammaf(ba)), dbb = gp * (ba / bb - tb);
  if (has_tau_grads) {
    dba = fmaf(dtb, tb_da, dba);
    dbb = fmaf(dtb, tb_db, dbb);
  }
  MfBiasGrad o;
  o.dba = dba;
  o.dbb = dbb;
  o.dtb = dtb;
  const float inv2 = 1.0f / (sb * sb);
  const float G = gbias + gp * (-2.0f * tb * bias) + gq * (-d * inv2);   // d loss / d bias
  o.dmu = G + gq * (d * inv2);
  const float dsb = (sample ? G * e : 0.f) + gq * (-1.0f / sb + d * d * inv2 / sb);
  o.drho = dsb * dsigma_drho(rho);
  return o;
}

// The layer's log prior from the five sums and the bias part gb (MF:148-150, 167-173): GaussGamma on n weights + gb +
// BetaBinomial with its element-independent lgamma terms
__device__ __forceinline__ float mf_log_prior(const float s[5], float gb, float a, float b, float tw, float pa, float pb, float n) {
  const float cw = gauss_gamma_const(a, b, tw);
  const float ggw = s[0] * cw - tw * s[1] + (n - s[0]) + n * 1e-8f;
  const float bbin = s[2] + n * (lgammaf(pa + pb) - lgammaf(1.0f + pa + pb) - lgammaf(pa) - lgammaf(pb));
  return ggw + gb + bbin;
}

// Gradients of mf_log_prior wrt its scalars, gp = dL/d log_prior, gq = dL/d log_q:
// d[0..4] = dL/ds0..4, d[5] = da, d[6] = db, d[7] = dtau_w, d[8] = dpa, d[9] = dpb (without the s2 part, psi(1+pb-g) per weight)
__device__ __forceinline__ void mf_log_prior_bwd(float gp, float gq, float s0, float s1, float a, float b, float tw, float pa,
                                                 float pb, float n, int has_tau_grads, float tw_da, float tw_db, float d[10]) {
  const float cw = gauss_gamma_const(a, b, tw);
  d[0] = gp * (cw - 1.0f);
  d[1] = gp * (-tw);
  d[2] = gp;
  d[3] = gq;
  d[4] = gq;
  const float dtw = gp * (s0 * ((a - 0.5f) - b) - s1);
  float da = gp * s0 * (logf(b) + tw - digammaf(a)), db = gp * s0 * (a / b - tw);
  if (has_tau_grads) {
    da = fmaf(dtw, tw_da, da);
    db = fmaf(dtw, tw_db, db);
  }
  d[5] = da;
  d[6] = db;
  d[7] = dtw;
  const float psi_s = digammaf(pa + pb) - digammaf(1.0f + pa + pb);
  d[8] = gp * n * (psi_s - digammaf(pa));
  d[9] = gp * n * (psi_s - digammaf(pb));
}

}  // namespace lbbnn
