// The MNF simulation study (LBBNN-GP-MF-MNFsim_study.py) in one launch: R independent repetitions of the in -> 1 MNF logistic
// regression (lbbnn.mnf.SimStudyNetwork: one MNF layer with RNVP z and r flows, sigmoid + BCELoss(sum), loss = nll +
// kl / num_batches) trained with torch.optim.Adam (one learning rate per group) for any number of epochs.  The repetitions
// share nothing but read-only data, so each is one CTA: no grid barrier, no host round trip, no launch per step.
//
// A replica's flows hold ~53 k parameters (two flows of two RNVP transforms with five 50-wide hidden layers at in = 20), too
// many for shared memory next to their Adam moments, so parameters and moments stay in global memory (L2) and are read with
// coherent loads: the CTA rewrites them every step.  Everything a step computes (the three flow rows' saved activations, the
// batch sums, the layer gradients) lives in shared memory.
//
// Layout of a step (all 256 threads, phases separated by __syncthreads):
//   0  draws (eps_z of both z rows, the masks of every transform of the three flow rows, eps_r), the layer tensors -> smem
//   1  z0 = q0_mean + sqrt(exp(q0_log_var)) eps for the activation row and the KL row, the z flow on both rows (z_k, z2,
//      log_det_q), the r flow on z2 (z_b, log_det_r): per Linear, one thread per (row, output neuron)
//   2  the batch: act = x (alpha mu z_k) + b_mu + sqrt(x^2 (sigma^2 alpha^2) + sigma_b^2) eps, sigmoid, BCE (torch's clamps)
//      and the batch sums of its backward, reduced in a fixed order (shuffle tree per warp, warps in order)
//   3  warp 0, lane = input feature: the weight / bias KL with z2, log q0, the auxiliary r(z|W) term, kl, the loss, and the
//      backward of all of it down to d z_k, d z2, d z_b and the layer tensors' direct gradients
//   4  the r flow backward, then the z flow backward on both rows: each flow weight's gradient is formed once (a fixed-order
//      sum over the live rows) and Adam is applied in the same pass, after the Linear's input gradient has read the weight
//   5  d q0_mean / d q0_log_var through the z0 draw, Adam on the layer tensors
#include "common.cuh"

namespace lbbnn {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kD = LBBNN_MNFSIM_MAX_IN;
constexpr int kT = LBBNN_MNFSIM_MAX_T;
constexpr int kH = LBBNN_MNFSIM_MAX_H;
constexpr int kNH = LBBNN_FLOW_MAX_HIDDEN;
constexpr int kRows = 3;                 // flow rows: 0 = activation row (z flow), 1 = KL row (z flow), 2 = z2 (r flow)
constexpr int kLayer = 8 * kD + 2;       // the ten layer tensors at in <= kD, out = 1

// packed layer tensors at in_features = D
__device__ __forceinline__ int off_wmu(int) { return 0; }
__device__ __forceinline__ int off_wrho(int D) { return D; }
__device__ __forceinline__ int off_lam(int D) { return 2 * D; }
__device__ __forceinline__ int off_bmu(int D) { return 3 * D; }
__device__ __forceinline__ int off_brho(int D) { return 3 * D + 1; }
__device__ __forceinline__ int off_q0m(int D) { return 3 * D + 2; }
__device__ __forceinline__ int off_q0lv(int D) { return 4 * D + 2; }
__device__ __forceinline__ int off_r0c(int D) { return 5 * D + 2; }
__device__ __forceinline__ int off_rb1(int D) { return 6 * D + 2; }
__device__ __forceinline__ int off_rb2(int D) { return 7 * D + 2; }
// the Adam group (lr index) of layer element e
__device__ __forceinline__ int layer_group(int e, int D) {
  if (e < 3 * D) return e / D;
  if (e < 3 * D + 2) return 3 + (e - 3 * D);
  return 5 + (e - 3 * D - 2) / D;
}

// Philox stream of one kind of draw of one step of one replica: replica < 2^24 in bits 40.., step < 2^36 in bits 4..39
__device__ __forceinline__ uint64_t sim_stream(int64_t replica, int64_t step, int kind) {
  return ((uint64_t)replica << 40) | ((uint64_t)step << 4) | (uint64_t)kind;
}

// element e of lbbnn_philox_normal / _uniform of a stream, as philox_normal1 / philox_uniform1 (selects, not a local array)
__device__ __forceinline__ float pick4(const float (&v)[4], uint64_t e) {
  const int k = (int)(e & 3);
  return k == 0 ? v[0] : (k == 1 ? v[1] : (k == 2 ? v[2] : v[3]));
}
__device__ __forceinline__ float draw_normal(uint64_t seed, uint64_t stream, uint64_t e) {
  float v[4];
  philox_normal4(seed, stream, e >> 2, v);
  return pick4(v, e);
}
__device__ __forceinline__ float draw_uniform(uint64_t seed, uint64_t stream, uint64_t e) {
  float v[4];
  philox_uniform4(seed, stream, e >> 2, v);
  return pick4(v, e);
}

// one RNVP flow of a replica: offsets (floats) of every tensor of a transform, PropagateFlow._params() order
struct FlowShape {
  int D, T, NH, H, per_t;
  int hid[kNH], oW[kNH], ob[kNH];
  int otW, otb, osW, osb;
};
__device__ __forceinline__ FlowShape flow_shape(const lbbnn_mnfsim& d) {
  FlowShape f;
  f.D = (int)d.in_features; f.T = d.n_transforms; f.NH = d.n_hidden;
  int o = 0, prev = f.D;
  for (int l = 0; l < kNH; ++l) {
    f.hid[l] = l < f.NH ? d.hidden[l] : 0;
    f.oW[l] = o; o += f.hid[l] * prev;
    f.ob[l] = o; o += f.hid[l];
    if (l < f.NH) prev = f.hid[l];
  }
  f.H = prev;
  f.otW = o; o += f.D * f.H;
  f.otb = o; o += f.D;
  f.osW = o; o += f.D * f.H;
  f.osb = o; o += f.D;
  f.per_t = o;
  return f;
}

struct Smem {
  float lp[kLayer];                 // layer tensors of this step
  float gl[kLayer];                 // their gradients
  float ez[2][kD];                  // eps of the two z0 draws
  float z[kRows][kD];               // current z of each flow row
  float zin[kRows][kT][kD];         // input of transform t
  float msk[kRows][kT][kD];
  float gate[kRows][kT][kD];
  float shf[kRows][kT][kD];
  float hs[kRows][kT][kNH][kH];     // hidden activations (post-activation)
  float dz[kRows][kD], dsh[kRows][kD], dsc[kRows][kD], dz2p[kD];
  float dh[kRows][kH], da[kRows][kH];
  float ld[kRows], dld[kRows];
  float Mz[kD], V[kD];
  float red[kWarps][2 * kD + 3];
  float step_size[12];
  float bc2_sqrt, eps_r, sigb;
};

struct AdamC { float b1, b2, eps, bc2_sqrt; };

// torch.optim.Adam on one element (exp_avg.lerp_(g, 1 - b1), exp_avg_sq = b2 v + (1 - b2) g^2,
// p -= step_size exp_avg / (sqrt(exp_avg_sq) / sqrt(1 - b2^t) + eps))
__device__ __forceinline__ void adam_el(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v, float* __restrict__ gout,
                                        int64_t i, float g, float step_size, const AdamC& c) {
  float mm = m[i], vv = v[i];
  mm = fmaf(1.0f - c.b1, g - mm, mm);
  vv = c.b2 * vv + (1.0f - c.b2) * g * g;
  p[i] = p[i] - step_size * (mm / (sqrtf(vv) / c.bc2_sqrt + c.eps));
  m[i] = mm;
  v[i] = vv;
  if (gout) gout[i] = g;
}

__device__ __forceinline__ float leaky(float a) { return a > 0.f ? a : 0.1f * a; }

// forward of one flow (params fp) on rows [rb, rb + nr): z[r] -> z[r], ld[r] += log_det; saves what the backward needs
__device__ __forceinline__ void flow_fwd(Smem& S, const float* fp, const FlowShape& f, int rb, int nr) {
  const int tid = threadIdx.x, D = f.D;
  for (int t = 0; t < f.T; ++t) {
    const float* tp = fp + (int64_t)t * f.per_t;
    for (int idx = tid; idx < nr * D; idx += kThreads) {
      const int r = rb + idx / D, dd = idx % D;
      S.zin[r][t][dd] = S.z[r][dd];
    }
    __syncthreads();
    int in = D;
    for (int l = 0; l < f.NH; ++l) {
      const int out = f.hid[l];
      const float* W = tp + f.oW[l];
      const float* b = tp + f.ob[l];
      for (int idx = tid; idx < nr * out; idx += kThreads) {
        const int r = rb + idx / out, j = idx % out;
        const float* w = W + j * in;
        float a = 0.f;
        if (l == 0) {
#pragma unroll 4
          for (int i = 0; i < in; ++i) a = fmaf(w[i], S.msk[r][t][i] * S.zin[r][t][i], a);
        } else {
#pragma unroll 4
          for (int i = 0; i < in; ++i) a = fmaf(w[i], S.hs[r][t][l - 1][i], a);
        }
        a += b[j];
        S.hs[r][t][l][j] = l < f.NH - 1 ? leaky(a) : a;     // the MLP drops its last activation (flows2:185)
      }
      __syncthreads();
      in = out;
    }
    const int H = f.H;
    for (int idx = tid; idx < nr * D; idx += kThreads) {
      const int r = rb + idx / D, dd = idx % D;
      const float* y = S.hs[r][t][f.NH - 1];
      const float* wt = tp + f.otW + dd * H;
      const float* ws = tp + f.osW + dd * H;
      float sh = 0.f, sc = 0.f;
#pragma unroll 4
      for (int i = 0; i < H; ++i) { sh = fmaf(wt[i], y[i], sh); sc = fmaf(ws[i], y[i], sc); }
      sh += tp[f.otb + dd];
      sc += tp[f.osb + dd];
      const float g = 1.0f / (1.0f + expf(-sc));
      const float m = S.msk[r][t][dd], z = S.zin[r][t][dd];
      S.gate[r][t][dd] = g;
      S.shf[r][t][dd] = sh;
      S.z[r][dd] = (1.0f - m) * z * g + (1.0f - g) * sh + m * z;   // flows2:215, (1 - g) shift on every dim
    }
    __syncthreads();
    if (tid < nr) {
      const int r = rb + tid;
      float s = 0.f;
      for (int dd = 0; dd < D; ++dd) s += (1.0f - S.msk[r][t][dd]) * logf(S.gate[r][t][dd]);
      S.ld[r] += s;
    }
  }
  __syncthreads();
}

// backward of one flow on rows [rb, rb + nr): dz[r] (gradient wrt the output) -> gradient wrt the input, with d log_det =
// dld[r]; every parameter's gradient (summed over the rows in order) goes straight into Adam
__device__ __forceinline__ void flow_bwd(Smem& S, float* fp, float* fm, float* fv, float* fg, const FlowShape& f, int rb, int nr, float step_size,
                         const AdamC& ac) {
  const int tid = threadIdx.x, D = f.D, H = f.H;
  for (int t = f.T - 1; t >= 0; --t) {
    const int64_t to = (int64_t)t * f.per_t;
    float* tp = fp + to;
    float* tm = fm + to;
    float* tv = fv + to;
    float* tg = fg ? fg + to : nullptr;
    for (int idx = tid; idx < nr * D; idx += kThreads) {
      const int r = rb + idx / D, dd = idx % D;
      const float m = S.msk[r][t][dd], z = S.zin[r][t][dd], g = S.gate[r][t][dd], sh = S.shf[r][t][dd], dx = S.dz[r][dd];
      const float dg = dx * ((1.0f - m) * z - sh) + S.dld[r] * (1.0f - m) / g;
      S.dsh[r][dd] = dx * (1.0f - g);
      S.dsc[r][dd] = dg * g * (1.0f - g);
      S.dz[r][dd] = dx * ((1.0f - m) * g + m);         // direct path; the path through the conditioner is added below
    }
    __syncthreads();
    // gradient wrt the conditioner output: dh[r][i] = sum_d Wt[d, i] dsh[r][d] + Ws[d, i] dsc[r][d]
    for (int idx = tid; idx < nr * H; idx += kThreads) {
      const int r = rb + idx / H, i = idx % H;
      float a = 0.f;
      for (int dd = 0; dd < D; ++dd) a = fmaf(tp[f.otW + dd * H + i], S.dsh[r][dd], fmaf(tp[f.osW + dd * H + i], S.dsc[r][dd], a));
      S.dh[r][i] = a;
    }
    __syncthreads();
    // heads: gradient + Adam (their weights have been read)
    for (int idx = tid; idx < D * H; idx += kThreads) {
      const int dd = idx / H, i = idx % H;
      float gt = 0.f, gs = 0.f;
      for (int r = rb; r < rb + nr; ++r) {
        const float y = S.hs[r][t][f.NH - 1][i];
        gt = fmaf(S.dsh[r][dd], y, gt);
        gs = fmaf(S.dsc[r][dd], y, gs);
      }
      adam_el(tp, tm, tv, tg, f.otW + idx, gt, step_size, ac);
      adam_el(tp, tm, tv, tg, f.osW + idx, gs, step_size, ac);
    }
    for (int dd = tid; dd < D; dd += kThreads) {
      float gt = 0.f, gs = 0.f;
      for (int r = rb; r < rb + nr; ++r) { gt += S.dsh[r][dd]; gs += S.dsc[r][dd]; }
      adam_el(tp, tm, tv, tg, f.otb + dd, gt, step_size, ac);
      adam_el(tp, tm, tv, tg, f.osb + dd, gs, step_size, ac);
    }
    // conditioner net, last hidden layer first
    for (int l = f.NH - 1; l >= 0; --l) {
      const int out = f.hid[l], in = l == 0 ? D : f.hid[l - 1];
      for (int idx = tid; idx < nr * out; idx += kThreads) {
        const int r = rb + idx / out, j = idx % out;
        const float h = S.hs[r][t][l][j];
        S.da[r][j] = S.dh[r][j] * (l == f.NH - 1 ? 1.0f : (h > 0.f ? 1.0f : 0.1f));
      }
      __syncthreads();
      const float* W = tp + f.oW[l];
      for (int idx = tid; idx < nr * in; idx += kThreads) {
        const int r = rb + idx / in, i = idx % in;
        float a = 0.f;
        for (int j = 0; j < out; ++j) a = fmaf(W[j * in + i], S.da[r][j], a);
        if (l == 0) S.dz[r][i] += S.msk[r][t][i] * a;     // the net's input was m * z
        else S.dh[r][i] = a;
      }
      __syncthreads();
      for (int idx = tid; idx < out * in; idx += kThreads) {
        const int j = idx / in, i = idx % in;
        float g = 0.f;
        for (int r = rb; r < rb + nr; ++r) {
          const float v = l == 0 ? S.msk[r][t][i] * S.zin[r][t][i] : S.hs[r][t][l - 1][i];
          g = fmaf(S.da[r][j], v, g);
        }
        adam_el(tp, tm, tv, tg, f.oW[l] + idx, g, step_size, ac);
      }
      for (int j = tid; j < out; j += kThreads) {
        float g = 0.f;
        for (int r = rb; r < rb + nr; ++r) g += S.da[r][j];
        adam_el(tp, tm, tv, tg, f.ob[l] + j, g, step_size, ac);
      }
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(kThreads) mnfsim_train_kernel(const lbbnn_mnfsim d, int epochs) {
  __shared__ Smem S;
  __shared__ FlowShape f;          // in shared memory: its per-layer arrays are indexed at run time
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int D = (int)d.in_features;
  if (tid == 0) f = flow_shape(d);
  __syncthreads();
  const int64_t B = d.batch, nb = d.rows / d.batch, steps = (int64_t)epochs * nb;
  const int64_t zoff = 8 * D + 2;                        // the z flow's first parameter
  const int64_t roff = zoff + (int64_t)f.T * f.per_t;
  const bool injected = d.eps_z != nullptr;
  const float gk = 1.0f / d.num_batches;                 // d loss / d kl
  const float LOG_PI = 1.1447298858494002f;
  const lbbnn_priors pr = d.priors;

  for (int64_t r = blockIdx.x; r < d.replicas; r += gridDim.x) {
    float* prm = d.params + r * d.param_stride;
    float* pm = d.exp_avg + r * d.param_stride;
    float* pv = d.exp_avg_sq + r * d.param_stride;
    const float* X = d.x + r * d.x_stride;
    const float* Y = d.y + r * d.y_stride;
    const int64_t step0 = d.step[r];
    __syncthreads();     // the previous replica's last reads of S are done
    for (int64_t s = 0; s < steps; ++s) {
      const int64_t gs = step0 + s;
      float* grow = (d.grads && s == steps - 1) ? d.grads + r * d.param_stride : nullptr;
      // ---- 0: layer tensors, draws ----
      for (int e = tid; e < 8 * D + 2; e += kThreads) { S.lp[e] = prm[e]; S.gl[e] = 0.f; }
      if (tid < kRows) { S.ld[tid] = 0.f; }
      if (tid == 0) {
        const double t = (double)(gs + 1);
        const double bc1 = 1.0 - pow((double)d.beta1, t), bc2 = 1.0 - pow((double)d.beta2, t);
        for (int g = 0; g < 12; ++g) S.step_size[g] = (float)((double)d.lr[g] / bc1);
        S.bc2_sqrt = (float)sqrt(bc2);
        S.eps_r = injected ? d.eps_r[r * steps + s] : draw_normal(d.seed, sim_stream(r, gs, LBBNN_MNFSIM_DRAW_EPS_R), 0);
      }
      {
        const int64_t o = r * steps + s;
        for (int idx = tid; idx < 2 * D; idx += kThreads) {
          const int row = idx / D, e = idx % D;
          S.ez[row][e] = injected ? (row ? d.eps_z2 : d.eps_z)[o * D + e]
                                  : draw_normal(d.seed, sim_stream(r, gs, row ? LBBNN_MNFSIM_DRAW_EPS_Z2 : LBBNN_MNFSIM_DRAW_EPS_Z), e);
        }
        for (int idx = tid; idx < kRows * f.T * D; idx += kThreads) {
          const int row = idx / (f.T * D), t = (idx / D) % f.T, e = idx % D;
          float m;
          if (injected) {
            const float* src = row == 0 ? d.z_masks : (row == 1 ? d.z_masks2 : d.r_masks);
            m = src[(o * f.T + t) * D + e];
          } else {
            const int kind = (row == 0 ? LBBNN_MNFSIM_DRAW_Z_MASK : (row == 1 ? LBBNN_MNFSIM_DRAW_Z_MASK2 : LBBNN_MNFSIM_DRAW_R_MASK)) + t;
            m = draw_uniform(d.seed, sim_stream(r, gs, kind), e) < 0.5f ? 1.0f : 0.0f;
          }
          S.msk[row][t][e] = m;
        }
      }
      __syncthreads();
      const AdamC ac{d.beta1, d.beta2, d.adam_eps, S.bc2_sqrt};
      // ---- 1: z0 draws and the flows ----
      for (int idx = tid; idx < 2 * D; idx += kThreads) {
        const int row = idx / D, e = idx % D;
        S.z[row][e] = S.lp[off_q0m(D) + e] + sqrtf(expf(S.lp[off_q0lv(D) + e])) * S.ez[row][e];
      }
      __syncthreads();
      flow_fwd(S, prm + zoff, f, 0, 2);
      for (int e = tid; e < D; e += kThreads) S.z[2][e] = S.z[1][e];
      __syncthreads();
      flow_fwd(S, prm + roff, f, 2, 1);
      for (int e = tid; e < D; e += kThreads) {
        const float al = alpha_of(S.lp[off_lam(D) + e]), sg = sigma_of(S.lp[off_wrho(D) + e]);
        S.Mz[e] = al * S.lp[off_wmu(D) + e] * S.z[0][e];
        S.V[e] = (sg * sg) * (al * al);
      }
      if (tid == 0) S.sigb = sigma_of(S.lp[off_brho(D)]);
      __syncthreads();

      // ---- 2: the batch ----
      {
        const int64_t k = s % nb;
        const float* Xb = X + k * B * D;
        const float* Yb = Y + k * B;
        const float sb2 = S.sigb * S.sigb, bmu = S.lp[off_bmu(D)];
        float aM[kD], aV[kD], nll = 0.f, dbl = 0.f, dvl = 0.f;
#pragma unroll
        for (int e = 0; e < kD; ++e) { aM[e] = 0.f; aV[e] = 0.f; }
        for (int64_t j = tid; j < B; j += kThreads) {
          const float* xr = Xb + j * D;
          float mean = 0.f, var = 0.f;
#pragma unroll
          for (int e = 0; e < kD; ++e) {
            if (e < D) {
              const float xv = __ldg(xr + e);
              mean = fmaf(xv, S.Mz[e], mean);
              var = fmaf(xv * xv, S.V[e], var);
            }
          }
          const float ep = injected ? d.eps[(r * steps + s) * B + j] : draw_normal(d.seed, sim_stream(r, gs, LBBNN_MNFSIM_DRAW_EPS), (uint64_t)j);
          const float sd = sqrtf(var + sb2);
          const float a = mean + bmu + sd * ep;
          const float p = 1.0f / (1.0f + expf(-a));
          const float y = __ldg(Yb + j);
          // binary_cross_entropy: log terms clamped at -100; backward (p - y) / max(p (1 - p), 1e-12), then sigmoid's p (1 - p)
          const float li = fmaxf(logf(p), -100.f), l1 = fmaxf(log1pf(-p), -100.f);
          nll += (y - 1.0f) * l1 - y * li;
          const float dp = (p - y) / fmaxf((1.0f - p) * p, 1e-12f);
          const float da = dp * (1.0f - p) * p;
          const float dvar = da * ep * 0.5f / sd;
          dbl += da;
          dvl += dvar;
#pragma unroll
          for (int e = 0; e < kD; ++e) {
            if (e < D) {
              const float xv = __ldg(xr + e);
              aM[e] = fmaf(da, xv, aM[e]);
              aV[e] = fmaf(dvar, xv * xv, aV[e]);
            }
          }
        }
#pragma unroll
        for (int e = 0; e < kD; ++e) {
          if (e < D) {
            const float m = warp_sum(aM[e]), v = warp_sum(aV[e]);
            if (lane == 0) { S.red[warp][e] = m; S.red[warp][kD + e] = v; }
          }
        }
        nll = warp_sum(nll);
        dbl = warp_sum(dbl);
        dvl = warp_sum(dvl);
        if (lane == 0) { S.red[warp][2 * kD] = nll; S.red[warp][2 * kD + 1] = dbl; S.red[warp][2 * kD + 2] = dvl; }
      }
      __syncthreads();

      // ---- 3: KL, loss and their backward (warp 0, lane = feature) ----
      if (warp == 0) {
        const bool el = lane < D;
        const int e = el ? lane : 0;
        float dMz = 0.f, dV = 0.f, nll = 0.f, dbl = 0.f, dvl = 0.f;
        for (int q = 0; q < kWarps; ++q) {
          if (el) { dMz += S.red[q][e]; dV += S.red[q][kD + e]; }
          nll += S.red[q][2 * kD];
          dbl += S.red[q][2 * kD + 1];
          dvl += S.red[q][2 * kD + 2];
        }
        const float mu = S.lp[off_wmu(D) + e], rho = S.lp[off_wrho(D) + e], lam = S.lp[off_lam(D) + e];
        const float lv = S.lp[off_q0lv(D) + e], rc = S.lp[off_r0c(D) + e], b1 = S.lp[off_rb1(D) + e], b2 = S.lp[off_rb2(D) + e];
        const float al = alpha_of(lam), sg = sigma_of(rho);
        const float zk = S.z[0][e], z2 = S.z[1][e];
        const float ezz = S.ez[1][e];
        // weight KL with mu z2 (MNF:230-233), log q0 (MNF:212-214; (z0 - q0_mean)^2 / exp(q0_log_var) = eps^2)
        const float muz = mu * z2, dm = muz - pr.mu;
        const float slab = logf(pr.sigma / sg) - 0.5f + logf(al / pr.alpha) + (sg * sg + dm * dm) / (2.0f * pr.sigma * pr.sigma);
        const float klw = el ? al * slab + (1.0f - al) * logf((1.0f - al) / (1.0f - pr.alpha)) : 0.f;
        const float lq0 = el ? -0.5f * LOG_PI - 0.5f * lv - 0.5f * ezz * ezz : 0.f;
        // auxiliary r(z | W) (MNF:216-227) at out = 1
        const float wm = z2 * mu * al, wv = (sg * sg) * (al * al);
        const float act_mu = warp_sum(el ? rc * wm : 0.f), act_var = warp_sum(el ? rc * rc * wv : 0.f);
        const float sdr = sqrtf(act_var);
        const float ar = tanhf(act_mu + sdr * S.eps_r);
        const float mr = b1 * ar, lvr = b2 * ar, zb = S.z[2][D - 1];
        const float diff = zb - mr, elv = expf(lvr);
        const float lrb = el ? -0.5f * LOG_PI - 0.5f * lvr - 0.5f * (diff * diff) / elv : 0.f;
        const float bmu = S.lp[off_bmu(D)], brho = S.lp[off_brho(D)], sigb = S.sigb;
        const float klb = kl_bias_elem(bmu, sigb, pr);
        const float kl = (klb + warp_sum(klw)) + (warp_sum(lq0) - S.ld[1]) - (S.ld[2] + warp_sum(lrb));
        if (lane == 0) {
          float* st = d.stats + (r * steps + s) * 3;
          st[0] = nll + kl * gk;
          st[1] = nll;
          st[2] = kl;
        }
        // backward, d loss / d kl = gk
        const float u = -gk;                                               // d loss / d log r_b
        const float dlvr = el ? u * (-0.5f + 0.5f * (diff * diff) / elv) : 0.f;
        const float dmr = el ? u * diff / elv : 0.f;
        const float dzb = -warp_sum(dmr);
        const float dar = warp_sum(dmr * b1 + dlvr * b2);
        const float dpre = dar * (1.0f - ar * ar);
        const float dvar_r = dpre * S.eps_r * 0.5f / sdr;
        const float dwm = dpre * rc, dwv = dvar_r * rc * rc;
        float dmu = gk * al * dm * z2 / (pr.sigma * pr.sigma) + dwm * z2 * al + dMz * al * zk;
        float dz2 = gk * al * dm * mu / (pr.sigma * pr.sigma) + dwm * mu * al;
        float dsg = gk * al * (sg / (pr.sigma * pr.sigma) - 1.0f / sg) + (dwv + dV) * 2.0f * sg * al * al;
        float dal = gk * (slab - logf((1.0f - al) / (1.0f - pr.alpha))) + dwm * z2 * mu + (dwv + dV) * 2.0f * sg * sg * al + dMz * mu * zk;
        if (el) {
          S.gl[off_wmu(D) + e] = dmu;
          S.gl[off_wrho(D) + e] = dsg * dsigma_drho(rho);
          S.gl[off_lam(D) + e] = dal * al * (1.0f - al);
          S.gl[off_q0lv(D) + e] = -0.5f * gk;
          S.gl[off_r0c(D) + e] = dpre * wm + dvar_r * 2.0f * rc * wv;
          S.gl[off_rb1(D) + e] = dmr * ar;
          S.gl[off_rb2(D) + e] = dlvr * ar;
          S.dz[0][e] = dMz * al * mu;
          S.dz2p[e] = dz2;
          S.dz[2][e] = e == D - 1 ? dzb : 0.f;
        }
        if (lane == 0) {
          const float pbs2 = pr.bias_sigma * pr.bias_sigma;
          S.gl[off_bmu(D)] = dbl + gk * (bmu - pr.bias_mu) / pbs2;
          S.gl[off_brho(D)] = (dvl * 2.0f * sigb + gk * (sigb / pbs2 - 1.0f / sigb)) * dsigma_drho(brho);
          S.dld[0] = 0.f;
          S.dld[1] = -gk;
          S.dld[2] = -gk;
        }
      }
      __syncthreads();

      // ---- 4: flow backwards with the fused Adam ----
      flow_bwd(S, prm + roff, pm + roff, pv + roff, grow ? grow + roff : nullptr, f, 2, 1, S.step_size[11], ac);
      for (int e = tid; e < D; e += kThreads) S.dz[1][e] = S.dz2p[e] + S.dz[2][e];
      __syncthreads();
      flow_bwd(S, prm + zoff, pm + zoff, pv + zoff, grow ? grow + zoff : nullptr, f, 0, 2, S.step_size[10], ac);

      // ---- 5: q0 through the z0 draws, Adam on the layer tensors ----
      for (int e = tid; e < D; e += kThreads) {
        const float sq = sqrtf(expf(S.lp[off_q0lv(D) + e]));
        S.gl[off_q0m(D) + e] = S.dz[0][e] + S.dz[1][e];
        S.gl[off_q0lv(D) + e] += 0.5f * sq * (S.dz[0][e] * S.ez[0][e] + S.dz[1][e] * S.ez[1][e]);
      }
      __syncthreads();
      for (int e = tid; e < 8 * D + 2; e += kThreads)
        adam_el(prm, pm, pv, grow, e, S.gl[e], S.step_size[layer_group(e, D)], ac);
      __syncthreads();
    }
    if (tid == 0) d.step[r] = step0 + steps;
  }
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" int64_t lbbnn_mnfsim_param_count(int64_t in_features, int n_transforms, int n_hidden, const int* hidden) {
  if (in_features < 1 || n_transforms < 1 || n_hidden < 1 || n_hidden > LBBNN_FLOW_MAX_HIDDEN || !hidden) return -1;
  int64_t per_t = 0, prev = in_features;
  for (int l = 0; l < n_hidden; ++l) {
    if (hidden[l] < 1) return -1;
    per_t += (prev + 1) * hidden[l];
    prev = hidden[l];
  }
  per_t += 2 * (prev + 1) * in_features;
  return 8 * in_features + 2 + 2 * (int64_t)n_transforms * per_t;
}

extern "C" int lbbnn_mnfsim_train_f32(const lbbnn_mnfsim* d, int epochs, lbbnn_stream s) {
  LBBNN_REQUIRE(d, "NULL descriptor");
  LBBNN_REQUIRE(epochs >= 1, "epochs must be >= 1, got %d", epochs);
  LBBNN_REQUIRE(d->replicas >= 1 && d->replicas < (1LL << 24), "replicas must be in [1, 2^24), got %lld", (long long)d->replicas);
  LBBNN_REQUIRE(d->in_features >= 1 && d->in_features <= LBBNN_MNFSIM_MAX_IN, "in_features must be in [1, %d], got %lld",
                LBBNN_MNFSIM_MAX_IN, (long long)d->in_features);
  LBBNN_REQUIRE(d->n_transforms >= 1 && d->n_transforms <= LBBNN_MNFSIM_MAX_T, "n_transforms must be in [1, %d], got %d",
                LBBNN_MNFSIM_MAX_T, d->n_transforms);
  LBBNN_REQUIRE(d->n_hidden >= 1 && d->n_hidden <= LBBNN_FLOW_MAX_HIDDEN, "n_hidden must be in [1, %d], got %d",
                LBBNN_FLOW_MAX_HIDDEN, d->n_hidden);
  for (int l = 0; l < d->n_hidden; ++l)
    LBBNN_REQUIRE(d->hidden[l] >= 1 && d->hidden[l] <= LBBNN_MNFSIM_MAX_H, "hidden width %d must be in [1, %d], got %d", l,
                  LBBNN_MNFSIM_MAX_H, d->hidden[l]);
  LBBNN_REQUIRE(d->batch >= 1 && d->rows >= d->batch && d->rows % d->batch == 0,
                "rows (%lld) must be a positive multiple of the batch size (%lld)", (long long)d->rows, (long long)d->batch);
  LBBNN_REQUIRE(d->params && d->exp_avg && d->exp_avg_sq && d->x && d->y && d->step && d->stats,
                "NULL params, exp_avg, exp_avg_sq, x, y, step or stats");
  LBBNN_REQUIRE(d->param_stride >= lbbnn_mnfsim_param_count(d->in_features, d->n_transforms, d->n_hidden, d->hidden),
                "param_stride too small");
  LBBNN_REQUIRE(d->x_stride == 0 || d->x_stride == d->rows * d->in_features, "x_stride must be 0 (shared) or rows * in_features");
  LBBNN_REQUIRE(d->y_stride == 0 || d->y_stride == d->rows, "y_stride must be 0 (shared) or rows");
  LBBNN_REQUIRE(d->num_batches > 0.f, "num_batches must be positive");
  LBBNN_REQUIRE(d->beta1 >= 0.f && d->beta1 < 1.f && d->beta2 >= 0.f && d->beta2 < 1.f && d->adam_eps >= 0.f,
                "Adam: betas must be in [0, 1) and eps >= 0");
  const bool inj = d->eps_z != nullptr;
  LBBNN_REQUIRE((d->eps_z2 != nullptr) == inj && (d->z_masks != nullptr) == inj && (d->z_masks2 != nullptr) == inj &&
                    (d->r_masks != nullptr) == inj && (d->eps != nullptr) == inj && (d->eps_r != nullptr) == inj,
                "injected noise: give all of eps_z, eps_z2, z_masks, z_masks2, r_masks, eps, eps_r or none");
  const int64_t cap = 4LL * sm_count();
  const unsigned grid = (unsigned)(d->replicas < cap ? d->replicas : cap);
  mnfsim_train_kernel<<<grid, kThreads, 0, (cudaStream_t)s>>>(*d, epochs);
  return check_launch("mnfsim_train");
}
