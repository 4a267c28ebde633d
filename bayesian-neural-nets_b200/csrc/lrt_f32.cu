// LRT layer, fp32 SIMT path ("parity mode": matches the reference within 1e-5, TF32 never used).
//
// Replaces BayesianLinear.forward of LBBNN-GP-MF-LRT.py:166-196 (and the GEMM part of
// LBBNN-GP-MF-MNF.py:190-206) and autograd through it.
//
// Structure (r01 ncu finding: transcendental chains fused into GEMM loaders/epilogues serialise at
// 8 warps/SM; as separate elementwise passes they run at full occupancy on all SMs):
//   prologue  elementwise over (mu,rho,lambda): M = alpha mu [z], V = sigma^2 alpha^2, KL partials
//   fwd GEMM  split-K dual GEMM  E += x M^T, S += x^2 V^T  -> partials
//   fwd epi   fixed-order sum of partials, + biases, sqrt / eps / FMA (/ relu); saves
//             ds_factor = eps / (2 sqrt(var_b)) = d act / d var_b for the backward; finalises KL
//   dW GEMM   dM = dE^T x, dV = dS^T x^2 (contraction over the batch), bias column sums
//   finalize  elementwise chain rule (dM,dV) -> (dmu,drho,dlambda) + closed-form KL gradient
//   dX GEMM   split-N  dx = dE M + 2 x (dS V) -> partials; epilogue sums (+ relu mask)
#include "common.cuh"
#include "lrt_chain.cuh"

namespace lbbnn {
namespace {

constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------------------
// guarded 4-wide loads (vector when the row is 16B aligned and fully in range, else element-wise)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 load4(const float* __restrict__ base, int64_t row, int64_t col, int64_t nrows,
                                        int64_t col_end, int64_t ld, bool vec) {
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
  if (row >= nrows) return r;
  const float* p = base + row * ld + col;
  if (vec && col + 3 < col_end) {
    r = __ldg(reinterpret_cast<const float4*>(p));
  } else {
    if (col + 0 < col_end) r.x = __ldg(p + 0);
    if (col + 1 < col_end) r.y = __ldg(p + 1);
    if (col + 2 < col_end) r.z = __ldg(p + 2);
    if (col + 3 < col_end) r.w = __ldg(p + 3);
  }
  return r;
}

__device__ __forceinline__ void store4(float* __restrict__ base, int64_t row, int64_t col, int64_t nrows,
                                       int64_t ncols, int64_t ld, bool vec, float4 v) {
  if (row >= nrows) return;
  float* p = base + row * ld + col;
  if (vec && col + 3 < ncols) {
    *reinterpret_cast<float4*>(p) = v;
  } else {
    const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (col + j < ncols) p[j] = e[j];
  }
}

// flat 4-wide access with a ragged tail
__device__ __forceinline__ void loadq(const float* __restrict__ p, int64_t e0, int64_t n, bool vec, float out[4]) {
  if (vec && e0 + 3 < n) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p + e0));
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = (e0 + j < n) ? __ldg(p + e0 + j) : 0.f;
  }
}
// same, for buffers written earlier in the same launch sequence is fine too (ld.global.nc is only
// unsafe within one kernel); partial buffers are read in a later kernel than the one writing them.
__device__ __forceinline__ void storeq(float* __restrict__ p, int64_t e0, int64_t n, bool vec, const float v[4],
                                       bool accumulate) {
  if (vec && e0 + 3 < n) {
    float4 o = make_float4(v[0], v[1], v[2], v[3]);
    if (accumulate) {
      const float4 c = *reinterpret_cast<const float4*>(p + e0);
      o.x += c.x; o.y += c.y; o.z += c.z; o.w += c.w;
    }
    *reinterpret_cast<float4*>(p + e0) = o;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < n) p[e0 + j] = accumulate ? p[e0 + j] + v[j] : v[j];
  }
}

// ================================================================================================
// prologue: M, V and the KL partial sums, elementwise over the (out,in) parameters
// ================================================================================================
struct PrologueArgs {
  const float *mu, *rho, *lam, *z, *z_kl;
  int64_t n, K;
  float *M, *V;     // V may be NULL (mean branch)
  double* kl_part;  // [gridDim.x] or NULL
  int var_mode;
  lbbnn_priors pri;
};

__global__ void __launch_bounds__(kThreads) lrt_f32_prologue(const PrologueArgs a) {
  __shared__ float red[32];
  const bool vec = (a.n % 4 == 0) && (a.K % 4 == 0) && aligned16(a.mu) && aligned16(a.rho) && aligned16(a.lam) &&
                   aligned16(a.M) && (a.V == nullptr || aligned16(a.V));
  const int64_t nq = ceil_div(a.n, 4);
  float kl = 0.f;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = q * 4;
    float mu[4], rho[4], lam[4], m[4], v[4];
    loadq(a.mu, e0, a.n, vec, mu);
    loadq(a.rho, e0, a.n, vec, rho);
    loadq(a.lam, e0, a.n, vec, lam);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      m[j] = v[j] = 0.f;
      if (e0 + j < a.n) {
        const float sg = sigma_of(rho[j]), al = alpha_of(lam[j]);
        const float zk = a.z ? __ldg(a.z + (e0 + j) % a.K) : 1.0f;
        const float zkl = a.z_kl ? __ldg(a.z_kl + (e0 + j) % a.K) : zk;
        const Moments mo = weight_moments(mu[j], sg, al, a.var_mode);
        m[j] = mo.m * zk;
        v[j] = mo.v;
        if (a.kl_part) kl += kl_weight_elem(mu[j] * zkl, sg, al, a.pri);
      }
    }
    storeq(a.M, e0, a.n, vec, m, false);
    if (a.V) storeq(a.V, e0, a.n, vec, v, false);
  }
  if (a.kl_part) {
    const float s = block_sum(kl, red);
    if (threadIdx.x == 0) a.kl_part[blockIdx.x] = (double)s;
  }
}

// ---- cheaper, algebraically identical forms of the per-weight KL terms for the wide (bandwidth-bound) passes -------------
// log(alpha) = -log1p(e^-lambda), log(1 - alpha) = log(alpha) - lambda, log(alpha / (1 - alpha)) = lambda exactly: one
// log1p instead of two logs and two divisions, and no 0 * log(0) when alpha rounds to 1.
struct KlConsts {
  float log_ps, inv_2ps2, log_pa, log_1mpa, logit_pa;
};
__device__ __forceinline__ KlConsts kl_consts(const lbbnn_priors& p) {
  KlConsts c;
  c.log_ps = logf(p.sigma);
  c.inv_2ps2 = 0.5f / (p.sigma * p.sigma);
  c.log_pa = logf(p.alpha);
  c.log_1mpa = logf(1.0f - p.alpha);
  c.logit_pa = c.log_pa - c.log_1mpa;
  return c;
}
// KL of one weight (LRT:189-192) from sigma, alpha, t = e^-lambda
__device__ __forceinline__ float kl_weight_elem_shared(float mu, float sg, float al, float t, float lam, const lbbnn_priors& p,
                                                       const KlConsts& c) {
  const float d = mu - p.mu;
  const float log_al = -log1pf(t);
  const float slab = (c.log_ps - logf(sg)) - 0.5f + (log_al - c.log_pa) + (sg * sg + d * d) * c.inv_2ps2;
  return al * slab + (1.0f - al) * ((log_al - lam) - c.log_1mpa);
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// ================================================================================================
// prologue of the bf16 tensor-core path: M, V as bf16 operands (out,in) AND their (in,out) transposes, plus the KL
// partial sums, in one pass over mu, rho, lambda (replaces lrt_f32_prologue -> fp32 M, V -> bf16_pack).  64x64 tile per
// block: row-major outputs straight from registers (4 bf16 = 8 bytes per store), transposed outputs through padded
// shared-memory tiles so both directions are written in full 8-byte pieces.
// ================================================================================================
struct PrologueBf16Args {
  const float *mu, *rho, *lam;
  int64_t rows, cols;                 // (out, in)
  __nv_bfloat16 *M, *V, *MT, *VT;     // MT, VT may be NULL
  float *M32, *V32;                   // optional fp32 copies (NULL = skip)
  double* kl_part;                    // [gridDim.x * gridDim.y] or NULL
  int var_mode;
  lbbnn_priors pri;
};

__device__ __forceinline__ uint2 pack4_bf16(const float v[4]) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
  return make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
}

__global__ void __launch_bounds__(kThreads) lrt_bf16_prologue(const PrologueBf16Args a) {
  // bf16 transpose tiles (17 KB): small enough for these CTAs to share an SM with a resident tc_dual_gemm CTA (~196 KB)
  // when the trainer issues the prologues on a side stream
  __shared__ __align__(8) __nv_bfloat16 tM[64][68], tV[64][68];
  __shared__ float red[32];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t c0 = (int64_t)blockIdx.x * 64, r0 = (int64_t)blockIdx.y * 64;
  const KlConsts kc = kl_consts(a.pri);
  float kl = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = ty + 16 * i;
    const int64_t r = r0 + rl, c = c0 + tx * 4;
    float m[4] = {0.f, 0.f, 0.f, 0.f}, v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < a.rows && c < a.cols) {            // cols % 4 == 0: the quad is entirely inside the row
      const int64_t e = r * a.cols + c;
      const float4 mu = __ldg(reinterpret_cast<const float4*>(a.mu + e));
      const float4 rho = __ldg(reinterpret_cast<const float4*>(a.rho + e));
      const float4 lam = __ldg(reinterpret_cast<const float4*>(a.lam + e));
      const float muv[4] = {mu.x, mu.y, mu.z, mu.w}, rhov[4] = {rho.x, rho.y, rho.z, rho.w};
      const float lamv[4] = {lam.x, lam.y, lam.z, lam.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float sg = sigma_of(rhov[j]);
        const float t = expf(-lamv[j]), al = 1.0f / (1.0f + t);          // = alpha_of(lambda)
        const Moments mo = weight_moments(muv[j], sg, al, a.var_mode);
        m[j] = mo.m;
        v[j] = mo.v;
        if (a.kl_part) kl += kl_weight_elem_shared(muv[j], sg, al, t, lamv[j], a.pri, kc);
      }
      *reinterpret_cast<uint2*>(a.M + e) = pack4_bf16(m);
      *reinterpret_cast<uint2*>(a.V + e) = pack4_bf16(v);
      if (a.M32) *reinterpret_cast<float4*>(a.M32 + e) = make_float4(m[0], m[1], m[2], m[3]);
      if (a.V32) *reinterpret_cast<float4*>(a.V32 + e) = make_float4(v[0], v[1], v[2], v[3]);
    }
    *reinterpret_cast<uint2*>(&tM[rl][tx * 4]) = pack4_bf16(m);       // same rounding as the row-major stores
    *reinterpret_cast<uint2*>(&tV[rl][tx * 4]) = pack4_bf16(v);
  }
  if (a.MT) {
    __syncthreads();
    const bool vec = (a.rows % 4 == 0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int cl = ty + 16 * i, rl = tx * 4;           // output row = input column c, 4 consecutive r
      const int64_t c = c0 + cl, r = r0 + rl;
      if (c >= a.cols || r >= a.rows) continue;
      const __nv_bfloat16 m[4] = {tM[rl][cl], tM[rl + 1][cl], tM[rl + 2][cl], tM[rl + 3][cl]};
      const __nv_bfloat16 v[4] = {tV[rl][cl], tV[rl + 1][cl], tV[rl + 2][cl], tV[rl + 3][cl]};
      if (vec) {
        auto bits = [](const __nv_bfloat16 lo, const __nv_bfloat16 hi) {
          return (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
        };
        *reinterpret_cast<uint2*>(a.MT + c * a.rows + r) = make_uint2(bits(m[0], m[1]), bits(m[2], m[3]));
        *reinterpret_cast<uint2*>(a.VT + c * a.rows + r) = make_uint2(bits(v[0], v[1]), bits(v[2], v[3]));
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (r + j < a.rows) {
            a.MT[c * a.rows + r + j] = m[j];
            a.VT[c * a.rows + r + j] = v[j];
          }
      }
    }
  }
  if (a.kl_part) {
    const float s = block_sum(kl, red);
    if (threadIdx.x == 0) a.kl_part[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] = (double)s;
  }
}

// ================================================================================================
// forward: split-K partial dual GEMM  E = x M^T,  S = x^2 V^T
// ================================================================================================
constexpr int F_BM = 128, F_BN = 64, F_BK = 16;

struct FwdArgs {
  const float *x, *M, *V;
  int64_t B, K, N;
  int chunks_per_split, splits, sample;
  float* part;  // [splits][2][B][N]
  // optional: rows [g * rows_per_group, (g + 1) * rows_per_group) use x .* rowscale[g] in the MEAN product only (the
  // variance product keeps x^2): MNF's multiplicative z, one per stacked MC sample (MNF:197-198)
  const float* rowscale;
  int64_t rows_per_group;
};

__global__ void __launch_bounds__(kThreads, 2) lrt_f32_fwd_partial(const FwdArgs a) {
  __shared__ __align__(16) float xs[F_BK][F_BM];
  __shared__ __align__(16) float xq[F_BK][F_BM];
  __shared__ __align__(16) float ms[F_BK][F_BN];
  __shared__ __align__(16) float vs[F_BK][F_BN];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // tx: 4 output features, ty: 8 batch rows
  const int64_t n0 = (int64_t)blockIdx.x * F_BN, m0 = (int64_t)blockIdx.y * F_BM;
  const int64_t kbeg = (int64_t)blockIdx.z * a.chunks_per_split * F_BK;
  const int64_t kend = min(a.K, kbeg + (int64_t)a.chunks_per_split * F_BK);
  const bool vec = (a.K % 4 == 0) && aligned16(a.x) && aligned16(a.M) && (a.V == nullptr || aligned16(a.V));

  float accE[8][4], accS[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) accE[i][j] = accS[i][j] = 0.f;

  float4 xr[2], zr[2], pm, pv;
  const int prow = tid >> 2, pkq = (tid & 3) * 4;  // loader coordinates for the weight tiles
  const bool vecz = a.rowscale != nullptr && (a.K % 4 == 0) && aligned16(a.rowscale);
  const int64_t ngroups = a.rowscale ? ceil_div(a.B, a.rows_per_group) : 0;

  auto gload = [&](int64_t k0) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int id = tid + i * kThreads;
      xr[i] = load4(a.x, m0 + (id >> 2), k0 + (id & 3) * 4, a.B, kend, a.K, vec);
      if (a.rowscale) zr[i] = load4(a.rowscale, (m0 + (id >> 2)) / a.rows_per_group, k0 + (id & 3) * 4, ngroups, kend, a.K, vecz);
    }
    pm = load4(a.M, n0 + prow, k0 + pkq, a.N, kend, a.K, vec);
    pv = a.sample ? load4(a.V, n0 + prow, k0 + pkq, a.N, kend, a.K, vec) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  auto sstore = [&]() {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int id = tid + i * kThreads;
      const int r = id >> 2, kq = (id & 3) * 4;
      const float e[4] = {xr[i].x, xr[i].y, xr[i].z, xr[i].w};
      const float z[4] = {zr[i].x, zr[i].y, zr[i].z, zr[i].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        xs[kq + j][r] = a.rowscale ? e[j] * z[j] : e[j];
        xq[kq + j][r] = e[j] * e[j];
      }
    }
    const float m[4] = {pm.x, pm.y, pm.z, pm.w}, v[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ms[pkq + j][prow] = m[j];
      vs[pkq + j][prow] = v[j];
    }
  };

  if (kbeg < kend) {
    gload(kbeg);
    for (int64_t k0 = kbeg; k0 < kend; k0 += F_BK) {
      __syncthreads();  // previous tile fully consumed
      sstore();
      __syncthreads();
      if (k0 + F_BK < kend) gload(k0 + F_BK);  // prefetch next tile into registers
#pragma unroll
      for (int k = 0; k < F_BK; ++k) {
        const float4 a0 = *reinterpret_cast<const float4*>(&xs[k][ty * 8]);
        const float4 a1 = *reinterpret_cast<const float4*>(&xs[k][ty * 8 + 4]);
        const float4 q0 = *reinterpret_cast<const float4*>(&xq[k][ty * 8]);
        const float4 q1 = *reinterpret_cast<const float4*>(&xq[k][ty * 8 + 4]);
        const float4 bm = *reinterpret_cast<const float4*>(&ms[k][tx * 4]);
        const float4 bv = *reinterpret_cast<const float4*>(&vs[k][tx * 4]);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float qv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
        const float mv[4] = {bm.x, bm.y, bm.z, bm.w}, vv[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            accE[i][j] = fmaf(av[i], mv[j], accE[i][j]);
            accS[i][j] = fmaf(qv[i], vv[j], accS[i][j]);
          }
      }
    }
  }

  float* pe = a.part + ((int64_t)blockIdx.z * 2 + 0) * a.B * a.N;
  float* ps = a.part + ((int64_t)blockIdx.z * 2 + 1) * a.B * a.N;
  const bool vst = (a.N % 4 == 0) && aligned16(a.part);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t gm = m0 + ty * 8 + i, gn = n0 + tx * 4;
    store4(pe, gm, gn, a.B, a.N, a.N, vst, make_float4(accE[i][0], accE[i][1], accE[i][2], accE[i][3]));
    if (a.sample) store4(ps, gm, gn, a.B, a.N, a.N, vst, make_float4(accS[i][0], accS[i][1], accS[i][2], accS[i][3]));
  }
}

struct FwdEpiArgs {
  const float* part;
  int splits;
  int64_t B, N;
  const float *bias_mu, *bias_rho;
  Noise noise;
  int flags;
  float *act, *dsf, *kl_out;
  const double* kl_part;
  int n_kl_part;
  lbbnn_priors pri;
  // optional: native noise drawn per row group -- rows [g R, (g + 1) R) take stream + g * group_stride, element index
  // (row - g R) * N + col: stacked MC samples each draw what a batch-R call on their own stream would (R N % 4 == 0)
  int64_t noise_group_rows;
  uint64_t noise_group_stride;
};

constexpr int kEpiThreads = 128;

constexpr int kEpiBatch = 8;      // splits whose partial tiles are in flight together (forward: E and S of each)
__global__ void __launch_bounds__(kEpiThreads) lrt_f32_fwd_epilogue(const FwdEpiArgs a) {
  __shared__ double dred[32];
  Noise nz = a.noise;
  nz.resolve();
  const bool sample = a.flags & LBBNN_FLAG_SAMPLE;
  const int64_t total = a.B * a.N;
  const bool vec = (total % 4 == 0) && aligned16(a.part) && aligned16(a.act) && (a.dsf == nullptr || aligned16(a.dsf)) &&
                   (nz.ptr == nullptr || aligned16(nz.ptr));
  const int64_t nquads = ceil_div(total, 4);
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nquads; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = q * 4;
    float E[4] = {0.f, 0.f, 0.f, 0.f}, S[4] = {0.f, 0.f, 0.f, 0.f}, ep[4] = {0.f, 0.f, 0.f, 0.f};
    // fixed summation order over the splits; loads issued kEpiBatch splits at a time for memory parallelism: the kernel is
    // a chain of (splits / batch) L2 round trips -- 49 splits at the 784-wide layer were 13 of them (6-8 us) four at a time
    for (int s0 = 0; s0 < a.splits; s0 += kEpiBatch) {
      float pe[kEpiBatch][4], ps[kEpiBatch][4];
#pragma unroll
      for (int u = 0; u < kEpiBatch; ++u) {
        if (s0 + u < a.splits) {
          loadq(a.part + ((int64_t)(s0 + u) * 2 + 0) * total, e0, total, vec, pe[u]);
          if (sample) loadq(a.part + ((int64_t)(s0 + u) * 2 + 1) * total, e0, total, vec, ps[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < kEpiBatch; ++u) {
        if (s0 + u < a.splits) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            E[j] += pe[u][j];
            if (sample) S[j] += ps[u][j];
          }
        }
      }
    }
    const bool moments = a.flags & LBBNN_FLAG_MOMENTS;
    if (sample && !moments) {
      if (nz.ptr) loadq(nz.ptr, e0, total, vec, ep);
      else if (a.noise_group_rows > 0) {
        const int64_t per = a.noise_group_rows * a.N, g = e0 / per;      // per % 4 == 0: the quad stays inside one group
        philox_normal4(nz.seed, nz.stream + (uint64_t)g * a.noise_group_stride, (uint64_t)((e0 - g * per) >> 2), ep);
      } else philox_normal4(nz.seed, nz.stream, (uint64_t)q, ep);
    }
    float out[4], df[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      out[j] = df[j] = 0.f;
      if (e0 + j < total) {
        const int64_t n = (e0 + j) % a.N;
        float v = E[j] + __ldg(a.bias_mu + n);
        if (moments) {            // e_b and var_b themselves (LRT:172-173), no noise: act <- e_b, dsf <- var_b
          const float sb = sigma_of(__ldg(a.bias_rho + n));
          out[j] = v;
          df[j] = S[j] + sb * sb;
          continue;
        }
        if (sample) {
          const float sb = sigma_of(__ldg(a.bias_rho + n));
          const float sd = sqrtf(S[j] + sb * sb);
          v = fmaf(sd, ep[j], v);
          df[j] = ep[j] / (2.0f * sd);  // d act / d var_b  (SURVEY.md §3.5: dS = G eps / (2 sqrt S))
        }
        out[j] = (a.flags & LBBNN_FLAG_RELU) ? fmaxf(v, 0.f) : v;
      }
    }
    storeq(a.act, e0, total, vec, out, false);
    if (a.dsf && sample) storeq(a.dsf, e0, total, vec, df, false);
  }
  // KL finalisation: fixed-order sum of the prologue's per-block partials in double + the bias term
  if ((a.flags & LBBNN_FLAG_KL) && blockIdx.x == 0) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < a.n_kl_part; i += blockDim.x) acc += a.kl_part[i];
    for (int64_t n = threadIdx.x; n < a.N; n += blockDim.x)
      acc += (double)kl_bias_elem(__ldg(a.bias_mu + n), sigma_of(__ldg(a.bias_rho + n)), a.pri);
    const double tot = block_sum(acc, dred);
    if (threadIdx.x == 0) *a.kl_out = (float)tot;
  }
}

// ================================================================================================
// backward wrt parameters, GEMM part: dM = dE^T x, dV = dS^T x^2, bias column sums
// ================================================================================================
constexpr int W_BN = 32, W_BK = 64, W_BB = 16;

struct BwdWArgs {
  const float *x, *g, *dsf;
  int64_t B, K, N;
  int sample;
  float *dM, *dV;   // (N,K) each
  float* colsum;    // [2][N]: sum_b dE, sum_b dS
};

__global__ void __launch_bounds__(kThreads) lrt_f32_bwd_w_gemm(const BwdWArgs a) {
  __shared__ __align__(16) float ge[W_BB][W_BN];
  __shared__ __align__(16) float gs[W_BB][W_BN];
  __shared__ __align__(16) float xs[W_BB][W_BK];
  __shared__ __align__(16) float xq[W_BB][W_BK];

  const int tid = threadIdx.x;
  const int tk = tid & 15, tn = tid >> 4;  // thread tile: 2 n x 4 k, lanes run along k
  const int64_t n0 = (int64_t)blockIdx.x * W_BN, k0 = (int64_t)blockIdx.y * W_BK;
  const bool vecn = (a.N % 4 == 0) && aligned16(a.g) && (a.dsf == nullptr || aligned16(a.dsf));
  const bool veck = (a.K % 4 == 0) && aligned16(a.x) && aligned16(a.dM) && aligned16(a.dV);

  float accM[2][4], accV[2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) accM[i][j] = accV[i][j] = 0.f;
  float be[4] = {0.f, 0.f, 0.f, 0.f}, bs[4] = {0.f, 0.f, 0.f, 0.f};

  const int gb = tid >> 3, gq = (tid & 7) * 4;   // G loader (threads 0..127): row b, 4 columns of the n-tile
  const int xb = tid >> 4, xk = (tid & 15) * 4;  // x loader (all threads)
  float4 rg = make_float4(0.f, 0.f, 0.f, 0.f), rs = rg, rx;

  auto gload = [&](int64_t b0) {
    if (tid < 128) {
      rg = load4(a.g, b0 + gb, n0 + gq, a.B, a.N, a.N, vecn);
      rs = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.sample) {
        const float4 f = load4(a.dsf, b0 + gb, n0 + gq, a.B, a.N, a.N, vecn);
        rs = make_float4(rg.x * f.x, rg.y * f.y, rg.z * f.z, rg.w * f.w);
      }
    }
    rx = load4(a.x, b0 + xb, k0 + xk, a.B, a.K, a.K, veck);
  };

  gload(0);
  for (int64_t b0 = 0; b0 < a.B; b0 += W_BB) {
    __syncthreads();
    if (tid < 128) {
      *reinterpret_cast<float4*>(&ge[gb][gq]) = rg;
      *reinterpret_cast<float4*>(&gs[gb][gq]) = rs;
      be[0] += rg.x; be[1] += rg.y; be[2] += rg.z; be[3] += rg.w;
      bs[0] += rs.x; bs[1] += rs.y; bs[2] += rs.z; bs[3] += rs.w;
    }
    *reinterpret_cast<float4*>(&xs[xb][xk]) = rx;
    *reinterpret_cast<float4*>(&xq[xb][xk]) = make_float4(rx.x * rx.x, rx.y * rx.y, rx.z * rx.z, rx.w * rx.w);
    __syncthreads();
    if (b0 + W_BB < a.B) gload(b0 + W_BB);
#pragma unroll
    for (int b = 0; b < W_BB; ++b) {
      const float2 e2 = *reinterpret_cast<const float2*>(&ge[b][tn * 2]);
      const float2 s2 = *reinterpret_cast<const float2*>(&gs[b][tn * 2]);
      const float4 x4 = *reinterpret_cast<const float4*>(&xs[b][tk * 4]);
      const float4 q4 = *reinterpret_cast<const float4*>(&xq[b][tk * 4]);
      const float ev[2] = {e2.x, e2.y}, sv[2] = {s2.x, s2.y};
      const float xv[4] = {x4.x, x4.y, x4.z, x4.w}, qv[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          accM[i][j] = fmaf(ev[i], xv[j], accM[i][j]);
          accV[i][j] = fmaf(sv[i], qv[j], accV[i][j]);
        }
    }
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int64_t n = n0 + tn * 2 + i, kc = k0 + tk * 4;
    store4(a.dM, n, kc, a.N, a.K, a.K, veck, make_float4(accM[i][0], accM[i][1], accM[i][2], accM[i][3]));
    if (a.sample) store4(a.dV, n, kc, a.N, a.K, a.K, veck, make_float4(accV[i][0], accV[i][1], accV[i][2], accV[i][3]));
  }
  // bias column sums over the batch (k-tile 0 CTAs only)
  if (blockIdx.y == 0) {
    __syncthreads();
    if (tid < 128) {
      *reinterpret_cast<float4*>(&ge[gb][gq]) = make_float4(be[0], be[1], be[2], be[3]);
      *reinterpret_cast<float4*>(&gs[gb][gq]) = make_float4(bs[0], bs[1], bs[2], bs[3]);
    }
    __syncthreads();
    if (tid < W_BN && n0 + tid < a.N) {
      float se = 0.f, ss = 0.f;
#pragma unroll
      for (int b = 0; b < W_BB; ++b) { se += ge[b][tid]; ss += gs[b][tid]; }
      a.colsum[n0 + tid] = se;
      a.colsum[a.N + n0 + tid] = ss;
    }
  }
}

// ================================================================================================
// finalize: chain rule through M = alpha mu z, V(sigma, alpha[, mu]) + closed-form KL gradient
// ================================================================================================
struct FinalizeArgs {
  const float *mu, *rho, *lam, *z, *z_kl, *bias_mu, *bias_rho;
  const float *dM, *dV, *colsum;
  int64_t N, K;
  int var_mode, sample, accumulate;
  int bias_only;                   // skip the weights (their update ran in the dW GEMM's epilogue)
  const float* klg_dev;
  float klg_host;
  lbbnn_priors pri;
  float *dmu, *drho, *dlam, *dbmu, *dbrho, *dz, *dz_kl;
  lbbnn_adam_layer_state adam;     // ADAM variant: the gradients go straight into torch.optim.Adam's update
};

// torch.optim.Adam update of 4 consecutive elements (same expressions as adam_kernel in util.cu)
__device__ __forceinline__ void adam_quad(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v, int64_t e0,
                                          int64_t n, bool vec, const float pv[4], const float g[4], float b1, float b2,
                                          float eps, float step_size, float bc2_sqrt) {
  float mv[4], vv[4], po[4];
  loadq(m, e0, n, vec, mv);
  loadq(v, e0, n, vec, vv);
  const float inv_bc2_sqrt = 1.0f / bc2_sqrt;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    mv[j] = mv[j] + (g[j] - mv[j]) * (1.0f - b1);
    vv[j] = b2 * vv[j] + (1.0f - b2) * g[j] * g[j];
    // sqrt.approx / fast division: <= 2 ulp on a step of size ~lr, i.e. ~1e-10 of the parameter (adam_kernel keeps the
    // IEEE forms; tests bound the difference)
    po[j] = pv[j] - step_size * __fdividef(mv[j], sqrt_approx(vv[j]) * inv_bc2_sqrt + eps);
  }
  storeq(p, e0, n, vec, po, false);
  storeq(m, e0, n, vec, mv, false);
  storeq(v, e0, n, vec, vv, false);
}

// chain rule + KL gradient (+ Adam) of the 4 consecutive weights e0 .. e0 + 3; the MNF z gradients of the quad's columns
// come back in dzk / dzkl (the caller reduces them)
template <bool ADAM>
__device__ __forceinline__ void finalize_quad(const FinalizeArgs& a, int64_t e0, int64_t n, bool vec, float klg, const lbbnn_priors& P,
                                              float inv_sp2, const KlConsts& kc, float (&dzk4)[4], float (&dzkl4)[4]) {
  float mu[4], rho[4], lam[4], dM[4], dV[4] = {0.f, 0.f, 0.f, 0.f}, gm[4], gr[4], gl[4];
  loadq(a.mu, e0, n, vec, mu);
  loadq(a.rho, e0, n, vec, rho);
  loadq(a.lam, e0, n, vec, lam);
  loadq(a.dM, e0, n, vec, dM);
  if (a.sample) loadq(a.dV, e0, n, vec, dV);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    gm[j] = gr[j] = gl[j] = 0.f;
    dzk4[j] = dzkl4[j] = 0.f;
    if (e0 + j >= n) continue;
    const float er = expf(rho[j]), sg = log1pf(er);                     // = sigma_of(rho); e^rho reused for d sigma / d rho
    const float al = 1.0f / (1.0f + expf(-lam[j]));                     // = alpha_of(lambda)
    float zk = 1.0f, zkl = 1.0f;
    if (a.z || a.z_kl) {                                                // MNF only
      const int64_t k = (e0 + j) % a.K;
      zk = a.z ? __ldg(a.z + k) : 1.0f;
      zkl = a.z_kl ? __ldg(a.z_kl + k) : zk;
    }
    const float dMz = dM[j] * zk;
    float dmu = al * dMz, dsg, dal, dzk = al * mu[j] * dM[j], dzkl = 0.f;
    if (a.var_mode == LBBNN_VAR_REFERENCE) {
      dsg = 2.0f * al * al * sg * dV[j];
      dal = mu[j] * dMz + 2.0f * al * sg * sg * dV[j];
    } else {
      dmu += 2.0f * al * (1.0f - al) * mu[j] * dV[j];
      dsg = 2.0f * al * sg * dV[j];
      dal = mu[j] * dMz + (sg * sg + (1.0f - 2.0f * al) * mu[j] * mu[j]) * dV[j];
    }
    if (klg != 0.f) {
      const float d = mu[j] * zkl - P.mu;
      dmu += klg * al * d * inv_sp2 * zkl;
      dsg += klg * al * (sg * inv_sp2 - __frcp_rn(sg));
      // log(ps / sg) - 1/2 + log(al / pa) - log((1 - al) / (1 - pa)) + ...: log(al / (1 - al)) = lambda exactly
      dal += klg * ((kc.log_ps - logf(sg)) - 0.5f + (lam[j] - kc.logit_pa) + (sg * sg + d * d) * 0.5f * inv_sp2);
      dzkl = klg * al * d * inv_sp2 * mu[j];
    }
    gm[j] = dmu;
    gr[j] = dsg * (er / (1.0f + er));                                   // d sigma / d rho
    gl[j] = dal * al * (1.0f - al);
    dzk4[j] = dzk;
    dzkl4[j] = dzkl;
  }
  if (ADAM) {
    const float ss = __ldg(a.adam.coef), bc = __ldg(a.adam.coef + 1);
    const bool va = vec && aligned16(a.adam.exp_avg[0]) && aligned16(a.adam.exp_avg[1]) && aligned16(a.adam.exp_avg[2]) &&
                    aligned16(a.adam.exp_avg_sq[0]) && aligned16(a.adam.exp_avg_sq[1]) && aligned16(a.adam.exp_avg_sq[2]);
    adam_quad(const_cast<float*>(a.mu), a.adam.exp_avg[0], a.adam.exp_avg_sq[0], e0, n, va, mu, gm, a.adam.beta1, a.adam.beta2,
              a.adam.eps, ss, bc);
    adam_quad(const_cast<float*>(a.rho), a.adam.exp_avg[1], a.adam.exp_avg_sq[1], e0, n, va, rho, gr, a.adam.beta1, a.adam.beta2,
              a.adam.eps, ss, bc);
    adam_quad(const_cast<float*>(a.lam), a.adam.exp_avg[2], a.adam.exp_avg_sq[2], e0, n, va, lam, gl, a.adam.beta1, a.adam.beta2,
              a.adam.eps, ss, bc);
  } else {
    storeq(a.dmu, e0, n, vec, gm, a.accumulate);
    storeq(a.drho, e0, n, vec, gr, a.accumulate);
    storeq(a.dlam, e0, n, vec, gl, a.accumulate);
  }
}

// ZRED (MNF, K % 4 == 0): the block is a (16 rows) x (32 column quads) patch, so the z gradients -- column sums over the
// out features -- are reduced in registers and shared memory first and reach memory as ONE atomic per column and block
// (one atomic per WEIGHT serialised on the <= 784 addresses in L2: 18-26 us per layer at MNIST shape)
constexpr int kZRows = 16;
template <bool ADAM, bool ZRED>
__global__ void __launch_bounds__(kThreads) lrt_f32_finalize(const FinalizeArgs a) {
  const int64_t n = a.bias_only ? 0 : a.N * a.K;
  const bool vec = (n % 4 == 0) && (a.K % 4 == 0) && aligned16(a.mu) && aligned16(a.rho) && aligned16(a.lam) &&
                   aligned16(a.dM) && aligned16(a.dV) && aligned16(a.dmu) && aligned16(a.drho) && aligned16(a.dlam);
  const float klg = (a.klg_dev ? __ldg(a.klg_dev) : 1.0f) * a.klg_host;
  const lbbnn_priors P = a.pri;
  const float inv_sp2 = 1.0f / (P.sigma * P.sigma);
  const KlConsts kc = kl_consts(P);
  if constexpr (ZRED) {
    static_assert(kThreads == 256, "8 warps: 32 column quads x 8 row lanes");
    __shared__ float red[2][8][32][4];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int qpr = (int)(a.K >> 2), ncb = (qpr + 31) / 32;
    const int cb = blockIdx.x % ncb, rb = blockIdx.x / ncb;
    const int cq = cb * 32 + tx;
    float sk[4] = {0.f, 0.f, 0.f, 0.f}, skl[4] = {0.f, 0.f, 0.f, 0.f};
    if (cq < qpr) {
      for (int64_t r = (int64_t)rb * kZRows + ty; r < min((int64_t)(rb + 1) * kZRows, a.N); r += 8) {
        float d1[4], d2[4];
        finalize_quad<ADAM>(a, r * a.K + 4 * cq, n, vec, klg, P, inv_sp2, kc, d1, d2);
#pragma unroll
        for (int j = 0; j < 4; ++j) { sk[j] += d1[j]; skl[j] += d2[j]; }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) { red[0][ty][tx][j] = sk[j]; red[1][ty][tx][j] = skl[j]; }
    __syncthreads();
    if (threadIdx.x < 128) {
      const int c = threadIdx.x >> 2, j = threadIdx.x & 3;     // column quad, element
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) { t0 += red[0][w][c][j]; t1 += red[1][w][c][j]; }
      const int k = (cb * 32 + c) * 4 + j;
      if (k < a.K) {
        if (a.dz_kl) { atomicAdd(a.dz_kl + k, t1); if (a.dz) atomicAdd(a.dz + k, t0); }
        else if (a.dz) atomicAdd(a.dz + k, t0 + t1);
      }
    }
  } else {
    const int64_t nq = ceil_div(n, 4);
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
      const int64_t e0 = q * 4;
      float d1[4], d2[4];
      finalize_quad<ADAM>(a, e0, n, vec, klg, P, inv_sp2, kc, d1, d2);
      if (a.dz || a.dz_kl) {                                                // MNF with K % 4 != 0; caller zeroes dz / dz_kl first
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (e0 + j >= n) continue;
          const int64_t k = (e0 + j) % a.K;
          if (a.dz_kl) { atomicAdd(a.dz_kl + k, d2[j]); if (a.dz) atomicAdd(a.dz + k, d1[j]); }
          else atomicAdd(a.dz + k, d1[j] + d2[j]);
        }
      }
    }
  }
  // biases: db_mu = sum_b dE, dsigma_b = 2 sigma_b sum_b dS, + KL (LRT:185-186); block 0 after its weights, or -- the
  // bias-only launch of the fused-update path -- every block a slice (one block took 33 us for 4096 biases)
  if (blockIdx.x == 0 || a.bias_only) {
    const int64_t i0 = a.bias_only ? (int64_t)blockIdx.x * blockDim.x + threadIdx.x : threadIdx.x;
    const int64_t di = a.bias_only ? (int64_t)gridDim.x * blockDim.x : blockDim.x;
    for (int64_t i = i0; i < a.N; i += di) {
      const float bm = __ldg(a.bias_mu + i), br = __ldg(a.bias_rho + i), sb = sigma_of(br);
      float dbm = a.colsum[i], dsb = a.sample ? 2.0f * sb * a.colsum[a.N + i] : 0.f;
      if (klg != 0.f) {
        const float inv = 1.0f / (P.bias_sigma * P.bias_sigma);
        dbm += klg * (bm - P.bias_mu) * inv;
        dsb += klg * (sb * inv - 1.0f / sb);
      }
      const float dbr = dsb * dsigma_drho(br);
      if (ADAM) {
        const float ss = __ldg(a.adam.coef), bc = __ldg(a.adam.coef + 1), b1 = a.adam.beta1, b2 = a.adam.beta2;
        float m = a.adam.exp_avg[3][i], v = a.adam.exp_avg_sq[3][i];
        m = m + (dbm - m) * (1.0f - b1);
        v = b2 * v + (1.0f - b2) * dbm * dbm;
        const_cast<float*>(a.bias_mu)[i] = bm - ss * (m / (sqrtf(v) / bc + a.adam.eps));
        a.adam.exp_avg[3][i] = m; a.adam.exp_avg_sq[3][i] = v;
        m = a.adam.exp_avg[4][i]; v = a.adam.exp_avg_sq[4][i];
        m = m + (dbr - m) * (1.0f - b1);
        v = b2 * v + (1.0f - b2) * dbr * dbr;
        const_cast<float*>(a.bias_rho)[i] = br - ss * (m / (sqrtf(v) / bc + a.adam.eps));
        a.adam.exp_avg[4][i] = m; a.adam.exp_avg_sq[4][i] = v;
        continue;
      }
      a.dbmu[i] = a.accumulate ? a.dbmu[i] + dbm : dbm;
      a.dbrho[i] = a.accumulate ? a.dbrho[i] + dbr : dbr;
    }
  }
}


// ================================================================================================
// data-parallel sharded update over NVSwitch multicast (NVLS)
// ================================================================================================
// Every rank holds this layer's raw gradients [dM | dV | colsum] of ITS minibatch shard in a buffer that is mapped into a
// multicast object spanning all ranks, and so are the parameters.  Rank r owns a contiguous 1/world of the weight quads:
//   multimem.ld_reduce  sums the owners' quads of dM, dV over all ranks inside the switch (the reduce-scatter),
//   chain rule + KL gradient (added once) + Adam run on the owner (its Adam moments are the only ones ever touched),
//   multimem.st         writes the updated mu, rho, lambda quads to every rank's copy (the all-gather).
// Per rank that is 1/world of the optimiser traffic of the replicated update and (8 + 12) B / weight over NVLink instead of
// the 2 x 8 B of an all-reduce of (dM, dV) followed by a full update on every rank.  The caller brackets the launch with
// cross-rank barriers (all ranks' dW GEMMs done before; all stores landed before the parameters are read again).

struct DpUpdateArgs {
  const float *mu, *rho, *lam, *bias_mu, *bias_rho;     // this rank's copies (read)
  float *mu_mc, *rho_mc, *lam_mc, *bias_mu_mc, *bias_rho_mc;   // multicast addresses (written)
  const float* raw_mc;                                    // multicast address of [dM | dV | colsum]
  int64_t N, K;
  int world, rank, var_mode, sample;
  float klg;
  lbbnn_priors pri;
  lbbnn_adam_layer_state adam;
};

__global__ void __launch_bounds__(kThreads) lrt_f32_finalize_adam_dp_kernel(const DpUpdateArgs a) {
  const int64_t nq = a.N * a.K / 4;                        // N K % 4 == 0 (checked on the host)
  const int64_t per = ceil_div(nq, a.world), q0 = a.rank * per, q1 = min(nq, q0 + per);
  const chain::Consts cc = chain::make_consts(a.pri, a.var_mode, a.klg, a.adam.beta1, a.adam.beta2, a.adam.eps, a.adam.coef);
  const float* dM_mc = a.raw_mc;
  const float* dV_mc = a.raw_mc + a.N * a.K;
  for (int64_t q = q0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < q1; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = q * 4;
    const float4 dM = mc_ld_reduce4(dM_mc + e0);
    const float4 dV = a.sample ? mc_ld_reduce4(dV_mc + e0) : make_float4(0.f, 0.f, 0.f, 0.f);
    float mu[4], rho[4], lam[4], mm[4], mr[4], ml[4], vm[4], vr[4], vl[4];
    loadq(a.mu, e0, nq * 4, true, mu); loadq(a.rho, e0, nq * 4, true, rho); loadq(a.lam, e0, nq * 4, true, lam);
    loadq(a.adam.exp_avg[0], e0, nq * 4, true, mm); loadq(a.adam.exp_avg[1], e0, nq * 4, true, mr); loadq(a.adam.exp_avg[2], e0, nq * 4, true, ml);
    loadq(a.adam.exp_avg_sq[0], e0, nq * 4, true, vm); loadq(a.adam.exp_avg_sq[1], e0, nq * 4, true, vr);
    loadq(a.adam.exp_avg_sq[2], e0, nq * 4, true, vl);
    const float d1[4] = {dM.x, dM.y, dM.z, dM.w}, d2[4] = {dV.x, dV.y, dV.z, dV.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float gm, gr, gl;
      chain::grads(cc, mu[t], rho[t], lam[t], d1[t], d2[t], gm, gr, gl);
      chain::adam(cc, mu[t], mm[t], vm[t], gm);
      chain::adam(cc, rho[t], mr[t], vr[t], gr);
      chain::adam(cc, lam[t], ml[t], vl[t], gl);
    }
    mc_st4(a.mu_mc + e0, mu); mc_st4(a.rho_mc + e0, rho); mc_st4(a.lam_mc + e0, lam);
    storeq(a.adam.exp_avg[0], e0, nq * 4, true, mm, false); storeq(a.adam.exp_avg[1], e0, nq * 4, true, mr, false);
    storeq(a.adam.exp_avg[2], e0, nq * 4, true, ml, false);
    storeq(a.adam.exp_avg_sq[0], e0, nq * 4, true, vm, false); storeq(a.adam.exp_avg_sq[1], e0, nq * 4, true, vr, false);
    storeq(a.adam.exp_avg_sq[2], e0, nq * 4, true, vl, false);
  }
  // biases: owned by rank 0 (2 N floats of column sums reduced in the switch, then the same bias update as lrt_f32_finalize)
  if (a.rank == 0 && blockIdx.x == 0) {
    const float* cs_mc = a.raw_mc + 2 * a.N * a.K;
    const float ss = __ldg(a.adam.coef), bc = __ldg(a.adam.coef + 1), b1 = a.adam.beta1, b2 = a.adam.beta2;
    for (int64_t i = threadIdx.x; i < a.N; i += blockDim.x) {
      const float bm = a.bias_mu[i], br = a.bias_rho[i], sb = sigma_of(br);
      float dbm = mc_ld_reduce1(cs_mc + i), dsb = a.sample ? 2.0f * sb * mc_ld_reduce1(cs_mc + a.N + i) : 0.f;
      if (a.klg != 0.f) {
        const float inv = 1.0f / (a.pri.bias_sigma * a.pri.bias_sigma);
        dbm += a.klg * (bm - a.pri.bias_mu) * inv;
        dsb += a.klg * (sb * inv - 1.0f / sb);
      }
      const float dbr = dsb * dsigma_drho(br);
      float m = a.adam.exp_avg[3][i], v = a.adam.exp_avg_sq[3][i];
      m = m + (dbm - m) * (1.0f - b1);
      v = b2 * v + (1.0f - b2) * dbm * dbm;
      mc_st1(a.bias_mu_mc + i, bm - ss * (m / (sqrtf(v) / bc + a.adam.eps)));
      a.adam.exp_avg[3][i] = m; a.adam.exp_avg_sq[3][i] = v;
      m = a.adam.exp_avg[4][i]; v = a.adam.exp_avg_sq[4][i];
      m = m + (dbr - m) * (1.0f - b1);
      v = b2 * v + (1.0f - b2) * dbr * dbr;
      mc_st1(a.bias_rho_mc + i, br - ss * (m / (sqrtf(v) / bc + a.adam.eps)));
      a.adam.exp_avg[4][i] = m; a.adam.exp_avg_sq[4][i] = v;
    }
  }
}

// ================================================================================================
// backward wrt the input: dx = dE M + 2 x (dS V), split over the out-feature contraction
// ================================================================================================
constexpr int X_BM = 128, X_BK = 64, X_BN = 16;

struct BwdXArgs {
  const float *x, *g, *dsf, *M, *V;
  int64_t B, K, N;
  int chunks_per_split, splits, sample;
  float* part;  // [splits][B][K]
};

__global__ void __launch_bounds__(kThreads, 2) lrt_f32_bwd_x_partial(const BwdXArgs a) {
  __shared__ __align__(16) float ge[X_BN][X_BM];
  __shared__ __align__(16) float gs[X_BN][X_BM];
  __shared__ __align__(16) float ms[X_BN][X_BK];
  __shared__ __align__(16) float vs[X_BN][X_BK];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // tx: 4 input features, ty: 8 batch rows
  const int64_t k0 = (int64_t)blockIdx.x * X_BK, m0 = (int64_t)blockIdx.y * X_BM;
  const int64_t nbeg = (int64_t)blockIdx.z * a.chunks_per_split * X_BN;
  const int64_t nend = min(a.N, nbeg + (int64_t)a.chunks_per_split * X_BN);
  const bool vecn = (a.N % 4 == 0) && aligned16(a.g) && (a.dsf == nullptr || aligned16(a.dsf));
  const bool veck = (a.K % 4 == 0) && aligned16(a.x) && aligned16(a.M) && (a.V == nullptr || aligned16(a.V)) && aligned16(a.part);

  float accE[8][4], accS[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) accE[i][j] = accS[i][j] = 0.f;

  float4 rg[2], rs[2], pm, pv;
  const int prow = tid >> 4, pkq = (tid & 15) * 4;

  auto gload = [&](int64_t nb) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int id = tid + i * kThreads;
      const int64_t b = m0 + (id >> 2), n = nb + (id & 3) * 4;
      rg[i] = load4(a.g, b, n, a.B, nend, a.N, vecn);
      rs[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.sample) {
        const float4 f = load4(a.dsf, b, n, a.B, nend, a.N, vecn);
        rs[i] = make_float4(rg[i].x * f.x, rg[i].y * f.y, rg[i].z * f.z, rg[i].w * f.w);
      }
    }
    pm = load4(a.M, nb + prow, k0 + pkq, nend, a.K, a.K, veck);
    pv = a.sample ? load4(a.V, nb + prow, k0 + pkq, nend, a.K, a.K, veck) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  auto sstore = [&]() {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int id = tid + i * kThreads;
      const int r = id >> 2, nq = (id & 3) * 4;
      const float e[4] = {rg[i].x, rg[i].y, rg[i].z, rg[i].w}, s[4] = {rs[i].x, rs[i].y, rs[i].z, rs[i].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ge[nq + j][r] = e[j];
        gs[nq + j][r] = s[j];
      }
    }
    *reinterpret_cast<float4*>(&ms[prow][pkq]) = pm;
    *reinterpret_cast<float4*>(&vs[prow][pkq]) = pv;
  };

  if (nbeg < nend) {
    gload(nbeg);
    for (int64_t nb = nbeg; nb < nend; nb += X_BN) {
      __syncthreads();
      sstore();
      __syncthreads();
      if (nb + X_BN < nend) gload(nb + X_BN);
#pragma unroll
      for (int n = 0; n < X_BN; ++n) {
        const float4 e0 = *reinterpret_cast<const float4*>(&ge[n][ty * 8]);
        const float4 e1 = *reinterpret_cast<const float4*>(&ge[n][ty * 8 + 4]);
        const float4 s0 = *reinterpret_cast<const float4*>(&gs[n][ty * 8]);
        const float4 s1 = *reinterpret_cast<const float4*>(&gs[n][ty * 8 + 4]);
        const float4 bm = *reinterpret_cast<const float4*>(&ms[n][tx * 4]);
        const float4 bv = *reinterpret_cast<const float4*>(&vs[n][tx * 4]);
        const float ev[8] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w};
        const float sv[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float mv[4] = {bm.x, bm.y, bm.z, bm.w}, vv[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            accE[i][j] = fmaf(ev[i], mv[j], accE[i][j]);
            accS[i][j] = fmaf(sv[i], vv[j], accS[i][j]);
          }
      }
    }
  }
  float* part = a.part + (int64_t)blockIdx.z * a.B * a.K;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t b = m0 + ty * 8 + i, kc = k0 + tx * 4;
    if (b >= a.B || kc >= a.K) continue;
    const float4 x4 = load4(a.x, b, kc, a.B, a.K, a.K, veck);
    const float4 o = make_float4(fmaf(2.0f * x4.x, accS[i][0], accE[i][0]), fmaf(2.0f * x4.y, accS[i][1], accE[i][1]),
                                 fmaf(2.0f * x4.z, accS[i][2], accE[i][2]), fmaf(2.0f * x4.w, accS[i][3], accE[i][3]));
    store4(part, b, kc, a.B, a.K, a.K, veck, o);
  }
}

__global__ void __launch_bounds__(kEpiThreads) lrt_f32_bwd_x_epilogue(const float* __restrict__ part, int splits,
                                                                      int64_t total, const float* __restrict__ x,
                                                                      int mask, int accumulate, float* __restrict__ dx) {
  const bool vec = (total % 4 == 0) && aligned16(part) && aligned16(x) && aligned16(dx);
  const int64_t nq = ceil_div(total, 4);
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = q * 4;
    float s[4] = {0.f, 0.f, 0.f, 0.f}, xv[4];
    for (int s0 = 0; s0 < splits; s0 += 2 * kEpiBatch) {
      float p[2 * kEpiBatch][4];
#pragma unroll
      for (int u = 0; u < 2 * kEpiBatch; ++u)
        if (s0 + u < splits) loadq(part + (int64_t)(s0 + u) * total, e0, total, vec, p[u]);
#pragma unroll
      for (int u = 0; u < 2 * kEpiBatch; ++u)
        if (s0 + u < splits) {
#pragma unroll
          for (int j = 0; j < 4; ++j) s[j] += p[u][j];
        }
    }
    if (mask) {
      loadq(x, e0, total, vec, xv);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (!(xv[j] > 0.f)) s[j] = 0.f;
    }
    storeq(dx, e0, total, vec, s, accumulate);
  }
}

// sum of the prologue's KL partials + the bias term -> kl_out (single block, fixed order)
__global__ void __launch_bounds__(kThreads) lrt_kl_finalize(const double* __restrict__ kl_part, int n_part,
                                                            const float* __restrict__ bias_mu,
                                                            const float* __restrict__ bias_rho, int64_t N,
                                                            const lbbnn_priors pri, float* __restrict__ kl_out) {
  __shared__ double dred[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_part; i += blockDim.x) acc += kl_part[i];
  for (int64_t n = threadIdx.x; n < N; n += blockDim.x)
    acc += (double)kl_bias_elem(__ldg(bias_mu + n), sigma_of(__ldg(bias_rho + n)), pri);
  const double tot = block_sum(acc, dred);
  if (threadIdx.x == 0) *kl_out = (float)tot;
}

// ---- split heuristics (shared by the workspace query and the launchers) ----------------------------
struct Split { int chunks_per_split, splits; };

Split pick_split(int64_t tiles, int64_t chunks) {
  const int64_t target = sm_count();
  int64_t want = tiles >= target ? 1 : ceil_div(target, tiles);
  if (want > chunks / 2) want = chunks / 2;  // at least two chunks per split: keep the prefetch pipeline busy
  if (want < 1) want = 1;
  Split s;
  s.chunks_per_split = (int)ceil_div(chunks, want);
  s.splits = (int)ceil_div(chunks, s.chunks_per_split);
  if (s.splits < 1) s.splits = 1;
  return s;
}
Split fwd_split(int64_t B, int64_t K, int64_t N) {
  return pick_split(ceil_div(B, F_BM) * ceil_div(N, F_BN), ceil_div(K, F_BK));
}
Split dx_split(int64_t B, int64_t K, int64_t N) {
  return pick_split(ceil_div(B, X_BM) * ceil_div(K, X_BK), ceil_div(N, X_BN));
}

int64_t elementwise_blocks(int64_t n) {
  int64_t b = ceil_div(ceil_div(n, 4), kThreads);
  const int64_t cap = 16LL * sm_count();
  return b < 1 ? 1 : (b > cap ? cap : b);
}

size_t align_up(size_t v) { return (v + 255) & ~size_t(255); }

// workspace layout: [ M | V | kl partials | GEMM scratch (fwd partials / dM,dV,colsum / dx partials) ]
struct WsLayout {
  size_t off_m, off_v, off_kl, off_scratch, total;
};
WsLayout ws_layout(int64_t B, int64_t K, int64_t N) {
  WsLayout w;
  const size_t nk = align_up((size_t)N * K * sizeof(float));
  w.off_m = 0;
  w.off_v = nk;
  w.off_kl = 2 * nk;
  w.off_scratch = w.off_kl + align_up((size_t)elementwise_blocks(N * K) * sizeof(double));
  const size_t fwd = (size_t)fwd_split(B, K, N).splits * 2 * B * N * sizeof(float);
  const size_t dw = 2 * nk + align_up((size_t)2 * N * sizeof(float));
  const size_t dx = (size_t)dx_split(B, K, N).splits * B * K * sizeof(float);
  size_t scratch = fwd > dw ? fwd : dw;
  if (dx > scratch) scratch = dx;
  w.total = w.off_scratch + align_up(scratch) + 256;
  return w;
}

inline bool aligned16_host(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int check_layer(const lbbnn_layer* L) {
  LBBNN_REQUIRE(L != nullptr, "layer is NULL");
  LBBNN_REQUIRE(L->in_features > 0 && L->out_features > 0, "bad layer shape (%lld,%lld)", (long long)L->out_features,
                (long long)L->in_features);
  LBBNN_REQUIRE(L->weight_mu && L->weight_rho && L->lambdal && L->bias_mu && L->bias_rho, "layer has NULL parameters");
  return LBBNN_OK;
}

int launch_prologue(const lbbnn_layer* L, const lbbnn_priors* pri, int var_mode, bool want_v, bool want_kl, float* M,
                    float* V, double* kl_part, cudaStream_t st) {
  PrologueArgs pa;
  pa.mu = L->weight_mu; pa.rho = L->weight_rho; pa.lam = L->lambdal; pa.z = L->z; pa.z_kl = L->z_kl;
  pa.n = L->in_features * L->out_features; pa.K = L->in_features;
  pa.M = M; pa.V = want_v ? V : nullptr; pa.kl_part = want_kl ? kl_part : nullptr;
  pa.var_mode = var_mode; pa.pri = *pri;
  lrt_f32_prologue<<<(unsigned)elementwise_blocks(pa.n), kThreads, 0, st>>>(pa);
  return check_launch("lrt_f32_prologue");
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" size_t lbbnn_lrt_f32_workspace_bytes(int64_t B, int64_t K, int64_t N) {
  if (B <= 0 || K <= 0 || N <= 0) return 0;
  return ws_layout(B, K, N).total;
}

extern "C" size_t lbbnn_lrt_f32_mv_bytes(int64_t K, int64_t N) {
  if (K <= 0 || N <= 0) return 0;
  return 2 * align_up((size_t)N * K * sizeof(float));
}

// act[s, b, n] = [relu](e_b[b, n] + sqrt(var_b[b, n]) eps_s[b, n]) for the samples of one launch (LRT:174-175 with the e_b, var_b
// of LRT:172-173 shared by all samples of a test batch, LRT:247); eps_s from stream + s * group_stride, or injected (S, B, N)
struct ExpandArgs {
  const float *e, *var;
  int64_t total;     // B * N
  int n_samples, relu;
  Noise noise;
  uint64_t group_stride;
  float* act;
};
__global__ void __launch_bounds__(kThreads) lrt_sample_expand_kernel(const ExpandArgs a) {
  Noise nz = a.noise;
  nz.resolve();
  const int64_t nq = ceil_div(a.total, 4);
  const bool vec = (a.total % 4 == 0) && aligned16(a.e) && aligned16(a.var) && aligned16(a.act) && (nz.ptr == nullptr || aligned16(nz.ptr));
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = q * 4;
    float ev[4], sd[4];
    loadq(a.e, e0, a.total, vec, ev);
    loadq(a.var, e0, a.total, vec, sd);
#pragma unroll
    for (int j = 0; j < 4; ++j) sd[j] = sqrtf(sd[j]);
    for (int s = 0; s < a.n_samples; ++s) {
      float ep[4], out[4];
      if (nz.ptr) loadq(nz.ptr + (int64_t)s * a.total, e0, a.total, vec, ep);
      else if (a.total % 4 == 0) philox_normal4(nz.seed, nz.stream + (uint64_t)s * a.group_stride, (uint64_t)q, ep);
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j) ep[j] = philox_normal1(nz.seed, nz.stream + (uint64_t)s * a.group_stride, (uint64_t)(e0 + j));
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float v = fmaf(sd[j], ep[j], ev[j]);
        out[j] = a.relu ? fmaxf(v, 0.f) : v;
      }
      storeq(a.act + (int64_t)s * a.total, e0, a.total, vec, out, false);
    }
  }
}

extern "C" int lbbnn_lrt_sample_expand(const float* e_b, const float* var_b, int64_t batch, int64_t out_features, int n_samples,
                                       const lbbnn_noise* nz, uint64_t noise_group_stride, int flags, float* act, lbbnn_stream s) {
  LBBNN_REQUIRE(e_b && var_b && act && nz && batch > 0 && out_features > 0 && n_samples > 0, "bad argument");
  ExpandArgs a;
  a.e = e_b; a.var = var_b; a.total = batch * out_features; a.n_samples = n_samples; a.relu = (flags & LBBNN_FLAG_RELU) ? 1 : 0;
  a.noise = make_noise(nz); a.group_stride = noise_group_stride; a.act = act;
  lrt_sample_expand_kernel<<<(unsigned)elementwise_blocks(a.total), kThreads, 0, (cudaStream_t)s>>>(a);
  return check_launch("lrt_sample_expand");
}

extern "C" int lbbnn_lrt_f32_fwd_ex(const lbbnn_layer* L, const float* x, int64_t B, const lbbnn_noise* nz,
                                    const lbbnn_priors* pri, int var_mode, int flags, float* act, float* ds_factor,
                                    float* kl_out, float* mv_cache, const float* rowscale, int64_t rows_per_group,
                                    uint64_t noise_group_stride, void* ws, size_t ws_bytes, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(rows_per_group >= 0 && (rowscale == nullptr || rows_per_group > 0), "rowscale needs rows_per_group > 0");
  LBBNN_REQUIRE(!(flags & LBBNN_FLAG_MOMENTS) || ((flags & LBBNN_FLAG_SAMPLE) && ds_factor), "FLAG_MOMENTS writes var_b into ds_factor");
  LBBNN_REQUIRE(noise_group_stride == 0 || (rows_per_group > 0 && (rows_per_group * L->out_features) % 4 == 0),
                "per-group noise streams need rows_per_group * out_features %% 4 == 0");
  LBBNN_REQUIRE(x && act && B > 0, "x/act NULL or empty batch");
  LBBNN_REQUIRE(pri != nullptr, "priors NULL");
  LBBNN_REQUIRE(var_mode == LBBNN_VAR_REFERENCE || var_mode == LBBNN_VAR_EXACT, "bad var_mode %d", var_mode);
  LBBNN_REQUIRE(!(flags & LBBNN_FLAG_KL) || kl_out, "FLAG_KL needs kl_out");
  const int64_t K = L->in_features, N = L->out_features;
  const WsLayout w = ws_layout(B, K, N);
  LBBNN_REQUIRE(ws && ws_bytes >= w.total, "workspace too small (%zu < %zu)", ws_bytes, w.total);
  const bool sample = flags & LBBNN_FLAG_SAMPLE, want_kl = flags & LBBNN_FLAG_KL;
  cudaStream_t st = (cudaStream_t)s;
  char* base = (char*)ws;
  float* M = mv_cache ? mv_cache : (float*)(base + w.off_m);
  float* V = mv_cache ? (float*)((char*)mv_cache + align_up((size_t)N * K * sizeof(float))) : (float*)(base + w.off_v);
  double* kl_part = (double*)(base + w.off_kl);
  if (int rc = launch_prologue(L, pri, var_mode, sample, want_kl, M, V, kl_part, st)) return rc;

  const Split sp = fwd_split(B, K, N);
  FwdArgs fa;
  fa.x = x; fa.M = M; fa.V = sample ? V : nullptr;
  fa.B = B; fa.K = K; fa.N = N;
  fa.chunks_per_split = sp.chunks_per_split; fa.splits = sp.splits; fa.sample = sample ? 1 : 0;
  fa.part = (float*)(base + w.off_scratch);
  fa.rowscale = rowscale; fa.rows_per_group = rows_per_group;
  dim3 grid((unsigned)ceil_div(N, F_BN), (unsigned)ceil_div(B, F_BM), (unsigned)sp.splits);
  lrt_f32_fwd_partial<<<grid, kThreads, 0, st>>>(fa);
  if (int rc = check_launch("lrt_f32_fwd_partial")) return rc;

  FwdEpiArgs ea;
  ea.part = fa.part; ea.splits = sp.splits; ea.B = B; ea.N = N;
  ea.bias_mu = L->bias_mu; ea.bias_rho = L->bias_rho;
  ea.noise = make_noise(nz);
  ea.flags = flags; ea.act = act; ea.dsf = ds_factor; ea.kl_out = kl_out;
  ea.kl_part = kl_part; ea.n_kl_part = (int)elementwise_blocks(N * K); ea.pri = *pri;
  ea.noise_group_rows = noise_group_stride ? rows_per_group : 0; ea.noise_group_stride = noise_group_stride;
  int64_t blocks = ceil_div(ceil_div(B * N, 4), kEpiThreads);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  lrt_f32_fwd_epilogue<<<(unsigned)blocks, kEpiThreads, 0, st>>>(ea);
  return check_launch("lrt_f32_fwd_epilogue");
}

extern "C" int lbbnn_lrt_f32_fwd(const lbbnn_layer* L, const float* x, int64_t B, const lbbnn_noise* nz,
                                 const lbbnn_priors* pri, int var_mode, int flags, float* act, float* ds_factor,
                                 float* kl_out, float* mv_cache, void* ws, size_t ws_bytes, lbbnn_stream s) {
  return lbbnn_lrt_f32_fwd_ex(L, x, B, nz, pri, var_mode, flags & ~LBBNN_FLAG_MOMENTS, act, ds_factor, kl_out, mv_cache, nullptr, 0,
                              0, ws, ws_bytes, s);
}

namespace lbbnn {
namespace {
// parameter gradients from (dM, dV, colsum); MNF layers with in_features % 4 == 0 take the patch-shaped launch whose z
// gradients are reduced per block (see lrt_f32_finalize<., true>)
int launch_finalize(const FinalizeArgs& f, cudaStream_t st) {
  if ((f.dz || f.dz_kl) && f.K % 4 == 0 && !f.bias_only) {
    const int64_t ncb = ceil_div(f.K / 4, 32), nrb = ceil_div(f.N, kZRows);
    lrt_f32_finalize<false, true><<<(unsigned)(ncb * nrb), kThreads, 0, st>>>(f);
  } else {
    lrt_f32_finalize<false, false><<<(unsigned)elementwise_blocks(f.N * f.K), kThreads, 0, st>>>(f);
  }
  return check_launch("lrt_f32_finalize");
}
}  // namespace
}  // namespace lbbnn

extern "C" int lbbnn_lrt_f32_bwd_params(const lbbnn_layer* L, const float* x, int64_t B, const float* gact,
                                        const float* ds_factor, const lbbnn_priors* pri, int var_mode, int flags,
                                        const float* kl_grad_dev, float kl_grad_host, const lbbnn_layer_grads* G,
                                        void* ws, size_t ws_bytes, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(x && gact && B > 0 && pri && G, "NULL argument");
  LBBNN_REQUIRE(G->weight_mu && G->weight_rho && G->lambdal && G->bias_mu && G->bias_rho, "NULL gradient buffer");
  const bool sample = flags & LBBNN_FLAG_SAMPLE;
  LBBNN_REQUIRE(!sample || ds_factor, "sample-branch backward needs the saved ds_factor");
  LBBNN_REQUIRE(G->z == nullptr || L->z != nullptr, "dz requested but the layer has no z");
  LBBNN_REQUIRE(G->z_kl == nullptr || L->z_kl != nullptr, "dz_kl requested but the layer has no z_kl");
  const int64_t K = L->in_features, N = L->out_features;
  const WsLayout w = ws_layout(B, K, N);
  LBBNN_REQUIRE(ws && ws_bytes >= w.total, "workspace too small (%zu < %zu)", ws_bytes, w.total);
  cudaStream_t st = (cudaStream_t)s;
  char* scratch = (char*)ws + w.off_scratch;
  const size_t nk = align_up((size_t)N * K * sizeof(float));
  BwdWArgs a;
  a.x = x; a.g = gact; a.dsf = ds_factor; a.B = B; a.K = K; a.N = N; a.sample = sample ? 1 : 0;
  a.dM = (float*)scratch; a.dV = (float*)(scratch + nk); a.colsum = (float*)(scratch + 2 * nk);
  dim3 grid((unsigned)ceil_div(N, W_BN), (unsigned)ceil_div(K, W_BK));
  lrt_f32_bwd_w_gemm<<<grid, kThreads, 0, st>>>(a);
  if (int rc = check_launch("lrt_f32_bwd_w_gemm")) return rc;

  FinalizeArgs f;
  f.bias_only = 0;
  f.mu = L->weight_mu; f.rho = L->weight_rho; f.lam = L->lambdal; f.z = L->z; f.z_kl = L->z_kl; f.bias_mu = L->bias_mu; f.bias_rho = L->bias_rho;
  f.dM = a.dM; f.dV = a.dV; f.colsum = a.colsum; f.N = N; f.K = K;
  f.var_mode = var_mode; f.sample = sample ? 1 : 0; f.accumulate = (flags & LBBNN_FLAG_ACCUMULATE) ? 1 : 0;
  f.klg_dev = kl_grad_dev; f.klg_host = kl_grad_host; f.pri = *pri;
  f.dmu = G->weight_mu; f.drho = G->weight_rho; f.dlam = G->lambdal; f.dbmu = G->bias_mu; f.dbrho = G->bias_rho; f.dz = G->z; f.dz_kl = G->z_kl;
  return launch_finalize(f, st);
}

extern "C" int lbbnn_lrt_f32_bwd_input(const lbbnn_layer* L, const float* x, int64_t B, const float* gact,
                                       const float* ds_factor, const lbbnn_priors* pri, int var_mode, int flags,
                                       const float* mv_cache, float* dx, void* ws, size_t ws_bytes, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(x && gact && dx && B > 0 && pri, "NULL argument");
  const bool sample = flags & LBBNN_FLAG_SAMPLE;
  LBBNN_REQUIRE(!sample || ds_factor, "sample-branch backward needs the saved ds_factor");
  const int64_t K = L->in_features, N = L->out_features;
  const WsLayout w = ws_layout(B, K, N);
  LBBNN_REQUIRE(ws && ws_bytes >= w.total, "workspace too small (%zu < %zu)", ws_bytes, w.total);
  cudaStream_t st = (cudaStream_t)s;
  char* base = (char*)ws;
  const float *M, *V;
  if (mv_cache) {  // M,V kept from the forward of this step
    M = mv_cache;
    V = (const float*)((const char*)mv_cache + align_up((size_t)N * K * sizeof(float)));
  } else {         // recompute them (parameters unchanged since the forward)
    if (int rc = launch_prologue(L, pri, var_mode, sample, false, (float*)(base + w.off_m), (float*)(base + w.off_v),
                                 nullptr, st))
      return rc;
    M = (const float*)(base + w.off_m);
    V = (const float*)(base + w.off_v);
  }
  const Split sp = dx_split(B, K, N);
  BwdXArgs a;
  a.x = x; a.g = gact; a.dsf = ds_factor; a.M = M; a.V = sample ? V : nullptr;
  a.B = B; a.K = K; a.N = N;
  a.chunks_per_split = sp.chunks_per_split; a.splits = sp.splits; a.sample = sample ? 1 : 0;
  a.part = (float*)(base + w.off_scratch);
  dim3 grid((unsigned)ceil_div(K, X_BK), (unsigned)ceil_div(B, X_BM), (unsigned)sp.splits);
  lrt_f32_bwd_x_partial<<<grid, kThreads, 0, st>>>(a);
  if (int rc = check_launch("lrt_f32_bwd_x_partial")) return rc;
  int64_t blocks = ceil_div(ceil_div(B * K, 4), kEpiThreads);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  lrt_f32_bwd_x_epilogue<<<(unsigned)blocks, kEpiThreads, 0, st>>>(a.part, sp.splits, B * K, x,
                                                                  (flags & LBBNN_FLAG_MASK_DX) ? 1 : 0,
                                                                  (flags & LBBNN_FLAG_ACCUMULATE) ? 1 : 0, dx);
  return check_launch("lrt_f32_bwd_x_epilogue");
}

extern "C" int lbbnn_lrt_f32_prologue(const lbbnn_layer* L, const lbbnn_priors* pri, int var_mode, int flags, float* M,
                                      float* V, float* kl_out, void* ws, size_t ws_bytes, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(pri && M, "NULL argument");
  const bool sample = flags & LBBNN_FLAG_SAMPLE;
  LBBNN_REQUIRE(!sample || V, "sample branch needs V");
  const int64_t n = L->in_features * L->out_features;
  const size_t need = align_up((size_t)elementwise_blocks(n) * sizeof(double));
  LBBNN_REQUIRE(kl_out == nullptr || (ws && ws_bytes >= need), "workspace too small for the KL partials");
  cudaStream_t st = (cudaStream_t)s;
  if (int rc = launch_prologue(L, pri, var_mode, sample, kl_out != nullptr, M, V, (double*)ws, st)) return rc;
  if (kl_out) {
    lrt_kl_finalize<<<1, kThreads, 0, st>>>((const double*)ws, (int)elementwise_blocks(n), L->bias_mu, L->bias_rho,
                                            L->out_features, *pri, kl_out);
    return check_launch("lrt_kl_finalize");
  }
  return LBBNN_OK;
}

extern "C" int lbbnn_lrt_f32_finalize(const lbbnn_layer* L, const float* dM, const float* dV, const float* colsum,
                                      const lbbnn_priors* pri, int var_mode, int flags, const float* kl_grad_dev,
                                      float kl_grad_host, const lbbnn_layer_grads* G, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(dM && colsum && pri && G, "NULL argument");
  LBBNN_REQUIRE(G->weight_mu && G->weight_rho && G->lambdal && G->bias_mu && G->bias_rho, "NULL gradient buffer");
  const bool sample = flags & LBBNN_FLAG_SAMPLE;
  LBBNN_REQUIRE(!sample || dV, "sample branch needs dV");
  FinalizeArgs f;
  f.bias_only = 0;
  f.mu = L->weight_mu; f.rho = L->weight_rho; f.lam = L->lambdal; f.z = L->z; f.z_kl = L->z_kl; f.bias_mu = L->bias_mu; f.bias_rho = L->bias_rho;
  f.dM = dM; f.dV = dV ? dV : dM; f.colsum = colsum; f.N = L->out_features; f.K = L->in_features;
  f.var_mode = var_mode; f.sample = sample ? 1 : 0; f.accumulate = (flags & LBBNN_FLAG_ACCUMULATE) ? 1 : 0;
  f.klg_dev = kl_grad_dev; f.klg_host = kl_grad_host; f.pri = *pri;
  f.dmu = G->weight_mu; f.drho = G->weight_rho; f.dlam = G->lambdal; f.dbmu = G->bias_mu; f.dbrho = G->bias_rho; f.dz = G->z; f.dz_kl = G->z_kl;
  return launch_finalize(f, (cudaStream_t)s);
}

extern "C" int lbbnn_lrt_f32_finalize_adam(const lbbnn_layer* L, const float* dM, const float* dV, const float* colsum,
                                           const lbbnn_priors* pri, int var_mode, int flags, const float* kl_grad_dev,
                                           float kl_grad_host, const lbbnn_adam_layer_state* adam, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(dM && colsum && pri && adam && adam->coef, "NULL argument");
  LBBNN_REQUIRE(L->z == nullptr && L->z_kl == nullptr, "the fused update is for LRT layers (no multiplicative z)");
  for (int i = 0; i < 5; ++i) LBBNN_REQUIRE(adam->exp_avg[i] && adam->exp_avg_sq[i], "NULL Adam state %d", i);
  const bool sample = flags & LBBNN_FLAG_SAMPLE;
  LBBNN_REQUIRE(!sample || dV, "sample branch needs dV");
  FinalizeArgs f;
  f.bias_only = 0;
  f.mu = L->weight_mu; f.rho = L->weight_rho; f.lam = L->lambdal; f.z = nullptr; f.z_kl = nullptr; f.bias_mu = L->bias_mu; f.bias_rho = L->bias_rho;
  f.dM = dM; f.dV = dV ? dV : dM; f.colsum = colsum; f.N = L->out_features; f.K = L->in_features;
  f.var_mode = var_mode; f.sample = sample ? 1 : 0; f.accumulate = 0;
  f.klg_dev = kl_grad_dev; f.klg_host = kl_grad_host; f.pri = *pri;
  f.dmu = f.drho = f.dlam = f.dbmu = f.dbrho = f.dz = f.dz_kl = nullptr;
  f.adam = *adam;
  lrt_f32_finalize<true, false><<<(unsigned)elementwise_blocks(f.N * f.K), kThreads, 0, (cudaStream_t)s>>>(f);
  return check_launch("lrt_f32_finalize_adam");
}

extern "C" int lbbnn_lrt_kl_finalize(const double* kl_part, int64_t n_part, const lbbnn_layer* L, const lbbnn_priors* pri,
                                     float* kl_out, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(kl_part && pri && kl_out && n_part > 0 && n_part < (1LL << 31), "bad argument");
  lrt_kl_finalize<<<1, kThreads, 0, (cudaStream_t)s>>>(kl_part, (int)n_part, L->bias_mu, L->bias_rho, L->out_features, *pri, kl_out);
  return check_launch("lrt_kl_finalize");
}

extern "C" int lbbnn_lrt_f32_finalize_adam_bias(const lbbnn_layer* L, const float* colsum, const lbbnn_priors* pri, int flags,
                                                float kl_grad_host, const lbbnn_adam_layer_state* adam, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(colsum && pri && adam && adam->coef, "NULL argument");
  for (int i = 3; i < 5; ++i) LBBNN_REQUIRE(adam->exp_avg[i] && adam->exp_avg_sq[i], "NULL Adam state %d", i);
  FinalizeArgs f;
  f.bias_only = 1;
  f.mu = L->weight_mu; f.rho = L->weight_rho; f.lam = L->lambdal; f.z = nullptr; f.z_kl = nullptr; f.bias_mu = L->bias_mu; f.bias_rho = L->bias_rho;
  f.dM = nullptr; f.dV = nullptr; f.colsum = colsum; f.N = L->out_features; f.K = L->in_features;
  f.var_mode = 0; f.sample = (flags & LBBNN_FLAG_SAMPLE) ? 1 : 0; f.accumulate = 0;
  f.klg_dev = nullptr; f.klg_host = kl_grad_host; f.pri = *pri;
  f.dmu = f.drho = f.dlam = f.dbmu = f.dbrho = f.dz = f.dz_kl = nullptr;
  f.adam = *adam;
  lrt_f32_finalize<true, false><<<(unsigned)ceil_div(f.N, kThreads), kThreads, 0, (cudaStream_t)s>>>(f);
  return check_launch("lrt_f32_finalize_adam_bias");
}

extern "C" int lbbnn_lrt_f32_finalize_adam_dp(const lbbnn_layer* L, const lbbnn_dp_layer* dp, const lbbnn_priors* pri, int var_mode,
                                              int flags, float kl_grad_host, const lbbnn_adam_layer_state* adam, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(dp && pri && adam && adam->coef, "NULL argument");
  LBBNN_REQUIRE(dp->world >= 1 && dp->rank >= 0 && dp->rank < dp->world, "bad rank %d of %d", dp->rank, dp->world);
  LBBNN_REQUIRE(dp->raw_mc && dp->weight_mu_mc && dp->weight_rho_mc && dp->lambdal_mc && dp->bias_mu_mc && dp->bias_rho_mc,
                "NULL multicast address");
  LBBNN_REQUIRE(L->z == nullptr && L->z_kl == nullptr, "the fused update is for LRT layers (no multiplicative z)");
  LBBNN_REQUIRE((L->in_features * L->out_features) % 4 == 0, "in_features * out_features must be a multiple of 4");
  for (int i = 0; i < 5; ++i) LBBNN_REQUIRE(adam->exp_avg[i] && adam->exp_avg_sq[i], "NULL Adam state %d", i);
  const void* al[] = {L->weight_mu, L->weight_rho, L->lambdal, dp->raw_mc, dp->weight_mu_mc, dp->weight_rho_mc, dp->lambdal_mc,
                      adam->exp_avg[0], adam->exp_avg[1], adam->exp_avg[2], adam->exp_avg_sq[0], adam->exp_avg_sq[1], adam->exp_avg_sq[2]};
  for (const void* p : al) LBBNN_REQUIRE((reinterpret_cast<uintptr_t>(p) & 15) == 0, "weight tensors / raw gradients must be 16B aligned");
  DpUpdateArgs a;
  a.mu = L->weight_mu; a.rho = L->weight_rho; a.lam = L->lambdal; a.bias_mu = L->bias_mu; a.bias_rho = L->bias_rho;
  a.mu_mc = dp->weight_mu_mc; a.rho_mc = dp->weight_rho_mc; a.lam_mc = dp->lambdal_mc; a.bias_mu_mc = dp->bias_mu_mc;
  a.bias_rho_mc = dp->bias_rho_mc; a.raw_mc = dp->raw_mc;
  a.N = L->out_features; a.K = L->in_features; a.world = dp->world; a.rank = dp->rank; a.var_mode = var_mode;
  a.sample = (flags & LBBNN_FLAG_SAMPLE) ? 1 : 0; a.klg = kl_grad_host; a.pri = *pri; a.adam = *adam;
  const int64_t shard = ceil_div(a.N * a.K / 4, (int64_t)dp->world);
  lrt_f32_finalize_adam_dp_kernel<<<(unsigned)elementwise_blocks(shard * 4), kThreads, 0, (cudaStream_t)s>>>(a);
  return check_launch("lrt_f32_finalize_adam_dp");
}

// ---- plain linear layer on the same kernels (mean-branch GEMM: E only) ---------------------------------
extern "C" int lbbnn_linear_f32_fwd(const float* x, const float* W, const float* bias, int64_t B, int64_t K, int64_t N,
                                    int flags, float* out, void* ws, size_t ws_bytes, lbbnn_stream s) {
  LBBNN_REQUIRE(x && W && bias && out && B > 0 && K > 0 && N > 0, "NULL argument");
  const WsLayout w = ws_layout(B, K, N);
  LBBNN_REQUIRE(ws && ws_bytes >= w.total, "workspace too small (%zu < %zu)", ws_bytes, w.total);
  cudaStream_t st = (cudaStream_t)s;
  const Split sp = fwd_split(B, K, N);
  FwdArgs fa;
  fa.x = x; fa.M = W; fa.V = nullptr; fa.B = B; fa.K = K; fa.N = N;
  fa.chunks_per_split = sp.chunks_per_split; fa.splits = sp.splits; fa.sample = 0;
  fa.part = (float*)((char*)ws + w.off_scratch);
  dim3 grid((unsigned)ceil_div(N, F_BN), (unsigned)ceil_div(B, F_BM), (unsigned)sp.splits);
  lrt_f32_fwd_partial<<<grid, kThreads, 0, st>>>(fa);
  if (int rc = check_launch("lrt_f32_fwd_partial")) return rc;
  FwdEpiArgs ea;
  ea.part = fa.part; ea.splits = sp.splits; ea.B = B; ea.N = N; ea.bias_mu = bias; ea.bias_rho = bias;
  ea.noise = make_noise(nullptr); ea.flags = flags & LBBNN_FLAG_RELU; ea.act = out; ea.dsf = nullptr; ea.kl_out = nullptr;
  ea.kl_part = nullptr; ea.n_kl_part = 0; ea.pri = lbbnn_priors{0.f, 1.f, 0.5f, 0.f, 1.f};
  int64_t blocks = ceil_div(ceil_div(B * N, 4), kEpiThreads);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  lrt_f32_fwd_epilogue<<<(unsigned)blocks, kEpiThreads, 0, st>>>(ea);
  return check_launch("lrt_f32_fwd_epilogue");
}

extern "C" int lbbnn_linear_f32_bwd_params(const float* x, const float* gout, int64_t B, int64_t K, int64_t N, float* dW,
                                           float* dbias, void* ws, size_t ws_bytes, lbbnn_stream s) {
  LBBNN_REQUIRE(x && gout && dW && dbias && B > 0 && K > 0 && N > 0, "NULL argument");
  LBBNN_REQUIRE(ws && ws_bytes >= (size_t)2 * N * sizeof(float), "workspace too small");
  BwdWArgs a;
  a.x = x; a.g = gout; a.dsf = nullptr; a.B = B; a.K = K; a.N = N; a.sample = 0;
  a.dM = dW; a.dV = dW; a.colsum = (float*)ws;
  dim3 grid((unsigned)ceil_div(N, W_BN), (unsigned)ceil_div(K, W_BK));
  lrt_f32_bwd_w_gemm<<<grid, kThreads, 0, (cudaStream_t)s>>>(a);
  if (int rc = check_launch("lrt_f32_bwd_w_gemm")) return rc;
  LBBNN_CUDA(cudaMemcpyAsync(dbias, ws, (size_t)N * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)s));
  return LBBNN_OK;
}

extern "C" int lbbnn_linear_f32_bwd_input(const float* x, const float* W, const float* gout, int64_t B, int64_t K,
                                          int64_t N, int flags, float* dx, void* ws, size_t ws_bytes, lbbnn_stream s) {
  LBBNN_REQUIRE(x && W && gout && dx && B > 0 && K > 0 && N > 0, "NULL argument");
  const WsLayout w = ws_layout(B, K, N);
  LBBNN_REQUIRE(ws && ws_bytes >= w.total, "workspace too small");
  const Split sp = dx_split(B, K, N);
  BwdXArgs a;
  a.x = x; a.g = gout; a.dsf = nullptr; a.M = W; a.V = nullptr; a.B = B; a.K = K; a.N = N;
  a.chunks_per_split = sp.chunks_per_split; a.splits = sp.splits; a.sample = 0;
  a.part = (float*)((char*)ws + w.off_scratch);
  dim3 grid((unsigned)ceil_div(K, X_BK), (unsigned)ceil_div(B, X_BM), (unsigned)sp.splits);
  lrt_f32_bwd_x_partial<<<grid, kThreads, 0, (cudaStream_t)s>>>(a);
  if (int rc = check_launch("lrt_f32_bwd_x_partial")) return rc;
  int64_t blocks = ceil_div(ceil_div(B * K, 4), kEpiThreads);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  lrt_f32_bwd_x_epilogue<<<(unsigned)blocks, kEpiThreads, 0, (cudaStream_t)s>>>(a.part, sp.splits, B * K, x,
                                                                  (flags & LBBNN_FLAG_MASK_DX) ? 1 : 0, 0, dx);
  return check_launch("lrt_f32_bwd_x_epilogue");
}

extern "C" size_t lbbnn_lrt_bf16_prologue_workspace_bytes(int64_t in_features, int64_t out_features) {
  if (in_features <= 0 || out_features <= 0) return 0;
  return align_up((size_t)(ceil_div(in_features, 64) * ceil_div(out_features, 64)) * sizeof(double));
}

static int bf16_prologue_impl(const lbbnn_layer* L, const lbbnn_priors* pri, int var_mode, void* M_bf, void* V_bf,
                              void* MT_bf, void* VT_bf, float* M32, float* V32, float* kl_out, bool kl_parts_only, void* ws,
                              size_t ws_bytes, lbbnn_stream s);

extern "C" int lbbnn_lrt_bf16_prologue(const lbbnn_layer* L, const lbbnn_priors* pri, int var_mode, void* M_bf, void* V_bf,
                                       void* MT_bf, void* VT_bf, float* M32, float* V32, float* kl_out, void* ws,
                                       size_t ws_bytes, lbbnn_stream s) {
  return bf16_prologue_impl(L, pri, var_mode, M_bf, V_bf, MT_bf, VT_bf, M32, V32, kl_out, false, ws, ws_bytes, s);
}

extern "C" size_t lbbnn_lrt_bf16_prologue_kl_parts(int64_t in_features, int64_t out_features) {
  return (size_t)(ceil_div(in_features, 64) * ceil_div(out_features, 64));
}

extern "C" int lbbnn_lrt_bf16_prologue_parts(const lbbnn_layer* L, const lbbnn_priors* pri, int var_mode, void* M_bf, void* V_bf,
                                             float* M32, float* V32, void* ws, size_t ws_bytes, lbbnn_stream s) {
  LBBNN_REQUIRE(ws != nullptr, "the KL partials need the workspace");
  return bf16_prologue_impl(L, pri, var_mode, M_bf, V_bf, nullptr, nullptr, M32, V32, nullptr, true, ws, ws_bytes, s);
}

static int bf16_prologue_impl(const lbbnn_layer* L, const lbbnn_priors* pri, int var_mode, void* M_bf, void* V_bf,
                              void* MT_bf, void* VT_bf, float* M32, float* V32, float* kl_out, bool kl_parts_only, void* ws,
                              size_t ws_bytes, lbbnn_stream s) {
  if (int rc = check_layer(L)) return rc;
  LBBNN_REQUIRE(pri && M_bf && V_bf, "NULL argument");
  LBBNN_REQUIRE((MT_bf == nullptr) == (VT_bf == nullptr), "transposed outputs come in pairs");
  LBBNN_REQUIRE(L->z == nullptr && L->z_kl == nullptr, "the bf16 prologue has no MNF z path");
  const int64_t K = L->in_features, N = L->out_features;
  LBBNN_REQUIRE(K % 4 == 0, "in_features must be a multiple of 4 (got %lld)", (long long)K);
  LBBNN_REQUIRE(aligned16_host(L->weight_mu) && aligned16_host(L->weight_rho) && aligned16_host(L->lambdal) &&
                    aligned16_host(M_bf) && aligned16_host(V_bf) && aligned16_host(MT_bf) && aligned16_host(VT_bf) &&
                    aligned16_host(M32) && aligned16_host(V32),
                "parameters and outputs must be 16-byte aligned");
  dim3 grid((unsigned)ceil_div(K, 64), (unsigned)ceil_div(N, 64));
  LBBNN_REQUIRE(grid.y <= 65535, "too many output features for one launch");
  const size_t need = lbbnn_lrt_bf16_prologue_workspace_bytes(K, N);
  LBBNN_REQUIRE((kl_out == nullptr && !kl_parts_only) || (ws && ws_bytes >= need), "workspace too small for the KL partials");
  cudaStream_t st = (cudaStream_t)s;
  PrologueBf16Args pa;
  pa.mu = L->weight_mu; pa.rho = L->weight_rho; pa.lam = L->lambdal; pa.rows = N; pa.cols = K;
  pa.M = (__nv_bfloat16*)M_bf; pa.V = (__nv_bfloat16*)V_bf; pa.MT = (__nv_bfloat16*)MT_bf; pa.VT = (__nv_bfloat16*)VT_bf;
  pa.M32 = M32; pa.V32 = V32; pa.kl_part = (kl_out || kl_parts_only) ? (double*)ws : nullptr; pa.var_mode = var_mode; pa.pri = *pri;
  lrt_bf16_prologue<<<grid, kThreads, 0, st>>>(pa);
  if (int rc = check_launch("lrt_bf16_prologue")) return rc;
  if (kl_out) {
    lrt_kl_finalize<<<1, kThreads, 0, st>>>((const double*)ws, (int)(grid.x * grid.y), L->bias_mu, L->bias_rho, N, *pri, kl_out);
    return check_launch("lrt_kl_finalize");
  }
  return LBBNN_OK;
}
