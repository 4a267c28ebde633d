// Whole training step of a small LRT stack as ONE persistent cooperative kernel (fp32, parity mode).
//
// Replaces the body of `train` for one minibatch (LBBNN-GP-MF-LRT.py:217-229): net(data, sample=True)
// (LRT:166-211), nll_loss(sum) + kl/NUM_BATCHES (LRT:223-224), backward, optim.Adam.step (LRT:358).
//
// Why one kernel: at MNIST shape / batch 100 a step is 546 MFLOP over ~20 MB of parameters that stay in the
// 126 MB L2; as ~20 separate launches the step is bound by launch + drain latency (r01 ncu: every kernel
// 5-15 us for < 2 us of work).  Here one CTA per SM runs all phases and meets the others at grid barriers:
//
//   F_l   split-K dual GEMM  E = x M^T, S = x^2 V^T; M = alpha mu, V = sigma^2 alpha^2 are computed in the weight
//         loader (each weight element is used by exactly one tile since batch <= 128), x^2 in registers
//   Fe_l  fixed-order sum of the split partials + biases + eps/sqrt/FMA + relu -> act_l, ds_factor_l
//         (last layer: log_softmax + nll + dlogits -> dE_L, dS_L, one warp per row)
//   B_l   dW tiles (dM = dE^T x, dV = dS^T x^2, contraction over the batch; bias column sums) and, on other
//         CTAs of the same phase, dX tiles (dx = dE M + 2 x (dS V), split over the out-feature contraction)
//   Xe_l  (only when dX was split) sum of the dX partials + relu mask -> dE_{l-1}, dS_{l-1}
//   U     elementwise over all parameters: chain rule (dM,dV) -> (dmu,drho,dlambda), closed-form KL gradient
//         and KL value (they share their logs), Adam update; gradients are only written out on request
//
// Every GEMM phase uses the same register-tiled routine: 4x8 outputs per thread for both products, thread
// groups split the contraction inside the CTA and are summed through shared memory in a fixed order, so results
// are deterministic.  Data-parallel training runs phases F..B in one launch, all-reduces the raw (dM, dV, colsum)
// buffer, and runs U as a second launch of the same kernel.
#pragma once
#include <cooperative_groups.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <initializer_list>
#include <cmath>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace lbbnn {
namespace {

#ifndef LBBNN_STEP_NT
#define LBBNN_STEP_NT 256
#endif
constexpr int NT = LBBNN_STEP_NT;            // threads per CTA
constexpr int kCtasPerSm = NT >= 512 ? 1 : 512 / NT;  // 512 threads per SM: 1 CTA of 512 or 2 CTAs of 256
constexpr int kMaxL = LBBNN_STEP_MAX_LAYERS;
constexpr size_t kSmemCap = 200 * 1024 / kCtasPerSm;  // per CTA = (kWOff + kWFloats) floats, see below

// Tile geometry of one GEMM phase of one layer, computed on the host for the FULL tile (edge tiles are zero-padded in
// shared memory and clipped on output): R rows x C columns per CTA, contraction chunk KC split over G thread groups.
struct TileCfg {
  int R, C, RP, CP, CG, TPG, G, kpg, KC, KS;  // KS = G * kpg >= KC: contraction extent of the smem tiles (zero-filled)
};

inline TileCfg make_cfg(int R, int C, int KC, int nt) {
  TileCfg t;
  t.R = R; t.C = C; t.KC = KC;
  t.RP = (R + 3) & ~3;
  t.CP = (C + 7) & ~7;
  t.CG = t.CP >> 3;
  t.TPG = (t.RP >> 2) * t.CG;
  int g = nt / t.TPG;
  if (g > 8) g = 8;  // the group reduction is one shared-memory round for G <= 8
  if (g > KC) g = KC;
  if (g < 1) g = 1;
  t.kpg = ((KC + g - 1) / g + 3) & ~3;  // multiple of 4: the MAC loop runs 4 contraction steps per trip
  t.G = (KC + t.kpg - 1) / t.kpg;
  t.KS = t.G * t.kpg;
  return t;
}

struct DevLayer {
  TileCfg fc, wc, xc;
  int K, N;
  int64_t off_mu, off_rho, off_lam, off_bmu, off_brho;
  float *dM, *dV, *colsum;     // raw gradients of the weight moments / bias column sums
  float *act, *dsf, *dE, *dS;  // (B,N)
  const float* eps;            // injected noise or NULL
  lbbnn_priors pri;
  int var_mode;
  int f_bn, f_kc, f_ntiles, f_splits;
  int w_rn, w_ck, w_rtiles, w_ctiles;
  int x_bk, x_nc, x_ctiles, x_splits;
};

struct DevStep {
  int L, B, phases, nll_ctas;
  int overlap_update;   // experimental (LBBNN_STEP_OVERLAP_UPDATE=1): see the kernel; measured slower on B200, off
  int small_last;   // the last layer is a small classifier (N <= 32): dedicated forward+loss and backward phases
  float* mv_last;   // its M and V, (2, N, K), computed once per launch
  DevLayer ly[kMaxL];
  float *flat, *m, *v, *grad;
  const float* x;
  const int64_t* y;
  float* part;
  double* kl_part;
  float* nll_part;
  unsigned* ticket;
  int64_t* step_dev;
  uint64_t seed;
  float lr, b1, b2, eps, klg;
  float* stats;
  long long* prof;  // optional: clock64 of CTA 0 at every phase boundary
  int prof_cta;     // CTA whose work items are stamped
  // data parallel inside the launch (lbbnn_step_dp): world > 1 switches it on
  int dp_world, dp_rank;
  float* flat_mc;
  const float* raw_mc;       // multicast address of the workspace head = the raw gradients of all layers
  const float* raw_base;     // local address of the same
  unsigned* dp_signal[8];
  double* dp_klx[8];
  unsigned long long* dp_epoch;
  int dp_p2p;                // peer-to-peer loads / stores instead of the multicast object
  float* flat_peer[8];
  const float* raw_peer[8];
  // replica launch (lbbnn_lrt_step_replicas_f32, the REP instantiation): R networks of one shape; replica r's parameters,
  // Adam state and gradients sit r * p_stride floats, its minibatch r * x_stride / y_stride elements and its workspace block
  // r * w_stride floats after replica 0's.  Every pointer above (and every DevLayer pointer) is replica 0's.
  int R;
  int64_t p_stride, x_stride, y_stride, w_stride;
  const uint64_t* seeds;     // device, R: replica r's Philox key
};

// Replica launch: REP ? <replica r's address / index> : <the single network's>.  The single-network instantiation keeps the
// second form verbatim, so it compiles from exactly the code it had before the replica axis existed.
#define REP_SEL(rep_form, single_form) (REP ? (rep_form) : (single_form))

// ---- NVLink flags / NVSwitch multicast (data parallel inside the launch) -------------------------------------------------
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// one thread: tell every peer this rank reached `epoch`, wait until all of them did
__device__ __forceinline__ void dp_flag_exchange(const DevStep& a, unsigned epoch) {
  __threadfence_system();
  for (int p = 0; p < a.dp_world; ++p) st_release_sys(a.dp_signal[p] + a.dp_rank, epoch);
  for (int q = 0; q < a.dp_world; ++q)
    while ((int)(ld_acquire_sys(a.dp_signal[a.dp_rank] + q) - epoch) < 0) {}
}

__device__ __forceinline__ void stamp(const DevStep& a, int& slot) {
  if (a.prof && (int)blockIdx.x == a.prof_cta && threadIdx.x == 0) a.prof[slot] = clock64();
  ++slot;
}

#define SUBSTAMP(a, idx) do { if ((a).prof && blockIdx.x == 0 && threadIdx.x == 0) (a).prof[40 + (idx)] = clock64(); } while (0)
#define ITEMSTAMP(a, base, l, idx) do { if ((a).prof && blockIdx.x == (a).prof_cta && threadIdx.x == 0) (a).prof[(base) + (l) * 8 + (idx)] = clock64(); } while (0)

// ---- guarded 4-wide global loads ----------------------------------------------------------------------
// COH: the buffer was written earlier in this launch by other CTAs -> L2-coherent load; else read-only path.
template <bool COH>
__device__ __forceinline__ float ld1(const float* p) { return COH ? __ldcg(p) : __ldg(p); }

template <bool COH>
__device__ __forceinline__ float4 ldrow4(const float* __restrict__ base, int64_t row, int64_t col, int64_t nrows,
                                         int64_t col_end, int64_t ld, bool vec) {
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
  if (row >= nrows || col >= col_end) return r;
  const float* p = base + row * ld + col;
  if (vec && col + 3 < col_end) {
    r = COH ? __ldcg(reinterpret_cast<const float4*>(p)) : __ldg(reinterpret_cast<const float4*>(p));
  } else {
    r.x = ld1<COH>(p);
    if (col + 1 < col_end) r.y = ld1<COH>(p + 1);
    if (col + 2 < col_end) r.z = ld1<COH>(p + 2);
    if (col + 3 < col_end) r.w = ld1<COH>(p + 3);
  }
  return r;
}

// ---- the register-tiled dual MAC ----------------------------------------------------------------------
// acc1[i][j] += A1[k][row i] * B1[k][col j], acc2 likewise with A2/B2 (or the squares of A1 / B1), for k in [kb, ke),
// ke - kb a multiple of 4.  Thread (rg, cg) owns rows rg*4..+3 and columns {cg*4..+3} U {CP/2 + cg*4..+3} (two float4
// per operand row, each contiguous across the threads of a warp: conflict-free LDS.128).
template <bool SQ_A, bool SQ_B>
__device__ __forceinline__ void tile_mac(const float* __restrict__ A1, const float* __restrict__ A2,
                                         const float* __restrict__ B1, const float* __restrict__ B2, const TileCfg& t,
                                         int kb, int ke, int rg, int cgi, float (&acc1)[4][8], float (&acc2)[4][8]) {
  const int cph = t.CP >> 1;
  const float* a1p = A1 + rg * 4 + kb * t.RP;
  const float* a2p = A2 + rg * 4 + kb * t.RP;
  const float* b1p = B1 + cgi * 4 + kb * t.CP;
  const float* b2p = B2 + cgi * 4 + kb * t.CP;
  for (int k = kb; k < ke; k += 4) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(a1p + kk * t.RP);
      float4 a2;
      if (SQ_A) a2 = make_float4(a.x * a.x, a.y * a.y, a.z * a.z, a.w * a.w);
      else a2 = *reinterpret_cast<const float4*>(a2p + kk * t.RP);
      const float4 b0 = *reinterpret_cast<const float4*>(b1p + kk * t.CP);
      const float4 b1 = *reinterpret_cast<const float4*>(b1p + kk * t.CP + cph);
      float4 c0, c1;
      if (SQ_B) {
        c0 = make_float4(b0.x * b0.x, b0.y * b0.y, b0.z * b0.z, b0.w * b0.w);
        c1 = make_float4(b1.x * b1.x, b1.y * b1.y, b1.z * b1.z, b1.w * b1.w);
      } else {
        c0 = *reinterpret_cast<const float4*>(b2p + kk * t.CP);
        c1 = *reinterpret_cast<const float4*>(b2p + kk * t.CP + cph);
      }
      const float av[4] = {a.x, a.y, a.z, a.w}, qv[4] = {a2.x, a2.y, a2.z, a2.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      const float cv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc1[i][j] = fmaf(av[i], bv[j], acc1[i][j]);
          acc2[i][j] = fmaf(qv[i], cv[j], acc2[i][j]);
        }
    }
    a1p += 4 * t.RP; a2p += 4 * t.RP; b1p += 4 * t.CP; b2p += 4 * t.CP;
  }
}

// Linear index -> (lo, hi) = (idx % m, idx / m) walked incrementally: one division per loop instead of per element.
struct Walk {
  int lo, hi, dlo, dhi, m;
  __device__ __forceinline__ Walk(int start, int stride, int mod) : m(mod) {
    lo = start % mod; hi = start / mod; dlo = stride % mod; dhi = stride / mod;
  }
  __device__ __forceinline__ void next() {
    lo += dlo; hi += dhi;
    if (lo >= m) { lo -= m; ++hi; }
  }
};

// Sum the accumulators of the G contraction groups into group 0's registers through shared memory, in a fixed order
// (deterministic): G <= 8: groups 1.. write once, group 0 adds them in order (2 barriers); larger G: a binary tree
// (upper half writes, lower half adds).  NW = 1: only acc1 is live.  Ends with a __syncthreads(): `red` is free.
template <int NW>
__device__ __forceinline__ void reduce_groups(float* __restrict__ red, const TileCfg& t, int g, int tg,
                                              float (&acc1)[4][8], float (&acc2)[4][8]) {
  constexpr int NACC = NW * 32;
  if (t.G == 1) return;
  __syncthreads();  // every thread is done reading the operand tiles that `red` aliases
  if (t.G <= 8) {
    if (g >= 1 && g < t.G) {
      float* dst = red + (g - 1) * NACC * t.TPG + tg;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          dst[(i * 8 + j) * t.TPG] = acc1[i][j];
          if (NW == 2) dst[(32 + i * 8 + j) * t.TPG] = acc2[i][j];
        }
    }
    __syncthreads();
    if (g == 0) {
      for (int gg = 1; gg < t.G; ++gg) {
        const float* src = red + (gg - 1) * NACC * t.TPG + tg;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            acc1[i][j] += src[(i * 8 + j) * t.TPG];
            if (NW == 2) acc2[i][j] += src[(32 + i * 8 + j) * t.TPG];
          }
      }
    }
    __syncthreads();
    return;
  }
  for (int cur = t.G; cur > 1;) {
    const int half = (cur + 1) >> 1;
    if (g >= half && g < cur) {
      float* dst = red + (g - half) * NACC * t.TPG + tg;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          dst[(i * 8 + j) * t.TPG] = acc1[i][j];
          if (NW == 2) dst[(32 + i * 8 + j) * t.TPG] = acc2[i][j];
        }
    }
    __syncthreads();
    if (g + half < cur) {
      const float* src = red + g * NACC * t.TPG + tg;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc1[i][j] += src[(i * 8 + j) * t.TPG];
          if (NW == 2) acc2[i][j] += src[(32 + i * 8 + j) * t.TPG];
        }
    }
    __syncthreads();
    cur = half;
  }
}

// store up to 4 consecutive floats of a row-major buffer; `n_ok` of them are inside the tile
__device__ __forceinline__ void st4_clip(float* p, float4 v, int n_ok, bool vec) {
  if (n_ok <= 0) return;
  if (vec && n_ok >= 4) {
    *reinterpret_cast<float4*>(p) = v;
  } else {
    p[0] = v.x;
    if (n_ok > 1) p[1] = v.y;
    if (n_ok > 2) p[2] = v.z;
    if (n_ok > 3) p[3] = v.w;
  }
}

__device__ __forceinline__ void zero_acc(float (&a)[4][8], float (&b)[4][8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) a[i][j] = b[i][j] = 0.f;
}

// M = alpha mu, V (var_mode) for 4 consecutive weights.  Branch-free so that the four dependent chains (exp, log1p,
// reciprocal) interleave; entries >= nvalid come out as zeros (their inputs are zero-filled loads).
__device__ __forceinline__ void moments4(const float4 qm, const float4 qr, const float4 ql, int var_mode, int nvalid,
                                         float (&m)[4], float (&v)[4]) {
  const float mm[4] = {qm.x, qm.y, qm.z, qm.w}, rr[4] = {qr.x, qr.y, qr.z, qr.w}, ll[4] = {ql.x, ql.y, ql.z, ql.w};
  const bool ref = var_mode == LBBNN_VAR_REFERENCE;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float sg = sigma_of(rr[j]), al = alpha_of(ll[j]);
    const float vr = (sg * sg) * (al * al);
    const float ve = al * (sg * sg + (1.0f - al) * mm[j] * mm[j]);
    const bool ok = j < nvalid;
    m[j] = ok ? mm[j] * al : 0.f;
    v[j] = ok ? (ref ? vr : ve) : 0.f;
  }
}

// Shared memory: [0, kWOff) = "A region": the activation-side operand tiles of the current item and, once the MAC loop
// is done, the reduction scratch; [kWOff, ..) = "W region": the weight-side operand tiles.  The W tiles of a phase
// depend on parameters (or on activations of the forward pass) only, never on the phase before it, so every CTA stages
// the W tiles of its NEXT item before it enters the grid barrier: the parameter loads and the exp/log1p/reciprocal
// chain of the prologue overlap the barrier wait instead of sitting on the critical path after it.
constexpr int kWOff = 34816 / kCtasPerSm;     // floats: 136 KB per SM
constexpr int kWFloats = 16384 / kCtasPerSm;  // 64 KB per SM

// ---- F_l: forward partial dual GEMM --------------------------------------------------------------------
// W tiles: M and V of columns [n0, n0+C) x contraction chunk [k0, kend), transposed to [k][n], rows >= kend zero
template <bool REP>
__device__ void fwd_stage_w(const DevStep& a, int l, int gitem, float* __restrict__ W) {
  const DevLayer& y = a.ly[l];
  const int K = y.K, N = y.N;
  const int rep = REP_SEL(gitem / (y.f_ntiles * y.f_splits), 0), item = REP_SEL(gitem - rep * y.f_ntiles * y.f_splits, gitem);
  const int tile = item % y.f_ntiles, split = item / y.f_ntiles;
  const int n0 = tile * y.f_bn, C = min(y.f_bn, N - n0);
  const int k0 = split * y.f_kc, kend = min(K, k0 + y.f_kc);
  const TileCfg& t = y.fc;
  float* B1 = W;
  float* B2 = W + t.KS * t.CP;
  const float* flat = REP_SEL(a.flat + rep * a.p_stride, a.flat);
  const float* mu = flat + y.off_mu;
  const float* rho = flat + y.off_rho;
  const float* lam = flat + y.off_lam;
  const bool vecw = (K % 4 == 0);  // flat offsets are 16-byte aligned
  const int tid = threadIdx.x;
  const int total = t.CP * (t.KS >> 2);
  Walk w(tid, NT, t.CP);  // lo = column, hi = k-quad
  for (int base = tid; base < total; base += 2 * NT) {
    float4 qm[2], qr[2], ql[2];
    int cc[2], kq[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      cc[u] = w.lo; kq[u] = w.hi;
      const bool ok = base + u * NT < total && w.lo < C;
      const int64_t n = ok ? n0 + w.lo : N;  // row N = out of range -> zeros
      qm[u] = ldrow4<false>(mu, n, k0 + w.hi * 4, N, kend, K, vecw);
      qr[u] = ldrow4<false>(rho, n, k0 + w.hi * 4, N, kend, K, vecw);
      ql[u] = ldrow4<false>(lam, n, k0 + w.hi * 4, N, kend, K, vecw);
      w.next();
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (base + u * NT >= total) break;
      float m[4], v[4];
      moments4(qm[u], qr[u], ql[u], y.var_mode, cc[u] < C ? kend - (k0 + kq[u] * 4) : 0, m, v);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        B1[(kq[u] * 4 + j) * t.CP + cc[u]] = m[j];
        B2[(kq[u] * 4 + j) * t.CP + cc[u]] = v[j];
      }
    }
  }
}

template <bool REP>
__device__ void fwd_item(const DevStep& a, int l, int gitem, float* __restrict__ sm, bool w_staged) {
  const DevLayer& y = a.ly[l];
  const int B = a.B, K = y.K, N = y.N;
  const int rep = REP_SEL(gitem / (y.f_ntiles * y.f_splits), 0), item = REP_SEL(gitem - rep * y.f_ntiles * y.f_splits, gitem);
  const int tile = item % y.f_ntiles, split = item / y.f_ntiles;
  const int n0 = tile * y.f_bn, C = min(y.f_bn, N - n0);
  const int k0 = split * y.f_kc, kend = min(K, k0 + y.f_kc);
  const TileCfg& t = y.fc;
  float* A1 = sm;
  float* B1 = sm + kWOff;
  float* B2 = B1 + t.KS * t.CP;
  const float* xin = REP_SEL(l == 0 ? a.x + rep * a.x_stride : a.ly[l - 1].act + rep * a.w_stride, l == 0 ? a.x : a.ly[l - 1].act);
  const bool vecx = (K % 4 == 0) && aligned16(xin);
  const int tid = threadIdx.x;
  ITEMSTAMP(a, 64, l, 0);
  if (!w_staged) fwd_stage_w<REP>(a, l, gitem, sm + kWOff);
  ITEMSTAMP(a, 64, l, 1);
  // activations of the previous layer (or the input batch), transposed to [k][b]; lanes run along b
  {
    const int total = t.RP * (t.KS >> 2);
    Walk w(tid, NT, t.RP);  // lo = row, hi = k-quad
    for (int base = tid; base < total; base += 4 * NT) {
      float4 v[4];
      int rr[4], kq[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        rr[u] = w.lo; kq[u] = w.hi;
        const int64_t r = base + u * NT < total ? w.lo : B;
        if (l == 0) v[u] = ldrow4<false>(xin, r, k0 + w.hi * 4, B, kend, K, vecx);
        else v[u] = ldrow4<true>(xin, r, k0 + w.hi * 4, B, kend, K, vecx);
        w.next();
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (base + u * NT >= total) break;
        float* d = A1 + (kq[u] * 4) * t.RP + rr[u];
        d[0] = v[u].x; d[t.RP] = v[u].y; d[2 * t.RP] = v[u].z; d[3 * t.RP] = v[u].w;
      }
    }
  }
  ITEMSTAMP(a, 64, l, 2);
  __syncthreads();
  ITEMSTAMP(a, 64, l, 3);
  float acc1[4][8], acc2[4][8];
  zero_acc(acc1, acc2);
  const int g = tid / t.TPG, tg = tid - g * t.TPG;
  if (g < t.G) tile_mac<true, false>(A1, A1, B1, B2, t, g * t.kpg, (g + 1) * t.kpg, tg / t.CG, tg % t.CG, acc1, acc2);
  float* pe = REP_SEL(a.part + rep * a.w_stride, a.part) + (int64_t)split * 2 * B * N;
  const bool vecp = (N % 4 == 0);
  ITEMSTAMP(a, 64, l, 4);
  reduce_groups<2>(sm, t, g, tg, acc1, acc2);
  if (g == 0) {  // group 0 holds the tile: rows rg*4.., columns {cg*4..} U {CP/2 + cg*4..}
    const int rg = tg / t.CG, cgi = tg - rg * t.CG, cph = t.CP >> 1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = rg * 4 + i;
      if (r >= B) break;
      float* pr = pe + (int64_t)r * N + n0;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c0 = h * cph + cgi * 4;
        st4_clip(pr + c0, make_float4(acc1[i][h * 4], acc1[i][h * 4 + 1], acc1[i][h * 4 + 2], acc1[i][h * 4 + 3]), C - c0, vecp);
        st4_clip(pr + (int64_t)B * N + c0, make_float4(acc2[i][h * 4], acc2[i][h * 4 + 1], acc2[i][h * 4 + 2], acc2[i][h * 4 + 3]), C - c0, vecp);
      }
    }
  }
  ITEMSTAMP(a, 64, l, 5);
}

// fixed-order sum over the split partials of element e; loads issued eight splits at a time
__device__ __forceinline__ void sum_splits2(const float* __restrict__ part, int splits, int64_t total, int64_t e,
                                            float& E, float& S) {
  E = 0.f; S = 0.f;
  int s = 0;
  for (; s + 8 <= splits; s += 8) {
    float pe[8], ps[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      pe[u] = __ldcg(part + (int64_t)(s + u) * 2 * total + e);
      ps[u] = __ldcg(part + (int64_t)(s + u) * 2 * total + total + e);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) { E += pe[u]; S += ps[u]; }
  }
  float pe[8], ps[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const bool ok = s + u < splits;
    pe[u] = ok ? __ldcg(part + (int64_t)(s + u) * 2 * total + e) : 0.f;
    ps[u] = ok ? __ldcg(part + (int64_t)(s + u) * 2 * total + total + e) : 0.f;
  }
#pragma unroll
  for (int u = 0; u < 8; ++u)
    if (s + u < splits) { E += pe[u]; S += ps[u]; }
}

// ---- Fe_l: hidden-layer epilogue, one element per thread ---------------------------------------------------
// (replica launch: the elements of all replicas, replica-major; e = the element within its replica)
template <bool REP>
__device__ void fwd_epilogue(const DevStep& a, int l, int64_t step) {
  const DevLayer& y = a.ly[l];
  const int64_t total = (int64_t)a.B * y.N;
  const float* bmu = a.flat + y.off_bmu;
  const float* brho = a.flat + y.off_brho;
  const uint64_t stream = (uint64_t)l + (uint64_t)step * (uint64_t)a.L;
  for (int64_t ge = (int64_t)blockIdx.x * NT + threadIdx.x; ge < REP_SEL(a.R * total, total); ge += (int64_t)gridDim.x * NT) {
    const int rep = REP_SEL((int)(ge / total), 0);
    const int64_t e = REP_SEL(ge - rep * total, ge);
    float E, S;
    sum_splits2(REP_SEL(a.part + rep * a.w_stride, a.part), y.f_splits, total, e, E, S);
    const float ep = y.eps ? __ldg(y.eps + ge) : philox_normal1(REP_SEL(__ldg(a.seeds + rep), a.seed), stream, (uint64_t)e);
    const int n = (int)(e % y.N);
    const float sb = sigma_of(__ldg(REP_SEL(brho + rep * a.p_stride, brho) + n));
    const float sd = sqrtf(S + sb * sb);
    const float v = fmaf(sd, ep, E + __ldg(REP_SEL(bmu + rep * a.p_stride, bmu) + n));
    REP_SEL(y.act + rep * a.w_stride, y.act)[e] = fmaxf(v, 0.f);
    REP_SEL(y.dsf + rep * a.w_stride, y.dsf)[e] = ep / (2.0f * sd);
  }
}

// ---- last layer: epilogue + log_softmax + nll + dlogits; one CTA per group of rows, one warp per row ---------
__device__ void loss_epilogue(const DevStep& a, int64_t step, float* __restrict__ sm) {
  const int l = a.L - 1;
  const DevLayer& y = a.ly[l];
  const int B = a.B, N = y.N;
  const int64_t total = (int64_t)B * N;
  if ((int)blockIdx.x >= a.nll_ctas) return;
  const int rows = (B + a.nll_ctas - 1) / a.nll_ctas;  // rows per CTA (<= NT/32)
  const int b0 = blockIdx.x * rows;
  const int nrow = min(rows, B - b0);
  const float* bmu = a.flat + y.off_bmu;
  const float* brho = a.flat + y.off_brho;
  const uint64_t stream = (uint64_t)l + (uint64_t)step * (uint64_t)a.L;
  float* logit = sm;  // [rows][N]
  // logits of this CTA's rows, one element per thread (all split loads of an element in flight together)
  for (int i = threadIdx.x; i < nrow * N; i += NT) {
    const int64_t e = (int64_t)b0 * N + i;
    float E, S;
    sum_splits2(a.part, y.f_splits, total, e, E, S);
    const float ep = y.eps ? __ldg(y.eps + e) : philox_normal1(a.seed, stream, (uint64_t)e);
    const int n = i % N;
    const float sb = sigma_of(__ldg(brho + n));
    const float sd = sqrtf(S + sb * sb);
    const float v = fmaf(sd, ep, E + __ldg(bmu + n));
    logit[i] = v;
    y.act[e] = v;
    y.dsf[e] = ep / (2.0f * sd);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float local = 0.f;
  if (warp < nrow) {
    const int b = b0 + warp;
    const float* row = logit + warp * N;
    float mx = -INFINITY;
    for (int n = lane; n < N; n += 32) mx = fmaxf(mx, row[n]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.f;
    for (int n = lane; n < N; n += 32) se += expf(row[n] - mx);
    se = warp_sum(se);
    const float lse = mx + logf(se);
    const int64_t tgt = a.y[b];
    for (int n = lane; n < N; n += 32) {
      const int64_t e = (int64_t)b * N + n;
      const float lp = row[n] - lse;
      const float gd = expf(lp) - (n == tgt ? 1.0f : 0.0f);
      y.dE[e] = gd;
      y.dS[e] = gd * y.dsf[e];
      if (n == tgt) local -= lp;
    }
  }
  __syncthreads();
  const float tot = block_sum(local, sm);
  if (threadIdx.x == 0) a.nll_part[blockIdx.x] = tot;
}

// log_softmax + nll + dlogits of one row of logits, by one warp: dE, dS (= dE * dsf) of the row's N classes; returns the
// row's nll on every lane (the warp's fixed shuffle tree).  Replica launch: its heads store one nll per row.
__device__ __forceinline__ float row_nll(const float* row, int N, int64_t tgt, float* dE, float* dS, const float* dsf) {
  const int lane = threadIdx.x & 31;
  float mx = -INFINITY;
  for (int n = lane; n < N; n += 32) mx = fmaxf(mx, row[n]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float se = 0.f;
  for (int n = lane; n < N; n += 32) se += expf(row[n] - mx);
  se = warp_sum(se);
  const float lse = mx + logf(se);
  float local = 0.f;
  for (int n = lane; n < N; n += 32) {
    const float lp = row[n] - lse;
    const float gd = expf(lp) - (n == tgt ? 1.0f : 0.0f);
    dE[n] = gd;
    dS[n] = gd * dsf[n];
    if (n == tgt) local -= lp;
  }
  return warp_sum(local);
}

// Replica launch, tiled head: the R x B rows of all replicas (replica-major), ceil(R B / nll_ctas) consecutive rows per CTA --
// any number of them: the CTA takes them NW at a time, one warp per row.  Row g's nll goes to nll_part[g].
__device__ void loss_epilogue_rows(const DevStep& a, int64_t step, float* __restrict__ sm) {
  constexpr int NW = NT / 32;
  const int l = a.L - 1;
  const DevLayer& y = a.ly[l];
  const int B = a.B, N = y.N, RB = a.R * a.B;
  const int64_t total = (int64_t)B * N;
  if ((int)blockIdx.x >= a.nll_ctas) return;
  const int rows = (RB + a.nll_ctas - 1) / a.nll_ctas;
  const int g0 = blockIdx.x * rows, gend = min(RB, g0 + rows);
  const uint64_t stream = (uint64_t)l + (uint64_t)step * (uint64_t)a.L;
  const int warp = threadIdx.x >> 5;
  float* logit = sm;  // [NW][N]
  for (int c0 = g0; c0 < gend; c0 += NW) {
    const int nrow = min(NW, gend - c0);
    __syncthreads();   // the previous rows' logits are consumed
    for (int i = threadIdx.x; i < nrow * N; i += NT) {
      const int g = c0 + i / N, n = i % N, rep = g / B;
      const int64_t e = (int64_t)(g - rep * B) * N + n, wo = rep * a.w_stride, po = rep * a.p_stride;
      float E, S;
      sum_splits2(a.part + wo, y.f_splits, total, e, E, S);
      const float ep = y.eps ? __ldg(y.eps + (int64_t)g * N + n) : philox_normal1(__ldg(a.seeds + rep), stream, (uint64_t)e);
      const float sb = sigma_of(__ldg(a.flat + po + y.off_brho + n));
      const float sd = sqrtf(S + sb * sb);
      const float v = fmaf(sd, ep, E + __ldg(a.flat + po + y.off_bmu + n));
      logit[i] = v;
      y.act[wo + e] = v;
      y.dsf[wo + e] = ep / (2.0f * sd);
    }
    __syncthreads();
    if (warp < nrow) {
      const int g = c0 + warp, rep = g / B, b = g - rep * B;
      const int64_t o = rep * a.w_stride + (int64_t)b * N;
      const float nll = row_nll(logit + warp * N, N, a.y[rep * a.y_stride + b], y.dE + o, y.dS + o, y.dsf + o);
      if ((threadIdx.x & 31) == 0) a.nll_part[g] = nll;
    }
  }
}

// ---- B_l: dW item ------------------------------------------------------------------------------------------
// W tile: x (activations of the forward pass) of columns [k0, k0+C), [b][k'], rows >= B zero
template <bool REP>
__device__ void dw_stage_w(const DevStep& a, int l, int gitem, float* __restrict__ W) {
  const DevLayer& y = a.ly[l];
  const int B = a.B, K = y.K;
  const int rep = REP_SEL(gitem / (y.w_rtiles * y.w_ctiles), 0), item = REP_SEL(gitem - rep * y.w_rtiles * y.w_ctiles, gitem);
  const int ct = item % y.w_ctiles;
  const int k0 = ct * y.w_ck, C = min(y.w_ck, K - k0);
  const TileCfg& t = y.wc;
  const float* xin = REP_SEL(l == 0 ? a.x + rep * a.x_stride : a.ly[l - 1].act + rep * a.w_stride, l == 0 ? a.x : a.ly[l - 1].act);
  const bool vecx = (K % 4 == 0) && aligned16(xin);
  const int tid = threadIdx.x;
  const int ncq = t.CP >> 2;
  const int total = t.KS * ncq;
  Walk w(tid, NT, ncq);  // lo = column quad (k'), hi = b
  for (int base = tid; base < total; base += 4 * NT) {
    float4 v[4];
    int cq[4], bb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      cq[u] = w.lo; bb[u] = w.hi;
      const int64_t b = base + u * NT < total ? w.hi : B;
      if (l == 0) v[u] = ldrow4<false>(xin, b, k0 + w.lo * 4, B, k0 + C, K, vecx);
      else v[u] = ldrow4<true>(xin, b, k0 + w.lo * 4, B, k0 + C, K, vecx);
      w.next();
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (base + u * NT >= total) break;
      *reinterpret_cast<float4*>(W + bb[u] * t.CP + cq[u] * 4) = v[u];
    }
  }
}

template <bool REP>
__device__ void dw_item(const DevStep& a, int l, int gitem, float* __restrict__ sm, bool w_staged) {
  const DevLayer& y = a.ly[l];
  const int B = a.B, K = y.K, N = y.N;
  const int rep = REP_SEL(gitem / (y.w_rtiles * y.w_ctiles), 0), item = REP_SEL(gitem - rep * y.w_rtiles * y.w_ctiles, gitem);
  const int ct = item % y.w_ctiles, rt = item / y.w_ctiles;
  const int n0 = rt * y.w_rn, R = min(y.w_rn, N - n0);
  const int k0 = ct * y.w_ck, C = min(y.w_ck, K - k0);
  const TileCfg& t = y.wc;
  float* A1 = sm;                   // [b][RP]  dE
  float* A2 = A1 + t.KS * t.RP;     // [b][RP]  dS
  float* B1 = sm + kWOff;           // [b][CP]  x
  const bool vecn = (N % 4 == 0);
  const int tid = threadIdx.x;
  const int nrq = t.RP >> 2;
  ITEMSTAMP(a, 96, l, 0);
  if (!w_staged) dw_stage_w<REP>(a, l, gitem, sm + kWOff);
  {
    const int total = t.KS * nrq;
    Walk w(tid, NT, nrq);  // lo = row quad (n), hi = b
    for (int base = tid; base < total; base += 2 * NT) {
      float4 e4[2], s4[2];
      int rq[2], bb[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        rq[u] = w.lo; bb[u] = w.hi;
        const int64_t b = base + u * NT < total ? w.hi : B;
        e4[u] = ldrow4<true>(REP_SEL(y.dE + rep * a.w_stride, y.dE), b, n0 + w.lo * 4, B, n0 + R, N, vecn);
        s4[u] = ldrow4<true>(REP_SEL(y.dS + rep * a.w_stride, y.dS), b, n0 + w.lo * 4, B, n0 + R, N, vecn);
        w.next();
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (base + u * NT >= total) break;
        *reinterpret_cast<float4*>(A1 + bb[u] * t.RP + rq[u] * 4) = e4[u];
        *reinterpret_cast<float4*>(A2 + bb[u] * t.RP + rq[u] * 4) = s4[u];
      }
    }
  }
  ITEMSTAMP(a, 96, l, 1);
  __syncthreads();
  ITEMSTAMP(a, 96, l, 2);
  // bias column sums over the batch (column-tile 0 only; fixed order)
  if (ct == 0) {
    for (int r = tid; r < R; r += NT) {
      float se = 0.f, ss = 0.f;
      for (int b = 0; b < B; ++b) { se += A1[b * t.RP + r]; ss += A2[b * t.RP + r]; }
      REP_SEL(y.colsum + rep * a.w_stride, y.colsum)[n0 + r] = se;
      REP_SEL(y.colsum + rep * a.w_stride, y.colsum)[N + n0 + r] = ss;
    }
  }
  float acc1[4][8], acc2[4][8];
  zero_acc(acc1, acc2);
  const int g = tid / t.TPG, tg = tid - g * t.TPG;
  if (g < t.G) tile_mac<false, true>(A1, A2, B1, B1, t, g * t.kpg, (g + 1) * t.kpg, tg / t.CG, tg % t.CG, acc1, acc2);
  const bool veck = (K % 4 == 0);
  ITEMSTAMP(a, 96, l, 3);
  reduce_groups<2>(sm, t, g, tg, acc1, acc2);
  ITEMSTAMP(a, 96, l, 4);
  if (g == 0) {
    const int rg = tg / t.CG, cgi = tg - rg * t.CG, cph = t.CP >> 1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = rg * 4 + i;
      if (r >= R) break;
      const int64_t o = REP_SEL(rep * a.w_stride + (int64_t)(n0 + r) * K + k0, (int64_t)(n0 + r) * K + k0);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c0 = h * cph + cgi * 4;
        st4_clip(y.dM + o + c0, make_float4(acc1[i][h * 4], acc1[i][h * 4 + 1], acc1[i][h * 4 + 2], acc1[i][h * 4 + 3]), C - c0, veck);
        st4_clip(y.dV + o + c0, make_float4(acc2[i][h * 4], acc2[i][h * 4 + 1], acc2[i][h * 4 + 2], acc2[i][h * 4 + 3]), C - c0, veck);
      }
    }
  }
  ITEMSTAMP(a, 96, l, 5);
}

// dE_{l-1} = dx * [x > 0], dS_{l-1} = dE_{l-1} * ds_factor_{l-1}  (x = relu output of layer l-1)
__device__ __forceinline__ void dx_finish(const DevStep& a, int l, int64_t e, float dx) {
  const DevLayer& p = a.ly[l - 1];
  const float xv = __ldcg(p.act + e);
  const float de = xv > 0.f ? dx : 0.f;
  p.dE[e] = de;
  p.dS[e] = de * __ldcg(p.dsf + e);
}

// ---- B_l: dX item --------------------------------------------------------------------------------------------
// W tiles: M and V of rows [nb, nend) (the contraction) x columns [k0, k0+C), [n][k'], rows >= nend zero
template <bool REP>
__device__ void dx_stage_w(const DevStep& a, int l, int gitem, float* __restrict__ W) {
  const DevLayer& y = a.ly[l];
  const int K = y.K, N = y.N;
  const int rep = REP_SEL(gitem / (y.x_ctiles * y.x_splits), 0), item = REP_SEL(gitem - rep * y.x_ctiles * y.x_splits, gitem);
  const int ct = item % y.x_ctiles, split = item / y.x_ctiles;
  const int k0 = ct * y.x_bk, C = min(y.x_bk, K - k0);
  const int nb = split * y.x_nc, nend = min(N, nb + y.x_nc);
  const TileCfg& t = y.xc;
  float* B1 = W;
  float* B2 = W + t.KS * t.CP;
  const bool vecw = (K % 4 == 0);
  const float* flat = REP_SEL(a.flat + rep * a.p_stride, a.flat);
  const float* mu = flat + y.off_mu;
  const float* rho = flat + y.off_rho;
  const float* lam = flat + y.off_lam;
  const int tid = threadIdx.x;
  const int ncq = t.CP >> 2;
  const int total = t.KS * ncq;
  Walk w(tid, NT, ncq);  // lo = column quad (k'), hi = contraction row (n)
  for (int base = tid; base < total; base += 2 * NT) {
    float4 qm[2], qr[2], ql[2];
    int cq[2], kk[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      cq[u] = w.lo; kk[u] = w.hi;
      const int64_t n = base + u * NT < total ? nb + w.hi : nend;
      qm[u] = ldrow4<false>(mu, n, k0 + w.lo * 4, nend, k0 + C, K, vecw);
      qr[u] = ldrow4<false>(rho, n, k0 + w.lo * 4, nend, k0 + C, K, vecw);
      ql[u] = ldrow4<false>(lam, n, k0 + w.lo * 4, nend, k0 + C, K, vecw);
      w.next();
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (base + u * NT >= total) break;
      float m[4], v[4];
      moments4(qm[u], qr[u], ql[u], y.var_mode, nb + kk[u] < nend ? C - cq[u] * 4 : 0, m, v);
      *reinterpret_cast<float4*>(B1 + kk[u] * t.CP + cq[u] * 4) = make_float4(m[0], m[1], m[2], m[3]);
      *reinterpret_cast<float4*>(B2 + kk[u] * t.CP + cq[u] * 4) = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

template <bool REP>
__device__ void dx_item(const DevStep& a, int l, int gitem, float* __restrict__ sm, bool w_staged) {
  const DevLayer& y = a.ly[l];
  const int B = a.B, K = y.K, N = y.N;
  const int rep = REP_SEL(gitem / (y.x_ctiles * y.x_splits), 0), item = REP_SEL(gitem - rep * y.x_ctiles * y.x_splits, gitem);
  const int ct = item % y.x_ctiles, split = item / y.x_ctiles;
  const int k0 = ct * y.x_bk, C = min(y.x_bk, K - k0);
  const int nb = split * y.x_nc, nend = min(N, nb + y.x_nc);
  const TileCfg& t = y.xc;
  float* A1 = sm;                   // [n][RP] dE^T
  float* A2 = A1 + t.KS * t.RP;     // [n][RP] dS^T
  float* B1 = sm + kWOff;           // [n][CP] M
  float* B2 = B1 + t.KS * t.CP;     // [n][CP] V
  const bool vecn = (N % 4 == 0);
  const bool vecw = (K % 4 == 0);
  const int tid = threadIdx.x;
  ITEMSTAMP(a, 128, l, 0);
  if (!w_staged) dx_stage_w<REP>(a, l, gitem, sm + kWOff);
  {
    const int total = t.RP * (t.KS >> 2);
    Walk w(tid, NT, t.RP);  // lo = row (b), hi = contraction quad (n)
    for (int base = tid; base < total; base += 2 * NT) {
      float4 e4[2], s4[2];
      int rr[2], nq[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        rr[u] = w.lo; nq[u] = w.hi;
        const int64_t r = base + u * NT < total ? w.lo : B;
        e4[u] = ldrow4<true>(REP_SEL(y.dE + rep * a.w_stride, y.dE), r, nb + w.hi * 4, B, nend, N, vecn);
        s4[u] = ldrow4<true>(REP_SEL(y.dS + rep * a.w_stride, y.dS), r, nb + w.hi * 4, B, nend, N, vecn);
        w.next();
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (base + u * NT >= total) break;
        float* d1 = A1 + (nq[u] * 4) * t.RP + rr[u];
        float* d2 = A2 + (nq[u] * 4) * t.RP + rr[u];
        d1[0] = e4[u].x; d1[t.RP] = e4[u].y; d1[2 * t.RP] = e4[u].z; d1[3 * t.RP] = e4[u].w;
        d2[0] = s4[u].x; d2[t.RP] = s4[u].y; d2[2 * t.RP] = s4[u].z; d2[3 * t.RP] = s4[u].w;
      }
    }
  }
  ITEMSTAMP(a, 128, l, 1);
  __syncthreads();
  ITEMSTAMP(a, 128, l, 2);
  float acc1[4][8], acc2[4][8];
  zero_acc(acc1, acc2);
  const int g = tid / t.TPG, tg = tid - g * t.TPG;
  const int rg = tg / t.CG, cgi = tg % t.CG;
  if (g < t.G) tile_mac<false, false>(A1, A2, B1, B2, t, g * t.kpg, (g + 1) * t.kpg, rg, cgi, acc1, acc2);
  ITEMSTAMP(a, 128, l, 3);
  reduce_groups<2>(sm, t, g, tg, acc1, acc2);
  ITEMSTAMP(a, 128, l, 4);
  if (g == 0) {
    // dx = dE M + 2 x (dS V); then either a partial (split contraction) or straight through the relu of layer l-1:
    // dE_{l-1} = dx [x > 0], dS_{l-1} = dE_{l-1} ds_factor_{l-1}.  All loads of the thread's 4x8 tile first.
    const DevLayer& p = a.ly[l - 1];
    const bool direct = y.x_splits == 1;
    float* part = a.part + (int64_t)split * B * K;
    const int cph = t.CP >> 1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = rg * 4 + i;
      if (r >= B) break;
      float4 xq[2], fq[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c0 = h * cph + cgi * 4;
        xq[h] = ldrow4<true>(REP_SEL(p.act + rep * a.w_stride, p.act), r, k0 + c0, B, k0 + C, K, vecw);
        fq[h] = direct ? ldrow4<true>(REP_SEL(p.dsf + rep * a.w_stride, p.dsf), r, k0 + c0, B, k0 + C, K, vecw) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c0 = h * cph + cgi * 4;
        const int64_t e = REP_SEL(rep * a.w_stride + (int64_t)r * K + k0 + c0, (int64_t)r * K + k0 + c0);
        const float xv[4] = {xq[h].x, xq[h].y, xq[h].z, xq[h].w};
        const float fv[4] = {fq[h].x, fq[h].y, fq[h].z, fq[h].w};
        float dx[4], ds[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          dx[j] = fmaf(2.0f * xv[j], acc2[i][h * 4 + j], acc1[i][h * 4 + j]);
          ds[j] = 0.f;
          if (direct) {
            dx[j] = xv[j] > 0.f ? dx[j] : 0.f;
            ds[j] = dx[j] * fv[j];
          }
        }
        if (!direct) {
          st4_clip(part + e, make_float4(dx[0], dx[1], dx[2], dx[3]), C - c0, vecw);
        } else {
          st4_clip(p.dE + e, make_float4(dx[0], dx[1], dx[2], dx[3]), C - c0, vecw);
          st4_clip(p.dS + e, make_float4(ds[0], ds[1], ds[2], ds[3]), C - c0, vecw);
        }
      }
    }
  }
  ITEMSTAMP(a, 128, l, 5);
}

// ---- Xe_l: sum of the dX partials ------------------------------------------------------------------------------
template <bool REP>
__device__ void dx_epilogue(const DevStep& a, int l) {
  const DevLayer& y = a.ly[l];
  const int64_t total = (int64_t)a.B * y.K;
  for (int64_t ge = (int64_t)blockIdx.x * NT + threadIdx.x; ge < REP_SEL(a.R * total, total); ge += (int64_t)gridDim.x * NT) {
    const int rep = REP_SEL((int)(ge / total), 0);
    const int64_t e = REP_SEL(ge - rep * total + rep * a.w_stride, ge);   // within the replica's workspace block
    float s = 0.f;
    int sp = 0;
    for (; sp < y.x_splits; sp += 8) {
      float p[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) p[u] = sp + u < y.x_splits ? __ldcg(a.part + (int64_t)(sp + u) * total + e) : 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (sp + u < y.x_splits) s += p[u];
    }
    dx_finish(a, l, e, s);
  }
}

// ---- U: chain rule + KL gradient/value + Adam ------------------------------------------------------------------
// The update phase is instruction-bound (r01 ncu: ~400 instructions per weight with IEEE div/sqrt/log slow paths), so it
// uses the approximate MUFU forms (<= 2 ulp; the parity bounds are 1e-5..5e-5): see tests/test_lrt_gpu.py.
__device__ __forceinline__ float fsqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void adam1(float& p, float g, float& m, float& v, float b1, float b2, float eps, float step_size,
                                      float inv_bc2_sqrt) {
  m = m + (g - m) * (1.0f - b1);  // lerp form, as torch's _single_tensor_adam
  v = b2 * v + (1.0f - b2) * g * g;
  const float denom = fmaf(fsqrt_approx(v), inv_bc2_sqrt, eps);
  p -= step_size * __fdividef(m, denom);
}

struct Q4 { float v[4]; };
template <bool COH>
__device__ __forceinline__ Q4 ldq4(const float* p, int cnt, bool vec) {
  Q4 r;
  if (vec) {
    const float4 t4 = COH ? __ldcg(reinterpret_cast<const float4*>(p)) : *reinterpret_cast<const float4*>(p);
    r.v[0] = t4.x; r.v[1] = t4.y; r.v[2] = t4.z; r.v[3] = t4.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) r.v[j] = j < cnt ? (COH ? __ldcg(p + j) : p[j]) : 0.f;
  }
  return r;
}
__device__ __forceinline__ void stq4(float* p, const Q4& q, int cnt, bool vec) {
  if (vec) {
    *reinterpret_cast<float4*>(p) = make_float4(q.v[0], q.v[1], q.v[2], q.v[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < cnt) p[j] = q.v[j];
  }
}

// one layer's weights: chain rule + KL + Adam over quads; VEC = all quads are full and 16-byte aligned
// chain rule + KL + Adam of quad q (4 consecutive weights) of one layer; returns the quad's KL contribution
// DP: the data-parallel exchange of lbbnn_step_dp is compiled in (a separate instantiation: its peer / multicast paths cost
// the single-GPU kernel registers -- 109 -> 128 us/step with spills when they shared one body)
// REP: the replica launch; po / wo = the replica's offset in the parameter-side buffers / in the workspace
template <bool VEC, bool REF, bool DP, bool REP = false>
__device__ __forceinline__ float update_quad(const DevStep& a, const DevLayer& y, float step_size, float inv_bc2_sqrt, int64_t q,
                                             int64_t po = 0, int64_t wo = 0) {
  const lbbnn_priors P = y.pri;
  const float klg = a.klg;
  const float inv_sp2 = 1.0f / (P.sigma * P.sigma);
  const float inv_omp = 1.0f / (1.0f - P.alpha), inv_ap = 1.0f / P.alpha;
  const int64_t n = (int64_t)y.N * y.K;
  float kl = 0.f;
  {
    const int64_t e0 = q * 4;
    const int cnt = VEC ? 4 : (int)min((int64_t)4, n - e0);
    Q4 mu = ldq4<false>(REP_SEL(a.flat + po, a.flat) + y.off_mu + e0, cnt, VEC), rho = ldq4<false>(REP_SEL(a.flat + po, a.flat) + y.off_rho + e0, cnt, VEC);
    Q4 lam = ldq4<false>(REP_SEL(a.flat + po, a.flat) + y.off_lam + e0, cnt, VEC);
    Q4 dM, dV;
    if (DP && VEC && a.dp_p2p) {   // this rank owns the quad: sum the ranks' copies over NVLink, in rank order
      const int64_t om = (y.dM - a.raw_base) + e0, ov = (y.dV - a.raw_base) + e0;
      float4 t0[8], t1[8];
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (q < a.dp_world) {
          t0[q] = __ldcg(reinterpret_cast<const float4*>(a.raw_peer[q] + om));
          t1[q] = __ldcg(reinterpret_cast<const float4*>(a.raw_peer[q] + ov));
        }
#pragma unroll
      for (int j = 0; j < 4; ++j) dM.v[j] = dV.v[j] = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (q < a.dp_world) {
          dM.v[0] += t0[q].x; dM.v[1] += t0[q].y; dM.v[2] += t0[q].z; dM.v[3] += t0[q].w;
          dV.v[0] += t1[q].x; dV.v[1] += t1[q].y; dV.v[2] += t1[q].z; dV.v[3] += t1[q].w;
        }
    } else if (DP && VEC) {   // summed over the ranks inside the switch (this rank owns the quad)
      const float4 t0 = mc_ld_reduce4(a.raw_mc + (y.dM - a.raw_base) + e0), t1 = mc_ld_reduce4(a.raw_mc + (y.dV - a.raw_base) + e0);
      dM.v[0] = t0.x; dM.v[1] = t0.y; dM.v[2] = t0.z; dM.v[3] = t0.w;
      dV.v[0] = t1.x; dV.v[1] = t1.y; dV.v[2] = t1.z; dV.v[3] = t1.w;
    } else {
      dM = ldq4<true>(REP_SEL(y.dM + wo, y.dM) + e0, cnt, VEC);
      dV = ldq4<true>(REP_SEL(y.dV + wo, y.dV) + e0, cnt, VEC);
    }
    Q4 m0 = ldq4<false>(REP_SEL(a.m + po, a.m) + y.off_mu + e0, cnt, VEC), m1 = ldq4<false>(REP_SEL(a.m + po, a.m) + y.off_rho + e0, cnt, VEC);
    Q4 m2 = ldq4<false>(REP_SEL(a.m + po, a.m) + y.off_lam + e0, cnt, VEC);
    Q4 v0 = ldq4<false>(REP_SEL(a.v + po, a.v) + y.off_mu + e0, cnt, VEC), v1 = ldq4<false>(REP_SEL(a.v + po, a.v) + y.off_rho + e0, cnt, VEC);
    Q4 v2 = ldq4<false>(REP_SEL(a.v + po, a.v) + y.off_lam + e0, cnt, VEC);
    Q4 g0, g1, g2;
#pragma unroll
    for (int j = 0; j < 4; ++j) {  // branch-free: the four elements' dependent chains interleave
      const float w = mu.v[j];
      const float er = __expf(rho.v[j]);
      const float sg = log1pf(er), al = __fdividef(1.0f, 1.0f + __expf(-lam.v[j]));
      const float inv_sg = __fdividef(1.0f, sg);
      float dmu = al * dM.v[j], dsg, dal;
      if (REF) {
        dsg = 2.0f * al * al * sg * dV.v[j];
        dal = w * dM.v[j] + 2.0f * al * sg * sg * dV.v[j];
      } else {
        dmu += 2.0f * al * (1.0f - al) * w * dV.v[j];
        dsg = 2.0f * al * sg * dV.v[j];
        dal = w * dM.v[j] + (sg * sg + (1.0f - 2.0f * al) * w * w) * dV.v[j];
      }
      // closed-form KL (LRT:189-192): value and gradient share their logs
      const float d = w - P.mu;
      const float om = 1.0f - al;
      const float l3 = __logf(om * inv_omp);
      const float slab = __logf(P.sigma * inv_sg) - 0.5f + __logf(al * inv_ap) + (sg * sg + d * d) * 0.5f * inv_sp2;
      const float klj = al * slab + om * l3;
      kl += (VEC || j < cnt) ? klj : 0.f;
      dmu += klg * al * d * inv_sp2;
      dsg += klg * al * (sg * inv_sp2 - inv_sg);
      dal += klg * (slab - l3);
      g0.v[j] = dmu;
      g1.v[j] = dsg * __fdividef(er, 1.0f + er);   // d sigma / d rho
      g2.v[j] = dal * al * om;
      adam1(mu.v[j], g0.v[j], m0.v[j], v0.v[j], a.b1, a.b2, a.eps, step_size, inv_bc2_sqrt);
      adam1(rho.v[j], g1.v[j], m1.v[j], v1.v[j], a.b1, a.b2, a.eps, step_size, inv_bc2_sqrt);
      adam1(lam.v[j], g2.v[j], m2.v[j], v2.v[j], a.b1, a.b2, a.eps, step_size, inv_bc2_sqrt);
    }
    if (DP && VEC && a.dp_p2p) {   // the new parameters go to every rank's copy (posted stores over NVLink)
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (q < a.dp_world) {
          stq4(a.flat_peer[q] + y.off_mu + e0, mu, 4, true); stq4(a.flat_peer[q] + y.off_rho + e0, rho, 4, true);
          stq4(a.flat_peer[q] + y.off_lam + e0, lam, 4, true);
        }
    } else if (DP && VEC) {   // the new parameters go to every rank's copy
      mc_st4(a.flat_mc + y.off_mu + e0, mu.v); mc_st4(a.flat_mc + y.off_rho + e0, rho.v); mc_st4(a.flat_mc + y.off_lam + e0, lam.v);
    } else {
      stq4(REP_SEL(a.flat + po, a.flat) + y.off_mu + e0, mu, cnt, VEC); stq4(REP_SEL(a.flat + po, a.flat) + y.off_rho + e0, rho, cnt, VEC);
      stq4(REP_SEL(a.flat + po, a.flat) + y.off_lam + e0, lam, cnt, VEC);
    }
    stq4(REP_SEL(a.m + po, a.m) + y.off_mu + e0, m0, cnt, VEC); stq4(REP_SEL(a.m + po, a.m) + y.off_rho + e0, m1, cnt, VEC); stq4(REP_SEL(a.m + po, a.m) + y.off_lam + e0, m2, cnt, VEC);
    stq4(REP_SEL(a.v + po, a.v) + y.off_mu + e0, v0, cnt, VEC); stq4(REP_SEL(a.v + po, a.v) + y.off_rho + e0, v1, cnt, VEC); stq4(REP_SEL(a.v + po, a.v) + y.off_lam + e0, v2, cnt, VEC);
    if (a.grad) {
      stq4(REP_SEL(a.grad + po, a.grad) + y.off_mu + e0, g0, cnt, VEC); stq4(REP_SEL(a.grad + po, a.grad) + y.off_rho + e0, g1, cnt, VEC);
      stq4(REP_SEL(a.grad + po, a.grad) + y.off_lam + e0, g2, cnt, VEC);
    }
  }
  return kl;
}

// Chain rule + KL + Adam of layers [l0, l1) by the CTAs [cta0, cta0 + ncta) of the grid (every CTA of that range
// calls this; `cta` = its index in the range).  The quads of all those layers form ONE index space that is dealt
// out round-robin, so every thread gets the same number of quads whatever the layer sizes; one CTA per layer also
// updates its biases.  Each CTA leaves its KL partial of every layer in kl_part[l][blockIdx.x].
template <bool DP>
__device__ void update_layers(const DevStep& a, int64_t step, int l0, int l1, int cta, int ncta, float* __restrict__ sm) {
  __shared__ float coef[2];
  constexpr int NW = NT / 32;
  __syncthreads();
  if (threadIdx.x == 0) {
    const double t = (double)(step + 1);
    coef[0] = a.lr / (float)(1.0 - pow((double)a.b1, t));
    coef[1] = (float)(1.0 / sqrt(1.0 - pow((double)a.b2, t)));
  }
  __syncthreads();
  const float step_size = coef[0], bc2_sqrt = coef[1];  // bc2_sqrt holds 1/sqrt(1 - beta2^t)
  const float klg = a.klg;
  float kl[kMaxL];
#pragma unroll
  for (int l = 0; l < kMaxL; ++l) kl[l] = 0.f;
  int64_t total = 0;
  for (int l = l0; l < l1; ++l) total += ((int64_t)a.ly[l].N * a.ly[l].K + 3) >> 2;
  // data parallel: this rank updates a contiguous 1 / world of the quads (and rank 0 the biases)
  int64_t g_first = 0, g_end = total;
  if (DP) {
    const int64_t per = (total + a.dp_world - 1) / a.dp_world;
    g_first = min(total, (int64_t)a.dp_rank * per);
    g_end = min(total, g_first + per);
  }
  for (int64_t g = g_first + (int64_t)cta * NT + threadIdx.x; g < g_end; g += (int64_t)ncta * NT) {
    int l = l0;
    int64_t q = g;
    for (;; ++l) {
      const int64_t nq = ((int64_t)a.ly[l].N * a.ly[l].K + 3) >> 2;
      if (q < nq) break;
      q -= nq;
    }
    const DevLayer& y = a.ly[l];
    const bool vec = (((int64_t)y.N * y.K) % 4 == 0);
    const bool ref = y.var_mode == LBBNN_VAR_REFERENCE;
    float k_;
    if (vec) k_ = ref ? update_quad<true, true, DP>(a, y, step_size, bc2_sqrt, q) : update_quad<true, false, DP>(a, y, step_size, bc2_sqrt, q);
    else k_ = ref ? update_quad<false, true, DP>(a, y, step_size, bc2_sqrt, q) : update_quad<false, false, DP>(a, y, step_size, bc2_sqrt, q);
#pragma unroll
    for (int j = 0; j < kMaxL; ++j) kl[j] += (j == l) ? k_ : 0.f;
  }
  // biases: db_mu = sum_b dE, dsigma_b = 2 sigma_b sum_b dS, + KL (LRT:185-186); one CTA per layer
  constexpr bool dp = DP;
  for (int l = l0; l < l1; ++l) {
    if (cta != (a.L - 1 - l) % ncta) continue;
    if (dp && a.dp_rank != 0) continue;
    const DevLayer& y = a.ly[l];
    const lbbnn_priors P = y.pri;
    const float inv = 1.0f / (P.bias_sigma * P.bias_sigma);
    float kb = 0.f;
    const float* cs_mc = dp ? a.raw_mc + (y.colsum - a.raw_base) : nullptr;
    for (int i = threadIdx.x; i < y.N; i += NT) {
      float bm = a.flat[y.off_bmu + i], br = a.flat[y.off_brho + i];
      const float sb = sigma_of(br);
      float dbm, dss;
      if (dp && a.dp_p2p) {
        dbm = dss = 0.f;
        for (int q = 0; q < a.dp_world; ++q) {
          const float* cq = a.raw_peer[q] + (y.colsum - a.raw_base);
          dbm += __ldcg(cq + i);
          dss += __ldcg(cq + y.N + i);
        }
      } else if (dp) {
        dbm = mc_ld_reduce1(cs_mc + i);
        dss = mc_ld_reduce1(cs_mc + y.N + i);
      } else {
        dbm = __ldcg(y.colsum + i);
        dss = __ldcg(y.colsum + y.N + i);
      }
      float dsb = 2.0f * sb * dss;
      kb += kl_bias_elem(bm, sb, P);
      dbm += klg * (bm - P.bias_mu) * inv;
      dsb += klg * (sb * inv - 1.0f / sb);
      const float dbr = dsb * dsigma_drho(br);
      if (a.grad) { a.grad[y.off_bmu + i] = dbm; a.grad[y.off_brho + i] = dbr; }
      float mm0 = a.m[y.off_bmu + i], vv0 = a.v[y.off_bmu + i], mm1 = a.m[y.off_brho + i], vv1 = a.v[y.off_brho + i];
      adam1(bm, dbm, mm0, vv0, a.b1, a.b2, a.eps, step_size, bc2_sqrt);
      adam1(br, dbr, mm1, vv1, a.b1, a.b2, a.eps, step_size, bc2_sqrt);
      if (dp && a.dp_p2p) {
        for (int q = 0; q < a.dp_world; ++q) { a.flat_peer[q][y.off_bmu + i] = bm; a.flat_peer[q][y.off_brho + i] = br; }
      } else if (dp) { mc_st1(a.flat_mc + y.off_bmu + i, bm); mc_st1(a.flat_mc + y.off_brho + i, br); }
      else { a.flat[y.off_bmu + i] = bm; a.flat[y.off_brho + i] = br; }
      a.m[y.off_bmu + i] = mm0; a.v[y.off_bmu + i] = vv0; a.m[y.off_brho + i] = mm1; a.v[y.off_brho + i] = vv1;
    }
#pragma unroll
    for (int j = 0; j < kMaxL; ++j) kl[j] += (j == l) ? kb : 0.f;
  }
  // per-layer KL partials of this CTA: warp shuffles, then the warps in order (one barrier for all layers)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < kMaxL; ++j) {
    const float w = warp_sum(kl[j]);
    if (lane == 0) sm[warp * kMaxL + j] = w;
  }
  __syncthreads();
  if ((int)threadIdx.x >= l0 && (int)threadIdx.x < l1) {
    double tot = 0.0;
    for (int w = 0; w < NW; ++w) tot += (double)sm[w * kMaxL + threadIdx.x];
    a.kl_part[(int64_t)threadIdx.x * gridDim.x + blockIdx.x] = tot;
  }
  __syncthreads();
}

// Replica launch: chain rule + KL + Adam of every layer of every replica.  One replica's quads (all its layers, as in
// update_layers) are padded to a multiple of NT, and the quads of all replicas form ONE index space dealt out round-robin in
// CTA-sized chunks: a chunk lies in one replica, so a CTA moves on to the next replica as a whole and then reduces the per-layer
// KL of the replica it leaves (warps in order) into kl_part[r][l][blockIdx.x].  Biases: one CTA per (replica, layer), added to
// that CTA's partial.  The per-element arithmetic is update_layers': each replica's parameters, moments and gradients come out
// bit-identical to the single-network step's.
__device__ void update_layers_rep(const DevStep& a, int64_t step, float* __restrict__ sm) {
  __shared__ float coef[2];
  constexpr int NW = NT / 32;
  const int L = a.L, G = gridDim.x;
  __syncthreads();
  if (threadIdx.x == 0) {
    const double t = (double)(step + 1);
    coef[0] = a.lr / (float)(1.0 - pow((double)a.b1, t));
    coef[1] = (float)(1.0 / sqrt(1.0 - pow((double)a.b2, t)));
  }
  // replicas this CTA has no quads or biases of keep a zero partial
  for (int i = threadIdx.x; i < a.R * L; i += NT) a.kl_part[(int64_t)i * G + blockIdx.x] = 0.0;
  __syncthreads();
  const float step_size = coef[0], bc2_sqrt = coef[1];
  const float klg = a.klg;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float kl[kMaxL];
#pragma unroll
  for (int l = 0; l < kMaxL; ++l) kl[l] = 0.f;
  // the CTA's per-layer KL of replica `rep` -> kl_part (+= when `add`: the bias pass after the quads)
  auto flush = [&](int rep, bool add) {
#pragma unroll
    for (int j = 0; j < kMaxL; ++j) {
      const float w = warp_sum(kl[j]);
      if (lane == 0) sm[warp * kMaxL + j] = w;
      kl[j] = 0.f;
    }
    __syncthreads();
    if ((int)threadIdx.x < L) {
      double tot = 0.0;
      for (int w = 0; w < NW; ++w) tot += (double)sm[w * kMaxL + threadIdx.x];
      double* dst = a.kl_part + ((int64_t)rep * L + threadIdx.x) * G + blockIdx.x;
      *dst = add ? *dst + tot : tot;
    }
    __syncthreads();
  };
  int64_t per = 0;
  for (int l = 0; l < L; ++l) per += ((int64_t)a.ly[l].N * a.ly[l].K + 3) >> 2;
  per = (per + NT - 1) / NT * NT;
  int cur = -1;
  for (int64_t g0 = (int64_t)blockIdx.x * NT; g0 < a.R * per; g0 += (int64_t)G * NT) {
    const int rep = (int)(g0 / per);
    if (rep != cur) {
      if (cur >= 0) flush(cur, false);
      cur = rep;
    }
    int l = 0;
    int64_t q = g0 - rep * per + threadIdx.x;
    for (; l < L; ++l) {
      const int64_t nq = ((int64_t)a.ly[l].N * a.ly[l].K + 3) >> 2;
      if (q < nq) break;
      q -= nq;
    }
    if (l == L) continue;   // padding
    const DevLayer& y = a.ly[l];
    const bool vec = (((int64_t)y.N * y.K) % 4 == 0);
    const bool ref = y.var_mode == LBBNN_VAR_REFERENCE;
    const int64_t po = rep * a.p_stride, wo = rep * a.w_stride;
    float k_;
    if (vec) k_ = ref ? update_quad<true, true, false, true>(a, y, step_size, bc2_sqrt, q, po, wo) : update_quad<true, false, false, true>(a, y, step_size, bc2_sqrt, q, po, wo);
    else k_ = ref ? update_quad<false, true, false, true>(a, y, step_size, bc2_sqrt, q, po, wo) : update_quad<false, false, false, true>(a, y, step_size, bc2_sqrt, q, po, wo);
#pragma unroll
    for (int j = 0; j < kMaxL; ++j) kl[j] += (j == l) ? k_ : 0.f;
  }
  if (cur >= 0) flush(cur, false);
  // biases (as update_layers): db_mu = sum_b dE, dsigma_b = 2 sigma_b sum_b dS, + KL (LRT:185-186)
  for (int t = blockIdx.x; t < a.R * L; t += G) {
    const int rep = t / L, l = L - 1 - (t - rep * L);
    const DevLayer& y = a.ly[l];
    const lbbnn_priors P = y.pri;
    const float inv = 1.0f / (P.bias_sigma * P.bias_sigma);
    const int64_t po = rep * a.p_stride, wo = rep * a.w_stride;
    float* flat = a.flat + po;
    float* am = a.m + po;
    float* av = a.v + po;
    float kb = 0.f;
    for (int i = threadIdx.x; i < y.N; i += NT) {
      float bm = flat[y.off_bmu + i], br = flat[y.off_brho + i];
      const float sb = sigma_of(br);
      float dbm = __ldcg(y.colsum + wo + i), dss = __ldcg(y.colsum + wo + y.N + i);
      float dsb = 2.0f * sb * dss;
      kb += kl_bias_elem(bm, sb, P);
      dbm += klg * (bm - P.bias_mu) * inv;
      dsb += klg * (sb * inv - 1.0f / sb);
      const float dbr = dsb * dsigma_drho(br);
      if (a.grad) { a.grad[po + y.off_bmu + i] = dbm; a.grad[po + y.off_brho + i] = dbr; }
      float mm0 = am[y.off_bmu + i], vv0 = av[y.off_bmu + i], mm1 = am[y.off_brho + i], vv1 = av[y.off_brho + i];
      adam1(bm, dbm, mm0, vv0, a.b1, a.b2, a.eps, step_size, bc2_sqrt);
      adam1(br, dbr, mm1, vv1, a.b1, a.b2, a.eps, step_size, bc2_sqrt);
      flat[y.off_bmu + i] = bm; flat[y.off_brho + i] = br;
      am[y.off_bmu + i] = mm0; av[y.off_bmu + i] = vv0; am[y.off_brho + i] = mm1; av[y.off_brho + i] = vv1;
    }
#pragma unroll
    for (int j = 0; j < kMaxL; ++j) kl[j] = (j == l) ? kb : 0.f;
    flush(rep, true);
  }
}

// The last CTA to arrive sums the per-CTA partials in a fixed order (deterministic) and bumps the step counter.
// Replica launch: one warp per (replica, sum) -- the replica's nll over its rows, each layer's KL over the CTAs.
template <bool DP, bool REP>
__device__ void finish_step(const DevStep& a, int64_t step, float* __restrict__ sm) {
  __shared__ int is_last;
  double* dred = reinterpret_cast<double*>(sm);
  if (DP) __threadfence_system();   // this CTA's multicast stores of parameters, before the closing flags
  else __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned tk = atomicAdd(a.ticket, 1u);
    is_last = (tk == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (a.prof && threadIdx.x == 0) a.prof[200] = clock64();
  if constexpr (REP) {
    const int L = a.L, lane = threadIdx.x & 31;
    for (int t = threadIdx.x >> 5; t < a.R * (L + 1); t += NT / 32) {
      const int rep = t / (L + 1), j = t - rep * (L + 1);
      double acc = 0.0;
      if (j == 0) {
        for (int b = lane; b < a.B; b += 32) acc += (double)__ldcg(a.nll_part + (int64_t)rep * a.B + b);
      } else {
        const double* kp = a.kl_part + ((int64_t)rep * L + j - 1) * gridDim.x;
        for (int c = lane; c < (int)gridDim.x; c += 32) acc += __ldcg(kp + c);
      }
      acc = warp_sum(acc);
      if (lane == 0) a.stats[(int64_t)rep * (L + 1) + j] = (float)acc;
    }
    if (threadIdx.x == 0) {
      *a.ticket = 0u;
      *a.step_dev = step + 1;
    }
  } else {
    for (int l = 0; l < a.L; ++l) {
      double acc = 0.0;
      for (int c = threadIdx.x; c < (int)gridDim.x; c += NT) acc += __ldcg(a.kl_part + (int64_t)l * gridDim.x + c);
      const double tot = block_sum(acc, dred);
      if (threadIdx.x == 0) {
        if (DP) {          // this rank's part of the layer's KL (its shard; rank 0: + the biases) -> every rank
          for (int p = 0; p < a.dp_world; ++p) a.dp_klx[p][a.dp_rank * kMaxL + l] = tot;
        } else a.stats[1 + l] = (float)tot;
      }
      __syncthreads();
    }
    if (DP && threadIdx.x == 0) {
      // closing exchange: every rank's parameter stores and KL partials have landed before anyone's next launch reads them
      const unsigned e = (unsigned)(*(volatile unsigned long long*)a.dp_epoch) + 1u;
      if (a.prof) a.prof[201] = clock64();
      dp_flag_exchange(a, e);
      if (a.prof) a.prof[202] = clock64();
      *a.dp_epoch = e;
      for (int l = 0; l < a.L; ++l) {
        double tot = 0.0;
        for (int q = 0; q < a.dp_world; ++q) tot += *(volatile double*)(a.dp_klx[a.dp_rank] + q * kMaxL + l);
        a.stats[1 + l] = (float)tot;
      }
    }
    {  // nll partials of the loss phase (written by this launch or, data-parallel, by the preceding one)
      double acc = 0.0;
      for (int c = threadIdx.x; c < a.nll_ctas; c += NT) acc += (double)__ldcg(a.nll_part + c);
      const double tot = block_sum(acc, dred);
      if (threadIdx.x == 0) a.stats[0] = (float)tot;
    }
    if (threadIdx.x == 0) {
      *a.ticket = 0u;
      *a.step_dev = step + 1;
    }
  }
}

// ---- small classifier head (last layer, N <= 32) --------------------------------------------------------------------
// A 600 -> 10 layer is 0.2 % of the step's FLOPs; as generic split-K tiles it costs a GEMM phase, an epilogue phase and a
// backward phase of fixed overheads.  Instead: M, V of the layer are computed once per launch (elementwise, at kernel
// start); `last_fwd_loss` gives every batch row to one CTA (warps own classes, lanes stride the contraction, so the
// sums have a fixed order) and goes straight on to log-softmax / nll / dlogits; `last_bwd` is elementwise over the
// (batch, in) inputs for dX and over the (out, in) weights for dM, dV.
template <bool REP>
__device__ void last_moments(const DevStep& a) {
  const DevLayer& y = a.ly[a.L - 1];
  const int64_t n = (int64_t)y.N * y.K;
  const float* mu = a.flat + y.off_mu;
  const float* rho = a.flat + y.off_rho;
  const float* lam = a.flat + y.off_lam;
  for (int64_t ge = (int64_t)blockIdx.x * NT + threadIdx.x; ge < REP_SEL(a.R * n, n); ge += (int64_t)gridDim.x * NT) {
    const int rep = REP_SEL((int)(ge / n), 0);
    const int64_t e = REP_SEL(ge - rep * n + rep * a.p_stride, ge);   // parameter side; the moments go to the replica's block
    const Moments mo = weight_moments(__ldg(mu + e), sigma_of(__ldg(rho + e)), alpha_of(__ldg(lam + e)), y.var_mode);
    REP_SEL(a.mv_last + rep * (a.w_stride - a.p_stride), a.mv_last)[e] = mo.m;
    REP_SEL(a.mv_last + rep * (a.w_stride - a.p_stride), a.mv_last)[n + e] = mo.v;
  }
}

// (replica launch: the R x B rows of all replicas, replica-major, at most NT / 32 per CTA; row g's nll goes to nll_part[g])
template <bool REP>
__device__ void last_fwd_loss(const DevStep& a, int64_t step, float* __restrict__ sm) {
  const int l = a.L - 1;
  const DevLayer& y = a.ly[l];
  const int B = a.B, K = y.K, N = y.N;
  if ((int)blockIdx.x >= a.nll_ctas) return;
  const int rows = (REP_SEL(a.R * B, B) + a.nll_ctas - 1) / a.nll_ctas;
  const int b0 = blockIdx.x * rows;
  const int nrow = min(rows, REP_SEL(a.R * B, B) - b0);
  const float* xin = l == 0 ? a.x : a.ly[l - 1].act;
  const float* M = a.mv_last;
  const float* V = a.mv_last + (int64_t)N * K;
  const float* bmu = a.flat + y.off_bmu;
  const float* brho = a.flat + y.off_brho;
  const uint64_t stream = (uint64_t)l + (uint64_t)step * (uint64_t)a.L;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = NT / 32;
  float* logit = sm;               // [rows][N]
  float* wred = sm + rows * N;     // [NW][2 N] per-warp partial sums of the current row
  for (int r = 0; r < nrow; ++r) {
    const int rep = REP_SEL((b0 + r) / B, 0), b = REP_SEL(b0 + r - rep * B, b0 + r);   // replica, its row
    const int64_t wo = REP_SEL(rep * a.w_stride, 0), po = REP_SEL(rep * a.p_stride, 0);
    const float* xr = REP_SEL((l == 0 ? xin + rep * a.x_stride : xin + wo) + (int64_t)b * K, xin + (int64_t)(b0 + r) * K);
    // the epilogue's noise and bias terms do not depend on the sums: computed while the loads below are in flight
    float ep = 0.f, sb2 = 0.f, bm = 0.f;
    if (threadIdx.x < N) {
      const int64_t ei = (int64_t)(b0 + r) * N + threadIdx.x;
      ep = y.eps ? __ldg(y.eps + ei) : philox_normal1(REP_SEL(__ldg(a.seeds + rep), a.seed), stream, REP_SEL((uint64_t)(b * N + threadIdx.x), (uint64_t)ei));
      const float sb = sigma_of(__ldg(REP_SEL(brho + po, brho) + threadIdx.x));
      sb2 = sb * sb;
      bm = __ldg(REP_SEL(bmu + po, bmu) + threadIdx.x);
    }
    // all threads stride the contraction; five classes' M, V loads (up to 30 per thread) are in flight together
    for (int n0 = 0; n0 < N; n0 += 5) {
      float e[5] = {0.f, 0.f, 0.f, 0.f, 0.f}, s_[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
      for (int k0 = threadIdx.x; k0 < K; k0 += NT * 3) {
        float xv[3], mv[5][3], vv[5][3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const int k = k0 + q * NT;
          xv[q] = k < K ? (l == 0 ? __ldg(xr + k) : __ldcg(xr + k)) : 0.f;
#pragma unroll
          for (int u = 0; u < 5; ++u) {
            const bool ok = k < K && n0 + u < N;
            mv[u][q] = ok ? __ldcg(REP_SEL(M + wo, M) + (int64_t)(n0 + u) * K + k) : 0.f;
            vv[u][q] = ok ? __ldcg(REP_SEL(V + wo, V) + (int64_t)(n0 + u) * K + k) : 0.f;
          }
        }
#pragma unroll
        for (int q = 0; q < 3; ++q)
#pragma unroll
          for (int u = 0; u < 5; ++u) {
            e[u] = fmaf(xv[q], mv[u][q], e[u]);
            s_[u] = fmaf(xv[q] * xv[q], vv[u][q], s_[u]);
          }
      }
#pragma unroll
      for (int u = 0; u < 5; ++u) {
        const float E = warp_sum(e[u]), S = warp_sum(s_[u]);
        if (lane == 0 && n0 + u < N) { wred[warp * 2 * N + n0 + u] = E; wred[warp * 2 * N + N + n0 + u] = S; }
      }
    }
    __syncthreads();
    if (threadIdx.x < N) {
      const int n = threadIdx.x;
      float E = 0.f, S = 0.f;
#pragma unroll
      for (int w = 0; w < NW; ++w) { E += wred[w * 2 * N + n]; S += wred[w * 2 * N + N + n]; }   // fixed order
      const int64_t ei = REP_SEL(wo + (int64_t)b * N + n, (int64_t)(b0 + r) * N + n);
      const float sd = sqrtf(S + sb2);
      const float v = fmaf(sd, ep, E + bm);
      logit[r * N + n] = v;
      y.act[ei] = v;
      y.dsf[ei] = ep / (2.0f * sd);
    }
    __syncthreads();
  }
  __syncthreads();
  if constexpr (REP) {
    if (warp < nrow) {
      const int g = b0 + warp, rep = g / B, b = g - rep * B;
      const int64_t o = rep * a.w_stride + (int64_t)b * N;
      const float nll = row_nll(logit + warp * N, N, a.y[rep * a.y_stride + b], y.dE + o, y.dS + o, y.dsf + o);
      if (lane == 0) a.nll_part[g] = nll;
    }
    return;
  }
  float local = 0.f;
  if (warp < nrow) {
    const int b = b0 + warp;
    const float* row = logit + warp * N;
    float mx = -INFINITY;
    for (int n = lane; n < N; n += 32) mx = fmaxf(mx, row[n]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.f;
    for (int n = lane; n < N; n += 32) se += expf(row[n] - mx);
    se = warp_sum(se);
    const float lse = mx + logf(se);
    const int64_t tgt = a.y[b];
    for (int n = lane; n < N; n += 32) {
      const int64_t e = (int64_t)b * N + n;
      const float lp = row[n] - lse;
      const float gd = expf(lp) - (n == tgt ? 1.0f : 0.0f);
      y.dE[e] = gd;
      y.dS[e] = gd * y.dsf[e];
      if (n == tgt) local -= lp;
    }
  }
  __syncthreads();
  const float tot = block_sum(local, sm);
  if (threadIdx.x == 0) a.nll_part[blockIdx.x] = tot;
}

// (replica launch: both index spaces run over all replicas, replica-major)
template <bool REP>
__device__ void last_bwd(const DevStep& a, float* __restrict__ sm) {
  const int l = a.L - 1;
  const DevLayer& y = a.ly[l];
  const int B = a.B, K = y.K, N = y.N;
  const float* M = a.mv_last;
  const float* V = a.mv_last + (int64_t)N * K;
  const float* xin = l == 0 ? a.x : a.ly[l - 1].act;
  const int G = gridDim.x;
  // dX (+ relu mask and ds_factor of the layer below): one (b, k) per thread, contraction over the N classes;
  // loads of up to 8 classes in flight before their FMAs.  CTAs are taken from the front of the grid.
  if (l > 0) {
    const DevLayer& p = a.ly[l - 1];
    for (int64_t ge = (int64_t)blockIdx.x * NT + threadIdx.x; ge < REP_SEL(a.R * (int64_t)B * K, (int64_t)B * K); ge += (int64_t)G * NT) {
      const int rep = REP_SEL((int)(ge / ((int64_t)B * K)), 0);
      const int64_t wo = REP_SEL(rep * a.w_stride, 0), e = REP_SEL(ge - rep * (int64_t)B * K + wo, ge);   // e: in the replica's block
      const int b = REP_SEL((int)((e - wo) / K), (int)(e / K)), k = REP_SEL((int)(e - wo - (int64_t)b * K), (int)(e - (int64_t)b * K));
      const float xv = __ldcg(p.act + e), fv = __ldcg(p.dsf + e);
      float de = 0.f, ds = 0.f;
      for (int n0 = 0; n0 < N; n0 += 8) {
        float ge_[8], gs[8], mm[8], vv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int n = n0 + u;
          const bool ok = n < N;
          ge_[u] = ok ? __ldcg(REP_SEL(y.dE + wo, y.dE) + (int64_t)b * N + n) : 0.f;
          gs[u] = ok ? __ldcg(REP_SEL(y.dS + wo, y.dS) + (int64_t)b * N + n) : 0.f;
          mm[u] = ok ? __ldcg(REP_SEL(M + wo, M) + (int64_t)n * K + k) : 0.f;
          vv[u] = ok ? __ldcg(REP_SEL(V + wo, V) + (int64_t)n * K + k) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) { de = fmaf(ge_[u], mm[u], de); ds = fmaf(gs[u], vv[u], ds); }
      }
      const float dx = xv > 0.f ? fmaf(2.0f * xv, ds, de) : 0.f;
      p.dE[e] = dx;
      p.dS[e] = dx * fv;
    }
  }
  // dM = dE^T x, dV = dS^T x^2 (+ the bias column sums): CTAs from the BACK of the grid take (32-wide chunk of k) x (quarter
  // of the 2 N output rows) tasks -- with whole chunks, 19 CTAs worked ~8.7 us at MNIST shape while 277 waited at the grid
  // barrier.  dE, dS and the chunk's columns of x are staged in shared memory (compact loops: this code runs once per
  // launch on a few CTAs, so its instruction footprint matters more than its issue rate); one (class, k) output per thread,
  // the batch summed in order.
  constexpr int NW = NT / 32;
  const int nchunk = (K + 31) / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* gE = sm;                    // [B][N]
  float* gS = gE + B * N;            // [B][N]
  float* xs = gS + B * N;            // [B][32]
  constexpr int kJSplit = 4;
  const int jper = (2 * N + kJSplit - 1) / kJSplit;
  for (int gtask = G - 1 - (int)blockIdx.x; gtask < REP_SEL(a.R * nchunk * kJSplit, nchunk * kJSplit); gtask += G) {
    const int rep = REP_SEL(gtask / (nchunk * kJSplit), 0), task = REP_SEL(gtask - rep * nchunk * kJSplit, gtask);
    const int64_t wo = REP_SEL(rep * a.w_stride, 0);
    const float* xr = REP_SEL(l == 0 ? xin + rep * a.x_stride : xin + wo, xin);
    const int chunk = task / kJSplit, js = task - chunk * kJSplit;
    const int j_lo = js * jper, j_hi = min(2 * N, j_lo + jper);
    __syncthreads();
    for (int i0 = threadIdx.x; i0 < B * N; i0 += NT * 4) {
      float te[4], ts[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = i0 + q * NT;
        te[q] = i < B * N ? __ldcg(REP_SEL(y.dE + wo, y.dE) + i) : 0.f;
        ts[q] = i < B * N ? __ldcg(REP_SEL(y.dS + wo, y.dS) + i) : 0.f;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = i0 + q * NT;
        if (i < B * N) { gE[i] = te[q]; gS[i] = ts[q]; }
      }
    }
    const int k = chunk * 32 + lane;
    for (int b0 = warp; b0 < B; b0 += NW * 4) {
      float xv[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int b = b0 + q * NW;
        xv[q] = (k < K && b < B) ? (l == 0 ? __ldg(xr + (int64_t)b * K + k) : __ldcg(xr + (int64_t)b * K + k)) : 0.f;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int b = b0 + q * NW;
        if (b < B) xs[b * 32 + lane] = xv[q];
      }
    }
    __syncthreads();
    for (int o = threadIdx.x; o < (j_hi - j_lo) * 32; o += NT) {
      const int ln = o & 31, j = j_lo + (o >> 5);      // j in [0, 2N): dM rows then dV rows
      const bool sq = j >= N;
      const float* src = (sq ? gS : gE) + (sq ? j - N : j);
      float a0 = 0.f, a1 = 0.f;
      int b = 0;
#pragma unroll 4
      for (; b + 1 < B; b += 2) {
        const float x0 = xs[b * 32 + ln], x1 = xs[(b + 1) * 32 + ln];
        a0 = fmaf(src[b * N], sq ? x0 * x0 : x0, a0);
        a1 = fmaf(src[(b + 1) * N], sq ? x1 * x1 : x1, a1);
      }
      if (b < B) { const float x0 = xs[b * 32 + ln]; a0 = fmaf(src[b * N], sq ? x0 * x0 : x0, a0); }
      const int kk = chunk * 32 + ln;
      if (kk < K) REP_SEL((sq ? y.dV : y.dM) + wo, (sq ? y.dV : y.dM))[(int64_t)(sq ? j - N : j) * K + kk] = a0 + a1;
    }
    if (chunk == nchunk - 1 && js == 0) {   // bias column sums over the batch: a warp per column, lanes over b, fixed shuffle tree
      for (int n = warp; n < 2 * N; n += NW) {
        const float* src = n < N ? gE : gS;
        const int c = n < N ? n : n - N;
        float s_ = 0.f;
        for (int b = lane; b < B; b += 32) s_ += src[b * N + c];
        s_ = warp_sum(s_);
        if (lane == 0) REP_SEL(y.colsum + wo, y.colsum)[n] = s_;
      }
    }
  }
}

// REP: the replica launch -- every phase's work items (and the elementwise index spaces) run over all a.R replicas,
// replica-major; the phases and grid barriers are the single network's.  DP and REP are exclusive.
template <bool DP, bool REP>
__global__ void __launch_bounds__(NT, kCtasPerSm) lrt_step_kernel(const __grid_constant__ DevStep a) {
  extern __shared__ __align__(16) float sm[];
  cg::grid_group grid = cg::this_grid();
  const int64_t step = *a.step_dev;  // read before anyone can bump it (the bump follows a grid-wide ticket)
  const int G = gridDim.x;
  const int R = REP ? a.R : 1;
  float* W = sm + kWOff;
  int slot = 0;
  stamp(a, slot);
  // Update overlap: with forward+backward and update in one launch, layers >= 1 are updated during layer 0's dW phase by
  // the CTAs that have no dW tile there (their raw gradients are final after phase B_1), if enough CTAs are idle.
  int u_first = 0;
  if (!REP && a.overlap_update && (a.phases & 3) == 3 && a.L >= 2) {
    const int nw0 = a.ly[0].w_rtiles * a.ly[0].w_ctiles;
    if (nw0 < G && (G - nw0) * 8 >= G) u_first = 1;
  }
  if (a.phases & 1) {
    // W tiles of this CTA's first item of a backward phase (dX items come first, then dW items)
    auto bwd_stage_w = [&](int l) {
      const DevLayer& y = a.ly[l];
      const int nx = l > 0 ? R * y.x_ctiles * y.x_splits : 0;
      const int item = blockIdx.x;
      if (item < nx) { dx_stage_w<REP>(a, l, item, W); return true; }
      if (item < nx + R * y.w_rtiles * y.w_ctiles) { dw_stage_w<REP>(a, l, item - nx, W); return true; }
      return false;
    };
    const int Lg = a.small_last ? a.L - 1 : a.L;   // layers that go through the generic tiled phases
    if (a.small_last) last_moments<REP>(a);
    bool staged = false;
    if (Lg > 0 && (int)blockIdx.x < R * a.ly[0].f_ntiles * a.ly[0].f_splits) { fwd_stage_w<REP>(a, 0, blockIdx.x, W); staged = true; }
    for (int rep = 0; rep < ((a.phases & 4) ? 2 : 1); ++rep)   // phases bit 2: debug, run the forward twice
    for (int l = 0; l < Lg; ++l) {
      const DevLayer& y = a.ly[l];
      for (int item = blockIdx.x; item < R * y.f_ntiles * y.f_splits; item += G) {
        // a CTA's next item overwrites the operand tiles, which an item with one thread group (TileCfg.G == 1) leaves
        // without a closing barrier; replica launches run many items per CTA
        if constexpr (REP) if (item != (int)blockIdx.x) __syncthreads();
        fwd_item<REP>(a, l, item, sm, staged && item == (int)blockIdx.x);
      }
      __syncthreads();
      // next GEMM phase's weight-side tiles, staged while the other CTAs finish
      if (l + 1 < Lg) {
        staged = (int)blockIdx.x < R * a.ly[l + 1].f_ntiles * a.ly[l + 1].f_splits;
        if (staged) fwd_stage_w<REP>(a, l + 1, blockIdx.x, W);
      } else {
        staged = a.small_last ? (Lg > 0 ? bwd_stage_w(Lg - 1) : false) : bwd_stage_w(a.L - 1);
      }
      stamp(a, slot);
      grid.sync();
      stamp(a, slot);
      if (l < a.L - 1) fwd_epilogue<REP>(a, l, step);
      else if constexpr (REP) loss_epilogue_rows(a, step, sm);
      else loss_epilogue(a, step, sm);
      stamp(a, slot);
      grid.sync();
      stamp(a, slot);
    }
    if (a.small_last) {
      if (Lg == 0) grid.sync();   // single-layer network: mv_last must be complete
      last_fwd_loss<REP>(a, step, sm);
      stamp(a, slot);
      grid.sync();
      stamp(a, slot);
      last_bwd<REP>(a, sm);
      stamp(a, slot);
      if (Lg > 0 || (a.phases & 2)) grid.sync();
      stamp(a, slot);
    }
    for (int l = Lg - 1; l >= 0; --l) {
      const DevLayer& y = a.ly[l];
      const int nx = l > 0 ? R * y.x_ctiles * y.x_splits : 0;
      const int nw = R * y.w_rtiles * y.w_ctiles;
      for (int item = blockIdx.x; item < nx + nw; item += G) {
        if constexpr (REP) if (item != (int)blockIdx.x) __syncthreads();   // as in the forward phases
        const bool st = staged && item == (int)blockIdx.x;
        if (item < nx) dx_item<REP>(a, l, item, sm, st);
        else dw_item<REP>(a, l, item - nx, sm, st);
      }
      __syncthreads();
      staged = l > 0 ? bwd_stage_w(l - 1) : false;
      if (!REP && l == 0 && u_first == 1) {
        // the raw gradients of layers >= 1 are complete: the CTAs without a layer-0 dW tile update those layers now
        const int busy = min(G, nw);
        if ((int)blockIdx.x >= busy) {
          if constexpr (!REP) update_layers<DP>(a, step, 1, a.L, blockIdx.x - busy, G - busy, sm);
        } else if (threadIdx.x == 0) {
          for (int ll = 1; ll < a.L; ++ll) a.kl_part[(int64_t)ll * G + blockIdx.x] = 0.0;
        }
      }
      stamp(a, slot);
      if (l > 0 || (a.phases & 2)) grid.sync();
      stamp(a, slot);
      if (l > 0 && y.x_splits > 1) {
        dx_epilogue<REP>(a, l);
        stamp(a, slot);
        grid.sync();
        stamp(a, slot);
      }
    }
  }
  if (a.phases & 2) {
    if (DP) {
      // every rank's raw gradients are complete (the grid barrier above + the peers' flags) before anyone reduces them
      if (blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned e = (unsigned)(*(volatile unsigned long long*)a.dp_epoch) + 1u;
        dp_flag_exchange(a, e);
        *a.dp_epoch = e;
      }
      stamp(a, slot);
      grid.sync();
      stamp(a, slot);
    }
    if constexpr (REP) update_layers_rep(a, step, sm);
    else update_layers<DP>(a, step, 0, u_first ? 1 : a.L, blockIdx.x, G, sm);   // layers >= 1 were done during B_0 if u_first
    stamp(a, slot);
    finish_step<DP, REP>(a, step, sm);
  }
  stamp(a, slot);
}

// ================================================================================================
// host: schedule + workspace layout
// ================================================================================================
size_t align256(size_t v) { return (v + 255) & ~size_t(255); }
int r4(int v) { return (v + 3) & ~3; }
int r8(int v) { return (v + 7) & ~7; }
int cdiv(int a, int b) { return (a + b - 1) / b; }

struct HostPlan {
  DevStep d;
  size_t smem;
  size_t off_raw, raw_floats, total;
  size_t rep_bytes;   // one replica's block of the workspace (raw gradients .. mv_last); the shared tail follows R of them
};

// per-item cost model in SM clocks (L2 -> SM at ~40 B/clk/SM, FFMA at ~70% of 128/clk)
double fma_clk(double fma) { return fma / (128.0 * 0.7); }

// Measured on B200 (profiles/r01_step_phases.txt): the MAC loop issues ~75 instructions per contraction step per warp at
// ~85% of the issue rate; a staging pass costs ~600 clk + ~450 clk per float4 unit per thread; the group reduction
// ~1000 clk + ~450 clk per extra group; writing a tile out ~1500 clk.
double mac_clk(const TileCfg& c) {
  const double warps_per_sched = std::ceil(c.G * c.TPG / 32.0) * kCtasPerSm / 4.0;
  return std::max(1.0, warps_per_sched) * c.kpg * 75.0 / 0.85 + 400.0;
}
double stage_clk(double float4_units) { return 600.0 + 450.0 * float4_units / NT; }
double reduce_clk(const TileCfg& c) { return (c.G > 1 ? 1000.0 + 450.0 * (c.G - 1) : 0.0) + 1500.0; }

// LBBNN_STEP_PLAN_L<l> = "bn,fsplits,rn,ck,bk,xsplits" forces layer l's forward column tile and split count, dW tile and
// dX column tile and split count (0 = left to the cost model; layer 0 has no dX phase).  v = all zeros when unset.
int env_plan(int l, int v[6]) {
  char name[64];
  snprintf(name, sizeof(name), "LBBNN_STEP_PLAN_L%d", l);
  for (int i = 0; i < 6; ++i) v[i] = 0;
  const char* s = getenv(name);
  if (!s) return LBBNN_OK;
  int end = -1;
  const int got = sscanf(s, "%d,%d,%d,%d,%d,%d%n", &v[0], &v[1], &v[2], &v[3], &v[4], &v[5], &end);
  bool ok = got == 6 && end >= 0 && s[end] == '\0';
  for (int i = 0; i < 6; ++i) ok = ok && v[i] >= 0;
  LBBNN_REQUIRE(ok, "%s=\"%s\": expected bn,fsplits,rn,ck,bk,xsplits (integers >= 0, 0 = free)", name, s);
  LBBNN_REQUIRE(l > 0 || (v[4] == 0 && v[5] == 0), "%s=\"%s\": layer 0 has no dX phase, bk and xsplits must be 0", name, s);
  return LBBNN_OK;
}

int plan_step_uncached(const lbbnn_step* S, int G, int R, const int (*ov)[6], bool generic_head, HostPlan* out);

// The schedule search costs ~1 ms; cache it per (G, replicas, batch, shapes, overrides) so eager (non-graph) steps do not pay
// it.  The overrides are part of the key: setting or clearing one replans.  R = 1 is the single-network step.
int plan_step(const lbbnn_step* S, int G, int R, HostPlan* out) {
  static std::mutex mu;
  static std::vector<int64_t> cached_key;
  static HostPlan cached;
  LBBNN_REQUIRE(S != nullptr, "step is NULL");
  std::vector<int64_t> key = {G, S->n_layers, S->batch, R};
  const bool sane = S->n_layers >= 1 && S->n_layers <= kMaxL;
  int ov[kMaxL][6] = {};
  for (int l = 0; sane && l < S->n_layers; ++l) {
    key.push_back(S->layer[l].in_features);
    key.push_back(S->layer[l].out_features);
    if (int rc = env_plan(l, ov[l])) return rc;
    key.insert(key.end(), ov[l], ov[l] + 6);
  }
  const bool generic_head = getenv("LBBNN_STEP_GENERIC_HEAD") != nullptr;
  key.push_back(generic_head);
  std::lock_guard<std::mutex> lock(mu);
  if (!sane || key != cached_key) {
    HostPlan P;
    if (int rc = plan_step_uncached(S, G, R, ov, generic_head, &P)) return rc;
    cached = P;
    cached_key = key;
  }
  *out = cached;
  // everything that is not schedule comes from the caller's struct
  for (int l = 0; l < S->n_layers; ++l) {
    const lbbnn_step_layer& s = S->layer[l];
    LBBNN_REQUIRE(s.var_mode == LBBNN_VAR_REFERENCE || s.var_mode == LBBNN_VAR_EXACT, "bad var_mode");
    LBBNN_REQUIRE((s.off_weight_mu | s.off_weight_rho | s.off_lambdal) % 4 == 0, "flat offsets of the weight tensors must be multiples of 4 floats");
    DevLayer& y = out->d.ly[l];
    y.off_mu = s.off_weight_mu; y.off_rho = s.off_weight_rho; y.off_lam = s.off_lambdal;
    y.off_bmu = s.off_bias_mu; y.off_brho = s.off_bias_rho;
    y.eps = s.eps; y.pri = s.priors; y.var_mode = s.var_mode;
  }
  return LBBNN_OK;
}

// R replicas of the network share every phase: a phase's item count is R times the single network's, which the cost model
// sees through the rounds of items per CTA (R = 1: the single-network plan).
int plan_step_uncached(const lbbnn_step* S, int G, int R, const int (*ovr)[6], bool generic_head, HostPlan* out) {
  LBBNN_REQUIRE(S != nullptr, "step is NULL");
  LBBNN_REQUIRE(S->n_layers >= 1 && S->n_layers <= kMaxL, "n_layers must be 1..%d", kMaxL);
  LBBNN_REQUIRE(S->batch >= 1 && S->batch <= 128, "the fused step kernel handles batch <= 128 (got %lld)", (long long)S->batch);
  HostPlan P;
  memset(&P, 0, sizeof(P));
  DevStep& d = P.d;
  d.L = S->n_layers;
  d.B = (int)S->batch;
  const int B = d.B, RPB = r4(B), RGB = RPB / 4;
  size_t smem = 32 * sizeof(double);
  size_t part_floats = 0;
  static const int kBn[] = {8, 16, 24, 32, 40, 48, 56, 64, 80, 96, 104, 128, 160};
  static const int kRn[] = {8, 12, 16, 20, 24, 32, 40, 48, 64};
  static const int kCk[] = {16, 24, 32, 40, 48, 56, 64, 80, 96, 112, 128};
  static const int kBk[] = {8, 16, 24, 32, 40, 48, 64, 80, 96, 104, 128, 160};
  for (int l = 0; l < d.L; ++l) {
    const lbbnn_step_layer& s = S->layer[l];
    LBBNN_REQUIRE(s.in_features > 0 && s.out_features > 0 && s.in_features < (1 << 24) && s.out_features < (1 << 24), "bad layer %d shape", l);
    LBBNN_REQUIRE(l == 0 || s.in_features == S->layer[l - 1].out_features, "layer %d input width does not chain", l);
    LBBNN_REQUIRE(s.var_mode == LBBNN_VAR_REFERENCE || s.var_mode == LBBNN_VAR_EXACT, "bad var_mode");
    LBBNN_REQUIRE((s.off_weight_mu | s.off_weight_rho | s.off_lambdal) % 4 == 0, "flat offsets of the weight tensors must be multiples of 4 floats");
    DevLayer& y = d.ly[l];
    y.K = (int)s.in_features; y.N = (int)s.out_features;
    y.off_mu = s.off_weight_mu; y.off_rho = s.off_weight_rho; y.off_lam = s.off_lambdal;
    y.off_bmu = s.off_bias_mu; y.off_brho = s.off_bias_rho;
    y.eps = s.eps; y.pri = s.priors; y.var_mode = s.var_mode;
    const int K = y.K, N = y.N;
    const int* ov = ovr[l];
    const bool forced = ov[0] || ov[1] || ov[2] || ov[3] || ov[4] || ov[5];
    auto red_floats = [](const TileCfg& c) {
      return (size_t)(c.G <= 1 ? 0 : (c.G <= 8 ? c.G - 1 : (c.G + 1) / 2)) * 64 * c.TPG;
    };
    // ---- forward: column tile bn x contraction splits ----
    double best = 1e300;
    for (int bn : kBn) {
      if (ov[0] && bn != ov[0]) continue;
      const int bnc = std::min(bn, r8(N));
      const int Cc = std::min(bnc, N);
      if (RGB * (r8(Cc) / 8) > NT) continue;
      const int ntiles = cdiv(N, bnc);
      const int max_splits = std::max(1, std::min(G / std::max(1, std::min(R * ntiles, G)), cdiv(K, 8)));
      // Replica launch: R multiplies the tiles, so the cap shrinks; past it the search goes on only as far as the first split
      // count whose chunk fits shared memory (and to a forced one), up to the single network's cap: every split count the
      // single network may run stays reachable.
      const int cap1 = std::max(1, std::min(G / std::max(1, std::min(ntiles, G)), cdiv(K, 8)));
      const int sp_end = R > 1 ? std::max({max_splits, cap1, ov[1]}) : max_splits;
      bool fit = false;
      for (int sp = 1; sp <= sp_end; ++sp) {
        if (sp > max_splits && fit && !ov[1]) break;
        if (ov[1] && sp != ov[1]) continue;
        const int kc = r4(cdiv(K, sp));
        const int s2 = cdiv(K, kc);
        const TileCfg c = make_cfg(B, Cc, kc, NT);
        if (std::max((size_t)c.KS * c.RP, red_floats(c)) > (size_t)kWOff || (size_t)2 * c.KS * c.CP > (size_t)kWFloats) continue;
        fit = true;
        const double rounds = cdiv(R * ntiles * s2, G);
        const double item = stage_clk(c.RP * c.KS / 4.0) + mac_clk(c) + reduce_clk(c) + 0.5 * stage_clk(3.0 * c.CP * c.KS / 4.0);
        // partials are written once and read once by the epilogue phase; the loss epilogue of the last layer
        // walks the splits serially (one warp per row, NT / 32 rows at a time)
        const double epi = l == d.L - 1 ? 2.0 * s2 * 60.0 * cdiv(cdiv(R * B, std::min(R * B, G)), NT / 32)
                                        : 2.0 * s2 * R * B * N * 4 / (40.0 * G) * 2 + 40.0 * s2;
        const double cost = rounds * item + epi;
        if (cost < best) {
          best = cost;
          y.f_bn = bnc; y.f_kc = kc; y.f_ntiles = ntiles; y.f_splits = s2;
        }
      }
    }
    LBBNN_REQUIRE(best < 1e300, "no forward schedule fits layer %d (%d -> %d) in shared memory%s", l, K, N,
                  forced ? " under the forced LBBNN_STEP_PLAN_L values" : "");
    part_floats = std::max(part_floats, (size_t)y.f_splits * 2 * B * N);
    // ---- backward: dW tiles (rn x ck) and dX tiles (bk columns x contraction splits) share a phase ----
    best = 1e300;
    for (int rn : kRn) {
      if (ov[2] && rn != ov[2]) continue;
      const int rnc = std::min(rn, r4(N));
      const int Rw = std::min(rnc, N);
      for (int ck : kCk) {
        if (ov[3] && ck != ov[3]) continue;
        const int ckc = std::min(ck, r8(K));
        const int Cw = std::min(ckc, K);
        if ((r4(Rw) / 4) * (r8(Cw) / 8) > NT) continue;
        const TileCfg cw = make_cfg(Rw, Cw, B, NT);
        if (std::max((size_t)2 * cw.KS * cw.RP, red_floats(cw)) > (size_t)kWOff || (size_t)cw.KS * cw.CP > (size_t)kWFloats) continue;
        const int nW = cdiv(N, rnc) * cdiv(K, ckc);
        const double cW = stage_clk(2.0 * cw.RP * cw.KS / 4.0) + mac_clk(cw) + reduce_clk(cw) + 0.5 * stage_clk(cw.CP * cw.KS / 4.0);
        const int nbk = l > 0 ? (int)(sizeof(kBk) / sizeof(int)) : 1;
        for (int bi = 0; bi < nbk; ++bi) {
          const int bk = kBk[bi];
          if (ov[4] && bk != ov[4]) continue;
          const int bkc = std::min(bk, r8(K));
          const int Cx = std::min(bkc, K);
          if (l > 0 && RGB * (r8(Cx) / 8) > NT) continue;
          const int xct = cdiv(K, bkc);
          const int max_sp = l > 0 ? std::max(1, std::min(cdiv(N, 4), G)) : 1;
          for (int sp = 1; sp <= max_sp; ++sp) {
            if (ov[5] && sp != ov[5]) continue;
            const int nc = r4(cdiv(N, sp));
            const int s2 = cdiv(N, nc);
            if (s2 != sp && sp > 1) continue;
            int nX = 0;
            double cX = 0.0, xe = 0.0;
            if (l > 0) {
              const TileCfg cx = make_cfg(B, Cx, nc, NT);
              if (std::max((size_t)2 * cx.KS * cx.RP, red_floats(cx)) > (size_t)kWOff || (size_t)2 * cx.KS * cx.CP > (size_t)kWFloats) continue;
              nX = xct * s2;
              cX = stage_clk(2.0 * cx.RP * cx.KS / 4.0) + mac_clk(cx) + reduce_clk(cx) + 1000.0 + 0.5 * stage_clk(3.0 * cx.CP * cx.KS / 4.0);
              if (s2 > 1) xe = 4500.0 + (double)s2 * R * B * K * 4 / (40.0 * G);
            }
            const double rounds = cdiv(R * (nW + nX), G);
            const double cost = rounds * std::max(cW, cX) + xe;
            if (cost < best) {
              best = cost;
              y.w_rn = rnc; y.w_ck = ckc; y.w_rtiles = cdiv(N, rnc); y.w_ctiles = cdiv(K, ckc);
              y.x_bk = bkc; y.x_nc = nc; y.x_ctiles = xct; y.x_splits = l > 0 ? s2 : 1;
            }
          }
        }
      }
    }
    LBBNN_REQUIRE(best < 1e300, "no backward schedule fits layer %d (%d -> %d) in shared memory%s", l, K, N,
                  forced ? " under the forced LBBNN_STEP_PLAN_L values" : "");
    y.fc = make_cfg(B, std::min(y.f_bn, N), y.f_kc, NT);
    y.wc = make_cfg(std::min(y.w_rn, N), std::min(y.w_ck, K), B, NT);
    y.xc = make_cfg(B, std::min(y.x_bk, K), y.x_nc, NT);
    if (l > 0 && y.x_splits > 1) part_floats = std::max(part_floats, (size_t)y.x_splits * B * K);
  }
  // loss epilogue: the logits of a CTA's rows in shared memory (the replica launch's loss_epilogue_rows: NT / 32 at a time)
  LBBNN_REQUIRE((size_t)std::min(NT / 32, cdiv(R * B, std::min(R * B, G))) * d.ly[d.L - 1].N + 64 <= (size_t)kWOff,
                "too many classes for the loss phase");
  smem = kSmemCap;
  d.R = R;
  d.nll_ctas = std::min(R * B, G);   // loss epilogue: ceil(R B / nll_ctas) rows per CTA, one warp per row
  {
    const int Nl = d.ly[d.L - 1].N;
    d.small_last = (Nl <= 32 && cdiv(R * B, d.nll_ctas) <= NT / 32 && 2 * B * Nl + 32 * B <= kWOff &&
                    !generic_head) ? 1 : 0;
  }
  LBBNN_REQUIRE(d.nll_ctas <= G, "batch too large for the loss phase");
  P.smem = smem;
  // workspace: R x [raw: dM,dV,colsum per layer | act,dsf,dE,dS per layer | partials | mv_last] | kl partials [R][L][G] |
  // nll partials (one per CTA; replica launch: one per row, [R][B]) | ticket
  size_t off = 0;
  P.off_raw = 0;
  for (int l = 0; l < d.L; ++l) {
    const size_t nk = (size_t)r4(d.ly[l].N * d.ly[l].K);
    off += 2 * nk + (size_t)r4(2 * d.ly[l].N);
  }
  P.raw_floats = off;
  off = align256(off * 4);
  for (int l = 0; l < d.L; ++l) off += 4 * align256((size_t)B * d.ly[l].N * 4);
  off += align256(part_floats * 4);
  off += align256((size_t)2 * d.ly[d.L - 1].N * d.ly[d.L - 1].K * 4);   // mv_last
  P.rep_bytes = off;
  d.w_stride = (int64_t)(off / 4);
  off *= R;
  off += align256((size_t)R * d.L * G * sizeof(double));
  off += align256((size_t)std::max(G, R * B) * sizeof(float));
  off += 256;
  P.total = off;
  *out = P;
  return LBBNN_OK;
}

void bind_workspace(HostPlan& P, char* ws, int G) {
  DevStep& d = P.d;
  float* raw = (float*)ws;
  size_t o = 0;
  for (int l = 0; l < d.L; ++l) {
    const size_t nk = (size_t)r4(d.ly[l].N * d.ly[l].K);
    d.ly[l].dM = raw + o; o += nk;
    d.ly[l].dV = raw + o; o += nk;
    d.ly[l].colsum = raw + o; o += (size_t)r4(2 * d.ly[l].N);
  }
  size_t off = align256(o * 4);
  for (int l = 0; l < d.L; ++l) {
    const size_t bn = align256((size_t)d.B * d.ly[l].N * 4);
    d.ly[l].act = (float*)(ws + off); off += bn;
    d.ly[l].dsf = (float*)(ws + off); off += bn;
    d.ly[l].dE = (float*)(ws + off); off += bn;
    d.ly[l].dS = (float*)(ws + off); off += bn;
  }
  d.part = (float*)(ws + off);
  off = P.rep_bytes - align256((size_t)2 * d.ly[d.L - 1].N * d.ly[d.L - 1].K * 4);
  d.mv_last = (float*)(ws + off);
  off = P.rep_bytes * d.R;
  d.kl_part = (double*)(ws + off); off += align256((size_t)d.R * d.L * G * sizeof(double));
  d.nll_part = (float*)(ws + off); off += align256((size_t)std::max(G, d.R * d.B) * sizeof(float));
  d.ticket = (unsigned*)(ws + off);
}

// `kernels`: the instantiations of lrt_step_kernel this translation unit launches (each must fit kCtasPerSm CTAs on an SM)
int step_grid(size_t smem, int* G, std::initializer_list<const void*> kernels) {
  static int cached_blocks = -1;
  static size_t cached_smem = 0;
  if (cached_blocks < 0 || smem > cached_smem) {
    for (const void* k : kernels) LBBNN_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap));
    for (const void* k : kernels) {
      int per_sm = 0;
      LBBNN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, NT, kSmemCap));
      LBBNN_REQUIRE(per_sm >= kCtasPerSm, "lrt_step_kernel does not fit %d CTAs on an SM", kCtasPerSm);
    }
    cached_blocks = sm_count() * kCtasPerSm;
    cached_smem = kSmemCap;
  }
  *G = cached_blocks;
  return LBBNN_OK;
}

// schedule dump for logs / DESIGN.md: "l0 F bn=.. splits=.. | W rn x ck (items) | X bk x splits (items); ... head=small|tiled smem=.."
// (head=small: the last layer runs last_fwd_loss / last_bwd, and its F / W / X entries are not used).  Items are per replica;
// the replica launch appends " replicas=R" when R > 1.
int describe_plan(const HostPlan& P, char* buf, size_t buf_bytes) {
  size_t o = 0;
  for (int l = 0; l < P.d.L && o < buf_bytes; ++l) {
    const DevLayer& y = P.d.ly[l];
    o += snprintf(buf + o, buf_bytes - o, "l%d(%d->%d) F bn=%d kc=%d items=%dx%d | W %dx%d items=%d | X bk=%d nc=%d items=%dx%d; ", l, y.K, y.N,
                  y.f_bn, y.f_kc, y.f_ntiles, y.f_splits, y.w_rn, y.w_ck, y.w_rtiles * y.w_ctiles, y.x_bk, y.x_nc,
                  l > 0 ? y.x_ctiles : 0, l > 0 ? y.x_splits : 0);
  }
  if (o < buf_bytes) o += snprintf(buf + o, buf_bytes - o, "head=%s smem=%zu", P.d.small_last ? "small" : "tiled", P.smem);
  if (P.d.R > 1 && o < buf_bytes) snprintf(buf + o, buf_bytes - o, " replicas=%d", P.d.R);
  return LBBNN_OK;
}

}  // namespace

// phase profile (lbbnn_lrt_step_profile): stamps buffer and stamped CTA of the following launches
extern long long* g_step_prof;
extern int g_step_prof_cta;
}  // namespace lbbnn
