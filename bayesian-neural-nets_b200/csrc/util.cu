// Error plumbing, noise export, loss head and optimizer kernels of liblbbnn.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace lbbnn {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
    return LBBNN_ERR_CUDA;
  }
  return LBBNN_OK;
}

int sm_count() {
  static int cached = 0;
  if (cached) return cached;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) == cudaSuccess &&
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
    cached = n;
  } else {
    cudaGetLastError();
    return 148;  // B200; only reached by size queries on a machine without a GPU
  }
  return cached;
}

namespace {

__global__ void philox_export_kernel(float* __restrict__ out, int64_t n, uint64_t seed, uint64_t stream, int normal) {
  const int64_t nquads = ceil_div(n, 4);
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nquads; q += (int64_t)gridDim.x * blockDim.x) {
    float v[4];
    if (normal) philox_normal4(seed, stream, (uint64_t)q, v);
    else philox_uniform4(seed, stream, (uint64_t)q, v);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (q * 4 + j < n) out[q * 4 + j] = v[j];
  }
}

int philox_export(float* out, int64_t n, uint64_t seed, uint64_t stream_id, int normal, lbbnn_stream s) {
  LBBNN_REQUIRE(out && n >= 0, "bad output");
  if (n == 0) return LBBNN_OK;
  int64_t blocks = ceil_div(ceil_div(n, 4), 256);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  philox_export_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(out, n, seed, stream_id, normal);
  return check_launch("philox_export");
}

// one warp per row: log_softmax(dim=1), nll(sum) and its gradient (LRT:210,223); single block so the
// nll sum has a fixed order
__global__ void logsoftmax_nll_kernel(const float* __restrict__ logits, const int64_t* __restrict__ target, int64_t B,
                                      int64_t C, float* __restrict__ logp, float* __restrict__ nll_sum,
                                      float* __restrict__ dlogits, float gscale, int64_t* step_inc) {
  __shared__ float red[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float local = 0.f;
  for (int64_t b = warp; b < B; b += nw) {
    const float* row = logits + b * C;
    float mx = -INFINITY;
    for (int64_t c = lane; c < C; c += 32) mx = fmaxf(mx, row[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.f;
    for (int64_t c = lane; c < C; c += 32) se += expf(row[c] - mx);
    se = warp_sum(se);
    const float lse = mx + logf(se);
    const int64_t t = target[b];
    for (int64_t c = lane; c < C; c += 32) {
      const float lp = row[c] - lse;
      if (logp) logp[b * C + c] = lp;
      if (dlogits) dlogits[b * C + c] = gscale * (expf(lp) - (c == t ? 1.0f : 0.0f));
      if (c == t) local -= lp;
    }
  }
  const float tot = block_sum(local, red);
  if (threadIdx.x == 0) {
    if (nll_sum) *nll_sum = tot;
    if (step_inc) *step_inc += 1;
  }
}

// The whole objective of a minibatch (LRT:221-224, MNF:267-270) in one block: the kernel above plus
//   loss = nll + sum_i scale_i term_i         out = [loss, nll]
// (scale_i = 1 / NUM_BATCHES for the layers' kl; the MF script's ELBO, MF:316-318, is the same with its log q terms at
// + 1 / NUM_BATCHES and its log prior terms at - 1 / NUM_BATCHES)
// so that a module-level training step (GraphedTrainer) goes from the logits straight to d loss / d logits: the torch
// formulation (log_softmax, nll_loss, the sum over the layers' kl, / NUM_BATCHES, + and their backward nodes) was ~20
// launches of 1-6 us each on the critical path between the forward and the backward.
constexpr int kMaxKlTerms = 16;
struct ObjectiveArgs {
  const float* logits;
  const int64_t* target;
  int64_t B, C;
  const float* kl[kMaxKlTerms];
  float scale[kMaxKlTerms];
  int n_kl;
  float *out, *dlogits;
};
__global__ void __launch_bounds__(1024) objective_kernel(const ObjectiveArgs a) {
  __shared__ float red[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // G lanes per row: 4 / 2 / 1 rows per warp pass for <= 8 / <= 16 / more classes (a 100 x 10 batch is one pass of the block,
  // not four dependent load -> max -> exp -> sum -> log chains per warp)
  const int G = a.C <= 8 ? 8 : (a.C <= 16 ? 16 : 32);
  const int gl = lane & (G - 1), rows_per_pass = nw * (32 / G);
  float local = 0.f;
  for (int64_t b0 = 0; b0 < a.B; b0 += rows_per_pass) {             // uniform trip count: the shuffles below are warp-wide
    const int64_t b = b0 + warp * (32 / G) + lane / G;
    const bool ok = b < a.B;
    const float* row = a.logits + (ok ? b : 0) * a.C;
    float mx = -INFINITY;
    for (int64_t c = gl; c < a.C; c += G) mx = fmaxf(mx, row[c]);
    for (int o = G >> 1; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float se = 0.f;
    for (int64_t c = gl; c < a.C; c += G) se += expf(row[c] - mx);
    for (int o = G >> 1; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
    const float lse = mx + logf(se);
    if (!ok) continue;
    const int64_t t = a.target[b];
    for (int64_t c = gl; c < a.C; c += G) {
      const float lp = row[c] - lse;
      if (a.dlogits) a.dlogits[b * a.C + c] = expf(lp) - (c == t ? 1.0f : 0.0f);
      if (c == t) local -= lp;
    }
  }
  const float nll = block_sum(local, red);
  if (threadIdx.x == 0) {
    float kl = 0.f;
    for (int i = 0; i < a.n_kl; ++i) kl = fmaf(a.scale[i], *a.kl[i], kl);   // in the order of sum(l.kl for l in layers)
    a.out[0] = nll + kl;
    a.out[1] = nll;
  }
}

// large batches: one warp per row over many blocks, per-block partial sums, then a fixed-order final sum
__global__ void __launch_bounds__(256) logsoftmax_nll_rows(const float* __restrict__ logits, const int64_t* __restrict__ target,
                                                           int64_t B, int64_t C, float* __restrict__ logp,
                                                           float* __restrict__ partial, float* __restrict__ dlogits,
                                                           float gscale) {
  __shared__ float red[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b = (int64_t)blockIdx.x * 8 + warp;
  float local = 0.f;
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
    const int64_t t = target[b];
    for (int64_t c = lane; c < C; c += 32) {
      const float lp = row[c] - lse;
      if (logp) logp[b * C + c] = lp;
      if (dlogits) dlogits[b * C + c] = gscale * (expf(lp) - (c == t ? 1.0f : 0.0f));
      if (c == t) local -= lp;
    }
  }
  const float tot = block_sum(local, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(256) nll_final_sum(const float* __restrict__ partial, int n, float* __restrict__ nll_sum,
                                                     int64_t* step_inc) {
  __shared__ double red[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += (double)partial[i];
  const double tot = block_sum(acc, red);
  if (threadIdx.x == 0) {
    if (nll_sum) *nll_sum = (float)tot;
    if (step_inc) *step_inc += 1;
  }
}

// torch.optim.Adam (single-tensor, non-amsgrad) on one flat fp32 buffer, 4 elements per thread
// bias corrections of step t, computed once (double pow) instead of in every block
__global__ void adam_prepare(const int64_t* __restrict__ step_dev, float lr, float b1, float b2, float* __restrict__ coef) {
  const double t = (double)(*step_dev);
  coef[0] = lr / (float)(1.0 - pow((double)b1, t));        // step_size = lr / bias_correction1
  coef[1] = (float)sqrt(1.0 - pow((double)b2, t));         // sqrt(bias_correction2)
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v, int64_t n,
                                                   float b1, float b2, float eps, const float* __restrict__ coef,
                                                   float decay) {       // decay = lr * weight_decay (AdamW), 0 for Adam
  const float step_size = __ldg(coef), bc2_sqrt = __ldg(coef + 1);
  const bool vec = (n % 4 == 0) && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v);
  const int64_t nq = ceil_div(n, 4);
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = q * 4;
    float pv[4], gv[4], mv[4], vv[4];
    if (vec && e0 + 3 < n) {
      const float4 a = *reinterpret_cast<const float4*>(p + e0), b = *reinterpret_cast<const float4*>(g + e0);
      const float4 c = *reinterpret_cast<const float4*>(m + e0), d = *reinterpret_cast<const float4*>(v + e0);
      pv[0] = a.x; pv[1] = a.y; pv[2] = a.z; pv[3] = a.w; gv[0] = b.x; gv[1] = b.y; gv[2] = b.z; gv[3] = b.w;
      mv[0] = c.x; mv[1] = c.y; mv[2] = c.z; mv[3] = c.w; vv[0] = d.x; vv[1] = d.y; vv[2] = d.z; vv[3] = d.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const bool ok = e0 + j < n;
        pv[j] = ok ? p[e0 + j] : 0.f; gv[j] = ok ? g[e0 + j] : 0.f;
        mv[j] = ok ? m[e0 + j] : 0.f; vv[j] = ok ? v[e0 + j] : 0.f;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (decay != 0.f) pv[j] *= 1.0f - decay;         // torch.optim.AdamW: param.mul_(1 - lr * weight_decay) first
      mv[j] = mv[j] + (gv[j] - mv[j]) * (1.0f - b1);   // lerp form, as torch's _single_tensor_adam
      vv[j] = b2 * vv[j] + (1.0f - b2) * gv[j] * gv[j];
      const float denom = sqrtf(vv[j]) / bc2_sqrt + eps;
      pv[j] -= step_size * (mv[j] / denom);
    }
    if (vec && e0 + 3 < n) {
      *reinterpret_cast<float4*>(p + e0) = make_float4(pv[0], pv[1], pv[2], pv[3]);
      *reinterpret_cast<float4*>(m + e0) = make_float4(mv[0], mv[1], mv[2], mv[3]);
      *reinterpret_cast<float4*>(v + e0) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (e0 + j < n) { p[e0 + j] = pv[j]; m[e0 + j] = mv[j]; v[e0 + j] = vv[j]; }
    }
  }
}

constexpr int kAdamSmemEntries = 512;
// adam_prepare for an optimizer that owns its step counter: t += 1, then the bias corrections of update t
__global__ void adam_prepare_inc(int64_t* __restrict__ step_dev, float lr, float b1, float b2, float* __restrict__ coef) {
  const int64_t ti = *step_dev + 1;
  *step_dev = ti;
  const double t = (double)ti;
  coef[0] = lr / (float)(1.0 - pow((double)b1, t));
  coef[1] = (float)sqrt(1.0 - pow((double)b2, t));
}

// adam_multi_kernel's table search for the data-parallel kernels below: the entry whose [first_block, next first_block) range
// holds block blk = block_lo + blockIdx.x.  Every thread of the block must call it (it synchronises the block).
// adam_multi_kernel keeps its own inline copy: through this function its SASS comes out different (same registers).
__device__ __forceinline__ int adam_table_find(const lbbnn_adam_entry* __restrict__ table, int n_entries, int64_t block_lo,
                                               int64_t* s_first, int64_t& blk) {
  const int ns = n_entries < kAdamSmemEntries ? n_entries : kAdamSmemEntries;
  for (int i = threadIdx.x; i < ns; i += blockDim.x) s_first[i] = table[i].first_block;
  __syncthreads();
  int lo = 0, hi = n_entries - 1;
  blk = block_lo + blockIdx.x;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    const int64_t fb = mid < ns ? s_first[mid] : table[mid].first_block;
    if (fb <= blk) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// The same update over a TABLE of tensors in one launch: block b works on 1024 consecutive elements of the tensor whose
// [first_block, next first_block) range holds b (binary search over the table, read through L2 by every block).
__global__ void __launch_bounds__(256) adam_multi_kernel(const lbbnn_adam_entry* __restrict__ table, int n_entries, float b1,
                                                         float b2, float eps, const float* __restrict__ coef) {
  // the table's block ranges go through shared memory first: ONE L2 round trip for all of them, then the search -- eight
  // dependent global loads per block (~4 us before the first useful load was issued) were half of this launch's 26 us
  __shared__ int64_t s_first[kAdamSmemEntries];
  const int ns = n_entries < kAdamSmemEntries ? n_entries : kAdamSmemEntries;
  for (int i = threadIdx.x; i < ns; i += blockDim.x) s_first[i] = table[i].first_block;
  __syncthreads();
  int lo = 0, hi = n_entries - 1;
  const int64_t blk = blockIdx.x;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    const int64_t fb = mid < ns ? s_first[mid] : table[mid].first_block;
    if (fb <= blk) lo = mid; else hi = mid - 1;
  }
  const lbbnn_adam_entry e = table[lo];
  const float step_size = __ldg(coef) * e.lr_scale, bc2_sqrt = __ldg(coef + 1);
  const int64_t e0 = (blk - e.first_block) * 1024 + (int64_t)threadIdx.x * 4;
  if (e0 >= e.n) return;
  float* p = e.param; const float* g = e.grad; float* m = e.exp_avg; float* v = e.exp_avg_sq;
  const bool vec = (e0 + 3 < e.n) && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v);
  float pv[4], gv[4], mv[4], vv[4];
  if (vec) {
    const float4 a = *reinterpret_cast<const float4*>(p + e0), b = *reinterpret_cast<const float4*>(g + e0);
    const float4 c = *reinterpret_cast<const float4*>(m + e0), d = *reinterpret_cast<const float4*>(v + e0);
    pv[0] = a.x; pv[1] = a.y; pv[2] = a.z; pv[3] = a.w; gv[0] = b.x; gv[1] = b.y; gv[2] = b.z; gv[3] = b.w;
    mv[0] = c.x; mv[1] = c.y; mv[2] = c.z; mv[3] = c.w; vv[0] = d.x; vv[1] = d.y; vv[2] = d.z; vv[3] = d.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool ok = e0 + j < e.n;
      pv[j] = ok ? p[e0 + j] : 0.f; gv[j] = ok ? g[e0 + j] : 0.f;
      mv[j] = ok ? m[e0 + j] : 0.f; vv[j] = ok ? v[e0 + j] : 0.f;
    }
  }
  // one reciprocal of the bias correction per thread, MUFU-based division for the update quotient: <= 2 ulp on a term that is
  // scaled by the learning rate (ncu: the IEEE divisions and sqrt chains kept this bandwidth kernel 55 % issue-active)
  const float inv_bc2 = 1.0f / bc2_sqrt;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (e.decay != 0.f) pv[j] *= 1.0f - e.decay;     // torch.optim.AdamW: param.mul_(1 - lr * weight_decay) first
    mv[j] = mv[j] + (gv[j] - mv[j]) * (1.0f - b1);
    vv[j] = b2 * vv[j] + (1.0f - b2) * gv[j] * gv[j];
    const float denom = fmaf(sqrtf(vv[j]), inv_bc2, eps);
    pv[j] -= step_size * __fdividef(mv[j], denom);
  }
  if (vec) {
    *reinterpret_cast<float4*>(p + e0) = make_float4(pv[0], pv[1], pv[2], pv[3]);
    *reinterpret_cast<float4*>(m + e0) = make_float4(mv[0], mv[1], mv[2], mv[3]);
    *reinterpret_cast<float4*>(v + e0) = make_float4(vv[0], vv[1], vv[2], vv[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < e.n) { p[e0 + j] = pv[j]; m[e0 + j] = mv[j]; v[e0 + j] = vv[j]; }
  }
}

// Data parallel: every entry's parameter lives in one symmetric-memory arena [parameters | packed gradients], its packed
// gradient grad_offset floats after it.  The pack copies autograd's gradient (entry.grad) of this rank's rows there.
__global__ void __launch_bounds__(256) adam_pack_kernel(const lbbnn_adam_entry* __restrict__ table, int n_entries,
                                                        int64_t grad_offset) {
  __shared__ int64_t s_first[kAdamSmemEntries];
  int64_t blk;
  const lbbnn_adam_entry e = table[adam_table_find(table, n_entries, 0, s_first, blk)];
  const int64_t e0 = (blk - e.first_block) * 1024 + (int64_t)threadIdx.x * 4;
  if (e0 >= e.n) return;
  const float* g = e.grad;
  float* d = e.param + grad_offset;
  if (e0 + 3 < e.n && aligned16(g) && aligned16(d)) {
    *reinterpret_cast<float4*>(d + e0) = *reinterpret_cast<const float4*>(g + e0);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (e0 + j < e.n) d[e0 + j] = g[e0 + j];
  }
}

// The sharded update: this rank runs table blocks [block_lo, block_lo + gridDim.x) only.  Per quad: the in-switch sum of the
// packed gradient over all ranks (multimem.ld_reduce: the reduce-scatter), the Adam step of adam_multi_kernel on this rank's
// moments, and the new parameter stored to every rank's copy (multimem.st: the all-gather).  Whole quads: the arena pads each
// tensor to 4 floats with zeros, a zero gradient keeps a zero moment and a zero parameter, so the pads stay zero.
__global__ void __launch_bounds__(256) adam_multi_dp_kernel(const lbbnn_adam_entry* __restrict__ table, int n_entries,
                                                            int64_t block_lo, const float* __restrict__ arena, float* arena_mc,
                                                            int64_t grad_offset, float b1, float b2, float eps,
                                                            const float* __restrict__ coef) {
  __shared__ int64_t s_first[kAdamSmemEntries];
  int64_t blk;
  const lbbnn_adam_entry e = table[adam_table_find(table, n_entries, block_lo, s_first, blk)];
  const float step_size = __ldg(coef) * e.lr_scale, bc2_sqrt = __ldg(coef + 1);
  const int64_t e0 = (blk - e.first_block) * 1024 + (int64_t)threadIdx.x * 4;
  if (e0 >= e.n) return;
  const int64_t off = (e.param - arena) + e0;              // float offset of this quad in the arena (a multiple of 4)
  const float4 gq = mc_ld_reduce4(arena_mc + off + grad_offset);
  const float4 a = *reinterpret_cast<const float4*>(e.param + e0);
  const float4 c = *reinterpret_cast<const float4*>(e.exp_avg + e0), d = *reinterpret_cast<const float4*>(e.exp_avg_sq + e0);
  float pv[4] = {a.x, a.y, a.z, a.w}, gv[4] = {gq.x, gq.y, gq.z, gq.w};
  float mv[4] = {c.x, c.y, c.z, c.w}, vv[4] = {d.x, d.y, d.z, d.w};
  const float inv_bc2 = 1.0f / bc2_sqrt;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (e.decay != 0.f) pv[j] *= 1.0f - e.decay;     // torch.optim.AdamW: param.mul_(1 - lr * weight_decay) first
    mv[j] = mv[j] + (gv[j] - mv[j]) * (1.0f - b1);
    vv[j] = b2 * vv[j] + (1.0f - b2) * gv[j] * gv[j];
    const float denom = fmaf(sqrtf(vv[j]), inv_bc2, eps);
    pv[j] -= step_size * __fdividef(mv[j], denom);
  }
  *reinterpret_cast<float4*>(e.exp_avg + e0) = make_float4(mv[0], mv[1], mv[2], mv[3]);
  *reinterpret_cast<float4*>(e.exp_avg_sq + e0) = make_float4(vv[0], vv[1], vv[2], vv[3]);
  mc_st4(arena_mc + off, pv);
}

__global__ void counter_inc_kernel(int64_t* c) { *c += 1; }

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" const char* lbbnn_last_error(void) { return g_err; }
extern "C" int lbbnn_abi_version(void) { return LBBNN_ABI_VERSION; }

extern "C" int lbbnn_device_ok(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return major == 10;
}

extern "C" int lbbnn_philox_normal(float* out, int64_t n, uint64_t seed, uint64_t stream_id, lbbnn_stream s) {
  return philox_export(out, n, seed, stream_id, 1, s);
}
extern "C" int lbbnn_philox_uniform(float* out, int64_t n, uint64_t seed, uint64_t stream_id, lbbnn_stream s) {
  return philox_export(out, n, seed, stream_id, 0, s);
}

namespace lbbnn {
namespace {
// N(0,1) draws of a full noise descriptor (its device step counter resolved in the kernel: fresh values on every replay of a
// captured graph), element i = what a fused kernel drawing from the same descriptor sees at index i
__global__ void __launch_bounds__(256) philox_noise_kernel(Noise nz, int64_t n, float* __restrict__ out) {
  nz.resolve();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = nz.ptr ? nz.ptr[i] : philox_normal1(nz.seed, nz.stream, (uint64_t)i);
}
}  // namespace
}  // namespace lbbnn

extern "C" int lbbnn_philox_normal_ex(float* out, int64_t n, const lbbnn_noise* noise, lbbnn_stream s) {
  LBBNN_REQUIRE(out && noise && n >= 0, "bad argument");
  if (n == 0) return LBBNN_OK;
  int64_t blocks = ceil_div(n, 256);
  if (blocks > 16LL * sm_count()) blocks = 16LL * sm_count();
  philox_noise_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(make_noise(noise), n, out);
  return check_launch("philox_noise");
}

extern "C" int lbbnn_nll_kl_objective_f32(const float* logits, const int64_t* target, int64_t B, int64_t C,
                                          const float* const* kl_terms, const float* term_scales, int n_kl, float kl_scale,
                                          float* out2, float* dlogits, lbbnn_stream s) {
  LBBNN_REQUIRE(logits && target && out2 && B > 0 && C > 0, "bad logits/target/output");
  LBBNN_REQUIRE(B <= 4096, "one-block objective: batch <= 4096 (got %lld)", (long long)B);
  LBBNN_REQUIRE(n_kl >= 0 && n_kl <= kMaxKlTerms && (n_kl == 0 || kl_terms), "0 <= n_kl <= %d", kMaxKlTerms);
  ObjectiveArgs a;
  a.logits = logits; a.target = target; a.B = B; a.C = C; a.n_kl = n_kl; a.out = out2; a.dlogits = dlogits;
  for (int i = 0; i < kMaxKlTerms; ++i) {
    a.kl[i] = i < n_kl ? kl_terms[i] : nullptr;
    a.scale[i] = i < n_kl ? kl_scale * (term_scales ? term_scales[i] : 1.0f) : 0.f;
  }
  for (int i = 0; i < n_kl; ++i) LBBNN_REQUIRE(a.kl[i], "NULL kl term %d", i);
  const int threads = B >= 32 ? 1024 : (int)(32 * B);
  objective_kernel<<<1, threads, 0, (cudaStream_t)s>>>(a);
  return check_launch("nll_kl_objective");
}

extern "C" int lbbnn_logsoftmax_nll_f32(const float* logits, const int64_t* target, int64_t B, int64_t C, float* logp,
                                        float* nll_sum, float* dlogits, float grad_scale, int64_t* step_inc,
                                        void* ws, size_t ws_bytes, lbbnn_stream s) {
  LBBNN_REQUIRE(logits && target && B > 0 && C > 0, "bad logits/target");
  if (B <= 512) {   // one block: no scratch needed
    logsoftmax_nll_kernel<<<1, 1024, 0, (cudaStream_t)s>>>(logits, target, B, C, logp, nll_sum, dlogits, grad_scale,
                                                           step_inc);
    return check_launch("logsoftmax_nll");
  }
  const int64_t blocks = ceil_div(B, 8);
  LBBNN_REQUIRE(ws && ws_bytes >= (size_t)blocks * sizeof(float), "loss workspace too small (need %lld bytes)",
                (long long)(blocks * sizeof(float)));
  logsoftmax_nll_rows<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(logits, target, B, C, logp, (float*)ws, dlogits,
                                                                     grad_scale);
  if (int rc = check_launch("logsoftmax_nll_rows")) return rc;
  nll_final_sum<<<1, 256, 0, (cudaStream_t)s>>>((const float*)ws, (int)blocks, nll_sum, step_inc);
  return check_launch("nll_final_sum");
}

extern "C" int lbbnn_adam_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                              float beta1, float beta2, float eps, const int64_t* step_dev, float* coef_scratch,
                              lbbnn_stream s) {
  LBBNN_REQUIRE(param && grad && exp_avg && exp_avg_sq && step_dev && coef_scratch && n > 0, "NULL argument");
  adam_prepare<<<1, 1, 0, (cudaStream_t)s>>>(step_dev, lr, beta1, beta2, coef_scratch);
  if (int rc = check_launch("adam_prepare")) return rc;
  const int64_t blocks = ceil_div(ceil_div(n, 4), 256);   // one quad per thread: no grid-stride loop
  LBBNN_REQUIRE(blocks < (1LL << 31), "flat buffer too large");
  adam_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(param, grad, exp_avg, exp_avg_sq, n, beta1, beta2, eps,
                                                             coef_scratch, 0.f);
  return check_launch("adam");
}

extern "C" int lbbnn_adamw_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                               float beta1, float beta2, float eps, float weight_decay, const int64_t* step_dev,
                               float* coef_scratch, lbbnn_stream s) {
  LBBNN_REQUIRE(param && grad && exp_avg && exp_avg_sq && step_dev && coef_scratch && n > 0, "NULL argument");
  adam_prepare<<<1, 1, 0, (cudaStream_t)s>>>(step_dev, lr, beta1, beta2, coef_scratch);
  if (int rc = check_launch("adam_prepare")) return rc;
  const int64_t blocks = ceil_div(ceil_div(n, 4), 256);
  LBBNN_REQUIRE(blocks < (1LL << 31), "flat buffer too large");
  adam_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(param, grad, exp_avg, exp_avg_sq, n, beta1, beta2, eps,
                                                             coef_scratch, lr * weight_decay);
  return check_launch("adamw");
}

extern "C" int lbbnn_adam_prepare(const int64_t* step_dev, float lr, float beta1, float beta2, float* coef, lbbnn_stream s) {
  LBBNN_REQUIRE(step_dev && coef, "NULL argument");
  adam_prepare<<<1, 1, 0, (cudaStream_t)s>>>(step_dev, lr, beta1, beta2, coef);
  return check_launch("adam_prepare");
}

extern "C" int lbbnn_adam_multi_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t total_blocks, float lr,
                                    float beta1, float beta2, float eps, const int64_t* step_dev, float* coef_scratch,
                                    lbbnn_stream s) {
  LBBNN_REQUIRE(table_dev && step_dev && coef_scratch && n_entries > 0 && total_blocks > 0 && total_blocks < (1LL << 31),
                "bad argument");
  adam_prepare<<<1, 1, 0, (cudaStream_t)s>>>(step_dev, lr, beta1, beta2, coef_scratch);
  if (int rc = check_launch("adam_prepare")) return rc;
  adam_multi_kernel<<<(unsigned)total_blocks, 256, 0, (cudaStream_t)s>>>(table_dev, n_entries, beta1, beta2, eps, coef_scratch);
  return check_launch("adam_multi");
}

extern "C" int lbbnn_adam_multi_step_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t total_blocks, float lr,
                                         float beta1, float beta2, float eps, int64_t* step_dev, float* coef_scratch,
                                         lbbnn_stream s) {
  LBBNN_REQUIRE(table_dev && step_dev && coef_scratch && n_entries > 0 && total_blocks > 0 && total_blocks < (1LL << 31),
                "bad argument");
  adam_prepare_inc<<<1, 1, 0, (cudaStream_t)s>>>(step_dev, lr, beta1, beta2, coef_scratch);
  if (int rc = check_launch("adam_prepare_inc")) return rc;
  adam_multi_kernel<<<(unsigned)total_blocks, 256, 0, (cudaStream_t)s>>>(table_dev, n_entries, beta1, beta2, eps, coef_scratch);
  return check_launch("adam_multi");
}

extern "C" int lbbnn_counter_inc(int64_t* counter, lbbnn_stream s) {
  LBBNN_REQUIRE(counter, "NULL counter");
  counter_inc_kernel<<<1, 1, 0, (cudaStream_t)s>>>(counter);
  return check_launch("counter_inc");
}

extern "C" int lbbnn_adam_pack_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t total_blocks, int64_t grad_offset,
                                   lbbnn_stream s) {
  LBBNN_REQUIRE(table_dev && n_entries > 0 && total_blocks > 0 && total_blocks < (1LL << 31), "bad argument");
  adam_pack_kernel<<<(unsigned)total_blocks, 256, 0, (cudaStream_t)s>>>(table_dev, n_entries, grad_offset);
  return check_launch("adam_pack");
}

extern "C" int lbbnn_adam_multi_dp_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t block_lo, int64_t block_hi,
                                       const float* arena, float* arena_mc, int64_t grad_offset, float lr, float beta1,
                                       float beta2, float eps, int64_t* step_dev, float* coef_scratch, int advance,
                                       lbbnn_stream s) {
  LBBNN_REQUIRE(table_dev && arena && arena_mc && step_dev && coef_scratch && n_entries > 0 && 0 <= block_lo &&
                block_lo <= block_hi && block_hi < (1LL << 31) && grad_offset % 4 == 0 &&
                (reinterpret_cast<uintptr_t>(arena) & 15u) == 0 && (reinterpret_cast<uintptr_t>(arena_mc) & 15u) == 0,
                "bad argument");
  if (advance) adam_prepare_inc<<<1, 1, 0, (cudaStream_t)s>>>(step_dev, lr, beta1, beta2, coef_scratch);
  else adam_prepare<<<1, 1, 0, (cudaStream_t)s>>>(step_dev, lr, beta1, beta2, coef_scratch);
  if (int rc = check_launch("adam_prepare")) return rc;
  if (block_hi == block_lo) return LBBNN_OK;                 // more ranks than blocks: this one owns nothing
  adam_multi_dp_kernel<<<(unsigned)(block_hi - block_lo), 256, 0, (cudaStream_t)s>>>(table_dev, n_entries, block_lo, arena, arena_mc,
                                                                                     grad_offset, beta1, beta2, eps, coef_scratch);
  return check_launch("adam_multi_dp");
}
