// Variational-dropout layer (variational_dropout.py:55-68, Kingma et al. 2015 with one dropout rate per output neuron) --
// SURVEY.md §8(f) rank 4.  theta is (n, m) = (in, out) row-major, i.e. the "NN" operand layout (the LBBNN layers keep
// (out, in)); alpha is (m,).
//
//   forward   phi = x theta, q = x^2 theta^2, delta = q alpha, act = phi + sqrt(delta) zeta            (VD:63-68)
//   backward  gD = g zeta / (2 sqrt(delta)), gS = gD alpha
//             d theta = x^T g + 2 theta .* (x^2^T gS)      d x = g theta^T + 2 x .* (gS (theta^2)^T)
//             d alpha = sum_b gD q
//
// One fp32 SIMT dual-GEMM kernel serves the three contractions (the reference runs fp32 with TF32 off; batch 100 does not
// fill a 128-row MMA tile): both products of a pair share the staged tiles, the squares are formed while staging.
// Operands are staged for either memory order (contraction index contiguous, or output index contiguous) so no transposed
// copy of x, theta or the gradients ever exists.  Small-M problems split the contraction over gridDim.z; the partial sums
// are added in a fixed order by the epilogue kernel, so results do not depend on the launch geometry of other calls.
// lbbnn_vd_fwd_ex runs the forward over stacked MC samples for the predictive loop (lbbnn.vd.EnsemblePredictor): a native
// noise stream per group of rows, or FLAG_MOMENTS (x theta and x^2 theta^2 without noise, once per test batch).
#include "common.cuh"

#include <algorithm>

namespace lbbnn {
namespace {

constexpr int BM = 32, BN = 64, BK = 16, kThreads = 128;
constexpr int PADM = BM + 4, PADN = BN + 4;      // rows stay 16-byte aligned for the float4 fragment reads

enum { OP_FWD = 0, OP_AXPY = 1 };

struct Epilogue {
  int op;
  // OP_FWD: act = s1 + sqrt(s2 alpha[col]) zeta, ds = zeta / (2 sqrt(delta)), q = s2;
  //         moments: act = s1, ds = delta, q = s2 (no noise)
  const float* alpha;
  Noise noise;
  int64_t rows_per_group;  // native noise: row r of group g = r / rows_per_group draws element (r % rows_per_group) * N + col
  uint64_t group_stride;   //   from stream noise.stream + g * group_stride
  int relu, moments;
  float* act;
  float* ds;
  float* q;
  // OP_AXPY: out = s1 + 2 base .* s2   (base, out indexed like the output)
  const float* base;
  float* out;
  int accumulate;
};

__device__ __forceinline__ void apply_epilogue(const Epilogue& e, int64_t row, int64_t col, int64_t N, float s1, float s2) {
  const int64_t idx = row * N + col;
  if (e.op == OP_FWD) {
    const float delta = s2 * __ldg(e.alpha + col);
    if (e.moments) {
      e.act[idx] = s1;
      if (e.ds) e.ds[idx] = delta;
      if (e.q) e.q[idx] = s2;
      return;
    }
    const float sd = sqrtf(delta);
    float z;
    if (e.noise.ptr) {
      z = __ldg(e.noise.ptr + idx);
    } else {
      const int64_t g = row / e.rows_per_group;
      const uint64_t el = (uint64_t)((row - g * e.rows_per_group) * N + col);
      float n4[4];      // philox_normal1, with the lane picked by selects (a dynamic index puts n4 on the stack here)
      philox_normal4(e.noise.seed, e.noise.stream + (uint64_t)g * e.group_stride, el >> 2, n4);
      const int lane = (int)(el & 3);
      z = lane == 0 ? n4[0] : lane == 1 ? n4[1] : lane == 2 ? n4[2] : n4[3];
    }
    float a = s1 + sd * z;
    if (e.relu) a = fmaxf(a, 0.f);
    e.act[idx] = a;
    if (e.ds) e.ds[idx] = z / (2.0f * sd);
    if (e.q) e.q[idx] = s2;
  } else {
    float v = s1 + 2.0f * __ldg(e.base + idx) * s2;
    if (e.accumulate) v += e.out[idx];
    e.out[idx] = v;
  }
}

struct GemmArgs {
  // C1 = A1 B1, C2 = A2 B2 with A (M x K), B (K x N).  A2 == nullptr: A2 = A1 .* A1; likewise B2.
  const float* A1; const float* A2; const float* B1; const float* B2;
  int64_t M, N, K, lda, ldb;
  int a_kc, b_kc;        // 1: element (r, k) at p[r * ld + k] (contraction index contiguous); 0: p[k * ld + r]
  int k_chunk;           // contraction elements per gridDim.z slice (multiple of BK)
  float* part;           // gridDim.z > 1: partial sums [z][2][M][N]
  Epilogue epi;
};

// Stage one R x BK operand tile into registers.  NV = R * BK / kThreads values per thread.
template <int R>
struct TileRegs { float v[R * BK / kThreads]; };

template <int R>
__device__ __forceinline__ void load_tile(TileRegs<R>& t, const float* __restrict__ p, int64_t ld, int kc, int64_t r0, int64_t k0,
                                          int64_t rows, int64_t kend, bool vec) {
  constexpr int NV = R * BK / kThreads;
  const int tid = threadIdx.x;
  if (vec) {       // whole tile in range, 16-byte aligned rows: one float4 per 4 values
#pragma unroll
    for (int i = 0; i < NV / 4; ++i) {
      const int e = tid + i * kThreads;
      float4 f;
      if (kc) {    // 4 consecutive k of row r
        const int r = e % R, k4 = e / R;
        f = __ldg(reinterpret_cast<const float4*>(p + (r0 + r) * ld + k0 + k4 * 4));
      } else {     // 4 consecutive r of contraction index k
        const int r4 = e % (R / 4), k = e / (R / 4);
        f = __ldg(reinterpret_cast<const float4*>(p + (k0 + k) * ld + r0 + r4 * 4));
      }
      t.v[i * 4 + 0] = f.x; t.v[i * 4 + 1] = f.y; t.v[i * 4 + 2] = f.z; t.v[i * 4 + 3] = f.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = tid + i * kThreads;
      int r, k;
      if (kc) { k = e % BK; r = e / BK; } else { r = e % R; k = e / R; }
      const bool ok = (r0 + r < rows) && (k0 + k < kend);
      t.v[i] = ok ? __ldg(p + (kc ? (r0 + r) * ld + k0 + k : (k0 + k) * ld + r0 + r)) : 0.f;
    }
  }
}

// registers -> shared S[k][r] (and the squares into S2 when the pair's second operand is implicit)
template <int R, int PAD>
__device__ __forceinline__ void store_tile(const TileRegs<R>& t, float (*S)[PAD], int kc, bool vec, bool square) {
  constexpr int NV = R * BK / kThreads;
  const int tid = threadIdx.x;
  if (vec) {
#pragma unroll
    for (int i = 0; i < NV / 4; ++i) {
      const int e = tid + i * kThreads;
      if (kc) {
        const int r = e % R, k4 = e / R;
#pragma unroll
        for (int j = 0; j < 4; ++j) { const float v = t.v[i * 4 + j]; S[k4 * 4 + j][r] = square ? v * v : v; }
      } else {
        const int r4 = e % (R / 4), k = e / (R / 4);
        float4 f = make_float4(t.v[i * 4], t.v[i * 4 + 1], t.v[i * 4 + 2], t.v[i * 4 + 3]);
        if (square) { f.x *= f.x; f.y *= f.y; f.z *= f.z; f.w *= f.w; }
        *reinterpret_cast<float4*>(&S[k][r4 * 4]) = f;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e = tid + i * kThreads;
      int r, k;
      if (kc) { k = e % BK; r = e / BK; } else { r = e % R; k = e / R; }
      const float v = t.v[i];
      S[k][r] = square ? v * v : v;
    }
  }
}

__device__ __forceinline__ bool tile_vec_ok(const float* p, int64_t ld, int kc, int64_t r0, int64_t k0, int R, int64_t rows,
                                            int64_t kend) {
  return (ld % 4 == 0) && aligned16(p) && (r0 + R <= rows) && (k0 + BK <= kend) && ((kc ? k0 : r0) % 4 == 0);
}

__global__ void __launch_bounds__(kThreads, 4) vd_dual_gemm_kernel(const GemmArgs a) {
  __shared__ __align__(16) float As1[BK][PADM], As2[BK][PADM], Bs1[BK][PADN], Bs2[BK][PADN];
  const int tid = threadIdx.x, tx = tid % (BN / 4), ty = tid / (BN / 4);
  const int64_t m0 = (int64_t)blockIdx.y * BM, n0 = (int64_t)blockIdx.x * BN;
  const int64_t kbeg = (int64_t)blockIdx.z * a.k_chunk;
  const int64_t kend = min((int64_t)a.K, kbeg + a.k_chunk);
  Epilogue epi = a.epi;
  epi.noise.resolve();

  float c1[4][4], c2[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) c1[i][j] = c2[i][j] = 0.f;

  TileRegs<BM> ra1, ra2;
  TileRegs<BN> rb1, rb2;
  bool va = false, vb = false;
  auto fetch = [&](int64_t k0) {
    va = tile_vec_ok(a.A1, a.lda, a.a_kc, m0, k0, BM, a.M, kend) && (!a.A2 || aligned16(a.A2));
    vb = tile_vec_ok(a.B1, a.ldb, a.b_kc, n0, k0, BN, a.N, kend) && (!a.B2 || aligned16(a.B2));
    load_tile<BM>(ra1, a.A1, a.lda, a.a_kc, m0, k0, a.M, kend, va);
    if (a.A2) load_tile<BM>(ra2, a.A2, a.lda, a.a_kc, m0, k0, a.M, kend, va);
    load_tile<BN>(rb1, a.B1, a.ldb, a.b_kc, n0, k0, a.N, kend, vb);
    if (a.B2) load_tile<BN>(rb2, a.B2, a.ldb, a.b_kc, n0, k0, a.N, kend, vb);
  };
  auto commit = [&]() {
    store_tile<BM, PADM>(ra1, As1, a.a_kc, va, false);
    if (a.A2) store_tile<BM, PADM>(ra2, As2, a.a_kc, va, false); else store_tile<BM, PADM>(ra1, As2, a.a_kc, va, true);
    store_tile<BN, PADN>(rb1, Bs1, a.b_kc, vb, false);
    if (a.B2) store_tile<BN, PADN>(rb2, Bs2, a.b_kc, vb, false); else store_tile<BN, PADN>(rb1, Bs2, a.b_kc, vb, true);
  };

  if (kbeg < kend) fetch(kbeg);
  for (int64_t k0 = kbeg; k0 < kend; k0 += BK) {
    __syncthreads();             // the previous tile's fragment reads are done
    commit();
    __syncthreads();
    if (k0 + BK < kend) fetch(k0 + BK);      // next tile's global loads fly under this tile's math
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a1 = *reinterpret_cast<const float4*>(&As1[k][ty * 4]);
      const float4 a2 = *reinterpret_cast<const float4*>(&As2[k][ty * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs1[k][tx * 4]);
      const float4 b2 = *reinterpret_cast<const float4*>(&Bs2[k][tx * 4]);
      const float av1[4] = {a1.x, a1.y, a1.z, a1.w}, av2[4] = {a2.x, a2.y, a2.z, a2.w};
      const float bv1[4] = {b1.x, b1.y, b1.z, b1.w}, bv2[4] = {b2.x, b2.y, b2.z, b2.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          c1[i][j] = fmaf(av1[i], bv1[j], c1[i][j]);
          c2[i][j] = fmaf(av2[i], bv2[j], c2[i][j]);
        }
    }
  }

  const int64_t MN = a.M * a.N;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t row = m0 + ty * 4 + i;
    if (row >= a.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t col = n0 + tx * 4 + j;
      if (col >= a.N) continue;
      if (gridDim.z == 1) {
        apply_epilogue(epi, row, col, a.N, c1[i][j], c2[i][j]);
      } else {
        float* p = a.part + (int64_t)blockIdx.z * 2 * MN + row * a.N + col;
        p[0] = c1[i][j];
        p[MN] = c2[i][j];
      }
    }
  }
}

// fixed-order sum of the contraction slices, then the epilogue
__global__ void __launch_bounds__(256) vd_reduce_epilogue_kernel(const float* __restrict__ part, int splits, int64_t M, int64_t N,
                                                                 Epilogue epi) {
  epi.noise.resolve();
  const int64_t MN = M * N;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < MN; i += (int64_t)gridDim.x * blockDim.x) {
    float s1 = 0.f, s2 = 0.f;
    for (int z = 0; z < splits; ++z) {
      s1 += __ldg(part + (int64_t)z * 2 * MN + i);
      s2 += __ldg(part + (int64_t)z * 2 * MN + MN + i);
    }
    apply_epilogue(epi, i / N, i % N, N, s1, s2);
  }
}

// backward staging: gE = g (masked by the relu that followed the layer), gS = gE ds alpha, d alpha = sum_b gE ds q.
// One block owns 32 columns; 8 row groups are summed through shared memory in a fixed order.
__global__ void __launch_bounds__(256) vd_bwd_prep_kernel(const float* __restrict__ g, const float* __restrict__ act,
                                                          const float* __restrict__ ds, const float* __restrict__ q,
                                                          const float* __restrict__ alpha, int64_t B, int64_t m, int relu,
                                                          float* __restrict__ gE, float* __restrict__ gS,
                                                          float* __restrict__ d_alpha, int accumulate) {
  __shared__ float red[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int64_t col = (int64_t)blockIdx.x * 32 + cx;
  float acc = 0.f;
  if (col < m) {
    const float al = __ldg(alpha + col);
    for (int64_t b = ry; b < B; b += 8) {
      const int64_t idx = b * m + col;
      float ge = __ldg(g + idx);
      if (relu && !(__ldg(act + idx) > 0.f)) ge = 0.f;
      const float gd = ge * __ldg(ds + idx);
      gE[idx] = ge;
      gS[idx] = gd * al;
      acc = fmaf(gd, __ldg(q + idx), acc);
    }
  }
  red[ry][cx] = acc;
  __syncthreads();
  if (ry == 0 && col < m && d_alpha) {
    float s = 0.f;
#pragma unroll
    for (int r = 0; r < 8; ++r) s += red[r][cx];
    d_alpha[col] = accumulate ? d_alpha[col] + s : s;
  }
}

// KL term of loss_fn (VD:98-102): sum_j 0.5 log a + c1 a + c2 a^2 + c3 a^3; d_alpha += grad_scale * d/da
__global__ void __launch_bounds__(256) vd_kl_kernel(const float* __restrict__ alpha, int64_t m, float* __restrict__ kl_out,
                                                    int kl_accumulate, float* __restrict__ d_alpha, float grad_scale) {
  __shared__ double red[32];
  constexpr double c1 = 1.16145124, c2 = -1.50204118, c3 = 0.58629921;
  double acc = 0.0;
  for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {      // m values: the terms cancel to ~1e-2 of their size, so fp64
    const double a = (double)alpha[j];
    acc += 0.5 * log(a) + a * (c1 + a * (c2 + a * c3));
    if (d_alpha) d_alpha[j] += grad_scale * (float)(0.5 / a + c1 + a * (2.0 * c2 + 3.0 * c3 * a));
  }
  const double tot = block_sum(acc, red);
  if (threadIdx.x == 0 && kl_out) *kl_out = (kl_accumulate ? *kl_out : 0.f) + (float)tot;
}

int pick_splits(int64_t M, int64_t N, int64_t K) {
  const int64_t tiles = ceil_div(M, BM) * ceil_div(N, BN);
  const int64_t ksteps = ceil_div(K, BK);
  int64_t want = ceil_div(4 * (int64_t)sm_count(), tiles);          // about four CTAs (16 warps) per SM
  want = std::min<int64_t>(want, ksteps / 4);                        // at least 4 k-steps per slice
  return (int)std::max<int64_t>(1, std::min<int64_t>(want, 32));
}

int launch_gemm(GemmArgs a, void* ws, size_t ws_bytes, cudaStream_t st, const char* what) {
  const int splits = pick_splits(a.M, a.N, a.K);
  const int64_t ksteps = ceil_div(a.K, BK);
  a.k_chunk = (int)(ceil_div(ksteps, splits) * BK);
  const int zs = (int)ceil_div(a.K, a.k_chunk);
  if (zs > 1) {
    const size_t need = (size_t)zs * 2 * a.M * a.N * sizeof(float);
    LBBNN_REQUIRE(ws && ws_bytes >= need, "%s: workspace too small (%zu < %zu)", what, ws_bytes, need);
    a.part = static_cast<float*>(ws);
  }
  dim3 grid((unsigned)ceil_div(a.N, BN), (unsigned)ceil_div(a.M, BM), (unsigned)zs);
  vd_dual_gemm_kernel<<<grid, kThreads, 0, st>>>(a);
  if (int rc = check_launch(what)) return rc;
  if (zs > 1) {
    const int64_t MN = a.M * a.N;
    const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(MN, 256), 4 * (int64_t)sm_count());
    vd_reduce_epilogue_kernel<<<blocks, 256, 0, st>>>(a.part, zs, a.M, a.N, a.epi);
    return check_launch("vd_reduce_epilogue");
  }
  return 0;
}

bool on_device(const void* p) {
  if (!p) return true;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

size_t split_bytes(int64_t M, int64_t N, int64_t K) {
  const int splits = pick_splits(M, N, K);
  return splits > 1 ? (size_t)splits * 2 * M * N * sizeof(float) : 0;
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" size_t lbbnn_vd_workspace_bytes(int64_t batch, int64_t n, int64_t m) {
  // [gE | gS] (batch, m) each, then the split-contraction partials of the largest of the three GEMMs
  const size_t g = (size_t)2 * batch * m * sizeof(float);
  const size_t part = std::max(split_bytes(batch, m, n), std::max(split_bytes(n, m, batch), split_bytes(batch, n, m)));
  return ((g + 255) / 256) * 256 + part + 256;
}

// launches of one dual GEMM (M x K)(K x N): 1, or 2 when its contraction is split (GEMM + fixed-order reduce/epilogue)
extern "C" int lbbnn_vd_gemm_launches(int64_t M, int64_t N, int64_t K) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  const int splits = pick_splits(M, N, K);
  const int64_t k_chunk = ceil_div(ceil_div(K, BK), splits) * BK;
  return ceil_div(K, k_chunk) > 1 ? 2 : 1;
}

extern "C" int lbbnn_vd_fwd_ex(const float* theta, const float* alpha, const float* x, int64_t batch, int64_t n, int64_t m,
                               const lbbnn_noise* noise, int flags, float* act, float* ds_factor, float* q,
                               int64_t rows_per_group, uint64_t noise_group_stride, void* workspace, size_t workspace_bytes,
                               lbbnn_stream s) {
  const bool moments = flags & LBBNN_FLAG_MOMENTS;
  LBBNN_REQUIRE(theta && alpha && x && act && (noise || moments), "vd_fwd: null argument");
  LBBNN_REQUIRE(batch > 0 && n > 0 && m > 0, "vd_fwd: empty shape");
  LBBNN_REQUIRE(rows_per_group > 0 && batch % rows_per_group == 0, "vd_fwd: batch %lld is not a multiple of rows_per_group %lld",
                (long long)batch, (long long)rows_per_group);
  LBBNN_REQUIRE(on_device(theta) && on_device(x) && on_device(act), "vd_fwd: host pointer (there is no CPU fallback)");
  GemmArgs a{};
  a.A1 = x; a.B1 = theta;                 // A2 = x^2, B2 = theta^2 formed while staging
  a.M = batch; a.N = m; a.K = n; a.lda = n; a.ldb = m; a.a_kc = 1; a.b_kc = 0;
  a.epi.op = OP_FWD; a.epi.alpha = alpha; a.epi.noise = make_noise(moments ? nullptr : noise);
  a.epi.rows_per_group = rows_per_group; a.epi.group_stride = noise_group_stride;
  a.epi.relu = (flags & LBBNN_FLAG_RELU) ? 1 : 0; a.epi.moments = moments ? 1 : 0;
  a.epi.act = act; a.epi.ds = ds_factor; a.epi.q = q;
  return launch_gemm(a, workspace, workspace_bytes, (cudaStream_t)s, "vd_fwd");
}

extern "C" int lbbnn_vd_fwd(const float* theta, const float* alpha, const float* x, int64_t batch, int64_t n, int64_t m,
                            const lbbnn_noise* noise, int flags, float* act, float* ds_factor, float* q, void* workspace,
                            size_t workspace_bytes, lbbnn_stream s) {
  LBBNN_REQUIRE(noise, "vd_fwd: null argument");
  return lbbnn_vd_fwd_ex(theta, alpha, x, batch, n, m, noise, flags & ~LBBNN_FLAG_MOMENTS, act, ds_factor, q, batch > 0 ? batch : 1,
                         0, workspace, workspace_bytes, s);
}

extern "C" int lbbnn_vd_bwd(const float* theta, const float* alpha, const float* x, const float* act, const float* ds_factor,
                            const float* q, const float* gact, int64_t batch, int64_t n, int64_t m, int flags,
                            float* d_theta, float* d_alpha, float* dx, void* workspace, size_t workspace_bytes,
                            lbbnn_stream s) {
  LBBNN_REQUIRE(theta && alpha && x && ds_factor && q && gact, "vd_bwd: null argument");
  LBBNN_REQUIRE(!(flags & LBBNN_FLAG_RELU) || act, "vd_bwd: FLAG_RELU needs the layer's output");
  LBBNN_REQUIRE(on_device(theta) && on_device(x) && on_device(gact), "vd_bwd: host pointer (there is no CPU fallback)");
  const size_t gbytes = (((size_t)2 * batch * m * sizeof(float) + 255) / 256) * 256;
  LBBNN_REQUIRE(workspace && workspace_bytes >= gbytes, "vd_bwd: workspace too small");
  cudaStream_t st = (cudaStream_t)s;
  float* gE = static_cast<float*>(workspace);
  float* gS = gE + batch * m;
  char* rest = static_cast<char*>(workspace) + gbytes;
  const size_t rest_bytes = workspace_bytes - gbytes;
  const int acc = (flags & LBBNN_FLAG_ACCUMULATE) ? 1 : 0;
  vd_bwd_prep_kernel<<<(unsigned)ceil_div(m, 32), 256, 0, st>>>(gact, act, ds_factor, q, alpha, batch, m,
                                                                 (flags & LBBNN_FLAG_RELU) ? 1 : 0, gE, gS, d_alpha, acc);
  if (int rc = check_launch("vd_bwd_prep")) return rc;
  if (d_theta) {      // (n, m) = x^T gE + 2 theta .* (x^2^T gS): contraction over the batch, both operands output-contiguous
    GemmArgs a{};
    a.A1 = x; a.B1 = gE; a.B2 = gS;
    a.M = n; a.N = m; a.K = batch; a.lda = n; a.ldb = m; a.a_kc = 0; a.b_kc = 0;
    a.epi.op = OP_AXPY; a.epi.base = theta; a.epi.out = d_theta; a.epi.accumulate = acc;
    if (int rc = launch_gemm(a, rest, rest_bytes, st, "vd_bwd_theta")) return rc;
  }
  if (dx) {           // (batch, n) = gE theta^T + 2 x .* (gS (theta^2)^T): contraction over m, both operands k-contiguous
    GemmArgs a{};
    a.A1 = gE; a.A2 = gS; a.B1 = theta;
    a.M = batch; a.N = n; a.K = m; a.lda = m; a.ldb = m; a.a_kc = 1; a.b_kc = 1;
    a.epi.op = OP_AXPY; a.epi.base = x; a.epi.out = dx; a.epi.accumulate = 0;
    if (int rc = launch_gemm(a, rest, rest_bytes, st, "vd_bwd_input")) return rc;
  }
  return 0;
}

extern "C" int lbbnn_vd_kl(const float* alpha, int64_t m, float* kl_out, int kl_accumulate, float* d_alpha, float grad_scale,
                           lbbnn_stream s) {
  LBBNN_REQUIRE(alpha && m > 0, "vd_kl: null argument");
  LBBNN_REQUIRE(on_device(alpha), "vd_kl: host pointer (there is no CPU fallback)");
  vd_kl_kernel<<<1, 256, 0, (cudaStream_t)s>>>(alpha, m, kl_out, kl_accumulate, d_alpha, grad_scale);
  return check_launch("vd_kl");
}
