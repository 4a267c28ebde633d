// fp32-accurate batched linear layer on the 5th-gen tensor cores: 3xTF32 split on tcgen05 / TMEM / TMA (sm_100a).
//
//   out[z][m][n] = act( sum_k A[z][m][k] W[z][n][k] + bias[z][n] )          (F.linear of LBBNN-GP-MF.py:255 per MC sample z)
//
// Every fp32 operand is carried as hi + lo, hi = the value rounded to TF32 (10-bit mantissa, exactly representable) and
// lo = x - hi (exact in fp32; the tensor core keeps its top 10 mantissa bits).  Per contraction step the kernel issues
// THREE kind::tf32 MMAs:  A_hi W_hi into a "main" fp32 accumulator in TMEM, A_hi W_lo + A_lo W_hi into a second, "small"
// one; the epilogue adds the two.  The dropped lo*lo term and the truncation of lo are ~2^-21 relative per product.  The
// tensor core truncates (rounds toward zero) when it adds into the accumulator, a bias that grows with the number of
// accumulations into the LARGE sum -- measured 5.4e-6 of max|out| at K = 784 with all three products in one accumulator;
// keeping the 2^-11-times-smaller cross terms out of it cuts the accumulations into the large sum (and the error) by 3x.
// The parity tests hold the kernel to the same 1e-5 as the CUDA-core path.
//
// Structure = tc_gemm.cu's: persistent, one CTA per SM, warp 0 TMA producer (3-D tile loads, SWIZZLE_128B, four 16 KB
// boxes of 128 rows x 32 fp32 per stage), warp 1 MMA issuer (M128 N128 K8), warps 2..9 epilogue (tcgen05.ld -> bias /
// relu -> fp32 out and, for the next layer, its hi / lo split), TMEM double-buffered.  The batch index z is the third
// tensor-map coordinate; operands may be strided views (row pitch / batch stride), which is how a layer reads the
// (batch, samples x features) output of the layer before it.
#include <cuda.h>

#include <cstdlib>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace lbbnn {
namespace {

using namespace tc;

constexpr int BM = 128, BN = 128, BKE = 32;     // CTA tile; BKE fp32 = 128 B = one swizzle row
constexpr int UMMA_K = 8;                       // kind::tf32: 8 elements (32 B) per instruction
constexpr int kStages = 3;
constexpr int kTileBytes = BM * BKE * 4;        // 16 KB per operand tile
constexpr int kStageBytes = 4 * kTileBytes;     // A_hi, A_lo, W_hi, W_lo
constexpr int kEpiWarps = 8;
constexpr int kThreads = 64 + kEpiWarps * 32;
constexpr int kTmemCols = 512;                  // 2 accumulator stages x (main + small) x 128 columns
constexpr int EW = 16;
constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256;

// kind::tf32 instruction descriptor: D = f32 (1 @4), A = B = tf32 (2 @7, 2 @10), both K-major, N>>3 @17, M>>4 @24
constexpr uint32_t kIdescTf32 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(kIdescTf32), "r"(accumulate)
      : "memory");
}

struct LinEpi {
  const float* bias;         // (Z, N)
  float *out, *out_hi, *out_lo;
  int64_t ldo, os;           // row pitch / batch stride of the outputs, in floats
  int relu;
};

__global__ void __launch_bounds__(kThreads, 1)
tc_linear_tf32x3_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                        const __grid_constant__ CUtensorMap tmWh, const __grid_constant__ CUtensorMap tmWl, const LinEpi epi,
                        int M, int N, int K, int Z) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* tfull_bar = bars + 2 * kStages;
  uint64_t* tempty_bar = bars + 2 * kStages + 2;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (M + BM - 1) / BM, num_n = (N + BN - 1) / BN;
  const int per_z = num_m * num_n;
  const int num_tiles = per_z * Z, num_kb = (K + BKE - 1) / BKE;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmAh); tma_prefetch_desc(&tmAl); tma_prefetch_desc(&tmWh); tma_prefetch_desc(&tmWl);
    for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_holder, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int z = t / per_z, r = t - z * per_z;
        const int m0 = (r % num_m) * BM, n0 = (r / num_m) * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * kStageBytes;
          mbar_expect_tx(&full_bar[stage], kStageBytes);
          tma_load_3d(sa + 0 * kTileBytes, &tmAh, &full_bar[stage], kb * BKE, m0, z);
          tma_load_3d(sa + 1 * kTileBytes, &tmAl, &full_bar[stage], kb * BKE, m0, z);
          tma_load_3d(sa + 2 * kTileBytes, &tmWh, &full_bar[stage], kb * BKE, n0, z);
          tma_load_3d(sa + 3 * kTileBytes, &tmWl, &full_bar[stage], kb * BKE, n0, z);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0; int it = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
        const int as = it & 1;
        mbar_wait(&tempty_bar[as], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + as * 256, dsm = d + 128;   // main / small accumulators
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kStageBytes);
          const uint64_t ah = umma_desc_kmajor_sw128(sa + 0 * kTileBytes), al = umma_desc_kmajor_sw128(sa + 1 * kTileBytes);
          const uint64_t wh = umma_desc_kmajor_sw128(sa + 2 * kTileBytes), wl = umma_desc_kmajor_sw128(sa + 3 * kTileBytes);
#pragma unroll
          for (int k = 0; k < BKE / UMMA_K; ++k) {
            const uint64_t koff = (uint64_t)((k * UMMA_K * 4) >> 4);   // 32 B per step inside the swizzle row
            const uint32_t acc = (kb | k) ? 1u : 0u;
            umma_tf32(dsm, al + koff, wh + koff, acc);
            umma_tf32(dsm, ah + koff, wl + koff, 1u);
            umma_tf32(d, ah + koff, wh + koff, acc);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[as]);
      }
    }
  } else {
    const int q = warp & 3, half = (warp - 2) >> 2;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int as = it & 1;
      const int z = t / per_z, r = t - z * per_z;
      const int m0 = (r % num_m) * BM, n0 = (r / num_m) * BN;
      mbar_wait(&tfull_bar[as], (it >> 1) & 1);
      tc_fence_after();
      const int64_t row = m0 + q * 32 + lane;
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + half * 64;
      const float* bias = epi.bias + (int64_t)z * N;
#pragma unroll 1
      for (int c = 0; c < 64 / EW; ++c) {
        float v[EW], sm[EW];
        tmem_ld16(tbase + c * EW, v);
        tmem_ld16(tbase + 128 + c * EW, sm);
        const int64_t col0 = n0 + half * 64 + c * EW;
        if (row < M && col0 < N) {
          float hi[EW], lo[EW];
#pragma unroll
          for (int j = 0; j < EW; ++j) {
            float o = (v[j] + sm[j]) + (col0 + j < N ? __ldg(bias + col0 + j) : 0.f);
            if (epi.relu) o = fmaxf(o, 0.f);
            v[j] = o;
            tf32_split(o, hi[j], lo[j]);
          }
          const int64_t off = (int64_t)z * epi.os + row * epi.ldo + col0;
          const bool v4 = (col0 + EW - 1 < N) && (epi.ldo % 4 == 0) && (epi.os % 4 == 0);
          if (v4) {
#pragma unroll
            for (int j = 0; j < EW; j += 4) {
              if (epi.out) *reinterpret_cast<float4*>(epi.out + off + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
              if (epi.out_hi) {
                *reinterpret_cast<float4*>(epi.out_hi + off + j) = make_float4(hi[j], hi[j + 1], hi[j + 2], hi[j + 3]);
                *reinterpret_cast<float4*>(epi.out_lo + off + j) = make_float4(lo[j], lo[j + 1], lo[j + 2], lo[j + 3]);
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < EW; ++j)
              if (col0 + j < N) {
                if (epi.out) epi.out[off + j] = v[j];
                if (epi.out_hi) { epi.out_hi[off + j] = hi[j]; epi.out_lo[off + j] = lo[j]; }
              }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---- CTA-pair variant (see tc_gemm.cu: tc_dual_gemm_bf16_pair) ----------------------------------------------------------
// 256 x 128 tiles on a cluster of two CTAs: each CTA stages its 128 rows of A_hi, A_lo and half (64 rows) of the W_hi,
// W_lo tiles -- 48 KB per stage instead of 64 KB for the same three MMAs, four stages -- and the leader issues
// tcgen05.mma.cta_group::2.kind::tf32 (M256 N128 K8).  The 1-CTA kernel was bound by operand delivery (tensor pipe 55 %).
constexpr int kStagesP = 4;
constexpr int kWHalfBytes = (BN / 2) * BKE * 4;                  // 8 KB
constexpr int kStageBytesP = 2 * kTileBytes + 2 * kWHalfBytes;   // 48 KB
constexpr int kSmemBytesP = kStagesP * kStageBytesP + 1024 + 256;
constexpr uint32_t kIdescTf32P = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);

__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(kIdescTf32P), "r"(accumulate)
      : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
tc_linear_tf32x3_pair_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                             const __grid_constant__ CUtensorMap tmWh, const __grid_constant__ CUtensorMap tmWl, const LinEpi epi,
                             int M, int N, int K, int Z) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStagesP * kStageBytesP);
  uint64_t* full_bar = bars;                        // the leader's is the live one
  uint64_t* empty_bar = bars + kStagesP;
  uint64_t* tfull_bar = bars + 2 * kStagesP;
  uint64_t* tempty_bar = bars + 2 * kStagesP + 2;   // the leader's is the live one
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * kStagesP + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int num_m2 = (M + 2 * BM - 1) / (2 * BM), num_n = (N + BN - 1) / BN;
  const int per_z = num_m2 * num_n;
  const int num_tiles = per_z * Z, num_kb = (K + BKE - 1) / BKE;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmAh); tma_prefetch_desc(&tmAl); tma_prefetch_desc(&tmWh); tma_prefetch_desc(&tmWl);
    for (int s = 0; s < kStagesP; ++s) { mbar_init(&full_bar[s], 2); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 2 * kEpiWarps); }
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 1) tmem_alloc_pair(tmem_holder, kTmemCols);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int t = cluster_id; t < num_tiles; t += num_clusters) {
        const int z = t / per_z, r = t - z * per_z;
        const int m0 = (r % num_m2) * 2 * BM + (int)rank * BM, n0h = (r / num_m2) * BN + (int)rank * (BN / 2);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * kStageBytesP;
          const uint32_t lead_full = mapa_u32(&full_bar[stage], 0);
          mbar_expect_tx_cluster(lead_full, kStageBytesP);
          tma_load_3d_pair(sa, &tmAh, lead_full, kb * BKE, m0, z);
          tma_load_3d_pair(sa + kTileBytes, &tmAl, lead_full, kb * BKE, m0, z);
          tma_load_3d_pair(sa + 2 * kTileBytes, &tmWh, lead_full, kb * BKE, n0h, z);
          tma_load_3d_pair(sa + 2 * kTileBytes + kWHalfBytes, &tmWl, lead_full, kb * BKE, n0h, z);
          if (++stage == kStagesP) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0; uint32_t phase = 0; int it = 0;
      for (int t = cluster_id; t < num_tiles; t += num_clusters, ++it) {
        const int as = it & 1;
        mbar_wait(&tempty_bar[as], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + as * 256, dsm = d + 128;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kStageBytesP);
          const uint64_t ah = umma_desc_kmajor_sw128(sa), al = umma_desc_kmajor_sw128(sa + kTileBytes);
          const uint64_t wh = umma_desc_kmajor_sw128(sa + 2 * kTileBytes);
          const uint64_t wl = umma_desc_kmajor_sw128(sa + 2 * kTileBytes + kWHalfBytes);
#pragma unroll
          for (int k = 0; k < BKE / UMMA_K; ++k) {
            const uint64_t koff = (uint64_t)((k * UMMA_K * 4) >> 4);
            const uint32_t acc = (kb | k) ? 1u : 0u;
            umma_tf32_pair(dsm, al + koff, wh + koff, acc);
            umma_tf32_pair(dsm, ah + koff, wl + koff, 1u);
            umma_tf32_pair(d, ah + koff, wh + koff, acc);
          }
          umma_commit_pair(&empty_bar[stage], 3);
          if (++stage == kStagesP) { stage = 0; phase ^= 1; }
        }
        umma_commit_pair(&tfull_bar[as], 3);
      }
    }
  } else {
    const int q = warp & 3, half = (warp - 2) >> 2;
    int it = 0;
    for (int t = cluster_id; t < num_tiles; t += num_clusters, ++it) {
      const int as = it & 1;
      const int z = t / per_z, r = t - z * per_z;
      const int m0 = (r % num_m2) * 2 * BM + (int)rank * BM, n0 = (r / num_m2) * BN;
      mbar_wait(&tfull_bar[as], (it >> 1) & 1);
      tc_fence_after();
      const int64_t row = m0 + q * 32 + lane;
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + half * 64;
      const float* bias = epi.bias + (int64_t)z * N;
#pragma unroll 1
      for (int c = 0; c < 64 / EW; ++c) {
        float v[EW], sm[EW];
        tmem_ld16(tbase + c * EW, v);
        tmem_ld16(tbase + 128 + c * EW, sm);
        const int64_t col0 = n0 + half * 64 + c * EW;
        if (row < M && col0 < N) {
          float hi[EW], lo[EW];
#pragma unroll
          for (int j = 0; j < EW; ++j) {
            float o = (v[j] + sm[j]) + (col0 + j < N ? __ldg(bias + col0 + j) : 0.f);
            if (epi.relu) o = fmaxf(o, 0.f);
            v[j] = o;
            tf32_split(o, hi[j], lo[j]);
          }
          const int64_t off = (int64_t)z * epi.os + row * epi.ldo + col0;
          const bool v4 = (col0 + EW - 1 < N) && (epi.ldo % 4 == 0) && (epi.os % 4 == 0);
          if (v4) {
#pragma unroll
            for (int j = 0; j < EW; j += 4) {
              if (epi.out) *reinterpret_cast<float4*>(epi.out + off + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
              if (epi.out_hi) {
                *reinterpret_cast<float4*>(epi.out_hi + off + j) = make_float4(hi[j], hi[j + 1], hi[j + 2], hi[j + 3]);
                *reinterpret_cast<float4*>(epi.out_lo + off + j) = make_float4(lo[j], lo[j + 1], lo[j + 2], lo[j + 3]);
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < EW; ++j)
              if (col0 + j < N) {
                if (epi.out) epi.out[off + j] = v[j];
                if (epi.out_hi) { epi.out_hi[off + j] = hi[j]; epi.out_lo[off + j] = lo[j]; }
              }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(&tempty_bar[as], 0));
    }
  }
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, kTmemCols);
  }
}

__global__ void __launch_bounds__(256) tf32_split_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ hi,
                                                         float* __restrict__ lo) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float h, l;
    tf32_split(__ldg(x + i), h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode3() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = (EncodeTiledFn)p;
  return fn;
}

// (Z, rows, K) fp32 view: K contiguous, row pitch / batch stride in floats; box = 32 (K) x 128 (rows) x 1, OOB -> zeros
int make_map3(CUtensorMap* map, const float* ptr, int64_t K, int64_t rows, int64_t Z, int64_t row_pitch, int64_t batch_stride,
              int box_rows = BM) {
  EncodeTiledFn enc = get_encode3();
  LBBNN_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  LBBNN_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && row_pitch % 4 == 0 && (Z == 1 || batch_stride % 4 == 0) &&
                    row_pitch >= K && (Z == 1 || batch_stride > 0),
                "TMA operand must be 16B aligned with 16B-multiple pitches (pitch %lld, batch stride %lld)",
                (long long)row_pitch, (long long)batch_stride);
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)Z};
  cuuint64_t strides[2] = {(cuuint64_t)row_pitch * 4, (cuuint64_t)(Z == 1 ? row_pitch * rows : batch_stride) * 4};
  cuuint32_t box[3] = {(cuuint32_t)BKE, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LBBNN_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) K=%lld rows=%lld Z=%lld", (int)r, (long long)K,
                (long long)rows, (long long)Z);
  return LBBNN_OK;
}

}  // namespace
}  // namespace lbbnn

using namespace lbbnn;

extern "C" int lbbnn_tf32_split(const float* x, int64_t n, float* hi, float* lo, lbbnn_stream s) {
  LBBNN_REQUIRE(x && hi && lo && n > 0, "NULL argument");
  int64_t blocks = ceil_div(n, 256);
  if (blocks > 8LL * sm_count()) blocks = 8LL * sm_count();
  tf32_split_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(x, n, hi, lo);
  return check_launch("tf32_split");
}

extern "C" int lbbnn_tc_linear_tf32x3(const float* a_hi, const float* a_lo, int64_t a_row_pitch, int64_t a_batch_stride,
                                      const float* w_hi, const float* w_lo, const float* bias, int64_t batches, int64_t M,
                                      int64_t N, int64_t K, int flags, float* out, float* out_hi, float* out_lo,
                                      int64_t out_row_pitch, int64_t out_batch_stride, lbbnn_stream s) {
  LBBNN_REQUIRE(a_hi && a_lo && w_hi && w_lo && bias && batches > 0 && M > 0 && N > 0 && K > 0, "bad argument");
  LBBNN_REQUIRE(out || out_hi, "no output requested");
  LBBNN_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), "hi / lo outputs come in pairs");
  LBBNN_REQUIRE(M < (1LL << 31) && N < (1LL << 31) && K < (1LL << 31) && batches < 65536, "dims must fit int32");
  LBBNN_REQUIRE(K % 4 == 0, "contraction length must be a multiple of 4 (16-byte TMA pitch), got %lld", (long long)K);
  // the epilogue stores float4 whenever both output pitches are multiples of 4 floats
  LBBNN_REQUIRE(out_row_pitch % 4 != 0 || out_batch_stride % 4 != 0 ||
                    ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(out_hi) |
                      reinterpret_cast<uintptr_t>(out_lo)) & 15) == 0,
                "outputs must be 16-byte aligned when their row pitch (%lld) and batch stride (%lld) are multiples of 4",
                (long long)out_row_pitch, (long long)out_batch_stride);
  CUtensorMap mAh, mAl, mWh, mWl;
  if (int rc = make_map3(&mAh, a_hi, K, M, batches, a_row_pitch, a_batch_stride)) return rc;
  if (int rc = make_map3(&mAl, a_lo, K, M, batches, a_row_pitch, a_batch_stride)) return rc;
  LinEpi e;
  e.bias = bias; e.out = out; e.out_hi = out_hi; e.out_lo = out_lo; e.ldo = out_row_pitch; e.os = out_batch_stride;
  e.relu = (flags & LBBNN_FLAG_RELU) ? 1 : 0;
  // CTA pairs (256-row tiles) when they fill the GPU; LBBNN_TC_PAIR=0 forces the 1-CTA kernel, 2 the pair kernel (tests)
  const char* pe = getenv("LBBNN_TC_PAIR");
  const int pair_mode = pe ? atoi(pe) : 1;
  const int64_t tiles2 = ceil_div(M, 2 * BM) * ceil_div(N, BN) * batches;
  if (pair_mode && M > BM && (pair_mode == 2 || tiles2 >= sm_count() / 2)) {
    if (int rc = make_map3(&mWh, w_hi, K, N, batches, K, N * K, BN / 2)) return rc;
    if (int rc = make_map3(&mWl, w_lo, K, N, batches, K, N * K, BN / 2)) return rc;
    static bool attrp_set = false;
    if (!attrp_set) {
      LBBNN_CUDA(cudaFuncSetAttribute(tc_linear_tf32x3_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytesP));
      attrp_set = true;
    }
    const int clusters = (int)(tiles2 < sm_count() / 2 ? tiles2 : sm_count() / 2);
    tc_linear_tf32x3_pair_kernel<<<2 * clusters, kThreads, kSmemBytesP, (cudaStream_t)s>>>(mAh, mAl, mWh, mWl, e, (int)M, (int)N,
                                                                                          (int)K, (int)batches);
    return check_launch("tc_linear_tf32x3_pair");
  }
  if (int rc = make_map3(&mWh, w_hi, K, N, batches, K, N * K)) return rc;
  if (int rc = make_map3(&mWl, w_lo, K, N, batches, K, N * K)) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    LBBNN_CUDA(cudaFuncSetAttribute(tc_linear_tf32x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  const int64_t tiles = ceil_div(M, BM) * ceil_div(N, BN) * batches;
  const int grid = (int)(tiles < sm_count() ? tiles : sm_count());
  tc_linear_tf32x3_kernel<<<grid, kThreads, kSmemBytes, (cudaStream_t)s>>>(mAh, mAl, mWh, mWl, e, (int)M, (int)N, (int)K,
                                                                          (int)batches);
  return check_launch("tc_linear_tf32x3");
}
