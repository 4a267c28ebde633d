/* liblbbnn -- C-ABI of the B200 (sm_100a) kernels behind the drop-in BayesianLinear layers.
 *
 * The reference (LarsELund/Bayesian-Neural-Nets) has no FFI: its boundary is the Python nn.Module
 * surface of `BayesianLinear` (SURVEY.md §8b).  The entry points below are what that surface binds
 * to in this repo: each one replaces a block of eager ATen calls inside a reference method, cited
 * as file:line (LRT = LBBNN-GP-MF-LRT.py, MNF = LBBNN-GP-MF-MNF.py, MF = LBBNN-GP-MF.py,
 * flows2 = flows2.py).  INTEGRATION.md shows the ctypes binding a maintainer adds on the
 * reference side.
 *
 * Conventions: plain device pointers, int64 sizes, row-major contiguous tensors, fp32 unless a
 * name says bf16; no allocation and no host synchronisation inside any call (the caller passes
 * outputs and workspace; *_workspace_bytes tells how much); every call enqueues on the given
 * cudaStream_t (pass the raw handle; 0 = legacy default stream) and is safe to capture in a CUDA
 * graph.  Return value 0 = ok, negative = error, message from lbbnn_last_error() (thread-local).
 * Host (CPU) pointers are rejected: there is no CPU fallback.
 */
#ifndef LBBNN_H
#define LBBNN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LBBNN_ABI_VERSION 2

enum { LBBNN_OK = 0, LBBNN_ERR_INVALID = -1, LBBNN_ERR_CUDA = -2, LBBNN_ERR_UNSUPPORTED = -3 };

/* variance of the masked weight: sigma^2 alpha^2 as the reference computes it (LRT:171, MNF:196)
 * or the spike-and-slab variance alpha(sigma^2+(1-alpha)mu^2) of BASELINE.json's north_star */
enum { LBBNN_VAR_REFERENCE = 0, LBBNN_VAR_EXACT = 1 };

enum {
  LBBNN_FLAG_SAMPLE = 1,      /* LRT sample branch (LRT:169-175); absent = mean branch (LRT:177-180) */
  LBBNN_FLAG_RELU = 2,        /* fwd: write relu(act) (the F.relu of LRT:208-209 fused in) */
  LBBNN_FLAG_KL = 4,          /* fwd: also reduce the layer's KL (LRT:182-194) into kl_out */
  LBBNN_FLAG_ACCUMULATE = 8,  /* bwd: grads += instead of = */
  LBBNN_FLAG_MASK_DX = 16,    /* bwd: dx *= (x > 0), i.e. back through the relu that produced x */
  LBBNN_FLAG_MOMENTS = 32     /* fwd_ex: no noise; act <- e_b, ds_factor <- var_b (LRT:172-173) */
};

typedef void* lbbnn_stream; /* cudaStream_t */

#if defined(__GNUC__)
#define LBBNN_API __attribute__((visibility("default")))
#else
#define LBBNN_API
#endif

/* fixed priors of the LRT/MNF layers (LRT:141-158; MNFsim:157-174 for the sim-study values) */
typedef struct lbbnn_priors {
  float mu, sigma, alpha, bias_mu, bias_sigma;
} lbbnn_priors;

/* variational parameters of one layer, the nn.Parameters of BayesianLinear (LRT:137-151):
 * weight_mu, weight_rho, lambdal are (out,in); bias_mu, bias_rho are (out,).  z is MNF's
 * multiplicative noise vector (in,) or NULL (MNF:197: mm(x*z, M^T) == mm(x, (M*z)^T)). */
typedef struct lbbnn_layer {
  const float* weight_mu;
  const float* weight_rho;
  const float* lambdal;
  const float* bias_mu;
  const float* bias_rho;
  const float* z;
  int64_t in_features, out_features;
  const float* z_kl; /* MNF: the z of the KL branch (MNF:210,230-233), a different draw than `z`; NULL = use z */
} lbbnn_layer;

typedef struct lbbnn_layer_grads {
  float* weight_mu;
  float* weight_rho;
  float* lambdal;
  float* bias_mu;
  float* bias_rho;
  float* z;    /* (in,) or NULL; accumulated with atomics, caller zeroes it */
  float* z_kl; /* (in,) or NULL; likewise */
} lbbnn_layer_grads;

/* Noise source of one call.  eps != NULL: injected tensor, indexed like the output it perturbs
 * (the parity tests feed the oracle's noise through this).  eps == NULL: native Philox4x32-10 with
 * key `seed` and stream  stream_id + (step_dev ? *step_dev * step_stride : 0); step_dev is a device
 * int64 so that a captured CUDA graph draws fresh noise on every replay. */
typedef struct lbbnn_noise {
  const float* eps;
  uint64_t seed;
  uint64_t stream_id;
  const int64_t* step_dev;
  uint64_t step_stride;
} lbbnn_noise;

LBBNN_API const char* lbbnn_last_error(void);
LBBNN_API int lbbnn_abi_version(void);
/* 1 if the current device is compute capability 10.x */
LBBNN_API int lbbnn_device_ok(void);

/* ---- noise --------------------------------------------------------------------------------
 * Native noise is Philox4x32-10 keyed by (seed, stream_id, element); these two calls materialise
 * exactly the values the fused kernels draw, so the CPU oracle can consume identical noise
 * (replaces torch.randn LRT:174 / torch.bernoulli's uniform, flows2:209). */
LBBNN_API int lbbnn_philox_normal(float* out, int64_t n, uint64_t seed, uint64_t stream_id, lbbnn_stream s);
LBBNN_API int lbbnn_philox_uniform(float* out, int64_t n, uint64_t seed, uint64_t stream_id, lbbnn_stream s);
/* the same for a full noise descriptor (step_dev honoured: a captured graph draws fresh values on every replay) */
LBBNN_API int lbbnn_philox_normal_ex(float* out, int64_t n, const lbbnn_noise* noise, lbbnn_stream s);

/* ---- LRT layer, fp32 SIMT path (parity mode) ---------------------------------------------------
 * fwd replaces BayesianLinear.forward LRT:166-196: an elementwise prologue (alpha, sigma, M, V, KL
 * terms), the two mm's as one split-K dual GEMM, and an epilogue (biases, eps, sqrt/FMA, optional
 * relu, KL total).  noise: see lbbnn_noise (shape (batch,out)).
 * Outputs: act (batch,out); ds_factor (batch,out) = eps/(2 sqrt(var_b)) = d act/d var_b, kept for the
 * backward (may be NULL when no backward follows); kl_out: one float (FLAG_KL); mv_cache (optional,
 * lbbnn_lrt_f32_mv_bytes) receives M,V so that bwd_input of the same step need not recompute them.
 * bwd_params / bwd_input replace autograd through the same lines (formulas: SURVEY.md §3.5).
 *   gact   = dL/d(act before relu) (batch,out)
 *   kl_grad_dev (device float or NULL) * kl_grad_host = dL/d(kl)
 * One workspace of lbbnn_lrt_f32_workspace_bytes serves all three calls (stream-ordered reuse).
 */
LBBNN_API size_t lbbnn_lrt_f32_workspace_bytes(int64_t batch, int64_t in_features, int64_t out_features);
LBBNN_API size_t lbbnn_lrt_f32_mv_bytes(int64_t in_features, int64_t out_features);

LBBNN_API int lbbnn_lrt_f32_fwd(const lbbnn_layer* layer, const float* x, int64_t batch,
                                const lbbnn_noise* noise, const lbbnn_priors* priors, int var_mode, int flags,
                                float* act, float* ds_factor, float* kl_out, float* mv_cache,
                                void* workspace, size_t workspace_bytes, lbbnn_stream s);

/* The same forward for the batched posterior-predictive loop (test_ensemble, LRT:239-265 / MNF:287-318), where `batch`
 * stacks rows_per_group input rows for each of several MC samples:
 *   rowscale (groups, in) or NULL: rows of group g enter the MEAN product as x .* rowscale[g] (MNF's z of that sample,
 *     MNF:197; the variance product keeps x^2, MNF:198) -- layer->z must then be NULL;
 *   noise_group_stride != 0: native noise per group -- rows of group g draw from stream_id + g * noise_group_stride with
 *     element index (row - g * rows_per_group) * out + col, i.e. what a rows_per_group-row call on that stream draws;
 *   FLAG_MOMENTS: no noise at all; act <- e_b (LRT:172), ds_factor <- var_b (LRT:173): what layer 1 computes ONCE per
 *     test batch when all samples share the input (LRT:247), expanded per sample by lbbnn_lrt_sample_expand. */
LBBNN_API int lbbnn_lrt_f32_fwd_ex(const lbbnn_layer* layer, const float* x, int64_t batch, const lbbnn_noise* noise,
                                   const lbbnn_priors* priors, int var_mode, int flags, float* act, float* ds_factor,
                                   float* kl_out, float* mv_cache, const float* rowscale, int64_t rows_per_group,
                                   uint64_t noise_group_stride, void* workspace, size_t workspace_bytes, lbbnn_stream s);

/* act (n_samples, batch, out) = [relu](e_b + sqrt(var_b) eps_s): the per-sample part of layer 1 of that loop; eps_s is
 * injected ((n_samples, batch, out) in noise->eps) or drawn from stream_id + s * noise_group_stride (FLAG_RELU honoured). */
LBBNN_API int lbbnn_lrt_sample_expand(const float* e_b, const float* var_b, int64_t batch, int64_t out_features,
                                      int n_samples, const lbbnn_noise* noise, uint64_t noise_group_stride, int flags,
                                      float* act, lbbnn_stream s);

LBBNN_API int lbbnn_lrt_f32_bwd_params(const lbbnn_layer* layer, const float* x, int64_t batch,
                                       const float* gact, const float* ds_factor,
                                       const lbbnn_priors* priors, int var_mode, int flags,
                                       const float* kl_grad_dev, float kl_grad_host,
                                       const lbbnn_layer_grads* grads,
                                       void* workspace, size_t workspace_bytes, lbbnn_stream s);

LBBNN_API int lbbnn_lrt_f32_bwd_input(const lbbnn_layer* layer, const float* x, int64_t batch,
                                      const float* gact, const float* ds_factor,
                                      const lbbnn_priors* priors, int var_mode, int flags,
                                      const float* mv_cache, float* dx,
                                      void* workspace, size_t workspace_bytes, lbbnn_stream s);

/* The elementwise halves of the LRT layer on their own (the tensor-core path composes them with the
 * bf16 GEMMs below).  prologue: M = alpha mu [z], V (LRT:170-171) as fp32 (out,in) + the layer KL
 * (LRT:182-194) into kl_out (NULL = skip).  finalize: chain rule from (dM, dV, colsum = [sum_b dE;
 * sum_b dS]) to the parameter gradients + closed-form KL gradient (SURVEY.md §3.5). */
LBBNN_API int lbbnn_lrt_f32_prologue(const lbbnn_layer* layer, const lbbnn_priors* priors, int var_mode, int flags,
                                     float* M, float* V, float* kl_out,
                                     void* workspace, size_t workspace_bytes, lbbnn_stream s);
LBBNN_API int lbbnn_lrt_f32_finalize(const lbbnn_layer* layer, const float* dM, const float* dV, const float* colsum,
                                     const lbbnn_priors* priors, int var_mode, int flags,
                                     const float* kl_grad_dev, float kl_grad_host,
                                     const lbbnn_layer_grads* grads, lbbnn_stream s);

/* ---- bf16 tensor-core path (tcgen05 / TMEM / TMA) ----------------------------------------------
 * One persistent warp-specialised kernel computes D1 = A1 B1^T and D2 = A2 B2^T (all operands K-major
 * bf16, fp32 accumulation in TMEM) and applies a fused epilogue.  Operands must be 16-byte aligned
 * with K % 8 == 0 (TMA pitch); ragged M/N/K tiles are zero-filled by TMA and masked in the epilogue.
 *   raw        D1, D2 as fp32 (M,N): the dW GEMM pair (dM = dE^T x, dV = dS^T x^2) and tests
 *   lrt_fwd    act = D1 + b_mu + sqrt(D2 + sigma_b^2) eps (LRT:172-175) [relu]; writes act and act^2
 *              in bf16 (batch,out), optionally their transposes (out,batch) for the next dW GEMM, the
 *              fp32 ds_factor and an fp32 copy of act.  bf16(act^2) is rounded from the fp32 act.
 *   lrt_bwd_input  dx = dE M + 2 x (dS V) [relu mask] = previous layer's dE; dS_prev = dE_prev *
 *              ds_factor_prev; both in bf16 (batch,in) and optionally transposed (in,batch). */
enum { LBBNN_TC_EPI_RAW = 0, LBBNN_TC_EPI_FWD = 1, LBBNN_TC_EPI_DX = 2, LBBNN_TC_EPI_DW_ADAM = 3 };
enum { LBBNN_PACK_PAIR = 0, LBBNN_PACK_SQUARE = 1, LBBNN_PACK_SCALE = 2 };

LBBNN_API int lbbnn_tc_dual_gemm_raw(const void* A1, const void* A2, const void* B1, const void* B2,
                                     int64_t M, int64_t N, int64_t K, float* D1, float* D2, lbbnn_stream s);
LBBNN_API int lbbnn_tc_lrt_fwd(const void* x_bf, const void* x2_bf, const void* M_bf, const void* V_bf,
                               int64_t batch, int64_t in_features, int64_t out_features,
                               const float* bias_mu, const float* bias_rho, const lbbnn_noise* noise, int flags,
                               void* act_bf, void* act2_bf, void* actT_bf, void* act2T_bf,
                               float* ds_factor, float* act_f32, lbbnn_stream s);
LBBNN_API int lbbnn_tc_lrt_bwd_input(const void* dE_bf, const void* dS_bf, const void* MT_bf, const void* VT_bf,
                                     int64_t batch, int64_t in_features, int64_t out_features,
                                     const void* x_bf, const float* ds_factor_prev, int flags,
                                     void* dE_prev_bf, void* dS_prev_bf, void* dE_prevT_bf, void* dS_prevT_bf,
                                     lbbnn_stream s);
/* fp32 (rows,cols) -> bf16 operand pairs, optionally also transposed (cols,rows):
 *   PAIR: (a, b)   SQUARE: (a, a*a)   SCALE: (a, a*b).   outT/out2T may be NULL. */
LBBNN_API int lbbnn_bf16_pack(const float* a, const float* b, int op, int64_t rows, int64_t cols,
                              void* out1, void* out2, void* out1T, void* out2T, lbbnn_stream s);
/* column sums over the batch: out[0..cols) = sum_r a, out[cols..2cols) = sum_r a*b (fixed order).
 * a_is_bf16: a and b(=second operand, already the product) are bf16 tensors dE, dS instead. */
/* Prologue of the bf16 path in one pass over mu, rho, lambda: M, V (LRT:170-171) as bf16 (out,in), their (in,out)
 * transposes (may be NULL), optional fp32 copies (M32, V32; NULL = skip) and the layer KL (LRT:182-194) into kl_out
 * (NULL = skip).  Same values as lbbnn_lrt_f32_prologue followed by lbbnn_bf16_pack(PACK_PAIR), without the fp32 round
 * trip.  in_features % 4 == 0; MNF's z is not supported here. */
LBBNN_API size_t lbbnn_lrt_bf16_prologue_workspace_bytes(int64_t in_features, int64_t out_features);
LBBNN_API int lbbnn_lrt_bf16_prologue(const lbbnn_layer* layer, const lbbnn_priors* priors, int var_mode, void* M_bf,
                                      void* V_bf, void* MT_bf, void* VT_bf, float* M32, float* V32, float* kl_out,
                                      void* workspace, size_t workspace_bytes, lbbnn_stream s);
/* The same pass without the closing one-block KL reduction: the per-tile KL partials (lbbnn_lrt_bf16_prologue_kl_parts
 * doubles) stay in `workspace` for a later lbbnn_lrt_kl_finalize(workspace, parts, ...), so that the forward GEMM waiting
 * for M, V does not wait for a scalar it does not read. */
LBBNN_API size_t lbbnn_lrt_bf16_prologue_kl_parts(int64_t in_features, int64_t out_features);
LBBNN_API int lbbnn_lrt_bf16_prologue_parts(const lbbnn_layer* layer, const lbbnn_priors* priors, int var_mode, void* M_bf,
                                            void* V_bf, float* M32, float* V32, void* workspace, size_t workspace_bytes,
                                            lbbnn_stream s);
/* Input gradient of a layer with out_features <= 12 (the classifier head) on the CUDA cores, fused with what
 * lbbnn_tc_lrt_bwd_input's epilogue produces for the layer below: dx = g M + 2 x .* ((g .* ds) V) through the relu that
 * produced x (FLAG_MASK_DX), dE = dx, dS = dx .* ds_prev as bf16 (batch,in) + transposes (in,batch; may be NULL), and
 * colsum = [sum_b dE; sum_b dS] (2*in floats, from the fp32 values; NULL = skip).  x_bf: the bf16 activations the
 * layer's forward GEMM consumed.  M32, V32: fp32 (out,in) from lbbnn_lrt_bf16_prologue. */
LBBNN_API size_t lbbnn_tc_lrt_bwd_input_small_workspace_bytes(int64_t batch, int64_t in_features);
LBBNN_API int lbbnn_tc_lrt_bwd_input_small(const float* gact, const float* ds_factor, const float* M32, const float* V32,
                                           int64_t batch, int64_t in_features, int64_t out_features, const void* x_bf,
                                           const float* ds_prev, int flags, void* dE_bf, void* dS_bf, void* dET_bf,
                                           void* dST_bf, float* colsum, void* workspace, size_t workspace_bytes,
                                           lbbnn_stream s);
/* The same forward and dW GEMM pairs for a layer with out_features <= 12 (the classifier head) on the CUDA cores: every SM
 * streams rows of the large operand against the few rows of the small one held in shared memory (bf16 operands, fp32
 * accumulation, like the tensor-core calls they replace).  fwd_small writes the fp32 activations (logits) and ds_factor;
 * it needs in_features * out_features * 4 B <= 192 KB.  raw_small: D1 (M, N) = A1 (M, K) B1 (N, K)^T, D2 likewise, M <= 12,
 * K % 8 == 0 -- lbbnn_tc_dual_gemm_raw's contract for dM = dE^T x, dV = dS^T x^2 of that layer. */
LBBNN_API int lbbnn_tc_lrt_fwd_small(const void* x_bf, const void* x2_bf, const void* M_bf, const void* V_bf, int64_t batch,
                                     int64_t in_features, int64_t out_features, const float* bias_mu, const float* bias_rho,
                                     const lbbnn_noise* noise, int flags, float* act_f32, float* ds_factor, lbbnn_stream s);
LBBNN_API int lbbnn_tc_dual_gemm_raw_small(const void* A1, const void* A2, const void* B1, const void* B2, int64_t M, int64_t N,
                                           int64_t K, float* D1, float* D2, lbbnn_stream s);
LBBNN_API size_t lbbnn_colsum2_workspace_bytes(int64_t rows, int64_t cols);
LBBNN_API int lbbnn_colsum2(const void* a, const void* b, int a_is_bf16, int64_t rows, int64_t cols,
                            float* out, void* workspace, size_t workspace_bytes, lbbnn_stream s);

/* ---- plain fp32 linear layer on the same SIMT GEMM kernels: out = x W^T + b  (F.linear, MF:255) ------
 * fwd (optional relu), bwd_params: dW = G^T x, db = sum_b G;  bwd_input: dx = G W (optional relu mask). */
LBBNN_API int lbbnn_linear_f32_fwd(const float* x, const float* W, const float* bias, int64_t batch,
                                   int64_t in_features, int64_t out_features, int flags, float* out,
                                   void* workspace, size_t workspace_bytes, lbbnn_stream s);
LBBNN_API int lbbnn_linear_f32_bwd_params(const float* x, const float* gout, int64_t batch, int64_t in_features,
                                          int64_t out_features, float* dW, float* dbias,
                                          void* workspace, size_t workspace_bytes, lbbnn_stream s);
LBBNN_API int lbbnn_linear_f32_bwd_input(const float* x, const float* W, const float* gout, int64_t batch,
                                         int64_t in_features, int64_t out_features, int flags, float* dx,
                                         void* workspace, size_t workspace_bytes, lbbnn_stream s);

/* ---- mean-field (full weight sampling) path, LBBNN-GP-MF.py ---------------------------------------
 * gamma_sample: gamma.rsample() (MF:105-117): exact -> [u < alpha]; else torch's RelaxedBernoulli
 *   reparameterisation at `temperature` (clamped probs / uniforms, clipped sigmoid).  alpha comes from
 *   lambdal (sigmoid) or is given; u: lbbnn_noise (injected uniform or native Philox).
 * sample_fwd: w = gamma (mu + sigma eps) | gamma mu | alpha mu (MF:232-242) + the five element sums the
 *   log-probs of MF:247-251 are built from (see csrc/mf.cu); sums = 5 floats.
 * sample_bwd: (dL/dw, dL/dsums) -> dmu, drho, dlambdal, dgamma (NULL = gamma needs no grad), dpb. */
enum { LBBNN_MF_SAMPLE = 0, LBBNN_MF_MEDIMEAN = 1, LBBNN_MF_JOINTMEAN = 2 };
enum {
  LBBNN_MF_FLAG_LOGPROBS = 1,
  LBBNN_MF_FLAG_LP_ON_WS = 2,       /* sim-study variant: log-probs at the unmasked ws (MFsim:233,237) */
  LBBNN_MF_FLAG_EXACT_GAMMA = 4,    /* gamma.exact       (MF:122-124) */
  LBBNN_MF_FLAG_EXACT_WPRIOR = 8,   /* weight_prior.exact (MF:142-146) */
  LBBNN_MF_FLAG_EXACT_GPRIOR = 16   /* gamma_prior.exact  (MF:163-164) */
};
LBBNN_API size_t lbbnn_mf_workspace_bytes(int64_t n);
LBBNN_API int lbbnn_mf_gamma_sample(const float* lambdal, const float* alpha, int64_t n, const lbbnn_noise* u,
                                    int exact, float temperature, float* gamma, lbbnn_stream s);
LBBNN_API int lbbnn_mf_gamma_sample_bwd(const float* lambdal, const float* alpha, const float* gamma,
                                        const float* dgamma, int64_t n, float temperature, float* dout, lbbnn_stream s);
LBBNN_API int lbbnn_mf_sample_fwd(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                                  const float* alpha_stale, const float* pb, int64_t n, const lbbnn_noise* eps,
                                  int mode, int flags, float* w, float* sums,
                                  void* workspace, size_t workspace_bytes, lbbnn_stream s);
/* Monte-Carlo posterior-predictive loop (test_ensemble, MF:345-436).  sample_predict: one launch per layer
 * draws the hard mask [u < sigmoid(lambdal)] natively (no gamma tensor), w = gamma (mu + sigma eps_w) and
 * bias = b_mu + sigma_b eps_b.  mc_accumulate: per weight sample, sum_logp += log_softmax(logits) and
 * sum_prob += row-normalised expit(log_softmax) (MF:397-406), both fp64 (batch,classes); bumps `counter`
 * (device int64, the sample index that keys the Philox streams of the next replay). */
LBBNN_API int lbbnn_mf_sample_predict(const lbbnn_layer* layer, const lbbnn_noise* gamma_u, const lbbnn_noise* eps_w,
                                      const lbbnn_noise* eps_b, float* w, float* bias, lbbnn_stream s);
LBBNN_API int lbbnn_mc_accumulate(const float* logits, int64_t batch, int64_t classes, double* sum_logp,
                                  double* sum_prob, int64_t* counter, lbbnn_stream s);
/* The same loop batched over weight samples (csrc/mc_predict.cu): n_samples samples per launch, sample s of a launch
 * has the global index *first_sample_dev + s and draws from Philox streams  stream_base + which + index * stream_stride
 * (which = 0: mask uniforms, 1: weight normals, 2: bias normals) -- with stream_base = layer * 4 and stream_stride =
 * 4 * n_layers these are exactly the draws of lbbnn_mf_sample_predict, so results do not depend on the batching.
 *   mc_sample            w (n_samples, out, in), bias (n_samples, out) of one layer
 *   linear_f32_batched   out[s] = x[s] W[s]^T + bias[s] (optional relu); x_stride = floats between the inputs of
 *                        consecutive samples (0: all samples read the same input, the first layer)
 *   mc_accumulate_batched  the two fp64 accumulators over the samples of the launch, in order; counter += n_samples */
LBBNN_API int lbbnn_mc_sample(const lbbnn_layer* layer, int n_samples, const int64_t* first_sample_dev, uint64_t seed,
                              uint64_t stream_base, uint64_t stream_stride, float* w, float* bias, lbbnn_stream s);
LBBNN_API int lbbnn_linear_f32_batched(const float* x, int64_t x_stride, const float* W, const float* bias, int n_samples,
                                       int64_t batch, int64_t in_features, int64_t out_features, int flags, float* out,
                                       lbbnn_stream s);
LBBNN_API int lbbnn_mc_accumulate_batched(const float* logits, int n_samples, int64_t batch, int64_t classes,
                                          double* sum_logp, double* sum_prob, int64_t* counter, lbbnn_stream s);
/* The F.linear of the loop (MF:255) at fp32 accuracy on the tensor cores (csrc/tc_gemm_tf32.cu): every fp32 operand is
 * carried as hi + lo (hi = the value rounded to TF32, lo = the exact remainder) and each contraction step issues
 * hi*hi + hi*lo + lo*hi as three tcgen05 kind::tf32 MMAs into one fp32 TMEM accumulator ("3xTF32").
 *   tf32_split           hi / lo of n floats (the test inputs, once per batch)
 *   mc_prepare           sigma = log1p(exp rho), alpha = sigmoid(lambda), sigma_b of one layer, once per parameter set
 *   mc_sample_split      = mc_sample with optional extras: w_lo != NULL -> the weights leave as w_hi / w_lo (w_hi + w_lo
 *                        is mc_sample's w, bit for bit); prepared != 0 -> the layer's weight_rho / lambdal / bias_rho
 *                        pointers hold mc_prepare's sigma / alpha / sigma_b (same values, not recomputed per sample)
 *   tc_linear_tf32x3     out[z][m][n] = act(sum_k a[z][m][k] w[z][n][k] + bias[z][n]),  z < batches.
 *                        a: row m of batch z starts at a + z * a_batch_stride + m * a_row_pitch (floats, multiples of 4);
 *                        w: (batches, N, K) contiguous; K % 4 == 0; outputs at z * out_batch_stride + m * out_row_pitch:
 *                        `out` (fp32, may be NULL) and/or the pair out_hi / out_lo (the split the next layer consumes).
 *                        All samples of a launch sharing one input (the first layer) = ONE problem with batches = 1 and
 *                        N = n_samples * out_features; its (batch, n_samples * out) output is the next layer's strided a. */
LBBNN_API int lbbnn_tf32_split(const float* x, int64_t n, float* hi, float* lo, lbbnn_stream s);
/* The LRT / MNF posterior-predictive loop (lbbnn.EnsemblePredictor) on the tensor cores (csrc/lrt_predict.cu): the LRT
 * forward of n stacked samples is E = A_E M^T and S = A_S V^T (M, V from lbbnn_lrt_f32_prologue, split by lbbnn_tf32_split),
 * each ONE lbbnn_tc_linear_tf32x3 call of n * batch rows with a zero bias; these two calls sit around them.
 *   lrt_mc_epilogue   act[s] = [relu](E[s] + b_mu + sqrt(S[s] + sigma_b^2) eps_s) for s < n_samples, the expressions of the
 *                     fp32 forward epilogue (LRT:172-175), sigma_b = log1p(exp bias_rho).  E[s] / S[s] (batch, out) start at
 *                     E + s * e_sample_stride (0 = shared by all samples: layer 1 of an LRT network, MNF layer 1's S).  eps_s
 *                     is injected ((n_samples, batch, out) in noise->eps) or drawn from stream_id + s * noise_group_stride
 *                     with element index row * out + col -- the draws of lbbnn_lrt_f32_fwd_ex / lbbnn_lrt_sample_expand.
 *                     Without FLAG_SAMPLE: act = [relu](E + b_mu) (LRT:177-180; S, bias_rho, noise unused).  Outputs, each
 *                     (n_samples, batch, out), NULL = skip: act (fp32); m_hi / m_lo = split of act .* rowscale[s] (rowscale
 *                     (n_samples, out) or NULL: the next MNF layer's z, MNF:197); v_hi / v_lo = split of act^2 (fp32 square).
 *   tf32_split_rows   for s < n_samples: hi / lo of x[s] .* rowscale[s] and sq_hi / sq_lo of x[s]^2, where x[s] (rows, cols)
 *                     starts at x + s * x_sample_stride (0 = one shared input); rowscale (n_samples, cols) or NULL; either
 *                     output pair may be NULL.  Splits are lbbnn_tf32_split's (hi + lo == value, bit for bit). */
LBBNN_API int lbbnn_lrt_mc_epilogue(const float* E, int64_t e_sample_stride, const float* S, int64_t s_sample_stride,
                                    const float* bias_mu, const float* bias_rho, int64_t batch, int64_t out_features,
                                    int n_samples, const lbbnn_noise* noise, uint64_t noise_group_stride, int flags,
                                    float* act, const float* rowscale, float* m_hi, float* m_lo, float* v_hi, float* v_lo,
                                    lbbnn_stream s);
LBBNN_API int lbbnn_tf32_split_rows(const float* x, int64_t x_sample_stride, int64_t rows, int64_t cols, int n_samples,
                                    const float* rowscale, float* hi, float* lo, float* sq_hi, float* sq_lo, lbbnn_stream s);
/* Classifier head + accumulation in one launch: logits[s] = h[s] W[s]^T + bias[s] for the n_samples samples of a launch
 * (h: sample s at h + s * h_stride, (batch, in_features) row-major; W (n_samples, classes, in_features); classes <= 16,
 * in_features % 4 == 0, 16 (classes + 8) in_features <= 220 KB of shared memory), then exactly mc_accumulate_batched on them (same expressions, samples in order).  The logits
 * are never written. */
LBBNN_API int lbbnn_mc_head_accumulate(const float* h, int64_t h_stride, const float* W, const float* bias, int n_samples,
                                       int64_t batch, int64_t in_features, int64_t classes, double* sum_logp,
                                       double* sum_prob, int64_t* counter, lbbnn_stream s);
LBBNN_API int lbbnn_mc_prepare(const lbbnn_layer* layer, float* sigma, float* alpha, float* bias_sigma, lbbnn_stream s);
LBBNN_API int lbbnn_mc_sample_split(const lbbnn_layer* layer, int n_samples, const int64_t* first_sample_dev, uint64_t seed,
                                    uint64_t stream_base, uint64_t stream_stride, int prepared, float* w_hi, float* w_lo,
                                    float* bias, lbbnn_stream s);
LBBNN_API int lbbnn_tc_linear_tf32x3(const float* a_hi, const float* a_lo, int64_t a_row_pitch, int64_t a_batch_stride,
                                     const float* w_hi, const float* w_lo, const float* bias, int64_t batches, int64_t M,
                                     int64_t N, int64_t K, int flags, float* out, float* out_hi, float* out_lo,
                                     int64_t out_row_pitch, int64_t out_batch_stride, lbbnn_stream s);
LBBNN_API int lbbnn_mf_sample_bwd(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                                  const float* pb, int64_t n, const lbbnn_noise* eps, int flags,
                                  const float* dw, const float* dsums,
                                  float* dmu, float* drho, float* dlambdal, float* dgamma, float* dpb,
                                  void* workspace, size_t workspace_bytes, lbbnn_stream s);
/* lbbnn_mf_sample_fwd / _bwd with the closing reductions (the five sums; dpb) done by the LAST block of the launch instead of one
 * / two further launches: `ticket` is a device counter that is zero on entry and is left zero (one per concurrent call site);
 * same summation order, bit-identical results. */
LBBNN_API int lbbnn_mf_sample_fwd_ticket(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                                         const float* alpha_stale, const float* pb, int64_t n, const lbbnn_noise* eps, int mode,
                                         int flags, float* w, float* sums, void* ws, size_t ws_bytes, unsigned int* ticket,
                                         lbbnn_stream s);
LBBNN_API int lbbnn_mf_sample_bwd_ticket(const float* mu, const float* rho, const float* lambdal, const float* gamma,
                                         const float* pb, int64_t n, const lbbnn_noise* eps, int flags, const float* dw,
                                         const float* dsums, float* dmu, float* drho, float* dlambdal, float* dgamma, float* dpb,
                                         void* ws, size_t ws_bytes, unsigned int* ticket, lbbnn_stream s);

/* The scalar tail of the MF layer's log-probabilities (MF:148-150 GaussGamma, MF:167-173 BetaBinomial, MF:246-251) in one
 * launch each way: from the five sums of lbbnn_mf_sample_fwd, the Gamma draws tau_w (1) / tau_b (out) and the hyper-
 * parameters to  bias = bias_mu + sigma_b eps_b  (sample_bias; bias_mu otherwise), logprobs2 = [log_prior, log_q]; see
 * csrc/mf.cu for the expressions (the reference's own, term for term).  eps_out keeps the bias draw for the backward.
 * bwd: d_scalars10 = [d s0..s4, d a, d b, d tau_w, d pa, d pb]; g_bias (out) = gradient arriving at `bias` from the
 * linear layer (NULL = none); every output is written. */
LBBNN_API int lbbnn_mf_prior_fwd(const float* sums5, const float* a, const float* b, const float* tau_w, const float* pa,
                                 const float* pb, const float* bias_a, const float* bias_b, const float* tau_b,
                                 const float* bias_mu, const float* bias_rho, const lbbnn_noise* eps_b, int sample_bias,
                                 int64_t out_features, double n_weights, float* bias, float* eps_out, float* logprobs2,
                                 lbbnn_stream s);
LBBNN_API int lbbnn_mf_prior_bwd(const float* sums5, const float* a, const float* b, const float* tau_w, const float* pa,
                                 const float* pb, const float* bias_a, const float* bias_b, const float* tau_b,
                                 const float* bias_mu, const float* bias_rho, const float* bias, const float* eps,
                                 int sample_bias, int64_t out_features, double n_weights, const float* g_log_prior,
                                 const float* g_log_q, const float* g_bias, float* d_scalars10, float* d_bias_a,
                                 float* d_bias_b, float* d_tau_b, float* d_bias_mu, float* d_bias_rho, lbbnn_stream s);
/* The same with the two Gamma precisions drawn OUTSIDE autograd (tau = g / b, g ~ standard Gamma(a)): dtau_*_da / dtau_*_db are
 * their partial derivatives (standard_gamma_grad(a, g) / b and -g / b^2; (1,) for the weights' precision, (out) for the
 * biases'; NULL pairs = none) and the gradient that reaches each tau is folded into d a, d b here (d tau is still written). */
LBBNN_API int lbbnn_mf_prior_bwd_tau(const float* sums5, const float* a, const float* b, const float* tau_w, const float* pa,
                                     const float* pb, const float* bias_a, const float* bias_b, const float* tau_b,
                                     const float* bias_mu, const float* bias_rho, const float* bias, const float* eps,
                                     int sample_bias, int64_t out_features, double n_weights, const float* g_log_prior,
                                     const float* g_log_q, const float* g_bias, const float* dtau_w_da, const float* dtau_w_db,
                                     const float* dtau_b_da, const float* dtau_b_db, float* d_scalars10, float* d_bias_a,
                                     float* d_bias_b, float* d_tau_b, float* d_bias_mu, float* d_bias_rho, lbbnn_stream s);

/* ---- normalizing flows of flows2.py: PropagateFlow (flows2:14-46) over RNVP (flows2:188-219) or the
 * IAF-style MNF transform (flows2:225-241), as fused small-MLP kernels (one CTA per row of z runs the
 * whole stack; see csrc/flows.cu).  Weights are nn.Linear layout (out,in).
 *   fwd:  z_out (rows,dim), logdet (rows,) [for the IAF kind the reference sums it over rows too, flows2:241:
 *         the caller adds the rows up]; masks: injected {0,1} floats (n_transforms, rows, dim) or NULL for
 *         native [u < 0.5] from Philox(seed, stream_id + transform); save: lbbnn_flow_save_floats floats
 *         kept for the backward (NULL = inference only).
 *   bwd:  dz_in (rows,dim) and the parameter gradients of EACH row into its own slice: every pointer in
 *         lbbnn_flow_grads addresses row 0, row r lives row_stride floats further (sum the rows afterwards). */
#define LBBNN_FLOW_MAX_T 8
#define LBBNN_FLOW_MAX_HIDDEN 6
enum { LBBNN_FLOW_RNVP = 0, LBBNN_FLOW_IAF = 1 };
typedef struct lbbnn_flow_linear { const float* W; const float* b; int in, out; } lbbnn_flow_linear;
typedef struct lbbnn_flow_transform {
  lbbnn_flow_linear hidden[LBBNN_FLOW_MAX_HIDDEN]; /* RNVP: network.{0,2,..}; IAF: f */
  lbbnn_flow_linear shift;                          /* RNVP: t; IAF: g */
  lbbnn_flow_linear scale;                          /* RNVP: s; IAF: k */
} lbbnn_flow_transform;
typedef struct lbbnn_flow {
  int kind, dim, n_transforms, n_hidden;
  lbbnn_flow_transform t[LBBNN_FLOW_MAX_T];
} lbbnn_flow;
typedef struct lbbnn_flow_linear_grad { float* dW; float* db; } lbbnn_flow_linear_grad;
typedef struct lbbnn_flow_transform_grads {
  lbbnn_flow_linear_grad hidden[LBBNN_FLOW_MAX_HIDDEN];
  lbbnn_flow_linear_grad shift, scale;
} lbbnn_flow_transform_grads;
typedef struct lbbnn_flow_grads {
  int64_t row_stride;
  lbbnn_flow_transform_grads t[LBBNN_FLOW_MAX_T];
} lbbnn_flow_grads;
LBBNN_API size_t lbbnn_flow_save_floats(const lbbnn_flow* flow, int64_t rows);
LBBNN_API int lbbnn_flow_fwd(const lbbnn_flow* flow, const float* z_in, int64_t rows, const float* masks,
                             const lbbnn_noise* mask_u, float* z_out, float* logdet, float* save, lbbnn_stream s);
LBBNN_API int lbbnn_flow_bwd(const lbbnn_flow* flow, const lbbnn_flow_grads* grads, int64_t rows, const float* masks,
                             const lbbnn_noise* mask_u, const float* dz_out, const float* dlogdet, const float* save,
                             float* dz_in, lbbnn_stream s);

/* ---- MNF auxiliary KL terms (MNF:208-235 minus the flows and the weight KL; csrc/mnf_aux.cu) -----------------------
 * out3 = [log_q0 - log_rb, log_q0, log_rb] with
 *   log_q0 = sum_i -0.5 log(pi) - 0.5 q0_log_var_i - 0.5 (z0_i - q0_mean_i)^2 / exp(q0_log_var_i)          (MNF:212-214)
 *   a_r    = tanh(M0 (r0_c * z2) + sqrt(V r0_c^2) * eps_r),  M0 = alpha mu, V = sigma^2 alpha^2 (out,in)   (MNF:211,216-219)
 *   log_rb = sum_i -0.5 log(pi) - 0.5 r0_b2_i mean(a_r) - 0.5 (z_b[in-1] - r0_b1_i mean(a_r))^2 / exp(r0_b2_i mean(a_r))
 * z0 = the KL row's pre-flow draw (what the reference leaves in self.z), z2 = its z-flow image, z_b = r_flow(z2).
 * save: lbbnn_mnf_aux_save_floats(out) floats kept for the backward; ticket: one zero-initialised device word per layer.
 * bwd: gout = d loss / d out3[0] (device scalar); every gradient is WRITTEN (not accumulated); dM0, dV are (out,in). */
typedef struct lbbnn_mnf_aux {
  int64_t in_features, out_features;
  const float *q0_mean, *q0_log_var, *z0;
  const float *r0_c, *r0_b1, *r0_b2;
  const float *z2, *M0, *V, *eps_r, *z_b;
} lbbnn_mnf_aux;
typedef struct lbbnn_mnf_aux_grads {
  float *d_q0_mean, *d_q0_log_var, *d_z0, *d_r0_c, *d_r0_b1, *d_r0_b2, *d_z2, *d_z_b;   /* (in,) each */
  float *dM0, *dV;                                                                      /* (out,in) */
} lbbnn_mnf_aux_grads;
LBBNN_API size_t lbbnn_mnf_aux_save_floats(int64_t out_features);
LBBNN_API int lbbnn_mnf_aux_kl_fwd(const lbbnn_mnf_aux* aux, float* out3, float* save, unsigned int* ticket, lbbnn_stream s);
LBBNN_API int lbbnn_mnf_aux_kl_bwd(const lbbnn_mnf_aux* aux, const float* save, const float* gout,
                                   const lbbnn_mnf_aux_grads* grads, lbbnn_stream s);

/* The elementwise glue of one MNF layer call, fused (csrc/mnf_aux.cu):
 *   draw      z0 (rows,in) = q0_mean + sqrt(exp(q0_log_var)) eps (MNF:183-185; eps injected (rows,in) or Philox, kept in eps_out for
 *             the backward) and, when eps_r != NULL, the auxiliary branch's eps_r (out,) (MNF:218) from its own noise source;
 *   draw_bwd  d q0_mean, d q0_log_var from d z0 (rows,in) + the auxiliary term's direct gradients (aux_* may be NULL; aux_d_z0 is
 *             added to row kl_row of d z0: the reference's log_q0 reads self.z = that row, MNF:212-214);
 *   kl_combine  kl = kl_wb + (log_q0 - log_rb) - log_det_q - log_det_r (MNF:235), device scalars;
 *   bwd_rows  dld2 = [0, g_scale * g] (log-det gradients of the activation row / the KL row) when dld2 != NULL, and, when rows2 != NULL,
 *             rows2 (2,in) = [dz_k or 0; a + b]: the z flow's output-gradient rows before the weight KL's share is accumulated. */
LBBNN_API int lbbnn_mnf_draw(const float* q0_mean, const float* q0_log_var, const lbbnn_noise* eps_z, int64_t rows,
                             int64_t in_features, float* eps_out, float* z0, const lbbnn_noise* eps_r_noise,
                             int64_t out_features, float* eps_r, lbbnn_stream s);
LBBNN_API int lbbnn_mnf_draw_bwd(const float* q0_log_var, const float* eps, const float* dz0, int64_t rows, int64_t in_features,
                                 int kl_row, const float* aux_d_q0_mean, const float* aux_d_q0_log_var, const float* aux_d_z0,
                                 float* d_q0_mean, float* d_q0_log_var, lbbnn_stream s);
LBBNN_API int lbbnn_mnf_kl_combine(const float* kl_wb, const float* aux_out, const float* log_det_q, const float* log_det_r,
                                   float* kl_out, lbbnn_stream s);
LBBNN_API int lbbnn_mnf_bwd_rows(const float* g, float g_scale, float* dld2, const float* dz_k, const float* a, const float* b,
                                 int64_t in_features, float* rows2, lbbnn_stream s);

/* ---- whole LRT training step as ONE persistent cooperative kernel (small stacks, batch <= 128) --------
 * Replaces the body of `train` for one minibatch (LRT:217-229): forward of every layer (LRT:166-211),
 * nll_loss(sum) + kl/NUM_BATCHES (LRT:223-224), backward, optim.Adam step (LRT:358); see csrc/lrt_step.cu.
 * Parameters, Adam state and (optionally) gradients are flat fp32 buffers; each layer names its five tensors
 * by float offsets (weight tensors at multiples of 4).  Noise of layer i: injected `eps` (batch,out) or
 * Philox(seed, stream = i + step * n_layers) with step = *step_dev before the call -- the same streams the
 * per-layer entry points draw.  stats = [nll, kl_1 .. kl_L] (KL at the pre-update parameters, like LRT:213).
 * phases: 1 = forward + loss + backward, leaving the raw (dM, dV, bias column sums) of all layers in the first
 *             lbbnn_lrt_step_raw_floats() floats of the workspace (the buffer a data-parallel run all-reduces);
 *         2 = chain rule + KL gradient (scaled by kl_scale = dL/dKL) + Adam on those raw gradients, writes
 *             stats, increments *step_dev;   3 = both in one launch.
 * The workspace must be zero-filled once before its first use and is otherwise opaque. */
#define LBBNN_STEP_MAX_LAYERS 8
typedef struct lbbnn_step_layer {
  int64_t in_features, out_features;
  int64_t off_weight_mu, off_weight_rho, off_lambdal, off_bias_mu, off_bias_rho;
  const float* eps;
  lbbnn_priors priors;
  int var_mode;
} lbbnn_step_layer;
typedef struct lbbnn_step {
  int n_layers;
  int64_t batch;
  lbbnn_step_layer layer[LBBNN_STEP_MAX_LAYERS];
  float* flat;        /* parameters */
  float* exp_avg;     /* Adam state, same layout */
  float* exp_avg_sq;
  float* grad;        /* same layout, or NULL: gradients are consumed in registers and never written */
  const float* x;     /* (batch, in_features of layer 0) */
  const int64_t* y;   /* (batch,) class indices */
  int64_t* step_dev;
  uint64_t seed;
  float lr, beta1, beta2, eps, kl_scale;
  float* stats;       /* 1 + n_layers floats */
  const struct lbbnn_step_dp* dp;   /* NULL, or the data-parallel exchange fused into the launch (phases == 3 only) */
} lbbnn_step;
/* Data-parallel training inside the ONE launch (SURVEY.md §8e; the reference has no multi-GPU path): after the backward
 * phases every rank signals its peers and waits for them (NVLink flags), the update phase then runs SHARDED -- rank r
 * reduces its contiguous 1/world of all weight quads over the ranks in the switch (multimem.ld_reduce on the raw gradients at
 * the head of the workspace), applies chain rule + KL gradient (kl_scale, added once) + Adam with its shard of the moments
 * and stores the new parameters to every rank (multimem.st); rank 0 owns the biases -- and a second flag exchange ends
 * the launch, also carrying every rank's per-layer KL partial so that stats[1..] is the whole KL on every rank (stats[0] stays
 * this rank's nll).  Setup: `flat` and the workspace lie at the same offsets of buffers bound to an NVSwitch multicast object
 * on every rank (flat_mc / ws_mc = their multicast addresses); signal[p] / klx[p] = rank p's signal pad (world uint32) and
 * KL exchange array (world * LBBNN_STEP_MAX_LAYERS doubles) as addressable from THIS rank (peer mappings; [rank] = own),
 * all zero-initialised once; epoch = one zero-initialised local device uint64.  grad must be NULL; every in*out % 4 == 0. */
typedef struct lbbnn_step_dp {
  int world, rank;
  float* flat_mc;
  const float* ws_mc;
  unsigned int* signal[8];
  double* klx[8];
  unsigned long long* epoch;
  /* optional peer-to-peer form of the same exchange (no multicast object needed): flat_peer[p] / ws_peer[p] = rank p's
   * parameter buffer / workspace as addressable from this rank.  When use_p2p != 0 the owner sums its shard of the raw
   * gradients with plain loads from every peer (rank order: deterministic) and writes the new parameters to every peer
   * with plain stores; flat_mc / ws_mc are then ignored. */
  int use_p2p;
  float* flat_peer[8];
  const float* ws_peer[8];
} lbbnn_step_dp;
LBBNN_API size_t lbbnn_lrt_step_workspace_bytes(const lbbnn_step* step);
LBBNN_API size_t lbbnn_lrt_step_raw_floats(const lbbnn_step* step);
LBBNN_API int lbbnn_lrt_step_f32(const lbbnn_step* step, int phases, void* workspace, size_t workspace_bytes,
                                 lbbnn_stream s);
/* Phase profile: while dev_stamps != NULL, CTA 0 of every following lbbnn_lrt_step_f32 launch writes its clock64()
 * at each phase boundary (before/after every grid barrier) and inside its last work item of every phase into dev_stamps
 * (256 int64; layout: see profiles/prof_fused_phases.py).  NULL switches it off. */
LBBNN_API int lbbnn_lrt_step_profile(long long* dev_stamps);
/* human-readable schedule (tile sizes / work items per phase) chosen for this step */
LBBNN_API int lbbnn_lrt_step_describe(const lbbnn_step* step, char* buf, size_t buf_bytes);

/* ---- loss head: F.log_softmax(dim=1) + F.nll_loss(reduction='sum') (LRT:210,223) ------------
 * logp (batch,classes) and dlogits (batch,classes) = grad_scale*(softmax - onehot) may be NULL.
 * step_inc (device int64 or NULL) is incremented by one: the trainer's step counter, bumped between
 * the forward (noise of step t) and the optimizer (bias correction t+1) without an extra launch.
 * batch > 512 runs multi-block and needs a workspace of ceil(batch/8) floats (NULL is fine below that). */
LBBNN_API int lbbnn_logsoftmax_nll_f32(const float* logits, const int64_t* target, int64_t batch, int64_t classes,
                                       float* logp, float* nll_sum, float* dlogits, float grad_scale,
                                       int64_t* step_inc, void* workspace, size_t workspace_bytes, lbbnn_stream s);
/* The whole training objective of one minibatch in ONE launch (LRT:221-224, MNF:267-270; MF:316-318):
 *   nll = F.nll_loss(F.log_softmax(logits, 1), target, reduction='sum')
 *   loss = nll + kl_scale * sum_i term_scales[i] * *kl_terms[i]
 * out2 = [loss, nll]; dlogits (batch,classes; may be NULL) = softmax - onehot = d loss / d logits, and d loss / d term_i is
 * kl_scale * term_scales[i].  kl_terms: HOST array of n_kl (<= 16) device pointers to scalar terms -- the layers' kl, or the
 * MF layers' log q (scale +1) and log prior (scale -1); term_scales: HOST array or NULL (all 1).  batch <= 4096. */
LBBNN_API int lbbnn_nll_kl_objective_f32(const float* logits, const int64_t* target, int64_t batch, int64_t classes,
                                         const float* const* kl_terms, const float* term_scales, int n_kl, float kl_scale,
                                         float* out2, float* dlogits, lbbnn_stream s);

/* ---- optimizer: torch.optim.Adam semantics (LRT:358), one flat buffer ----------------------------
 * step_dev: device int64 holding t, the 1-based index of THIS update; coef_scratch: 2 device floats
 * (the bias-corrected step size is computed once on the device, so a graph replay needs no host input). */
LBBNN_API int lbbnn_adam_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                             float lr, float beta1, float beta2, float eps, const int64_t* step_dev,
                             float* coef_scratch, lbbnn_stream s);
/* Chain rule + KL gradient + Adam in one pass (the wide trainer): lbbnn_lrt_f32_finalize with the three weight
 * gradients and the two bias gradients consumed in registers by torch.optim.Adam's update -- the layer's parameters and
 * their Adam state are updated IN PLACE (the layer struct's pointers are written through) and no gradient is stored.
 * exp_avg / exp_avg_sq: [weight_mu, weight_rho, lambdal, bias_mu, bias_rho]; coef: the 2 floats lbbnn_adam_prepare
 * wrote for this step (step size / bias-correction, computed on the device from *step_dev). */
typedef struct lbbnn_adam_layer_state {
  float* exp_avg[5];
  float* exp_avg_sq[5];
  const float* coef;
  float beta1, beta2, eps;
} lbbnn_adam_layer_state;
LBBNN_API int lbbnn_adam_prepare(const int64_t* step_dev, float lr, float beta1, float beta2, float* coef, lbbnn_stream s);
LBBNN_API int lbbnn_lrt_f32_finalize_adam(const lbbnn_layer* layer, const float* dM, const float* dV, const float* colsum,
                                          const lbbnn_priors* priors, int var_mode, int flags, const float* kl_grad_dev,
                                          float kl_grad_host, const lbbnn_adam_layer_state* adam, lbbnn_stream s);
/* Biases only (sum_b dE, sum_b dS -> d bias_mu, d bias_rho + KL gradient -> Adam): the companion of lbbnn_tc_lrt_dw_adam,
 * whose GEMM epilogue updates the three weight tensors. */
LBBNN_API int lbbnn_lrt_f32_finalize_adam_bias(const lbbnn_layer* layer, const float* colsum, const lbbnn_priors* priors,
                                               int flags, float kl_grad_host, const lbbnn_adam_layer_state* adam,
                                               lbbnn_stream s);

/* ---- data-parallel update over NVSwitch multicast (NVLS) ------------------------------------------------------------------
 * The reference has no multi-GPU path; this is the data-parallel exchange of SURVEY.md §8(e) as ONE kernel per layer instead of
 * an all-reduce of the raw gradients followed by the full update on every rank.  Setup (the binder's job: cuMemCreate /
 * cuMulticastCreate + cuMulticastBindMem, or torch.distributed._symmetric_memory as lbbnn/engine.py does): every rank places
 * the layer's parameters and its raw gradient buffer [dM (out,in) | dV (out,in) | sum_b dE (out) | sum_b dS (out)] at the SAME
 * offsets of a buffer bound to a multicast object spanning all ranks; *_mc are the multicast virtual addresses.
 * finalize_adam_dp, launched by every rank after ALL ranks' dW GEMMs of the layer have completed (cross-rank barrier):
 *   rank r reduces its contiguous 1/world of the (dM, dV) quads over all ranks in the switch (multimem.ld_reduce), applies
 *   chain rule + KL gradient (once) + Adam with ITS shard of the Adam moments, and stores the updated mu, rho, lambda to every
 *   rank's copy (multimem.st); rank 0 does the same for the biases.  A second cross-rank barrier must precede the next read
 *   of the parameters.  `layer` holds this rank's LOCAL addresses (the old values are read from them). */
typedef struct lbbnn_dp_layer {
  int world, rank;
  const float* raw_mc;
  float *weight_mu_mc, *weight_rho_mc, *lambdal_mc, *bias_mu_mc, *bias_rho_mc;
} lbbnn_dp_layer;
LBBNN_API int lbbnn_lrt_f32_finalize_adam_dp(const lbbnn_layer* layer, const lbbnn_dp_layer* dp, const lbbnn_priors* priors,
                                             int var_mode, int flags, float kl_grad_host, const lbbnn_adam_layer_state* adam,
                                             lbbnn_stream s);

/* ---- bf16 tensor-core path, operands read in place (r02) -------------------------------------------------------------
 * The GEMM kernels also take "MN-major" operands: the row-major (K, rows) tensor, i.e. one whose ROW index is the
 * contraction index, fetched by TMA as 64 x 64 boxes into tcgen05's MN-major SWIZZLE_128B layout.  With them the three
 * GEMM pairs of a layer read the same row-major tensors and no transposed copy of x, act, dE, dS, M or V exists:
 *   raw_ex        lbbnn_tc_dual_gemm_raw with a major flag per operand side (a_mn: A1, A2 are (K, M); b_mn: B1, B2 are
 *                 (K, N)); rows % 8 == 0 for an MN-major side (TMA pitch).
 *   bwd_input_mn  lbbnn_tc_lrt_bwd_input reading M_bf, V_bf (out, in) as they are (no M^T, V^T), without transposed
 *                 outputs, and optionally writing the bias-gradient partial sums of the layer below: colsum_part
 *                 [ceil(batch/32)][2*in] (sum over each 32 batch rows of dE | dS, from the fp32 values);
 *                 lbbnn_tc_colsum_reduce sums them in a fixed order into colsum[2*in] -- replaces lbbnn_colsum2 there.
 *   dw_adam       the dW pair dM = dE^T x, dV = dS^T x^2 (contraction over the batch; dE, dS (batch, out) and x, x^2
 *                 (batch, in) read in place) with chain rule + closed-form KL gradient (weight kl_grad = 1/NUM_BATCHES)
 *                 + torch.optim.Adam applied to the accumulators in the epilogue: weight_mu, weight_rho, lambdal and
 *                 their Adam moments are updated IN PLACE, dM / dV never reach memory (LRT:225-226 for the weights of
 *                 one layer).  in/out_features % 8 == 0.  Biases: lbbnn_lrt_f32_finalize_adam_bias. */
LBBNN_API int lbbnn_tc_dual_gemm_raw_ex(const void* A1, const void* A2, const void* B1, const void* B2, int64_t M, int64_t N,
                                        int64_t K, int a_mn, int b_mn, float* D1, float* D2, lbbnn_stream s);
LBBNN_API size_t lbbnn_tc_colsum_part_floats(int64_t batch, int64_t in_features);
LBBNN_API int lbbnn_tc_colsum_reduce(const float* colsum_part, int64_t batch, int64_t in_features, float* colsum,
                                     lbbnn_stream s);
LBBNN_API int lbbnn_tc_lrt_bwd_input_mn(const void* dE_bf, const void* dS_bf, const void* M_bf, const void* V_bf,
                                        int64_t batch, int64_t in_features, int64_t out_features, const void* x_bf,
                                        const float* ds_factor_prev, int flags, void* dE_prev_bf, void* dS_prev_bf,
                                        float* colsum_part, lbbnn_stream s);
LBBNN_API int lbbnn_tc_lrt_dw_adam(const void* dE_bf, const void* dS_bf, const void* x_bf, const void* x2_bf,
                                   const lbbnn_layer* layer, int64_t batch, const lbbnn_priors* priors, int var_mode,
                                   float kl_grad, const lbbnn_adam_layer_state* adam, lbbnn_stream s);
/* dw_adam that also emits what the NEXT step's forward needs from the updated parameters, so that step runs without a
 * prologue pass for this layer: next_M_bf, next_V_bf (out,in) bf16 = lbbnn_lrt_bf16_prologue's M, V of the new mu, rho,
 * lambda, and next_kl_part = lbbnn_tc_lrt_dw_adam_kl_parts() doubles, per-warp partial sums of the weights' KL terms
 * (LRT:189-192); lbbnn_lrt_kl_finalize adds them in a fixed order together with the bias term (LRT:185-186) of the
 * layer's (already updated) biases into kl_out.  The arrays may be NULL (then identical to lbbnn_tc_lrt_dw_adam). */
LBBNN_API size_t lbbnn_tc_lrt_dw_adam_kl_parts(void);
LBBNN_API int lbbnn_tc_lrt_dw_adam_next(const void* dE_bf, const void* dS_bf, const void* x_bf, const void* x2_bf,
                                        const lbbnn_layer* layer, int64_t batch, const lbbnn_priors* priors, int var_mode,
                                        float kl_grad, const lbbnn_adam_layer_state* adam, void* next_M_bf, void* next_V_bf,
                                        double* next_kl_part, lbbnn_stream s);
LBBNN_API int lbbnn_lrt_kl_finalize(const double* kl_part, int64_t n_part, const lbbnn_layer* layer,
                                    const lbbnn_priors* priors, float* kl_out, lbbnn_stream s);

/* The same update for a whole parameter list in ONE launch (optim.Adam(net.parameters()) of the MNF script, MNF:352,
 * and the 33 per-tensor parameter groups of the MF script, MF:520-553: learning rates 1e-4 for weights / biases, 1e-3
 * for pa / pb, 1e-5 for the Gamma hyper-parameters, 0.1 for lambdal): table_dev = device array of n_entries records;
 * block b of the launch updates elements [(b - first_block) * 1024, +1024) of the tensor with the largest
 * first_block <= b, so first_block is the running sum of ceil(n / 1024) and total_blocks its final value.  Each entry's
 * learning rate is lr * lr_scale (its parameter group's lr relative to the call's).  decay = lr_group * weight_decay of the
 * entry's group (computed by the caller: coef holds the bias-corrected step size, not the raw lr): non-zero makes the entry's
 * update torch.optim.AdamW's (variational_dropout.py:110), param *= 1 - decay before the Adam step; 0 is torch.optim.Adam,
 * bit for bit. */
typedef struct lbbnn_adam_entry {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t n;
  int64_t first_block;
  float lr_scale;
  float decay;
} lbbnn_adam_entry;
LBBNN_API int lbbnn_adam_multi_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t total_blocks, float lr,
                                   float beta1, float beta2, float eps, const int64_t* step_dev, float* coef_scratch,
                                   lbbnn_stream s);
/* The same with the optimizer's step counter advanced by the call: *step_dev += 1 first (the 1-based index of this update),
 * then the update -- one launch fewer than lbbnn_counter_inc + lbbnn_adam_multi_f32. */
LBBNN_API int lbbnn_adam_multi_step_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t total_blocks, float lr,
                                        float beta1, float beta2, float eps, int64_t* step_dev, float* coef_scratch,
                                        lbbnn_stream s);
/* Data-parallel form of the table update above, for the training step of LBBNN-GP-MF-MNF.py:263-275,
 * LBBNN-GP-MF.py:325-343 and variational_dropout.py:160-166 with the minibatch sharded over ranks: torch.optim.Adam (entries
 * with decay != 0: torch.optim.AdamW) of the SUM over ranks of the gradients.
 * Every entry's param lies in one symmetric-memory arena [parameters | packed gradients] that is bound to an NVSwitch
 * multicast object (arena_mc is its multicast address), each tensor at a 16-byte aligned offset and padded with zeros to a
 * multiple of 4 floats; its packed gradient sits grad_offset floats (a multiple of 4) after it.
 *   pack:  param[grad_offset + i] = grad[i] for every entry -- this rank's gradients into its region of the arena.
 *   dp:    blocks [block_lo, block_hi) of the table (one rank's share, 1024 elements each; the ranks' shares cover every
 *          block once): in-switch sum over ranks of the packed gradient (multimem.ld_reduce), Adam on this rank's exp_avg /
 *          exp_avg_sq with lr * lr_scale and the entry's decay, the new parameter stored to every rank's arena
 *          (multimem.st).  advance != 0:
 *          *step_dev += 1 first, as lbbnn_adam_multi_step_f32; 0: as lbbnn_adam_multi_f32.
 * The caller orders the dp launch between two cross-rank barriers: every rank packed before, every store landed after. */
LBBNN_API int lbbnn_adam_pack_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t total_blocks, int64_t grad_offset,
                                  lbbnn_stream s);
LBBNN_API int lbbnn_adam_multi_dp_f32(const lbbnn_adam_entry* table_dev, int n_entries, int64_t block_lo, int64_t block_hi,
                                      const float* arena, float* arena_mc, int64_t grad_offset, float lr, float beta1,
                                      float beta2, float eps, int64_t* step_dev, float* coef_scratch, int advance,
                                      lbbnn_stream s);
LBBNN_API int lbbnn_counter_inc(int64_t* counter, lbbnn_stream s);
/* torch.optim.AdamW (variational_dropout.py:110): the update above preceded by param *= 1 - lr * weight_decay */
LBBNN_API int lbbnn_adamw_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                              float lr, float beta1, float beta2, float eps, float weight_decay,
                              const int64_t* step_dev, float* coef_scratch, lbbnn_stream s);

/* ---- variational-dropout layer (VD = variational_dropout.py; SURVEY.md §8f rank 4) -----------------------------
 * BayesianLayer.forward VD:63-68 and autograd through it.  theta is (n, m) = (in, out) row-major -- the "NN" operand
 * layout, unlike the (out, in) weights above -- alpha is (m,), x is (batch, n).
 *   fwd: act = x theta + sqrt((x^2 theta^2) alpha) zeta (FLAG_RELU: relu of it, the F.relu of VD:81-83 fused in);
 *        saved for the backward: ds_factor = zeta / (2 sqrt(delta)) and q = x^2 theta^2, both (batch, m); either may be
 *        NULL when no backward follows.  noise: zeta, shape (batch, m) (see lbbnn_noise).
 *   bwd: gact = dL/d(act) (with FLAG_RELU: dL/d(relu output), masked here by act > 0).  Writes d_theta (n, m)
 *        (FLAG_ACCUMULATE: +=), d_alpha (m,) and dx (batch, n); each may be NULL.
 *   kl:  the layer's term of loss_fn VD:98-102, sum_j 0.5 log a_j + c1 a_j + c2 a_j^2 + c3 a_j^3, written (or added)
 *        to *kl_out; d_alpha (may be NULL) += grad_scale * d kl / d alpha.
 * One workspace of lbbnn_vd_workspace_bytes serves fwd and bwd (stream-ordered reuse). */
LBBNN_API size_t lbbnn_vd_workspace_bytes(int64_t batch, int64_t n, int64_t m);
/* kernel launches of one of the path's dual GEMMs (M x K)(K x N): 2 when its contraction is split, else 1
 * (fwd: (batch, m, n); d_theta: (n, m, batch); dx: (batch, n, m)) -- for launch accounting only */
LBBNN_API int lbbnn_vd_gemm_launches(int64_t M, int64_t N, int64_t K);
LBBNN_API int lbbnn_vd_fwd(const float* theta, const float* alpha, const float* x, int64_t batch, int64_t n, int64_t m,
                           const lbbnn_noise* noise, int flags, float* act, float* ds_factor, float* q, void* workspace,
                           size_t workspace_bytes, lbbnn_stream s);
LBBNN_API int lbbnn_vd_bwd(const float* theta, const float* alpha, const float* x, const float* act, const float* ds_factor,
                           const float* q, const float* gact, int64_t batch, int64_t n, int64_t m, int flags,
                           float* d_theta, float* d_alpha, float* dx, void* workspace, size_t workspace_bytes,
                           lbbnn_stream s);
LBBNN_API int lbbnn_vd_kl(const float* alpha, int64_t m, float* kl_out, int kl_accumulate, float* d_alpha, float grad_scale,
                          lbbnn_stream s);

#ifdef __cplusplus
}
#endif
#endif /* LBBNN_H */
