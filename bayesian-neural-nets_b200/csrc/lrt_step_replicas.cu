// The replica launch of the one-launch LRT step (lbbnn_lrt_step_replicas_*): R networks of one shape trained side by side by
// lrt_step_kernel<false, true> (lrt_step.cuh).  A translation unit of its own: see lrt_step.cu.
#include "lrt_step.cuh"

using namespace lbbnn;

// ---- replica launch ---------------------------------------------------------------------------------------------------
namespace {
int check_replicas(const lbbnn_step* S, const lbbnn_step_replicas* Rp) {
  LBBNN_REQUIRE(S != nullptr && Rp != nullptr, "step or replicas is NULL");
  LBBNN_REQUIRE(Rp->replicas >= 1 && Rp->replicas <= LBBNN_STEP_MAX_REPLICAS, "replicas must be 1..%d (got %d)",
                LBBNN_STEP_MAX_REPLICAS, Rp->replicas);
  LBBNN_REQUIRE(Rp->param_stride > 0 && Rp->param_stride % 4 == 0, "param_stride must be a positive multiple of 4 floats (got %lld)",
                (long long)Rp->param_stride);
  LBBNN_REQUIRE(Rp->x_stride >= 0 && Rp->y_stride >= 0, "x_stride and y_stride must be >= 0 (got %lld, %lld)",
                (long long)Rp->x_stride, (long long)Rp->y_stride);
  LBBNN_REQUIRE(S->dp == nullptr, "the replica launch has no data-parallel exchange (dp must be NULL)");
  LBBNN_REQUIRE(S->n_layers >= 1 && S->n_layers <= kMaxL, "n_layers must be 1..%d", kMaxL);
  for (int l = 0; l < S->n_layers; ++l) {   // one replica's tensors lie inside its stride
    const lbbnn_step_layer& y = S->layer[l];
    const int64_t nk = y.in_features * y.out_features, n = y.out_features;
    const int64_t end = std::max({y.off_weight_mu + nk, y.off_weight_rho + nk, y.off_lambdal + nk, y.off_bias_mu + n, y.off_bias_rho + n});
    const int64_t lo = std::min({y.off_weight_mu, y.off_weight_rho, y.off_lambdal, y.off_bias_mu, y.off_bias_rho});
    LBBNN_REQUIRE(lo >= 0 && end <= Rp->param_stride, "layer %d's tensors end at float %lld, past param_stride %lld", l,
                  (long long)end, (long long)Rp->param_stride);
  }
  return LBBNN_OK;
}
}  // namespace

extern "C" size_t lbbnn_lrt_step_replicas_workspace_bytes(const lbbnn_step* S, const lbbnn_step_replicas* Rp) {
  HostPlan P;
  if (check_replicas(S, Rp) != LBBNN_OK) return 0;
  if (plan_step(S, sm_count() * kCtasPerSm, Rp->replicas, &P) != LBBNN_OK) return 0;
  return P.total;
}

extern "C" int lbbnn_lrt_step_replicas_describe(const lbbnn_step* S, const lbbnn_step_replicas* Rp, char* buf, size_t buf_bytes) {
  HostPlan P;
  if (int rc = check_replicas(S, Rp)) return rc;
  if (int rc = plan_step(S, sm_count() * kCtasPerSm, Rp->replicas, &P)) return rc;
  return describe_plan(P, buf, buf_bytes);
}

extern "C" int lbbnn_lrt_step_replicas_f32(const lbbnn_step* S, const lbbnn_step_replicas* Rp, void* ws, size_t ws_bytes,
                                           lbbnn_stream s) {
  if (int rc = check_replicas(S, Rp)) return rc;
  int G = 0;
  HostPlan P;
  if (int rc = plan_step(S, sm_count() * kCtasPerSm, Rp->replicas, &P)) return rc;
  if (int rc = step_grid(P.smem, &G, {(const void*)lrt_step_kernel<false, true>})) return rc;
  LBBNN_REQUIRE(G == sm_count() * kCtasPerSm, "grid size mismatch");
  LBBNN_REQUIRE(ws && ws_bytes >= P.total, "workspace too small (%zu < %zu)", ws_bytes, P.total);
  LBBNN_REQUIRE(S->flat && S->exp_avg && S->exp_avg_sq && S->x && S->y && S->step_dev && S->stats && Rp->seeds, "NULL argument");
  bind_workspace(P, (char*)ws, G);
  DevStep& d = P.d;
  d.phases = 3;
  d.flat = S->flat; d.m = S->exp_avg; d.v = S->exp_avg_sq; d.grad = S->grad;
  d.x = S->x; d.y = S->y; d.step_dev = S->step_dev; d.seed = 0;
  d.lr = S->lr; d.b1 = S->beta1; d.b2 = S->beta2; d.eps = S->eps; d.klg = S->kl_scale;
  d.stats = S->stats;
  d.prof = g_step_prof;
  d.prof_cta = g_step_prof_cta;
  d.dp_p2p = 0;
  for (int p = 0; p < 8; ++p) { d.flat_peer[p] = nullptr; d.raw_peer[p] = nullptr; d.dp_signal[p] = nullptr; d.dp_klx[p] = nullptr; }
  d.dp_world = 1; d.dp_rank = 0; d.flat_mc = nullptr; d.raw_mc = nullptr; d.raw_base = (const float*)ws; d.dp_epoch = nullptr;
  d.overlap_update = 0;
  d.p_stride = Rp->param_stride; d.x_stride = Rp->x_stride; d.y_stride = Rp->y_stride; d.seeds = Rp->seeds;
  void* args[] = {(void*)&d};
  LBBNN_CUDA(cudaLaunchCooperativeKernel((const void*)lrt_step_kernel<false, true>, dim3((unsigned)G), dim3(NT), args, kSmemCap,
                                         (cudaStream_t)s));
  return check_launch("lrt_step_kernel");
}
