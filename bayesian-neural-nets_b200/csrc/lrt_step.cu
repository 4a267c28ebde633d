// Whole training step of a small LRT stack as ONE persistent cooperative kernel: the single-network entry points (the kernel,
// its phases and the planner are in lrt_step.cuh; the replica launch is compiled in lrt_step_replicas.cu, so that this
// translation unit holds only the single-network and data-parallel instantiations and compiles to the same code as before the
// replica axis existed).
#include "lrt_step.cuh"

using namespace lbbnn;

namespace lbbnn {
long long* g_step_prof = nullptr;
int g_step_prof_cta = 0;
}  // namespace lbbnn

extern "C" int lbbnn_lrt_step_profile(long long* dev_stamps) {
  g_step_prof = dev_stamps;
  const char* e = getenv("LBBNN_STEP_PROF_CTA");
  g_step_prof_cta = e ? atoi(e) : 0;
  return LBBNN_OK;
}

extern "C" size_t lbbnn_lrt_step_workspace_bytes(const lbbnn_step* S) {
  HostPlan P;
  if (plan_step(S, sm_count() * kCtasPerSm, 1, &P) != LBBNN_OK) return 0;
  return P.total;
}

extern "C" size_t lbbnn_lrt_step_raw_floats(const lbbnn_step* S) {
  HostPlan P;
  if (plan_step(S, sm_count() * kCtasPerSm, 1, &P) != LBBNN_OK) return 0;
  return P.raw_floats;
}

extern "C" int lbbnn_lrt_step_f32(const lbbnn_step* S, int phases, void* ws, size_t ws_bytes, lbbnn_stream s) {
  LBBNN_REQUIRE(phases >= 1 && phases <= 7, "phases must be 1 (forward+backward), 2 (update) or 3 (both)");
  int G = 0;
  HostPlan P;
  if (int rc = plan_step(S, sm_count() * kCtasPerSm, 1, &P)) return rc;
  if (int rc = step_grid(P.smem, &G, {(const void*)lrt_step_kernel<false, false>, (const void*)lrt_step_kernel<true, false>})) return rc;
  LBBNN_REQUIRE(G == sm_count() * kCtasPerSm, "grid size mismatch");
  LBBNN_REQUIRE(ws && ws_bytes >= P.total, "workspace too small (%zu < %zu)", ws_bytes, P.total);
  LBBNN_REQUIRE(S->flat && S->exp_avg && S->exp_avg_sq && S->x && S->y && S->step_dev && S->stats, "NULL argument");
  bind_workspace(P, (char*)ws, G);
  DevStep& d = P.d;
  d.phases = phases;
  d.flat = S->flat; d.m = S->exp_avg; d.v = S->exp_avg_sq; d.grad = S->grad;
  d.x = S->x; d.y = S->y; d.step_dev = S->step_dev; d.seed = S->seed;
  d.lr = S->lr; d.b1 = S->beta1; d.b2 = S->beta2; d.eps = S->eps; d.klg = S->kl_scale;
  d.stats = S->stats;
  d.prof = g_step_prof;
  d.dp_p2p = 0;
  for (int p = 0; p < 8; ++p) { d.flat_peer[p] = nullptr; d.raw_peer[p] = nullptr; }
  d.dp_world = 1; d.dp_rank = 0; d.flat_mc = nullptr; d.raw_mc = nullptr; d.raw_base = (const float*)ws; d.dp_epoch = nullptr;
  for (int p = 0; p < 8; ++p) { d.dp_signal[p] = nullptr; d.dp_klx[p] = nullptr; }
  if (S->dp && S->dp->world > 1) {
    const lbbnn_step_dp* D = S->dp;
    LBBNN_REQUIRE(phases == 3, "the in-launch data-parallel exchange needs phases == 3");
    LBBNN_REQUIRE(D->world <= 8 && D->rank >= 0 && D->rank < D->world, "bad data-parallel rank %d of %d", D->rank, D->world);
    LBBNN_REQUIRE(D->epoch && (D->use_p2p || (D->flat_mc && D->ws_mc)), "NULL multicast address / epoch");
    LBBNN_REQUIRE(S->grad == nullptr, "the sharded update does not materialise gradients (grad must be NULL)");
    for (int p = 0; p < D->world; ++p) LBBNN_REQUIRE(D->signal[p] && D->klx[p], "NULL peer mapping %d", p);
    for (int l = 0; l < d.L; ++l)
      LBBNN_REQUIRE(((int64_t)d.ly[l].N * d.ly[l].K) % 4 == 0, "sharded update needs in*out %% 4 == 0 (layer %d)", l);
    d.dp_world = D->world; d.dp_rank = D->rank; d.flat_mc = D->flat_mc; d.raw_mc = D->ws_mc; d.dp_epoch = D->epoch;
    for (int p = 0; p < D->world; ++p) { d.dp_signal[p] = D->signal[p]; d.dp_klx[p] = D->klx[p]; }
    d.dp_p2p = D->use_p2p ? 1 : 0;
    for (int p = 0; p < D->world; ++p) {
      LBBNN_REQUIRE(!D->use_p2p || (D->flat_peer[p] && D->ws_peer[p]), "NULL peer buffer %d", p);
      d.flat_peer[p] = D->flat_peer[p]; d.raw_peer[p] = D->ws_peer[p];
    }
  }
  d.overlap_update = (getenv("LBBNN_STEP_OVERLAP_UPDATE") && d.dp_world == 1) ? 1 : 0;
  d.prof_cta = g_step_prof_cta;
  void* args[] = {(void*)&d};
  const void* kern = d.dp_world > 1 ? (const void*)lrt_step_kernel<true, false> : (const void*)lrt_step_kernel<false, false>;
  LBBNN_CUDA(cudaLaunchCooperativeKernel(kern, dim3((unsigned)G), dim3(NT), args, kSmemCap, (cudaStream_t)s));
  return check_launch("lrt_step_kernel");
}

extern "C" int lbbnn_lrt_step_describe(const lbbnn_step* S, char* buf, size_t buf_bytes) {
  HostPlan P;
  if (int rc = plan_step(S, sm_count() * kCtasPerSm, 1, &P)) return rc;
  return describe_plan(P, buf, buf_bytes);
}

