// extern "C" entry points that are not tied to one kernel file: error string, launch counter,
// packing and the score / stats dispatch.
#include <cstdarg>
#include <cstdlib>
#include <mutex>
#include <string>

#include "common.cuh"

namespace ssp {

static thread_local char g_err[1024] = "";
static std::atomic<int64_t> g_launches{0};
// per-kernel launch counts since the last reset (names are string literals: compared by content, few entries)
static std::mutex g_log_mu;
static const char* g_log_name[64];
static int64_t g_log_count[64];
static int g_log_n = 0;
static char g_log_text[4096];

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(const char* name) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  std::lock_guard<std::mutex> lk(g_log_mu);
  for (int i = 0; i < g_log_n; ++i)
    if (g_log_name[i] == name || strcmp(g_log_name[i], name) == 0) { ++g_log_count[i]; return; }
  if (g_log_n < 64) { g_log_name[g_log_n] = name; g_log_count[g_log_n++] = 1; }
}

}  // namespace ssp

extern "C" int ssp_abi_version(void) { return SSP_ABI_VERSION; }
extern "C" const char* ssp_last_error(void) { return ssp::g_err; }
extern "C" int64_t ssp_launch_count(void) { return ssp::g_launches.load(); }
extern "C" void ssp_reset_launch_count(void) {
  ssp::g_launches.store(0);
  std::lock_guard<std::mutex> lk(ssp::g_log_mu);
  ssp::g_log_n = 0;
}
extern "C" const char* ssp_launch_log(void) {
  std::lock_guard<std::mutex> lk(ssp::g_log_mu);
  size_t o = 0;
  ssp::g_log_text[0] = 0;
  for (int i = 0; i < ssp::g_log_n && o + 128 < sizeof(ssp::g_log_text); ++i)
    o += snprintf(ssp::g_log_text + o, sizeof(ssp::g_log_text) - o, "%s%s:%lld", i ? "," : "", ssp::g_log_name[i],
                  (long long)ssp::g_log_count[i]);
  return ssp::g_log_text;
}

// Workspaces of the statistics, posterior and shared-variance calls: the tensor-core kernels write the operand images
// with 16-byte (uint4) stores and stream them into shared memory with cp.async.bulk, whose global source must be 16-byte
// aligned.  Every section inside a workspace starts at a multiple of 256 bytes from its base, so the base is what counts.
static constexpr uintptr_t kWorkspaceAlign = 16;

// The workspace argument of `fn`: 16-byte aligned (NULL passes), and at least `need` bytes where the call needs one (no
// silent slower path: a short workspace is the caller's error).  `query` names the entry point that gives `need`.
static int check_workspace(const char* fn, const void* workspace, int64_t workspace_bytes, int64_t need, const char* query) {
  SSP_REQUIRE(((uintptr_t)workspace & (kWorkspaceAlign - 1)) == 0, "%s: workspace must be %d-byte aligned", fn,
              (int)kWorkspaceAlign);
  SSP_REQUIRE(need == 0 || (workspace && workspace_bytes >= need), "%s: workspace of %lld bytes, need %lld (%s)", fn,
              (long long)(workspace ? workspace_bytes : 0), (long long)need, query);
  return SSP_OK;
}

extern "C" int64_t ssp_gmm_pack_bytes(const ssp_gmm_dims* dims) {
  ssp::PackLayout L;
  if (!ssp::make_layout(dims, &L)) return 0;
  return (int64_t)L.bytes;
}

extern "C" int ssp_gmm_pack_models(const double* weights, const double* means, const double* variances,
                                   const ssp_gmm_dims* dims, void* out_pack, void* stream) {
  ssp::PackLayout L;
  SSP_REQUIRE(ssp::make_layout(dims, &L), "ssp_gmm_pack_models: unsupported dims (need 1 <= D <= %d)", ssp::kMaxFeat);
  SSP_REQUIRE(weights && means && variances && out_pack, "ssp_gmm_pack_models: null pointer");
  SSP_REQUIRE(((uintptr_t)out_pack & 127) == 0, "ssp_gmm_pack_models: out_pack must be 128-byte aligned");
  return ssp::launch_pack(weights, means, variances, L, out_pack, (cudaStream_t)stream);
}

extern "C" int ssp_gmm_score(const float* feats, const int64_t* frame_offsets, int64_t n_utts, int64_t total_frames,
                             const void* pack, const ssp_gmm_dims* dims, int32_t precision, double* out_scores,
                             float* out_frame_lse, void* stream) {
  ssp::PackLayout L;
  SSP_REQUIRE(ssp::make_layout(dims, &L), "ssp_gmm_score: unsupported dims");
  SSP_REQUIRE(frame_offsets && pack && out_scores && (feats || total_frames == 0), "ssp_gmm_score: null pointer");
  SSP_REQUIRE(n_utts >= 0 && total_frames >= 0, "ssp_gmm_score: negative size");
  if (n_utts == 0) return SSP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == SSP_PREC_FP32)
    return ssp::launch_score_simt(feats, frame_offsets, n_utts, total_frames, pack, L, true, out_scores, out_frame_lse, st);
  if (precision == SSP_PREC_TF32 || precision == SSP_PREC_TF32X2 || precision == SSP_PREC_TF32X3)
    return ssp::launch_score_tc(feats, frame_offsets, n_utts, total_frames, pack, L,
                                precision == SSP_PREC_TF32 ? 1 : precision == SSP_PREC_TF32X2 ? 2 : 3, true, out_scores,
                                out_frame_lse, st);
  SSP_REQUIRE(false, "ssp_gmm_score: unknown precision %d", precision);
}

extern "C" int64_t ssp_gmm_shared_pack_bytes(const ssp_gmm_dims* dims) {
  ssp::SvLayout L;
  if (!ssp::make_sv_layout(dims, &L)) return 0;
  return (int64_t)L.bytes;
}

extern "C" int ssp_gmm_pack_shared(const double* weights, const double* variances, const double* means,
                                   const ssp_gmm_dims* dims, int32_t ref_model, void* out_pack, void* stream) {
  ssp::SvLayout L;
  SSP_REQUIRE(ssp::make_sv_layout(dims, &L), "ssp_gmm_pack_shared: unsupported dims (need 1 <= D <= %d)", ssp::kSvMaxFeat);
  SSP_REQUIRE(weights && variances && means && out_pack, "ssp_gmm_pack_shared: null pointer");
  SSP_REQUIRE(((uintptr_t)out_pack & 127) == 0, "ssp_gmm_pack_shared: out_pack must be 128-byte aligned");
  SSP_REQUIRE(ref_model >= 0 && ref_model < L.n_models, "ssp_gmm_pack_shared: ref_model %d outside [0, %d)", ref_model,
              L.n_models);
  return ssp::launch_pack_sv(weights, variances, means, L, ref_model, out_pack, (cudaStream_t)stream);
}

extern "C" int64_t ssp_gmm_score_shared_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames) {
  ssp::SvLayout L;
  if (!ssp::make_sv_layout(dims, &L) || total_frames < 0) return 0;
  return ssp::score_sv_workspace_bytes(L, total_frames);
}

extern "C" int ssp_gmm_score_shared(const float* feats, const int64_t* frame_offsets, int64_t n_utts, int64_t total_frames,
                                    const void* pack, const ssp_gmm_dims* dims, double* out_scores, float* out_frame_lse,
                                    void* workspace, int64_t workspace_bytes, void* stream) {
  ssp::SvLayout L;
  SSP_REQUIRE(ssp::make_sv_layout(dims, &L), "ssp_gmm_score_shared: unsupported dims");
  SSP_REQUIRE(frame_offsets && pack && out_scores && (feats || total_frames == 0), "ssp_gmm_score_shared: null pointer");
  SSP_REQUIRE(n_utts >= 0 && total_frames >= 0, "ssp_gmm_score_shared: negative size");
  int rc = check_workspace("ssp_gmm_score_shared", workspace, workspace_bytes, ssp::score_sv_workspace_bytes(L, total_frames),
                           "ssp_gmm_score_shared_workspace_bytes");
  if (rc != SSP_OK || n_utts == 0) return rc;
  return ssp::launch_score_sv(feats, frame_offsets, n_utts, total_frames, pack, L, true, out_scores, out_frame_lse, workspace,
                              (cudaStream_t)stream);
}

extern "C" int64_t ssp_gmm_stats_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames, int64_t n_segs) {
  ssp::PackLayout L;
  if (!ssp::make_layout(dims, &L) || total_frames < 0 || n_segs < 0) return 0;
  return ssp::stats_tc_workspace_bytes(L, total_frames, n_segs);
}

extern "C" int ssp_gmm_stats(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                             const void* pack, const ssp_gmm_dims* dims, float* frame_lse, double* out_n, double* out_f,
                             double* out_s, double* out_loglik, void* workspace, int64_t workspace_bytes, int32_t reuse_images,
                             void* stream) {
  ssp::PackLayout L;
  SSP_REQUIRE(ssp::make_layout(dims, &L), "ssp_gmm_stats: unsupported dims");
  SSP_REQUIRE(dims->n_models == 1 || dims->n_models == n_segs,
              "ssp_gmm_stats: %d models for %lld segments (one model for all segments, or one per segment)", dims->n_models,
              (long long)n_segs);
  SSP_REQUIRE(seg_offsets && pack && frame_lse && out_n && out_f && out_s && out_loglik, "ssp_gmm_stats: null pointer");
  SSP_REQUIRE(n_segs >= 0 && total_frames >= 0, "ssp_gmm_stats: negative size");
  // only the tensor-core path takes a workspace (0 bytes otherwise)
  int rc = check_workspace("ssp_gmm_stats", workspace, workspace_bytes,
                           n_segs ? ssp::stats_tc_workspace_bytes(L, total_frames, n_segs) : 0, "ssp_gmm_stats_workspace_bytes");
  if (rc != SSP_OK || n_segs == 0) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // The tensor-core kernels serve every feature width they support (D <= 39); the FP32 CUDA-core kernels serve wider
  // features only.
  if (ssp::stats_tc_supported(L)) {
    return ssp::launch_stats_tc(feats, seg_offsets, n_segs, total_frames, pack, L, frame_lse, out_n, out_f, out_s, out_loglik,
                                workspace, reuse_images != 0, st);
  }
  if (dims->n_models != 1) {
    ssp::set_error("ssp_gmm_stats: per-segment models need the tensor-core path (D <= 39, n_models <= %d)", ssp::kMaxTrainModels);
    return SSP_EUNSUP;
  }
  // FP32 CUDA-core path (D > 39).  pass 1: per-frame log-likelihood and the per-segment sum of frame log-likelihoods (the EM
  // lower bound numerator, sklearn _base.py:558); pass 2: posteriors and N/F/S
  rc = ssp::launch_score_simt(feats, seg_offsets, n_segs, total_frames, pack, L, false, out_loglik, frame_lse, st);
  if (rc != SSP_OK) return rc;
  return ssp::launch_stats_simt(feats, seg_offsets, n_segs, total_frames, pack, L, frame_lse, out_n, out_f, out_s, st);
}

extern "C" int64_t ssp_gmm_posteriors_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames, int64_t n_segs) {
  ssp::PackLayout L;
  if (!ssp::make_layout(dims, &L) || total_frames < 0 || n_segs < 0) return 0;
  if (ssp::stats_tc_supported(L)) return ssp::stats_tc_workspace_bytes(L, total_frames, n_segs);
  return L.n_models == 1 ? ssp::posteriors_simt_workspace_bytes(total_frames, n_segs) : 0;
}

extern "C" int ssp_gmm_posteriors(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                                  const void* pack, const ssp_gmm_dims* dims, float* out_resp, int64_t* out_label,
                                  float* out_frame_lse, void* workspace, int64_t workspace_bytes, int32_t reuse_images,
                                  void* stream) {
  ssp::PackLayout L;
  SSP_REQUIRE(ssp::make_layout(dims, &L), "ssp_gmm_posteriors: unsupported dims");
  SSP_REQUIRE(dims->n_models == 1 || dims->n_models == n_segs,
              "ssp_gmm_posteriors: %d models for %lld segments (one model for all segments, or one per segment)",
              dims->n_models, (long long)n_segs);
  SSP_REQUIRE(out_resp || out_label, "ssp_gmm_posteriors: out_resp and out_label are both NULL (nothing to compute)");
  SSP_REQUIRE(seg_offsets && pack && (feats || total_frames == 0), "ssp_gmm_posteriors: null pointer");
  SSP_REQUIRE(n_segs >= 0 && total_frames >= 0, "ssp_gmm_posteriors: negative size");
  const bool empty = n_segs == 0 || total_frames == 0;
  int rc = check_workspace("ssp_gmm_posteriors", workspace, workspace_bytes,
                           empty ? 0 : ssp_gmm_posteriors_workspace_bytes(dims, total_frames, n_segs),
                           "ssp_gmm_posteriors_workspace_bytes");
  if (rc != SSP_OK || empty) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (ssp::stats_tc_supported(L)) {
    return ssp::launch_posteriors_tc(feats, seg_offsets, n_segs, total_frames, pack, L, out_resp, out_label, out_frame_lse,
                                     workspace, reuse_images != 0, st);
  }
  if (dims->n_models != 1) {
    ssp::set_error("ssp_gmm_posteriors: per-segment models need the tensor-core path (D <= 39, n_models <= %d)",
                   ssp::kMaxTrainModels);
    return SSP_EUNSUP;
  }
  return ssp::launch_posteriors_simt(feats, seg_offsets, n_segs, total_frames, pack, L, out_resp, out_label, out_frame_lse,
                                     workspace, st);
}

extern "C" int64_t ssp_gmm_top_components_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames, int64_t n_segs,
                                                          int32_t c) {
  ssp::PackLayout L;
  if (!ssp::make_layout(dims, &L) || L.n_models != 1 || total_frames < 0 || n_segs < 0 || c < 1 || c > ssp::kTopcMaxC)
    return 0;
  return ssp::topc_tc_workspace_bytes(L, total_frames, n_segs, c);
}

extern "C" int ssp_gmm_top_components(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                                      const void* pack, const ssp_gmm_dims* dims, int32_t c, int32_t* out_idx, float* out_logit,
                                      void* workspace, int64_t workspace_bytes, int32_t reuse_images, void* stream) {
  ssp::PackLayout L;
  SSP_REQUIRE(ssp::make_layout(dims, &L), "ssp_gmm_top_components: unsupported dims");
  SSP_REQUIRE(dims->n_models == 1, "ssp_gmm_top_components: %d models (selection runs under one model)", dims->n_models);
  if (!ssp::stats_tc_supported(L)) {
    ssp::set_error("ssp_gmm_top_components: D = %d (the selection kernels take D <= %d)", L.D, ssp::kTopcMaxFeat);
    return SSP_EUNSUP;
  }
  SSP_REQUIRE(c >= 1 && c <= L.K && c <= ssp::kTopcMaxC, "ssp_gmm_top_components: C = %d outside [1, min(K = %d, %d)]", c, L.K,
              ssp::kTopcMaxC);
  SSP_REQUIRE(seg_offsets && pack && out_idx && out_logit && (feats || total_frames == 0), "ssp_gmm_top_components: null pointer");
  SSP_REQUIRE(n_segs >= 0 && total_frames >= 0, "ssp_gmm_top_components: negative size");
  const bool empty = n_segs == 0 || total_frames == 0;
  int rc = check_workspace("ssp_gmm_top_components", workspace, workspace_bytes,
                           empty ? 0 : ssp::topc_tc_workspace_bytes(L, total_frames, n_segs, c),
                           "ssp_gmm_top_components_workspace_bytes");
  if (rc != SSP_OK || empty) return rc;
  return ssp::launch_topc_tc(feats, seg_offsets, n_segs, total_frames, pack, L, c, out_idx, out_logit, workspace,
                             reuse_images != 0, (cudaStream_t)stream);
}

static bool topc_dims_ok(const ssp_gmm_dims* dims) {
  return dims && dims->n_models >= 1 && dims->n_comp >= 1 && dims->n_feat >= 1 && dims->n_feat <= ssp::kTopcMaxFeat;
}

extern "C" int64_t ssp_gmm_topc_pack_bytes(const ssp_gmm_dims* dims) {
  return topc_dims_ok(dims) ? ssp::topc_pack_bytes(dims->n_models, dims->n_comp, dims->n_feat) : 0;
}

extern "C" int ssp_gmm_pack_topc(const double* variances, const double* means, const ssp_gmm_dims* dims, int32_t ref_model,
                                 void* out_pack, void* stream) {
  SSP_REQUIRE(topc_dims_ok(dims), "ssp_gmm_pack_topc: unsupported dims (need 1 <= D <= %d)", ssp::kTopcMaxFeat);
  SSP_REQUIRE(variances && means && out_pack, "ssp_gmm_pack_topc: null pointer");
  SSP_REQUIRE(((uintptr_t)out_pack & 15) == 0, "ssp_gmm_pack_topc: out_pack must be 16-byte aligned");
  SSP_REQUIRE(ref_model >= 0 && ref_model < dims->n_models, "ssp_gmm_pack_topc: ref_model %d outside [0, %d)", ref_model,
              dims->n_models);
  return ssp::launch_pack_topc(variances, means, dims->n_models, dims->n_comp, dims->n_feat, ref_model, out_pack,
                               (cudaStream_t)stream);
}

extern "C" int64_t ssp_gmm_topc_adapted_pack_bytes(const ssp_gmm_dims* dims) {
  return topc_dims_ok(dims) ? ssp::topc_adapted_pack_bytes(dims->n_models, dims->n_comp, dims->n_feat) : 0;
}

extern "C" int ssp_gmm_pack_topc_adapted(const double* weights, const double* means, const double* variances,
                                         const ssp_gmm_dims* dims, int32_t ref_model, void* out_pack, void* stream) {
  SSP_REQUIRE(topc_dims_ok(dims), "ssp_gmm_pack_topc_adapted: unsupported dims (need 1 <= D <= %d)", ssp::kTopcMaxFeat);
  SSP_REQUIRE(weights && means && variances && out_pack, "ssp_gmm_pack_topc_adapted: null pointer");
  SSP_REQUIRE(((uintptr_t)out_pack & 15) == 0, "ssp_gmm_pack_topc_adapted: out_pack must be 16-byte aligned");
  SSP_REQUIRE(ref_model >= 0 && ref_model < dims->n_models, "ssp_gmm_pack_topc_adapted: ref_model %d outside [0, %d)",
              ref_model, dims->n_models);
  return ssp::launch_pack_topc_adapted(weights, means, variances, dims->n_models, dims->n_comp, dims->n_feat, ref_model,
                                       out_pack, (cudaStream_t)stream);
}

extern "C" int64_t ssp_gmm_topc_chunk_frames(void) { return ssp::kTopcChunkFrames; }

extern "C" int64_t ssp_gmm_score_topc_workspace_bytes(const ssp_gmm_dims* dims, int32_t c, int64_t total_frames) {
  if (!topc_dims_ok(dims) || c < 1 || c > dims->n_comp || c > ssp::kTopcMaxC || total_frames < 0) return 0;
  return ssp::score_topc_workspace_bytes(dims->n_models, dims->n_comp, c, total_frames);
}

// ssp_gmm_score_topc (adapted == false) and ssp_gmm_score_topc_adapted: the same checks, the same workspace
static int score_topc(const char* fn, bool adapted, const float* feats, const int64_t* frame_offsets, int64_t n_utts,
                      int64_t total_frames, const int32_t* idx, const float* logit, int32_t c, const void* pack,
                      const ssp_gmm_dims* dims, double* out_scores, float* out_frame_lse, void* workspace,
                      int64_t workspace_bytes, void* stream) {
  SSP_REQUIRE(topc_dims_ok(dims), "%s: unsupported dims (need 1 <= D <= %d)", fn, ssp::kTopcMaxFeat);
  SSP_REQUIRE(c >= 1 && c <= dims->n_comp && c <= ssp::kTopcMaxC, "%s: C = %d outside [1, min(K = %d, %d)]", fn, c,
              dims->n_comp, ssp::kTopcMaxC);
  SSP_REQUIRE(frame_offsets && pack && out_scores && ((feats && idx && logit) || total_frames == 0), "%s: null pointer", fn);
  SSP_REQUIRE(((uintptr_t)pack & 15) == 0, "%s: pack must be 16-byte aligned", fn);
  SSP_REQUIRE(n_utts >= 0 && total_frames >= 0, "%s: negative size", fn);
  int rc = check_workspace(fn, workspace, workspace_bytes,
                           ssp::score_topc_workspace_bytes(dims->n_models, dims->n_comp, c, total_frames),
                           "ssp_gmm_score_topc_workspace_bytes");
  if (rc != SSP_OK || n_utts == 0) return rc;
  return ssp::launch_score_topc(feats, frame_offsets, n_utts, total_frames, idx, logit, c, pack, dims->n_models, dims->n_comp,
                                dims->n_feat, adapted, out_scores, out_frame_lse, workspace, (cudaStream_t)stream);
}

extern "C" int ssp_gmm_score_topc(const float* feats, const int64_t* frame_offsets, int64_t n_utts, int64_t total_frames,
                                  const int32_t* idx, const float* logit, int32_t c, const void* pack, const ssp_gmm_dims* dims,
                                  double* out_scores, float* out_frame_lse, void* workspace, int64_t workspace_bytes,
                                  void* stream) {
  return score_topc("ssp_gmm_score_topc", false, feats, frame_offsets, n_utts, total_frames, idx, logit, c, pack, dims,
                    out_scores, out_frame_lse, workspace, workspace_bytes, stream);
}

extern "C" int ssp_gmm_score_topc_adapted(const float* feats, const int64_t* frame_offsets, int64_t n_utts,
                                          int64_t total_frames, const int32_t* idx, const float* logit, int32_t c,
                                          const void* pack, const ssp_gmm_dims* dims, double* out_scores,
                                          float* out_frame_lse, void* workspace, int64_t workspace_bytes, void* stream) {
  return score_topc("ssp_gmm_score_topc_adapted", true, feats, frame_offsets, n_utts, total_frames, idx, logit, c, pack, dims,
                    out_scores, out_frame_lse, workspace, workspace_bytes, stream);
}
