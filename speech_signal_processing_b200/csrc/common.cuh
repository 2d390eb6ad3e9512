// Shared host/device helpers for the ssp_b200 library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdio>
#include <cstring>

#include "../../include/ssp_b200.h"

namespace ssp {

// ---------------------------------------------------------------- error / launch bookkeeping
void set_error(const char* fmt, ...);
void count_launch(const char* kernel_name);

#define SSP_CUDA_OK(expr)                                                              \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      ::ssp::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return SSP_ECUDA;                                                                \
    }                                                                                  \
  } while (0)

#define SSP_REQUIRE(cond, ...)          \
  do {                                  \
    if (!(cond)) {                      \
      ::ssp::set_error(__VA_ARGS__);    \
      return SSP_EINVAL;                \
    }                                   \
  } while (0)

#define SSP_LAUNCH_CHECK(name)          \
  do {                                  \
    ::ssp::count_launch(name);          \
    SSP_CUDA_OK(cudaGetLastError());    \
  } while (0)

// ---------------------------------------------------------------- packed-model layout
// One buffer holds both operand forms of every model (see ssp_gmm_pack_models):
//   E (exact, CUDA-core kernels): ab[m][c][d] = (mu/var, -1/(2 var)) float2, d < DP (zero padded),
//                                 cst[m][c]   = log w - 0.5(D log 2pi + sum mu^2/var) + 0.5 sum log(1/var)
//   T (tensor, tcgen05 kernel):   tile[m][c/128] = shared-memory image [KD/4][128] float4 of the
//                                 TF32-rounded, log2(e)-scaled rows [mu/var, -1/(2var), c_hi, c_lo, 0..]
constexpr int kTileN = 128;  // components per tensor tile / padding granule of K
constexpr int kMaxFeat = 80;
constexpr int kMaxTrainModels = 1024;  // model sets up to this size carry the BF16 images ssp_gmm_stats needs

struct PackLayout {
  int n_models, K, D;
  int Kp;  // K rounded up to kTileN (padded components have cst = -1e30, zero rows)
  int DP;  // D padded for the CUDA-core kernels: 16, 32, 40, 64 or 80
  int KD;  // contraction length of the tensor kernel: roundup(2D + 2, 8)
  size_t off_ab, off_cst, off_tile, off_tile_lo, off_tile_bf, off_tile_h, off_tile_hl, off_flag, bytes;  // off_tile_bf == 0: no BF16 images (n_models > 1)
  int KDb() const { return (2 * D + 2 + 15) / 16 * 16; }  // contraction length of the BF16 / FP16 images (multiple of 16)
  size_t tile_floats() const { return (size_t)kTileN * KD; }
};

// Shared-variance model sets (gmm_score_sv.cu): every model has the base model's weights and variances and its own
// means.  One buffer of tcgen05 shared-memory images (K-major, no swizzle), [Kp/64 tiles][kSvBaseImages + n_models]
// [KS/8][64][8] FP16, all scaled by log2(e), + a 128-byte tail (overflow flag of the pack kernel).  The common part is
// the full logit of the REFERENCE member, contraction [x^2 | x | 1, 1] of length KQ, as two FP16 pieces (hi + lo exact
// to ~2^-22) cut into ring-slot-sized column ranges:
//   images 0, 1  = hi piece, columns [0, KS) and [KS, KQ) of [-1/(2 var) | mu_ref/var | c1, c2 | 0..]
//   images 2, 3  = lo piece, same columns ................ of [residuals ..................| c3, 0 | 0..]
//                  c = log w - D/2 log 2pi - 1/2 sum log var - 1/2 sum mu_ref^2 / var as three pieces
//   image 4 + s  = model s MINUS the reference  [(mu_s - mu_ref)/var, ca, cb, 0..] against [x, 1, 1024]:
//                  ca + 1024 cb = ck_s - ck_ref,  ck = -1/2 sum mu^2/var
constexpr int kSvTileN = 64;
constexpr int kSvMaxKS = 64;
constexpr int kSvBaseImages = 4;
constexpr float kSvConstScale = 1024.f;  // second "one" column of the per-model frame operand (range of the model constants)
// shape of gmm_score_sv_kernel (here because it bounds the feature width the layout accepts)
constexpr int kSvStages = 12, kSvSlots = 6, kSvChunk = 32, kSvUnit = 256;
constexpr size_t kMaxDynSmem = 232448;  // 227 KB per CTA on sm_100
constexpr int kSvMaxFeat = 39;          // widest feature vector whose operands fit (sv_smem_bytes)
struct SvLayout {
  int n_models, K, D;
  int Kp;  // K rounded up to kSvTileN
  int KS;  // contraction length of the per-model part: roundup(D + 2, 16)
  int KQ;  // contraction length of the common part: roundup(2 D + 2, 16) <= 2 KS
  size_t flag_offset;  // int32 at the tail: set by the pack kernel when a value leaves FP16's range
  size_t bytes;
};
inline size_t sv_smem_bytes(int KS, int KQ) {
  return (size_t)2 * kSvUnit * KQ * 2 + (size_t)kSvStages * kSvTileN * KS * 2 + (size_t)2 * kSvChunk * kSvUnit * 4 +
         (2 * kSvStages + 2 * kSvSlots + 2) * 8 + 16 + kSvUnit * 4;
}
inline bool make_sv_layout(const ssp_gmm_dims* dims, SvLayout* L) {
  if (!dims || dims->n_models < 1 || dims->n_comp < 1 || dims->n_feat < 1) return false;
  L->n_models = dims->n_models;
  L->K = dims->n_comp;
  L->D = dims->n_feat;
  L->Kp = (L->K + kSvTileN - 1) / kSvTileN * kSvTileN;
  L->KS = (L->D + 2 + 15) / 16 * 16;
  L->KQ = (2 * L->D + 2 + 15) / 16 * 16;
  if (L->KS > kSvMaxKS || sv_smem_bytes(L->KS, L->KQ) > kMaxDynSmem) return false;  // D <= kSvMaxFeat
  L->flag_offset = (size_t)(L->Kp / kSvTileN) * (size_t)(L->n_models + kSvBaseImages) * kSvTileN * L->KS * 2;
  L->bytes = L->flag_offset + 128;
  return true;
}

inline int pad_feat(int d) {
  if (d <= 16) return 16;
  if (d <= 32) return 32;
  if (d <= 40) return 40;
  if (d <= 64) return 64;
  return 80;
}

inline bool make_layout(const ssp_gmm_dims* dims, PackLayout* L) {
  if (!dims || dims->n_models < 1 || dims->n_comp < 1 || dims->n_feat < 1 || dims->n_feat > kMaxFeat) return false;
  L->n_models = dims->n_models;
  L->K = dims->n_comp;
  L->D = dims->n_feat;
  L->Kp = (L->K + kTileN - 1) / kTileN * kTileN;
  L->DP = pad_feat(L->D);
  L->KD = (2 * L->D + 2 + 7) / 8 * 8;
  auto up = [](size_t x) { return (x + 127) / 128 * 128; };
  size_t o = 0;
  L->off_ab = o;
  o = up(o + (size_t)L->n_models * L->Kp * L->DP * sizeof(float2));
  L->off_cst = o;
  o = up(o + (size_t)L->n_models * L->Kp * sizeof(float));
  L->off_tile = o;
  o = up(o + (size_t)L->n_models * L->Kp * L->KD * sizeof(float));
  // residual ("lo") tiles: B = hi + lo to ~2^-22 -- the 3xTF32 EM kernels and the 2- / 3-pass scoring rungs
  L->off_tile_lo = o;
  o = up(o + (size_t)L->n_models * L->Kp * L->KD * sizeof(float));
  // BF16 hi + lo images for the EM / MAP statistics kernels (the UBM, or a small set of models trained together --
  // one per segment): [model][Kp/128 tiles][hi | lo][KDb/8][128][8 bf16]; the constant rides as three BF16 pieces
  // (hi: columns 2D, 2D+1; lo: 2D)
  L->off_tile_bf = 0;
  if (L->n_models <= kMaxTrainModels && 2 * L->D + 2 <= 80) {
    L->off_tile_bf = o;
    o = up(o + (size_t)L->n_models * (L->Kp / kTileN) * 512 * L->KDb());
  }
  // FP16 images of the same rows for the tensor scoring rungs (kind::f16: K = 16 per MMA, half the bytes; an FP16
  // significand has TF32's 11 bits): [model][Kp/128 tiles][KDb/8][128][8 half], hi and residual, + a flag the pack kernel
  // raises when a value leaves FP16's range (ssp_gmm_score then streams the TF32 images instead)
  L->off_tile_h = 0;
  L->off_tile_hl = 0;
  L->off_flag = 0;
  if (2 * L->D + 2 <= 80) {
    L->off_tile_h = o;
    o = up(o + (size_t)L->n_models * L->Kp * L->KDb() * 2);
    L->off_tile_hl = o;   // residual FP16 images (hi + lo exact to ~2^-22): the 2- and 3-pass rungs
    o = up(o + (size_t)L->n_models * L->Kp * L->KDb() * 2);
    L->off_flag = o;
    o = up(o + 128);
  }
  L->bytes = o;
  return true;
}

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// index u with offsets[u] <= x < offsets[u+1]; offsets has n+1 non-decreasing entries
// (empty segments allowed).  Returns -1 if x is outside [offsets[0], offsets[n]).
__device__ __forceinline__ int find_segment(const int64_t* __restrict__ offsets, int64_t n, int64_t x) {
  if (x < offsets[0] || x >= offsets[n]) return -1;
  int64_t lo = 0, hi = n;  // invariant: offsets[lo] <= x < offsets[hi]
  while (hi - lo > 1) {
    int64_t mid = (lo + hi) >> 1;
    if (offsets[mid] <= x) lo = mid; else hi = mid;
  }
  return (int)lo;
}

// Sum `val` over runs of equal `seg` among the 32 lanes (runs are contiguous) and let the first
// lane of each run add it to out[seg * stride + col] (double atomics).  seg < 0: lane inactive.
__device__ __forceinline__ void warp_segmented_atomic_add(double* out, int seg, int64_t stride, int64_t col, float val,
                                                          int lane) {
  const unsigned full = 0xffffffffu;
  float v = seg >= 0 ? val : 0.f;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    float ov = __shfl_down_sync(full, v, d);
    int os = __shfl_down_sync(full, seg, d);
    if (lane + d < 32 && os == seg) v += ov;
  }
  int prev = __shfl_up_sync(full, seg, 1);
  bool head = (lane == 0) || (prev != seg);
  if (head && seg >= 0) atomicAdd(out + (int64_t)seg * stride + col, (double)v);
}
#endif

// kernels / launchers implemented in the .cu files ------------------------------------------
int launch_pack(const double* w, const double* mu, const double* var, const PackLayout& L, void* pack, cudaStream_t st);
int launch_score_simt(const float* feats, const int64_t* offsets, int64_t n_utts, int64_t total_frames, const void* pack,
                      const PackLayout& L, bool normalize, double* scores, float* frame_lse, cudaStream_t st);
// host-side note of which packs may be scored from their FP16 images (gmm_score_tc.cu): reset by every pack call, resolved by
// one read-back of the pack's overflow flag the first time the pack is scored in a single pass
void note_pack(const void* pack);
int launch_score_tc(const float* feats, const int64_t* offsets, int64_t n_utts, int64_t total_frames, const void* pack,
                    const PackLayout& L, int parts, bool normalize, double* scores, float* frame_lse, cudaStream_t st);
int launch_stats_tc(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames, const void* pack,
                    const PackLayout& L, float* frame_lse, double* out_n, double* out_f, double* out_s, double* out_loglik,
                    void* workspace, bool reuse_images, cudaStream_t st);
bool stats_tc_supported(const PackLayout& L);
int launch_pack_sv(const double* w, const double* var, const double* mu, const SvLayout& L, int ref_model, void* pack,
                   cudaStream_t st);
int64_t score_sv_workspace_bytes(const SvLayout& L, int64_t total_frames);
int launch_score_sv(const float* feats, const int64_t* offsets, int64_t n_utts, int64_t total_frames, const void* pack,
                    const SvLayout& L, bool normalize, double* scores, float* frame_lse, void* workspace, cudaStream_t st);
int64_t stats_tc_workspace_bytes(const PackLayout& L, int64_t total_frames, int64_t n_segs);
int launch_posteriors_tc(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames, const void* pack,
                         const PackLayout& L, float* out_resp, int64_t* out_label, float* out_frame_lse, void* workspace,
                         bool reuse_images, cudaStream_t st);
// workspace of the CUDA-core posterior path: per-segment sums of the scoring kernel, then the per-frame lse
inline int64_t posteriors_simt_lse_offset(int64_t n_segs) { return (8 * n_segs + 255) / 256 * 256; }
inline int64_t posteriors_simt_workspace_bytes(int64_t total_frames, int64_t n_segs) {
  return posteriors_simt_lse_offset(n_segs) + 4 * total_frames;
}
int launch_posteriors_simt(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                           const void* pack, const PackLayout& L, float* out_resp, int64_t* out_label, float* out_frame_lse,
                           void* workspace, cudaStream_t st);
int launch_stats_simt(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                      const void* pack, const PackLayout& L, const float* frame_lse, double* out_n, double* out_f,
                      double* out_s, cudaStream_t st);

}  // namespace ssp
