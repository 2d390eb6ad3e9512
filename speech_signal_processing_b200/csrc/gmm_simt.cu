// CUDA-core FP32 GMM kernels: exact scoring (SSP_PREC_FP32) and the posterior / N-F-S statistics
// pass used by UBM EM and MAP enrolment.  Same math as sklearn _gaussian_mixture.py:536-553 and
// _base.py:552-582, evaluated as sum_d x_d * (a1_d + a2_d * x_d) + cst with a1 = mu/var, a2 = -1/(2var).
#include "common.cuh"

namespace ssp {

// ------------------------------------------------------------------------------------------------
// Exact scoring.  grid = (ceil(frames/64), n_models), block = 128: thread = (frame f = tid%64, half h).
// Each half walks 16 of every 32 staged components; online (max, sum-exp) per thread, halves merged
// through shared memory; per-utterance mean via a warp-segmented double atomic.
// ------------------------------------------------------------------------------------------------
constexpr int kSF = 64;   // frames per block
constexpr int kSC = 32;   // components staged per step

template <int DP>
__global__ void __launch_bounds__(128) gmm_score_simt_kernel(const float* __restrict__ feats,
                                                            const int64_t* __restrict__ offsets, int64_t n_utts,
                                                            int64_t total_frames, const float2* __restrict__ ab,
                                                            const float* __restrict__ cst, int Kp, int D, int n_models,
                                                            int normalize, double* __restrict__ scores,
                                                            float* __restrict__ frame_lse) {
  __shared__ __align__(16) float2 s_ab[kSC * DP];
  __shared__ float s_c[kSC];
  __shared__ float s_m[kSF], s_s[kSF];
  const int tid = threadIdx.x, f = tid % kSF, h = tid / kSF;
  const int model = blockIdx.y;
  const int64_t frame = (int64_t)blockIdx.x * kSF + f;
  const bool valid = frame < total_frames;
  float x[DP];
#pragma unroll
  for (int d = 0; d < DP; ++d) x[d] = (valid && d < D) ? feats[frame * D + d] : 0.f;

  const float2* ab_m = ab + (int64_t)model * Kp * DP;
  const float* c_m = cst + (int64_t)model * Kp;
  float m_run = -3.0e38f, s_run = 0.f;
  for (int c0 = 0; c0 < Kp; c0 += kSC) {
    __syncthreads();
    for (int i = tid; i < kSC * DP; i += 128) s_ab[i] = ab_m[(int64_t)c0 * DP + i];
    if (tid < kSC) s_c[tid] = c_m[c0 + tid];
    __syncthreads();
    float l[kSC / 2];
    float cmax = -3.0e38f;
#pragma unroll
    for (int j = 0; j < kSC / 2; ++j) {
      const int c = h * (kSC / 2) + j;
      const float4* row = reinterpret_cast<const float4*>(s_ab + c * DP);
      float acc0 = s_c[c], acc1 = 0.f;
#pragma unroll
      for (int d = 0; d < DP; d += 2) {
        float4 p = row[d >> 1];  // (a1[d], a2[d], a1[d+1], a2[d+1])
        acc0 = fmaf(x[d], fmaf(p.y, x[d], p.x), acc0);
        acc1 = fmaf(x[d + 1], fmaf(p.w, x[d + 1], p.z), acc1);
      }
      l[j] = acc0 + acc1;
      cmax = fmaxf(cmax, l[j]);
    }
    const float m_new = fmaxf(m_run, cmax);
    float add = 0.f;
#pragma unroll
    for (int j = 0; j < kSC / 2; ++j) add += expf(l[j] - m_new);
    s_run = s_run * expf(m_run - m_new) + add;
    m_run = m_new;
  }
  if (h == 1) { s_m[f] = m_run; s_s[f] = s_run; }
  __syncthreads();
  if (h == 0) {
    const float m2 = s_m[f], s2 = s_s[f];
    const float m_new = fmaxf(m_run, m2);
    const float s_tot = s_run * expf(m_run - m_new) + s2 * expf(m2 - m_new);
    const float lse = m_new + logf(s_tot);
    if (valid && frame_lse) frame_lse[(int64_t)model * total_frames + frame] = lse;
    int u = valid ? find_segment(offsets, n_utts, frame) : -1;
    float wgt = 1.f;
    if (u >= 0 && normalize) wgt = 1.f / (float)(offsets[u + 1] - offsets[u]);
    warp_segmented_atomic_add(scores, u, n_models, model, lse * wgt, tid & 31);
  }
}

int launch_score_simt(const float* feats, const int64_t* offsets, int64_t n_utts, int64_t total_frames, const void* pack,
                      const PackLayout& L, bool normalize, double* scores, float* frame_lse, cudaStream_t st) {
  const char* base = (const char*)pack;
  const float2* ab = (const float2*)(base + L.off_ab);
  const float* cst = (const float*)(base + L.off_cst);
  SSP_CUDA_OK(cudaMemsetAsync(scores, 0, sizeof(double) * n_utts * L.n_models, st));
  if (total_frames == 0) return SSP_OK;
  dim3 grid((unsigned)((total_frames + kSF - 1) / kSF), (unsigned)L.n_models);
  SSP_REQUIRE(L.n_models <= 65535, "ssp_gmm_score(fp32): n_models %d > 65535", L.n_models);
#define SSP_CASE(dp)                                                                                               \
  case dp:                                                                                                         \
    gmm_score_simt_kernel<dp><<<grid, 128, 0, st>>>(feats, offsets, n_utts, total_frames, ab, cst, L.Kp, L.D,     \
                                                     L.n_models, normalize ? 1 : 0, scores, frame_lse);            \
    break;
  switch (L.DP) {
    SSP_CASE(16) SSP_CASE(32) SSP_CASE(40) SSP_CASE(64) SSP_CASE(80)
    default: SSP_REQUIRE(false, "unsupported padded feature dim %d", L.DP);
  }
#undef SSP_CASE
  SSP_LAUNCH_CHECK("gmm_score_simt_kernel");
  return SSP_OK;
}

// ------------------------------------------------------------------------------------------------
// Posteriors (D > 39, one model).  Same block shape and logit arithmetic as gmm_score_simt_kernel, whose per-frame lse
// this pass consumes: gamma[t, c] = exp(L[t, c] - lse_t) is staged per 32 components in shared memory and written as
// rows of 32 consecutive components (one 128-byte row segment per warp store); the label is the lowest component index
// reaching the maximum logit.
// ------------------------------------------------------------------------------------------------
template <int DP>
__global__ void __launch_bounds__(128) gmm_post_simt_kernel(const float* __restrict__ feats, int64_t total_frames,
                                                           const float2* __restrict__ ab, const float* __restrict__ cst,
                                                           int K, int Kp, int D, const float* __restrict__ frame_lse,
                                                           float* __restrict__ out_resp, int64_t* __restrict__ out_label) {
  __shared__ __align__(16) float2 s_ab[kSC * DP];
  __shared__ float s_c[kSC];
  __shared__ float s_g[kSF * (kSC + 1)];
  __shared__ float s_m[kSF];
  __shared__ int s_i[kSF];
  const int tid = threadIdx.x, f = tid % kSF, h = tid / kSF;
  const int64_t f0 = (int64_t)blockIdx.x * kSF, frame = f0 + f;
  const bool valid = frame < total_frames;
  float x[DP];
#pragma unroll
  for (int d = 0; d < DP; ++d) x[d] = (valid && d < D) ? feats[frame * D + d] : 0.f;
  const float lse = (valid && out_resp) ? frame_lse[frame] : 0.f;
  float bm = -3.0e38f;
  int bi = 0;
  for (int c0 = 0; c0 < Kp; c0 += kSC) {
    __syncthreads();
    for (int i = tid; i < kSC * DP; i += 128) s_ab[i] = ab[(int64_t)c0 * DP + i];
    if (tid < kSC) s_c[tid] = cst[c0 + tid];
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < kSC / 2; ++j) {
      const int c = h * (kSC / 2) + j;
      const float4* row = reinterpret_cast<const float4*>(s_ab + c * DP);
      float acc0 = s_c[c], acc1 = 0.f;
#pragma unroll
      for (int d = 0; d < DP; d += 2) {
        float4 p = row[d >> 1];
        acc0 = fmaf(x[d], fmaf(p.y, x[d], p.x), acc0);
        acc1 = fmaf(x[d + 1], fmaf(p.w, x[d + 1], p.z), acc1);
      }
      const float l = acc0 + acc1;
      if (c0 + c < K && l > bm) { bm = l; bi = c0 + c; }
      if (out_resp) s_g[f * (kSC + 1) + c] = expf(l - lse);
    }
    if (out_resp) {
      __syncthreads();
      // warp w writes rows w, w + 4, ...: 32 lanes = 32 consecutive components of one frame
      const int lane = tid & 31;
      for (int r = tid >> 5; r < kSF; r += 4)
        if (f0 + r < total_frames && c0 + lane < K) __stcs(out_resp + (f0 + r) * K + c0 + lane, s_g[r * (kSC + 1) + lane]);
    }
  }
  if (out_label) {
    // half 0 holds components [c0, c0 + 16) of every chunk, half 1 [c0 + 16, c0 + 32): on a tie the lower index wins
    if (h == 1) { s_m[f] = bm; s_i[f] = bi; }
    __syncthreads();
    if (h == 0 && valid) {
      const float m1 = s_m[f];
      const int i1 = s_i[f];
      out_label[frame] = (m1 > bm || (m1 == bm && i1 < bi)) ? i1 : bi;
    }
  }
}

int launch_posteriors_simt(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                           const void* pack, const PackLayout& L, float* out_resp, int64_t* out_label, float* out_frame_lse,
                           void* workspace, cudaStream_t st) {
  if (total_frames == 0) return SSP_OK;
  const char* base = (const char*)pack;
  const float2* ab = (const float2*)(base + L.off_ab);
  const float* cst = (const float*)(base + L.off_cst);
  // workspace: per-segment sums of gmm_score_simt_kernel (unused), then the per-frame lse unless the caller takes it
  double* seg_sums = (double*)workspace;
  float* lse = out_frame_lse ? out_frame_lse : (float*)((char*)workspace + posteriors_simt_lse_offset(n_segs));
  if (out_resp || out_frame_lse) {
    const int rc = launch_score_simt(feats, seg_offsets, n_segs, total_frames, pack, L, false, seg_sums, lse, st);
    if (rc != SSP_OK) return rc;
  }
  if (!out_resp && !out_label) return SSP_OK;
  const unsigned grid = (unsigned)((total_frames + kSF - 1) / kSF);
#define SSP_CASE(dp)                                                                                                   \
  case dp:                                                                                                             \
    gmm_post_simt_kernel<dp><<<grid, 128, 0, st>>>(feats, total_frames, ab, cst, L.K, L.Kp, L.D, lse, out_resp, out_label); \
    break;
  switch (L.DP) {  // the tensor-core pass serves D <= 39
    SSP_CASE(40) SSP_CASE(64) SSP_CASE(80)
    default: SSP_REQUIRE(false, "unsupported padded feature dim %d", L.DP);
  }
#undef SSP_CASE
  SSP_LAUNCH_CHECK("gmm_post_simt_kernel");
  return SSP_OK;
}

// ------------------------------------------------------------------------------------------------
// Statistics pass.  grid = (frame chunks, component groups of 64), block = 256.
//   phase A: thread = (frame t = tid%64, quarter q): gamma[t, c] = exp(L[t,c] - lse_t) for 16 components
//   phase B: thread = (component c = tid%64, quarter q): F/S accumulators for DP/4 dims (+N on q == 0)
// FP32 accumulators are folded into double registers every 16 tiles; one double atomic per output at
// segment / chunk end.  Tiles never straddle a segment boundary.
// ------------------------------------------------------------------------------------------------
constexpr int kTF = 64;  // frames per tile
constexpr int kTG = 64;  // components per group

template <int DP>
struct StatsSmem {
  static constexpr int DPB = (DP + 15) / 16 * 16;  // phase-B row stride: quarters of DPB/4 dims stay 16-byte aligned
  float2 ab[kTG * DP];
  float cst[kTG];
  float xs[kTF * DPB];        // row-major tile of frames (phase B broadcast reads)
  float xt[DP * (kTF + 1)];   // transposed copy (phase A, conflict-free per-frame reads)
  float g[kTG * (kTF + 1)];   // gamma[c][t]
  float lse[kTF];
};

template <int DP>
__global__ void __launch_bounds__(256) gmm_stats_simt_kernel(const float* __restrict__ feats,
                                                            const int64_t* __restrict__ seg, int64_t n_segs,
                                                            int64_t total_frames, int64_t chunk,
                                                            const float2* __restrict__ ab, const float* __restrict__ cst,
                                                            int K, int D, const float* __restrict__ frame_lse,
                                                            double* __restrict__ out_n, double* __restrict__ out_f,
                                                            double* __restrict__ out_s) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  StatsSmem<DP>& sm = *reinterpret_cast<StatsSmem<DP>*>(smem_raw);
  constexpr int DPB = StatsSmem<DP>::DPB;
  constexpr int DQ = DPB / 4;  // multiple of 4
  const int tid = threadIdx.x;
  const int c0 = blockIdx.y * kTG;
  const int64_t begin = (int64_t)blockIdx.x * chunk;
  const int64_t end = min(begin + chunk, total_frames);
  if (begin >= end) return;

  for (int i = tid; i < kTG * DP; i += 256) sm.ab[i] = ab[(int64_t)c0 * DP + i];
  if (tid < kTG) sm.cst[tid] = cst[c0 + tid];

  // phase A / B identities
  const int a_t = tid % kTF, a_q = tid / kTF;
  const int b_c = tid % kTG, b_q = tid / kTG;
  float accF[DQ], accS[DQ], accN = 0.f;
  double dF[DQ], dS[DQ], dN = 0.0;
#pragma unroll
  for (int j = 0; j < DQ; ++j) { accF[j] = accS[j] = 0.f; dF[j] = dS[j] = 0.0; }

  int cur_seg = find_segment(seg, n_segs, begin);
  int64_t seg_end = cur_seg >= 0 ? seg[cur_seg + 1] : begin;
  int tiles_since_fold = 0;

  auto fold = [&]() {
#pragma unroll
    for (int j = 0; j < DQ; ++j) { dF[j] += accF[j]; dS[j] += accS[j]; accF[j] = accS[j] = 0.f; }
    dN += accN; accN = 0.f;
    tiles_since_fold = 0;
  };
  auto flush = [&](int s) {
    fold();
    const int c = c0 + b_c;
    if (s >= 0 && c < K) {
      if (b_q == 0) atomicAdd(out_n + (int64_t)s * K + c, dN);
#pragma unroll
      for (int j = 0; j < DQ; ++j) {
        const int d = b_q * DQ + j;
        if (d < D) {
          atomicAdd(out_f + ((int64_t)s * K + c) * D + d, dF[j]);
          atomicAdd(out_s + ((int64_t)s * K + c) * D + d, dS[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < DQ; ++j) dF[j] = dS[j] = 0.0;
    dN = 0.0;
  };

  int64_t t0 = begin;
  while (t0 < end) {
    if (cur_seg < 0 || t0 >= seg_end) {  // advance to the segment containing t0 (skips empty segments)
      flush(cur_seg);
      cur_seg = find_segment(seg, n_segs, t0);
      if (cur_seg < 0) break;
      seg_end = seg[cur_seg + 1];
    }
    const int nt = (int)min((int64_t)kTF, min(end, seg_end) - t0);
    __syncthreads();  // previous tile's phase B done (and parameter staging on the first trip)
    // stage the tile: coalesced read of nt*D contiguous floats, two shared copies
    for (int i = tid; i < kTF * DPB; i += 256) {
      const int t = i / DPB, d = i % DPB;
      float v = (t < nt && d < D) ? feats[(t0 + t) * D + d] : 0.f;
      sm.xs[i] = v;
      if (d < DP) sm.xt[d * (kTF + 1) + t] = v;
    }
    if (tid < kTF) sm.lse[tid] = tid < nt ? frame_lse[t0 + tid] : 0.f;
    __syncthreads();
    // ---- phase A
    {
      float x[DP];
#pragma unroll
      for (int d = 0; d < DP; ++d) x[d] = sm.xt[d * (kTF + 1) + a_t];
      const float lse = sm.lse[a_t];
      const bool live = a_t < nt;
#pragma unroll 4
      for (int j = 0; j < kTG / 4; ++j) {
        const int c = a_q * (kTG / 4) + j;
        const float4* row = reinterpret_cast<const float4*>(sm.ab + c * DP);
        float acc0 = sm.cst[c], acc1 = 0.f;
#pragma unroll
        for (int d = 0; d < DP; d += 2) {
          float4 p = row[d >> 1];
          acc0 = fmaf(x[d], fmaf(p.y, x[d], p.x), acc0);
          acc1 = fmaf(x[d + 1], fmaf(p.w, x[d + 1], p.z), acc1);
        }
        sm.g[c * (kTF + 1) + a_t] = live ? expf(acc0 + acc1 - lse) : 0.f;
      }
    }
    __syncthreads();
    // ---- phase B
    {
      const float* grow = sm.g + b_c * (kTF + 1);
      for (int t = 0; t < nt; ++t) {
        const float g = grow[t];
        const float4* xr = reinterpret_cast<const float4*>(sm.xs + t * DPB + b_q * DQ);
        accN += g;
#pragma unroll
        for (int j4 = 0; j4 < DQ / 4; ++j4) {
          float4 xv = xr[j4];
          float gx;
          gx = g * xv.x; accF[4 * j4 + 0] += gx; accS[4 * j4 + 0] = fmaf(gx, xv.x, accS[4 * j4 + 0]);
          gx = g * xv.y; accF[4 * j4 + 1] += gx; accS[4 * j4 + 1] = fmaf(gx, xv.y, accS[4 * j4 + 1]);
          gx = g * xv.z; accF[4 * j4 + 2] += gx; accS[4 * j4 + 2] = fmaf(gx, xv.z, accS[4 * j4 + 2]);
          gx = g * xv.w; accF[4 * j4 + 3] += gx; accS[4 * j4 + 3] = fmaf(gx, xv.w, accS[4 * j4 + 3]);
        }
      }
    }
    if (++tiles_since_fold >= 16) fold();
    t0 += nt;
  }
  flush(cur_seg);
}

int launch_stats_simt(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                      const void* pack, const PackLayout& L, const float* frame_lse, double* out_n, double* out_f,
                      double* out_s, cudaStream_t st) {
  if (total_frames == 0) return SSP_OK;
  const char* base = (const char*)pack;
  const float2* ab = (const float2*)(base + L.off_ab);
  const float* cst = (const float*)(base + L.off_cst);
  const int groups = L.Kp / kTG;
  // chunk: aim for ~8 CTAs per SM over the whole grid, at least one tile, at most 64 Ki frames
  int64_t want_ctas = 148 * 8;
  int64_t chunks = (want_ctas + groups - 1) / groups;
  int64_t chunk = (total_frames + chunks - 1) / chunks;
  chunk = (chunk + kTF - 1) / kTF * kTF;
  if (chunk < 4 * kTF) chunk = 4 * kTF;
  if (chunk > 65536) chunk = 65536;
  dim3 grid((unsigned)((total_frames + chunk - 1) / chunk), (unsigned)groups);
#define SSP_CASE(dp)                                                                                                  \
  case dp: {                                                                                                          \
    size_t smem = sizeof(StatsSmem<dp>);                                                                              \
    SSP_CUDA_OK(cudaFuncSetAttribute(gmm_stats_simt_kernel<dp>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    gmm_stats_simt_kernel<dp><<<grid, 256, smem, st>>>(feats, seg_offsets, n_segs, total_frames, chunk, ab, cst, L.K,  \
                                                        L.D, frame_lse, out_n, out_f, out_s);                         \
  } break;
  switch (L.DP) {
    SSP_CASE(16) SSP_CASE(32) SSP_CASE(40) SSP_CASE(64) SSP_CASE(80)
    default: SSP_REQUIRE(false, "unsupported padded feature dim %d", L.DP);
  }
#undef SSP_CASE
  SSP_LAUNCH_CHECK("gmm_stats_simt_kernel");
  return SSP_OK;
}

}  // namespace ssp
