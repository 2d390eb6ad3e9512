// Model packing, M-step and MAP adaptation: small double-precision kernels that keep the whole
// EM / enrolment loop resident in HBM (no host round trip of parameters between iterations).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace ssp {

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// One thread per (model, padded component).  Follows sklearn/mixture/_gaussian_mixture.py:536-553:
//   L[t,c] = log w_c - 0.5 (D log 2pi + sum_d (mu^2 p - 2 x mu p + x^2 p)) + 0.5 sum_d log p,  p = 1/var
// which is the contraction [x, x^2, 1] . [mu p, -p/2, cst_c].
__global__ void gmm_pack_kernel(const double* __restrict__ w, const double* __restrict__ mu,
                                const double* __restrict__ var, int n_models, int K, int Kp, int D, int DP, int KD,
                                float2* __restrict__ ab, float* __restrict__ cst, float* __restrict__ tiles,
                                float* __restrict__ tiles_lo, __nv_bfloat16* __restrict__ tiles_bf, int KDb,
                                __half* __restrict__ tiles_h, __half* __restrict__ tiles_hl, int* __restrict__ h_overflow) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n_models * Kp) return;
  int m = (int)(idx / Kp), c = (int)(idx % Kp);
  float2* ab_row = ab + idx * DP;
  // tile image: [KD/4][128] float4, element (kc, n) holds row n, columns 4kc..4kc+3
  float* tile = tiles + ((int64_t)m * (Kp / kTileN) + c / kTileN) * (int64_t)kTileN * KD;
  const int n = c % kTileN;
  auto tile_at = [&](int j) -> float& { return tile[((j >> 2) * kTileN + n) * 4 + (j & 3)]; };
  // residual image (same layout): B = hi + lo to ~2^-22, used by the 3xTF32 EM kernels
  float* tlo = tiles_lo ? tiles_lo + ((int64_t)m * (Kp / kTileN) + c / kTileN) * (int64_t)kTileN * KD : nullptr;
  auto lo_at = [&](int j) -> float& { return tlo[((j >> 2) * kTileN + n) * 4 + (j & 3)]; };
  // BF16 image of the tile (EM kernels): [hi | lo][KDb/8][128][8], element (part, j, n) at ((part*KDb/8 + j/8)*128 + n)*8 + j%8
  __nv_bfloat16* tbf = tiles_bf ? tiles_bf + ((int64_t)m * (Kp / kTileN) + c / kTileN) * 2 * kTileN * KDb : nullptr;
  auto bf_at = [&](int part, int j) -> __nv_bfloat16& {
    return tbf[(((int64_t)part * (KDb >> 3) + (j >> 3)) * kTileN + n) * 8 + (j & 7)];
  };
  auto bf_split = [&](int j, double v) {
    const __nv_bfloat16 h = __float2bfloat16_rn((float)v);
    bf_at(0, j) = h;
    bf_at(1, j) = __float2bfloat16_rn((float)(v - (double)__bfloat162float(h)));
  };
  if (tbf)
    for (int j = 0; j < KDb; ++j) { bf_at(0, j) = __float2bfloat16_rn(0.f); bf_at(1, j) = __float2bfloat16_rn(0.f); }
  // FP16 image of the tile (single-pass scoring rung): element (j, n) at ((j/8)*128 + n)*8 + j%8
  __half* th = tiles_h ? tiles_h + ((int64_t)m * (Kp / kTileN) + c / kTileN) * (int64_t)kTileN * KDb : nullptr;
  bool h_bad = false;
  __half* thl = tiles_hl ? tiles_hl + ((int64_t)m * (Kp / kTileN) + c / kTileN) * (int64_t)kTileN * KDb : nullptr;
  auto h_put = [&](int j, double v, bool with_residual = true) {   // hi image: fp16(v); residual image: fp16(v - hi); returns hi
    const __half h = __float2half_rn((float)v);
    if (!(fabs((double)__half2float(h)) <= 65504.0)) h_bad = true;
    const int64_t at = (((int64_t)(j >> 3)) * kTileN + n) * 8 + (j & 7);
    th[at] = h;
    if (thl && with_residual) thl[at] = __float2half_rn((float)(v - (double)__half2float(h)));
    return (double)__half2float(h);
  };
  if (th)
    for (int j = 0; j < KDb; ++j) {
      th[(((int64_t)(j >> 3)) * kTileN + n) * 8 + (j & 7)] = __float2half_rn(0.f);
      if (thl) thl[(((int64_t)(j >> 3)) * kTileN + n) * 8 + (j & 7)] = __float2half_rn(0.f);
    }
  const double LOG2E = 1.4426950408889634074;
  if (c >= K) {
    if (th) h_put(2 * D, -60000.0, false);  // 2^-60000 == 0: padded components never contribute
    if (tbf) bf_at(0, 2 * D) = __float2bfloat16_rn(-1e30f);
    for (int d = 0; d < DP; ++d) ab_row[d] = make_float2(0.f, 0.f);
    cst[idx] = -1e30f;
    for (int j = 0; j < KD; ++j) tile_at(j) = 0.f;
    tile_at(2 * D) = to_tf32(-1e30f);
    if (tlo)
      for (int j = 0; j < KD; ++j) lo_at(j) = 0.f;
    return;
  }
  const double* mu_r = mu + ((int64_t)m * K + c) * D;
  const double* var_r = var + ((int64_t)m * K + c) * D;
  double quad = 0.0, logdet = 0.0;
  for (int d = 0; d < D; ++d) {
    double p = 1.0 / var_r[d];
    double a1 = mu_r[d] * p, a2 = -0.5 * p;
    quad += mu_r[d] * mu_r[d] * p;
    logdet += log(p);
    ab_row[d] = make_float2((float)a1, (float)a2);
    const float h1 = to_tf32((float)(a1 * LOG2E)), h2 = to_tf32((float)(a2 * LOG2E));
    tile_at(d) = h1;
    tile_at(D + d) = h2;
    if (tlo) {
      lo_at(d) = to_tf32((float)(a1 * LOG2E - (double)h1));
      lo_at(D + d) = to_tf32((float)(a2 * LOG2E - (double)h2));
    }
    if (tbf) {
      bf_split(d, a1 * LOG2E);
      bf_split(D + d, a2 * LOG2E);
    }
    if (th) {
      h_put(d, a1 * LOG2E);
      h_put(D + d, a2 * LOG2E);
    }
  }
  for (int d = D; d < DP; ++d) ab_row[d] = make_float2(0.f, 0.f);
  double cc = log(w[(int64_t)m * K + c]) - 0.5 * (D * 1.8378770664093454836 + quad) + 0.5 * logdet;
  if (!(cc > -1e30)) cc = -1e30;  // w == 0 -> log w = -inf; keep finite so exp() underflows cleanly
  cst[idx] = (float)cc;
  // the constant goes through the TF32 MMA as two exactly-representable pieces times A columns of 1.0
  double c2 = cc * LOG2E;
  float hi = to_tf32((float)c2);
  float lo = to_tf32((float)(c2 - (double)hi));
  tile_at(2 * D) = hi;
  tile_at(2 * D + 1) = lo;
  for (int j = 2 * D + 2; j < KD; ++j) tile_at(j) = 0.f;
  if (tlo) {
    lo_at(2 * D) = to_tf32((float)(c2 - (double)hi - (double)lo));  // third piece of the constant
    for (int j = 2 * D + 1; j < KD; ++j) lo_at(j) = 0.f;
  }
  if (th) {  // two FP16 pieces of the constant against the two "one" columns
    const double ch = c2 > -60000.0 ? c2 : -60000.0;   // (zero-weight components)
    // the constant as three FP16 pieces: two in the hi image (so that the single-pass rung has it to ~2^-22), the third in
    // the residual image
    const double c1 = h_put(2 * D, ch, false);
    const double c2 = h_put(2 * D + 1, ch - c1, false);
    if (thl) thl[(((int64_t)((2 * D) >> 3)) * kTileN + n) * 8 + ((2 * D) & 7)] = __float2half_rn((float)(ch - c1 - c2));
    if (h_bad) *h_overflow = 1;
  }
  if (tbf) {  // three BF16 pieces of the constant (24 bits) against the two "one" columns of the frame operand
    const __nv_bfloat16 p1 = __float2bfloat16_rn((float)c2);
    const double r1 = c2 - (double)__bfloat162float(p1);
    const __nv_bfloat16 p2 = __float2bfloat16_rn((float)r1);
    bf_at(0, 2 * D) = p1;
    bf_at(0, 2 * D + 1) = p2;
    bf_at(1, 2 * D) = __float2bfloat16_rn((float)(r1 - (double)__bfloat162float(p2)));
  }
}

int launch_pack(const double* w, const double* mu, const double* var, const PackLayout& L, void* pack, cudaStream_t st) {
  char* base = (char*)pack;
  int64_t n = (int64_t)L.n_models * L.Kp;
  int threads = 128;
  int64_t blocks = (n + threads - 1) / threads;
  if (L.off_flag) SSP_CUDA_OK(cudaMemsetAsync(base + L.off_flag, 0, 128, st));
  gmm_pack_kernel<<<(unsigned)blocks, threads, 0, st>>>(w, mu, var, L.n_models, L.K, L.Kp, L.D, L.DP, L.KD,
                                                       (float2*)(base + L.off_ab), (float*)(base + L.off_cst),
                                                       (float*)(base + L.off_tile),
                                                       L.off_tile_lo ? (float*)(base + L.off_tile_lo) : nullptr,
                                                       L.off_tile_bf ? (__nv_bfloat16*)(base + L.off_tile_bf) : nullptr, L.KDb(),
                                                       L.off_tile_h ? (__half*)(base + L.off_tile_h) : nullptr,
                                                       L.off_tile_hl ? (__half*)(base + L.off_tile_hl) : nullptr,
                                                       L.off_flag ? (int*)(base + L.off_flag) : nullptr);
  note_pack(pack);
  SSP_LAUNCH_CHECK("gmm_pack_kernel");
  return SSP_OK;
}

// Shared-variance pack (SvLayout, common.cuh): one thread per (image, padded component), FP16 images.  The common part
// (images 0..3) is the full logit of the reference member as hi + lo FP16 pieces; image kSvBaseImages + s holds model s
// as its DIFFERENCE from the reference, so rounding acts on (mu_s - mu_ref) / var -- an order of magnitude smaller than
// mu_s / var for MAP-adapted speakers -- and the reference model's own image is exactly zero.
__global__ void gmm_pack_sv_kernel(const double* __restrict__ w, const double* __restrict__ var, const double* __restrict__ mu,
                                   int S, int K, int Kp, int D, int KS, int KQ, int ref, __half* __restrict__ tiles,
                                   int* __restrict__ overflow) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int n_images = S + kSvBaseImages;
  if (idx >= (int64_t)n_images * Kp) return;
  const int image = (int)(idx / Kp), c = (int)(idx % Kp);
  const int n = c % kSvTileN;
  __half* tile = tiles + ((int64_t)(c / kSvTileN) * n_images + image) * (int64_t)kSvTileN * KS;
  auto tile_at = [&](int j) -> __half& { return tile[((j >> 3) * kSvTileN + n) * 8 + (j & 7)]; };
  for (int j = 0; j < KS; ++j) tile_at(j) = __float2half_rn(0.f);
  const double LOG2E = 1.4426950408889634074;
  const double kFloor = -60000.0;  // FP16-exact; 2^-60000 == 0: padded or zero-weight components never contribute
  bool bad = false;
  auto put = [&](int j, double v, int piece) {  // piece 0, 1, 2 of v as FP16 values (v ~ p0 + p1 + p2)
    const __half p0 = __float2half_rn((float)v);
    const double r1 = v - (double)__half2float(p0);
    const __half p1 = __float2half_rn((float)r1);
    const __half pc = piece == 0 ? p0 : piece == 1 ? p1 : __float2half_rn((float)(r1 - (double)__half2float(p1)));
    if (!(fabs((double)__half2float(p0)) <= 65504.0)) bad = true;
    tile_at(j) = pc;
  };
  if (image < kSvBaseImages) {
    // column range [j0, j1) of the common contraction [x^2 (D) | x (D) | 1, 1 | 0..] and which piece
    const int j0 = (image & 1) ? KS : 0, j1 = (image & 1) ? KQ : KS, lo = image >> 1;
    if (c >= K) {
      if (!lo && 2 * D >= j0 && 2 * D < j1) tile_at(2 * D - j0) = __float2half_rn((float)kFloor);
      return;
    }
    const double* var_r = var + (int64_t)c * D;
    const double* ref_r = mu + ((int64_t)ref * K + c) * D;
    double logdet = 0.0, quad = 0.0;
    for (int d = 0; d < D; ++d) {
      const double p = 1.0 / var_r[d];
      logdet += log(p);
      quad += ref_r[d] * ref_r[d] * p;
      if (d >= j0 && d < j1) put(d - j0, -0.5 * p * LOG2E, lo);
      if (D + d >= j0 && D + d < j1) put(D + d - j0, ref_r[d] * p * LOG2E, lo);
    }
    // log w - D/2 log 2pi - 1/2 sum log var - 1/2 sum mu_ref^2 / var, as three FP16 pieces against the two columns of 1.0
    double cc = (log(w[c]) - 0.5 * D * 1.8378770664093454836 + 0.5 * logdet - 0.5 * quad) * LOG2E;
    if (!(cc > kFloor)) cc = kFloor;  // w == 0
    if (2 * D >= j0 && 2 * D < j1) put(2 * D - j0, cc, lo ? 2 : 0);
    if (!lo && 2 * D + 1 >= j0 && 2 * D + 1 < j1) put(2 * D + 1 - j0, cc, 1);
  } else if (c < K) {  // [x, 1, 1] . log2(e) [(mu_s - mu_ref) / var, ck_s - ck_ref as two pieces]
    const double* var_r = var + (int64_t)c * D;
    const double* ref_r = mu + ((int64_t)ref * K + c) * D;
    const double* mu_r = mu + ((int64_t)(image - kSvBaseImages) * K + c) * D;
    double dquad = 0.0;
    for (int d = 0; d < D; ++d) {
      const double p = 1.0 / var_r[d], dm = mu_r[d] - ref_r[d];
      dquad += dm * (mu_r[d] + ref_r[d]) * p;
      put(d, dm * p * LOG2E, 0);
    }
    // the constant against the frame operand's columns [1, 1024]: cb * 1024 + ca, so that a model far from the
    // reference (|constant| up to 6.7e7; its scores go through sv_fixup_kernel) stays inside FP16's range
    const double cd = -0.5 * dquad * LOG2E;
    const __half cb = __float2half_rn((float)(cd / kSvConstScale));
    const __half ca = __float2half_rn((float)(cd - kSvConstScale * (double)__half2float(cb)));
    if (!(fabs((double)__half2float(cb)) <= 65504.0)) bad = true;
    tile_at(D) = ca;
    tile_at(D + 1) = cb;
  }
  if (bad) *overflow = 1;
}

int launch_pack_sv(const double* w, const double* var, const double* mu, const SvLayout& L, int ref_model, void* pack,
                   cudaStream_t st) {
  const int64_t n = (int64_t)(L.n_models + kSvBaseImages) * L.Kp;
  const int threads = 128;
  int* flag = (int*)((char*)pack + L.flag_offset);
  SSP_CUDA_OK(cudaMemsetAsync(flag, 0, 128, st));
  gmm_pack_sv_kernel<<<(unsigned)((n + threads - 1) / threads), threads, 0, st>>>(w, var, mu, L.n_models, L.K, L.Kp, L.D, L.KS,
                                                                              L.KQ, ref_model, (__half*)pack, flag);
  SSP_LAUNCH_CHECK("gmm_pack_sv_kernel");
  // packing is rare (once per model set): one read-back tells the caller that the set does not fit FP16
  int h_flag = 0;
  SSP_CUDA_OK(cudaMemcpyAsync(&h_flag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  SSP_CUDA_OK(cudaStreamSynchronize(st));
  if (h_flag) {
    set_error("ssp_gmm_pack_shared: a model parameter leaves the FP16 range of the shared-variance kernel (|value| > 65504: "
              "means / variances far from normalised features); score the set with ssp_gmm_score instead");
    return SSP_EUNSUP;
  }
  return SSP_OK;
}

// ------------------------------------------------------------------------------------------ M-step
// sklearn _gaussian_mixture.py:312-313 (nk = resp.sum + 10 eps), :250-252 (diag covariance),
// :898 (weights /= weights.sum()).  One block; K*D is small.
__global__ void gmm_mstep_kernel(const double* __restrict__ n, const double* __restrict__ f, const double* __restrict__ s,
                                 int K, int D, double reg_covar, double nk_eps, double* __restrict__ ow,
                                 double* __restrict__ omu, double* __restrict__ ovar) {
  __shared__ double red[32];
  __shared__ double total_s;
  // one block per model (statistics and parameters of model m at offset m * K (* D))
  n += (int64_t)blockIdx.x * K; ow += (int64_t)blockIdx.x * K;
  f += (int64_t)blockIdx.x * K * D; s += (int64_t)blockIdx.x * K * D;
  omu += (int64_t)blockIdx.x * K * D; ovar += (int64_t)blockIdx.x * K * D;
  double part = 0.0;
  for (int c = threadIdx.x; c < K; c += blockDim.x) part += n[c] + nk_eps;
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (blockDim.x + 31) / 32; ++i) t += red[i];
    total_s = t;
  }
  __syncthreads();
  const double total = total_s;
  for (int c = threadIdx.x; c < K; c += blockDim.x) ow[c] = (n[c] + nk_eps) / total;
  for (int i = threadIdx.x; i < K * D; i += blockDim.x) {
    double nk = n[i / D] + nk_eps;
    double m = f[i] / nk;
    omu[i] = m;
    ovar[i] = s[i] / nk - m * m + reg_covar;
  }
}

// ------------------------------------------------------------------------------------------ MAP
// Reynolds, Quatieri, Dunn (2000) eq. 11-14.  One block per speaker.  A speaker or component without data keeps the
// UBM's parameters: alpha = 0 when n = 0 (also at relevance 0, where n / (n + r) would be 0 / 0), and the weight term
// alpha n / T is 0 for a speaker of T = 0 frames.
__global__ void gmm_map_kernel(const double* __restrict__ n, const double* __restrict__ f, const double* __restrict__ s,
                               const int64_t* __restrict__ seg, const double* __restrict__ uw,
                               const double* __restrict__ umu, const double* __restrict__ uvar, int K, int D,
                               double relevance, int flags, double* __restrict__ ow, double* __restrict__ omu,
                               double* __restrict__ ovar) {
  const int spk = blockIdx.x;
  const double* n_s = n + (int64_t)spk * K;
  const double* f_s = f + (int64_t)spk * K * D;
  const double* s_s = s + (int64_t)spk * K * D;
  __shared__ double red[32];
  __shared__ double total_s;
  if (ow) {
    const double T = (double)(seg[spk + 1] - seg[spk]);
    double part = 0.0;
    for (int c = threadIdx.x; c < K; c += blockDim.x) {
      double a = n_s[c] > 0.0 ? n_s[c] / (n_s[c] + relevance) : 0.0;
      const double wn = T > 0.0 ? a * n_s[c] / T : 0.0;
      double v = (flags & 2) ? wn + (1.0 - a) * uw[c] : uw[c];
      ow[(int64_t)spk * K + c] = v;
      part += v;
    }
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < (blockDim.x + 31) / 32; ++i) t += red[i];
      total_s = t;
    }
    __syncthreads();
    if (flags & 2)
      for (int c = threadIdx.x; c < K; c += blockDim.x) ow[(int64_t)spk * K + c] /= total_s;
  }
  for (int i = threadIdx.x; i < K * D; i += blockDim.x) {
    int c = i / D;
    double nc = n_s[c];
    double a = nc > 0.0 ? nc / (nc + relevance) : 0.0;
    double safe = nc > 1e-300 ? nc : 1e-300;
    double m_new = (flags & 1) ? a * (f_s[i] / safe) + (1.0 - a) * umu[i] : umu[i];
    if (omu) omu[(int64_t)spk * K * D + i] = m_new;
    if (ovar) {
      double v = uvar[i];
      if (flags & 4) v = a * (s_s[i] / safe) + (1.0 - a) * (uvar[i] + umu[i] * umu[i]) - m_new * m_new;
      ovar[(int64_t)spk * K * D + i] = v;
    }
  }
}

}  // namespace ssp

extern "C" int ssp_gmm_mstep(const double* n, const double* f, const double* s, int32_t n_models, int32_t n_comp, int32_t n_feat,
                             double reg_covar, double nk_eps, double* out_weights, double* out_means,
                             double* out_variances, void* stream) {
  SSP_REQUIRE(n && f && s && out_weights && out_means && out_variances, "ssp_gmm_mstep: null pointer");
  SSP_REQUIRE(n_models > 0 && n_comp > 0 && n_feat > 0, "ssp_gmm_mstep: bad dims");
  ssp::gmm_mstep_kernel<<<(unsigned)n_models, 1024, 0, (cudaStream_t)stream>>>(n, f, s, n_comp, n_feat, reg_covar, nk_eps,
                                                                              out_weights, out_means, out_variances);
  SSP_LAUNCH_CHECK("gmm_mstep_kernel");
  return SSP_OK;
}

extern "C" int ssp_gmm_map_adapt(const double* n, const double* f, const double* s, const int64_t* seg_offsets,
                                 int64_t n_spk, const double* ubm_weights, const double* ubm_means,
                                 const double* ubm_variances, int32_t n_comp, int32_t n_feat, double relevance,
                                 int32_t flags, double* out_weights, double* out_means, double* out_variances,
                                 void* stream) {
  SSP_REQUIRE(n && f && s && seg_offsets && ubm_weights && ubm_means && ubm_variances, "ssp_gmm_map_adapt: null pointer");
  SSP_REQUIRE(n_spk > 0 && n_comp > 0 && n_feat > 0 && relevance >= 0.0, "ssp_gmm_map_adapt: bad dims");
  ssp::gmm_map_kernel<<<(unsigned)n_spk, 256, 0, (cudaStream_t)stream>>>(n, f, s, seg_offsets, ubm_weights, ubm_means,
                                                                       ubm_variances, n_comp, n_feat, relevance, flags,
                                                                       out_weights, out_means, out_variances);
  SSP_LAUNCH_CHECK("gmm_map_kernel");
  return SSP_OK;
}
