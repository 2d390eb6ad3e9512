// Top-C fast scoring of model sets that share weights and variances (Reynolds, Quatieri & Dunn 2000): every frame is
// scored under each model over the C components the reference member (the UBM) ranks highest for that frame only.
//
//   l_s(t) = log sum_{c in S_t} exp(L_s,c(t)),   L_s,c(t) = L_r,c(t) + a_s,c . x_t + b_s,c
//
// L_r,c(t) and S_t come from ssp_gmm_top_components (the selection pass of gmm_em_tc.cu); a and b are the difference of
// model s from the reference, which is all that is left of a model once weights and variances are shared:
//   a_s,c = (mu_s,c - mu_r,c) / var_c,   b_s,c = -1/2 sum_d (mu_s,c - mu_r,c)(mu_s,c + mu_r,c) / var_c.
// The frames are taken in chunks of kTopcChunkFrames; per chunk
//   topc_route (once for all chunks)  counting sort of the (frame, slot) pairs by selected component
//   topc_product_kernel               per component: its routed pairs x all models on the FP32 FMA pipe ->
//                                     v = L_r,c(t) + a_s,c . x_t + b_s,c, log domain, chunk buffer [frame][slot][model]
//   topc_combine_kernel               max-shifted log-sum-exp over the C slots of every (frame, model), per-utterance
//                                     sums in double
// At a chunk of 4096 frames a component receives about 4096 C / K routed pairs (20 at C = 5, K = 1024): too few rows
// for a 128-row tcgen05 tile, so the product runs on the CUDA cores, where the difference term is FP32-exact.
//
// Model sets MAP-adapted in weights and variances too (ssp_gmm_score_topc_adapted) keep the component correspondence
// with the reference and differ from it by a quadratic form.  The product block of component c centres its frames on
// mu_r,c (y = x - mu_r,c, delta = mu_s,c - mu_r,c), and topc_adapted_product_kernel computes
//   L_s,c(t) = L_r,c(t) + a . y + b . y^2 + k,   a = delta / var_s,   b = -1/2 (1/var_s - 1/var_r),
//   k = log(w_s / w_r) - 1/2 sum_d log(var_s / var_r) - 1/2 sum_d delta^2 / var_s
// with the frames routed to c being the ones that selected it, |y| is of the order of sigma, and a member (or component)
// with the reference's parameters has a row of zeros, so its value is L_r,c(t) bit for bit.  Routing, combine and
// finalize are the same kernels for both forms.
#include <algorithm>

#include "common.cuh"

namespace ssp {
namespace topc {

constexpr int kThreads = 128;     // models per block of the product and combine kernels
constexpr int kBatch = 64;        // routed pairs staged in shared memory at a time
constexpr int kCombineFrames = 64;

// ------------------------------------------------------------------------------------------------ pack
// pack[c][s][0 .. DA) = a_s,c (D values), b_s,c, zeros; one thread per (component, model), double inside
__global__ void __launch_bounds__(256) topc_pack_kernel(const double* __restrict__ var, const double* __restrict__ mu, int S, int K,
                                                        int D, int DA, int ref, float* __restrict__ pack) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= (int64_t)K * S) return;
  const int c = (int)(i / S), s = (int)(i % S);
  const double* ms = mu + ((int64_t)s * K + c) * D;
  const double* mr = mu + ((int64_t)ref * K + c) * D;
  const double* v = var + (int64_t)c * D;
  float* row = pack + i * DA;
  double b = 0.0;
  for (int d = 0; d < D; ++d) {
    const double diff = ms[d] - mr[d];
    row[d] = (float)(diff / v[d]);
    b += diff * (ms[d] + mr[d]) / v[d];
  }
  row[D] = (float)(-0.5 * b);
  for (int d = D + 1; d < DA; ++d) row[d] = 0.f;
}

// pack[c][s][0 .. DA) = a_s,c (D values), b_s,c (D values), k_s,c, zeros; after the K * S rows, mur[c][0 .. DR) = mu_r,c
// in FP32, zero padded (the centring of the product's staging).  One thread per (component, model), double inside.
__global__ void __launch_bounds__(256) topc_adapted_pack_kernel(const double* __restrict__ w, const double* __restrict__ mu,
                                                                const double* __restrict__ var, int S, int K, int D, int DA,
                                                                int DR, int ref, float* __restrict__ pack) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= (int64_t)K * S) return;
  const int c = (int)(i / S), s = (int)(i % S);
  const int64_t os = ((int64_t)s * K + c) * D, orf = ((int64_t)ref * K + c) * D;
  float* row = pack + i * DA;
  double k = log(w[(int64_t)s * K + c] / w[(int64_t)ref * K + c]);
  for (int d = 0; d < D; ++d) {
    const double delta = mu[os + d] - mu[orf + d], vs = var[os + d], vr = var[orf + d];
    row[d] = (float)(delta / vs);
    row[D + d] = (float)(-0.5 * (1.0 / vs - 1.0 / vr));
    k -= 0.5 * (log(vs / vr) + delta * delta / vs);
  }
  row[2 * D] = (float)k;
  for (int d = 2 * D + 1; d < DA; ++d) row[d] = 0.f;
  if (s == 0) {
    float* m = pack + (int64_t)K * S * DA + (int64_t)c * DR;
    for (int d = 0; d < DR; ++d) m[d] = d < D ? (float)mu[orf + d] : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------ routing
struct Route {
  const int32_t* idx;    // [T][C]
  int64_t T;
  int C, K;
  int32_t* cnt;          // [n_chunks][K] pairs routed to (chunk, component)
  int32_t* off;          // [n_chunks][K] exclusive prefix of cnt within the chunk; after the scatter: end of the run
  int32_t* list;         // [n_chunks][kTopcChunkFrames * C] pair index t_local * C + j, grouped by component
  int64_t n_chunks;
};

__global__ void __launch_bounds__(256) topc_hist_kernel(const Route r) {
  const int64_t n = r.T * r.C;
  for (int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x; g < n; g += (int64_t)gridDim.x * 256) {
    const int c = __ldg(r.idx + g);
    if (c >= 0 && c < r.K) atomicAdd(r.cnt + (g / ((int64_t)kTopcChunkFrames * r.C)) * r.K + c, 1);
  }
}

// one block per chunk: exclusive scan of its K counts (a thread sums a contiguous range)
__global__ void __launch_bounds__(1024) topc_scan_kernel(const Route r) {
  __shared__ int32_t part[1024];
  const int tid = threadIdx.x;
  const int32_t* cnt = r.cnt + (int64_t)blockIdx.x * r.K;
  int32_t* off = r.off + (int64_t)blockIdx.x * r.K;
  const int per = (r.K + 1023) / 1024;
  const int c0 = min(tid * per, r.K), c1 = min(c0 + per, r.K);
  int32_t sum = 0;
  for (int c = c0; c < c1; ++c) sum += cnt[c];
  part[tid] = sum;
  __syncthreads();
  if (tid == 0) {
    int32_t run = 0;
    for (int i = 0; i < 1024; ++i) { const int32_t v = part[i]; part[i] = run; run += v; }
  }
  __syncthreads();
  int32_t run = part[tid];
  for (int c = c0; c < c1; ++c) { off[c] = run; run += cnt[c]; }
}

__global__ void __launch_bounds__(256) topc_scatter_kernel(const Route r) {
  const int64_t n = r.T * r.C, per_chunk = (int64_t)kTopcChunkFrames * r.C;
  for (int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x; g < n; g += (int64_t)gridDim.x * 256) {
    const int c = __ldg(r.idx + g);
    if (c < 0 || c >= r.K) continue;
    const int64_t ch = g / per_chunk;
    const int pos = atomicAdd(r.off + ch * r.K + c, 1);
    r.list[ch * per_chunk + pos] = (int32_t)(g - ch * per_chunk);
  }
}

// ------------------------------------------------------------------------------------------------ product
// grid = (K, model tiles of kThreads); thread == model: its row (a, b) of the block's component in registers, the routed
// pairs' frames [x, 1, 0..] staged in shared memory and read as broadcasts
struct Product {
  const float* feats;
  const float* logit;    // [T][C]
  const float* pack;     // [K][S][DA]
  const int32_t* cnt;    // of this chunk
  const int32_t* off;    // of this chunk (run ends)
  const int32_t* list;   // of this chunk
  int64_t t0;            // first frame of the chunk
  int C, K, S, D;
  float* v;              // [kTopcChunkFrames][C][S]
};

template <int NQ>  // DA / 4
__global__ void __launch_bounds__(kThreads) topc_product_kernel(const Product p) {
  constexpr int DA = 4 * NQ;
  __shared__ __align__(16) float sx[kBatch][DA];
  __shared__ float sl[kBatch];
  __shared__ int32_t sq[kBatch];
  const int c = blockIdx.x, tid = threadIdx.x;
  const int n = p.cnt[c];
  if (n == 0) return;
  const int start = p.off[c] - n;
  const int s = blockIdx.y * kThreads + tid;
  const bool live = s < p.S;
  float4 a[NQ];
  {
    const float4* row = reinterpret_cast<const float4*>(p.pack + ((int64_t)c * p.S + (live ? s : 0)) * DA);
#pragma unroll
    for (int q = 0; q < NQ; ++q) a[q] = __ldg(row + q);
  }
  for (int b0 = 0; b0 < n; b0 += kBatch) {
    const int nb = min(kBatch, n - b0);
    __syncthreads();
    if (tid < nb) {
      const int q = __ldg(p.list + start + b0 + tid);
      sq[tid] = q;
      sl[tid] = __ldg(p.logit + p.t0 * p.C + q);
    }
    for (int e = tid; e < nb * DA; e += kThreads) {
      const int i = e / DA, d = e % DA;
      const int q = __ldg(p.list + start + b0 + i);
      const int64_t t = p.t0 + q / p.C;
      sx[i][d] = d < p.D ? __ldg(p.feats + t * p.D + d) : (d == p.D ? 1.f : 0.f);
    }
    __syncthreads();
    if (live) {
#pragma unroll 2
      for (int i = 0; i < nb; ++i) {
        const float4* x = reinterpret_cast<const float4*>(sx[i]);
        float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          const float4 xv = x[q];
          acc0 = fmaf(a[q].x, xv.x, acc0);
          acc1 = fmaf(a[q].y, xv.y, acc1);
          acc0 = fmaf(a[q].z, xv.z, acc0);
          acc1 = fmaf(a[q].w, xv.w, acc1);
        }
        __stcg(p.v + (int64_t)sq[i] * p.S + s, sl[i] + (acc0 + acc1));
      }
    }
  }
}

// The adapted form: as topc_product_kernel, with the row (a, b, k) of topc_adapted_pack_kernel and the routed frames
// staged as [y, y^2, 1, 0..], y = x - mu_r,c (mur: the FP32 reference means after the table)
template <int NQ>  // roundup(2D + 1, 4) / 4
__global__ void __launch_bounds__(kThreads) topc_adapted_product_kernel(const Product p, const float* __restrict__ mur) {
  constexpr int DA = 4 * NQ;
  __shared__ __align__(16) float sx[kBatch][DA];
  __shared__ float sl[kBatch];
  __shared__ int32_t sq[kBatch];
  const int c = blockIdx.x, tid = threadIdx.x;
  const int n = p.cnt[c];
  if (n == 0) return;
  const int start = p.off[c] - n;
  const int s = blockIdx.y * kThreads + tid;
  const bool live = s < p.S;
  const float* m = mur + (int64_t)c * ((p.D + 3) / 4 * 4);
  float4 a[NQ];
  {
    const float4* row = reinterpret_cast<const float4*>(p.pack + ((int64_t)c * p.S + (live ? s : 0)) * DA);
#pragma unroll
    for (int q = 0; q < NQ; ++q) a[q] = __ldg(row + q);
  }
  for (int b0 = 0; b0 < n; b0 += kBatch) {
    const int nb = min(kBatch, n - b0);
    __syncthreads();
    if (tid < nb) {
      const int q = __ldg(p.list + start + b0 + tid);
      sq[tid] = q;
      sl[tid] = __ldg(p.logit + p.t0 * p.C + q);
    }
    for (int e = tid; e < nb * DA; e += kThreads) {
      const int i = e / DA, d = e % DA;
      float val = d == 2 * p.D ? 1.f : 0.f;
      if (d < 2 * p.D) {
        const int j = d < p.D ? d : d - p.D;
        const int64_t t = p.t0 + __ldg(p.list + start + b0 + i) / p.C;
        const float y = __ldg(p.feats + t * p.D + j) - __ldg(m + j);
        val = d < p.D ? y : y * y;
      }
      sx[i][d] = val;
    }
    __syncthreads();
    if (live) {
#pragma unroll 2
      for (int i = 0; i < nb; ++i) {
        const float4* x = reinterpret_cast<const float4*>(sx[i]);
        float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          const float4 xv = x[q];
          acc0 = fmaf(a[q].x, xv.x, acc0);
          acc1 = fmaf(a[q].y, xv.y, acc1);
          acc0 = fmaf(a[q].z, xv.z, acc0);
          acc1 = fmaf(a[q].w, xv.w, acc1);
        }
        __stcg(p.v + (int64_t)sq[i] * p.S + s, sl[i] + (acc0 + acc1));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ combine
// grid = (model tiles, frame groups of kCombineFrames); thread == model, walking the group's frames in order and carrying
// the running sum of the current utterance until it changes
struct Combine {
  const float* v;
  const int32_t* idx;        // [T][C]
  const int64_t* offsets;    // [n_utts + 1]
  int64_t n_utts, T, t0, t1; // frames of the chunk: [t0, t1)
  int C, K, S;
  double* scores;            // [n_utts][S], sums
  float* frame_lse;          // [S][T] or NULL
};

__global__ void __launch_bounds__(kThreads) topc_combine_kernel(const Combine p) {
  const int s = blockIdx.x * kThreads + threadIdx.x;
  const int64_t f0 = p.t0 + (int64_t)blockIdx.y * kCombineFrames;
  const int64_t f1 = min(f0 + kCombineFrames, p.t1);
  if (s >= p.S || f0 >= f1) return;
  int64_t u = find_segment(p.offsets, p.n_utts, f0);
  int64_t u_end = __ldg(p.offsets + u + 1);
  double acc = 0.0;
  for (int64_t t = f0; t < f1; ++t) {
    if (t >= u_end) {
      atomicAdd(p.scores + u * p.S + s, acc);
      acc = 0.0;
      do { ++u; u_end = __ldg(p.offsets + u + 1); } while (t >= u_end);
    }
    const float* vt = p.v + (t - p.t0) * p.C * (int64_t)p.S + s;
    const int32_t* it = p.idx + t * p.C;
    float m = -INFINITY;
    for (int j = 0; j < p.C; ++j) {
      const int c = __ldg(it + j);
      if (c >= 0 && c < p.K) m = fmaxf(m, vt[(int64_t)j * p.S]);
    }
    float sum = 0.f;
    for (int j = 0; j < p.C; ++j) {
      const int c = __ldg(it + j);
      if (c >= 0 && c < p.K) sum += __expf(vt[(int64_t)j * p.S] - m);
    }
    const float l = m + logf(sum);
    if (p.frame_lse) p.frame_lse[(int64_t)s * p.T + t] = l;
    acc += (double)l;
  }
  atomicAdd(p.scores + u * p.S + s, acc);
}

// sums -> means; an empty utterance scores 0
__global__ void __launch_bounds__(256) topc_finalize_kernel(double* scores, const int64_t* offsets, int64_t n_utts, int S) {
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n_utts * S; i += (int64_t)gridDim.x * 256) {
    const int64_t u = i / S, n = offsets[u + 1] - offsets[u];
    scores[i] = n > 0 ? scores[i] / (double)n : 0.0;
  }
}

struct Ws {
  int64_t n_chunks;
  size_t o_cnt, o_off, o_list, o_v, bytes;
};
static Ws ws_layout(int K, int S, int C, int64_t T) {
  Ws w;
  w.n_chunks = (T + kTopcChunkFrames - 1) / kTopcChunkFrames;
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  size_t o = 0;
  w.o_cnt = o;  o = up(o + sizeof(int32_t) * (size_t)w.n_chunks * K);
  w.o_off = o;  o = up(o + sizeof(int32_t) * (size_t)w.n_chunks * K);
  w.o_list = o; o = up(o + sizeof(int32_t) * (size_t)w.n_chunks * kTopcChunkFrames * C);
  w.o_v = o;    o = up(o + sizeof(float) * (size_t)kTopcChunkFrames * C * S);
  w.bytes = T > 0 ? o : 0;
  return w;
}

}  // namespace topc

int64_t topc_pack_bytes(int S, int K, int D) { return (int64_t)K * S * topc_row_floats(D) * (int64_t)sizeof(float); }

int launch_pack_topc(const double* var, const double* mu, int S, int K, int D, int ref, void* pack, cudaStream_t st) {
  const int64_t n = (int64_t)K * S;
  topc::topc_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(var, mu, S, K, D, topc_row_floats(D), ref, (float*)pack);
  SSP_LAUNCH_CHECK("topc_pack_kernel");
  return SSP_OK;
}

int64_t topc_adapted_pack_bytes(int S, int K, int D) {
  return ((int64_t)K * S * topc_adapted_row_floats(D) + (int64_t)K * topc_ref_floats(D)) * (int64_t)sizeof(float);
}

int launch_pack_topc_adapted(const double* w, const double* mu, const double* var, int S, int K, int D, int ref, void* pack,
                             cudaStream_t st) {
  const int64_t n = (int64_t)K * S;
  topc::topc_adapted_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w, mu, var, S, K, D, topc_adapted_row_floats(D),
                                                                              topc_ref_floats(D), ref, (float*)pack);
  SSP_LAUNCH_CHECK("topc_adapted_pack_kernel");
  return SSP_OK;
}

int64_t score_topc_workspace_bytes(int S, int K, int C, int64_t T) { return (int64_t)topc::ws_layout(K, S, C, T).bytes; }

int launch_score_topc(const float* feats, const int64_t* offsets, int64_t n_utts, int64_t T, const int32_t* idx,
                      const float* logit, int C, const void* pack, int S, int K, int D, bool adapted, double* scores,
                      float* frame_lse, void* workspace, cudaStream_t st) {
  using namespace topc;
  SSP_CUDA_OK(cudaMemsetAsync(scores, 0, sizeof(double) * n_utts * S, st));
  if (T > 0) {
    const Ws w = ws_layout(K, S, C, T);
    unsigned char* base = (unsigned char*)workspace;
    Route r;
    r.idx = idx;
    r.T = T;
    r.C = C;
    r.K = K;
    r.cnt = (int32_t*)(base + w.o_cnt);
    r.off = (int32_t*)(base + w.o_off);
    r.list = (int32_t*)(base + w.o_list);
    r.n_chunks = w.n_chunks;
    SSP_CUDA_OK(cudaMemsetAsync(r.cnt, 0, sizeof(int32_t) * (size_t)w.n_chunks * K, st));
    const int64_t pairs = T * C;
    const unsigned g_pairs = (unsigned)std::min<int64_t>((pairs + 255) / 256, 4096);
    topc_hist_kernel<<<g_pairs, 256, 0, st>>>(r);
    SSP_LAUNCH_CHECK("topc_hist_kernel");
    topc_scan_kernel<<<(unsigned)w.n_chunks, 1024, 0, st>>>(r);
    SSP_LAUNCH_CHECK("topc_scan_kernel");
    topc_scatter_kernel<<<g_pairs, 256, 0, st>>>(r);
    SSP_LAUNCH_CHECK("topc_scatter_kernel");
    float* v = (float*)(base + w.o_v);
    const int DA = adapted ? topc_adapted_row_floats(D) : topc_row_floats(D);
    const float* mur = (const float*)pack + (int64_t)K * S * DA;   // adapted: the reference means after the table
    const unsigned m_tiles = (unsigned)((S + kThreads - 1) / kThreads);
    for (int64_t ch = 0; ch < w.n_chunks; ++ch) {
      const int64_t t0 = ch * kTopcChunkFrames, t1 = std::min<int64_t>(T, t0 + kTopcChunkFrames);
      Product p;
      p.feats = feats;
      p.logit = logit;
      p.pack = (const float*)pack;
      p.cnt = r.cnt + ch * K;
      p.off = r.off + ch * K;
      p.list = r.list + ch * (int64_t)kTopcChunkFrames * C;
      p.t0 = t0;
      p.C = C;
      p.K = K;
      p.S = S;
      p.D = D;
      p.v = v;
      const dim3 grid((unsigned)K, m_tiles);
      if (adapted) {
#define SSP_TOPC_PRODUCT(nq) \
  case nq: topc_adapted_product_kernel<nq><<<grid, kThreads, 0, st>>>(p, mur); break;
        switch (DA / 4) {
          SSP_TOPC_PRODUCT(1) SSP_TOPC_PRODUCT(2) SSP_TOPC_PRODUCT(3) SSP_TOPC_PRODUCT(4) SSP_TOPC_PRODUCT(5)
          SSP_TOPC_PRODUCT(6) SSP_TOPC_PRODUCT(7) SSP_TOPC_PRODUCT(8) SSP_TOPC_PRODUCT(9) SSP_TOPC_PRODUCT(10)
          SSP_TOPC_PRODUCT(11) SSP_TOPC_PRODUCT(12) SSP_TOPC_PRODUCT(13) SSP_TOPC_PRODUCT(14) SSP_TOPC_PRODUCT(15)
          SSP_TOPC_PRODUCT(16) SSP_TOPC_PRODUCT(17) SSP_TOPC_PRODUCT(18) SSP_TOPC_PRODUCT(19) SSP_TOPC_PRODUCT(20)
          default: SSP_REQUIRE(false, "ssp_gmm_score_topc_adapted: feature width %d", D);
        }
#undef SSP_TOPC_PRODUCT
        SSP_LAUNCH_CHECK("topc_adapted_product_kernel");
      } else {
#define SSP_TOPC_PRODUCT(nq) \
  case nq: topc_product_kernel<nq><<<grid, kThreads, 0, st>>>(p); break;
        switch (DA / 4) {
          SSP_TOPC_PRODUCT(1) SSP_TOPC_PRODUCT(2) SSP_TOPC_PRODUCT(3) SSP_TOPC_PRODUCT(4) SSP_TOPC_PRODUCT(5)
          SSP_TOPC_PRODUCT(6) SSP_TOPC_PRODUCT(7) SSP_TOPC_PRODUCT(8) SSP_TOPC_PRODUCT(9) SSP_TOPC_PRODUCT(10)
          default: SSP_REQUIRE(false, "ssp_gmm_score_topc: feature width %d", D);
        }
#undef SSP_TOPC_PRODUCT
        SSP_LAUNCH_CHECK("topc_product_kernel");
      }
      Combine q;
      q.v = v;
      q.idx = idx;
      q.offsets = offsets;
      q.n_utts = n_utts;
      q.T = T;
      q.t0 = t0;
      q.t1 = t1;
      q.C = C;
      q.K = K;
      q.S = S;
      q.scores = scores;
      q.frame_lse = frame_lse;
      topc_combine_kernel<<<dim3(m_tiles, (unsigned)((t1 - t0 + kCombineFrames - 1) / kCombineFrames)), kThreads, 0, st>>>(q);
      SSP_LAUNCH_CHECK("topc_combine_kernel");
    }
  }
  const unsigned g = (unsigned)std::min<int64_t>((n_utts * S + 255) / 256, 4096);
  topc_finalize_kernel<<<g, 256, 0, st>>>(scores, offsets, n_utts, S);
  SSP_LAUNCH_CHECK("topc_finalize_kernel");
  return SSP_OK;
}

}  // namespace ssp
