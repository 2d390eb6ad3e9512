// Dynamic time warping (dtw 1.4 `accelerated_dtw`: symmetric step pattern, no window, no slope weights) between
// every pair of two ragged sets of sequences (MFCC_DTW.py's template loop), FP32 CUDA cores.
//
//   D[i, j] = C[i, j] + min(D[i-1, j-1], D[i-1, j], D[i, j-1]),  D[-1, -1] = 0, rest of row / column -1 = +inf,
//   C[i, j] = sum_k (x_ik - y_jk)^2 (sqrt of it for 'euclidean') or sum_k |x_ik - y_jk|, in difference form: the Gram
//   form x.x - 2 x.y + y.y cancels digits near zero distance, and the min-plus recurrence has no MMA form anyway.
//
//   dtw_kernel      : one CTA per column-side sequence, staged in shared memory as [j][S] with an odd row stride S
//                     (lane l reads row j - l: 32 different banks).  Each warp runs one row-side sequence against it as
//                     an anti-diagonal wavefront: lane l owns rows l, l + 32, l + 64, ... (its feature vector in
//                     registers) and at step t computes column t - l of its current row.  "Up" D[i-1, j] is what lane
//                     l - 1 produced one step earlier (shuffle), "diagonal" D[i-1, j-1] is the "up" this lane received
//                     one step before that, "left" D[i, j-1] is the lane's own previous value.  Lane 31 writes its row
//                     to a per-warp row buffer in shared memory, which lane 0 reads when it starts the next row; a
//                     lane moves to its next row every max(m, 32) steps, so the strips follow each other without a
//                     ramp in between (steps = ceil(n / 32) * max(m, 32) + 31 per pair).
//   dtw_full_kernel : the same code compiled with FULL = true for one pair: also stores C and D (row-major n x m) for
//                     the host's traceback (accelerated_dtw drop-in).
#include <math.h>

#include "common.cuh"

namespace ssp {
namespace dtw {

constexpr int kWarps = 8;
constexpr int kMaxDim = 64;

// Feature widths are padded (with zeros on both sides, which add nothing to either metric) to one of these, so that
// the per-cell loop is unrolled over a compile-time length; 1, 13, 26 and 39 (MFCC_lib flattened, 13-d MFCC with
// 0 / 1 / 2 delta orders) are exact.
inline int dim_bucket(int dim) {
  const int b[] = {1, 2, 4, 8, 13, 16, 20, 26, 32, 39, 48, kMaxDim};
  for (int v : b)
    if (dim <= v) return v;
  return 0;
}
inline int row_stride(int dim) { return dim_bucket(dim) | 1; }
// shared memory: the column sequence [len][S] + one row buffer of len floats per warp
inline size_t smem_bytes(int dim, int64_t len) { return (size_t)len * (row_stride(dim) + kWarps) * sizeof(float); }

struct Args {
  const float* rows;           // row side, [total frames][dim]
  const int64_t* row_offsets;  // device int64[n_rows + 1], or NULL: one sequence of row_len frames
  int64_t n_rows, row_len;
  const float* cols;           // column side (shared memory)
  const int64_t* col_offsets;  // device int64[n_cols + 1], or NULL: one sequence of col_len frames
  int64_t n_cols, col_len;
  int dim, max_col_len, root;  // root: C = sqrt(sum of squares) ('euclidean')
  float* out;                  // dtw_kernel: dist[row * n_cols + col]
  float* cost;                 // dtw_full_kernel: C and D, [row_len][col_len]
  float* acc;
};

template <int DB, bool ABS, bool FULL>
__global__ void __launch_bounds__(kWarps * 32) dtw_kernel(const Args a) {
  constexpr int S = DB | 1;
  constexpr float INF = __builtin_huge_valf();
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t c = blockIdx.x;
  const int64_t c0 = a.col_offsets ? a.col_offsets[c] : 0;
  const int64_t m64 = a.col_offsets ? a.col_offsets[c + 1] - c0 : a.col_len;
  const bool fits = m64 >= 1 && m64 <= a.max_col_len;  // the host guarantees it; anything else yields NaN
  const int m = fits ? (int)m64 : 0;
  float* ys = smem;
  float* rb = smem + (size_t)a.max_col_len * S + (size_t)warp * a.max_col_len;
  {
    const float* y = a.cols + c0 * a.dim;
    for (int e = threadIdx.x; e < m * S; e += blockDim.x) {
      const int j = e / S, k = e - j * S;
      ys[e] = k < a.dim ? y[(int64_t)j * a.dim + k] : 0.f;
    }
  }
  __syncthreads();
  const int M = m > 32 ? m : 32;  // steps between two rows of one lane
  for (int64_t q = (int64_t)blockIdx.y * kWarps + warp; q < a.n_rows; q += (int64_t)gridDim.y * kWarps) {
    const int64_t q0 = a.row_offsets ? a.row_offsets[q] : 0;
    const int64_t n64 = a.row_offsets ? a.row_offsets[q + 1] - q0 : a.row_len;
    if (!fits || n64 < 1 || n64 > INT32_MAX / 2) {
      if (!FULL && lane == 0) a.out[q * a.n_cols + c] = NAN;
      continue;
    }
    const int n = (int)n64;
    const float* x = a.rows + q0 * a.dim;
    float xr[DB];
    int i = lane, j = -lane;
#pragma unroll
    for (int k = 0; k < DB; ++k) xr[k] = (k < a.dim && i < n) ? x[(int64_t)i * a.dim + k] : 0.f;
    float recv = INF, diag = INF, left = INF;
    // ceil(n / 32) * M + 31 steps can exceed INT32_MAX (a row of 10 644 257 frames against 6 456): they run in chunks of
    // at most 2^30, each counted in 32 bits (one chunk for any realistic pair, and the same inner loop as one count)
    for (int64_t remaining = (int64_t)((n + 31) >> 5) * M + 31; remaining > 0; remaining -= 1 << 30) {
      const int steps = remaining < (1 << 30) ? (int)remaining : 1 << 30;
      for (int t = 0; t < steps; ++t) {
        const bool col_ok = j >= 0 && j < m;
        float up = recv;
        if (lane == 0) up = (col_ok && i >= 32 && i < n) ? rb[j] : INF;
        float cur = INF;
        if (col_ok && i < n) {
          const float* yj = ys + j * S;
          float s = 0.f;
#pragma unroll
          for (int k = 0; k < DB; ++k) {
            const float d = xr[k] - yj[k];
            s = ABS ? s + fabsf(d) : fmaf(d, d, s);
          }
          if (a.root) s = sqrtf(s);
          const float dg = j == 0 ? (i == 0 ? 0.f : INF) : diag;
          const float lf = j == 0 ? INF : left;
          cur = s + fminf(dg, fminf(up, lf));
          if (FULL) {
            a.cost[(int64_t)i * m + j] = s;
            a.acc[(int64_t)i * m + j] = cur;
          } else if (i == n - 1 && j == m - 1) {
            a.out[q * a.n_cols + c] = cur;
          }
          if (lane == 31) rb[j] = cur;
        }
        left = cur;
        diag = up;
        __syncwarp();  // orders lane 31's row-buffer store before lane 0's load of it (M >= 32 steps later, or the next)
        recv = __shfl_up_sync(0xffffffffu, cur, 1);
        if (++j == M) {
          j = 0;
          i += 32;
#pragma unroll
          for (int k = 0; k < DB; ++k) xr[k] = (k < a.dim && i < n) ? x[(int64_t)i * a.dim + k] : 0.f;
        }
      }
    }
    __syncwarp();
  }
}

template <int DB, bool FULL>
int launch_db(const Args& a, int metric, cudaStream_t st) {
  const dim3 block(kWarps * 32);
  const int64_t gy = (a.n_rows + kWarps - 1) / kWarps;
  const dim3 grid((unsigned)a.n_cols, (unsigned)(gy < 65535 ? gy : 65535));
  const size_t smem = smem_bytes(DB, a.max_col_len);
  auto kern = metric == SSP_DTW_CITYBLOCK ? dtw_kernel<DB, true, FULL> : dtw_kernel<DB, false, FULL>;
  if (smem > 48 * 1024) SSP_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, block, smem, st>>>(a);
  SSP_LAUNCH_CHECK(FULL ? "dtw_full_kernel" : "dtw_kernel");
  return SSP_OK;
}

template <bool FULL>
int launch(const Args& a, int metric, cudaStream_t st) {
  switch (dim_bucket(a.dim)) {
    case 1: return launch_db<1, FULL>(a, metric, st);
    case 2: return launch_db<2, FULL>(a, metric, st);
    case 4: return launch_db<4, FULL>(a, metric, st);
    case 8: return launch_db<8, FULL>(a, metric, st);
    case 13: return launch_db<13, FULL>(a, metric, st);
    case 16: return launch_db<16, FULL>(a, metric, st);
    case 20: return launch_db<20, FULL>(a, metric, st);
    case 26: return launch_db<26, FULL>(a, metric, st);
    case 32: return launch_db<32, FULL>(a, metric, st);
    case 39: return launch_db<39, FULL>(a, metric, st);
    case 48: return launch_db<48, FULL>(a, metric, st);
    case kMaxDim: return launch_db<kMaxDim, FULL>(a, metric, st);
  }
  set_error("dtw: dim %d outside [1, %d]", a.dim, kMaxDim);
  return SSP_EUNSUP;
}

}  // namespace dtw
}  // namespace ssp

extern "C" int64_t ssp_dtw_max_len(int32_t dim) {
  using namespace ssp::dtw;
  if (dim < 1 || dim > kMaxDim) return 0;
  return (int64_t)(ssp::kMaxDynSmem / smem_bytes(dim, 1));
}

static int dtw_check_common(const char* fn, int32_t dim, int32_t metric, int64_t col_len) {
  SSP_REQUIRE(metric == SSP_DTW_EUCLIDEAN || metric == SSP_DTW_SQEUCLIDEAN || metric == SSP_DTW_CITYBLOCK,
              "%s: unknown metric %d", fn, metric);
  if (dim < 1 || dim > ssp::dtw::kMaxDim) {
    ssp::set_error("%s: dim %d outside [1, %d]", fn, dim, ssp::dtw::kMaxDim);
    return SSP_EUNSUP;
  }
  if (col_len > ssp_dtw_max_len(dim)) {
    ssp::set_error("%s: column-side sequences of %lld frames, the kernel holds at most %lld at dim %d", fn,
                   (long long)col_len, (long long)ssp_dtw_max_len(dim), dim);
    return SSP_EUNSUP;
  }
  return SSP_OK;
}

extern "C" int ssp_dtw_batch(const float* q, const int64_t* q_offsets, int64_t n_q, const float* r, const int64_t* r_offsets,
                             int64_t n_r, int32_t dim, int32_t metric, int64_t max_r_len, float* out_dist, void* stream) {
  SSP_REQUIRE(q && q_offsets && r && r_offsets && out_dist, "ssp_dtw_batch: null pointer");
  SSP_REQUIRE(n_q >= 0 && n_r >= 0 && n_r <= INT32_MAX && max_r_len >= 1, "ssp_dtw_batch: bad sizes");
  const int rc = dtw_check_common("ssp_dtw_batch", dim, metric, max_r_len);
  if (rc != SSP_OK) return rc;
  if (n_q == 0 || n_r == 0) return SSP_OK;
  ssp::dtw::Args a = {};
  a.rows = q;
  a.row_offsets = q_offsets;
  a.n_rows = n_q;
  a.cols = r;
  a.col_offsets = r_offsets;
  a.n_cols = n_r;
  a.dim = dim;
  a.max_col_len = (int)max_r_len;
  a.root = metric == SSP_DTW_EUCLIDEAN;
  a.out = out_dist;
  return ssp::dtw::launch<false>(a, metric, (cudaStream_t)stream);
}

extern "C" int ssp_dtw_full(const float* x, int64_t n_x, const float* y, int64_t n_y, int32_t dim, int32_t metric,
                            float* out_cost, float* out_acc, void* stream) {
  SSP_REQUIRE(x && y && out_cost && out_acc, "ssp_dtw_full: null pointer");
  SSP_REQUIRE(n_x >= 1 && n_y >= 1 && n_x <= INT32_MAX / 2, "ssp_dtw_full: empty or oversized sequence (%lld x %lld)",
              (long long)n_x, (long long)n_y);
  const int rc = dtw_check_common("ssp_dtw_full", dim, metric, n_y);
  if (rc != SSP_OK) return rc;
  ssp::dtw::Args a = {};
  a.rows = x;
  a.n_rows = 1;
  a.row_len = n_x;
  a.cols = y;
  a.n_cols = 1;
  a.col_len = n_y;
  a.dim = dim;
  a.max_col_len = (int)n_y;
  a.root = metric == SSP_DTW_EUCLIDEAN;
  a.cost = out_cost;
  a.acc = out_acc;
  return ssp::dtw::launch<true>(a, metric, (cudaStream_t)stream);
}
