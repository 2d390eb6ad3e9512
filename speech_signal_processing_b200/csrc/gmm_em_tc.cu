// EM / MAP sufficient statistics on the tensor cores (sm_100a): posteriors and N/F/S as two chained GEMMs fed by
// bulk copies of operand images that are built ONCE per set of frames.
//
// The frames of an EM run never change, only the model does.  ssp_gmm_stats therefore splits into
//
//   prepare (once per feats / seg_offsets; skipped when the caller says the workspace still holds the images):
//     em_plan_kernel   segments are padded to multiples of 64 frames ("blocks"); block -> (segment, first frame, frames)
//     em_prep_kernel   per block: the tcgen05 shared-memory images of its frames
//                        Fb  [x, x^2, 1, 1, 0..] as BF16 hi + lo, K-major rows of 128 frames  (logit GEMMs, both passes)
//                        Xt  the same columns as FP16 hi + lo with the FRAME index contiguous (statistics GEMM)
//   per call (one EM iteration / one enrolment):
//     gmm_em_lse_kernel    logits[frame, comp] for a PAIR of 128-component tiles per CTA, 128 frames per step:
//                          3 x BF16 (hi.hi + lo.hi + hi.lo, FP32 accumulation in TMEM; emulated on the CPU: per-frame
//                          log-likelihood within 4e-7 relative of float64, N/F/S indistinguishable from 3xTF32 --
//                          the TF32 rounding of gamma below dominates) at twice the TF32 issue rate;
//                          thread == frame row -> (max, sum 2^x) per 64-component half tile -> workspace
//     em_merge_kernel      partials -> per-frame log2-likelihood, frame_lse, per-segment log-likelihood
//     gmm_em_stats_kernel  TRANSPOSED logits[comp, frame] (same images, model tile as the M-side operand), 64 frames
//                          per step, thread == component row: gamma = 2^(L - lse[frame]) is written by tcgen05.st IN
//                          PLACE over the logits and is the TMEM-side operand of the statistics GEMM
//                          stats[comp, :] += gamma . Xt (kind::f16: gamma as FP16 -- the 11-bit significand a TF32 gamma
//                          had -- scaled by 2^12 so that posteriors down to 1e-11 survive FP16's range, Xt as FP16
//                          hi + lo; K = 16 frames per MMA: 8 MMAs per step instead of the 16 of the TF32 form),
//                          accumulated in TMEM over all blocks of a segment and added, unscaled, to the float64
//                          N / F / S outputs at segment ends.
//
// No thread builds an operand any more: the producer warp streams images with cp.async.bulk, one warp issues the MMAs,
// sixteen warps do the exponentials.  (Round 1 split the frames into hi / lo in every CTA of every pass of every
// iteration -- 8x per iteration at K = 512 -- and was bound by that thread work: tensor pipe 37-40 % busy.)
// Blocks never straddle a segment, so one kernel set serves UBM EM (one segment) and batched MAP enrolment (one
// segment per speaker).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace ssp {
namespace em {

using namespace tc;

constexpr int BN = 128;        // components per tile
constexpr int IMG = 128;       // frames per Fb image = rows of one LSE step
constexpr int BLK = 64;        // frames per block: padding granule of a segment, rows of one STATS step
constexpr int EPI = 512;       // 16 epilogue warps
constexpr int THREADS = 64 + EPI;
constexpr int MAX_KD = 80;
constexpr int NS_L = 3;        // Fb stages of the LSE pass
constexpr float kGammaScale = 4096.f;   // gamma rides the statistics GEMM as FP16(gamma * 2^12); the merge kernel folds it into lse2

// ------------------------------------------------------------------------------------------------ workspace
struct Ws {
  int64_t nb_max, P;           // upper bound on the number of blocks (even), padded frames = nb_max * BLK
  int KDb;                     // contraction length, a multiple of 16: roundup(2D + 2, 16); also the N of the statistics GEMM
  size_t o_blk_start, o_blk_seg, o_blk_t0, o_blk_nt, o_lse2, o_partial, o_fb, o_xt, bytes;
  size_t img_bytes() const { return (size_t)512 * KDb; }   // Fb image of 128 frames == model tile image of 128 components
  size_t xt_bytes() const { return (size_t)256 * KDb; }    // Xt image of one 64-frame block (FP16 hi + lo)
};
static Ws ws_layout(const PackLayout& L, int64_t total_frames, int64_t n_segs) {
  Ws w;
  w.KDb = (2 * L.D + 2 + 15) / 16 * 16;
  w.nb_max = (total_frames / BLK + 2 * n_segs + 2) & ~(int64_t)1;  // per-segment models pad segments to whole 128-frame images
  w.P = w.nb_max * BLK;
  auto up = [](size_t x) { return (x + 1023) / 1024 * 1024; };
  size_t o = 0;
  w.o_blk_start = o; o = up(o + sizeof(int64_t) * (n_segs + 2));
  w.o_blk_seg = o;   o = up(o + sizeof(int32_t) * w.nb_max);
  w.o_blk_t0 = o;    o = up(o + sizeof(int64_t) * w.nb_max);
  w.o_blk_nt = o;    o = up(o + sizeof(int32_t) * w.nb_max);
  w.o_lse2 = o;      o = up(o + sizeof(float) * w.P);
  w.o_fb = o;        o = up(o + w.img_bytes() * (w.nb_max / 2));
  w.o_xt = o;        o = up(o + w.xt_bytes() * w.nb_max);
  // last: the only section whose size depends on K, so that the images stay valid for a model of another size
  w.o_partial = o;   o = up(o + sizeof(float2) * 2 * (L.Kp / BN) * w.P);
  w.bytes = o;
  return w;
}

struct Args {
  const float* feats;
  const int64_t* seg;
  int64_t n_segs, total_frames;
  // workspace
  int64_t* blk_start;       // [n_segs + 1]; blk_start[n_segs] = number of blocks
  int32_t* blk_seg;         // [nb_max] segment of a block, -1: padding
  int64_t* blk_t0;          // [nb_max] first frame
  int32_t* blk_nt;          // [nb_max] frames (1..64; 0: padding)
  float* lse2;              // [P] per padded frame: log2-likelihood - log2(kGammaScale); 3e38 for dead rows
  float2* partial;          // [2 n_tiles][P]
  const unsigned char* fb;  // [nb_max / 2] images: [hi | lo][KDb/8][128 rows][8 bf16]
  const unsigned char* xt;  // [nb_max] images:     [hi | lo][8][KDb rows][8 half]
  int64_t nb_max, P;
  // model
  const unsigned char* tiles;  // [model][n_tiles] images [hi | lo][KDb/8][128 comps][8 bf16]
  int K, D, KDb, n_tiles;
  int per_seg_model;           // 1: segment s is scored under model s (grid z = segment; segments padded to whole Fb images)
  // outputs
  float* frame_lse;          // may be NULL (ssp_gmm_posteriors)
  double* out_n;
  double* out_f;
  double* out_s;
  double* out_loglik;        // may be NULL (ssp_gmm_posteriors)
  float* out_resp;           // [total_frames][K] (posterior pass)
  int64_t* out_label;        // [total_frames]    (posterior pass)
  int resp_vec;              // out_resp rows are 16-byte aligned (K % 4 == 0 and an aligned base): float4 stores
};

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_st16u(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tc_st32(uint32_t taddr, const float (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
        "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]), "f"(v[16]), "f"(v[17]), "f"(v[18]), "f"(v[19]),
        "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]), "f"(v[24]), "f"(v[25]), "f"(v[26]), "f"(v[27]), "f"(v[28]), "f"(v[29]),
        "f"(v[30]), "f"(v[31])
      : "memory");
}
__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// share of the LSE pass's exponentials on the FMA pipe (pairs of 16), measured at config 3 (36 M frames, K = 512):
// 2 / 4 / 6 / 8 pairs -> 30.0 / 27.8 / 26.3 / 27.3 ms per call
constexpr int kPolyPairs = 6;

// sum over 32 accumulator columns of 2^(r - cm); kPolyPairs of the 16 column pairs on the FMA pipe (degree-4 minimax
// polynomial after a magic-number range reduction, 2.7e-6 relative), the rest MUFU ex2 (see gmm_score_sv.cu)
__device__ __forceinline__ float exp_sum32(const uint32_t (&r)[32], float cm) {
  static_assert(kPolyPairs % 2 == 0 && kPolyPairs <= 16, "pairs are consumed two at a time");
  const float MAGIC = 12582912.f;  // 1.5 * 2^23
  const float2 mg = make_float2(MAGIC, MAGIC), nmg = make_float2(-MAGIC, -MAGIC), neg1 = make_float2(-1.f, -1.f);
  const float2 ncm = make_float2(-cm, -cm);
  float2 accp = make_float2(0.f, 0.f), accm0 = accp, accm1 = accp;
#pragma unroll
  for (int i = 0; i < kPolyPairs; ++i) {
    float2 d = __fadd2_rn(make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1])), ncm);
    d.x = fmaxf(d.x, -126.f);
    d.y = fmaxf(d.y, -126.f);
    const float2 t = __fadd2_rn(d, mg);
    const float2 nn = __fadd2_rn(t, nmg);
    const float2 f = __ffma2_rn(nn, neg1, d);
    float2 p = __ffma2_rn(make_float2(0.009570102207362652f, 0.009570102207362652f), f, make_float2(0.05591785907745361f, 0.05591785907745361f));
    p = __ffma2_rn(p, f, make_float2(0.240247443318367f, 0.240247443318367f));
    p = __ffma2_rn(p, f, make_float2(0.6931217908859253f, 0.6931217908859253f));
    p = __ffma2_rn(p, f, make_float2(0.9999992847442627f, 0.9999992847442627f));
    float2 e;
    e.x = __uint_as_float(__float_as_uint(p.x) + (__float_as_uint(t.x) << 23));
    e.y = __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(t.y) << 23));
    accp = __fadd2_rn(accp, e);
  }
#pragma unroll
  for (int i = kPolyPairs; i < 16; i += 2) {
    const float2 d0 = __fadd2_rn(make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1])), ncm);
    const float2 d1 = __fadd2_rn(make_float2(__uint_as_float(r[2 * i + 2]), __uint_as_float(r[2 * i + 3])), ncm);
    accm0 = __fadd2_rn(accm0, make_float2(ex2(d0.x), ex2(d0.y)));
    accm1 = __fadd2_rn(accm1, make_float2(ex2(d1.x), ex2(d1.y)));
  }
  const float2 tot = __fadd2_rn(__fadd2_rn(accm0, accm1), accp);
  return tot.x + tot.y;
}

// ================================================================================================ prepare
// blk_start[s] = number of 64-frame blocks of the segments before s (one block, chunked scan)
__global__ void __launch_bounds__(1024) em_plan_kernel(const Args a) {
  __shared__ int64_t part[1024];
  const int tid = threadIdx.x;
  const int64_t per = (a.n_segs + 1023) / 1024;
  const int64_t s0 = min((int64_t)tid * per, a.n_segs), s1 = min(s0 + per, a.n_segs);
  // blocks of a segment; with per-segment models an even number, so that no Fb image straddles two models
  auto n_blk = [&](int64_t s) {
    const int64_t nbk = (a.seg[s + 1] - a.seg[s] + BLK - 1) / BLK;
    return a.per_seg_model ? (nbk + 1) & ~(int64_t)1 : nbk;
  };
  int64_t sum = 0;
  for (int64_t s = s0; s < s1; ++s) sum += n_blk(s);
  part[tid] = sum;
  __syncthreads();
  if (tid == 0) {
    int64_t run = 0;
    for (int i = 0; i < 1024; ++i) { const int64_t v = part[i]; part[i] = run; run += v; }
    a.blk_start[a.n_segs] = run;
  }
  __syncthreads();
  int64_t run = part[tid];
  for (int64_t s = s0; s < s1; ++s) {
    a.blk_start[s] = run;
    run += n_blk(s);
  }
}

__device__ __forceinline__ float feat_col(const float* xr, int j, int D) {
  if (j < D) return xr[j];
  if (j < 2 * D) { const float x = xr[j - D]; return x * x; }
  return j < 2 * D + 2 ? 1.f : 0.f;
}

// one CTA per block: block table entry + the block's half of an Fb image + its Xt image
__global__ void __launch_bounds__(256) em_prep_kernel(const Args a) {
  __shared__ float sx[BLK * (MAX_KD / 2)];
  __shared__ int s_nt;
  __shared__ int64_t s_t0;
  const int64_t b = blockIdx.x;
  const int64_t nb = a.blk_start[a.n_segs];
  if (b >= ((nb + 1) & ~(int64_t)1)) return;
  const int tid = threadIdx.x, D = a.D, KDb = a.KDb;
  if (tid == 0) {
    int seg = -1, nt = 0;
    int64_t t0 = 0;
    if (b < nb) {
      seg = find_segment(a.blk_start, a.n_segs, b);
      t0 = a.seg[seg] + (b - a.blk_start[seg]) * BLK;
      nt = (int)max((int64_t)0, min((int64_t)BLK, a.seg[seg + 1] - t0));  // 0: the padding block of an odd-sized segment
    }
    s_nt = nt; s_t0 = t0;
    a.blk_seg[b] = seg;
    a.blk_t0[b] = t0;
    a.blk_nt[b] = nt;
  }
  __syncthreads();
  const int nt = s_nt;
  const float* src = a.feats + s_t0 * D;
  for (int i = tid; i < BLK * D; i += 256) sx[i] = i < nt * D ? __ldg(src + i) : 0.f;
  __syncthreads();
  // ---- Fb: rows (b & 1) * 64 .. + 63 of image b / 2; item = (chunk of 8 columns, row) -> 16 bytes of hi and of lo
  {
    unsigned char* img = const_cast<unsigned char*>(a.fb) + (size_t)(b >> 1) * 512 * KDb;
    const size_t part_bytes = (size_t)256 * KDb;  // [KDb/8][128][16 B]
    const int row0 = (int)(b & 1) * BLK;
    for (int it = tid; it < (KDb >> 3) * BLK; it += 256) {
      const int c = it / BLK, r = it % BLK;
      const bool live = r < nt;
      const float* xr = sx + r * D;
      __align__(16) __nv_bfloat16 h[8], l[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float v = live ? feat_col(xr, 8 * c + e, D) : 0.f;
        h[e] = __float2bfloat16_rn(v);
        l[e] = __float2bfloat16_rn(v - __bfloat162float(h[e]));
      }
      const size_t off = ((size_t)c * IMG + row0 + r) * 16;
      *reinterpret_cast<uint4*>(img + off) = *reinterpret_cast<const uint4*>(h);
      *reinterpret_cast<uint4*>(img + part_bytes + off) = *reinterpret_cast<const uint4*>(l);
    }
  }
  // ---- Xt: item = (chunk of 8 frames, column j) -> 16 bytes (8 FP16) of hi and of lo
  {
    unsigned char* img = const_cast<unsigned char*>(a.xt) + (size_t)b * 256 * KDb;
    const size_t part_bytes = (size_t)128 * KDb;  // [8][KDb][16 B]
    for (int it = tid; it < 8 * KDb; it += 256) {
      const int fc = it / KDb, j = it % KDb;
      __align__(16) __half h[8], l[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int r = 8 * fc + e;
        // column 2D + 1 (the second "one" of the logit operand) is dead weight here: N is column 2D
        const float v = (r < nt && j <= 2 * D) ? feat_col(sx + r * D, j, D) : 0.f;
        h[e] = __float2half_rn(v);
        l[e] = __float2half_rn(v - __half2float(h[e]));
      }
      *reinterpret_cast<uint4*>(img + (size_t)it * 16) = *reinterpret_cast<const uint4*>(h);
      *reinterpret_cast<uint4*>(img + part_bytes + (size_t)it * 16) = *reinterpret_cast<const uint4*>(l);
    }
  }
}

// ================================================================================================ pass LSE / posteriors
// grid = (image chunks, tile pairs).  Shared memory: the pair's model tiles (BF16 hi + lo) + NS_L Fb stages; tensor
// memory: 2 tiles x 2 buffers of 128 accumulator columns.  The epilogue is chosen at compile time:
//   kEpiLse    (gmm_em_lse_kernel)   (max, sum 2^x) of each 64-component half tile -> partial
//   kEpiResp   (gmm_em_post_kernel)  gamma = 2^(L - lse2) -> out_resp[frame][comp], live frames and components only
//   kEpiLabel  (gmm_em_post_kernel)  (max logit, lowest component reaching it) of each half tile -> partial, in the
//                                    slots of the LSE partials (em_label_merge_kernel reduces them)
constexpr int kEpiLse = 0, kEpiResp = 1, kEpiLabel = 2;

template <int kEpi>
__device__ __forceinline__ void logit_pass(const Args& a) {
  constexpr bool kResp = (kEpi & kEpiResp) != 0, kLabel = (kEpi & kEpiLabel) != 0;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int KDb = a.KDb;
  const uint32_t TB = 512u * (uint32_t)KDb;  // bytes of one image (hi + lo)
  unsigned char* sB = smem;                  // [2][TB]
  unsigned char* sF = smem + 2 * (size_t)TB; // [NS_L][TB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sF + (size_t)NS_L * TB);
  uint64_t* b_full = bars;                   // model tiles landed
  uint64_t* f_full = bars + 1;               // [NS_L]
  uint64_t* f_empty = f_full + NS_L;         // [NS_L]
  uint64_t* t_full = f_empty + NS_L;         // [4] accumulator (buffer, tile) holds a step's logits
  uint64_t* t_empty = t_full + 4;            // [4]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 4);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tile0 = 2 * blockIdx.y;
  const int ntl = min(2, a.n_tiles - tile0);
  if (tid == 0) {
    mbar_init(b_full, 1);
    for (int i = 0; i < NS_L; ++i) { mbar_init(f_full + i, 1); mbar_init(f_empty + i, 1); }
    for (int i = 0; i < 4; ++i) { mbar_init(t_full + i, 1); mbar_init(t_empty + i, 2 * IMG); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // images of this CTA: a chunk of all images, or (per-segment models) a chunk of the images of segment blockIdx.z
  int64_t img_lo = 0, img_hi = (a.blk_start[a.n_segs] + 1) >> 1;
  const unsigned char* tiles = a.tiles;
  if (a.per_seg_model) {
    img_lo = a.blk_start[blockIdx.z] >> 1;
    img_hi = a.blk_start[blockIdx.z + 1] >> 1;
    tiles += (size_t)blockIdx.z * a.n_tiles * TB;
  }
  const int64_t per = (img_hi - img_lo + gridDim.x - 1) / gridDim.x;
  const int64_t i0 = img_lo + (int64_t)blockIdx.x * per, i1 = min(i0 + per, img_hi);

  if (warp == 0) {
    // ===================== producer =====================
    if (i0 < i1) {
      if (elect_one()) {
        mbar_arrive_expect_tx(b_full, (uint32_t)ntl * TB);
        for (int t = 0; t < ntl; ++t) bulk_g2s(sB + (size_t)t * TB, tiles + (size_t)(tile0 + t) * TB, TB, b_full);
      }
      __syncwarp();
      uint32_t k = 0;
      for (int64_t i = i0; i < i1; ++i, ++k) {
        const uint32_t st = k % NS_L, ph = (k / NS_L) & 1u;
        mbar_wait_relaxed(f_empty + st, ph ^ 1u);
        if (elect_one()) {
          mbar_arrive_expect_tx(f_full + st, TB);
          bulk_g2s(sF + (size_t)st * TB, a.fb + (size_t)i * TB, TB, f_full + st);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (i0 < i1) {
      constexpr uint32_t lbo = IMG * 16u, sbo = 128u;  // 128-row K-major images: chunk stride 2 KB, 8-row groups contiguous
      constexpr uint32_t kstep = (2u * lbo) >> 4;      // one K = 16 step = two 16-byte chunks
      const uint32_t idesc = make_idesc_bf16(IMG, BN);
      const int ksteps = KDb >> 4;
      const uint32_t half_units = (TB >> 1) >> 4;      // hi -> lo inside an image, in descriptor units
      const uint64_t b_desc0 = make_desc(smem_u32(sB), lbo, sbo), f_desc0 = make_desc(smem_u32(sF), lbo, sbo);
      mbar_wait_relaxed(b_full, 0);
      uint32_t k = 0;
      for (int64_t i = i0; i < i1; ++i, ++k) {
        const uint32_t st = k % NS_L, ph = (k / NS_L) & 1u;
        mbar_wait_relaxed(f_full + st, ph);
        tc_fence_after();
        const uint64_t fh = f_desc0 + (uint64_t)(st * (TB >> 4)), fl = fh + half_units;
        for (int t = 0; t < ntl; ++t) {
          const uint32_t slot = 2u * (k & 1u) + (uint32_t)t;
          mbar_wait_relaxed(t_empty + slot, ((k >> 1) & 1u) ^ 1u);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t d = tmem_base + slot * BN;
            const uint64_t bh = b_desc0 + (uint64_t)(t * (TB >> 4)), bl = bh + half_units;
            for (int q = 0; q < ksteps; ++q) mma_bf16_ss(d, fh + (uint64_t)(q * kstep), bh + (uint64_t)(q * kstep), idesc, q > 0 ? 1u : 0u);
            for (int q = 0; q < ksteps; ++q) mma_bf16_ss(d, fl + (uint64_t)(q * kstep), bh + (uint64_t)(q * kstep), idesc, 1u);
            for (int q = 0; q < ksteps; ++q) mma_bf16_ss(d, fh + (uint64_t)(q * kstep), bl + (uint64_t)(q * kstep), idesc, 1u);
            tc_commit(t_full + slot);
          }
          __syncwarp();
        }
        if (elect_one()) tc_commit(f_empty + st);
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue: thread == (frame row, 64 of a tile's 128 columns) =====================
    const int ew = warp - 2;
    const int t = ew >> 3, half = (ew >> 2) & 1, quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    if (t < ntl && i0 < i1) {
      float2* dst = a.partial + (size_t)(2 * (tile0 + t) + half) * a.P + row;
      const int comp0 = (2 * (tile0 + t) + half) * 64;  // component of column 0 of this thread's half tile
      uint32_t k = 0;
      for (int64_t i = i0; i < i1; ++i, ++k) {
        // posteriors: the row's frame and merged lse2, loaded before the wait for the logits
        int live = 0;
        int64_t frame = 0;
        float l2 = 0.f;
        if constexpr (kResp) {
          const int64_t b = 2 * i + (row >> 6);
          live = (row & 63) < __ldg(a.blk_nt + b);
          frame = __ldg(a.blk_t0 + b) + (row & 63);
          l2 = __ldg(a.lse2 + i * IMG + row) + 12.f;  // undo the gamma scale of the statistics pass: log2(kGammaScale) = 12
        }
        const uint32_t slot = 2u * (k & 1u) + (uint32_t)t;
        mbar_wait(t_full + slot, (k >> 1) & 1u);
        tc_fence_after();
        uint32_t ra[32], rb[32];
        const uint32_t taddr = tmem_base + lane_addr + slot * BN + half * 64;
        tc_ld32_issue(taddr, ra);
        tc_ld32_issue(taddr + 32, rb);
        tc_ld_wait2(ra, rb);
        tc_fence_before();
        mbar_arrive(t_empty + slot);
        if constexpr (kEpi == kEpiLse) {
          float cm = max3(__uint_as_float(ra[0]), __uint_as_float(ra[1]), __uint_as_float(rb[0]));
#pragma unroll
          for (int e = 2; e < 32; e += 2) cm = max3(cm, __uint_as_float(ra[e]), __uint_as_float(ra[e + 1]));
#pragma unroll
          for (int e = 1; e < 31; e += 2) cm = max3(cm, __uint_as_float(rb[e]), __uint_as_float(rb[e + 1]));
          cm = fmaxf(cm, __uint_as_float(rb[31]));
          const float s = exp_sum32(ra, cm) + exp_sum32(rb, cm);
          dst[i * IMG] = make_float2(cm, s);
        }
        if constexpr (kLabel) {
          // strict > in component order: the lowest index wins a tie (numpy's argmax); padded components never compete
          const int n_live = a.K - comp0;  // columns of real components (may be <= 0: a half tile of padding)
          float bm = -3.0e38f;
          int bi = 0;
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const float v = __uint_as_float(ra[e]);
            if (e < n_live && v > bm) { bm = v; bi = e; }
          }
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const float v = __uint_as_float(rb[e]);
            if (32 + e < n_live && v > bm) { bm = v; bi = 32 + e; }
          }
          dst[i * IMG] = make_float2(bm, __int_as_float(comp0 + bi));
        }
        if constexpr (kResp) {
          if (live) {
            float* out = a.out_resp + frame * a.K + comp0;
            if (a.resp_vec && comp0 + 64 <= a.K) {
              float4* o4 = reinterpret_cast<float4*>(out);
#pragma unroll
              for (int q = 0; q < 8; ++q)
                __stcs(o4 + q, make_float4(ex2(__uint_as_float(ra[4 * q]) - l2), ex2(__uint_as_float(ra[4 * q + 1]) - l2),
                                           ex2(__uint_as_float(ra[4 * q + 2]) - l2), ex2(__uint_as_float(ra[4 * q + 3]) - l2)));
#pragma unroll
              for (int q = 0; q < 8; ++q)
                __stcs(o4 + 8 + q, make_float4(ex2(__uint_as_float(rb[4 * q]) - l2), ex2(__uint_as_float(rb[4 * q + 1]) - l2),
                                               ex2(__uint_as_float(rb[4 * q + 2]) - l2), ex2(__uint_as_float(rb[4 * q + 3]) - l2)));
            } else {
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (comp0 + e < a.K) __stcs(out + e, ex2(__uint_as_float(ra[e]) - l2));
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (comp0 + 32 + e < a.K) __stcs(out + 32 + e, ex2(__uint_as_float(rb[e]) - l2));
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

__global__ void __launch_bounds__(THREADS, 1) gmm_em_lse_kernel(const Args a) { logit_pass<kEpiLse>(a); }

template <int kEpi>
__global__ void __launch_bounds__(THREADS, 1) gmm_em_post_kernel(const Args a) { logit_pass<kEpi>(a); }

// label partials -> out_label: thread == padded frame; partial slots ascend with the component index, so strict > keeps
// the lowest index of a tie
__global__ void __launch_bounds__(256) em_label_merge_kernel(const Args a) {
  const int64_t n_rows = ((a.blk_start[a.n_segs] + 1) & ~(int64_t)1) * BLK;
  const int n_part = 2 * a.n_tiles;
  for (int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x; p < n_rows; p += (int64_t)gridDim.x * 256) {
    const int64_t b = p >> 6;
    const int r = (int)(p & 63);
    if (r >= __ldg(a.blk_nt + b)) continue;
    const float2 q0 = __ldg(a.partial + p);
    float bm = q0.x, bi = q0.y;
#pragma unroll 4
    for (int y = 1; y < n_part; ++y) {
      const float2 q = __ldg(a.partial + (size_t)y * a.P + p);
      if (q.x > bm) { bm = q.x; bi = q.y; }
    }
    a.out_label[__ldg(a.blk_t0 + b) + r] = __float_as_int(bi);
  }
}

// partials -> lse2 per padded frame, frame_lse per frame, log-likelihood per segment.  Persistent CTAs walk groups of 4
// blocks; the partials of a frame are loaded in one batch (independent loads in flight) and merged from registers.  A thread
// carries the log-likelihood of its frames until the segment changes, so a UBM iteration (one segment) ends in a few
// thousand double atomics on its address -- one per warp and 32 frames, as before, was 1.1 M serialised L2 atomics at
// config 3 and most of this kernel's 2.6 ms.
__global__ void __launch_bounds__(256) em_merge_kernel(const Args a) {
  const int64_t nb = a.blk_start[a.n_segs];
  const int64_t nb2 = (nb + 1) & ~(int64_t)1;
  const int r = threadIdx.x & 63, lane = threadIdx.x & 31;
  double acc = 0.0;
  int seg_acc = -1;
  auto flush = [&]() {   // warp-uniform: the 32 lanes of a warp share a block, hence a segment
    double tot = acc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    if (lane == 0 && seg_acc >= 0 && tot != 0.0 && a.out_loglik) atomicAdd(a.out_loglik + seg_acc, tot);
    acc = 0.0;
  };
  for (int64_t b = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 6); b < nb2; b += (int64_t)gridDim.x * 4) {
    const int nt = a.blk_nt[b];
    const int seg = a.blk_seg[b];
    const int64_t p = b * BLK + r;
    float lse2 = 3.0e38f, ll = 0.f;  // dead rows: gamma = 2^(x - huge) = 0
    if (r < nt) {
      const int n_part = 2 * a.n_tiles;
      float m = -3.0e38f, s = 0.f;
      for (int y0 = 0; y0 < n_part; y0 += 8) {
        float2 q[8];
#pragma unroll
        for (int y = 0; y < 8; ++y) q[y] = y0 + y < n_part ? __ldg(a.partial + (size_t)(y0 + y) * a.P + p) : make_float2(-3.0e38f, 0.f);
        float mg = m;
#pragma unroll
        for (int y = 0; y < 8; ++y) mg = fmaxf(mg, q[y].x);
        s *= ex2(m - mg);
#pragma unroll
        for (int y = 0; y < 8; ++y) s += q[y].y * ex2(q[y].x - mg);
        m = mg;
      }
      lse2 = m + lg2(s);
      ll = lse2 * 0.69314718055994530942f;
      if (a.frame_lse) a.frame_lse[a.blk_t0[b] + r] = ll;
    }
    a.lse2[p] = lse2 < 1.0e38f ? lse2 - 12.f : lse2;   // log2(kGammaScale) = 12
    if (seg != seg_acc) {
      flush();
      seg_acc = seg;
    }
    acc += (double)ll;
  }
  flush();
}

// ================================================================================================ pass STATS
// grid = (block chunks, tile pairs).  Shared memory: the pair's model tiles, a ring of NF (Fb half image + 64 lse values)
// stages for the logit GEMM and a ring of NX Xt images for the statistics GEMM; tensor memory: logits / gamma
// [tile][buffer] 64 columns each, statistics [tile] KDb columns.  Tensor-pipe order per step k: GEMM1(k) (logits),
// GEMM2(k - 1) (statistics); both rings are released by the completion of GEMM2(k), so the loads of step k + 1 are
// issued two GEMMs before they are needed.
namespace p3 {
// ring depths, measured at config 3 (ms per statistics call, three runs each on one box; single runs scatter by up to 5 ms):
// (NF, NX) = (3, 2) 21.6 / 21.6 / 22.6, (4, 3) 21.5 / 21.3 / 21.1, (3, 4) 21.0 / 20.8 -- the FP16 Xt images freed the shared
// memory for the deeper Xt ring
constexpr int NF = 3, NX = 4;
constexpr uint32_t COL_LOGIT = 0;    // + 64 * (2 * tile + buffer)
constexpr uint32_t COL_STAT = 256;   // + KDb * tile
constexpr int CTRL = 96;             // warp 0: producer; warps 1, 2: MMA issuers of tile 0 / tile 1 (a step's MMAs are 32-40
                                     // tensor cycles each: one issuing lane cannot keep up with two tiles)
constexpr int THREADS_S = CTRL + EPI;
}

template <int KSTEPS>
__global__ void __launch_bounds__(p3::THREADS_S, 1) gmm_em_stats_kernel(const Args a) {
  using namespace p3;
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int KDb = KSTEPS * 16;
  const int D = a.D;
  constexpr uint32_t TB = 512u * (uint32_t)KDb;  // model tile image
  constexpr uint32_t XB = 256u * (uint32_t)KDb;  // Xt image of a step (FP16 hi + lo)
  constexpr uint32_t FB = TB >> 1;               // the 64-row half of an Fb image (hi + lo)
  constexpr uint32_t FST = FB + 256u;            // F stage: + 64 lse values
  unsigned char* sB = smem;                      // [2][TB]
  unsigned char* sF = smem + 2 * (size_t)TB;     // [NF][FST]
  unsigned char* sX = sF + (size_t)NF * FST;     // [NX][XB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sX + (size_t)NX * XB);
  uint64_t* b_full = bars;           // model tiles landed
  uint64_t* f_full = bars + 1;       // [NF]
  uint64_t* f_empty = f_full + NF;   // [NF] the statistics GEMMs of the step are complete (its lse values are dead too)
  uint64_t* x_full = f_empty + NF;   // [NX]
  uint64_t* x_empty = x_full + NX;   // [NX]
  uint64_t* l_full = x_empty + NX;   // [4] logits of (tile, buffer) are in TMEM
  uint64_t* g_full = l_full + 4;     // [4] gamma of (tile, buffer) is in TMEM
  uint64_t* st_done = g_full + 4;    // [2] per tile: every statistics GEMM issued so far is complete
  uint64_t* drained = st_done + 2;   // [2] per tile: the accumulator has been read out after a segment end
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tile0 = 2 * blockIdx.y;
  const int ntl = min(2, a.n_tiles - tile0);
  if (tid == 0) {
    mbar_init(b_full, 1);
    for (int i = 0; i < NF; ++i) { mbar_init(f_full + i, 1); mbar_init(f_empty + i, (uint32_t)ntl); }
    for (int i = 0; i < NX; ++i) { mbar_init(x_full + i, 1); mbar_init(x_empty + i, (uint32_t)ntl); }
    for (int i = 0; i < 4; ++i) { mbar_init(l_full + i, 1); mbar_init(g_full + i, EPI / 2); }
    for (int i = 0; i < 2; ++i) { mbar_init(st_done + i, 1); mbar_init(drained + i, EPI / 2); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // blocks of this CTA: a chunk of all blocks, or (per-segment models) a chunk of the blocks of segment blockIdx.z
  int64_t blk_lo = 0, blk_hi = a.blk_start[a.n_segs];
  const unsigned char* tiles = a.tiles;
  if (a.per_seg_model) {
    blk_lo = a.blk_start[blockIdx.z];
    blk_hi = a.blk_start[blockIdx.z + 1];
    tiles += (size_t)blockIdx.z * a.n_tiles * TB;
  }
  const int64_t per = (blk_hi - blk_lo + gridDim.x - 1) / gridDim.x;
  const int64_t b0 = blk_lo + (int64_t)blockIdx.x * per, b1 = min(b0 + per, blk_hi);

  if (warp == 0) {
    // ===================== producer =====================
    if (b0 < b1) {
      if (elect_one()) {
        mbar_arrive_expect_tx(b_full, (uint32_t)ntl * TB);
        for (int t = 0; t < ntl; ++t) bulk_g2s(sB + (size_t)t * TB, tiles + (size_t)(tile0 + t) * TB, TB, b_full);
      }
      __syncwarp();
      constexpr int n_pieces = 2 * (KDb >> 3);  // (hi | lo) x chunk: 1 KB each, 64 rows x 16 B out of a 128-row chunk
      uint32_t k = 0;
      for (int64_t b = b0; b < b1; ++b, ++k) {
        const uint32_t fs = k % NF, xs = k % NX;
        mbar_wait_relaxed(f_empty + fs, ((k / NF) & 1u) ^ 1u);
        unsigned char* dst = sF + (size_t)fs * FST;
        if (lane == 0) mbar_arrive_expect_tx(f_full + fs, FST);
        __syncwarp();
        const unsigned char* img = a.fb + (size_t)(b >> 1) * TB + (size_t)(b & 1) * (BLK * 16);
        for (int pc = lane; pc < n_pieces; pc += 32) bulk_g2s(dst + (size_t)pc * 1024, img + (size_t)pc * 2048, 1024u, f_full + fs);
        if (lane == 31) bulk_g2s(dst + FB, a.lse2 + b * BLK, 256u, f_full + fs);
        __syncwarp();
        mbar_wait_relaxed(x_empty + xs, ((k / NX) & 1u) ^ 1u);
        if (elect_one()) {
          mbar_arrive_expect_tx(x_full + xs, XB);
          bulk_g2s(sX + (size_t)xs * XB, a.xt + (size_t)b * XB, XB, x_full + xs);
        }
        __syncwarp();
      }
    }
  } else if (warp < CTRL / 32) {
    // ===================== MMA issuer of tile t =====================
    const int t = warp - 1;
    if (t < ntl && b0 < b1) {
      constexpr uint32_t sbo = 128u;
      constexpr uint32_t lbo_b = BN * 16u, lbo_f = BLK * 16u, lbo_x = (uint32_t)KDb * 16u;
      constexpr uint32_t ks_b = (2u * lbo_b) >> 4, ks_f = (2u * lbo_f) >> 4, ks_x = (2u * lbo_x) >> 4;
      constexpr uint32_t idesc1 = make_idesc_bf16(BN, BLK);
      constexpr uint32_t idesc2 = make_idesc_f16(BN, KDb);
      const uint32_t sF_u = smem_u32(sF), sX_u = smem_u32(sX);
      const uint64_t bh = make_desc(smem_u32(sB) + (uint32_t)t * TB, lbo_b, sbo), bl = bh + (uint64_t)((TB >> 1) >> 4);
      const uint32_t t_stat = tmem_base + COL_STAT + (uint32_t)(t * KDb);
      mbar_wait_relaxed(b_full, 0);
      bool pending_drain = false;
      uint32_t n_drains = 0;
      // statistics GEMM of step p: stats += gamma (TMEM, in the logit columns of buffer p & 1) . Xt (stage p % NX)
      auto gemm2 = [&](uint32_t p, bool first, bool flush) {
        const uint32_t xs = p % NX, lb = 2u * (uint32_t)t + (p & 1u);
        mbar_wait_relaxed(x_full + xs, (p / NX) & 1u);
        mbar_wait_relaxed(g_full + lb, (p >> 1) & 1u);
        if (pending_drain) {
          mbar_wait_relaxed(drained + t, n_drains & 1u);
          ++n_drains;
          pending_drain = false;
        }
        tc_fence_after();
        if (elect_one()) {
          const uint64_t xhi = make_desc(sX_u + xs * XB, lbo_x, sbo), xlo = xhi + (uint64_t)((XB >> 1) >> 4);
          const uint32_t t_gam = tmem_base + COL_LOGIT + 64u * lb;
          // K = 16 frames per MMA; the gamma of frames [32 h, 32 h + 32) sits packed in columns [32 h, 32 h + 16) of the buffer
#pragma unroll
          for (int q = 0; q < BLK / 16; ++q)
            mma_f16_ts(t_stat, t_gam + 32u * (q >> 1) + 8u * (q & 1), xhi + (uint64_t)(q * ks_x), idesc2, (first && q == 0) ? 0u : 1u);
          // the residual (lo) FP16 piece of the frames too: leaving it out saves 4 of 23 MMAs per step (19.7 vs 21.0 ms per
          // call at config 3), but the 11-bit x and x^2 cancel in S/N - mean^2: variances off by up to 60 % in
          // test_em_trajectory_matches_sklearn
#pragma unroll
          for (int q = 0; q < BLK / 16; ++q)
            mma_f16_ts(t_stat, t_gam + 32u * (q >> 1) + 8u * (q & 1), xlo + (uint64_t)(q * ks_x), idesc2, 1u);
          if (flush) tc_commit(st_done + t);
          tc_commit(f_empty + p % NF);
          tc_commit(x_empty + xs);
        }
        __syncwarp();
        pending_drain = flush;
      };
      uint32_t k = 0;
      bool prev_first = true, prev_flush = false;
      int seg_cur = a.blk_seg[b0];
      bool first_in_seg = true;
      for (int64_t b = b0; b < b1; ++b, ++k) {
        const int seg_next = (b + 1 < b1) ? __ldg(a.blk_seg + b + 1) : -2;  // issued early, used at the bottom
        const uint32_t fs = k % NF, lb = 2u * (uint32_t)t + (k & 1u);
        mbar_wait_relaxed(f_full + fs, (k / NF) & 1u);
        tc_fence_after();
        // the logit buffer (t, k & 1) was last read by the statistics GEMM of step k - 2, issued before this one
        if (elect_one()) {
          const uint64_t fh = make_desc(sF_u + fs * FST, lbo_f, sbo), fl = fh + (uint64_t)((FB >> 1) >> 4);
          const uint32_t d = tmem_base + COL_LOGIT + 64u * lb;
#pragma unroll
          for (int q = 0; q < KSTEPS; ++q) mma_bf16_ss(d, bh + (uint64_t)(q * ks_b), fh + (uint64_t)(q * ks_f), idesc1, q > 0 ? 1u : 0u);
#pragma unroll
          for (int q = 0; q < KSTEPS; ++q) mma_bf16_ss(d, bh + (uint64_t)(q * ks_b), fl + (uint64_t)(q * ks_f), idesc1, 1u);
#pragma unroll
          for (int q = 0; q < KSTEPS; ++q) mma_bf16_ss(d, bl + (uint64_t)(q * ks_b), fh + (uint64_t)(q * ks_f), idesc1, 1u);
          tc_commit(l_full + lb);
        }
        __syncwarp();
        if (k > 0) gemm2(k - 1, prev_first, prev_flush);
        prev_first = first_in_seg;
        prev_flush = seg_next != seg_cur;
        first_in_seg = prev_flush;
        seg_cur = seg_next;
      }
      gemm2(k - 1, prev_first, prev_flush);
    }
  } else {
    // ===================== epilogue: thread == (component row, 32 of a step's 64 frames) =====================
    const int ew = warp - CTRL / 32;
    const int t = ew >> 3, cq = (ew >> 2) & 1, quad = warp & 3;
    const int row = quad * 32 + lane;  // TMEM lane == component row within the tile
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    if (t < ntl && b0 < b1) {
      const int comp = (tile0 + t) * BN + row;
      uint32_t k = 0, n_flush = 0;
      int seg_cur = a.blk_seg[b0];
      for (int64_t b = b0; b < b1; ++b, ++k) {
        const int seg_next = (b + 1 < b1) ? __ldg(a.blk_seg + b + 1) : -2;  // issued early, used at the bottom
        const uint32_t fs = k % NF, lb = 2u * (uint32_t)t + (k & 1u);
        mbar_wait(f_full + fs, (k / NF) & 1u);   // the stage's lse values (written by the bulk copy) are visible
        const float* lse = reinterpret_cast<const float*>(sF + (size_t)fs * FST + FB) + 32 * cq;
        float4 ls[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) ls[q] = *reinterpret_cast<const float4*>(lse + 4 * q);
        mbar_wait(l_full + lb, (k >> 1) & 1u);
        tc_fence_after();
        const uint32_t t_log = tmem_base + lane_addr + COL_LOGIT + 64u * lb + 32u * (uint32_t)cq;
        uint32_t r[32];
        tc_ld32_issue(t_log, r);
        tc_ld_wait(r);
        // gamma * 2^12 (the scale is folded into lse2) as FP16, two frames per column over this thread's own logits
        uint32_t gam[16];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const __half2 g0 = __floats2half2_rn(ex2(__uint_as_float(r[4 * q + 0]) - ls[q].x), ex2(__uint_as_float(r[4 * q + 1]) - ls[q].y));
          const __half2 g1 = __floats2half2_rn(ex2(__uint_as_float(r[4 * q + 2]) - ls[q].z), ex2(__uint_as_float(r[4 * q + 3]) - ls[q].w));
          gam[2 * q] = *reinterpret_cast<const uint32_t*>(&g0);
          gam[2 * q + 1] = *reinterpret_cast<const uint32_t*>(&g1);
        }
        tc_st16u(t_log, gam);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        mbar_arrive(g_full + lb);
        if (seg_next != seg_cur) {
          // last step of a segment inside this chunk: wait for its statistics GEMMs, add the accumulator to the outputs
          mbar_wait(st_done + t, n_flush & 1u);
          ++n_flush;
          tc_fence_after();
          const uint32_t saddr = tmem_base + lane_addr + COL_STAT + (uint32_t)(t * KDb);
          constexpr int half_cols = KDb >> 1;  // a multiple of 8
#pragma unroll 1
          for (int c0 = cq * half_cols; c0 < (cq + 1) * half_cols; c0 += 8) {
            uint32_t s8[8];
            tc_ld8(saddr + c0, s8);
            if (comp < a.K) {
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                const int jj = c0 + e;
                const double v = (double)__uint_as_float(s8[e]) * (1.0 / (double)kGammaScale);
                if (jj < D) atomicAdd(a.out_f + ((int64_t)seg_cur * a.K + comp) * D + jj, v);
                else if (jj < 2 * D) atomicAdd(a.out_s + ((int64_t)seg_cur * a.K + comp) * D + (jj - D), v);
                else if (jj == 2 * D) atomicAdd(a.out_n + (int64_t)seg_cur * a.K + comp, v);
              }
            }
          }
          tc_fence_before();
          mbar_arrive(drained + t);
        }
        seg_cur = seg_next;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

}  // namespace em

bool stats_tc_supported(const PackLayout& L) { return L.KD <= em::MAX_KD && L.off_tile_bf != 0; }

int64_t stats_tc_workspace_bytes(const PackLayout& L, int64_t total_frames, int64_t n_segs) {
  return stats_tc_supported(L) ? (int64_t)em::ws_layout(L, total_frames, n_segs).bytes : 0;
}

static int g_num_sms = 0;
static int query_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    SSP_CUDA_OK(cudaGetDevice(&dev));
    SSP_CUDA_OK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  return SSP_OK;
}

// Arguments shared by the statistics and posterior calls: the workspace carve-up (images at the same place for both) and
// the model.  Outputs are left NULL.
static em::Args em_args(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames, const void* pack,
                        const PackLayout& L, const em::Ws& w, void* workspace) {
  using namespace em;
  unsigned char* base = (unsigned char*)workspace;
  Args a = {};
  a.feats = feats;
  a.seg = seg_offsets;
  a.n_segs = n_segs;
  a.total_frames = total_frames;
  a.blk_start = (int64_t*)(base + w.o_blk_start);
  a.blk_seg = (int32_t*)(base + w.o_blk_seg);
  a.blk_t0 = (int64_t*)(base + w.o_blk_t0);
  a.blk_nt = (int32_t*)(base + w.o_blk_nt);
  a.lse2 = (float*)(base + w.o_lse2);
  a.partial = (float2*)(base + w.o_partial);
  a.fb = base + w.o_fb;
  a.xt = base + w.o_xt;
  a.nb_max = w.nb_max;
  a.P = w.P;
  a.tiles = (const unsigned char*)pack + L.off_tile_bf;
  a.K = L.K;
  a.D = L.D;
  a.KDb = w.KDb;
  a.n_tiles = L.Kp / BN;
  a.per_seg_model = L.n_models > 1 ? 1 : 0;
  return a;
}

// grids of the passes: the number of blocks is a device value (segment padding); size them from its host-side bounds
struct EmGrid {
  int n_pairs;
  unsigned gz;
  int64_t gx_l, gx_s;  // image chunks of the logit passes, block chunks of the statistics pass
  size_t smem_lse;
};
static int em_grid(const em::Args& a, const em::Ws& w, int64_t n_segs, int64_t total_frames, const char* who, EmGrid* g) {
  using namespace em;
  const int rc = query_sms();
  if (rc != SSP_OK) return rc;
  const int sms = g_num_sms;
  g->n_pairs = (a.n_tiles + 1) / 2;
  const int64_t nb_lo = (total_frames + BLK - 1) / BLK;
  g->gz = a.per_seg_model ? (unsigned)n_segs : 1u;
  SSP_REQUIRE(!a.per_seg_model || n_segs <= 65535, "%s: %lld per-segment models (at most 65535)", who, (long long)n_segs);
  int64_t gx = sms / ((int64_t)g->n_pairs * g->gz);
  if (gx < 1) gx = 1;
  g->gx_l = min(gx, (nb_lo + 1) / 2);
  g->gx_s = min(gx, nb_lo);
  g->smem_lse = (2 + NS_L) * w.img_bytes() + 16 * sizeof(uint64_t) + 64;
  return SSP_OK;
}

// plan + images (skipped on reuse), then the LSE pass and the merge: lse2 per padded frame (+ frame_lse / loglik if set)
static int em_prepare_and_lse(em::Args& a, const em::Ws& w, const EmGrid& g, bool reuse_images, bool lse, cudaStream_t st) {
  using namespace em;
  if (!reuse_images) {
    em_plan_kernel<<<1, 1024, 0, st>>>(a);
    SSP_LAUNCH_CHECK("em_plan_kernel");
    em_prep_kernel<<<(unsigned)w.nb_max, 256, 0, st>>>(a);
    SSP_LAUNCH_CHECK("em_prep_kernel");
  }
  if (!lse) return SSP_OK;
  SSP_CUDA_OK(cudaFuncSetAttribute(gmm_em_lse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem_lse));
  gmm_em_lse_kernel<<<dim3((unsigned)g.gx_l, (unsigned)g.n_pairs, g.gz), THREADS, g.smem_lse, st>>>(a);
  SSP_LAUNCH_CHECK("gmm_em_lse_kernel");
  {
    const int64_t groups = (w.nb_max + 3) / 4, cap = 8 * (int64_t)g_num_sms;
    em_merge_kernel<<<(unsigned)(groups < cap ? groups : cap), 256, 0, st>>>(a);
  }
  SSP_LAUNCH_CHECK("em_merge_kernel");
  return SSP_OK;
}

int launch_stats_tc(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames, const void* pack,
                    const PackLayout& L, float* frame_lse, double* out_n, double* out_f, double* out_s, double* out_loglik,
                    void* workspace, bool reuse_images, cudaStream_t st) {
  using namespace em;
  SSP_CUDA_OK(cudaMemsetAsync(out_loglik, 0, sizeof(double) * n_segs, st));
  if (total_frames == 0) return SSP_OK;
  const Ws w = ws_layout(L, total_frames, n_segs);
  Args a = em_args(feats, seg_offsets, n_segs, total_frames, pack, L, w, workspace);
  a.frame_lse = frame_lse;
  a.out_n = out_n;
  a.out_f = out_f;
  a.out_s = out_s;
  a.out_loglik = out_loglik;
  EmGrid g;
  int rc = em_grid(a, w, n_segs, total_frames, "ssp_gmm_stats", &g);
  if (rc != SSP_OK) return rc;
  rc = em_prepare_and_lse(a, w, g, reuse_images, true, st);
  if (rc != SSP_OK) return rc;
  const size_t TB = w.img_bytes();
  const size_t smem_stats = 2 * TB + p3::NF * (TB / 2 + 256) + p3::NX * (TB / 2) + (13 + 2 * p3::NF + 2 * p3::NX) * sizeof(uint64_t) + 64;
#define SSP_EM_STATS(ks)                                                                                                  \
  case ks:                                                                                                                \
    SSP_CUDA_OK(cudaFuncSetAttribute(gmm_em_stats_kernel<ks>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_stats)); \
    gmm_em_stats_kernel<ks><<<dim3((unsigned)g.gx_s, (unsigned)g.n_pairs, g.gz), p3::THREADS_S, smem_stats, st>>>(a);   \
    break;
  switch (w.KDb >> 4) {
    SSP_EM_STATS(1) SSP_EM_STATS(2) SSP_EM_STATS(3) SSP_EM_STATS(4) SSP_EM_STATS(5)
    default: SSP_REQUIRE(false, "ssp_gmm_stats: contraction length %d", w.KDb);
  }
#undef SSP_EM_STATS
  SSP_LAUNCH_CHECK("gmm_em_stats_kernel");
  return SSP_OK;
}

int launch_posteriors_tc(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames, const void* pack,
                         const PackLayout& L, float* out_resp, int64_t* out_label, float* out_frame_lse, void* workspace,
                         bool reuse_images, cudaStream_t st) {
  using namespace em;
  if (total_frames == 0) return SSP_OK;
  const Ws w = ws_layout(L, total_frames, n_segs);
  Args a = em_args(feats, seg_offsets, n_segs, total_frames, pack, L, w, workspace);
  a.frame_lse = out_frame_lse;
  a.out_resp = out_resp;
  a.out_label = out_label;
  a.resp_vec = (L.K % 4 == 0 && ((uintptr_t)out_resp & 15) == 0) ? 1 : 0;
  EmGrid g;
  int rc = em_grid(a, w, n_segs, total_frames, "ssp_gmm_posteriors", &g);
  if (rc != SSP_OK) return rc;
  // labels alone need no log-sum-exp: the argmax of the logits is the argmax of the posteriors
  rc = em_prepare_and_lse(a, w, g, reuse_images, out_resp || out_frame_lse, st);
  if (rc != SSP_OK) return rc;
  if (!out_resp && !out_label) return SSP_OK;
  const dim3 grid((unsigned)g.gx_l, (unsigned)g.n_pairs, g.gz);
#define SSP_EM_POST(epi, name)                                                                                          \
  SSP_CUDA_OK(cudaFuncSetAttribute(gmm_em_post_kernel<epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem_lse)); \
  gmm_em_post_kernel<epi><<<grid, THREADS, g.smem_lse, st>>>(a);                                                        \
  SSP_LAUNCH_CHECK(name);
  if (out_resp && out_label) {
    SSP_EM_POST(kEpiResp | kEpiLabel, "gmm_em_post_kernel<resp+labels>")
  } else if (out_resp) {
    SSP_EM_POST(kEpiResp, "gmm_em_post_kernel<resp>")
  } else {
    SSP_EM_POST(kEpiLabel, "gmm_em_post_kernel<labels>")
  }
#undef SSP_EM_POST
  if (out_label) {
    const int64_t blocks = (w.P + 255) / 256, cap = 8 * (int64_t)g_num_sms;
    em_label_merge_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(a);
    SSP_LAUNCH_CHECK("em_label_merge_kernel");
  }
  return SSP_OK;
}

}  // namespace ssp
