// GMM-UBM scoring on the 5th-generation tensor cores (sm_100a, tcgen05 + TMEM + TMA bulk copies).
//
// The diagonal-Gaussian log-likelihood (sklearn _gaussian_mixture.py:536-553) is the dense contraction
//     L2[t, c] = [x_t, x_t^2, 1, 1] . [mu_c/var_c, -1/(2 var_c), c_hi, c_lo] * log2(e)
// with frames as M, (model, component) as N and 2D+2 as the K dimension.  One persistent CTA per SM owns
// 256 frames at a time ("unit"): the frames' [x, x^2, 1, 1] rows are rounded to TF32 (cvt.rna) and laid
// out ONCE in shared memory as two 128-row UMMA operands, then every model's component tiles (pre-packed
// as shared-memory images by gmm_pack_kernel) stream through a 3-stage cp.async.bulk ring.  All CTAs walk
// the same tile sequence, so each tile is read from HBM once per wave and served to the other SMs by L2.
//
//   warp 0      : producer   - one lane issues cp.async.bulk (global -> smem) + mbarrier expect_tx
//   warp 1      : MMA issuer - the warp walks the tile loop uniformly, one elected lane issues tcgen05.mma
//                 kind::tf32 (M128 x N128 x K8) into 4 TMEM slots (descriptors stay in uniform registers;
//                 a divergent single-lane loop cost ~135 cycles per 64-cycle MMA), tcgen05.commit signals
//                 "slot full" / "stage free"
//   warps 2..17 : epilogue   - 4 warps per SM sub-partition (2 row blocks x 2 column halves x 4 TMEM lane
//                 quadrants); tcgen05.ld 32 lanes x 32 columns; thread == (frame row, 64 columns); sum of
//                 2^(x - stabiliser) across a model's tiles (MUFU ex2 + a small FMA-pipe polynomial share),
//                 the two column halves merged through shared memory -> per-frame log-likelihood ->
//                 warp-segmented per-utterance sum -> one double atomic per (warp, utterance, model).
//                 The T x K logits never leave the SM.
//
// The log-constant rides through the MMA as two TF32-exact pieces (c_hi + c_lo) against A columns of 1.0,
// so the epilogue is max / ex2 / add only.
#include <cuda_fp16.h>

#include <mutex>
#include <unordered_map>

#include "tc_common.cuh"

namespace ssp {

namespace tc {
constexpr int BM = 128;      // rows per accumulator (TMEM lanes)
constexpr int BN = kTileN;   // components per tile
constexpr int NSTAGE = 3;
constexpr int NSLOT = 4;     // TMEM accumulator slots (BN fp32 columns each) = all 512 columns
constexpr int MAX_KD = 80;
// Precision rungs (SURVEY section 7 ladder), all FP32 accumulation in TMEM:
//   NPARTS 1: A_hi.B_hi                       single-pass TF32, 1e-4 relative at the named workloads (K >= 512)
//   NPARTS 2: + A_hi.B_lo                     model side exact to 2^-22 (the systematic part of the error)
//   NPARTS 3: + A_lo.B_hi                     FP32-grade (3xTF32): frame side split as well
// MB = row blocks of 128 frames per unit: 2 (16 epilogue warps: 4 per SM sub-partition = two row blocks x two 64-column
// halves x four lane quadrants), or 1 for the 3-part rung, whose A_lo operand takes the second row block's shared
// memory (8 epilogue warps).
constexpr int threads_of(int mb) { return 64 + 8 * mb * 32; }
// Measured on B200 under the 1 kW cap (10k utts x 1001 models): pairs 0/2/4/6/8 -> 523/539/526/496/486 TFLOP/s.
// The kernel is power-bound, not pipe-bound: a MUFU ex2 costs less energy than the ~7 FMA-pipe instructions that
// replace it, so only a small share is worth moving.
constexpr int kPolyPairs = 2;

// Sum of 2^(v - m_stab) over 32 accumulator columns of one row, plus their maximum.
//
// m_stab is a stabiliser chosen BEFORE the tile is seen (the previous model's maximum for this frame: speaker
// models adapted from one UBM peak within a few units of each other), so the exponentials do not depend on the
// tile's own maximum and the whole tile is one dependency-free instruction stream; the caller checks the
// maximum afterwards and redoes the tile on the (rare) rows where the stabiliser was off by more than 2^64.
//
// The MUFU (16 ex2/clk/SM) would otherwise be the binding pipe, so kPolyPairs of the 16 column pairs are
// evaluated on the FMA pipe: 2^x = 2^n * p(f), n = round(x) via the 1.5*2^23 magic add, f = x - n in
// [-0.5, 0.5], p = degree-4 minimax polynomial (max relative error 2.7e-6), 2^n applied by adding n to the
// exponent field.  Packed FADD2 / FFMA2 halve the issue slots; FMNMX3 halves the max chain.
__device__ __forceinline__ void chunk_sum(const uint32_t (&r)[32], float m_stab, float2& accp, float2& accm0, float2& accm1,
                                          float& cmax) {
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
  float cm = max3(v[0], v[1], v[2]);
#pragma unroll
  for (int i = 3; i < 31; i += 2) cm = max3(cm, v[i], v[i + 1]);
  cmax = max3(cmax, cm, v[31]);
  const float2 nm = make_float2(-m_stab, -m_stab);
  const float MAGIC = 12582912.f;  // 1.5 * 2^23
  const float2 mg = make_float2(MAGIC, MAGIC), nmg = make_float2(-MAGIC, -MAGIC), neg1 = make_float2(-1.f, -1.f);
  const float2 c0 = make_float2(0.9999992847442627f, 0.9999992847442627f);
  const float2 c1 = make_float2(0.6931218504905701f, 0.6931218504905701f);
  const float2 c2 = make_float2(0.240247443318367f, 0.240247443318367f);
  const float2 c3 = make_float2(0.05591766536235809f, 0.05591766536235809f);
  const float2 c4 = make_float2(0.009570018388330936f, 0.009570018388330936f);
#pragma unroll
  for (int i = 0; i < kPolyPairs; ++i) {
    float2 d = __fadd2_rn(make_float2(v[2 * i], v[2 * i + 1]), nm);
    d.x = fmaxf(d.x, -126.f);
    d.y = fmaxf(d.y, -126.f);
    const float2 t = __fadd2_rn(d, mg);
    const float2 nn = __fadd2_rn(t, nmg);
    const float2 f = __ffma2_rn(nn, neg1, d);
    float2 p = __ffma2_rn(c4, f, c3);
    p = __ffma2_rn(p, f, c2);
    p = __ffma2_rn(p, f, c1);
    p = __ffma2_rn(p, f, c0);
    float2 e;
    e.x = __uint_as_float(__float_as_uint(p.x) + (__float_as_uint(t.x) << 23));
    e.y = __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(t.y) << 23));
    accp = __fadd2_rn(accp, e);
  }
  static_assert(kPolyPairs % 2 == 0 && kPolyPairs <= 16, "pairs are consumed two at a time");
#pragma unroll
  for (int i = kPolyPairs; i < 16; i += 2) {
    const float2 d0 = __fadd2_rn(make_float2(v[2 * i], v[2 * i + 1]), nm);
    const float2 d1 = __fadd2_rn(make_float2(v[2 * i + 2], v[2 * i + 3]), nm);
    accm0 = __fadd2_rn(accm0, make_float2(ex2(d0.x), ex2(d0.y)));
    accm1 = __fadd2_rn(accm1, make_float2(ex2(d1.x), ex2(d1.y)));
  }
}
// plain MUFU version used by the redo path
__device__ __forceinline__ float chunk_sum_exact(const uint32_t (&r)[32], float m) {
  float a0 = 0.f, a1 = 0.f;
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    a0 += ex2(__uint_as_float(r[i]) - m);
    a1 += ex2(__uint_as_float(r[i + 1]) - m);
  }
  return a0 + a1;
}

// cute::UMMA::InstrDescriptor: c_format F32 (1) @4, a/b_format TF32 (2) @7/@10, K-major A and B,
// n_dim = N>>3 @17, m_dim = M>>4 @24.
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

struct Args {
  const float* feats;
  const int64_t* offsets;
  int64_t n_utts, total_frames;
  const float* tiles;  // [n_models][Kp/BN][KD/4][BN] float4 images
  const float* tiles_lo;  // residual images (same layout), parts 2 and 3
  int n_models, tiles_per_model, D, KD;
  int normalize;
  double* scores;
  float* frame_lse;
};

// kH: FP16 operands (kind::f16, K = 16 per MMA: half the MMA instructions, half the bytes of a model tile and of the frame
// operand; an FP16 significand has TF32's 11 bits, so every rung keeps its error).  a.KD is then the FP16 contraction length.
template <int MB, int NPARTS, bool kH>
__global__ void __launch_bounds__(threads_of(MB), 1) gmm_score_tc_kernel(const Args a) {
  static_assert(NPARTS >= 1 && NPARTS <= 3 && (MB == 1 || MB == 2) && (NPARTS < 3 || MB == 1), "see the rung table");
  constexpr uint32_t ELT = kH ? 2u : 4u;
  constexpr int UNIT = BM * MB, EPI_WARPS = 8 * MB;
  constexpr int A_IMAGES = MB * (NPARTS == 3 ? 2 : 1);  // hi images of every row block, then the lo images
  extern __shared__ __align__(1024) unsigned char smem[];
  const int KD = a.KD;
  const uint32_t tile_bytes = (uint32_t)BN * KD * ELT;
  float* sA = reinterpret_cast<float*>(smem);                     // [A_IMAGES][KC][BM][4]   (kH: [KD/8][BM][8] half)
  unsigned char* sB = smem + (size_t)A_IMAGES * tile_bytes;       // [NSTAGE][KC][BN][4]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + (size_t)NSTAGE * tile_bytes);
  uint64_t* b_full = bars;
  uint64_t* b_empty = bars + NSTAGE;
  uint64_t* t_full = bars + 2 * NSTAGE;
  uint64_t* t_empty = t_full + NSLOT;
  uint64_t* a_full = t_empty + NSLOT;
  uint64_t* a_empty = a_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_empty + 1);
  float2* comb = reinterpret_cast<float2*>(tmem_slot + 4);  // [model parity][row block][row]: (m, s) of column half 1

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < NSTAGE; ++i) { mbar_init(b_full + i, 1); mbar_init(b_empty + i, 1); }
    for (int i = 0; i < NSLOT; ++i) { mbar_init(t_full + i, 1); mbar_init(t_empty + i, 2 * BM); }
    mbar_init(a_full, EPI_WARPS * 32);
    mbar_init(a_empty, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)(NSLOT * BN))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t n_units = (a.total_frames + UNIT - 1) / UNIT;
  const int tiles_per_unit = a.n_models * a.tiles_per_model;
  const size_t tile_floats = (size_t)BN * KD;

  if (warp == 0) {
    // ===================== producer: stream every model's tiles, once per unit =====================
    uint32_t it = 0;
    for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x) {
      for (int t = 0; t < tiles_per_unit; ++t) {
#pragma unroll
        for (int part = 0; part < (NPARTS >= 2 ? 2 : 1); ++part, ++it) {  // the hi image, then the residual image
          const uint32_t stage = it % NSTAGE, ph = (it / NSTAGE) & 1u;
          mbar_wait(b_empty + stage, ph ^ 1u);
          if (elect_one()) {
            mbar_arrive_expect_tx(b_full + stage, tile_bytes);
            bulk_g2s(sB + (size_t)stage * tile_bytes,
                     reinterpret_cast<const unsigned char*>(part == 0 ? a.tiles : a.tiles_lo) + (size_t)t * tile_bytes, tile_bytes,
                     b_full + stage);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp walks the loop, one elected lane issues) =====================
    constexpr uint32_t lbo = BM * 16u, sbo = 128u;  // chunk stride = 128 rows x 16 B; 8-row groups are contiguous
    constexpr uint32_t kstep = (2u * lbo) >> 4;      // one K=8 step = two 16-byte chunks, in descriptor address units
    const uint64_t a_desc0 = make_desc(smem_u32(sA), lbo, sbo);
    const uint64_t b_desc0 = make_desc(smem_u32(sB), lbo, sbo);
    const uint32_t tile_units = tile_bytes >> 4;
    const int ksteps = kH ? KD >> 4 : KD >> 3;
    constexpr uint32_t idesc = kH ? make_idesc_f16(BM, BN) : kIdesc;
    uint32_t it = 0, q = 0, unit_idx = 0;
    for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x, ++unit_idx) {
      mbar_wait(a_full, unit_idx & 1u);
      tc_fence_after();
      for (int t = 0; t < tiles_per_unit; ++t) {
        const uint32_t stage = it % NSTAGE, ph = (it / NSTAGE) & 1u;
        mbar_wait(b_full + stage, ph);
        uint32_t stage_lo = 0;
        if (NPARTS >= 2) {
          stage_lo = (it + 1) % NSTAGE;
          mbar_wait(b_full + stage_lo, ((it + 1) / NSTAGE) & 1u);
        }
        it += NPARTS >= 2 ? 2 : 1;
        tc_fence_after();
        const uint64_t bd0 = b_desc0 + (uint64_t)(stage * tile_units), bl0 = b_desc0 + (uint64_t)(stage_lo * tile_units);
#pragma unroll
        for (int mb = 0; mb < MB; ++mb, ++q) {
          const uint32_t slot = q % NSLOT, sph = (q / NSLOT) & 1u;
          mbar_wait(t_empty + slot, sph ^ 1u);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + slot * BN;
          const uint64_t ad0 = a_desc0 + (uint64_t)(mb * tile_units), al0 = a_desc0 + (uint64_t)((MB + mb) * tile_units);
          if (elect_one()) {
            auto mma = [&](uint64_t ad, uint64_t bd, uint32_t acc) {
              if (kH) mma_f16_ss(d_tmem, ad, bd, idesc, acc);
              else tc_mma_tf32(d_tmem, ad, bd, idesc, acc);
            };
            mma(ad0, bd0, 0u);
            for (int k = 1; k < ksteps; ++k) mma(ad0 + (uint64_t)(k * kstep), bd0 + (uint64_t)(k * kstep), 1u);
            if (NPARTS >= 2)
              for (int k = 0; k < ksteps; ++k) mma(ad0 + (uint64_t)(k * kstep), bl0 + (uint64_t)(k * kstep), 1u);
            if (NPARTS == 3)
              for (int k = 0; k < ksteps; ++k) mma(al0 + (uint64_t)(k * kstep), bd0 + (uint64_t)(k * kstep), 1u);
            tc_commit(t_full + slot);
          }
          __syncwarp();
        }
        if (elect_one()) {
          tc_commit(b_empty + stage);
          if (NPARTS >= 2) tc_commit(b_empty + stage_lo);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(a_empty);
      __syncwarp();
    }
  } else {
    // ===================== epilogue warps (also build the A operand) =====================
    const int etid = tid - 64;                 // 0..511
    const int ew = warp - 2;                   // 0..15
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int g = MB == 2 ? (ew >> 2) & 1 : 0;  // row block whose accumulators this thread reads
    const int half = ew >> (MB == 2 ? 3 : 2);  // which 64 of the tile's 128 columns
    const int row = quad * 32 + lane;          // accumulator row within the row block
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    const float LN2 = 0.69314718055994530942f;
    uint32_t n = 0, unit_idx = 0;
    for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x, ++unit_idx) {
      const int64_t frame0 = u * UNIT;
      // ---- A operand: row r of block mb at float index ((mb*KC + j/4)*BM + r)*4 + j%4; two threads per row
      mbar_wait(a_empty, (unit_idx & 1u) ^ 1u);
      {
        const int brow = etid & (UNIT - 1), part = etid / UNIT;
        const int64_t fr = frame0 + brow;
        const bool live = fr < a.total_frames;
        const float* xr = a.feats + fr * a.D;
        float* dst = sA + (size_t)(brow >> 7) * tile_floats + (size_t)(brow & (BM - 1)) * 4;
        __half* dst_h = reinterpret_cast<__half*>(sA) + (size_t)(brow >> 7) * tile_floats + (size_t)(brow & (BM - 1)) * 8;
        const int j0 = part * (KD >> 1), j1 = j0 + (KD >> 1);
        for (int j = j0; j < j1; ++j) {
          float v = 0.f;
          if (j < a.D) v = live ? xr[j] : 0.f;
          else if (j < 2 * a.D) { float x = live ? xr[j - a.D] : 0.f; v = x * x; }
          else if (j < 2 * a.D + 2) v = 1.f;
          if (kH) {   // a frame outside FP16's range gives inf -> NaN scores for its utterance; see launch_score_tc
            const __half h = __float2half_rn(v);
            dst_h[(size_t)(j >> 3) * (BM * 8) + (j & 7)] = h;
            if (NPARTS == 3) dst_h[(size_t)MB * tile_floats + (size_t)(j >> 3) * (BM * 8) + (j & 7)] = __float2half_rn(v - __half2float(h));
            continue;
          }
          const float hi = rna_tf32(v);
          dst[(size_t)(j >> 2) * (BM * 4) + (j & 3)] = hi;
          if (NPARTS == 3) dst[(size_t)MB * tile_floats + (size_t)(j >> 2) * (BM * 4) + (j & 3)] = rna_tf32(v - hi);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(a_full);
      }
      // ---- the frame this thread scores (column half 0 finalises the row)
      const int64_t fe = frame0 + (int64_t)g * BM + row;
      const bool live = fe < a.total_frames;
      int utt = -1;
      float wgt = 1.f;
      if (half == 0) {
        utt = live ? find_segment(a.offsets, a.n_utts, fe) : -1;
        if (utt >= 0 && a.normalize) wgt = 1.f / (float)(a.offsets[utt + 1] - a.offsets[utt]);
      }

      float m_stab = -3.0e38f;  // carried from model to model (see chunk_sum)
      for (int model = 0; model < a.n_models; ++model) {
        float s_run = 0.f;
        for (int t = 0; t < a.tiles_per_model; ++t, ++n) {
          const uint32_t qj = n * MB + (uint32_t)g, slot = qj % NSLOT, ph = (qj / NSLOT) & 1u;
          mbar_wait(t_full + slot, ph);
          tc_fence_after();
          const uint32_t taddr = tmem_base + lane_addr + slot * BN + half * 64;
          uint32_t ra[32], rb[32];
          float2 accp = make_float2(0.f, 0.f), accm0 = make_float2(0.f, 0.f), accm1 = make_float2(0.f, 0.f);
          float cmax = -3.0e38f;
          tc_ld32_issue(taddr, ra);
          tc_ld32_issue(taddr + 32, rb);
          tc_ld_wait2(ra, rb);
          chunk_sum(ra, m_stab, accp, accm0, accm1, cmax);
          chunk_sum(rb, m_stab, accp, accm0, accm1, cmax);
          const float2 tot = __fadd2_rn(__fadd2_rn(accm0, accm1), accp);
          float s_tile = tot.x + tot.y;
          // stabiliser check: too low (overflow risk) on any tile, too high (underflow of everything) on a
          // model's first tile.  Warp-uniform branch: the redo re-reads TMEM with .sync.aligned loads.
          const bool redo = (cmax > m_stab + 64.f) || (t == 0 && cmax < m_stab - 64.f);
          if (__any_sync(0xffffffffu, redo)) {
            float s_new = 0.f;
#pragma unroll 1
            for (int c = 0; c < 2; ++c) {
              tc_ld32_issue(taddr + c * 32, ra);
              tc_ld_wait(ra);
              s_new += chunk_sum_exact(ra, cmax);
            }
            if (redo) {
              s_run = (t == 0) ? 0.f : s_run * ex2(m_stab - cmax);
              s_tile = s_new;
              m_stab = cmax;
            }
          }
          tc_fence_before();
          mbar_arrive(t_empty + slot);
          s_run += s_tile;
        }
        // ---- merge the two column halves of the row: half 1 publishes (m, s), half 0 finalises
        float2* cb = comb + ((model & 1) * MB + g) * BM;
        if (half == 1) cb[row] = make_float2(m_stab, s_run);
        asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "r"(2 * BM) : "memory");
        if (half == 0) {
          const float2 o = cb[row];
          const float m = fmaxf(m_stab, o.x);
          const float ssum = s_run * ex2(m_stab - m) + o.y * ex2(o.x - m);
          const float lse = (m + lg2(ssum)) * LN2;
          if (live && a.frame_lse) a.frame_lse[(int64_t)model * a.total_frames + fe] = lse;
          warp_segmented_atomic_add(a.scores, utt, a.n_models, model, lse * wgt, lane);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(NSLOT * BN))
                 : "memory");
  }
}

// FP16 operands: a frame outside FP16's range (|x| > 255: x^2 overflows) turns the scores of its utterance into NaN / inf.
// One warp per (utterance, model) pair scans the score matrix and re-scores such pairs in FP32 from the exact section
// of the pack (ab = (mu/var, -1/(2 var)), cst), online log-sum-exp per frame.
struct FixArgs {
  const float* feats;
  const int64_t* offsets;
  int64_t n_utts, total_frames;
  const float2* ab;
  const float* cst;
  int n_models, Kp, K, D, DP, normalize;
  double* scores;
  float* frame_lse;
};
__global__ void __launch_bounds__(256) tc_fixup_kernel(const FixArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n_pairs = a.n_utts * a.n_models;
  for (int64_t p = warp0; p < n_pairs; p += n_warps) {
    const double cur = a.scores[p];
    if (cur == cur && fabs(cur) < 1.0e300) continue;
    const int64_t utt = p / a.n_models;
    const int m = (int)(p % a.n_models);
    const int64_t t0 = a.offsets[utt], t1 = a.offsets[utt + 1];
    double total = 0.0;
    for (int64_t t = t0; t < t1; ++t) {
      const float* xr = a.feats + t * a.D;
      float mrun = -3.0e38f, srun = 0.f;
      for (int c = lane; c < a.K; c += 32) {
        const float2* row = a.ab + ((int64_t)m * a.Kp + c) * a.DP;
        float l = a.cst[(int64_t)m * a.Kp + c];
        for (int j = 0; j < a.D; ++j) {
          const float x = xr[j];
          l = fmaf(x, row[j].x, l);
          l = fmaf(x * x, row[j].y, l);
        }
        const float mn = fmaxf(mrun, l);
        srun = srun * __expf(mrun - mn) + __expf(l - mn);
        mrun = mn;
      }
      const float mall = warp_max(mrun);
      const float sall = warp_sum(srun * __expf(mrun - mall));
      const float lse = mall + __logf(sall);
      if (lane == 0 && a.frame_lse) a.frame_lse[(int64_t)m * a.total_frames + t] = lse;
      total += (double)lse;
    }
    if (lane == 0) a.scores[p] = a.normalize && t1 > t0 ? total / (double)(t1 - t0) : total;
  }
}

}  // namespace tc

// ---- which packs may be scored from their FP16 images
static std::mutex g_pack_mu;
static std::unordered_map<const void*, int> g_pack_h;   // -1: not read back yet, 0: a value left FP16's range, 1: usable
void note_pack(const void* pack) {
  std::lock_guard<std::mutex> lk(g_pack_mu);
  g_pack_h[pack] = -1;
}
static bool pack_h_usable(const void* pack, const PackLayout& L, cudaStream_t st) {
  if (!L.off_tile_h) return false;
  std::lock_guard<std::mutex> lk(g_pack_mu);
  auto it = g_pack_h.find(pack);
  if (it == g_pack_h.end()) return false;   // a pack this process did not build (copied buffer): TF32 images are always valid
  if (it->second < 0) {
    int flag = 1;
    if (cudaMemcpyAsync(&flag, (const char*)pack + L.off_flag, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
      return false;
    it->second = flag ? 0 : 1;
  }
  return it->second == 1;
}

int launch_score_tc(const float* feats, const int64_t* offsets, int64_t n_utts, int64_t total_frames, const void* pack,
                    const PackLayout& L, int parts, bool normalize, double* scores, float* frame_lse, cudaStream_t st) {
  using namespace tc;
  if (L.KD > MAX_KD) {
    set_error("ssp_gmm_score(tf32): feature dim %d needs a contraction of %d > %d; use SSP_PREC_FP32", L.D, L.KD, MAX_KD);
    return SSP_EUNSUP;
  }
  SSP_REQUIRE(parts >= 1 && parts <= 3, "ssp_gmm_score: %d TF32 passes requested (1, 2 or 3)", parts);
  SSP_REQUIRE(parts == 1 || L.off_tile_lo != 0, "ssp_gmm_score: this pack carries no residual tiles");
  SSP_CUDA_OK(cudaMemsetAsync(scores, 0, sizeof(double) * n_utts * L.n_models, st));
  if (total_frames == 0) return SSP_OK;
  Args a;
  a.feats = feats;
  a.offsets = offsets;
  a.n_utts = n_utts;
  a.total_frames = total_frames;
  a.tiles = (const float*)((const char*)pack + L.off_tile);
  a.tiles_lo = (const float*)((const char*)pack + L.off_tile_lo);
  a.n_models = L.n_models;
  a.tiles_per_model = L.Kp / BN;
  a.D = L.D;
  a.KD = L.KD;
  a.normalize = normalize ? 1 : 0;
  a.scores = scores;
  a.frame_lse = frame_lse;
  const int mb = parts == 3 ? 1 : 2, unit = BM * mb;
  const bool use_h = pack_h_usable(pack, L, st);
  if (use_h) {
    a.tiles = (const float*)((const char*)pack + L.off_tile_h);
    a.tiles_lo = (const float*)((const char*)pack + L.off_tile_hl);
    a.KD = L.KDb();
  }
  const size_t tile_bytes = (size_t)BN * a.KD * (use_h ? 2 : 4);
  const size_t smem = (2 + NSTAGE) * tile_bytes + (2 * NSTAGE + 2 * NSLOT + 2) * sizeof(uint64_t) + 16 +
                      2 * mb * BM * sizeof(float2);
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    SSP_CUDA_OK(cudaGetDevice(&dev));
    SSP_CUDA_OK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int64_t n_units = (total_frames + unit - 1) / unit;
  const unsigned grid = (unsigned)(n_units < num_sms ? n_units : num_sms);
#define SSP_TC_LAUNCH(MBv, NP)                                                                                                  \
  do {                                                                                                                          \
    if (use_h) {                                                                                                                \
      SSP_CUDA_OK(cudaFuncSetAttribute(gmm_score_tc_kernel<MBv, NP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      gmm_score_tc_kernel<MBv, NP, true><<<grid, threads_of(MBv), smem, st>>>(a);                                               \
    } else {                                                                                                                    \
      SSP_CUDA_OK(cudaFuncSetAttribute(gmm_score_tc_kernel<MBv, NP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      gmm_score_tc_kernel<MBv, NP, false><<<grid, threads_of(MBv), smem, st>>>(a);                                              \
    }                                                                                                                           \
  } while (0)
  if (parts == 1) SSP_TC_LAUNCH(2, 1);
  else if (parts == 2) SSP_TC_LAUNCH(2, 2);
  else SSP_TC_LAUNCH(1, 3);
#undef SSP_TC_LAUNCH
  SSP_LAUNCH_CHECK(parts == 1 ? "gmm_score_tc_kernel" : parts == 2 ? "gmm_score_tc_kernel<2 passes>" : "gmm_score_tc_kernel<3 passes>");
  if (use_h) {
    FixArgs f;
    f.feats = feats;
    f.offsets = offsets;
    f.n_utts = n_utts;
    f.total_frames = total_frames;
    f.ab = (const float2*)((const char*)pack + L.off_ab);
    f.cst = (const float*)((const char*)pack + L.off_cst);
    f.n_models = L.n_models;
    f.Kp = L.Kp;
    f.K = L.K;
    f.D = L.D;
    f.DP = L.DP;
    f.normalize = normalize ? 1 : 0;
    f.scores = scores;
    f.frame_lse = frame_lse;
    const int64_t n_pairs = n_utts * L.n_models, want = (n_pairs + 7) / 8, cap = 4 * (int64_t)num_sms;
    tc_fixup_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(f);
    SSP_LAUNCH_CHECK("tc_fixup_kernel");
  }
  return SSP_OK;
}

}  // namespace ssp
