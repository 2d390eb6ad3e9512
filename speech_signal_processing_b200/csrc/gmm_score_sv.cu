// GMM-UBM scoring for model sets that SHARE weights and variances (sm_100a, tcgen05 + TMEM).
//
// Mean-only relevance-MAP enrolment (Reynolds 2000; the north-star's "MAP adaptation + scoring" workload) gives
// every speaker the UBM's weights and variances and its own means.  The diagonal-Gaussian log-likelihood
// (sklearn _gaussian_mixture.py:536-553) then splits into a part that is common to all speakers and a part that is
// linear in the frame (log2 domain):
//
//     L2[t, s, c] = q[t, c] + r[t, s, c]
//     q[t, c]     = [x_t^2, x_t, 1, 1] . [-1/(2 var_c), mu_ref,c/var_c, c..] * log2(e)     the full logit of a REFERENCE member
//     r[t, s, c]  = [x_t, 1, 1024] . [(mu_sc - mu_ref,c)/var_c, ca, cb] * log2(e)           speaker s MINUS the reference
//
// so the per-speaker contraction is D + 2 long (41 -> 48 at D = 39) instead of 2D + 2 (80), and the common part is
// computed once per (256 frames, 64 components, 32 models) and kept in registers.
//
// Operands are FP16 (kind::f16, FP32 accumulation): an FP16 significand has the 11 bits of TF32, one MMA covers K = 16
// instead of 8 -- half the tcgen05.mma instructions (an M128 x N64 instruction costs ~49 cycles whatever its kind,
// benchmarks/ubench_mma.cu), half the bytes per model image.  Cepstra after CMVN and (mu_s - mu_ref)/var are far inside
// FP16's range; a frame outside it turns its scores into NaN, which sv_fixup_kernel re-scores in FP32, and
// ssp_gmm_pack_shared refuses models outside it.
//   * r rounds only the DIFFERENCE of a speaker from the reference: its error scales with |mu_s - mu_ref|, and the
//     reference model's own r is exactly zero;
//   * q is evaluated to FP32 grade in the 3-pass manner, A_hi.B_hi + A_lo.B_hi + A_hi.B_lo with FP16 pieces of the
//     frame operand (built per unit in shared memory) and of the model operand (two images), 15 MMAs per 32 models.
//
//   one persistent CTA per SM, unit = 256 frames (two 128-row blocks), component tile = 64
//   loop order per unit:  chunk of 32 models (outer)  x  component tile j  x  model in the chunk (inner)
//   warp 0      : producer   - cp.async.bulk of the 6 KB tile images through a 12-stage ring
//   warps 1, 2  : MMA issuers, one per row block - r-tiles: tcgen05.mma kind::f16 with the FRAME operand in TMEM
//                 (written once per unit by tcgen05.st, thread == row) and the model tile in shared memory -> no
//                 shared-memory traffic for the frames at all; q-tiles: both operands in shared memory.
//                 M128 x N64 x K16, 6 accumulator slots (3 per row block) so the tensor core runs ahead of the epilogue
//   (warps 0..3 shrink to 32 registers, the epilogue warps grow to 112: setmaxnreg)
//   warps 4..19 : epilogue   - thread == (frame row, 32 of the tile's 64 columns); keeps the weights P = 2^(q - m_t) of its
//                 32 columns in registers across the models of a chunk; per model job: tcgen05.ld, release the slot,
//                 sum_c P_c 2^r_c (MUFU ex2 + an FMA-pipe polynomial share, one packed FMA per pair), added to the
//                 (model, frame) partial sum in shared memory
//   per-frame stabiliser m_t = round(max_c logit of the reference model), found in a short pre-pass, fixed for the whole
//   unit, so partial sums of different component tiles simply add.  After a chunk's last tile the partial sums become
//   per-frame log-likelihoods, are summed per utterance inside the warp and added to the (utterance, model) scores.
//   A sum outside [2^-100, 2^100] (a model nowhere near the reference) turns the score into NaN and
//   sv_fixup_kernel re-scores that (utterance, model) pair with a plain FP32 online log-sum-exp.
#include <cuda_fp16.h>

#include <cstdlib>

#include "tc_common.cuh"

namespace ssp {
namespace sv {
using namespace tc;

constexpr int BM = 128;
constexpr int MB = 2;
constexpr int UNIT = BM * MB;
static_assert(UNIT == kSvUnit, "sv_smem_bytes");
constexpr int BN = kSvTileN;
constexpr int NSTAGE = kSvStages;
constexpr int NSLOT = kSvSlots;                 // 3 per row block
constexpr int EPI_WARPS = 16;
constexpr int EPI = EPI_WARPS * 32;
constexpr int CTRL = 128;                // warpgroup 0: producer, two MMA issuers, one idle warp (setmaxnreg is per warpgroup)
constexpr int THREADS = CTRL + EPI;
constexpr int CTRL_REGS = 32, EPI_REGS = 112;  // launched at 96: 128 x (96 - 32) registers released == 512 x (112 - 96) acquired
constexpr int NQ = kSvBaseImages;          // ring slots of the common part: B_hi columns [0, KS) and [KS, KQ), B_lo likewise
constexpr int CHUNK = kSvChunk;                // models per chunk: partial sums [2 column halves][CHUNK][UNIT] fp32 = 64 KB
constexpr uint32_t ACC_COL0 = 128;       // TMEM: [0, 2 KS) frame operand of the two row blocks, [128, 512) accumulators
constexpr uint32_t kRelaxNs = 1000;      // suspend-time hint of the control warps' mbarrier waits
// Share of the exponentials on the FMA pipe, measured on B200 (bench.py config 4, ms per scoring call, profiles/r2k_sv_ab.txt E;
// the float64 oracle check reads 1.35e-5 / 1.36e-5 relative for degree 4 / 3): FP16 kernel, (pairs, degree) = (2,4) 728, (4,4) 711,
// (6,4) 706, (6,3) 691, (8,3) 720.  (The TF32 kernel of round 1, power-capped and with twice the MMA instructions, was best at (4,4).)
constexpr int kPolyPairs = 6;
constexpr int kPolyDeg = 3;

struct Args {
  const float* feats;
  const int64_t* offsets;
  int64_t n_utts, total_frames;
  const __half* tiles;  // [n_tiles][NQ + S][KS/8][BN][8] FP16 images of the WHOLE set (S models); images 0..NQ-1 of a tile are the common q part
  // One launch scores the models [model0, model0 + n_models) of the set -- an L2-resident group (see launch_score_sv):
  const __half* tiles_group;  // == tiles + model0 images: image NQ + m of a tile is model model0 + m
  int n_models;              // models of this launch
  int set_images;            // NQ + S: images per tile
  int set_models;            // S: row stride of the score matrix
  int n_tiles, D, KS, normalize;
  int KQ;              // contraction length of the common part: roundup(2 D + 2, 16) <= 2 KS
  float* stab;         // [total_frames] per-frame exponent stabiliser: written by the first launch (kFirst), read by the others
  double* scores;      // + model0
  float* frame_lse;    // + model0 * total_frames
};

__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// Barriers are addressed by their 32-bit shared-memory address, computed once per thread: going through generic
// pointers re-derives the shared window (S2UR + ULEA) at every use, which is most of a wait's instructions.
__device__ __forceinline__ bool bar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// spin on an mbarrier phase; a protocol bug must trap (after seconds), not hang the GPU.
// No printf here: a call would cost the control warps more registers than setmaxnreg leaves them.
// The bound is clock64(): its reads are 5 % of the kernel's executed instructions, but a poll counter instead makes it
// SLOWER: measured on one box, config 4, ms per call (profiles/r2e_sv_ab.txt): clock64 706 / 708, poll counter 718 / 727,
// counter + nanosleep(20 / 60) 712 / 713 -- a waiting epilogue warp that polls faster takes issue slots and mbarrier
// bandwidth from the three working warps of its sub-partition; the clock read is the cheapest throttle found.
__device__ __forceinline__ void bar_spin(uint32_t bar, uint32_t parity) {
  if (bar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!bar_try_wait(bar, parity)) {
    if (clock64() - t0 > (1ll << 31)) __trap();
  }
}
// the control warps' version: a failed poll parks the warp in hardware for up to ~1 us instead of re-issuing the wait
// loop, which would steal issue slots from the four epilogue warps that share the sub-partition
__device__ __forceinline__ void bar_spin_relaxed(uint32_t bar, uint32_t parity) {
  if (bar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(kRelaxNs)
        : "memory");
    if (ok) return;
    if (clock64() - t0 > (1ll << 31)) __trap();
  }
}
__device__ __forceinline__ void bar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void bar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_g2s_u32(uint32_t smem_dst, const void* gmem_src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
               "l"(gmem_src), "r"(bytes), "r"(bar)
               : "memory");
}

__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}

// sum_c qm_c 2^r_c over 32 accumulator columns, qm holding the WEIGHTS 2^(q - m_t) of the common part: one packed FMA
// per column pair.  kPolyPairs of the 16 column pairs go to the FMA pipe:
// 2^d = 2^n p(f), n = round(d) by the 1.5 * 2^23 magic add, f = d - n in [-0.5, 0.5], p = degree-3 minimax polynomial
// (7.5e-5 relative -- 3e-5 absolute on a frame's log-likelihood at this share, 5e-7 of its magnitude; degree 4 would be
// 2.7e-6), 2^n applied by adding n to the exponent field; the rest is MUFU ex2.
__device__ __forceinline__ float exp_sum32(const uint32_t (&r)[32], const float (&qm)[32]) {
  static_assert(kPolyPairs % 2 == 0 && kPolyPairs <= 16, "pairs are consumed two at a time");
  static_assert(kPolyDeg == 3, "the coefficients below are those of the degree-3 polynomial");
  const float MAGIC = 12582912.f;  // 1.5 * 2^23
  const float2 mg = make_float2(MAGIC, MAGIC), nmg = make_float2(-MAGIC, -MAGIC), neg1 = make_float2(-1.f, -1.f);
  float2 accp = make_float2(0.f, 0.f), accm0 = accp, accm1 = accp;
#pragma unroll
  for (int i = 0; i < kPolyPairs; ++i) {
    float2 d = make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
    d.x = fmaxf(d.x, -126.f);
    d.y = fmaxf(d.y, -126.f);
    const float2 t = __fadd2_rn(d, mg);
    const float2 nn = __fadd2_rn(t, nmg);
    const float2 f = __ffma2_rn(nn, neg1, d);
    float2 p = __ffma2_rn(make_float2(0.0551716685295105f, 0.0551716685295105f), f, make_float2(0.2426111251115799f, 0.2426111251115799f));
    p = __ffma2_rn(p, f, make_float2(0.6932609677314758f, 0.6932609677314758f));
    p = __ffma2_rn(p, f, make_float2(0.9999280571937561f, 0.9999280571937561f));
    float2 e;
    e.x = __uint_as_float(__float_as_uint(p.x) + (__float_as_uint(t.x) << 23));
    e.y = __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(t.y) << 23));
    accp = __ffma2_rn(e, make_float2(qm[2 * i], qm[2 * i + 1]), accp);
  }
#pragma unroll
  for (int i = kPolyPairs; i < 16; i += 2) {
    const float2 d0 = make_float2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
    const float2 d1 = make_float2(__uint_as_float(r[2 * i + 2]), __uint_as_float(r[2 * i + 3]));
    accm0 = __ffma2_rn(make_float2(ex2(d0.x), ex2(d0.y)), make_float2(qm[2 * i], qm[2 * i + 1]), accm0);
    accm1 = __ffma2_rn(make_float2(ex2(d1.x), ex2(d1.y)), make_float2(qm[2 * i + 2], qm[2 * i + 3]), accm1);
  }
  const float2 tot = __fadd2_rn(__fadd2_rn(accm0, accm1), accp);
  return tot.x + tot.y;
}

// kFirst: this launch finds the stabilisers (pre-pass over the reference model) and, if a.stab is set, leaves them for
// the launches of the other model groups; !kFirst: reads them.  A template flag, so that the control warps (32
// registers after setmaxnreg) compile exactly as for a single launch.
template <int KSTEPS, bool kFirst>
__global__ void __launch_bounds__(THREADS, 1) gmm_score_sv_kernel(const Args a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int KS = KSTEPS * 16;
  constexpr uint32_t tile_bytes = (uint32_t)BN * KS * 2u;       // one model tile image (one ring stage)
  const uint32_t aq_block_bytes = (uint32_t)a.KQ * BM * 2u;     // q operand of one row block
  __half* sAh = reinterpret_cast<__half*>(smem);                                  // [MB][KQ/8][BM][8]  fp16([x^2, x, 1, 1, 0..])
  __half* sAl = reinterpret_cast<__half*>(smem + (size_t)MB * aq_block_bytes);    // same shape: what that rounding dropped
  unsigned char* sB = smem + (size_t)2 * MB * aq_block_bytes;                     // [NSTAGE][KS/8][BN][8]
  float* sPart = reinterpret_cast<float*>(sB + (size_t)NSTAGE * tile_bytes);    // [2][CHUNK][UNIT]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sPart + 2 * CHUNK * UNIT);
  const uint32_t b_full = smem_u32(bars);  // barrier i of a group at +8 i
  const uint32_t b_empty = b_full + 8u * NSTAGE;
  const uint32_t t_full = b_empty + 8u * NSTAGE;
  const uint32_t t_empty = t_full + 8u * NSLOT;
  const uint32_t a_full = t_empty + 8u * NSLOT;
  const uint32_t a_empty = a_full + 8u;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NSTAGE + 2 * NSLOT + 2);
  float* mstab = reinterpret_cast<float*>(tmem_slot + 4);  // [UNIT] per-frame stabiliser
  float* mx = sPart;  // [2][UNIT] row maxima of the two column halves: pre-pass only, the partial sums are idle (zero) then

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < NSTAGE; ++i) { mbar_init(bars + i, 1); mbar_init(bars + NSTAGE + i, MB); }
    for (int i = 0; i < NSLOT; ++i) { mbar_init(bars + 2 * NSTAGE + i, 1); mbar_init(bars + 2 * NSTAGE + NSLOT + i, EPI_WARPS / MB); }
    mbar_init(bars + 2 * NSTAGE + 2 * NSLOT, EPI);
    mbar_init(bars + 2 * NSTAGE + 2 * NSLOT + 1, MB);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid >= CTRL)
    for (int i = tid - CTRL; i < 2 * CHUNK * UNIT; i += EPI) sPart[i] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t n_units = (a.total_frames + UNIT - 1) / UNIT;
  const int S = a.n_models, NT = a.n_tiles;
  constexpr size_t tile_halfs = (size_t)BN * KS;

  if (warp < CTRL / 32) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(CTRL_REGS));
  if (warp == 0) {
    // ===================== producer =====================
    const uint32_t sB_u32 = smem_u32(sB);
    uint32_t stage = 0, ph = 0;
    auto load = [&](const __half* src) {
      bar_spin_relaxed(b_empty + 8u * stage, ph ^ 1u);
      if (elect_one()) {
        bar_arrive_expect_tx(b_full + 8u * stage, tile_bytes);
        bulk_g2s_u32(sB_u32 + stage * tile_bytes, src, tile_bytes, b_full + 8u * stage);
      }
      __syncwarp();
      if (++stage == NSTAGE) { stage = 0; ph ^= 1u; }
    };
    const size_t tile_stride = (size_t)a.set_images * tile_halfs;
    for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x) {
      if (kFirst)
        for (int j = 0; j < NT; ++j) {
          const __half* tj = a.tiles + (size_t)j * tile_stride;
          for (int i = 0; i < NQ; ++i, tj += tile_halfs) load(tj);
        }
      for (int m0 = 0; m0 < S; m0 += CHUNK) {
        const int nm = min(CHUNK, S - m0);
        for (int j = 0; j < NT; ++j) {
          const __half* tj = a.tiles + (size_t)j * tile_stride;
          for (int i = 0; i < NQ; ++i, tj += tile_halfs) load(tj);
          const __half* src = a.tiles_group + (size_t)j * tile_stride + (size_t)(NQ + m0) * tile_halfs;
          for (int m = 0; m < nm; ++m, src += tile_halfs) load(src);
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ===================== MMA issuers: warp 1 owns row block 0, warp 2 row block 1 =====================
    const int g = warp - 1;
    constexpr uint32_t lbo_a = BM * 16u, lbo_b = BN * 16u, sbo = 128u;
    constexpr uint32_t ks_a = (2u * lbo_a) >> 4, ks_b = (2u * lbo_b) >> 4;  // one K = 16 step (two 16-byte chunks) in descriptor units
    constexpr uint32_t tile_units = tile_bytes >> 4;
    const uint64_t ah_desc = make_desc(smem_u32(sAh) + (uint32_t)g * aq_block_bytes, lbo_a, sbo);
    const uint64_t al_desc = make_desc(smem_u32(sAl) + (uint32_t)g * aq_block_bytes, lbo_a, sbo);
    const uint64_t b_desc0 = make_desc(smem_u32(sB), lbo_b, sbo);
    const uint32_t at = tmem_base + (uint32_t)(g * (KS / 2));   // two FP16 per TMEM column
    constexpr uint32_t idesc = make_idesc_f16(BM, BN);
    const int steps_b = (a.KQ - KS) >> 4;                       // K steps of the q columns beyond the first KS
    uint32_t stage = 0, bph = 0, s3 = 0, sph = 0, unit_idx = 0;
    auto next_stage = [&]() { if (++stage == NSTAGE) { stage = 0; bph ^= 1u; } };
    auto next_slot = [&]() { if (++s3 == 3) { s3 = 0; sph ^= 1u; } };
    // one accumulator job of this row block: r part only (frame operand in TMEM)
    auto job_r = [&]() {
      bar_spin_relaxed(b_full + 8u * stage, bph);
      const uint32_t slot = (uint32_t)g + 2u * s3;
      bar_spin_relaxed(t_empty + 8u * slot, sph ^ 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d_tmem = tmem_base + ACC_COL0 + slot * BN;
        const uint64_t bd = b_desc0 + (uint64_t)(stage * tile_units);
#pragma unroll
        for (int k = 0; k < KSTEPS; ++k) mma_f16_ts(d_tmem, at + 8u * k, bd + (uint64_t)(k * ks_b), idesc, k > 0 ? 1u : 0u);
        bar_commit(t_full + 8u * slot);
        bar_commit(b_empty + 8u * stage);
      }
      __syncwarp();
      next_stage();
      next_slot();
    };
    // common part = full logit of the reference model, FP32 grade: ring slots 0, 1 hold the columns [0, KS) and [KS, KQ)
    // of B_hi and multiply A_hi and A_lo, slots 2, 3 the same columns of B_lo and multiply A_hi; all into one
    // accumulator; a slot's ring stage is released as soon as its MMAs retire
    auto job_q = [&]() {
      const uint32_t slot = (uint32_t)g + 2u * s3;
      bar_spin_relaxed(t_empty + 8u * slot, sph ^ 1u);
      const uint32_t d_tmem = tmem_base + ACC_COL0 + slot * BN;
#pragma unroll
      for (int part = 0; part < NQ; ++part) {
        bar_spin_relaxed(b_full + 8u * stage, bph);
        tc_fence_after();
        if (elect_one()) {
          // straight-line issue: compile-time descriptor offsets, the steps beyond KQ masked by a uniform predicate (a
          // rolled loop cost this warp ~17 instructions per MMA and left the epilogue waiting for every common part)
          const uint64_t bd = b_desc0 + (uint64_t)(stage * tile_units);
          const bool second = (part & 1) != 0;
          const uint64_t a_off = second ? (uint64_t)(KSTEPS * ks_a) : 0ull;
#pragma unroll
          for (int k = 0; k < KSTEPS; ++k)
            if (!second || k < steps_b)
              mma_f16_ss(d_tmem, ah_desc + a_off + (uint64_t)(k * ks_a), bd + (uint64_t)(k * ks_b), idesc, (part | k) ? 1u : 0u);
          if (part < 2) {
#pragma unroll
            for (int k = 0; k < KSTEPS; ++k)
              if (!second || k < steps_b)
                mma_f16_ss(d_tmem, al_desc + a_off + (uint64_t)(k * ks_a), bd + (uint64_t)(k * ks_b), idesc, 1u);
          }
          if (part == NQ - 1) bar_commit(t_full + 8u * slot);
          bar_commit(b_empty + 8u * stage);
        }
        __syncwarp();
        next_stage();
      }
      next_slot();
    };
    for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x, ++unit_idx) {
      bar_spin_relaxed(a_full, unit_idx & 1u);
      tc_fence_after();
      if (kFirst)
        for (int j = 0; j < NT; ++j) job_q();       // pre-pass: logits of the reference model
      for (int m0 = 0; m0 < S; m0 += CHUNK) {
        const int nm = min(CHUNK, S - m0);
        for (int j = 0; j < NT; ++j) {
          job_q();                                // common part of tile j
#pragma unroll 1
          for (int m = 0; m < nm; ++m) job_r();
        }
      }
      if (elect_one()) bar_commit(a_empty);
      __syncwarp();
    }
  }
  } else {
    // ===================== epilogue warps (also build the frame operands) =====================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(EPI_REGS));
    const int etid = tid - CTRL;               // 0..511
    const int ew = warp - CTRL / 32;           // 0..15
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int g = (ew >> 2) & 1;               // row block
    const int half = ew >> 3;                  // which 32 of the tile's 64 columns
    const int row = quad * 32 + lane;          // accumulator row within the row block
    const int urow = g * BM + row;             // row within the unit
    const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
    const int frow = etid & (UNIT - 1), fpart = etid >> 8;  // finalisation role: frame row, model parity
    const float LN2 = 0.69314718055994530942f;
    float* my_part = sPart + (size_t)half * CHUNK * UNIT + urow;
    uint32_t s3 = 0, sph = 0, unit_idx = 0;

    // wait for the next accumulator job of this row block, pull this thread's 32 columns, free the slot
    const uint32_t my_tmem = tmem_base + lane_addr + ACC_COL0 + (uint32_t)(g * BN + half * 32);  // slot s3 at + 2 BN s3
    const uint32_t my_full = t_full + 8u * g, my_empty = t_empty + 8u * g;                       // slot s3 at + 16 s3
    const bool lane0 = lane == 0;
    auto fetch = [&](uint32_t (&r)[32]) {
      bar_spin(my_full + 16u * s3, sph);
      tc_fence_after();
      tc_ld32_issue(my_tmem + 2u * BN * s3, r);
      tc_ld_wait(r);
      tc_fence_before();
      __syncwarp();
      if (lane0) bar_arrive(my_empty + 16u * s3);
      if (++s3 == 3) { s3 = 0; sph ^= 1u; }
    };

    for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x, ++unit_idx) {
      const int64_t frame0 = u * UNIT;
      bar_spin(a_empty, (unit_idx & 1u) ^ 1u);
      tc_fence_after();
      {
        // ---- q operand [x^2 | x | 1, 1, 0..] in shared memory as two FP16 pieces (A_hi, and what that rounding dropped):
        //      (row r, column j) of block mb at ((mb*KQ/8 + j/8)*BM + r)*8 + j%8
        const int64_t fr = frame0 + frow;
        const bool live = fr < a.total_frames;
        const float* xr = a.feats + fr * a.D;
        const size_t at0 = (size_t)(frow >> 7) * (BM * a.KQ) + (size_t)(frow & (BM - 1)) * 8;
        const int j0 = fpart * (a.KQ >> 1), j1 = j0 + (a.KQ >> 1);
        for (int j = j0; j < j1; ++j) {
          float y = 0.f;
          if (j < 2 * a.D) {
            if (live) { const float x = xr[j < a.D ? j : j - a.D]; y = j < a.D ? x * x : x; }
          } else if (j < 2 * a.D + 2) {
            y = 1.f;
          }
          const __half h = __float2half_rn(y);
          const size_t at1 = at0 + (size_t)(j >> 3) * (BM * 8) + (j & 7);
          sAh[at1] = h;
          sAl[at1] = __float2half_rn(y - __half2float(h));
        }
      }
      {
        // ---- r operand [x, 1, 1024, 0..] as FP16 straight into TMEM: lane == row, column c holds contraction indices 2c, 2c + 1
        const int64_t fe = frame0 + urow;
        const bool live = fe < a.total_frames;
        const float* xr = a.feats + fe * a.D;
        for (int c = half; c < KSTEPS; c += 2) {
          uint32_t v[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float x2[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int j = 16 * c + 2 * e + i;
              float x = 0.f;
              if (j < a.D) x = live ? xr[j] : 0.f;
              else if (j == a.D) x = 1.f;
              else if (j == a.D + 1) x = kSvConstScale;
              x2[i] = x;
            }
            const __half2 hh = __floats2half2_rn(x2[0], x2[1]);   // .x (low half) = the lower contraction index
            v[e] = *reinterpret_cast<const uint32_t*>(&hh);
          }
          tc_st8(tmem_base + lane_addr + (uint32_t)(g * (KS / 2) + 8 * c), v);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      bar_arrive(a_full);

      // ---- finalisation bookkeeping for frame `frow`
      const int64_t ff = frame0 + frow;
      const bool flive = ff < a.total_frames;
      const int futt = flive ? find_segment(a.offsets, a.n_utts, ff) : -1;
      float fwgt = 1.f;
      if (futt >= 0 && a.normalize) fwgt = 1.f / (float)(a.offsets[futt + 1] - a.offsets[futt]);

      // ---- per-frame stabiliser: round(maximum logit of the reference model), from a pre-pass in the first launch
      float m_t;
      if (kFirst) {
        float rmax = -3.0e38f;
        for (int j = 0; j < NT; ++j) {
          uint32_t r[32];
          fetch(r);
          float cm = max3(__uint_as_float(r[0]), __uint_as_float(r[1]), __uint_as_float(r[2]));
#pragma unroll
          for (int i = 3; i < 31; i += 2) cm = max3(cm, __uint_as_float(r[i]), __uint_as_float(r[i + 1]));
          rmax = max3(rmax, cm, __uint_as_float(r[31]));
        }
        mx[half * UNIT + urow] = rmax;
        named_bar_sync(1 + g, 2 * BM);
        m_t = rintf(fmaxf(mx[urow], mx[UNIT + urow]));
        named_bar_sync(1 + g, 2 * BM);
        if (half == 0) { mx[urow] = 0.f; mx[UNIT + urow] = 0.f; }  // both are partial sums of this thread (models 0 and 1)
        if (half == 0 && a.stab && frame0 + urow < a.total_frames) a.stab[frame0 + urow] = m_t;
      } else {
        m_t = frame0 + urow < a.total_frames ? a.stab[frame0 + urow] : 0.f;
      }
      if (half == 0) mstab[urow] = m_t;

      // ---- main pass, a chunk of models at a time
      for (int m0 = 0; m0 < S; m0 += CHUNK) {
        const int nm = min(CHUNK, S - m0);
        for (int j = 0; j < NT; ++j) {
          // sum_c 2^(q - m_t + r) = sum_c P_c 2^r_c with the weights P = 2^(q - m_t) of this thread's 32 columns kept in
          // registers for the models of the chunk: one MUFU per column and tile, and a model job is tcgen05.ld, release,
          // 32 x (ex2 | polynomial) and a packed FMA per pair.  (Round 1 left q - m_t in the accumulator slot for the MMA
          // three jobs ahead to run on top of: a tcgen05.st + wait per job, and the slot was released only after it.)
          float qm[32];
          {
            uint32_t r[32];
            fetch(r);
#pragma unroll
            for (int i = 0; i < 32; ++i) qm[i] = ex2(__uint_as_float(r[i]) - m_t);
          }
          float* dst = my_part;
          // (Reading an accumulator as two 16-column halves, the next job's first half in flight behind the second, was 18 %
          // SLOWER -- 793 vs 672 ms: every tcgen05.wait::ld costs a fixed ~100 cycles, so one 32-column load per job it is.)
#pragma unroll 1
          for (int m = 0; m < nm; ++m, dst += UNIT) {
            uint32_t r[32];
            fetch(r);
            *dst += exp_sum32(r, qm);
          }
        }
        // ---- partial sums of this chunk -> per-frame log-likelihood -> per-utterance score
        named_bar_sync(3, EPI);
        {
          const float mf = mstab[frow];
          float* p0 = sPart + (size_t)fpart * UNIT + frow;
          for (int m = fpart; m < nm; m += 2, p0 += 2 * UNIT) {
            const float v = p0[0] + p0[CHUNK * UNIT];
            p0[0] = 0.f;
            p0[CHUNK * UNIT] = 0.f;
            float lse = (mf + lg2(v)) * LN2;
            if (!(v > 7.9e-31f && v < 1.2e30f)) lse = __int_as_float(0x7fc00000);  // outside [2^-100, 2^100]: sv_fixup_kernel
            if (flive && a.frame_lse) a.frame_lse[(int64_t)(m0 + m) * a.total_frames + ff] = lse;
            warp_segmented_atomic_add(a.scores, futt, a.set_models, m0 + m, lse * fwgt, lane);
          }
        }
        named_bar_sync(3, EPI);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
}

// Re-score the (utterance, model) pairs the tensor kernel gave up on (NaN score): one warp per pair, FP32 online
// log-sum-exp over the same FP16 model images, exact frames.
__global__ void __launch_bounds__(256) sv_fixup_kernel(const Args a, int64_t n_pairs) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int S = a.set_models, KS = a.KS, KQ = a.KQ, D = a.D;   // launched once over the whole set
  const size_t tile_halfs = (size_t)BN * KS;
  const float LN2 = 0.69314718055994530942f;
  for (int64_t p = warp0; p < n_pairs; p += n_warps) {
    const double cur = a.scores[p];
    if (cur == cur && fabs(cur) < 1.0e300) continue;
    const int64_t utt = p / S;
    const int m = (int)(p % S);
    const int64_t t0 = a.offsets[utt], t1 = a.offsets[utt + 1];
    double total = 0.0;
    for (int64_t t = t0; t < t1; ++t) {
      const float* xr = a.feats + t * D;
      float mrun = -3.0e38f, srun = 0.f;
      for (int c = lane; c < a.n_tiles * BN; c += 32) {
        const __half* tq = a.tiles + ((size_t)(c / BN) * (S + NQ)) * tile_halfs;   // B_hi [0, KS), [KS, KQ); B_lo likewise
        const __half* tr = tq + (size_t)(NQ + m) * tile_halfs;                      // model minus reference
        const int n = c % BN;
        auto at = [&](const __half* tile, int j) { return __half2float(tile[((size_t)(j >> 3) * BN + n) * 8 + (j & 7)]); };
        auto bq = [&](int j) {  // column j of the common part, hi + lo
          const __half* t_hi = j < KS ? tq : tq + tile_halfs;
          const int jj = j < KS ? j : j - KS;
          return at(t_hi, jj) + at(t_hi + 2 * tile_halfs, jj);
        };
        float l = at(tr, D) + kSvConstScale * at(tr, D + 1);
        for (int j = 2 * D; j < KQ; ++j) l += bq(j);
        for (int j = 0; j < D; ++j) {
          const float x = xr[j];
          l = fmaf(x, at(tr, j) + bq(D + j), l);
          l = fmaf(x * x, bq(j), l);
        }
        const float mn = fmaxf(mrun, l);
        srun = srun * exp2f(mrun - mn) + exp2f(l - mn);
        mrun = mn;
      }
      const float mall = warp_max(mrun);
      const float sall = warp_sum(srun * exp2f(mrun - mall));
      const float lse = (mall + log2f(sall)) * LN2;
      if (lane == 0 && a.frame_lse) a.frame_lse[(int64_t)m * a.total_frames + t] = lse;
      total += (double)lse;
    }
    if (lane == 0) a.scores[p] = a.normalize && t1 > t0 ? total / (double)(t1 - t0) : total;
  }
}

static int g_num_sms = 0;
static int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      g_num_sms = 148;
  }
  return g_num_sms;
}

template <int KSTEPS>
static int launch_one(const Args& a, unsigned grid, bool first, cudaStream_t st) {
  const size_t smem = sv_smem_bytes(KSTEPS * 16, a.KQ);  // make_sv_layout has checked it against the 227 KB limit
  if (first) {
    SSP_CUDA_OK(cudaFuncSetAttribute(gmm_score_sv_kernel<KSTEPS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gmm_score_sv_kernel<KSTEPS, true><<<grid, THREADS, smem, st>>>(a);
  } else {
    SSP_CUDA_OK(cudaFuncSetAttribute(gmm_score_sv_kernel<KSTEPS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gmm_score_sv_kernel<KSTEPS, false><<<grid, THREADS, smem, st>>>(a);
  }
  return SSP_OK;
}
static int launch_ks(const Args& a, unsigned grid, bool first, cudaStream_t st) {
  switch (a.KS) {
    case 16: return launch_one<1>(a, grid, first, st);
    case 32: return launch_one<2>(a, grid, first, st);
    case 48: return launch_one<3>(a, grid, first, st);
    case 64: return launch_one<4>(a, grid, first, st);
  }
  set_error("ssp_gmm_score_shared: contraction length %d is not a multiple of 16 in [16, 64]", a.KS);
  return SSP_EINVAL;
}

}  // namespace sv

// Large model sets are scored in GROUPS whose tile images stay resident in L2 while all frames pass by: one launch per
// group over the same frames, the per-frame stabilisers of the first launch kept in the workspace.  (Round 1 streamed the
// whole set -- 197 MB of TF32 images at config 4 -- once per 256-frame unit: 36 GB of DRAM reads per call, 48x the
// algorithmic bytes.)  SSP_SV_GROUP_MB caps a group's footprint (default 48 MB; 0 = one launch over the whole set); the
// groups are balanced, so a set just above the cap is not split into a full group and a sliver.  Measured at config 4 with
// the 99 MB of FP16 images, ms per call / DRAM bytes per call: 24 MB (4 launches) 673 / 2.26 GB, 48 MB (2 launches) 671,
// one launch 668 / 8.44 GB -- the 126 MB L2 does not hold a 99 MB set that every SM streams, and 0.5 % of time is not
// worth 13x the algorithmic traffic.
static int sv_group_models(const SvLayout& L) {
  static double mb = -1.0;
  if (mb < 0.0) {
    const char* e = getenv("SSP_SV_GROUP_MB");
    mb = e ? atof(e) : 48.0;
  }
  if (mb <= 0.0) return L.n_models;
  const double per_model = (double)L.Kp * L.KS * 2.0;  // FP16 images
  int cap = (int)(mb * 1048576.0 / per_model) / sv::CHUNK * sv::CHUNK;
  if (cap < sv::CHUNK) cap = sv::CHUNK;
  if (cap >= L.n_models) return L.n_models;
  const int n_groups = (L.n_models + cap - 1) / cap;
  int g = ((L.n_models + n_groups - 1) / n_groups + sv::CHUNK - 1) / sv::CHUNK * sv::CHUNK;
  return g >= L.n_models ? L.n_models : g;
}

int64_t score_sv_workspace_bytes(const SvLayout& L, int64_t total_frames) {
  return sv_group_models(L) < L.n_models ? (int64_t)sizeof(float) * total_frames : 0;
}

int launch_score_sv(const float* feats, const int64_t* offsets, int64_t n_utts, int64_t total_frames, const void* pack,
                    const SvLayout& L, bool normalize, double* scores, float* frame_lse, void* workspace, cudaStream_t st) {
  using namespace sv;
  SSP_CUDA_OK(cudaMemsetAsync(scores, 0, sizeof(double) * n_utts * L.n_models, st));
  if (total_frames == 0) return SSP_OK;
  const int group = sv_group_models(L);
  Args a;
  a.feats = feats;
  a.offsets = offsets;
  a.n_utts = n_utts;
  a.total_frames = total_frames;
  a.tiles = (const __half*)pack;
  a.set_images = L.n_models + NQ;
  a.set_models = L.n_models;
  a.n_tiles = L.Kp / BN;
  a.D = L.D;
  a.KS = L.KS;
  a.KQ = L.KQ;
  a.normalize = normalize ? 1 : 0;
  a.stab = group < L.n_models ? (float*)workspace : nullptr;
  const int64_t n_units = (total_frames + UNIT - 1) / UNIT;
  const unsigned grid = (unsigned)(n_units < num_sms() ? n_units : num_sms());
  for (int m0 = 0; m0 < L.n_models; m0 += group) {
    a.n_models = L.n_models - m0 < group ? L.n_models - m0 : group;
    a.tiles_group = a.tiles + (size_t)m0 * BN * L.KS;   // images are BN * KS FP16 values
    a.scores = scores + m0;
    a.frame_lse = frame_lse ? frame_lse + (size_t)m0 * total_frames : nullptr;
    const int rc = launch_ks(a, grid, m0 == 0, st);
    if (rc != SSP_OK) return rc;
    SSP_LAUNCH_CHECK("gmm_score_sv_kernel");
  }
  // the fix-up pass sees the whole set
  a.n_models = L.n_models;
  a.tiles_group = a.tiles;
  a.scores = scores;
  a.frame_lse = frame_lse;
  const int64_t n_pairs = n_utts * L.n_models;
  const int64_t want = (n_pairs + 7) / 8, cap = 4 * (int64_t)num_sms();
  sv_fixup_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(a, n_pairs);
  SSP_LAUNCH_CHECK("sv_fixup_kernel");
  return SSP_OK;
}

}  // namespace ssp
