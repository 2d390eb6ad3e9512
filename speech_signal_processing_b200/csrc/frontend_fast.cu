// Fast path of the fused front-end for nfft = 512 (25 ms frames at 16 kHz, the reference's setting).
//
// Same contract as frontend_kernel (frontend.cu) with a cheaper per-frame pipeline:
//   * the samples of 8 consecutive frames (one per warp) are staged once in shared memory as floats,
//     so each PCM sample is read from global memory once per CTA instead of 2 x 2.5 times;
//   * the 256-point complex FFT of the packed frame lives in REGISTERS: 8 points per lane, radix-8
//     butterfly, one shared-memory transpose (bank-conflict-free, row stride 36), second radix-8, and the
//     last radix-4 across lane quadruples with warp shuffles -- 2 shared-memory round trips instead of 4
//     Stockham passes;
//   * the real-FFT split handles bins k and 256-k together;
//   * the triangular filterbank is cut into 8-bin segments that start on a multiple of 4 bins (weights zero-padded),
//     spread over the 32 lanes: a segment is two 16-byte loads of weights, two of the spectrum and 8 FMAs, and a
//     lane per filter is no longer bound by the widest triangle; per-filter sums in a fixed order (deterministic);
//   * int16 PCM is staged with 16-byte loads (8 samples) when the utterance starts on a 16-byte boundary;
//   * delta and delta-delta are materialised once in shared memory when the utterance is short enough,
//     and the CMVN statistics / output passes read them instead of re-deriving 16 taps per element.
//   * kSk = true is the instantiation for the reference's own setting (sidekit recipe at 16 kHz: 400-sample frames, hop
//     160, per-frame pre-emphasis, power spectrum, 24 filters, natural log, 13 cepstra, every frame complete): frame
//     geometry and conventions are compile-time constants, the window, the real-FFT twiddles and the DCT rows live in
//     registers, samples are read as aligned 8-byte pairs (round 1: 4-byte loads at stride 2 floats, the bulk of the
//     26 % bank-conflict wavefronts), the DCT runs two lanes per cepstrum, and log is lg2.approx * ln 2 (|error| ~1e-6).
#include <type_traits>

#include "frontend_common.cuh"

namespace ssp {

namespace ff {
// CTAs per SM the register allocation aims at.  3 (<= 85 registers: 80 + 292 bytes of spills, and no materialised deltas
// to fit the shared memory) measured 108.6 ms at config 2 against 33.2 ms
constexpr int kMinCtas = 2;
constexpr int W = 8;          // warps per CTA == frames per batch
constexpr int NH = 256;       // complex FFT length
constexpr int EXS = 36;       // float2 row stride of the transpose buffer (conflict-free for 64-bit accesses)
constexpr int EXN = 8 * EXS;  // 288 float2 >= 268 needed for the padded spectrum
constexpr int MAXSEG = 128;   // 8-bin filterbank segments (two-sided 40-filter bank: ~92)
constexpr int PWN = 272;      // spectrum row: 257 bins + zero padding read by the last aligned segment
constexpr int MAXF = 64;      // filters
constexpr int MAXC = 32;      // cepstra

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ void dft4(float2& a0, float2& a1, float2& a2, float2& a3) {
  const float2 s0 = cadd(a0, a2), s1 = csub(a0, a2), s2 = cadd(a1, a3), d = csub(a1, a3);
  const float2 s3 = make_float2(d.y, -d.x);  // (a1 - a3) * (-i)
  a0 = cadd(s0, s2);
  a1 = cadd(s1, s3);
  a2 = csub(s0, s2);
  a3 = csub(s1, s3);
}
// in-place 8-point DFT, natural order in and out (decimation in frequency)
__device__ __forceinline__ void dft8(float2 (&v)[8]) {
  const float R = 0.70710678118654752440f;
  float2 a0 = cadd(v[0], v[4]), a1 = cadd(v[1], v[5]), a2 = cadd(v[2], v[6]), a3 = cadd(v[3], v[7]);
  float2 b0 = csub(v[0], v[4]);
  const float2 t1 = csub(v[1], v[5]), t2 = csub(v[2], v[6]), t3 = csub(v[3], v[7]);
  float2 b1 = make_float2((t1.x + t1.y) * R, (t1.y - t1.x) * R);   // * (1 - i)/sqrt2
  float2 b2 = make_float2(t2.y, -t2.x);                           // * (-i)
  float2 b3 = make_float2((t3.y - t3.x) * R, -(t3.x + t3.y) * R);  // * (-1 - i)/sqrt2
  dft4(a0, a1, a2, a3);
  dft4(b0, b1, b2, b3);
  v[0] = a0; v[2] = a1; v[4] = a2; v[6] = a3;
  v[1] = b0; v[3] = b1; v[5] = b2; v[7] = b3;
}
__device__ __forceinline__ float2 shfl_xor2(float2 v, int m) {
  return make_float2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
}

__host__ __device__ inline size_t carve_floats(const ssp_frontend_cfg& c, int max_frames, bool mat, int* per_warp_out,
                                                int* stg_out) {
  const int FLp = (c.frame_len + 3) & ~3;
  const int stg = ((W - 1) * c.frame_shift + c.frame_len + 1 + 3) & ~3;
  const int per_warp = 2 * EXN + PWN + MAXSEG + MAXF;
  if (per_warp_out) *per_warp_out = per_warp;
  if (stg_out) *stg_out = stg;
  size_t f = 2 * (NH + 2) + FLp + ((c.n_ceps * (c.n_filt | 1) + 3) & ~3) + 8 * MAXSEG + 2 * MAXSEG + (MAXF + 4) + 4 + 256 + 64 + 64 +
             2 * (stg + 12) + (size_t)W * per_warp;
  f += (size_t)max_frames * c.n_ceps * (mat ? (1 + c.delta_order) : 1);
  return f;
}

// the configuration the kSk instantiation is compiled for (sidekit recipe at 16 kHz, GMM_UBM.py:89)
constexpr int SK_FL = 400, SK_SH = 160, SK_NF = 24, SK_NC = 13;

template <typename PcmT, bool kSk>
__global__ void __launch_bounds__(256, kMinCtas) frontend512_kernel(const FrontendArgs a, const int flags, const int64_t n_utts) {
  const int materialize = flags & 1;  // bit 0: delta / delta-delta are materialised in shared memory
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ssp_frontend_cfg& cfg = a.cfg;
  const int NC = kSk ? SK_NC : cfg.n_ceps, NF = kSk ? SK_NF : cfg.n_filt, FL = kSk ? SK_FL : cfg.frame_len,
            SH = kSk ? SK_SH : cfg.frame_shift;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
  const int OD = NC * (1 + cfg.delta_order);
  // ---- carve-up (mirrors carve_floats)
  int per_warp, stg;
  carve_floats(cfg, 0, false, &per_warp, &stg);
  float* p = reinterpret_cast<float*>(smem_raw);
  float2* tw_real = reinterpret_cast<float2*>(p); p += 2 * (NH + 2);
  float* win = p; p += (FL + 3) & ~3;
  const int DS = NF | 1;  // odd row stride: lanes reading different rows hit different banks
  float* dct = p; p += (NC * DS + 3) & ~3;
  float* segw = p; p += 8 * MAXSEG;  // [2 halves][MAXSEG][4]: lane == segment reads 16 bytes at stride 16 (no conflicts)
  int* seg_start = reinterpret_cast<int*>(p); p += MAXSEG;
  int* seg_filt = reinterpret_cast<int*>(p); p += MAXSEG;
  int* filt_seg0 = reinterpret_cast<int*>(p); p += MAXF + 4;
  int* meta = reinterpret_cast<int*>(p); p += 4;
  float* red = p; p += 256;
  float* mean = p; p += 64;
  float* istd = p; p += 64;
  // two staging buffers (batch b in buffer b & 1: one CTA barrier per batch instead of two); "+ 3": sample 0 of a batch sits
  // at a 16-byte boundary (stage[1]), so 8 samples are staged with two 16-byte stores and frames read aligned pairs
  float* stage0 = p + 3; p += 2 * (stg + 12);
  const int stage_stride = stg + 12;
  float* wb = p + (size_t)warp * per_warp; p += (size_t)W * per_warp;
  float* ceps = p;
  float2* ex = reinterpret_cast<float2*>(wb);
  float* pw = wb + 2 * EXN;
  float* segsum = pw + PWN;
  float* mel = segsum + MAXSEG;

  // ---- per-CTA tables (built once: a CTA walks utterances blockIdx.x, + gridDim.x, ...)
  for (int k = tid; k <= NH; k += 256) {
    float s, c;
    sincospif(-(float)k / 256.0f, &s, &c);  // e^{-2 pi i k / 512}
    tw_real[k] = make_float2(c, s);
  }
  for (int i = tid; i < FL; i += 256) win[i] = a.window[i];
  for (int i = tid; i < NC * NF; i += 256) dct[(i / NF) * DS + (i % NF)] = a.dct[i];
  // filterbank CSR (3 x NF ints) is pulled in cooperatively; every triangle is cut into 8-bin segments that start
  // on a multiple of 4 bins
  int* csr = reinterpret_cast<int*>(stage0);  // the staging buffers are free until the first batch
  for (int i = tid; i < NF; i += 256) {
    csr[i] = a.fb_len[i];
    csr[MAXF + i] = a.fb_start[i];
    csr[2 * MAXF + i] = a.fb_offset[i];
  }
  __syncthreads();
  if (tid == 0) {
    int s = 0;
    for (int m = 0; m < NF; ++m) {
      filt_seg0[m] = s;
      const int len = csr[m], st = csr[MAXF + m];
      if (len > 0) s += (st + len - (st & ~3) + 7) >> 3;
    }
    filt_seg0[NF] = s;
    meta[0] = s;
  }
  __syncthreads();
  const int n_seg = meta[0];  // <= MAXSEG is checked on the host side of the launch (frontend_fast_supported + fallback)
  for (int m = tid; m < NF; m += 256) {
    const int st = csr[MAXF + m];
    for (int sg = filt_seg0[m], b = st & ~3; sg < filt_seg0[m + 1] && sg < MAXSEG; ++sg, b += 8) {
      seg_start[sg] = b;
      seg_filt[sg] = m;
    }
  }
  __syncthreads();
  for (int idx = tid; idx < 8 * min(n_seg, MAXSEG); idx += 256) {
    const int sg = idx >> 3, j = idx & 7, m = seg_filt[sg];
    const int rel = seg_start[sg] + j - csr[MAXF + m];
    const float w = (rel >= 0 && rel < csr[m]) ? a.fb_weights[csr[2 * MAXF + m] + rel] : 0.f;
    segw[((j >> 2) * MAXSEG + sg) * 4 + (j & 3)] = w;
  }
  for (int i = lane; i < PWN; i += 32) pw[i] = 0.f;  // the padding bins stay zero; 0..256 are rewritten every frame
  // per-lane twiddles, constant across frames
  float2 tw1[8], tw2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    float s, c;
    sincospif(-(float)(lane * k) / 128.0f, &s, &c);  // W_256^{lane k}
    tw1[k] = make_float2(c, s);
    sincospif(-(float)((lane & 3) * k) / 16.0f, &s, &c);  // W_32^{b k}
    tw2[k] = make_float2(c, s);
  }
  __syncthreads();

  // real-FFT twiddles of the bins this lane splits (k = 1 + lane + 32 j), constant across frames
  float2 twr[4];
#pragma unroll
  for (int jx = 0; jx < 4; ++jx) {
    float sn, cs;
    sincospif(-(float)(1 + lane + 32 * jx) / 256.0f, &sn, &cs);
    twr[jx] = make_float2(cs, sn);
  }
  // kSk: window taps of this lane's samples (i = 64 j + 2 lane, + 1) and its half DCT row (lane = 2 cepstrum + half)
  float2 wreg[7];
  float dreg[SK_NF / 2];
  if (kSk) {
#pragma unroll
    for (int jx = 0; jx < 7; ++jx) {
      const int i = 64 * jx + 2 * lane;
      wreg[jx] = i < SK_FL ? make_float2(a.window[i], a.window[i + 1]) : make_float2(0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < SK_NF / 2; ++i) dreg[i] = lane < 2 * SK_NC ? a.dct[(lane >> 1) * SK_NF + (lane & 1) * (SK_NF / 2) + i] : 0.f;
  }
  // kSk: this lane's filterbank bookkeeping in registers (first bin of its <= 4 segments, segment range of its filter)
  int sgs[4] = {0, 0, 0, 0}, fs0 = 0, fs1 = 0;
  if (kSk) {
#pragma unroll
    for (int q = 0; q < 4; ++q) sgs[q] = (lane + 32 * q < n_seg && n_seg <= MAXSEG) ? seg_start[lane + 32 * q] : -1;
    // a filterbank wider than the segment table leaves the range empty: segsum holds MAXSEG floats and is not written
    // then, so the per-filter sum reads nothing and the plain dot product below serves the filter
    if (lane < SK_NF && n_seg <= MAXSEG) { fs0 = filt_seg0[lane]; fs1 = filt_seg0[lane + 1]; }
  }
  const float pre = cfg.preemph;
  const int pmode = kSk ? 1 : cfg.preemph_mode;
  const float LOG10_E = 0.43429448190325176f;

  for (int64_t u = blockIdx.x; u < n_utts; u += gridDim.x) {
  const int64_t s_begin = a.sample_offsets[u];
  const int64_t n_samp = a.sample_offsets[u + 1] - s_begin;
  const int64_t f_begin = a.frame_offsets[u];
  const int T = (int)(a.frame_offsets[u + 1] - f_begin);
  if (T <= 0) continue;
  const int n_batches = (T + W - 1) / W;

  // everything of a frame after the windowed samples: FFT, spectrum, filterbank, log, DCT -> cepstra of frame f
  auto finish_frame = [&](const int f, float2 (&v)[8], float energy) {
    energy = warp_sum(energy);

    // ---- 256-point FFT: n = 32 n1 + n2 (n2 = lane), k = k1 + 8 k2
    dft8(v);
#pragma unroll
    for (int k = 1; k < 8; ++k) v[k] = cmul(v[k], tw1[k]);
#pragma unroll
    for (int k = 0; k < 8; ++k) ex[k * EXS + lane] = v[k];
    __syncwarp();
    const int k1 = lane >> 2, bq = lane & 3;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = ex[k1 * EXS + 4 * j + bq];
    __syncwarp();
    dft8(v);
#pragma unroll
    for (int c = 1; c < 8; ++c) v[c] = cmul(v[c], tw2[c]);
    // radix-4 across the lane quadruple: after the two shuffle stages lane b holds output d = {0,2,1,3}[b]
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float2 q = shfl_xor2(v[c], 2);
      v[c] = (lane & 2) ? csub(q, v[c]) : cadd(v[c], q);
      if (bq == 3) v[c] = make_float2(v[c].y, -v[c].x);
      q = shfl_xor2(v[c], 1);
      v[c] = (lane & 1) ? csub(q, v[c]) : cadd(v[c], q);
    }
    {
      const int d = ((bq & 1) << 1) | (bq >> 1);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int k = k1 + 8 * c + 64 * d;
        ex[k + 4 * (k >> 6)] = v[c];  // padded by 4 per 64 so the four d-blocks land in different banks
      }
    }
    __syncwarp();

    // ---- real-input split, bins k and 256 - k together; power / magnitude spectrum
    float etot = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = 1 + lane + 32 * j, km = NH - k;  // k in 1..128
      const float2 zk = ex[k + 4 * (k >> 6)], zm = ex[km + 4 * (km >> 6)];
      const float2 t = twr[j];
      const float2 xe = make_float2(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
      const float2 xo = make_float2(0.5f * (zk.y + zm.y), -0.5f * (zk.x - zm.x));
      const float2 x = cmul(t, xo);
      // X[k] = xe + t xo ;  X[256-k] = conj(xe) + (-conj t) * conj(xo)... = conj(xe - t xo)
      const float re = xe.x + x.x, im = xe.y + x.y;
      const float re2 = xe.x - x.x, im2 = xe.y - x.y;
      float p1 = fmaf(re, re, im * im), p2 = fmaf(re2, re2, im2 * im2);
      if (!kSk) {
        if (cfg.spec_type == 1) { p1 = sqrtf(p1); p2 = sqrtf(p2); }
        p1 *= cfg.spec_scale;
        p2 *= cfg.spec_scale;
      }
      pw[k] = p1;
      if (km != k) { pw[km] = p2; etot += p2; }
      etot += p1;
    }
    if (lane == 0) {
      const float2 z0 = ex[0];
      float p0 = (z0.x + z0.y) * (z0.x + z0.y), pn = (z0.x - z0.y) * (z0.x - z0.y);
      if (!kSk) {
        if (cfg.spec_type == 1) { p0 = sqrtf(p0); pn = sqrtf(pn); }
        p0 *= cfg.spec_scale;
        pn *= cfg.spec_scale;
      }
      pw[0] = p0;
      pw[NH] = pn;
      etot += p0 + pn;
    }
    if (!kSk && cfg.energy_mode == 2) etot = warp_sum(etot);
    __syncwarp();

    // ---- filterbank: bounded-width segments spread over the lanes, then a fixed-order sum per filter
    if (kSk) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (sgs[q] >= 0) {
          const int sg = lane + 32 * q;
          const float4* q4 = reinterpret_cast<const float4*>(pw + sgs[q]);
          const float4 w0 = reinterpret_cast<const float4*>(segw)[sg], w1 = reinterpret_cast<const float4*>(segw)[MAXSEG + sg];
          const float4 q0 = q4[0], q1 = q4[1];
          float acc = w0.x * q0.x;
          acc = fmaf(w0.y, q0.y, acc);
          acc = fmaf(w0.z, q0.z, acc);
          acc = fmaf(w0.w, q0.w, acc);
          acc = fmaf(w1.x, q1.x, acc);
          acc = fmaf(w1.y, q1.y, acc);
          acc = fmaf(w1.z, q1.z, acc);
          acc = fmaf(w1.w, q1.w, acc);
          segsum[sg] = acc;
        }
      }
      __syncwarp();
      if (lane < SK_NF) {
        // the loads of up to 8 segments are independent (issued back to back); wider filters finish in the loop
        float part[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) part[q] = fs0 + q < fs1 ? segsum[fs0 + q] : 0.f;
        float acc = part[0];
#pragma unroll
        for (int q = 1; q < 8; ++q) acc += part[q];   // same order as the sequential sum (zeros pad the tail)
        for (int sg = fs0 + 8; sg < fs1; ++sg) acc += segsum[sg];
        if (n_seg > MAXSEG) {  // (24 filters wider than the segment table holds: plain dot products, as in the generic path)
          acc = 0.f;
          const float* w = a.fb_weights + a.fb_offset[lane];
          const float* q = pw + a.fb_start[lane];
          for (int i = 0; i < a.fb_len[lane]; ++i) acc = fmaf(w[i], q[i], acc);
        }
        mel[lane] = __logf(acc);
      }
      __syncwarp();
    } else {
    for (int sg = lane; sg < n_seg && n_seg <= MAXSEG; sg += 32) {
      const float4* q4 = reinterpret_cast<const float4*>(pw + seg_start[sg]);
      const float4 w0 = reinterpret_cast<const float4*>(segw)[sg], w1 = reinterpret_cast<const float4*>(segw)[MAXSEG + sg];
      const float4 q0 = q4[0], q1 = q4[1];
      float acc = w0.x * q0.x;
      acc = fmaf(w0.y, q0.y, acc);
      acc = fmaf(w0.z, q0.z, acc);
      acc = fmaf(w0.w, q0.w, acc);
      acc = fmaf(w1.x, q1.x, acc);
      acc = fmaf(w1.y, q1.y, acc);
      acc = fmaf(w1.z, q1.z, acc);
      acc = fmaf(w1.w, q1.w, acc);
      segsum[sg] = acc;
    }
    __syncwarp();
    for (int m = lane; m < NF; m += 32) {
      float acc = 0.f;
      if (n_seg <= MAXSEG) {
        for (int sg = filt_seg0[m]; sg < filt_seg0[m + 1]; ++sg) acc += segsum[sg];
      } else {  // a filterbank too wide for the segment table: plain per-filter dot product from global memory
        const float* w = a.fb_weights + a.fb_offset[m];
        const float* q = pw + a.fb_start[m];
        for (int i = 0; i < a.fb_len[m]; ++i) acc = fmaf(w[i], q[i], acc);
      }
      if (cfg.log_zero_floor > 0.f && acc == 0.f) acc = cfg.log_zero_floor;
      acc += cfg.log_add;
      mel[m] = cfg.log_type == 2 ? acc : (cfg.log_type == 1 ? logf(acc) * LOG10_E : logf(acc));
    }
    __syncwarp();
    }
    // ---- DCT
    if (kSk) {
      // two lanes per cepstrum, 12 filters each, coefficients in registers
      const float4* mh = reinterpret_cast<const float4*>(mel + (lane & 1) * (SK_NF / 2));
      float acc = 0.f;
#pragma unroll
      for (int q = 0; q < SK_NF / 8; ++q) {
        const float4 mv = mh[q];
        acc = fmaf(dreg[4 * q + 0], mv.x, acc);
        acc = fmaf(dreg[4 * q + 1], mv.y, acc);
        acc = fmaf(dreg[4 * q + 2], mv.z, acc);
        acc = fmaf(dreg[4 * q + 3], mv.w, acc);
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      if (lane < 2 * SK_NC && (lane & 1) == 0) ceps[f * SK_NC + (lane >> 1)] = acc;
    } else {
    for (int j = lane; j < NC; j += 32) {
      const float* row = dct + j * DS;
      float acc0 = 0.f, acc1 = 0.f;
      int m = 0;
      for (; m + 1 < NF; m += 2) {
        acc0 = fmaf(row[m], mel[m], acc0);
        acc1 = fmaf(row[m + 1], mel[m + 1], acc1);
      }
      if (m < NF) acc0 = fmaf(row[m], mel[m], acc0);
      float acc = acc0 + acc1;
      if (cfg.energy_mode == 2 && j == 0) {
        float e = etot;
        if (cfg.log_zero_floor > 0.f && e == 0.f) e = cfg.log_zero_floor;
        acc = logf(e);
      }
      ceps[f * NC + j] = acc;
    }
    }
    if (lane == 0 && a.out_log_energy && cfg.energy_mode == 1) a.out_log_energy[f_begin + f] = kSk ? __logf(energy) : logf(energy);
  };

  // kSk, int16 PCM on a 4-byte boundary: NO staging and no CTA barrier per batch.  A lane's samples of a frame are seven
  // aligned pairs z[32 j + lane] = (x[64 j + 2 lane], x[.. + 1]) -- seven coalesced 4-byte loads straight from global memory
  // (a sample is read by the 2.5 frames that cover it, from L1 after the first), the sample before a pair comes from the
  // neighbouring lane by shuffle, and the loads of the warp's NEXT frame are in flight while this one is transformed.  The
  // warps of a CTA run decoupled until the delta / CMVN phase.
  const bool direct = kSk && sizeof(PcmT) == 2 && ((reinterpret_cast<uintptr_t>(a.pcm) & 3) == 0);
  if (direct) {
    // an utterance that starts on an odd sample reads the pairs one sample earlier: word = (x[i - 1], x[i]), x[i + 1] comes
    // from the lane above
    const bool odd = (s_begin & 1) != 0;
    const int16_t* pcm16 = reinterpret_cast<const int16_t*>(a.pcm) + s_begin;
    const uint32_t* pairs = reinterpret_cast<const uint32_t*>(pcm16 - (odd ? 1 : 0)) + lane;
    constexpr int LAST = (SK_FL - 384) / 2;   // lanes of pair row 6 inside the frame
    uint32_t cur[7], nxt[7];
    auto load_frame = [&](int f, uint32_t (&wd)[7]) {
      const uint32_t* q = pairs + (int64_t)f * (SK_SH / 2);
#pragma unroll
      for (int j = 0; j < 6; ++j) wd[j] = __ldg(q + 32 * j);
      wd[6] = lane < LAST ? __ldg(q + 192) : 0u;
      // odd start: lane LAST holds (x[399], x[400]); only x[399] is part of the frame (and of the buffer)
      if (odd && lane == LAST) wd[6] = (uint32_t)(uint16_t)pcm16[(int64_t)f * SK_SH + SK_FL - 1];
    };
    // (one loop per alignment, chosen per utterance: with both unpack variants inside one loop the kernel lost the 10 % the
    // direct loads had gained)
    auto run = [&](auto odd_tag) {
      constexpr bool kOdd = decltype(odd_tag)::value;
      if (warp < T) load_frame(warp, cur);
      for (int f = warp; f < T; f += W) {
        if (f + W < T) load_frame(f + W, nxt);
        float2 v[8];
        float energy = 0.f;
        if (!kOdd) {
          float hi_prev = 0.f;
#pragma unroll
          for (int j = 0; j < 7; ++j) {
            const float lo = (float)(int16_t)(cur[j] & 0xffffu), hi = (float)(int16_t)(cur[j] >> 16);
            // x[i - 1]: the odd sample of the lane below; lane 0 takes lane 31's odd sample of the previous pair row
            float xm1 = __shfl_sync(0xffffffffu, lane == 31 ? hi_prev : hi, (lane + 31) & 31);
            if (j == 0 && lane == 0) xm1 = lo;   // per-frame pre-emphasis: the first sample is its own predecessor
            hi_prev = hi;
            float y0 = fmaf(-pre, xm1, lo), y1 = fmaf(-pre, lo, hi);
            if (j == 6 && lane >= LAST) { y0 = 0.f; y1 = 0.f; }
            energy = fmaf(y0, y0, fmaf(y1, y1, energy));
            v[j] = make_float2(y0 * wreg[j].x, y1 * wreg[j].y);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 7; ++j) {
            const float xm = (float)(int16_t)(cur[j] & 0xffffu), x0 = (float)(int16_t)(cur[j] >> 16);   // x[i - 1], x[i]
            const float lo_next_row = j < 6 ? (float)(int16_t)(cur[j < 6 ? j + 1 : j] & 0xffffu) : 0.f;
            // x[i + 1]: the even-position sample of the lane above; lane 31 takes lane 0's of the next pair row
            const float x1 = __shfl_sync(0xffffffffu, lane == 0 ? lo_next_row : xm, (lane + 1) & 31);
            float y0 = fmaf(-pre, (j == 0 && lane == 0) ? x0 : xm, x0), y1 = fmaf(-pre, x0, x1);
            if (j == 6 && lane >= LAST) { y0 = 0.f; y1 = 0.f; }
            energy = fmaf(y0, y0, fmaf(y1, y1, energy));
            v[j] = make_float2(y0 * wreg[j].x, y1 * wreg[j].y);
          }
        }
        v[7] = make_float2(0.f, 0.f);
        finish_frame(f, v, energy);
#pragma unroll
        for (int j = 0; j < 7; ++j) cur[j] = nxt[j];
      }
    };
    if (odd) run(std::true_type{}); else run(std::false_type{});
    __syncthreads();
  } else {
  // The staging loads of batch b+1 are issued before batch b is processed and only written to shared memory
  // after it, so their global-memory latency hides behind a whole frame of FFT work.
  constexpr int PF = 8;  // samples per thread per batch: (W-1)*shift + frame_len + 1 <= 256 * PF
  float pf[PF];
  // int16 PCM whose utterance starts on a 16-byte boundary: thread t stages samples [8t, 8t + 8) of the batch with one
  // 16-byte load (W * shift is a multiple of 8, so every batch stays aligned); the sample before the batch (needed by
  // the pre-emphasis) goes through thread 255.  Otherwise: one sample per load, 8 loads per thread.
  const bool vec = sizeof(PcmT) == 2 && ((s_begin & 7) == 0) && ((reinterpret_cast<uintptr_t>(a.pcm) & 15) == 0);
  auto prefetch = [&](int b) {
    const int64_t base = (int64_t)b * W * SH;
    if (vec) {
      const int64_t j = base + 8 * tid;
      if (8 * tid < stg - 1 && j + 7 < n_samp) {
        const uint4 raw = *reinterpret_cast<const uint4*>(reinterpret_cast<const int16_t*>(a.pcm) + s_begin + j);
        pf[0] = __uint_as_float(raw.x); pf[1] = __uint_as_float(raw.y); pf[2] = __uint_as_float(raw.z); pf[3] = __uint_as_float(raw.w);
      } else {
        // tail of the utterance: per-sample loads, packed the same way so that the unpack below is shared
        uint32_t wds[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int64_t g = j + 2 * e;
          const int lo = (8 * tid < stg - 1 && g < n_samp) ? (int)reinterpret_cast<const int16_t*>(a.pcm)[s_begin + g] : 0;
          const int hi = (8 * tid < stg - 1 && g + 1 < n_samp) ? (int)reinterpret_cast<const int16_t*>(a.pcm)[s_begin + g + 1] : 0;
          wds[e] = ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16);
        }
        pf[0] = __uint_as_float(wds[0]); pf[1] = __uint_as_float(wds[1]); pf[2] = __uint_as_float(wds[2]); pf[3] = __uint_as_float(wds[3]);
      }
      pf[4] = (tid == 255 && base > 0 && base - 1 < n_samp) ? load_pcm<PcmT>(a.pcm, s_begin + base - 1) : 0.f;
      return;
    }
    const int64_t g0 = base - 1;
#pragma unroll
    for (int r = 0; r < PF; ++r) {
      const int i = tid + 256 * r;
      const int64_t g = g0 + i;
      pf[r] = (i < stg && g >= 0 && g < n_samp) ? load_pcm<PcmT>(a.pcm, s_begin + g) : 0.f;
    }
  };
  prefetch(0);
  for (int b = 0; b < n_batches; ++b) {
    float* stage = stage0 + (b & 1) * stage_stride;
    if (vec) {
      if (8 * tid < stg - 1) {
        float smp[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const uint32_t wd = __float_as_uint(pf[e]);
          smp[2 * e] = (float)(int16_t)(wd & 0xffffu);
          smp[2 * e + 1] = (float)(int16_t)(wd >> 16);
        }
        float4* dst = reinterpret_cast<float4*>(stage + 1 + 8 * tid);   // 16-byte aligned; the buffer has slack for whole stores
        dst[0] = make_float4(smp[0], smp[1], smp[2], smp[3]);
        dst[1] = make_float4(smp[4], smp[5], smp[6], smp[7]);
      }
      if (tid == 255) stage[0] = pf[4];
    } else {
#pragma unroll
      for (int r = 0; r < PF; ++r) {
        const int i = tid + 256 * r;
        if (i < stg) stage[i] = pf[r];
      }
    }
    __syncthreads();  // batch b is staged; buffer (b + 1) & 1 was last read in batch b - 1, which every warp has left
    if (b + 1 < n_batches) prefetch(b + 1);
    const int f = b * W + warp;
    if (f >= T) continue;
    const float* s = stage + 1 + warp * SH;              // s[i] = sample i of this frame, s[-1] the one before
    const int64_t s0 = (int64_t)f * SH;
    const int n_valid = (int)min((int64_t)FL, n_samp - s0);  // samples of the frame that exist (zero padded tail)

    // ---- load + pre-emphasis + energy + window, packed z[n] = (x[2n], x[2n+1]); lane holds z[32 j + lane]
    float2 v[8];
    float energy = 0.f;
    if (kSk) {
      // every frame is complete (framing 0): no tail handling; samples as aligned pairs, window taps from registers
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const int i = 64 * j + 2 * lane;
        float2 x = make_float2(0.f, 0.f);
        float xm1 = 0.f;
        if (j < 6 || i < SK_FL) {
          x = *reinterpret_cast<const float2*>(s + i);
          xm1 = (j == 0 && lane == 0) ? x.x : s[i - 1];
        }
        const float y0 = fmaf(-pre, xm1, x.x), y1 = fmaf(-pre, x.x, x.y);
        energy = fmaf(y0, y0, fmaf(y1, y1, energy));
        v[j] = make_float2(y0 * wreg[j].x, y1 * wreg[j].y);
      }
      v[7] = make_float2(0.f, 0.f);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = 64 * j + 2 * lane;
        float y0 = 0.f, y1 = 0.f;
        if (i < n_valid) {
          const float x0 = s[i];
          float xm1 = s[i - 1];
          if (i == 0 && pmode == 1) xm1 = x0;
          y0 = pmode ? fmaf(-pre, xm1, x0) : x0;
          if (i + 1 < n_valid) {
            const float x1 = s[i + 1];
            y1 = pmode ? fmaf(-pre, x0, x1) : x1;
          }
        }
        energy = fmaf(y0, y0, fmaf(y1, y1, energy));
        const float w0 = i < FL ? win[i] : 0.f, w1 = i + 1 < FL ? win[i + 1] : 0.f;
        v[j] = make_float2(y0 * w0, y1 * w1);
      }
    }
    finish_frame(f, v, energy);
  }
  __syncthreads();
  }  // staged path

  // ---- delta / delta-delta / CMVN
  const int N = cfg.delta_n;
  float den = 0.f;
  for (int n = 1; n <= N; ++n) den += 2.f * n * n;
  const float inv_den = den > 0.f ? 1.f / den : 0.f;
  float* out = a.out_feats + f_begin * OD;
  const int total = T * OD;
  const int j = tid & 63, g = tid >> 6;         // feature column / frame phase for the column passes
  const int ord_j = j >= 2 * NC ? 2 : (j >= NC ? 1 : 0), jj_j = j - ord_j * NC;
  if (materialize && cfg.delta_order > 0) {
    // all orders laid out as [order][T][NC] right behind the cepstra; thread = (column tid % 16.., frame phase)
    const int cols = NC <= 16 ? 16 : 32, jj = tid & (cols - 1), tg = tid / cols, tstep = 256 / cols;
    for (int ord = 1; ord <= cfg.delta_order; ++ord) {
      const float* src = ceps + (size_t)(ord - 1) * T * NC;
      float* dst = ceps + (size_t)ord * T * NC;
      if (jj < NC)
        for (int t = tg; t < T; t += tstep) dst[t * NC + jj] = delta_at(src, NC, T, t, jj, N, inv_den);
      __syncthreads();
    }
  }
  auto value = [&](int t, int ord, int jj, int jfull) -> float {
    if (materialize) return ceps[((size_t)ord * T + t) * NC + jj];
    return feat_at(ceps, NC, T, t, jfull, N, inv_den);
  };
  if (cfg.cmvn) {
    float part = 0.f;
    if (j < OD)
      for (int t = g; t < T; t += 4) part += value(t, ord_j, jj_j, j);
    red[tid] = part;
    __syncthreads();
    if (tid < 64) mean[tid] = (red[tid] + red[64 + tid] + red[128 + tid] + red[192 + tid]) / (float)T;
    __syncthreads();
    part = 0.f;
    if (j < OD) {
      const float mu = mean[j];
      for (int t = g; t < T; t += 4) {
        const float d = value(t, ord_j, jj_j, j) - mu;
        part = fmaf(d, d, part);
      }
    }
    red[tid] = part;
    __syncthreads();
    if (tid < 64) {
      float sd = sqrtf((red[tid] + red[64 + tid] + red[128 + tid] + red[192 + tid]) / (float)T);
      if (sd < 10.f * 1.1920929e-7f) sd = 1.f;  // sklearn/preprocessing/_data.py:127
      istd[tid] = 1.f / sd;
    }
    __syncthreads();
  }
  // flattened, fully coalesced store; (t, column) advance incrementally: no integer division in the loop
  {
    const int dq = 256 / OD, dr = 256 - dq * OD;
    int t = tid / OD, jc = tid - t * OD;
    for (int idx = tid; idx < total; idx += 256) {
      const int ord = jc >= 2 * NC ? 2 : (jc >= NC ? 1 : 0);
      float val = value(t, ord, jc - ord * NC, jc);
      if (cfg.cmvn) val = (val - mean[jc]) * istd[jc];
      out[idx] = val;
      t += dq;
      jc += dr;
      if (jc >= OD) { jc -= OD; ++t; }
    }
  }
  __syncthreads();  // the cepstra / statistics of this utterance are dead: the next one may overwrite them
  }  // utterances
}

}  // namespace ff

bool frontend_fast_supported(const ssp_frontend_cfg& c) {
  return c.nfft == 512 && c.framing <= 2 && c.log_type <= 2 && c.n_filt <= ff::MAXF && c.n_ceps <= ff::MAXC &&
         c.frame_len >= 2 && c.frame_shift >= 1 &&
         (ff::W - 1) * c.frame_shift + c.frame_len + 1 <= 256 * 8;
}

size_t frontend_fast_smem(const ssp_frontend_cfg& c, int max_frames, bool mat) {
  return ff::carve_floats(c, max_frames, mat, nullptr, nullptr) * sizeof(float);
}

int launch_frontend_fast(const FrontendArgs& a, int64_t n_utts, size_t* smem_out, cudaStream_t st) {
  // materialise delta / delta-delta when that still leaves room for two CTAs per SM
  const size_t with = frontend_fast_smem(a.cfg, a.max_frames, true);
  const bool mat = a.cfg.delta_order > 0 && with <= 110 * 1024;
  const size_t smem = mat ? with : frontend_fast_smem(a.cfg, a.max_frames, false);
  if (smem_out) *smem_out = smem;
  // persistent CTAs: the per-CTA tables (twiddles, filterbank segments) are built once and amortised over the utterances
  // a CTA walks; 16 CTAs per SM slot keep the block scheduler's dynamic balancing for ragged batches
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    SSP_CUDA_OK(cudaGetDevice(&dev));
    SSP_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const unsigned grid = (unsigned)(n_utts < 16 * (int64_t)sms ? n_utts : 16 * (int64_t)sms);
  const ssp_frontend_cfg& c = a.cfg;
  const bool sk = c.frame_len == ff::SK_FL && c.frame_shift == ff::SK_SH && c.n_filt == ff::SK_NF && c.n_ceps == ff::SK_NC &&
                  c.framing == 0 && c.preemph_mode == 1 && c.spec_type == 0 && c.spec_scale == 1.0f && c.log_type == 0 &&
                  c.log_add == 0.0f && c.log_zero_floor == 0.0f && c.energy_mode <= 1;
#define SSP_FE_LAUNCH(T, SK)                                                                                              \
  do {                                                                                                                    \
    SSP_CUDA_OK(cudaFuncSetAttribute(ff::frontend512_kernel<T, SK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    ff::frontend512_kernel<T, SK><<<grid, 256, smem, st>>>(a, mat ? 1 : 0, n_utts);                                       \
  } while (0)
  if (c.pcm_dtype == 0) {
    if (sk) SSP_FE_LAUNCH(int16_t, true); else SSP_FE_LAUNCH(int16_t, false);
  } else {
    if (sk) SSP_FE_LAUNCH(float, true); else SSP_FE_LAUNCH(float, false);
  }
#undef SSP_FE_LAUNCH
  // the sidekit instantiation keeps the plain name (the benchmark's launch log); the other one says which it is
  SSP_LAUNCH_CHECK(sk ? "frontend512_kernel" : "frontend512_kernel<generic>");
  return SSP_OK;
}

}  // namespace ssp
