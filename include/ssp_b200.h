/*
 * ssp_b200.h -- C ABI of the B200-native MFCC -> diag-GMM-UBM hot path.
 *
 * The reference (kleinzcy/speech_signal_processing) is pure Python; its "plugin API" for
 * this path is a set of module-level Python names (SURVEY.md section 8(b)).  Each entry point below
 * names the reference call it replaces; the modules of speech_signal_processing_b200 bind them with
 * ctypes and re-expose the reference's own signatures (mfcc, MFCC, delta, scale,
 * GaussianMixture.fit/score, GMM()).  See INTEGRATION.md for the reference-side binding.
 *
 * Conventions
 *   - every pointer marked "device" is a CUDA device pointer into caller-owned memory
 *     (torch CUDA tensors in the Python host); nothing is allocated behind the caller's back;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); calls are asynchronous;
 *   - return value: 0 on success, negative SSP_E* on error, message via ssp_last_error();
 *   - there is NO CPU fallback: every entry point launches sm_100a kernels or fails.
 */
#ifndef SSP_B200_H_
#define SSP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSP_OK 0
#define SSP_EINVAL (-1)   /* bad argument / unsupported shape */
#define SSP_ECUDA (-2)    /* CUDA runtime error (see ssp_last_error) */
#define SSP_EUNSUP (-3)   /* valid request this build does not implement */

#define SSP_ABI_VERSION 1

int ssp_abi_version(void);
const char* ssp_last_error(void);
/* How many kernels this library has launched since load / the last reset, and which:
 * "kernel_name:count,kernel_name:count,..." (valid until the next call); evidence for bench.py's
 * "gpu_launches" and for the tests that assert WHICH kernel served a call. */
int64_t ssp_launch_count(void);
void ssp_reset_launch_count(void);
const char* ssp_launch_log(void);

/* ------------------------------------------------------------------------------------------
 * Front-end: PCM -> cepstra (+delta, +delta-delta, +per-utterance CMVN) in ONE kernel.
 * Replaces, per utterance: sidekit.frontend.features.mfcc (bound at GMM_UBM.py:20, called
 * GMM_UBM.py:89), GMM_UBM.delta (GMM_UBM.py:53-69), np.hstack (:91), preprocessing.scale
 * (:93); and utils.processing.MFCC (utils/processing.py:110-144) with the "processing" tables.
 * ---------------------------------------------------------------------------------------- */
typedef struct ssp_frontend_cfg {
  int32_t frame_len;     /* samples per frame (400)                                          */
  int32_t frame_shift;   /* hop (160)                                                        */
  int32_t nfft;          /* [64, 4096], >= frame_len; a power of two runs an FFT, any other
                            length (utils/processing.py:129: nfft = frame length) a direct DFT */
  int32_t n_filt;        /* mel filters (24 sidekit, 26 psf, 40 processing.py)               */
  int32_t n_ceps;        /* cepstra kept (13); n_ceps*(1+delta_order) <= 64, or up to n_filt
                            (<= 256) with delta_order 0 and cmvn 0                            */
  int32_t framing;       /* 0: floor((N-len)/shift)+1, no padding (sidekit)
                            1: 1+ceil((N-len)/shift), zero-padded tail (psf)
                            2: ceil(N/shift), zero-padded tail (utils/processing.py:27)
                            3: 1+floor(N/shift), frame f centred on sample f*shift, edges
                               mirrored (librosa center=True, pad_mode='reflect'); preemph_mode 0
                            4: as 3 with zero padding (pad_mode='constant')                    */
  int32_t preemph_mode;  /* 0 none; 1 per frame, y[0]=x[0]-p*x[0] (sidekit);
                            2 whole signal, y[0]=x[0] (psf)                                    */
  float preemph;         /* 0.97                                                             */
  int32_t spec_type;     /* 0 power re^2+im^2; 1 magnitude                                    */
  float spec_scale;      /* spectrum multiplied by this (1/nfft for psf and processing.py)   */
  int32_t log_type;      /* 0 natural log; 1 log10; 2 none (PLP: raw critical-band energies);
                            3 dB: 10 log10(max(x, log_zero_floor)) (librosa power_to_db, amin)  */
  float log_add;         /* added before the log (1e-8 at utils/processing.py:105)           */
  float log_zero_floor;  /* if > 0: exact zeros are replaced by this before the log (psf eps) */
  int32_t energy_mode;   /* 0 none; 1 sidekit ln(sum y^2) of the pre-emphasised, un-windowed
                            frame -> out_log_energy; 2 psf: c0 := ln(sum of scaled spectrum)  */
  int32_t delta_order;   /* 0, 1 (reference, 26-d) or 2 (39-d)                                 */
  int32_t delta_n;       /* regression half-width N (2)                                       */
  int32_t cmvn;          /* 1: per-utterance mean/variance normalisation (ddof=0, std<10eps->1) */
  int32_t pcm_dtype;     /* 0 int16, 1 float32                                                 */
} ssp_frontend_cfg;

/* Number of frames the framing rule yields for n_samples (0 if the utterance is too short). */
int64_t ssp_frontend_num_frames(const ssp_frontend_cfg* cfg, int64_t n_samples);
/* Longest utterance (in frames) the fused single-pass kernel accepts (shared-memory bound). */
int64_t ssp_frontend_max_frames(const ssp_frontend_cfg* cfg);

/*
 * pcm            device, int16 or float32 samples of all utterances back to back
 * sample_offsets device int64[n_utts+1], start of each utterance in `pcm` (16-byte aligned
 *                starts are not required)
 * window         device float[frame_len]
 * fb_start/len   device int32[n_filt]: first FFT bin and number of bins of each triangle
 * fb_offset      device int32[n_filt]: offset of the triangle's weights in fb_weights
 * fb_weights     device float[sum(fb_len)]
 * dct            device float[n_ceps * n_filt] (row-major; lifter folded in)
 * frame_offsets  device int64[n_utts+1], prefix sum of ssp_frontend_num_frames per utterance
 * out_feats      device float[total_frames * n_ceps*(1+delta_order)]
 * out_log_energy device float[total_frames] or NULL
 */
int ssp_frontend_batch(const void* pcm, const int64_t* sample_offsets, int64_t n_utts,
                       const ssp_frontend_cfg* cfg, const float* window, const int32_t* fb_start,
                       const int32_t* fb_len, const int32_t* fb_offset, const float* fb_weights,
                       const float* dct, const int64_t* frame_offsets, int64_t max_frames_per_utt,
                       float* out_feats, float* out_log_energy, void* stream);

/*
 * Back half of sidekit.frontend.features.plp (bound at GMM_UBM.py:20, called :94-99 for feature_type 'PLP'; a port of
 * rastamat's rastaplp): critical-band energies (ssp_frontend_batch with a Bark filterbank, log_type 2 and an identity
 * "DCT") -> RASTA filtering of the log energies along time (optional) -> equal-loudness weighting and cube-root
 * compression (^0.33), first / last band replicated -> autocorrelation (real inverse DFT of the even extension, given
 * as the matrix `idft`) -> Levinson-Durbin of order n_ceps - 1 -> LPC cepstra -> lifter.  Double precision inside.
 * bands         device float[total_frames * n_bands], OVERWRITTEN (RASTA runs in place)
 * eql           device double[n_bands]           equal-loudness weights
 * idft          device double[n_ceps * n_bands]  r[k] = sum_i idft[k, i] * post[i]
 * lift          device double[n_ceps]
 * out_ceps      device float[total_frames * n_ceps]
 */
int ssp_plp_post(float* bands, const int64_t* frame_offsets, int64_t n_utts, int32_t n_bands, int32_t n_ceps,
                 const double* eql, const double* idft, const double* lift, int32_t rasta, float* out_ceps,
                 void* stream);

/*
 * Back half of librosa.feature.mfcc as MFCC_DTW.py:27-30 calls it (MFCC_lib; SURVEY 8(f).3): log-mel power in dB
 * (ssp_frontend_batch with framing 3, log_type 3 and an identity "DCT") -> power_to_db's top_db clip against the maximum
 * of the whole utterance -> DCT-II rows.
 * mel_db        device float[total_frames * n_mels]
 * dct           device float[n_ceps * n_mels]
 * top_db        clip to (utterance max - top_db); negative: no clip (librosa top_db=None)
 * out_ceps      device float[total_frames * n_ceps]
 */
int ssp_mel_db_post(const float* mel_db, const int64_t* frame_offsets, int64_t n_utts, int32_t n_mels, int32_t n_ceps,
                    const float* dct, float top_db, float* out_ceps, void* stream);

/* GMM_UBM.delta (GMM_UBM.py:53-69) on a (T, F) float32 device matrix. */
int ssp_delta(const float* feat, int64_t n_frames, int32_t n_feat, int32_t delta_n, float* out,
              void* stream);
/* sklearn.preprocessing.scale (GMM_UBM.py:93) per utterance over concatenated (T, F) features. */
int ssp_cmvn(const float* feat, const int64_t* frame_offsets, int64_t n_utts, int32_t n_feat,
             float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Voice-activity pre-filter (reference VAD.py; SURVEY 8(f).4 -- the report runs it in front of GMM-UBM).
 * ---------------------------------------------------------------------------------------- */
typedef struct ssp_vad_cfg {
  int32_t frame_len;       /* 256 (VAD.py:22; also the FFT length)                                   */
  int32_t frame_shift;     /* 128 = frame_len - overlap (VAD.py:23); == frame_len for pre-framed input */
  int32_t n_blocks;        /* sub-bands of the spectral entropy, 10 (VAD.py:79)                      */
  int32_t normalize_peak;  /* 1: divide each utterance by max|x| first (VAD.py:133)                  */
  int32_t pcm_dtype;       /* 0 int16, 1 float32                                                      */
  float eps;               /* 1e-8 (VAD.py:79)                                                        */
} ssp_vad_cfg;

/* ceil(n_samples / frame_shift) frames, zero-padded tail (VAD.py:36). */
int64_t ssp_vad_num_frames(const ssp_vad_cfg* cfg, int64_t n_samples);
/*
 * Per-frame features of VAD.py:52-108 for a batch of utterances in one launch:
 * out_zcr[f]     number of strictly negative products of neighbouring samples (ZCR, :52-63; the caller applies
 *                the `* (power > 0.1)` gate of feature(), :115)
 * out_power[f]   sum of squares in double (energy, :66-76)
 * out_entropy[f] spectral entropy of |FFT|[:128] over n_blocks sub-bands (:79-108)
 * pcm / sample_offsets / frame_offsets as in ssp_frontend_batch (frame_offsets = prefix sum of ssp_vad_num_frames).
 */
int ssp_vad_features(const void* pcm, const int64_t* sample_offsets, int64_t n_utts, const ssp_vad_cfg* cfg,
                     const int64_t* frame_offsets, float* out_zcr, double* out_power, float* out_entropy,
                     void* stream);
/*
 * VAD_detection (VAD.py:137-182): the double-threshold state machine, one utterance per thread.
 * zcr must already carry the power gate.  out_speech[f] = 1 for speech frames.  Where the reference's backward
 * search would run past index -n (IndexError) the search stops there.
 */
int ssp_vad_detect(const float* zcr, const double* power, const int64_t* frame_offsets, int64_t n_utts,
                   float zcr_gate, double ampl, double amph, int32_t min_len, uint8_t* out_speech, void* stream);

/* ------------------------------------------------------------------------------------------
 * GMM: packed models, scoring, EM/MAP sufficient statistics.
 * Replaces sklearn.mixture.GaussianMixture(covariance_type='diag').score / .fit internals as
 * called at GMM_UBM.py:158-160,169-170,185,194 (sklearn/mixture/_gaussian_mixture.py:536-553,
 * _base.py:373,393,552-582).
 * ---------------------------------------------------------------------------------------- */
typedef struct ssp_gmm_dims {
  int32_t n_models;
  int32_t n_comp;   /* K                                         */
  int32_t n_feat;   /* D (<= 80)                                 */
} ssp_gmm_dims;

/* Bytes of the packed-model buffer for these dims (0 if unsupported). */
int64_t ssp_gmm_pack_bytes(const ssp_gmm_dims* dims);
/*
 * weights   device double[n_models*K], means/variances device double[n_models*K*D].
 * out_pack  device, ssp_gmm_pack_bytes() bytes, 128-byte aligned.  Holds, per model,
 *           (a) exact fp32 rows [mu/var, -1/(2 var)] + log-constant for the CUDA-core kernels and
 *           (b) TF32-rounded, log2(e)-scaled [mu/var, -1/(2 var), c_hi, c_lo] tiles laid out as
 *               tcgen05 shared-memory images (one bulk copy per 128-component tile), their residuals (2- / 3-pass
 *               rungs), FP16 images of the same rows (single-pass rung) and BF16 hi + lo images (ssp_gmm_stats).
 */
int ssp_gmm_pack_models(const double* weights, const double* means, const double* variances,
                        const ssp_gmm_dims* dims, void* out_pack, void* stream);

#define SSP_PREC_FP32 0 /* CUDA-core FP32 FMA, ~1e-7 relative                              */
#define SSP_PREC_TF32 1 /* one tcgen05 pass, operands rounded to an 11-bit significand, FP32 accumulate in TMEM:
                           1e-4 relative on the utterance score at K >= 512 components and ~300 frames            */
#define SSP_PREC_TF32X2 2 /* two passes, A.B_hi + A.B_lo: the model operand exact to 2^-22 (its rounding is the
                             systematic part of the one-pass error), frames still rounded                       */
#define SSP_PREC_TF32X3 3 /* three passes, A_hi.B_hi + A_hi.B_lo + A_lo.B_hi: FP32-grade, ~5e-7 relative;
                             what LLRs of small models / short utterances need (abs 1e-3)                       */
/* The three tensor rungs are issued as kind::f16 from FP16 images of the pack (FP16 has TF32's 11-bit significand, one
 * MMA covers K = 16 instead of 8, tiles are half the bytes) when every model value fits FP16's range, else as kind::tf32
 * from the TF32 images; a frame outside that range (|x| > 255) is re-scored in FP32 by tc_fixup_kernel. */

/*
 * scores[u, m] = mean over the frames of utterance u of log sum_c w_c N(x_t; mu_mc, var_mc)
 * -- GaussianMixture.score for every (utterance, model) pair in one launch (GMM_UBM.py:182-197
 * makes S*N*2 separate calls).
 * feats          device float[total_frames * D]
 * frame_offsets  device int64[n_utts+1]; total_frames == frame_offsets[n_utts] (host copy, so that
 *                the launch needs no device read-back)
 * out_scores     device double[n_utts * n_models], overwritten
 * out_frame_lse  device float[n_models * total_frames] or NULL: per-frame log-likelihood
 *                (GaussianMixture.score_samples)
 */
int ssp_gmm_score(const float* feats, const int64_t* frame_offsets, int64_t n_utts,
                  int64_t total_frames, const void* pack, const ssp_gmm_dims* dims, int32_t precision,
                  double* out_scores, float* out_frame_lse, void* stream);

/*
 * Scoring of model sets that SHARE weights and variances and differ in their means only -- what mean-only
 * relevance-MAP enrolment from a UBM produces (ssp_gmm_map_adapt with flags == 1), i.e. the speaker models of
 * GMM_UBM.py:182-197 when they are adapted instead of trained from scratch.  The log-likelihood splits into a part
 * common to all models -- the full logit of a REFERENCE member of the set, [x^2, x, 1] . [-1/(2 var), mu_ref/var,
 * const], computed once per frame block with the model operand split in two TF32 pieces -- and a per-model part
 * linear in the frame, [x, 1] . [(mu - mu_ref)/var, const], so the per-model tensor-core contraction is D + 2 long
 * instead of 2D + 2 and TF32 rounding acts on the DIFFERENCE from the reference only: scores agree with
 * ssp_gmm_score(SSP_PREC_TF32) on the expanded set to TF32 rounding or better, and log-likelihood ratios against the
 * reference member are an order of magnitude tighter for MAP-adapted speakers.
 *
 * dims->n_models = number of mean sets S; weights double[K], variances double[K*D], means double[S*K*D] (device).
 * ref_model      (at pack time) index of the reference member: the UBM's own means if they are part of the set,
 *                else any member.  Its per-frame maximum logit also stabilises the exponentials.
 * workspace      device, ssp_gmm_score_shared_workspace_bytes() bytes, 16-byte aligned (else SSP_EINVAL); may be NULL
 *                when that is 0.  Large model sets
 *                are scored in groups whose tile images stay resident in L2 while all frames pass by; the per-frame
 *                exponent stabilisers found while the first group is scored live here (4 bytes per frame).
 */
int64_t ssp_gmm_shared_pack_bytes(const ssp_gmm_dims* dims);
int ssp_gmm_pack_shared(const double* weights, const double* variances, const double* means,
                        const ssp_gmm_dims* dims, int32_t ref_model, void* out_pack, void* stream);
int64_t ssp_gmm_score_shared_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames);
int ssp_gmm_score_shared(const float* feats, const int64_t* frame_offsets, int64_t n_utts,
                         int64_t total_frames, const void* pack, const ssp_gmm_dims* dims, double* out_scores,
                         float* out_frame_lse, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * Posterior-weighted sufficient statistics over segments of frames:
 *   N[s,c] = sum_t g_tc, F[s,c,:] = sum_t g_tc x_t, S[s,c,:] = sum_t g_tc x_t^2, loglik[s] = sum_t log p(x_t);
 *   g = posterior (sklearn _base.py:552-582; M-step inputs of _gaussian_mixture.py:312-313,250-252).
 * dims->n_models == 1: every segment under the ONE model (all frames = one segment for UBM EM; one segment per speaker
 *   for MAP enrolment).
 * dims->n_models == n_segs > 1: segment s under model s -- S models trained together, the per-speaker loop of
 *   GMM_UBM.py:154-165 as one call per EM iteration (D <= 39, n_models <= 1024).
 * Outputs are ACCUMULATED into (caller zeroes them).
 * frame_lse      device float[total_frames]: per-frame log-likelihood under the model (written by this call)
 * workspace      device, ssp_gmm_stats_workspace_bytes() bytes, 16-byte aligned (else SSP_EINVAL: the frame images
 *                are written with 16-byte stores and read by cp.async.bulk).  The tensor-core path (tcgen05,
 *                D <= 39) keeps there (a) the tcgen05 operand images of the frames -- [x, x^2, 1, 1] as BF16 hi + lo
 *                rows and as TF32 hi + lo with the frame index contiguous, segments padded to 64 frames: 12 * roundup(2D+2,
 *                16) bytes per frame, 960 at D = 39 -- and (b) per-component-tile log-sum-exp partials.  A NULL or short
 *                workspace is SSP_EINVAL (the FP32 CUDA-core kernels serve D > 39 only, never as a silent fallback).
 * reuse_images   nonzero: the workspace still holds the images of THIS feats / seg_offsets from an earlier call (the
 *                frames of an EM run never change, only the model does): the preparation pass is skipped.
 */
int ssp_gmm_stats(const float* feats, const int64_t* seg_offsets, int64_t n_segs,
                  int64_t total_frames, const void* pack, const ssp_gmm_dims* dims, float* frame_lse, double* out_n,
                  double* out_f, double* out_s, double* out_loglik, void* workspace, int64_t workspace_bytes,
                  int32_t reuse_images, void* stream);
/* Scratch bytes ssp_gmm_stats needs for these dims, frames and segments (0: none). */
int64_t ssp_gmm_stats_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames, int64_t n_segs);

/*
 * Frame posteriors (GaussianMixture.predict_proba / predict, sklearn _base.py:552-582 and argmax of it):
 *   gamma[t, c] = w_c N(x_t; c) / sum_c' w_c' N(x_t; c'),  label[t] = lowest c maximising log w_c + log N(x_t; c)
 *   (numpy's argmax rule on ties).
 * Models and segments as in ssp_gmm_stats: dims->n_models == 1 puts every segment under the one model,
 * dims->n_models == n_segs puts segment s under model s (D <= 39 only; SSP_EUNSUP above).
 * Always FP32 grade: for D <= 39 the logits are the 3 x BF16 tcgen05 products of ssp_gmm_stats (same frame images,
 * same per-frame log-likelihood), for 40 <= D <= 80 the FP32 CUDA-core kernels of SSP_PREC_FP32.
 * out_resp       device float[total_frames * K] (row-major, K unpadded) or NULL
 * out_label      device int64[total_frames] or NULL; at least one of the two (both NULL is SSP_EINVAL).  Labels alone
 *                skip the log-sum-exp pass.
 * out_frame_lse  device float[total_frames] or NULL: per-frame log-likelihood (computed when out_resp or this is set)
 * workspace      device, ssp_gmm_posteriors_workspace_bytes() bytes, 16-byte aligned (else SSP_EINVAL).  For D <= 39 it
 *                has the layout
 *                of the ssp_gmm_stats workspace (same size, frame images at the same place), so one workspace serves both
 *                calls on the same frames and reuse_images works across them (label the frames of an EM run
 *                without preparing them again).
 * reuse_images   nonzero: the workspace still holds the images of THIS feats / seg_offsets (see ssp_gmm_stats).
 */
int ssp_gmm_posteriors(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                       const void* pack, const ssp_gmm_dims* dims, float* out_resp, int64_t* out_label,
                       float* out_frame_lse, void* workspace, int64_t workspace_bytes, int32_t reuse_images,
                       void* stream);
/* Scratch bytes ssp_gmm_posteriors needs for these dims, frames and segments (0: unsupported dims). */
int64_t ssp_gmm_posteriors_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames, int64_t n_segs);

/*
 * Top-C Gaussian selection (the first half of the fast scoring of Reynolds, Quatieri & Dunn 2000): for every frame the C
 * components with the largest L_c(t) = log w_c + log N(x_t; c) under ONE model, in descending order, the lower index
 * first on equal values.  D <= 39 (SSP_EUNSUP above), 1 <= C <= min(K, 64) (else SSP_EINVAL), dims->n_models == 1.
 * FP32 grade: the logits are the 3 x BF16 tcgen05 products of ssp_gmm_posteriors.
 * out_idx        device int32[total_frames * C]
 * out_logit      device float[total_frames * C]: L_c(t) of the selected components
 * workspace      device, ssp_gmm_top_components_workspace_bytes() bytes, 16-byte aligned (else SSP_EINVAL).  The layout of
 *                the ssp_gmm_stats / ssp_gmm_posteriors workspace with a longer last section: the frame images sit at the
 *                same place, so reuse_images works across the three calls on the same frames.
 */
int ssp_gmm_top_components(const float* feats, const int64_t* seg_offsets, int64_t n_segs, int64_t total_frames,
                           const void* pack, const ssp_gmm_dims* dims, int32_t c, int32_t* out_idx, float* out_logit,
                           void* workspace, int64_t workspace_bytes, int32_t reuse_images, void* stream);
/* Scratch bytes ssp_gmm_top_components needs (0: unsupported dims or C). */
int64_t ssp_gmm_top_components_workspace_bytes(const ssp_gmm_dims* dims, int64_t total_frames, int64_t n_segs, int32_t c);

/*
 * Top-C scoring of a model set that shares weights and variances (the second half of the fast scoring): with S_t the
 * selection of ssp_gmm_top_components under the reference member r,
 *   l_s(t) = log sum_{c in S_t} exp(L_s,c(t)),   L_s,c(t) = L_r,c(t) + a_s,c . x_t + b_s,c,
 *   a_s,c = (mu_s,c - mu_r,c) / var_c,   b_s,c = -1/2 sum_d (mu_s,c - mu_r,c)(mu_s,c + mu_r,c) / var_c,
 * scores[u, s] = mean of l_s(t) over the frames of utterance u (0 for an empty utterance).  With C = K this is the exact
 * score.  The (a, b) table is the pack: FP32, component-major ([K][S][roundup(D + 1, 4)]); the weights cancel in L_s - L_r
 * and are not part of it.  dims->n_models = S, weights / variances / means as in ssp_gmm_pack_shared, D <= 39.
 * The frames are scored in chunks of ssp_gmm_topc_chunk_frames() frames: each chunk's (frame, slot) pairs are routed by
 * component, the difference terms of a component for all models are FP32 FMAs, the log-sum-exp over the C slots is taken
 * per (frame, model) in FP32 and the utterance sums are double.
 * idx, logit     device int32 / float [total_frames * C] from ssp_gmm_top_components (entries outside [0, K) are skipped)
 * out_scores     device double[n_utts * S]
 * out_frame_lse  device float[S * total_frames] or NULL: l_s(t)
 * workspace      device, ssp_gmm_score_topc_workspace_bytes() bytes, 16-byte aligned (else SSP_EINVAL)
 */
int64_t ssp_gmm_topc_pack_bytes(const ssp_gmm_dims* dims);
int ssp_gmm_pack_topc(const double* variances, const double* means, const ssp_gmm_dims* dims, int32_t ref_model,
                      void* out_pack, void* stream);
int64_t ssp_gmm_topc_chunk_frames(void);
int64_t ssp_gmm_score_topc_workspace_bytes(const ssp_gmm_dims* dims, int32_t c, int64_t total_frames);
int ssp_gmm_score_topc(const float* feats, const int64_t* frame_offsets, int64_t n_utts, int64_t total_frames,
                       const int32_t* idx, const float* logit, int32_t c, const void* pack, const ssp_gmm_dims* dims,
                       double* out_scores, float* out_frame_lse, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * Top-C scoring of a model set MAP-adapted from its reference member r in weights and variances too (component c of
 * every model is component c of r): as ssp_gmm_score_topc, with
 *   L_s,c(t) = L_r,c(t) + k_s,c + a_s,c . y + b_s,c . y^2,   y = x_t - mu_r,c,   delta = mu_s,c - mu_r,c,
 *   a = delta / var_s,c,   b = -1/2 (1/var_s,c - 1/var_r,c),
 *   k = log(w_s,c / w_r,c) - 1/2 sum_d log(var_s,c / var_r,c) - 1/2 sum_d delta^2 / var_s,c.
 * A model (or component) with the reference's parameters has a row of zeros and scores L_r,c(t) bit for bit.
 * The pack: the table [K][S][roundup(2D + 1, 4)] FP32 rows [a (D), b (D), k, 0..] computed in double, then the reference
 * means [K][roundup(D, 4)] in FP32; ssp_gmm_topc_adapted_pack_bytes() bytes, 16-byte aligned.  weights [S][K], means and
 * variances [S][K][D] double (positive, finite weights and variances: the table takes their logarithms), D <= 39,
 * ref_model in [0, S).  ssp_gmm_score_topc_adapted takes the arguments of ssp_gmm_score_topc, with this pack, and its
 * workspace from ssp_gmm_score_topc_workspace_bytes().
 */
int64_t ssp_gmm_topc_adapted_pack_bytes(const ssp_gmm_dims* dims);
int ssp_gmm_pack_topc_adapted(const double* weights, const double* means, const double* variances, const ssp_gmm_dims* dims,
                              int32_t ref_model, void* out_pack, void* stream);
int ssp_gmm_score_topc_adapted(const float* feats, const int64_t* frame_offsets, int64_t n_utts, int64_t total_frames,
                               const int32_t* idx, const float* logit, int32_t c, const void* pack, const ssp_gmm_dims* dims,
                               double* out_scores, float* out_frame_lse, void* workspace, int64_t workspace_bytes,
                               void* stream);

/*
 * M-step on device (sklearn _gaussian_mixture.py:312-313,250-252,898): from (all-reduced)
 * statistics to weights/means/variances, double precision, for n_models models at once (arrays [n_models][K](xD)).
 * nk = N + 10*eps_of(stat_dtype); mu = F/nk; var = S/nk - mu^2 + reg_covar; w = nk/sum(nk).
 */
int ssp_gmm_mstep(const double* n, const double* f, const double* s, int32_t n_models, int32_t n_comp, int32_t n_feat,
                  double reg_covar, double nk_eps, double* out_weights, double* out_means,
                  double* out_variances, void* stream);

/*
 * Relevance-MAP adaptation (Reynolds et al. 2000; absent from the reference code, SURVEY F4)
 * for a batch of speakers from their UBM statistics: alpha = n/(n+r);
 * mu^ = alpha F/n + (1-alpha) mu_ubm.  flags bit0: adapt means, bit1: weights, bit2: variances.
 */
int ssp_gmm_map_adapt(const double* n, const double* f, const double* s, const int64_t* seg_offsets,
                      int64_t n_spk, const double* ubm_weights, const double* ubm_means,
                      const double* ubm_variances, int32_t n_comp, int32_t n_feat, double relevance,
                      int32_t flags, double* out_weights, double* out_means, double* out_variances,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * Dynamic time warping: the template-matching stage of the MFCC+DTW recogniser (MFCC_DTW.py, dtw 1.4
 * `accelerated_dtw`).  Symmetric step pattern, no window, no slope weights, no normalisation:
 *   D[i,j] = C[i,j] + min(D[i-1,j-1], D[i-1,j], D[i,j-1]),  D[-1,-1] = 0, the rest of row / column -1 = +inf,
 *   distance = D[n-1, m-1];  C = scipy cdist(x, y, metric), computed in FP32 in difference form.
 * The distance is exactly symmetric in its two arguments; the "column" side (r, y) is staged in shared memory and
 * bounds the length (ssp_dtw_max_len), the "row" side takes sequences of up to INT32_MAX / 2 frames (a pair with a
 * longer one comes out NaN).
 * ---------------------------------------------------------------------------------------- */
#define SSP_DTW_EUCLIDEAN 0   /* sqrt(sum (x - y)^2) */
#define SSP_DTW_SQEUCLIDEAN 1 /* sum (x - y)^2       */
#define SSP_DTW_CITYBLOCK 2   /* sum |x - y|         */

/* Longest column-side sequence (frames) the kernels accept at this feature width; 0 if dim is outside [1, 64]. */
int64_t ssp_dtw_max_len(int32_t dim);
/*
 * out_dist[a * n_r + b] = DTW distance of q sequence a and r sequence b, every pair in one launch (dtw_kernel).
 * q, r           device float[total frames * dim], sequences back to back
 * q_offsets      device int64[n_q + 1]; r_offsets device int64[n_r + 1] (every sequence at least one frame)
 * max_r_len      host: longest r sequence (sizes the shared memory; <= ssp_dtw_max_len(dim), else SSP_EUNSUP)
 * out_dist       device float[n_q * n_r]
 */
int ssp_dtw_batch(const float* q, const int64_t* q_offsets, int64_t n_q, const float* r, const int64_t* r_offsets,
                  int64_t n_r, int32_t dim, int32_t metric, int64_t max_r_len, float* out_dist, void* stream);
/*
 * One pair with its matrices (dtw_full_kernel): out_cost = C, out_acc = D, both device float[n_x * n_y] row-major.
 * n_y <= ssp_dtw_max_len(dim), else SSP_EUNSUP.
 */
int ssp_dtw_full(const float* x, int64_t n_x, const float* y, int64_t n_y, int32_t dim, int32_t metric,
                 float* out_cost, float* out_acc, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SSP_B200_H_ */
