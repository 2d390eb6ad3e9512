"""GMM kernels at the count bounds of their loops, against the float64 oracle.

The width tests (test_gpu_gmm_widths.py) take every feature width and the first component tile.  This file takes the
other axis: the counts each kernel loops over, where state carried from one iteration to the next (exponent
stabilisers, TMEM ring phases, partial-sum chunks, per-segment running sums) is first reused.

* ``gmm_score_tc_kernel`` (all four rungs of ``ssp_gmm_score``): component tiles of 128, model counts around the 4 TMEM
  slots and the model-parity comb buffer, a stabiliser redo on tiles other than the first, frames per persistent wave.
* ``gmm_score_sv_kernel`` (``ssp_gmm_score_shared``): model chunks of 32, model groups in L2, frames per wave.
* ``tc_fixup_kernel`` and ``sv_fixup_kernel``: partly padded component tiles, more NaN pairs than the grid has warps.
* ``em_plan_kernel`` .. ``gmm_em_stats_kernel`` (``ssp_gmm_stats``) and the posterior kernels (``ssp_gmm_posteriors``):
  segments around the plan's 1024-thread scan, tile pairs with and without a half-empty pair, per-segment models up to
  ``kMaxTrainModels``, grids on both sides of one CTA per SM.
* ``warp_segmented_atomic_add``: 100 000 utterances of 0 to 3 frames, many runs per warp.
* The CUDA-core kernels (D > 39) at their frame and component block sizes.

Tolerances are the derived per-frame bounds of test_gpu_gmm_widths.py (C_BOUND * u * terms, and for the statistics the
FP16 pieces of the posteriors and frame values); posteriors follow from the same logit bound.  Every GPU test prints its
largest error in units of u * terms or of its bound (profiles/r3e_pytest_gpu_gmm_counts.log).
``test_count_lists_straddle_every_kernel_bound`` parses the counts out of the CUDA sources and checks that the cases
below sit on both sides of each.
"""
import ctypes as C
import functools
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pytest

from oracle import gmm as ogmm
from test_gpu_gmm_widths import C_BOUND, EM_SIMT_KERNELS, EM_TENSOR_KERNELS, U, U_GAMMA, _check_scores, _check_stats, \
    frame_bound_terms
from test_gpu_posteriors import MARGIN, SIMT, TENSOR, reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "speech_signal_processing_b200", "csrc")
RUNGS = ("fp32", "tf32", "tf32x2", "tf32x3")
TC_KERNEL = {"tf32": "gmm_score_tc_kernel", "tf32x2": "gmm_score_tc_kernel<2 passes>",
             "tf32x3": "gmm_score_tc_kernel<3 passes>"}


# ------------------------------------------------------------------------------------------------ kernel counts
def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _int(pattern, text):
    m = re.search(pattern, text)
    assert m, pattern
    return int(m.group(1))


@functools.lru_cache(maxsize=None)
def kernel_counts():
    """The loop counts of the GMM kernels, parsed out of the CUDA sources (on first use, so that a pattern that stops
    matching fails the tests that need it, not the collection of this file)."""
    common, tc, sv, em, simt = (_source(n) for n in ("common.cuh", "gmm_score_tc.cu", "gmm_score_sv.cu", "gmm_em_tc.cu",
                                                      "gmm_simt.cu"))
    with open(os.path.join(ROOT, "speech_signal_processing_b200", "mixture.py")) as f:
        mixture = f.read()
    return {
        "kTileN": _int(r"constexpr int kTileN = (\d+);", common),
        "kSvTileN": _int(r"constexpr int kSvTileN = (\d+);", common),
        "kSvChunk": _int(r"kSvChunk = (\d+)", common),
        "kSvSlots": _int(r"kSvSlots = (\d+)", common),
        "kSvUnit": _int(r"kSvUnit = (\d+);", common),
        "kMaxTrainModels": _int(r"constexpr int kMaxTrainModels = (\d+);", common),
        "FIT_BATCH_MAX": _int(r"or n_models > (\d+):", mixture),
        "TC_BM": _int(r"constexpr int BM = (\d+);", tc),
        "TC_NSLOT": _int(r"constexpr int NSLOT = (\d+);", tc),
        "TC_MB1": _int(r"if \(parts == 1\) SSP_TC_LAUNCH\((\d+), 1\);", tc),
        "TC_MB2": _int(r"else if \(parts == 2\) SSP_TC_LAUNCH\((\d+), 2\);", tc),
        "TC_MB3": _int(r"else SSP_TC_LAUNCH\((\d+), 3\);", tc),
        "TC_FIX_CTAS_PER_SM": _int(r"cap = (\d+) \* \(int64_t\)num_sms;", tc),
        "TC_FIX_THREADS": _int(r"tc_fixup_kernel<<<\(unsigned\)\(want < cap \? want : cap\), (\d+),", tc),
        "SV_FIX_CTAS_PER_SM": _int(r"cap = (\d+) \* \(int64_t\)num_sms\(\);", sv),
        "SV_FIX_THREADS": _int(r"sv_fixup_kernel<<<\(unsigned\)\(want < cap \? want : cap\), (\d+),", sv),
        "EM_BN": _int(r"constexpr int BN = (\d+);", em),
        "EM_IMG": _int(r"constexpr int IMG = (\d+);", em),
        "EM_BLK": _int(r"constexpr int BLK = (\d+);", em),
        "EM_PLAN_THREADS": _int(r"em_plan_kernel<<<1, (\d+),", em),
        "EM_PLAN_SCAN": _int(r"\(a\.n_segs \+ \d+\) / (\d+);", em),
        "EM_PLAN_SHARED": _int(r"__shared__ int64_t part\[(\d+)\];", em),
        "kSF": _int(r"constexpr int kSF = (\d+);", simt),
        "kSC": _int(r"constexpr int kSC = (\d+);", simt),
        "kTF": _int(r"constexpr int kTF = (\d+);", simt),
        "kTG": _int(r"constexpr int kTG = (\d+);", simt),
    }


# the values the cases of this file were written for: a change to one of them fails here until the cases follow
PINNED = {"kTileN": 128, "kSvTileN": 64, "kSvChunk": 32, "kSvSlots": 6, "kSvUnit": 256, "kMaxTrainModels": 1024,
          "FIT_BATCH_MAX": 1024, "TC_BM": 128, "TC_NSLOT": 4, "TC_MB1": 2, "TC_MB2": 2, "TC_MB3": 1,
          "TC_FIX_CTAS_PER_SM": 4, "TC_FIX_THREADS": 256, "SV_FIX_CTAS_PER_SM": 4, "SV_FIX_THREADS": 256, "EM_BN": 128,
          "EM_IMG": 128, "EM_BLK": 64, "EM_PLAN_THREADS": 1024, "EM_PLAN_SCAN": 1024, "EM_PLAN_SHARED": 1024,
          "kSF": 64, "kSC": 32, "kTF": 64, "kTG": 64}

# cases
TC_K = (255, 256, 257, 1023, 1025, 2047, 2049)       # components of the general scorer, at TC_D
TC_D = (13, 39)
TC_MODELS = (1, 3, 4, 5, 8, 9)                        # around the 4 TMEM slots and the model-parity comb
SV_MODELS = (31, 32, 33, 63, 64, 65)                  # around the 32-model partial-sum chunks
SV_K = (65, 127, 1024)
SV_GROUP_SETS = (32, 33, 64, 65)                      # scored with groups capped at SV_GROUP_CAP models
SV_GROUP_CAP = 32
FIX_K = (65, 129)                                     # the last component tile partly padded in both kernels
WAVES = ((1, -1), (1, 1), (2, 1))                     # frames = waves * SMs * unit + delta
EM_SEGS = (1023, 1024, 1025, 2048, 2049, 100003)      # around the plan kernel's 1024-thread scan
EM_K = (128, 129, 256, 257, 384, 385)                 # 1 .. 4 tiles: whole and half-empty tile pairs
EM_LONG = (63, 64, 65, 129, 2000)                     # long segments mixed into the 0 .. 3 frame ones
SEG_MODELS = (1, 2, "sms", 1023, 1024)                # per-segment models ("sms": the device's SM count)
SEG_MODELS_REFUSED = 1025
TINY_UTTS = 100003
SIMT_K = (31, 32, 33, 63, 64, 65)                     # the CUDA-core kernels (D = 40) ...
SIMT_LENS = (1, 63, 64, 65, 129)                      # ... and their 64-frame blocks


def _straddles(values, unit):
    """Some multiple of unit in values with its two neighbours."""
    return any(v % unit == 0 and v - 1 in values and v + 1 in values for v in values)


def _both_sides(values, bound):
    return any(v <= bound for v in values) and any(v > bound for v in values)


def _n_tiles(k, tile):
    return -(-k // tile)


def test_count_lists_straddle_every_kernel_bound():
    B = kernel_counts()
    assert B == PINNED, "a GMM kernel count changed: move the cases of this file with it"
    # general scorer: tile edges at 2, 8 and 16 tiles; models around the TMEM slots, both parities above them
    assert _straddles(TC_K, B["kTileN"]) and {1023, 1025, 2047, 2049} <= set(TC_K)
    assert all(_n_tiles(k, B["kTileN"]) > 1 for k in TC_K)
    n = B["TC_NSLOT"]
    assert {n - 1, n, n + 1, 2 * n, 2 * n + 1} <= set(TC_MODELS) and 1 in TC_MODELS
    assert {B["TC_MB1"], B["TC_MB2"], B["TC_MB3"]} == {1, 2}             # units of 128 and 256 frames: WAVES per rung
    # shared-variance scorer: chunks of 32 models (and more models than accumulator slots), tiles of 64
    c = B["kSvChunk"]
    assert set(SV_MODELS) == {c - 1, c, c + 1, 2 * c - 1, 2 * c, 2 * c + 1} and min(SV_MODELS) > B["kSvSlots"]
    assert any(k % B["kSvTileN"] for k in SV_K) and any(k % B["kSvTileN"] == 0 for k in SV_K)    # padded and whole tiles
    assert SV_GROUP_CAP % c == 0 and set(SV_GROUP_SETS) == {SV_GROUP_CAP, SV_GROUP_CAP + 1, 2 * SV_GROUP_CAP, 2 * SV_GROUP_CAP + 1}
    # fix-up passes: a partly padded last tile in both kernels (the pair count is derived from the parsed grid)
    assert all(k % B["kTileN"] and k % B["kSvTileN"] and k > B["kSvTileN"] for k in FIX_K)
    # EM: the plan scan, tile pairs (odd and even tile counts, one and two pairs), blocks and images of a segment
    t = B["EM_PLAN_THREADS"]
    assert B["EM_PLAN_SCAN"] == B["EM_PLAN_SHARED"] == t
    assert _straddles(EM_SEGS, t) and {2 * t, 2 * t + 1} <= set(EM_SEGS) and max(EM_SEGS) > 64 * t
    tiles = [_n_tiles(k, B["EM_BN"]) for k in EM_K]
    assert {1, 2, 3, 4} <= set(tiles) and {k % B["EM_BN"] for k in EM_K} == {0, 1}
    assert _straddles(EM_LONG, B["EM_BLK"]) and B["EM_IMG"] + 1 in EM_LONG and max(EM_LONG) > 8 * B["EM_IMG"]
    # per-segment models: up to kMaxTrainModels accepted, one more refused; fit_batch batches exactly those
    m = B["kMaxTrainModels"]
    assert {m - 1, m} <= set(SEG_MODELS) and SEG_MODELS_REFUSED == m + 1 and B["FIT_BATCH_MAX"] == m
    # CUDA-core kernels: component steps of kSC, groups of kTG, frame blocks of kSF / kTF
    assert _straddles(SIMT_K, B["kSC"]) and _straddles(SIMT_K, B["kTG"])
    assert _straddles(SIMT_LENS, B["kSF"]) and _straddles(SIMT_LENS, B["kTF"]) and max(SIMT_LENS) > 2 * B["kSF"]


# ------------------------------------------------------------------------------------------------ helpers
def _sms():
    import torch

    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _ubms(n_models, k, d, seed):
    """n_models GMMs (S, K) / (S, K, D) from synth_ubm with consecutive seeds."""
    from speech_signal_processing_b200 import synth

    ps = [synth.synth_ubm(k, d, seed=seed + s) for s in range(n_models)]
    return tuple(np.stack([p[i] for p in ps]) for i in range(3))


def _ragged(total, seed, hi=600):
    """Utterance lengths in [1, hi] summing to total."""
    rs = np.random.RandomState(seed)
    lens = []
    while sum(lens) < total:
        lens.append(int(min(rs.randint(1, hi + 1), total - sum(lens))))
    return lens


def _offsets(lens):
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


def _sample(w, mu, var, lens, seed):
    from speech_signal_processing_b200 import synth

    total = int(np.sum(lens))
    return synth.sample_gmm(w, mu, var, max(total, 1), seed=seed)[:total], _offsets(lens)


def _tiny_lens(n, seed):
    """n segments of 0 .. 3 frames."""
    return np.random.RandomState(seed).randint(0, 4, size=n)


def _score(ms, x, offs, precision):
    import torch

    from speech_signal_processing_b200 import _lib

    _lib.load().ssp_reset_launch_count()
    got, lse = ms.score(torch.as_tensor(x, device=ms.device), offs, precision=precision, want_frame_lse=True)
    log = _lib.launch_log()
    if precision == "fp32":
        assert set(log) == {"gmm_score_simt_kernel"}, log
    else:
        assert TC_KERNEL[precision] in log and set(log) <= {TC_KERNEL[precision], "tc_fixup_kernel"}, log
    return got.cpu().numpy(), lse.cpu().numpy()


def _score_rungs(w, mu, var, x, offs, what, rungs=RUNGS):
    import speech_signal_processing_b200 as ssp

    ms = ssp.ModelSet(w, mu, var)
    report = []
    for precision in rungs:
        got, lse = _score(ms, x, offs, precision)
        c = _check_scores(got, lse, x, offs, w, mu, var, U[precision], f"{what} {precision}")
        empty = np.diff(offs) == 0
        assert (got[empty] == 0).all()
        report.append(f"{precision} {c:.2f}")
    print(f"{what}: largest error / (u * terms): " + ", ".join(report))


def _score_shared(sms, x, offs):
    import torch

    from speech_signal_processing_b200 import _lib

    _lib.load().ssp_reset_launch_count()
    got, lse = sms.score(torch.as_tensor(x, device=sms.device), offs, want_frame_lse=True)
    log = _lib.launch_log()
    assert set(log) == {"gmm_score_sv_kernel", "sv_fixup_kernel"}, log
    return got.cpu().numpy(), lse.cpu().numpy(), log


def _check_shared(got, lse, x, offs, w, var, means, what):
    """Speakers (all but the last model) with u = 2^-11, the reference member (last) with its measured u."""
    s = len(means)
    W, V = np.tile(w, (s, 1)), np.tile(var, (s, 1, 1))
    spk = _check_scores(got[:, :-1], lse[:-1], x, offs, W[:-1], means[:-1], V[:-1], U["tf32"], f"{what} speakers")
    ref = _check_scores(got[:, -1:], lse[-1:], x, offs, W[-1:], means[-1:], V[-1:], U["sv_reference"], f"{what} reference")
    assert (got[np.diff(offs) == 0] == 0).all()
    return spk, ref


def _shared_models(n_spk, k, d, seed):
    from speech_signal_processing_b200 import synth

    w, mu, var = synth.synth_ubm(k, d, seed=seed)
    means = np.concatenate([synth.synth_speaker_means(mu, n_spk, seed=seed + 1, shift=0.3), mu[None]])   # last = reference
    return w, var, means


def _check_posteriors(g, lab, lse, x, seg, params, u, per_segment=False):
    """Posteriors, labels and per-frame log-likelihoods against float64, under params[0] for every frame or (per_segment)
    params[s] for segment s.  A logit and the frame's log-likelihood are each within C_BOUND * u * terms_t (u = 2^-18 for
    the 3 x BF16 logits of the tensor kernels, 2^-22 for the FP32 CUDA-core kernels), so a posterior is within
    gamma * expm1(2 C_BOUND u terms_t), plus the FP32 rounding of its exponential (2^-22 of itself) and FP32's underflow
    (2^-126).  Labels on the frames whose float64 top-2 margin exceeds MARGIN, as in test_gpu_posteriors.py.  Returns
    the largest posterior error (over the posteriors FP32 represents as normal numbers) and log-likelihood error in units
    of their bounds."""
    w, mu, var = params
    if per_segment:
        spans = [(s, a, b) for s, (a, b) in enumerate(zip(seg[:-1], seg[1:])) if b > a]
        refs = [reference(x[a:b], w[s], mu[s], var[s]) + (frame_bound_terms(x[a:b], w[s], mu[s], var[s]),) for s, a, b in spans]
        r_lse, r_g, r_lab, margin, terms = (np.concatenate(p) for p in zip(*refs))
    else:
        r_lse, r_g, r_lab, margin = reference(x, w[0], mu[0], var[0])
        terms = frame_bound_terms(x, w[0], mu[0], var[0])
    cg = cl = 0.0
    if g is not None:
        bound = r_g * (np.expm1(2 * C_BOUND * u * terms)[:, None] + U["fp32"]) + 2.0 ** -126
        err = np.abs(g - r_g)
        normal = r_g >= 2.0 ** -126                 # the ratio where underflow does not decide it
        cg = float((err[normal] / bound[normal]).max())
        assert (err <= bound).all(), cg
    if lse is not None:
        err = np.abs(lse - r_lse)
        cl = float((err / (C_BOUND * u * terms)).max())
        assert (err <= C_BOUND * u * terms).all(), cl
    if lab is not None:
        ok = margin > MARGIN
        np.testing.assert_array_equal(lab[ok], r_lab[ok])
    return cg, cl


# ------------------------------------------------------------------------------------------------ general scorer
@pytest.mark.gpu
@pytest.mark.parametrize("d", TC_D)
@pytest.mark.parametrize("k", TC_K)
def test_general_scorer_component_tiles(k, d):
    """2 .. 17 component tiles per model: the stabiliser and the running sum cross every tile edge of a model."""
    w, mu, var = _ubms(2, k, d, seed=k + d)
    x, offs = _sample(w[0], mu[0], var[0], [1, 300, 2, 129], seed=k)
    _score_rungs(w, mu, var, x, offs, f"K {k} D {d}")


@pytest.mark.gpu
@pytest.mark.parametrize("n_models", TC_MODELS)
def test_general_scorer_model_counts(n_models):
    """Tiles of consecutive models cycle through the 4 TMEM slots; the column halves merge through a comb buffer that
    alternates with the model's parity."""
    w, mu, var = _ubms(n_models, 129, 13, seed=100 + n_models)
    x, offs = _sample(w[0], mu[0], var[0], [300, 1, 257, 64, 2], seed=n_models)
    _score_rungs(w, mu, var, x, offs, f"{n_models} models K 129 D 13")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [257, 1025])
def test_general_scorer_redo_beyond_the_first_tile(k):
    """The stabiliser is carried from model to model and checked on every tile.  Models alternate between thousands of
    nats apart (``far``) and ``split`` models whose first tile lies ~160 nats below the rest: after the first tile has set
    the stabiliser, the second tile's maximum exceeds it by more than 2^64 and the running sum of the first must be
    rescaled (a redo on a tile other than the first).  ``flip`` has the far components last (no redo: they vanish)."""
    from speech_signal_processing_b200 import synth

    d = 13
    w, mu, var = synth.synth_ubm(k, d, seed=k)
    far = mu + 25.0                        # every component ~25 sigma from the frames: log-likelihood ~ -5000
    split = mu.copy()
    split[:128] += 5.0                     # tile 0: ~ -160 nats below the other tiles
    flip = mu.copy()
    flip[128:] += 5.0
    models_mu = np.stack([split, far, split, mu, split, flip, far, split])
    s = len(models_mu)
    W, V = np.tile(w, (s, 1)), np.tile(var, (s, 1, 1))
    x, offs = _sample(w, mu, var, [300, 257, 40, 1], seed=k + 1)
    _score_rungs(W, models_mu, V, x, offs, f"redo K {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("waves,delta", WAVES)
def test_general_scorer_frames_per_wave(waves, delta):
    """Persistent CTAs take units of 256 frames (128 in the 3-pass rung) in turn: one frame short of a full wave, one
    frame more, and two waves and a frame.  The mbarrier phases follow the unit count of each CTA."""
    B = kernel_counts()
    w, mu, var = _ubms(3, 129, 13, seed=200)
    for precision in ("tf32", "tf32x2", "tf32x3"):
        unit = B["TC_BM"] * (B["TC_MB3"] if precision == "tf32x3" else B["TC_MB1"])
        total = waves * _sms() * unit + delta
        x, offs = _sample(w[0], mu[0], var[0], _ragged(total, seed=total), seed=total)
        _score_rungs(w, mu, var, x, offs, f"{total} frames ({waves} x SMs x {unit} {delta:+d})", rungs=(precision,))


# ------------------------------------------------------------------------------------------------ shared variance
@pytest.mark.gpu
@pytest.mark.parametrize("k", SV_K)
@pytest.mark.parametrize("n_spk", SV_MODELS)
def test_shared_variance_model_chunks(n_spk, k):
    """Models are scored in chunks of 32 whose partial sums are cleared after each read; the last chunk has S % 32
    models.  The set is n_spk speakers plus the reference member."""
    import speech_signal_processing_b200 as ssp

    w, var, means = _shared_models(n_spk - 1, k, 13, seed=300 + k + n_spk)   # n_spk models with the reference
    x, offs = _sample(w, means[0], var, [1, 300, 255, 2], seed=n_spk)
    sms = ssp.SharedModelSet(w, var, means)
    got, lse, _ = _score_shared(sms, x, offs)
    spk, ref = _check_shared(got, lse, x, offs, w, var, means, f"{n_spk} models K {k}")
    print(f"{n_spk} models K {k}: largest error / (u * terms): speakers {spk:.2f}, reference member {ref:.2f}")


@pytest.mark.gpu
@pytest.mark.parametrize("waves,delta", WAVES)
def test_shared_variance_frames_per_wave(waves, delta):
    import speech_signal_processing_b200 as ssp

    total = waves * _sms() * kernel_counts()["kSvUnit"] + delta
    w, var, means = _shared_models(34, 65, 13, seed=400)
    x, offs = _sample(w, means[1], var, _ragged(total, seed=total), seed=total + 1)
    got, lse, _ = _score_shared(ssp.SharedModelSet(w, var, means), x, offs)
    spk, ref = _check_shared(got, lse, x, offs, w, var, means, f"{total} frames")
    print(f"{total} frames ({waves} x SMs x 256 {delta:+d}): largest error / (u * terms): speakers {spk:.2f}, "
          f"reference member {ref:.2f}")


GROUP_SCRIPT = r"""
import os, sys
import numpy as np, torch
sys.path.insert(0, %r)
import speech_signal_processing_b200 as ssp
from speech_signal_processing_b200 import synth
k, d = 65, 13
w, mu, var = synth.synth_ubm(k, d, seed=500)
lens = [298, 1, 300, 255, 257, 129]
out = {}
for s in %r:
    means = np.concatenate([synth.synth_speaker_means(mu, s - 1, seed=501, shift=0.3), mu[None]])
    utts = [synth.sample_gmm(w, means[i %% s], var, n, seed=502 + i) for i, n in enumerate(lens)]
    sms = ssp.SharedModelSet(w, var, means)
    feats, offs = ssp.mixture.concat_utterances(utts, sms.device)
    got, lse = sms.score(feats, offs, want_frame_lse=True)
    out[f"scores_{s}"], out[f"lse_{s}"] = got.cpu().numpy(), lse.cpu().numpy()
    out[f"grouped_{s}"] = np.array(sms._ws is not None)
np.savez(sys.argv[1], **out)
"""


@pytest.mark.gpu
def test_shared_variance_group_splits(tmp_path):
    """Model groups in L2 (SSP_SV_GROUP_MB is read once per process, hence a subprocess per cap): with groups capped at
    32 models, 32 models are one launch, 33 are 32 + 1, 64 are 32 + 32 and 65 are 32 + 32 + 1.  Every grouped result is
    bit-equal to the single-group result, and against the oracle."""
    from speech_signal_processing_b200 import synth

    per_model = 128 * 16 * 2                              # Kp = 128 components, KS = 16 FP16 columns
    cap_mb = (SV_GROUP_CAP + 0.5) * per_model / 1048576   # rounds down to SV_GROUP_CAP models
    script = tmp_path / "groups.py"
    script.write_text(GROUP_SCRIPT % (ROOT, SV_GROUP_SETS))
    out = {}
    for mb in (f"{cap_mb:.6f}", "0"):
        path = str(tmp_path / f"groups_{mb}.npz")
        r = subprocess.run([sys.executable, str(script), path], env=dict(os.environ, SSP_SV_GROUP_MB=mb), capture_output=True,
                           text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        out[mb] = dict(np.load(path))
    grouped, single = out[f"{cap_mb:.6f}"], out["0"]
    w, mu, var = synth.synth_ubm(65, 13, seed=500)
    lens = [298, 1, 300, 255, 257, 129]
    for s in SV_GROUP_SETS:
        assert bool(grouped[f"grouped_{s}"]) == (s > SV_GROUP_CAP) and not bool(single[f"grouped_{s}"])
        np.testing.assert_array_equal(grouped[f"scores_{s}"], single[f"scores_{s}"])
        np.testing.assert_array_equal(grouped[f"lse_{s}"], single[f"lse_{s}"])
        means = np.concatenate([synth.synth_speaker_means(mu, s - 1, seed=501, shift=0.3), mu[None]])
        x = np.concatenate([synth.sample_gmm(w, means[i % s], var, n, seed=502 + i) for i, n in enumerate(lens)])
        spk, ref = _check_shared(grouped[f"scores_{s}"], grouped[f"lse_{s}"], x, _offsets(lens), w, var, means, f"{s} grouped")
        print(f"{s} models, groups of {SV_GROUP_CAP}: bit-equal to one group; largest error / (u * terms): speakers "
              f"{spk:.2f}, reference member {ref:.2f}")


# ------------------------------------------------------------------------------------------------ fix-up passes
def _wild(x, offs, which, value=300.0):
    """One frame of |x| > 255 (x^2 leaves FP16's range) in each utterance of `which`."""
    x = x.copy()
    for j in which:
        if offs[j + 1] > offs[j]:
            x[(offs[j] + offs[j + 1]) // 2, j % x.shape[1]] = value if j % 2 else -value
    return x


def _subset(got, lse, x, offs, utts):
    """Rows of the utterances `utts`, their frames and the matching offsets."""
    idx = np.concatenate([np.arange(offs[j], offs[j + 1]) for j in utts]) if len(utts) else np.zeros(0, np.int64)
    return got[utts], lse[:, idx], x[idx], _offsets([offs[j + 1] - offs[j] for j in utts])


def _fixup_split(got, lse, x, offs, wild, w, mu, var, u_fix, u_tensor, what):
    """The re-scored utterances (FP32 fix-up) and the others (tensor kernel) against the oracle, each within its bound."""
    utts = np.arange(len(offs) - 1)
    cf = _check_scores(*_subset(got, lse, x, offs, utts[wild]), w, mu, var, u_fix, f"{what} fix-up")
    ct = _check_scores(*_subset(got, lse, x, offs, utts[~wild]), w, mu, var, u_tensor, f"{what} tensor") if (~wild).any() else 0.0
    assert np.isfinite(got).all()
    return cf, ct


@pytest.mark.gpu
@pytest.mark.parametrize("k", FIX_K)
def test_fixup_on_a_partly_padded_tile(k):
    """Frames outside FP16's range turn the single-pass rung's and the shared-variance kernel's scores of their
    utterance to NaN; ``tc_fixup_kernel`` re-scores over the K real components, ``sv_fixup_kernel`` over whole tiles of
    64 (the padded components of the last tile must add nothing)."""
    import speech_signal_processing_b200 as ssp

    d = 13
    w, mu, var = _ubms(2, k, d, seed=600 + k)
    lens = [64, 130, 1, 300, 7]
    x, offs = _sample(w[0], mu[0], var[0], lens, seed=k)
    wild = np.array([False, True, True, False, True])
    x = _wild(x, offs, np.flatnonzero(wild))
    got, lse = _score(ssp.ModelSet(w, mu, var), x, offs, "tf32")
    cf, ct = _fixup_split(got, lse, x, offs, wild, w, mu, var, U["fp32"], U["tf32"], f"tc K {k}")
    print(f"tc_fixup_kernel K {k}: largest error / (u * terms): fix-up {cf:.2f}, tensor {ct:.2f}")
    sw, sv, smeans = _shared_models(2, k, d, seed=610 + k)
    xs = _wild(_sample(sw, smeans[0], sv, lens, seed=k + 1)[0], offs, np.flatnonzero(wild))
    got, lse, _ = _score_shared(ssp.SharedModelSet(sw, sv, smeans), xs, offs)
    # the fix-up pass uses the FP16 images of the speakers' differences (11-bit) and the FP16 hi + lo common part
    W, V = np.tile(sw, (3, 1)), np.tile(sv, (3, 1, 1))
    cs = _fixup_split(got[:, :2], lse[:2], xs, offs, wild, W[:2], smeans[:2], V[:2], U["tf32"], U["tf32"], f"sv K {k}")
    cr = _fixup_split(got[:, 2:], lse[2:], xs, offs, wild, W[2:], smeans[2:], V[2:], U["sv_reference"], U["sv_reference"],
                      f"sv reference K {k}")
    print(f"sv_fixup_kernel K {k}: largest error / (u * terms): speakers fix-up {cs[0]:.2f} / tensor {cs[1]:.2f}, "
          f"reference member {cr[0]:.2f} / {cr[1]:.2f}")


@pytest.mark.gpu
def test_fixup_with_more_pairs_than_warps():
    """Every (utterance, model) pair needs the fix-up pass and there are more pairs than the fix-up grid has warps
    (ctas per SM x SMs x threads / 32): each warp takes several pairs in its grid-stride loop."""
    import speech_signal_processing_b200 as ssp

    B = kernel_counts()
    sms = _sms()
    d, n_models = 13, 3
    for kernel, ctas, threads in (("tc", B["TC_FIX_CTAS_PER_SM"], B["TC_FIX_THREADS"]),
                                  ("sv", B["SV_FIX_CTAS_PER_SM"], B["SV_FIX_THREADS"])):
        warps = ctas * sms * threads // 32
        n_utts = warps // n_models + 700
        lens = 1 + np.random.RandomState(7).randint(0, 3, size=n_utts)
        k = 65
        if kernel == "tc":
            w, mu, var = _ubms(n_models, k, d, seed=700)
            x, offs = _sample(w[0], mu[0], var[0], lens, seed=701)
            x = _wild(x, offs, range(n_utts))
            got, lse = _score(ssp.ModelSet(w, mu, var), x, offs, "tf32")
            c = _check_scores(got, lse, x, offs, w, mu, var, U["fp32"], "tc fix-up pairs")
            report = f"{c:.2f}"
        else:
            sw, sv, smeans = _shared_models(n_models - 1, k, d, seed=710)
            x, offs = _sample(sw, smeans[0], sv, lens, seed=711)
            x = _wild(x, offs, range(n_utts))
            got, lse, _ = _score_shared(ssp.SharedModelSet(sw, sv, smeans), x, offs)
            spk, ref = _check_shared(got, lse, x, offs, sw, sv, smeans, "sv fix-up pairs")
            report = f"speakers {spk:.2f}, reference member {ref:.2f}"
        assert n_utts * n_models > warps
        print(f"{kernel} fix-up: {n_utts * n_models} pairs over {warps} warps: largest error / (u * terms): {report}")


# ------------------------------------------------------------------------------------------------ EM statistics
def _em_lens(n_segs, seed):
    """0 .. 3 frames per segment, empty segments at the edges of the plan kernel's per-thread chunks, and the EM_LONG
    segments at seeded positions."""
    t = kernel_counts()["EM_PLAN_THREADS"]
    per = -(-n_segs // t)
    lens = _tiny_lens(n_segs, seed)
    edges = np.arange(0, n_segs, per)
    if per > 1:
        lens[edges[::7]] = 0
        lens[np.minimum(edges[3::7] + per - 1, n_segs - 1)] = 0
    else:
        lens[::97] = 0
    lens[0] = lens[-1] = 0
    pos = np.random.RandomState(seed + 1).choice(np.arange(1, n_segs - 1), size=len(EM_LONG), replace=False)
    lens[pos] = EM_LONG
    return lens


def _check_stats_all(stats, x, seg, w, mu, var, sample=None):
    """Every segment: sum(N) is its length, its log-likelihood is the oracle's within the bound of _check_stats, an empty
    segment is exactly zero.  Then N, F, S of every segment (or of a seeded sample) with _check_stats.  Returns the
    largest log-likelihood error in units of u * terms."""
    import torch

    n, f, s, ll = (t.cpu().numpy() for t in stats)
    lens = np.diff(seg)
    empty = lens == 0
    assert (n[empty] == 0).all() and (f[empty] == 0).all() and (s[empty] == 0).all() and (ll[empty] == 0).all()
    assert (np.abs(n.sum(axis=1) - lens) <= 2 * U_GAMMA * lens).all()
    lse = ogmm.score_samples(x, w, mu, var)
    terms = frame_bound_terms(x, w, mu, var)
    cl, ct = np.concatenate([[0], np.cumsum(lse)]), np.concatenate([[0], np.cumsum(terms)])
    ref, tsum = cl[seg[1:]] - cl[seg[:-1]], ct[seg[1:]] - ct[seg[:-1]]
    err = np.abs(ll - ref)
    assert (err <= C_BOUND * U["stats"] * tsum).all(), float((err / np.maximum(tsum, 1e-300)).max())
    worst = float((err[~empty] / (U["stats"] * tsum[~empty])).max())
    idx = np.arange(len(lens)) if sample is None else np.sort(np.random.RandomState(0).choice(len(lens), sample, replace=False))
    idx = np.union1d(idx, np.flatnonzero(lens > 3))        # the long segments always
    sub = tuple(torch.from_numpy(a[idx]) for a in (n, f, s, ll))
    xs = np.concatenate([x[seg[i] : seg[i + 1]] for i in idx])
    _check_stats(sub, xs, _offsets(lens[idx]), lambda i: (w, mu, var))
    return worst, len(idx)


EM_CASES = [(1023, 129), (1024, 128), (1025, 257), (2048, 256), (2049, 385), (100003, 129)] + \
           [(1025, k) for k in EM_K if k not in (257,)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_segs,k", EM_CASES)
def test_em_statistics_segment_counts(n_segs, k):
    """One model, n_segs segments of 0 .. 3 frames with long ones mixed in.  The plan kernel gives each of its 1024
    threads ceil(n_segs / 1024) segments; the merge kernel carries a segment's log-likelihood until the segment changes;
    the statistics pass flushes TMEM at segment ends; one CTA per pair of 128-component tiles.  At 100 003 segments the
    N / log-likelihood identities are checked for every segment and N, F, S for a seeded sample of 400."""
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    d = 13
    w, mu, var = _ubms(1, k, d, seed=800 + k)
    lens = _em_lens(n_segs, seed=n_segs)
    x, seg = _sample(w[0], mu[0] * 0.9, var[0] * 1.2, lens, seed=n_segs + k)
    ms = ssp.ModelSet(w, mu, var)
    _lib.load().ssp_reset_launch_count()
    stats = ms.stats(torch.as_tensor(x, device=ms.device), seg)
    assert set(_lib.launch_log()) == EM_TENSOR_KERNELS, _lib.launch_log()
    worst, checked = _check_stats_all(stats, x, seg, w[0], mu[0], var[0], sample=400 if n_segs > 4096 else None)
    print(f"{n_segs} segments ({int(seg[-1])} frames) K {k}: N, F, S of {checked} segments; largest log-likelihood "
          f"error / (u * terms): {worst:.2f}")


@pytest.mark.gpu
def test_em_grid_cases_straddle_one_cta_per_sm():
    """The statistics and LSE passes size their grids as min(SMs / tile pairs, blocks of the frame total): the cases above
    have fewer and more 64-frame blocks than CTAs."""
    B = kernel_counts()
    sms = _sms()
    sides = set()
    for n_segs, k in EM_CASES:
        total = int(_em_lens(n_segs, seed=n_segs).sum())
        gx = max(1, sms // ((_n_tiles(k, B["EM_BN"]) + 1) // 2))
        nb_lo = -(-total // B["EM_BLK"])
        sides |= {nb_lo > gx, (nb_lo + 1) // 2 > gx}     # block chunks (statistics), image chunks (LSE, posteriors)
    assert sides == {True, False}


# ------------------------------------------------------------------------------------------------ per-segment models
def _seg_model_count(n):
    return _sms() if n == "sms" else n


def _per_segment_case(n, k, d, seed):
    """n models and n segments (0 .. 3 frames, a few longer), segment s drawn from model s."""
    from speech_signal_processing_b200 import synth

    w, mu, var = _ubms(n, k, d, seed=seed)
    lens = _tiny_lens(n, seed)
    lens[:: max(1, n // 3)] = 65
    if n > 2:
        lens[1] = 0
    x = np.concatenate([synth.sample_gmm(w[s], mu[s], var[s], max(int(c), 1), seed=seed + s)[: int(c)]
                        for s, c in enumerate(lens)])
    return w, mu, var, x, _offsets(lens)


@pytest.mark.gpu
@pytest.mark.parametrize("n", SEG_MODELS)
def test_per_segment_models(n):
    """ssp_gmm_stats and ssp_gmm_posteriors with n_models == n_segs: grid z = segment, SMs / (pairs x segments) CTAs per
    segment (clamped to 1 from SMs segments on), up to kMaxTrainModels models."""
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    n = _seg_model_count(n)
    k, d = 129, 13
    w, mu, var, x, seg = _per_segment_case(n, k, d, seed=900 + n)
    ms = ssp.ModelSet(w, mu, var)
    feats = torch.as_tensor(x, device=ms.device)
    _lib.load().ssp_reset_launch_count()
    stats = ms.stats(feats, seg)
    assert set(_lib.launch_log()) == EM_TENSOR_KERNELS, _lib.launch_log()
    c = _check_stats(stats, x, seg, lambda i: (w[i], mu[i], var[i]))
    _lib.load().ssp_reset_launch_count()
    g, lab, lse = ms.posteriors(feats, seg, resp=True, labels=True)
    assert set(_lib.launch_log()) == TENSOR["both"], _lib.launch_log()
    cg, cl = _check_posteriors(g.cpu().numpy(), lab.cpu().numpy(), lse.cpu().numpy(), x, seg, (w, mu, var), U["stats"],
                               per_segment=n > 1)
    print(f"{n} per-segment models ({int(seg[-1])} frames): statistics log-likelihood {c:.2f} of u * terms; posteriors "
          f"{cg:.2f} and frame lse {cl:.2f} of their bounds")


@pytest.mark.gpu
def test_per_segment_models_beyond_the_training_limit():
    """kMaxTrainModels + 1 models carry no statistics images: both entry points refuse per-segment models cleanly, and
    fit_batch trains such a batch one model at a time with the result of the per-model loop."""
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib, synth

    n = SEG_MODELS_REFUSED
    w, mu, var, x, seg = _per_segment_case(n, 129, 13, seed=950)
    ms = ssp.ModelSet(w, mu, var)
    feats = torch.as_tensor(x, device=ms.device)
    with pytest.raises(NotImplementedError, match="per-segment models"):
        ms.stats(feats, seg)
    with pytest.raises(NotImplementedError, match="per-segment models"):
        ms.posteriors(feats, seg)
    k, d = 4, 13
    xs, inits = [], []
    for i in range(n):
        wi, mi, vi = synth.synth_ubm(k, d, seed=960 + i)
        xs.append(synth.sample_gmm(wi, mi, vi, 8, seed=970 + i))
        inits.append((wi, mi + 0.2, np.ones_like(vi)))
    kw = dict(covariance_type="diag", max_iter=1)
    _lib.load().ssp_reset_launch_count()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        batched = ssp.fit_batch(xs, n_components=k, weights_init=[a for a, _, _ in inits], means_init=[b for _, b, _ in inits],
                                precisions_init=[1.0 / c for _, _, c in inits], **kw)
        assert _lib.launch_log()["gmm_em_stats_kernel"] >= n, _lib.launch_log()   # one statistics call per model at least
        sample = np.random.RandomState(1).choice(n, 16, replace=False)
        looped = [ssp.GaussianMixture(n_components=k, weights_init=inits[i][0], means_init=inits[i][1],
                                      precisions_init=1.0 / inits[i][2], **kw).fit(xs[i]) for i in sample]
    assert len(batched) == n
    for i, b in zip(sample, looped):     # (float64 atomics: the same sums in another order)
        a = batched[i]
        assert abs(a.lower_bound_ - b.lower_bound_) <= 1e-12 * abs(b.lower_bound_)
        np.testing.assert_allclose(a.means_, b.means_, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(a.covariances_, b.covariances_, rtol=1e-9, atol=1e-12)


# ------------------------------------------------------------------------------------------------ posteriors
@pytest.mark.gpu
@pytest.mark.parametrize("n_segs,k", EM_CASES[:6])
def test_posteriors_segment_counts(n_segs, k):
    """resp, labels and both through the C ABI into canary-filled buffers longer than T x K / T, at the segment counts
    of the statistics tests: only live frames and components are written, every frame within the stated bounds, labels
    on the frames whose float64 top-2 margin exceeds MARGIN."""
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    d = 13
    w, mu, var = _ubms(1, k, d, seed=1000 + k)
    lens = _em_lens(n_segs, seed=n_segs)
    x, seg = _sample(w[0], mu[0], var[0], lens, seed=n_segs + 1)
    ms = ssp.ModelSet(w, mu, var)
    total, pad = int(seg[-1]), 4096
    lib = _lib.load()
    feats, d_off = torch.as_tensor(x, device="cuda"), torch.as_tensor(seg, device="cuda")
    ws_bytes = int(lib.ssp_gmm_posteriors_workspace_bytes(C.byref(ms.dims), total, n_segs))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    for mode, (want_resp, want_lab) in {"resp": (True, False), "labels": (False, True), "both": (True, True)}.items():
        resp = torch.full((total * k + pad,), -7.0, dtype=torch.float32, device="cuda")
        lab = torch.full((total + pad,), -7, dtype=torch.int64, device="cuda")
        lse = torch.full((total + pad,), -7.0, dtype=torch.float32, device="cuda")
        lib.ssp_reset_launch_count()
        rc = lib.ssp_gmm_posteriors(feats.data_ptr(), d_off.data_ptr(), n_segs, total, ms.pack.data_ptr(), C.byref(ms.dims),
                                    resp.data_ptr() if want_resp else None, lab.data_ptr() if want_lab else None,
                                    lse.data_ptr() if want_resp else None, ws.data_ptr(), ws_bytes, 0, _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_posteriors")
        assert set(_lib.launch_log()) == TENSOR[mode], (mode, _lib.launch_log())
        r, lb, ls = resp.cpu().numpy(), lab.cpu().numpy(), lse.cpu().numpy()
        assert (r[total * k :] == -7.0).all() and (lb[total:] == -7).all() and (ls[total:] == -7.0).all()
        if want_resp:
            assert not (r[: total * k] == -7.0).any() and not (ls[:total] == -7.0).any()
        else:
            assert (r == -7.0).all() and (ls == -7.0).all()
        if want_lab:
            assert not (lb[:total] == -7).any()
        else:
            assert (lb == -7).all()
        cg, cl = _check_posteriors(r[: total * k].reshape(total, k) if want_resp else None, lb[:total] if want_lab else None,
                                   ls[:total] if want_resp else None, x, seg, (w, mu, var), U["stats"])
        print(f"{n_segs} segments ({total} frames) K {k} {mode}: posteriors {cg:.2f} and frame lse {cl:.2f} of their bounds")


# ------------------------------------------------------------------------------------------------ tiny utterances
@pytest.mark.gpu
def test_scoring_many_tiny_utterances():
    """100 003 utterances of 0 .. 3 frames under 2 models: every warp of the scoring epilogues folds several runs of
    equal utterance in warp_segmented_atomic_add.  Every score against the mean of its frames' float64
    log-likelihoods, every frame_lse within its bound, empty utterances exactly 0."""
    import speech_signal_processing_b200 as ssp

    k, d = 65, 13
    lens = _tiny_lens(TINY_UTTS, seed=11)
    lens[:: 1000] = 0
    w, mu, var = _ubms(2, k, d, seed=1100)
    x, offs = _sample(w[0], mu[0], var[0], lens, seed=1101)
    _score_rungs(w, mu, var, x, offs, f"{TINY_UTTS} utterances of 0 .. 3 frames", rungs=("fp32", "tf32", "tf32x3"))
    sw, sv, smeans = _shared_models(1, k, d, seed=1110)
    xs, _ = _sample(sw, smeans[0], sv, lens, seed=1111)
    got, lse, _ = _score_shared(ssp.SharedModelSet(sw, sv, smeans), xs, offs)
    spk, ref = _check_shared(got, lse, xs, offs, sw, sv, smeans, "tiny utterances shared")
    print(f"{TINY_UTTS} utterances, shared variance: largest error / (u * terms): speakers {spk:.2f}, reference member "
          f"{ref:.2f}")


# ------------------------------------------------------------------------------------------------ CUDA-core kernels
@pytest.mark.gpu
@pytest.mark.parametrize("k", SIMT_K)
def test_cuda_core_kernels_at_their_block_sizes(k):
    """D = 40: gmm_score_simt_kernel (64-frame blocks, 32 components staged per step), gmm_stats_simt_kernel (64-frame
    tiles, 64-component groups) and gmm_post_simt_kernel, on segments of 1, 63, 64, 65 and 129 frames."""
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    d = 40
    w, mu, var = _ubms(2, k, d, seed=1200 + k)
    lens = list(SIMT_LENS) + [0]
    x, offs = _sample(w[0], mu[0] * 0.9, var[0] * 1.2, lens, seed=k)
    _score_rungs(w, mu, var, x, offs, f"CUDA cores K {k}", rungs=("fp32",))
    ms = ssp.ModelSet(w[:1], mu[:1], var[:1])
    feats = torch.as_tensor(x, device=ms.device)
    _lib.load().ssp_reset_launch_count()
    stats = ms.stats(feats, offs)
    assert set(_lib.launch_log()) == EM_SIMT_KERNELS, _lib.launch_log()
    c = _check_stats(stats, x, offs, lambda i: (w[0], mu[0], var[0]))
    print(f"CUDA cores K {k}: statistics log-likelihood {c:.2f} of u * terms")
    _lib.load().ssp_reset_launch_count()
    g, lab, lse = ms.posteriors(feats, offs, resp=True, labels=True)
    assert set(_lib.launch_log()) == SIMT["both"], _lib.launch_log()
    cg, cl = _check_posteriors(g.cpu().numpy(), lab.cpu().numpy(), lse.cpu().numpy(), x, offs, (w[:1], mu[:1], var[:1]), U["fp32"])
    print(f"CUDA cores K {k}: posteriors {cg:.2f} and frame lse {cl:.2f} of their bounds")
