"""Every path of the two front-end kernels, and every size bound they choose by, against a float64 recipe reference.

``ssp_frontend_batch`` picks one of three kernels from the configuration:

* ``frontend512_kernel``: the sidekit instantiation of the nfft = 512 kernel (400 / 160 framing, 24 filters, 13 cepstra,
  sidekit conventions).  On int16 PCM whose base is 4-byte aligned it loads sample pairs straight from global memory
  (one loop for utterances that start on an even sample, one for odd); otherwise it stages int16 or float32 samples.
* ``frontend512_kernel<generic>``: the same kernel for any other nfft = 512 recipe inside its support.  It stages int16
  with 16-byte loads when the utterance starts on a 16-byte boundary, otherwise one sample per load, and float32 PCM
  one sample per load.
* ``frontend_kernel``: everything else (other FFT lengths, wider filterbanks, longer hops).

Inside the fast kernel, a filterbank of more than MAXSEG 8-bin segments falls back to per-filter dot products, and
delta / delta-delta are materialised in shared memory while the launch's longest utterance fits 110 KB.  Utterances
longer than ``ssp_frontend_max_frames`` take the chunked path of ``FrontEnd._extract_mixed``.

``reference`` below restates any ``Recipe`` in float64; ``test_reference_matches_the_oracle`` pins it to the oracle's
restatements of the reference front-ends, and ``test_kernel_constants_and_bounds`` pins the kernel constants and the
shared-memory sizes the bounds are derived from.  Both run without a device.

Tolerances: cepstra and features without CMVN |d| <= 1e-4 * max(1, |c|) (SURVEY 8(c)); log-energy 2e-5 relative;
features after CMVN the absolute tolerances of tests/test_gpu_frontend.py (5e-4 sidekit, 2e-3 otherwise).  Every test
prints its largest error (profiles/r3c_pytest_gpu_frontend_paths.log).  Largest errors measured on a B200 (1 000 W):
cepstra and deltas 9.5e-5 (sidekit convention, full-scale square wave of period 11; every other case <= 3.1e-5), load
paths 5.1e-6 (sidekit), 1.1e-5 (psf), 6.8e-7 (processing), path against path 2.9e-6, log-energy 1.1e-7, CMVN features
1.1e-4 (sidekit geometry, 128 segments) and <= 5.6e-5 elsewhere.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import frontend as ofe
from speech_signal_processing_b200 import frontend as sfe
from speech_signal_processing_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "speech_signal_processing_b200", "csrc")

CEPS_TOL = 1e-4
LOGE_TOL = 2e-5
CMVN_ATOL = {"sidekit": 5e-4}
CMVN_ATOL_OTHER = 2e-3


# ------------------------------------------------------------------------------------------------ kernel constants
def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def kernel_constants():
    """The constants the fast kernel's support, shared-memory carve-up and path choices are built from, parsed out of the
    CUDA sources (so the boundary cases below move with them)."""
    fast, gen = _source("frontend_fast.cu"), _source("frontend.cu")
    k = {}
    for name in ("W", "NH", "EXS", "MAXSEG", "PWN", "MAXF", "MAXC", "PF"):
        m = re.search(r"constexpr int %s = (\d+);" % name, fast)
        assert m, name
        k[name] = int(m.group(1))
    m = re.search(r"constexpr int EXN = (\d+) \* EXS;", fast)
    k["EXN"] = int(m.group(1)) * k["EXS"]
    m = re.search(r"constexpr int SK_FL = (\d+), SK_SH = (\d+), SK_NF = (\d+), SK_NC = (\d+);", fast)
    k["SK_FL"], k["SK_SH"], k["SK_NF"], k["SK_NC"] = (int(g) for g in m.groups())
    m = re.search(r"with <= (\d+) \* 1024", fast)
    k["MAT_BYTES"] = int(m.group(1)) * 1024
    m = re.search(r"\(ff::W - 1\) \* c\.frame_shift \+ c\.frame_len \+ 1 <= 256 \* (\d+)", fast)
    k["STAGE_SAMPLES"] = 256 * int(m.group(1))
    m = re.search(r"c\.frame_len >= (\d+)", fast)
    k["MIN_FL"] = int(m.group(1))
    m = re.search(r"kFrontendSmemMax = (\d+) \* 1024", gen)
    k["SMEM_MAX"] = int(m.group(1)) * 1024
    m = re.search(r"return nfft <= (\d+) \? (\d+) : \(nfft <= (\d+) \? (\d+) : (\d+)\);", gen)
    k["WARPS"] = tuple(int(g) for g in m.groups())
    return k


# the values the boundary cases of this file were written for: a change to one of them fails here until they follow
PINNED = {"W": 8, "NH": 256, "EXS": 36, "EXN": 288, "MAXSEG": 128, "PWN": 272, "MAXF": 64, "MAXC": 32, "PF": 8,
          "SK_FL": 400, "SK_SH": 160, "SK_NF": 24, "SK_NC": 13, "MAT_BYTES": 110 * 1024, "STAGE_SAMPLES": 2048,
          "MIN_FL": 2, "SMEM_MAX": 226 * 1024, "WARPS": (512, 8, 1024, 4, 2)}
K = kernel_constants()


def cfg_of(recipe, delta_order=0, delta_n=2, cmvn=False, pcm_dtype=0):
    """``FrontEnd._cfg`` without a device."""
    from speech_signal_processing_b200 import _lib

    r = recipe
    return _lib.FrontendCfg(r.frame_len, r.frame_shift, r.nfft, r.fbank.shape[0], r.dct.shape[0], r.framing, r.preemph_mode,
                            r.preemph, r.spec_type, r.spec_scale, r.log_type, r.log_add, r.log_zero_floor, r.energy_mode,
                            delta_order, delta_n, int(cmvn), pcm_dtype)


def fast_supported(c):
    return (c.nfft == 512 and c.framing <= 2 and c.log_type <= 2 and c.n_filt <= K["MAXF"] and c.n_ceps <= K["MAXC"]
            and c.frame_len >= K["MIN_FL"] and c.frame_shift >= 1
            and (K["W"] - 1) * c.frame_shift + c.frame_len + 1 <= K["STAGE_SAMPLES"])


def is_sk(c):
    return (c.frame_len == K["SK_FL"] and c.frame_shift == K["SK_SH"] and c.n_filt == K["SK_NF"] and c.n_ceps == K["SK_NC"]
            and c.framing == 0 and c.preemph_mode == 1 and c.spec_type == 0 and c.spec_scale == 1.0 and c.log_type == 0
            and c.log_add == 0.0 and c.log_zero_floor == 0.0 and c.energy_mode <= 1)


def kernel_of(recipe, pcm_dtype=0):
    c = cfg_of(recipe, pcm_dtype=pcm_dtype)
    if fast_supported(c):
        return "frontend512_kernel" if is_sk(c) else "frontend512_kernel<generic>"
    return "frontend_kernel"


def carve_floats(c, max_frames, mat):
    """``ff::carve_floats`` (csrc/frontend_fast.cu)."""
    W, MAXSEG, MAXF = K["W"], K["MAXSEG"], K["MAXF"]
    flp = (c.frame_len + 3) & ~3
    stg = ((W - 1) * c.frame_shift + c.frame_len + 1 + 3) & ~3
    per_warp = 2 * K["EXN"] + K["PWN"] + MAXSEG + MAXF
    f = (2 * (K["NH"] + 2) + flp + ((c.n_ceps * (c.n_filt | 1) + 3) & ~3) + 8 * MAXSEG + 2 * MAXSEG + (MAXF + 4) + 4 + 256
         + 64 + 64 + 2 * (stg + 12) + W * per_warp)
    return f + max_frames * c.n_ceps * ((1 + c.delta_order) if mat else 1)


def generic_smem_floats(c, max_frames):
    """``frontend_smem`` (csrc/frontend.cu) in floats."""
    lo, w_lo, mid, w_mid, w_hi = K["WARPS"]
    nh, nw = c.nfft // 2, (w_lo if c.nfft <= lo else (w_mid if c.nfft <= mid else w_hi))
    f = 2 * nh + 2 * (nh + 2) + ((c.frame_len + 3) & ~3) + nw * 32 + 128
    f += nw * ((4 * nh + (nh + 4) + ((c.n_filt + 3) & ~3) + 3) & ~3)
    return f + max_frames * c.n_ceps


def max_frames(c):
    """``ssp_frontend_max_frames`` for a valid configuration."""
    fixed = 4 * (carve_floats(c, 0, False) if fast_supported(c) else generic_smem_floats(c, 0))
    return 0 if fixed >= K["SMEM_MAX"] else (K["SMEM_MAX"] - fixed) // (4 * c.n_ceps)


def mat_max_frames(c):
    """Longest launch (frames of its longest utterance) for which the fast kernel materialises the deltas."""
    return (K["MAT_BYTES"] // 4 - carve_floats(c, 0, True)) // (c.n_ceps * (1 + c.delta_order))


def n_segments(recipe):
    """8-bin segments starting on a multiple of 4 bins, over the nonzero range of every filter (the kernel's table)."""
    s = 0
    for row in np.asarray(recipe.fbank, dtype=np.float64):
        nz = np.nonzero(row)[0]
        if nz.size:
            st, ln = int(nz[0]), int(nz[-1]) + 1 - int(nz[0])
            s += (st + ln - (st & ~3) + 7) >> 3
    return s


# ------------------------------------------------------------------------------------------------ float64 reference
def frame_count(recipe, n):
    L, S = recipe.frame_len, recipe.frame_shift
    if n <= 0:
        return 0
    if recipe.framing == 0:
        return 0 if n < L else (n - L) // S + 1
    if recipe.framing == 1:
        return 1 if n <= L else 1 + -(-(n - L) // S)
    if recipe.framing == 2:
        return -(-n // S)
    raise NotImplementedError("centred framing is covered through oracle.librosa_mfcc")


def samples_for(recipe, T):
    """An utterance length that gives exactly T >= 1 frames."""
    n = T * recipe.frame_shift if recipe.framing == 2 else recipe.frame_len + (T - 1) * recipe.frame_shift
    assert frame_count(recipe, n) == T
    return n


def reference(recipe, sig, delta_order=0, delta_n=2, cmvn=False, preemph32=True):
    """Any framing 0-2 recipe in float64: (features (T, n_ceps * (1 + delta_order)), log-energy (T,) or None).

    ``preemph32``: use the pre-emphasis coefficient as the kernel holds it (float32).  x[i] - p x[i - 1] cancels where
    neighbouring samples are close, and 0.97 and float32(0.97) differ by 1.3e-8 relative, which one-sample frames turn
    into 2e-4 on the cepstra."""
    r = recipe
    pre = float(np.float32(r.preemph)) if preemph32 else r.preemph
    x = np.asarray(sig, dtype=np.float64)
    n, L, S = x.shape[0], r.frame_len, r.frame_shift
    T = frame_count(r, n)
    nc = r.dct.shape[0]
    if T == 0:
        return np.zeros((0, nc * (1 + delta_order))), (np.zeros(0) if r.energy_mode == 1 else None)
    if r.preemph_mode == 2:      # whole signal, y[0] = x[0]
        x = np.concatenate([x[:1], x[1:] - pre * x[:-1]])
    idx = np.arange(L)[None, :] + S * np.arange(T)[:, None]
    valid = idx < n
    padded = np.zeros(max(n, int(idx.max()) + 1))
    padded[:n] = x
    fr = padded[idx]
    if r.preemph_mode == 1:      # per frame, the first sample is its own predecessor
        fr = fr - pre * np.concatenate([fr[:, :1], fr[:, :-1]], axis=1)
    fr = np.where(valid, fr, 0.0)
    energy = (fr * fr).sum(axis=1)
    spec = np.abs(np.fft.rfft(fr * np.asarray(r.window, dtype=np.float64)[None, :], r.nfft, axis=1)) ** 2
    if r.spec_type == 1:
        spec = np.sqrt(spec)
    spec = spec * r.spec_scale
    mel = spec @ np.asarray(r.fbank, dtype=np.float64).T
    with np.errstate(divide="ignore", invalid="ignore"):
        if r.log_zero_floor > 0:
            mel = np.where(mel == 0, r.log_zero_floor, mel)
        mel = mel + r.log_add
        mel = {0: np.log, 1: np.log10, 2: lambda v: v}[r.log_type](mel)
        ceps = mel @ np.asarray(r.dct, dtype=np.float64).T
        if r.energy_mode == 2:
            e = spec.sum(axis=1)
            ceps[:, 0] = np.log(np.where(e == 0, r.log_zero_floor, e) if r.log_zero_floor > 0 else e)
        log_e = np.log(energy) if r.energy_mode == 1 else None
    parts, d = [ceps], ceps
    for _ in range(delta_order):
        d = ofe.delta(d, delta_n)
        parts.append(d)
    feats = np.hstack(parts)
    if cmvn:
        mu = feats.mean(axis=0)
        sd = np.sqrt(((feats - mu) ** 2).mean(axis=0))
        feats = (feats - mu) / np.where(sd < 10 * np.finfo(np.float64).eps, 1.0, sd)
    return feats, log_e


def custom_fbank(seg_counts, n_bins=257, seed=0):
    """Filters of exactly the given numbers of 8-bin segments: filter m covers bins [4 m, 4 m + 8 s_m) with positive
    weights (first and last bin nonzero)."""
    rs = np.random.RandomState(seed)
    fb = np.zeros((len(seg_counts), n_bins))
    for m, s in enumerate(seg_counts):
        st = 4 * m
        assert st + 8 * s <= n_bins
        fb[m, st : st + 8 * s] = 0.05 + rs.uniform(size=8 * s)
    return fb


def sk_geometry_recipe(fbank, name="sk-custom"):
    """sidekit conventions and geometry at 16 kHz with another 24-filter bank (still the sidekit instantiation)."""
    return sfe.Recipe(name, 400, 160, 512, np.hanning(400), fbank, sfe.dct_rows(13, fbank.shape[0], first=1), framing=0,
                      preemph_mode=1, preemph=0.97, energy_mode=1)


def psf_conventions_recipe(fbank, n_ceps=13, frame_len=400, shift=160, name="psf-custom"):
    """python_speech_features conventions (generic instantiation) with another filterbank or geometry."""
    return sfe.Recipe(name, frame_len, shift, 512, np.ones(frame_len), fbank, sfe.dct_rows(n_ceps, fbank.shape[0]), framing=1,
                      preemph_mode=2, preemph=0.97, spec_scale=1.0 / 512, log_zero_floor=float(np.finfo(float).eps),
                      energy_mode=2)


# segment counts of 24 filters: 128 in all with one filter of 9 segments (the sidekit per-filter sum's loop beyond 8),
# and the same with one segment more
SEGS_128 = [9] + [5] * 19 + [6] * 4
SEGS_129 = [9] + [5] * 18 + [6] * 4 + [6]


# ------------------------------------------------------------------------------------------------ CPU tests
@pytest.fixture(scope="module")
def lib():
    from speech_signal_processing_b200 import _lib, build

    build.build()
    return _lib.load()


def test_reference_matches_the_oracle():
    """The recipe reference equals the oracle's restatements of sidekit, python_speech_features, utils/processing.py and
    GMM_UBM.extract_feature, so the comparisons below are comparisons with those front-ends."""
    for n in (16000, 4321, 400):
        sig = synth.synth_utterance(5, n % 97, n)
        got, le = reference(sfe.sidekit_recipe(), sig, preemph32=False)
        want = ofe.sidekit_mfcc(sig)
        np.testing.assert_allclose(got, want[0], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(le, want[1], rtol=1e-12)
        got, le = reference(sfe.psf_recipe(), sig, preemph32=False)
        assert le is None
        np.testing.assert_allclose(got, ofe.psf_mfcc(sig), rtol=1e-9, atol=1e-9)
    for fs, fsz, step in ((8000, 512, 256), (16000, 400, 160), (8000, 255, 100)):
        sig = synth.synth_utterance(4, 3, 2 * fs + 123, fs)
        got, _ = reference(sfe.processing_recipe(fs, fsz, step), sig)
        np.testing.assert_allclose(got, ofe.processing_mfcc(sig, fs, fsz, step), rtol=1e-9, atol=1e-9)
    sig = synth.synth_utterance(3, 1, 20000)
    for preset, recipe, kw in (("sidekit", sfe.sidekit_recipe(), {}), ("psf", sfe.psf_recipe(), {}),
                               ("processing", sfe.processing_recipe(16000, 512, 160),
                                dict(fs=16000, frame_size=512, step=160))):
        for order in (1, 2):
            got, _ = reference(recipe, sig, delta_order=order, cmvn=True, preemph32=False)
            np.testing.assert_allclose(got, ofe.features(sig, preset=preset, delta_order=order, cmvn=True, **kw),
                                       rtol=1e-9, atol=1e-9)
    # any N: the oracle's edge-padded delta, including T <= 2N + 1
    c = np.random.RandomState(0).standard_normal((3, 2))
    got, _ = reference(sfe.sidekit_recipe(), synth.synth_utterance(1, 1, 720), delta_order=1, delta_n=9)
    assert got.shape == (3, 26)
    den = 2 * sum(n * n for n in range(1, 10))
    want = [sum(n * (c[min(t + n, 2)] - c[max(t - n, 0)]) for n in range(1, 10)) / den for t in range(3)]
    np.testing.assert_allclose(ofe.delta(c, 9), np.array(want), rtol=1e-12)


def test_kernel_constants_and_bounds(lib):
    """The parsed constants are the ones the boundary cases were written for, and the restated shared-memory sizes give
    the library's ``ssp_frontend_max_frames`` on both sides of every support bound."""
    assert K == PINNED, "a front-end kernel constant changed: move the boundary cases of this file with it"
    recipes = [sfe.sidekit_recipe(), sfe.psf_recipe(), sfe.processing_recipe(), sfe.processing_recipe(16000, 512, 160),
               sfe.sidekit_recipe(fs=8000, maxfreq=4000), sfe.sidekit_recipe(fs=32000, maxfreq=16000),
               sfe.sidekit_recipe(fs=48000, maxfreq=24000), sfe.psf_recipe(numcep=20), sfe.psf_recipe(numcep=32, nfilt=40),
               sfe.processing_recipe(16000, 4096, 1024)] + [r for r, _ in support_cases()]
    kinds = set()
    for r in recipes:
        for order, cmvn in ((0, False), (1, True), (2, True)):
            c = cfg_of(r, order, 2, cmvn)
            if c.n_ceps * (1 + order) > 64:
                assert lib.ssp_frontend_max_frames(C.byref(c)) == 0
                continue
            assert lib.ssp_frontend_max_frames(C.byref(c)) == max_frames(c), (r.name, r.frame_len, r.frame_shift, order)
            kinds.add(fast_supported(c))
            if fast_supported(c) and order:
                t = mat_max_frames(c)
                assert 4 * carve_floats(c, t, True) <= K["MAT_BYTES"] < 4 * carve_floats(c, t + 1, True)
                assert t < max_frames(c)
    assert kinds == {True, False}
    for r, want in support_cases():
        assert kernel_of(r) == want, (r.name, want)
    # utils/processing.py's default (8 kHz, 512 / 256) has exactly MAXSEG segments, but its hop is past the staging bound
    assert n_segments(sfe.processing_recipe()) == K["MAXSEG"] and kernel_of(sfe.processing_recipe()) == "frontend_kernel"
    assert n_segments(sk_geometry_recipe(custom_fbank(SEGS_128))) == K["MAXSEG"]
    assert n_segments(sk_geometry_recipe(custom_fbank(SEGS_129))) == K["MAXSEG"] + 1
    assert n_segments(bark_sidekit_recipe()) > K["MAXSEG"]
    assert n_segments(sfe.sidekit_recipe()) < K["MAXSEG"]


def max_shift(frame_len):
    """Longest hop whose 8-frame batch still fits the fast kernel's staging buffer."""
    return (K["STAGE_SAMPLES"] - 1 - frame_len) // (K["W"] - 1)


def support_cases():
    """(recipe, kernel) on both sides of every bound of ``frontend_fast_supported``."""
    g, generic = "frontend512_kernel<generic>", "frontend_kernel"
    fb26 = sfe.psf_filterbank(16000, 512, 26)
    cases = []
    for fl in (512, 200):
        s = max_shift(fl)
        cases += [(psf_conventions_recipe(fb26, frame_len=fl, shift=s, name=f"fl{fl}-s{s}"), g),
                  (psf_conventions_recipe(fb26, frame_len=fl, shift=s + 1, name=f"fl{fl}-s{s + 1}"), generic)]
    for nf in (K["MAXF"], K["MAXF"] + 1):
        # (mel triangles from 100 Hz: python_speech_features' own bank gives 64 filters one that holds the DC bin alone,
        # whose power after pre-emphasis is at the level of the float32 FFT's rounding)
        cases.append((psf_conventions_recipe(sfe.sidekit_filterbank(16000, 512, 100, 8000, nf), name=f"nfilt{nf}"),
                      g if nf <= K["MAXF"] else generic))
    fb40 = sfe.psf_filterbank(16000, 512, 40)
    for ncep in (K["MAXC"], K["MAXC"] + 1):
        cases.append((psf_conventions_recipe(fb40, n_ceps=ncep, name=f"nceps{ncep}"), g if ncep <= K["MAXC"] else generic))
    for fl in (K["MIN_FL"], K["MIN_FL"] - 1):
        cases.append((psf_conventions_recipe(fb26, frame_len=fl, shift=1, name=f"fl{fl}"), g if fl >= K["MIN_FL"] else generic))
    return cases


def bark_sidekit_recipe():
    """Bark-band cepstra with sidekit conventions: 24 filters nonzero on all 257 bins (792 segments)."""
    return sk_geometry_recipe(sfe.bark_filterbank(16000, 512, nfilts=24), name="bark24")


# ------------------------------------------------------------------------------------------------ GPU helpers
WORST = {}


def note(key, err):
    WORST[key] = max(WORST.get(key, 0.0), float(err))
    print(f"  {key}: {err:.3e}")


def scaled_err(got, want):
    """max |got - want| / max(1, |want|) over the finite entries; the non-finite entries must be the same."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    for pred in (np.isnan, np.isposinf, np.isneginf):
        assert np.array_equal(pred(got), pred(want)), f"{pred.__name__} positions differ"
    fin = np.isfinite(want)
    if not fin.any():
        return 0.0
    return float((np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))).max())


def check(key, got, want, tol=CEPS_TOL):
    err = scaled_err(got, want)
    note(key, err)
    assert err <= tol, f"{key}: scaled error {err:.3e} > {tol}"


def check_loge(key, got, want):
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape
    for pred in (np.isnan, np.isposinf, np.isneginf):
        assert np.array_equal(pred(got), pred(want)), f"{key}: {pred.__name__} positions differ"
    fin = np.isfinite(want)
    err = float((np.abs(got[fin] - want[fin]) / np.abs(want[fin])).max()) if fin.any() else 0.0
    note(key + " log-energy", err)
    assert err <= LOGE_TOL, f"{key}: log-energy relative error {err:.3e}"


def check_cmvn(key, preset, got, want):
    atol = CMVN_ATOL.get(preset, CMVN_ATOL_OTHER)
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape
    err = float(np.abs(got - want).max()) if got.size else 0.0
    note(key + " cmvn", err)
    assert err <= atol, f"{key}: CMVN features off by {err:.3e} > {atol}"


def check_utts(key, preset, feats, offs, sigs, recipe, delta_order, delta_n, cmvn, log_e=None):
    for i, s in enumerate(sigs):
        want, wle = reference(recipe, s, delta_order, delta_n, cmvn)
        got = feats[offs[i] : offs[i + 1]]
        if cmvn:
            check_cmvn(key, preset, got, want)
        else:
            check(key, got, want)
        if log_e is not None:
            check_loge(key, log_e[offs[i] : offs[i + 1]], wle)


@pytest.fixture(scope="module")
def gpu():
    import torch

    from speech_signal_processing_b200 import _lib

    _lib.load()
    yield torch
    print("\nworst errors of this module:")
    for k in sorted(WORST):
        print(f"  {k}: {WORST[k]:.3e}")


def run(fe, sigs, want_log_energy=False):
    """FrontEnd.extract on a list of signals -> (feats, offsets, log_e, launch log)."""
    from speech_signal_processing_b200 import _lib

    _lib.load().ssp_reset_launch_count()
    feats, offs, le = fe.extract(sigs, want_log_energy)
    return feats.cpu().numpy(), offs, (le.cpu().numpy() if le is not None else None), _lib.launch_log()


def run_device(fe, pcm, offs, want_log_energy=False):
    from speech_signal_processing_b200 import _lib

    _lib.load().ssp_reset_launch_count()
    feats, foffs, le = fe.extract_device(pcm, offs, want_log_energy)
    return feats.cpu().numpy(), foffs, (le.cpu().numpy() if le is not None else None), _lib.launch_log()


def slices(base, lens, seed=0):
    """Utterances of the given lengths cut from one long signal at random offsets."""
    rs = np.random.RandomState(seed)
    return [base[o : o + n].copy() for n, o in zip(lens, rs.randint(0, len(base) - max(lens) - 1, size=len(lens)))]


PRESETS = {
    "sidekit": (sfe.sidekit_recipe, 16000),
    "psf": (sfe.psf_recipe, 16000),
    "processing": (lambda: sfe.processing_recipe(16000, 512, 160), 16000),
    "generic-kernel sidekit 8 kHz": (lambda: sfe.sidekit_recipe(fs=8000, maxfreq=4000), 8000),
}


def preset_of(name):
    return "sidekit" if name.startswith("sidekit") else name


# ------------------------------------------------------------------------------------------------ load paths
def load_path(sk, itemsize, base, s_begin):
    """The loads the fast kernel chooses for an utterance from the PCM base address and the utterance's first sample
    (frontend_fast.cu: ``direct`` and ``vec``)."""
    if itemsize == 4:
        return "staged-float" if sk else "float"
    if sk:
        return ("direct-odd" if s_begin & 1 else "direct-even") if base % 4 == 0 else "staged-int16"
    return "vec" if s_begin % 8 == 0 and base % 16 == 0 else "scalar-int16"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sidekit", "psf", "processing-16k"])
def test_every_load_path_matches_the_reference(gpu, name):
    """Views pcm[k:], k = 0..7, of one device buffer set the base alignment (2 to 16 bytes); the preceding utterance
    lengths set the parity of each utterance's first sample and its offset mod 8; float32 PCM takes the staged float path.
    Every path gives the reference's cepstra (and log-energy), and all of them agree with each other."""
    torch = gpu
    recipe = sfe.processing_recipe(16000, 512, 160) if name == "processing-16k" else PRESETS[name][0]()
    sk = kernel_of(recipe) == "frontend512_kernel"
    assert kernel_of(recipe) == ("frontend512_kernel" if name == "sidekit" else "frontend512_kernel<generic>")
    lens = [4003, 4000, 4005, 4002, 4008, 4001, 4007, 4004, 4006, 4011]
    sigs = slices(synth.synth_utterance(11, 2, 60000), lens)
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    cat = np.concatenate(sigs)
    fe = sfe.FrontEnd(recipe)
    want_le = recipe.energy_mode == 1
    refs = [reference(recipe, s) for s in sigs]
    buf = torch.zeros(len(cat) + 8, dtype=torch.int16, device="cuda")
    covered, results = set(), []
    for k in range(8):
        buf[k : k + len(cat)].copy_(torch.from_numpy(cat))
        pcm = buf[k : k + len(cat)]
        paths = {load_path(sk, 2, pcm.data_ptr(), int(o)) for o in offs[:-1]}
        covered |= paths
        feats, foffs, le, log = run_device(fe, pcm, offs, want_le)
        assert log == {kernel_of(recipe): 1}, log
        for i, (want, wle) in enumerate(refs):
            check(f"{name} {sorted(paths)}", feats[foffs[i] : foffs[i + 1]], want)
            if want_le:
                check_loge(f"{name} {sorted(paths)}", le[foffs[i] : foffs[i + 1]], wle)
        results.append(feats)
    fpcm = torch.from_numpy(cat.astype(np.float32)).cuda()
    covered.add(load_path(sk, 4, fpcm.data_ptr(), 0))
    feats, foffs, le, log = run_device(fe, fpcm, offs, want_le)
    assert log == {kernel_of(recipe, 1): 1}, log
    for i, (want, wle) in enumerate(refs):
        check(f"{name} float32", feats[foffs[i] : foffs[i + 1]], want)
        if want_le:
            check_loge(f"{name} float32", le[foffs[i] : foffs[i + 1]], wle)
    results.append(feats)
    assert covered == ({"direct-even", "direct-odd", "staged-int16", "staged-float"} if sk else {"vec", "scalar-int16", "float"})
    for other in results[1:]:
        err = scaled_err(other, results[0].astype(np.float64))
        note(f"{name} path against path", err)
        assert err <= CEPS_TOL


# ------------------------------------------------------------------------------------------------ bounds
@pytest.mark.gpu
@pytest.mark.parametrize("case", range(10))
def test_fast_path_support_bounds(gpu, case):
    """Both sides of the hop (staging buffer), filter-count, cepstrum-count and frame-length bounds: the kernel the
    launch log names, and the reference's cepstra either way."""
    recipe, want_kernel = support_cases()[case]
    fe = sfe.FrontEnd(recipe)
    n = [recipe.frame_len + 7 * recipe.frame_shift + 5, 3000, recipe.frame_len]
    sigs = slices(synth.synth_utterance(6, case, 40000), n, seed=case)
    feats, offs, _, log = run(fe, sigs)
    assert log == {want_kernel: 1}, log
    check_utts(f"support {recipe.name} -> {want_kernel}", "psf", feats, offs, sigs, recipe, 0, 2, False)


SEG_CASES = {
    "sk 128": (lambda: sk_geometry_recipe(custom_fbank(SEGS_128)), "frontend512_kernel"),
    "sk 129": (lambda: sk_geometry_recipe(custom_fbank(SEGS_129)), "frontend512_kernel"),
    "sk bark 792": (bark_sidekit_recipe, "frontend512_kernel"),
    "generic 128": (lambda: psf_conventions_recipe(custom_fbank(SEGS_128)), "frontend512_kernel<generic>"),
    "generic 129": (lambda: psf_conventions_recipe(custom_fbank(SEGS_129)), "frontend512_kernel<generic>"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SEG_CASES))
def test_segment_table_bound(gpu, case):
    """MAXSEG segments use the table, one more takes the per-filter fallback, in both instantiations; the sidekit
    fallback at T = 1 (every warp's segment scratch unused but the first) and at T >= 47, alone and in one batch."""
    make, want_kernel = SEG_CASES[case]
    recipe = make()
    fs = 16000
    fe = sfe.FrontEnd(recipe, delta_order=2, cmvn=True)
    fe0 = sfe.FrontEnd(recipe)
    base = synth.synth_utterance(8, 1, 20 * fs, fs)
    for lens in ([samples_for(recipe, 1)], [samples_for(recipe, 60)], [samples_for(recipe, t) for t in (1, 47, 2, 100, 9)]):
        sigs = slices(base, lens, seed=len(lens))
        feats, offs, le, log = run(fe0, sigs, recipe.energy_mode == 1)
        assert log == {want_kernel: 1}, log
        check_utts(f"segments {case}", "x", feats, offs, sigs, recipe, 0, 2, False, le)
        feats, offs, _, log = run(fe, sigs)
        assert log == {want_kernel: 1}, log
        check_utts(f"segments {case}", preset_of(recipe.name), feats, offs, sigs, recipe, 2, 2, True)


MAT_CASES = {
    "13 cepstra, delta-delta": (sfe.sidekit_recipe, 2),
    "20 cepstra, delta-delta (OD 60)": (lambda: sfe.psf_recipe(numcep=20), 2),
    "32 cepstra, delta (OD 64)": (lambda: sfe.psf_recipe(numcep=32, nfilt=40), 1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(MAT_CASES))
def test_delta_materialisation_bound(gpu, case):
    """The longest launch that still materialises delta / delta-delta in shared memory, and one frame more (recomputed
    from the cepstra), with and without CMVN."""
    make, order = MAT_CASES[case]
    recipe = make()
    c = cfg_of(recipe, order, 2, True)
    t_mat = mat_max_frames(c)
    base = synth.synth_utterance(9, 3, samples_for(recipe, t_mat + 1) + 20000)
    for t in (t_mat, t_mat + 1):
        sigs = slices(base, [samples_for(recipe, t), samples_for(recipe, 3)], seed=t)
        for cmvn in (False, True):
            fe = sfe.FrontEnd(recipe, delta_order=order, cmvn=cmvn)
            feats, offs, _, log = run(fe, sigs)
            assert log == {kernel_of(recipe): 1}, log
            side = "materialised" if t == t_mat else "recomputed"
            # (the 3-frame utterance's CMVN divides by the spread of 3 frames: compared without CMVN only)
            check_utts(f"{case} {side}", preset_of(recipe.name), feats, offs[:2] if cmvn else offs, sigs[:1] if cmvn else sigs,
                       recipe, order, 2, cmvn)


MAXF_CASES = {
    "sidekit (fast, sidekit instantiation)": lambda: sfe.sidekit_recipe(),
    "sidekit 8 kHz (generic kernel)": lambda: sfe.sidekit_recipe(fs=8000, maxfreq=4000),
    "processing 16 kHz (framing 2)": lambda: sfe.processing_recipe(16000, 512, 160),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(MAXF_CASES))
def test_fused_frame_bound_and_chunks(gpu, case):
    """``ssp_frontend_max_frames`` frames run fused, one more frame takes the chunked path (chunks of at most 2048
    frames, then ssp_delta / ssp_cmvn over the utterance); delta orders 0, 1, 2 with and without CMVN."""
    recipe = MAXF_CASES[case]()
    fs = 8000 if "8 kHz" in case else 16000
    kern = kernel_of(recipe)
    t_max = max_frames(cfg_of(recipe))
    base = synth.synth_utterance(12, 4, samples_for(recipe, t_max + 1) + 1000, fs)
    for t in (t_max, t_max + 1):
        sig = base[: samples_for(recipe, t)]
        ceps, le = reference(recipe, sig)
        for order in (0, 1, 2):
            parts, d = [ceps], ceps
            for _ in range(order):
                d = ofe.delta(d, 2)
                parts.append(d)
            raw = np.hstack(parts)
            for cmvn in (False, True):
                fe = sfe.FrontEnd(recipe, delta_order=order, cmvn=cmvn)
                feats, offs, got_le, log = run(fe, [sig], recipe.energy_mode == 1)
                if t == t_max:
                    assert log == {kern: 1}, log
                else:
                    want_log = {kern: -(-t // min(t_max, 2048))}
                    if order:
                        want_log["delta_kernel"] = order
                    if cmvn:
                        want_log["cmvn_kernel"] = 1
                    assert log == want_log, log
                key = f"{case} T={'max' if t == t_max else 'max+1'}"
                if cmvn:
                    mu, sd = raw.mean(0), raw.std(0)
                    check_cmvn(key, preset_of(recipe.name), feats, (raw - mu) / np.where(sd < 10 * np.finfo(float).eps, 1, sd))
                else:
                    check(key, feats, raw)
                if le is not None:
                    check_loge(key, got_le, le)


@pytest.mark.gpu
def test_chunk_cap(gpu):
    """2 * 2048 + 1 frames: chunks of 2048, 2048 and 1 frames, with log-energy, deltas and CMVN."""
    recipe = sfe.sidekit_recipe()
    t = 2 * 2048 + 1
    assert t > max_frames(cfg_of(recipe))
    sig = synth.synth_utterance(13, 2, samples_for(recipe, t))
    short = synth.synth_utterance(13, 3, 16000)
    fe = sfe.FrontEnd(recipe, delta_order=2, cmvn=True)
    feats, offs, le, log = run(fe, [short, sig], True)
    assert log == {"frontend512_kernel": 1 + 3, "delta_kernel": 2, "cmvn_kernel": 1}, log
    check_utts("chunk cap", "sidekit", feats, offs, [short, sig], recipe, 2, 2, True, le)


@pytest.mark.gpu
def test_feature_width_64_fused_and_wider_served_exactly(gpu):
    """OD = 64 (32 cepstra + delta) runs fused; the C entry point rejects OD = 65 and 66, and FrontEnd serves them
    through the chunked path with the reference's numbers -- an error or the right output, never a wrong one."""
    from speech_signal_processing_b200 import _lib

    torch = gpu
    sigs = slices(synth.synth_utterance(14, 1, 80000), [16000, 9000, 400], seed=3)
    r64 = sfe.psf_recipe(numcep=32, nfilt=40)
    feats, offs, _, log = run(sfe.FrontEnd(r64, delta_order=1, cmvn=True), sigs)
    assert log == {"frontend512_kernel<generic>": 1}, log
    check_utts("OD 64", "psf", feats, offs, sigs[:2], r64, 1, 2, True)
    for recipe, order in ((sfe.psf_recipe(numcep=22, nfilt=26), 2), (psf_conventions_recipe(sfe.psf_filterbank(16000, 512, 70), 65), 0)):
        assert recipe.dct.shape[0] * (1 + order) in (65, 66)
        fe = sfe.FrontEnd(recipe, delta_order=order, cmvn=True)
        cfg = fe._cfg(0)
        assert fe.lib.ssp_frontend_max_frames(C.byref(cfg)) == 0
        pcm = torch.from_numpy(np.concatenate(sigs)).cuda()
        soff = torch.tensor([0, 16000], dtype=torch.int64, device="cuda")
        foff = torch.tensor([0, fe.num_frames(16000)], dtype=torch.int64, device="cuda")
        out = torch.empty((1000, 70), dtype=torch.float32, device="cuda")
        rc = fe.lib.ssp_frontend_batch(_lib.ptr(pcm), _lib.ptr(soff), 1, C.byref(cfg), _lib.ptr(fe.t_window),
                                       _lib.ptr(fe.t_fb_start), _lib.ptr(fe.t_fb_len), _lib.ptr(fe.t_fb_off), _lib.ptr(fe.t_fb_w),
                                       _lib.ptr(fe.t_dct), _lib.ptr(foff), fe.num_frames(16000), _lib.ptr(out), None,
                                       _lib.stream_ptr())
        with pytest.raises(ValueError):
            _lib.check(rc, "ssp_frontend_batch")
        feats, offs, _, log = run(fe, sigs)
        assert "cmvn_kernel" in log, log
        check_utts(f"OD {recipe.dct.shape[0] * (1 + order)} chunked", "psf", feats, offs, sigs[:2], recipe, order, 2, True)


# ------------------------------------------------------------------------------------------------ edges
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PRESETS))
def test_short_utterances_and_delta_edges(gpu, name):
    """T = 1, 2, N, N + 1 and 2N + 1 for N = 1, 2, 3, 9, where edge padding decides every delta, with empty and
    shorter-than-a-frame utterances in the batch; on the fast kernel once with materialised deltas and once with a
    long neighbour that makes the launch recompute them."""
    make, fs = PRESETS[name]
    recipe = make()
    kern = kernel_of(recipe)
    base = synth.synth_utterance(15, 5, 40 * fs, fs)
    for N in (1, 2, 3, 9):
        ts = sorted({1, 2, N, N + 1, 2 * N + 1})
        lens = [0, 1, recipe.frame_len - 1] + [samples_for(recipe, t) for t in ts]
        sigs = slices(base, lens, seed=N)
        batches = [("materialised" if kern.startswith("frontend512") else "fused", sigs)]
        if kern.startswith("frontend512"):
            t_long = mat_max_frames(cfg_of(recipe, 2, N, False)) + 1
            batches.append(("recomputed", sigs + [base[: samples_for(recipe, t_long)]]))
        for side, batch in batches:
            fe = sfe.FrontEnd(recipe, delta_order=2, delta_n=N, cmvn=False)
            feats, offs, le, log = run(fe, batch, recipe.energy_mode == 1)
            assert log == {kern: 1}, log
            assert [offs[i + 1] - offs[i] for i in range(len(lens))] == [frame_count(recipe, n) for n in lens]
            check_utts(f"{name} edges {side}", preset_of(name), feats, offs, batch, recipe, 2, N, False, le)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PRESETS))
def test_digital_silence_and_full_scale(gpu, name):
    """Leading, trailing and full digital silence, and full-scale int16 square waves (+32767 / -32768).  Finite outputs
    match; under the sidekit convention (no log floor) the NaN and -inf of silent frames sit where the reference's do."""
    make, fs = PRESETS[name]
    recipe = make()
    n = samples_for(recipe, 40)
    speech = synth.synth_utterance(16, 1, n, fs)
    gap = 5 * recipe.frame_shift + 37
    lead, trail = speech.copy(), speech.copy()
    lead[:gap] = 0
    trail[-gap:] = 0
    i = np.arange(n)
    squares = [np.where((i // p) % 2 == 0, 32767, -32768).astype(np.int16) for p in (37, 11)]
    sigs = [lead, trail, np.zeros(n, np.int16)] + squares
    fe = sfe.FrontEnd(recipe)
    feats, offs, le, log = run(fe, sigs, recipe.energy_mode == 1)
    assert log == {kernel_of(recipe): 1}, log
    for j, s in enumerate(sigs):
        want, wle = reference(recipe, s)
        if j < 3 and name.startswith("sidekit"):
            assert not np.isfinite(want).all()
        tag = ["leading silence", "trailing silence", "silence", "square 37", "square 11"][j]
        check(f"{name} {tag}", feats[offs[j] : offs[j + 1]], want)
        if wle is not None:
            check_loge(f"{name} {tag}", le[offs[j] : offs[j + 1]], wle)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sidekit", "psf"])
def test_more_utterances_than_the_persistent_grid(gpu, name):
    """At least 3 x 16 x SMs short ragged utterances: every persistent CTA walks several, reusing its tables and shared
    memory."""
    torch = gpu
    make, fs = PRESETS[name]
    recipe = make()
    n_utts = 3 * 16 * torch.cuda.get_device_properties(0).multi_processor_count + 7
    rs = np.random.RandomState(1)
    lens = rs.randint(0, samples_for(recipe, 6), size=n_utts)
    sigs = slices(synth.synth_utterance(17, 2, 200000, fs), lens.tolist(), seed=2)
    fe = sfe.FrontEnd(recipe, delta_order=2, cmvn=False)
    feats, offs, le, log = run(fe, sigs, recipe.energy_mode == 1)
    assert log == {kernel_of(recipe): 1}, log
    check_utts(f"{name} {n_utts} utterances", name, feats, offs, sigs, recipe, 2, 2, False, le)


GENERIC_KERNEL_RECIPES = {
    "sidekit 8 kHz (nfft 256, 8 warps)": (lambda: sfe.sidekit_recipe(fs=8000, maxfreq=4000), 8000),
    "sidekit 32 kHz (nfft 1024, 4 warps)": (lambda: sfe.sidekit_recipe(fs=32000, maxfreq=16000), 32000),
    "sidekit 48 kHz (nfft 2048, 2 warps)": (lambda: sfe.sidekit_recipe(fs=48000, maxfreq=24000), 48000),
    "psf 32 kHz (nfft 1024)": (lambda: sfe.psf_recipe(samplerate=32000, nfft=1024), 32000),
    "psf 48 kHz (nfft 2048)": (lambda: sfe.psf_recipe(samplerate=48000, nfft=2048), 48000),
    "processing 4096": (lambda: sfe.processing_recipe(16000, 4096, 1024), 16000),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(GENERIC_KERNEL_RECIPES))
def test_generic_kernel_conventions_and_fused_epilogue(gpu, case):
    """``frontend_kernel`` at 8, 4 and 2 warps per CTA under the sidekit, psf and processing conventions, with its fused
    delta / delta-delta / CMVN epilogue."""
    make, fs = GENERIC_KERNEL_RECIPES[case]
    recipe = make()
    assert kernel_of(recipe) == "frontend_kernel"
    preset = preset_of(recipe.name)
    base = synth.synth_utterance(18, 3, 6 * fs, fs)
    sigs = slices(base, [fs, fs // 2 + 77, recipe.frame_len, 2 * fs + 5], seed=4)
    for order, cmvn in ((0, False), (2, False), (2, True)):
        fe = sfe.FrontEnd(recipe, delta_order=order, cmvn=cmvn)
        feats, offs, le, log = run(fe, sigs, recipe.energy_mode == 1)
        assert log == {"frontend_kernel": 1}, log
        check_utts(f"{case} order {order}", preset, feats, offs, sigs, recipe, order, 2, cmvn, le)
