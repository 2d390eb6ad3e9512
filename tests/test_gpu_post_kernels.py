"""The small kernels behind the front ends and the GMM loop, each on its own inputs through the C ABI, against float64.

* ``plp_post_kernel`` (``ssp_plp_post``): RASTA, equal loudness, autocorrelation, Levinson-Durbin and the cepstra of PLP.
* ``mel_db_dct_kernel`` (``ssp_mel_db_post``): the utterance-wide ``top_db`` clip and the DCT of the librosa MFCC.
* ``delta_kernel`` and ``cmvn_kernel`` (``ssp_delta``, ``ssp_cmvn``): the stand-alone delta and CMVN of chunked utterances.
* ``gmm_mstep_kernel`` and ``gmm_map_kernel`` (``ssp_gmm_mstep``, ``ssp_gmm_map_adapt``): the EM M-step and MAP.
* ``vad_features_kernel`` and ``vad_detect_kernel`` (``ssp_vad_features``, ``ssp_vad_detect``): the VAD front filter.

Every GPU test feeds a kernel its own device buffers, compares with a float64 restatement on the same inputs and checks
the launch log.  The tolerances follow from each kernel's arithmetic:

* PLP: double inside, float32 out.  The RASTA output is stored in the float32 band buffer between the two phases; it
  is checked to one float32 ulp of float64 RASTA, and the cepstra against the float64 back half of that stored buffer:
  |d| <= 2^-24 |c| + PLP_ATOL max(1, |c|).
* mel-dB: float32 with two interleaved partial sums: |d| <= sum_m |dct_jm| |v_m| (n_mels / 2 + 2) 2^-24.
* delta: |d| <= sum_n n (|hi| + |lo|) (N + 3) 2^-24 / den.
* CMVN: float32 sums over ceil(T / G) + G sequential terms (G = 256 / F frame groups).  This bound is statistical, not
  a worst case: the rounding of a sum of n terms as a random walk, 4 sqrt(n) 2^-24 (four standard deviations), on the
  mean (relative to mean |x|) and on the variance.  The seeds are fixed, so the measured margin below holds.
* M-step and MAP: double; means and variances a few ulps of their terms; weights the depth of the kernel's and numpy's
  summation trees in ulps.
* VAD: zero-crossing counts and decisions exact, energy 1e-12 relative, spectral entropy 2e-4 absolute (float32 FFT).

``test_kernel_bounds_and_parametrisations`` parses the bounds out of the CUDA sources and checks that the cases below
sit on both sides of each.  Every GPU test prints its largest error (profiles/r3d_pytest_gpu_post_kernels.log).
Largest errors measured on a B200 (1 000 W): PLP back half none beyond the float32 rounding of the output; ``ssp.plp``
against the oracle 4.1e-7 (at 8 to 48 kHz and up to 6 000 frames); mel-dB 0.28 of its bound; delta 0.51 of its bound;
CMVN 1.6e-4 absolute at 200 000 frames (on the mean-60, spread-0.3 column: 0.097 of the statistical bound) and at most
1.5e-4 on the shorter utterances; M-step and MAP at most 0.32 of their bounds, M-step means bit-exact; VAD energy
2.8e-15 relative and spectral entropy 2.7e-6 absolute (against the stated 2e-4), zero-crossing counts and decisions
exact.
"""
import ctypes as C
import functools
import math
import os
import re

import numpy as np
import pytest

from oracle import frontend as ofe
from oracle import gmm as ogmm
from oracle import vad as ov
from speech_signal_processing_b200 import frontend as sfe
from speech_signal_processing_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "speech_signal_processing_b200", "csrc")
U32, U64 = 2.0 ** -24, 2.0 ** -53
PLP_ATOL = 1e-9
ENT_ATOL = 2e-4


# ------------------------------------------------------------------------------------------------ kernel bounds
def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _int(pattern, text):
    m = re.search(pattern, text)
    assert m, pattern
    return int(m.group(1))


@functools.lru_cache(maxsize=None)
def kernel_bounds():
    """The support bounds and block sizes of the eight kernels, parsed out of the CUDA sources (on first use, so that a
    pattern that stops matching fails the tests that need it, not the collection of this file)."""
    plp, mel, vad, fe, gmm = (_source(n) for n in ("plp.cu", "mel_db.cu", "vad.cu", "frontend.cu", "gmm_pack.cu"))
    return {
        "PLP_MAXB": _int(r"constexpr int MAXB = (\d+);", plp),
        "PLP_MAXC": _int(r"constexpr int MAXC = (\d+);", plp),
        "PLP_MINB": _int(r"n_bands >= (\d+) &&", plp),
        "PLP_MINC": _int(r"n_ceps >= (\d+) &&", plp),
        "MEL_PRODUCT": _int(r"\(int64_t\)n_mels \* n_ceps <= (\d+)", mel),
        "VAD_FL": _int(r"constexpr int FL = (\d+);", vad),
        "VAD_MAX_BLOCKS": _int(r"cfg->n_blocks >= 1 && cfg->n_blocks <= (\d+)", vad),
        "VAD_SHIFT_MAX_IS_FL": int("cfg->frame_shift >= 1 && cfg->frame_shift <= FL" in vad),
        "CMVN_BLOCK": _int(r"for \(int j0 = 0; j0 < F; j0 \+= (\d+)\)", fe),
        "CMVN_THREADS": _int(r"cmvn_kernel<<<\(unsigned\)n_utts, (\d+),", fe),
        "MSTEP_THREADS": _int(r"gmm_mstep_kernel<<<\(unsigned\)n_models, (\d+),", gmm),
        "MAP_THREADS": _int(r"gmm_map_kernel<<<\(unsigned\)n_spk, (\d+),", gmm),
        "PLP_THREADS": _int(r"plp_post_kernel<<<\(unsigned\)n_utts, (\d+),", plp),
        "MEL_THREADS": _int(r"mel_db_dct_kernel<<<\(unsigned\)n_utts, (\d+),", mel),
    }


# the values the cases of this file were written for: a change to one of them fails here until the cases follow
PINNED = {"PLP_MAXB": 32, "PLP_MAXC": 16, "PLP_MINB": 3, "PLP_MINC": 2, "MEL_PRODUCT": 8192, "VAD_FL": 256,
          "VAD_MAX_BLOCKS": 32, "VAD_SHIFT_MAX_IS_FL": 1, "CMVN_BLOCK": 256, "CMVN_THREADS": 256, "MSTEP_THREADS": 1024,
          "MAP_THREADS": 256, "PLP_THREADS": 128, "MEL_THREADS": 256}

# cases (accepted, then rejected, where the entry point has a bound)
PLP_BANDS = (3, 16, 17, 21, 28, 32)
PLP_CEPS = (2, 3, 13, 16)
PLP_T = (1, 0, 4, 5, 6, 127, 128, 129, 300)       # RASTA's FIR-only start-up frames, the 128-thread frame loop
PLP_REJECT = ((2, 2), (33, 13), (21, 1), (21, 17), (13, 14))   # (n_bands, n_ceps)
MEL_SHAPES = ((128, 13), (41, 41), (127, 20), (1, 1), (128, 64), (8192, 1), (13, 12))   # (n_mels, n_ceps)
MEL_REJECT = ((2731, 3), (8193, 1), (12, 13), (0, 1))
DELTA_N = (1, 2, 3, 9)
DELTA_F = (1, 13, 39, 257)
CMVN_F = (1, 39, 255, 256, 257, 600)
VAD_SHIFTS = (1, 2, 127, 128, 129, 255, 256)
VAD_SHIFT_REJECT = (0, 257)
VAD_BLOCKS = (1, 3, 10, 32)
VAD_BLOCK_REJECT = (0, 33)
VAD_LENS = (0, 1, 255, 256, 257)
GMM_K = (1, 255, 256, 257, 1023, 1024, 1025, 4096)


def _both_sides(values, bound):
    return any(v <= bound for v in values) and any(v > bound for v in values)


# ------------------------------------------------------------------------------------------------ references
def plp_tables(nb, nc, fmax):
    """``plp_recipe``'s tables for any band and cepstrum count: equal-loudness weights, the real IDFT of the even
    extension as an (nc, nb) matrix, and the lifter."""
    cf = 600.0 * np.sinh(np.linspace(0.0, float(ofe.hz2bark(fmax)), nb) / 6.0)
    fsq = cf ** 2
    eql = (fsq / (fsq + 1.6e5)) ** 2 * ((fsq + 1.44e6) / (fsq + 9.61e6))
    n = 2 * (nb - 1)
    k, i = np.arange(nc)[:, None], np.arange(nb)[None, :]
    idft = 2.0 * np.cos(2.0 * np.pi * k * i / n) / n
    idft[:, 0] = 1.0 / n
    idft[:, nb - 1] = ((-1.0) ** np.arange(nc)) / n
    lift = np.concatenate([[1.0], np.arange(1, nc, dtype=np.float64) ** 0.6])
    return eql, idft, lift


def plp_post_ref(bands, eql, idft, lift, rasta, round32=True):
    """``ssp_plp_post`` of one utterance in float64 from the kernel's own tables: (cepstra (T, nc), band buffer after the
    call).  ``round32``: the RASTA output goes through the float32 band buffer, as in the kernel."""
    x = np.asarray(bands, dtype=np.float64)
    after = np.asarray(bands).copy()
    if x.shape[0] == 0:
        return np.zeros((0, idft.shape[0])), after
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        if rasta:
            x = np.exp(ofe.rasta_filt(np.log(x)))
            if round32:
                after = x.astype(np.float32)
                x = after.astype(np.float64)
        post = (eql[None, :] * x) ** 0.33
        post[:, 0] = post[:, 1]
        post[:, -1] = post[:, -2]
        r = post @ idft.T
        nc = idft.shape[0]
        a, e = ofe.levinson(r, nc - 1)
        cep = np.zeros((x.shape[0], nc))
        cep[:, 0] = np.log(e)
        for n in range(1, nc):
            s = np.zeros(x.shape[0])
            for m in range(1, n):
                s += (n - m) * a[:, m] * cep[:, n - m]
            cep[:, n] = -(a[:, n] + s / n)
    return cep * lift[None, :], after


def speech_bands(nb, T, seed, fs=16000):
    """Critical-band energies (T, nb) float32 of a synthetic utterance: sidekit framing, pre-emphasis, Hann window,
    power spectrum and an nb-band rastamat Bark filterbank."""
    if T == 0:
        return np.zeros((0, nb), np.float32)
    sig = synth.synth_utterance(seed % 7, seed, 400 + (T - 1) * 160, fs).astype(np.float64)
    fr = ofe.sidekit_frames(sig, 400, 160)
    fr = fr - 0.97 * np.concatenate([fr[:, :1], fr[:, :-1]], axis=1)
    spec = np.abs(np.fft.rfft(fr * np.hanning(400), 512, axis=1)) ** 2
    return (spec @ ofe.fft2barkmx(512, fs, nb).T).astype(np.float32)


def mel_db_ref(x, dct32, top_db):
    """``ssp_mel_db_post`` of one utterance: float64 DCT of the float32 clipped values (the clip floor in float32)."""
    mx = np.float32(x.max())
    floor = np.float32(mx - np.float32(top_db)) if top_db >= 0 else -np.inf
    v = np.maximum(x, floor).astype(np.float64)
    d = dct32.astype(np.float64)
    return v @ d.T, np.abs(v) @ np.abs(d).T


def vad_ref(sig, shift, n_blocks, normalize, eps=1e-8):
    """oracle.vad's framing, ZCR, energy and spectral entropy at any hop and sub-band count: three (T,) float64 arrays."""
    with np.errstate(divide="ignore", invalid="ignore"):
        w = ov.wav_normalise(sig) if normalize else np.asarray(sig, dtype=np.float64)
        fr = ov.enframe(w, 256, 256 - shift)
        return ov.zcr(fr)[:, 0], ov.energy(fr)[:, 0], ov.spectral_entropy(fr, n_blocks, eps)[:, 0]


def offsets(lens):
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


# ------------------------------------------------------------------------------------------------ CPU tests
@pytest.fixture(scope="module")
def lib():
    from speech_signal_processing_b200 import _lib, build

    build.build()
    return _lib.load()


def frontend_cfg(recipe):
    from speech_signal_processing_b200 import _lib

    r = recipe
    return _lib.FrontendCfg(r.frame_len, r.frame_shift, r.nfft, r.fbank.shape[0], r.dct.shape[0], r.framing, r.preemph_mode,
                            r.preemph, r.spec_type, r.spec_scale, r.log_type, r.log_add, r.log_zero_floor, r.energy_mode,
                            0, 2, 0, 0)


# fused-kernel frame bounds of the PLP band front end and the librosa recipe (ssp_frontend_max_frames)
PLP_RATES = {8000: (17, 256, 3026), 16000: (21, 512, 2065), 22050: (23, 1024, 1941), 44100: (27, 2048, 1561),
             48000: (28, 2048, 1502)}
LIBROSA_PRESETS = {"defaults": ({}, 320), "16 kHz, 40 bands": (dict(sr=16000, n_fft=400, hop_length=160, n_mels=40), 1197)}


def test_kernel_bounds_and_parametrisations(lib):
    """The parsed bounds are the ones the cases were written for, every case list spans both sides of its bound, and
    the fused frame bounds the long-utterance cases are built on are the library's."""
    B = kernel_bounds()
    assert B == PINNED, "a post-kernel bound changed: move the cases of this file with it"
    assert _both_sides(PLP_BANDS + tuple(b for b, _ in PLP_REJECT), B["PLP_MAXB"])
    assert _both_sides(PLP_BANDS + tuple(b for b, _ in PLP_REJECT), B["PLP_MINB"] - 1)
    assert B["PLP_MAXB"] in PLP_BANDS and B["PLP_MINB"] in PLP_BANDS
    assert _both_sides(PLP_CEPS + tuple(c for _, c in PLP_REJECT), B["PLP_MAXC"])
    assert B["PLP_MAXC"] in PLP_CEPS and B["PLP_MINC"] in PLP_CEPS and B["PLP_MINC"] - 1 in [c for _, c in PLP_REJECT]
    assert any(c > b for b, c in PLP_REJECT) and any(b == c for b in PLP_BANDS for c in PLP_CEPS)
    assert _both_sides(PLP_T, B["PLP_THREADS"]) and B["PLP_THREADS"] in PLP_T and {0, 1, 4, 5} <= set(PLP_T)
    prods = [m * c for m, c in MEL_SHAPES + MEL_REJECT]
    assert B["MEL_PRODUCT"] in [m * c for m, c in MEL_SHAPES] and B["MEL_PRODUCT"] + 1 in [m * c for m, c in MEL_REJECT]
    assert _both_sides(prods, B["MEL_PRODUCT"]) and any(m % 2 for m, _ in MEL_SHAPES) and any(m == c for m, c in MEL_SHAPES)
    assert B["VAD_SHIFT_MAX_IS_FL"] and _both_sides(VAD_SHIFTS + VAD_SHIFT_REJECT, B["VAD_FL"])
    assert B["VAD_FL"] in VAD_SHIFTS and 1 in VAD_SHIFTS and 0 in VAD_SHIFT_REJECT
    assert _both_sides(VAD_BLOCKS + VAD_BLOCK_REJECT, B["VAD_MAX_BLOCKS"]) and B["VAD_MAX_BLOCKS"] in VAD_BLOCKS
    assert _both_sides(VAD_LENS, B["VAD_FL"]) and B["VAD_FL"] in VAD_LENS
    assert B["CMVN_BLOCK"] == B["CMVN_THREADS"] and _both_sides(CMVN_F, B["CMVN_BLOCK"]) and B["CMVN_BLOCK"] in CMVN_F
    assert B["CMVN_BLOCK"] - 1 in CMVN_F and max(CMVN_F) > 2 * B["CMVN_BLOCK"]
    for t in ("MSTEP_THREADS", "MAP_THREADS"):
        assert _both_sides(GMM_K, B[t]) and B[t] in GMM_K and B[t] - 1 in GMM_K and B[t] + 1 in GMM_K
    assert max(GMM_K) > 2 * B["MSTEP_THREADS"]
    for fs, (nb, nfft, t_max) in PLP_RATES.items():
        r = sfe.plp_recipe(fs=fs)
        assert (r.fbank.shape[0], r.nfft) == (nb, nfft)
        assert lib.ssp_frontend_max_frames(C.byref(frontend_cfg(r))) == t_max, fs
    for kw, t_max in LIBROSA_PRESETS.values():
        assert lib.ssp_frontend_max_frames(C.byref(frontend_cfg(sfe.librosa_recipe(**kw)))) == t_max


def test_plp_reference_matches_the_oracle():
    """The table form above (IDFT matrix, the kernel's cepstrum recursion) equals the oracle's rastaplp back half (IFFT
    of the even extension, lpc / e) on positive bands, and its tables are ``plp_recipe``'s."""
    rs = np.random.RandomState(0)
    for nb in PLP_BANDS:
        for nc in PLP_CEPS:
            if nc > nb:
                continue
            bands = np.exp(rs.standard_normal((40, nb)) * 2.0 + 10.0)
            for rasta in (True, False):
                got, _ = plp_post_ref(bands, *plp_tables(nb, nc, 8000.0), rasta, round32=False)
                want = ofe.plp_post(bands, nc, 8000.0, rasta)
                np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-9)
    for fs in PLP_RATES:
        for order in (2, 13, 16):
            r = sfe.plp_recipe(fs=fs, plp_order=order)
            for name, table in zip(("eql", "idft", "lift"), plp_tables(r.fbank.shape[0], order, fs / 2.0)):
                np.testing.assert_allclose(table, r.extra[name], rtol=1e-15, atol=1e-15)
            np.testing.assert_allclose(r.extra["eql"], ofe.postaud_weights(r.fbank.shape[0], fs / 2.0), rtol=1e-15)
    # the float32 rounding between the phases is visible at the tolerance the GPU test uses
    nb, nc = 21, 13
    bands = speech_bands(nb, 60, 3)
    a, _ = plp_post_ref(bands, *plp_tables(nb, nc, 8000.0), True, round32=True)
    b, _ = plp_post_ref(bands, *plp_tables(nb, nc, 8000.0), True, round32=False)
    assert (np.abs(a - b) > U32 * np.abs(a) + PLP_ATOL * np.maximum(1.0, np.abs(a))).any()


def test_vad_reference_matches_the_oracle_defaults():
    """``vad_ref`` at the reference's hop and sub-band count is the oracle's feature set."""
    sig = synth.synth_utterance(2, 1, 5000)
    z, p, e = vad_ref(sig, 128, 10, True)
    fr = ov.enframe(ov.wav_normalise(sig))
    np.testing.assert_array_equal(z, ov.zcr(fr)[:, 0])
    np.testing.assert_array_equal(p, ov.energy(fr)[:, 0])
    np.testing.assert_array_equal(e, ov.spectral_entropy(fr)[:, 0])


# ------------------------------------------------------------------------------------------------ GPU helpers
WORST = {}


def note(key, err):
    WORST[key] = max(WORST.get(key, 0.0), float(err))
    print(f"  {key}: {err:.3e}")


@pytest.fixture(scope="module")
def gpu():
    import torch

    from speech_signal_processing_b200 import _lib

    _lib.load()
    yield torch
    print("\nworst errors of this module:")
    for k in sorted(WORST):
        print(f"  {k}: {WORST[k]:.3e}")


def dev(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a), device="cuda")


def run(name, *args):
    """Call a C entry point on the current stream, synchronise, and return the launch log of the call."""
    import torch

    from speech_signal_processing_b200 import _lib

    lib = _lib.load()
    lib.ssp_reset_launch_count()
    _lib.check(getattr(lib, name)(*args, _lib.stream_ptr()), name)
    torch.cuda.synchronize()
    _ALIVE.clear()
    return _lib.launch_log()


def rejected(name, *args):
    from speech_signal_processing_b200 import _lib

    lib = _lib.load()
    lib.ssp_reset_launch_count()
    with pytest.raises(ValueError):
        _lib.check(getattr(lib, name)(*args, _lib.stream_ptr()), name)
    _ALIVE.clear()
    assert _lib.launch_log() == {}


def same_nonfinite(got, want, key):
    for pred in (np.isnan, np.isposinf, np.isneginf):
        assert np.array_equal(pred(got), pred(want)), f"{key}: {pred.__name__} positions differ"


_ALIVE = []


def P(t):
    """Device pointer of t; t stays alive until the next ``run`` has synchronised (``P(dev(a))`` would otherwise hand
    the allocator the block back before the call, and the next ``dev`` could reuse it)."""
    from speech_signal_processing_b200 import _lib

    _ALIVE.append(t)
    return _lib.ptr(t)


# ------------------------------------------------------------------------------------------------ PLP back half
@pytest.mark.gpu
@pytest.mark.parametrize("nb", PLP_BANDS)
def test_plp_post_matches_float64(gpu, nb):
    """Every cepstrum count up to min(16, n_bands), RASTA on and off, utterances of 1, 0, 4, 5, 6, 127, 128, 129 and 300
    frames and one of digital silence in one launch: the cepstra within the float32 rounding of the output, the band
    buffer rewritten with RASTA's float32 output (and left alone without RASTA), NaN and inf where the reference has
    them and only in the silent utterance."""
    torch = gpu
    lens = list(PLP_T) + [10]
    offs = offsets(lens)
    bands = np.concatenate([speech_bands(nb, t, 11 * nb + i) for i, t in enumerate(lens[:-1])] + [np.zeros((10, nb), np.float32)])
    d_off = dev(offs)
    for nc in [c for c in PLP_CEPS if c <= nb]:
        tables = plp_tables(nb, nc, 8000.0)
        d_tab = [dev(t.astype(np.float64)) for t in tables]
        for rasta in (True, False):
            d_bands = dev(bands)
            out = torch.full((int(offs[-1]), nc), float("nan"), dtype=torch.float32, device="cuda")
            log = run("ssp_plp_post", P(d_bands), P(d_off), len(lens), nb, nc, *(P(t) for t in d_tab), int(rasta), P(out))
            assert log == {"plp_post_kernel": 1}, log
            got, after = out.cpu().numpy().astype(np.float64), d_bands.cpu().numpy()
            key = f"plp_post nb={nb} nc={nc} rasta={int(rasta)}"
            worst = 0.0
            for u in range(len(lens)):
                sl = slice(offs[u], offs[u + 1])
                want, want_after = plp_post_ref(bands[sl], *tables, rasta)
                same_nonfinite(got[sl], want, key)
                if rasta:
                    # phase 2 on the kernel's own float32 RASTA output, checked to one ulp below: the float64 filters
                    # agree to ~1e-14, which can still put a value on the other side of a float32 rounding boundary
                    want, _ = plp_post_ref(after[sl], *tables, False)
                    same_nonfinite(got[sl], want, key)
                same_nonfinite(after[sl].astype(np.float64), want_after.astype(np.float64), key + " bands")
                if u < len(lens) - 1:
                    assert np.isfinite(want).all() and np.isfinite(want_after).all()
                    # the table form is the oracle's rastaplp back half on the same bands
                    x2 = after[sl] if rasta else bands[sl]
                    np.testing.assert_allclose(want, ofe.plp_post(x2.astype(np.float64), nc, 8000.0, False), rtol=1e-9, atol=1e-9)
                else:
                    assert not np.isfinite(want).all()
                fin = np.isfinite(want)
                g, w = got[sl][fin], want[fin]
                excess = (np.abs(g - w) - U32 * np.abs(w)) / np.maximum(1.0, np.abs(w))
                if excess.size:
                    worst = max(worst, float(excess.max()))
                fa = np.isfinite(want_after)
                a, wa = after[sl][fa].astype(np.float64), want_after[fa].astype(np.float64)
                if rasta:
                    assert (np.abs(a - wa) <= np.spacing(np.abs(want_after[fa]).astype(np.float32))).all(), key
                else:
                    assert np.array_equal(a, wa), key
            note(key + " (error beyond the float32 rounding, of max(1, |c|))", worst)
            assert worst <= PLP_ATOL, f"{key}: {worst:.3e}"


@pytest.mark.gpu
def test_plp_post_rejects_out_of_range_shapes(gpu):
    """2 and 33 bands, 1 and 17 cepstra, and more cepstra than bands."""
    torch = gpu
    d_off = dev(np.array([0, 3], np.int64))
    bands = torch.ones((3, 40), dtype=torch.float32, device="cuda")
    tab = torch.ones(40 * 40, dtype=torch.float64, device="cuda")
    out = torch.empty((3, 40), dtype=torch.float32, device="cuda")
    for nb, nc in PLP_REJECT:
        rejected("ssp_plp_post", P(bands), P(d_off), 1, nb, nc, P(tab), P(tab), P(tab), 1, P(out))


# ------------------------------------------------------------------------------------------------ PLP end to end
@pytest.mark.gpu
@pytest.mark.parametrize("fs", sorted(PLP_RATES))
def test_plp_at_every_sample_rate(gpu, fs):
    """``ssp.plp`` against the oracle's sidekit / rastamat PLP at 8, 16, 22.05, 44.1 and 48 kHz, model orders 2, 13 and
    16, RASTA on and off (the tolerance of tests/test_gpu_frontend.py::test_plp_matches_oracle)."""
    import speech_signal_processing_b200 as ssp

    sig = synth.synth_utterance(3, fs % 13, int(1.3 * fs), fs)
    for order in (2, 13, 16):
        for rasta in (True, False):
            got = ssp.plp(sig, fs=fs, plp_order=order, rasta=rasta)
            want = ofe.sidekit_plp(sig, fs=fs, plp_order=order, rasta=rasta)
            assert got[0].shape == want[0].shape and got[0].shape[1] == order
            err = float(np.abs(got[0] - want[0]).max())
            note(f"plp {fs} Hz order {order} rasta={int(rasta)}", err)
            assert err <= 2e-3
            np.testing.assert_allclose(got[1], want[1], rtol=2e-5)


@pytest.mark.gpu
def test_plp_long_utterances_take_the_chunked_path(gpu):
    """At 16 kHz: the fused bound of the band front end, one frame more, and 60 s; the launch log shows the chunks and
    RASTA runs over the whole utterance."""
    from speech_signal_processing_b200 import _lib

    t_max = PLP_RATES[16000][2]
    fe = sfe.PlpFrontEnd(sfe.plp_recipe())
    base = synth.synth_utterance(5, 2, 400 + 5999 * 160)
    for t in (t_max, t_max + 1, 6000):
        sig = base[: 400 + (t - 1) * 160]
        _lib.load().ssp_reset_launch_count()
        feats, offs, _ = fe.extract([sig])
        log = _lib.launch_log()
        chunks = 1 if t <= t_max else -(-t // min(t_max, 2048))
        assert log == {"frontend512_kernel<generic>": chunks, "plp_post_kernel": 1}, log
        got, want = feats.cpu().numpy(), ofe.sidekit_plp(sig)[0]
        assert got.shape == want.shape == (t, 13)
        err = float(np.abs(got - want).max())
        note(f"plp 16 kHz T={t}", err)
        assert err <= 2e-3


@pytest.mark.gpu
def test_extract_feature_plp_with_a_long_utterance(gpu):
    """``extract_feature(feature_type='PLP')`` on short utterances around one beyond the fused bound (the tolerance of
    tests/test_gpu_frontend.py::test_extract_feature_plp_batched)."""
    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    x = [synth.synth_utterance(1, 1, 16000), synth.synth_utterance(2, 2, 400 + 2500 * 160), synth.synth_utterance(3, 3, 8000)]
    _lib.load().ssp_reset_launch_count()
    feats, _ = ssp.extract_feature(x, ["a", "b", "c"], feature_type="PLP")
    log = _lib.launch_log()
    # band front end: one fused launch for each run of short utterances around the long one (2), and the 2501-frame
    # utterance in chunks of 2048 frames (2); one PLP back half for the batch; one delta launch per utterance; one CMVN
    assert log == {"frontend512_kernel<generic>": 2 + 2, "plp_post_kernel": 1, "delta_kernel": 3, "cmvn_kernel": 1}, log
    for sig, f in zip(x, feats):
        c = ofe.sidekit_plp(sig)[0]
        ref = ofe.scale(np.hstack([c, ofe.delta(c)]))
        assert f.shape == ref.shape
        err = float(np.abs(f - ref).max())
        note(f"extract_feature PLP T={len(c)}", err)
        assert err <= 2e-2


# ------------------------------------------------------------------------------------------------ mel-dB back half
def mel_inputs(nm, lens, seed):
    """Log-mel power in dB (float32): a smooth spectral envelope over -100 .. +30 dB per frame."""
    rs = np.random.RandomState(seed)
    env = np.cumsum(rs.standard_normal((sum(lens), nm)), axis=1) * 2.0
    return (env - env.mean(axis=1, keepdims=True) - 40.0 + 15.0 * rs.standard_normal((sum(lens), 1))).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", MEL_SHAPES)
def test_mel_db_post_matches_float64(gpu, shape):
    """top_db 80, 0 and negative (no clip); the utterance maximum at its first and at its last element; utterances of
    1, 0, 37 and 3000 frames (the block-wide maximum loops) in one launch."""
    torch = gpu
    nm, nc = shape
    lens = [1, 0, 37, 3000, 37, 5] if nm * nc <= 2048 else [1, 0, 37, 300, 37, 5]
    offs = offsets(lens)
    x = mel_inputs(nm, lens, nm + nc)
    x[offs[2], 0] = x[offs[2] : offs[3]].max() + 7.0            # maximum at the first element
    x[offs[5] - 1, -1] = x[offs[4] : offs[5]].max() + 7.0        # ... and at the last
    dct32 = sfe.dct_rows(nc, nm).astype(np.float32)
    d_x, d_off, d_dct = dev(x), dev(offs), dev(dct32)
    for top_db in (80.0, 0.0, -1.0):
        out = torch.full((int(offs[-1]), nc), float("nan"), dtype=torch.float32, device="cuda")
        log = run("ssp_mel_db_post", P(d_x), P(d_off), len(lens), nm, nc, P(d_dct), top_db, P(out))
        assert log == {"mel_db_dct_kernel": 1}, log
        got = out.cpu().numpy().astype(np.float64)
        worst = 0.0
        for u in range(len(lens)):
            sl = slice(offs[u], offs[u + 1])
            if lens[u] == 0:
                continue
            want, mag = mel_db_ref(x[sl], dct32, top_db)
            bound = mag * (nm / 2 + 2) * U32
            err = np.abs(got[sl] - want)
            assert (err <= bound).all(), f"mel-dB {shape} top_db {top_db} utterance {u}"
            worst = max(worst, float((err / np.maximum(bound, 1e-300)).max()))
        note(f"mel_db {nm}x{nc} top_db={top_db} (error / bound)", worst)


@pytest.mark.gpu
def test_mel_db_post_rejects_out_of_range_shapes(gpu):
    """n_mels * n_ceps of 8193, n_ceps > n_mels and n_mels 0."""
    torch = gpu
    d_off = dev(np.array([0, 1], np.int64))
    buf = torch.zeros(9000 * 3, dtype=torch.float32, device="cuda")
    for nm, nc in MEL_REJECT:
        rejected("ssp_mel_db_post", P(buf), P(d_off), 1, nm, nc, P(buf), 80.0, P(buf))


@pytest.mark.gpu
@pytest.mark.parametrize("preset", sorted(LIBROSA_PRESETS))
def test_librosa_mfcc_at_the_fused_bound(gpu, preset):
    """The librosa recipe at its fused frame bound matches the oracle; one frame more raises NotImplementedError
    (centred framing is not chunked)."""
    import speech_signal_processing_b200 as ssp

    kw, t_max = LIBROSA_PRESETS[preset]
    full = dict(sr=8000, n_mfcc=13)
    full.update(kw)
    hop = kw.get("hop_length", 512)
    sig = synth.synth_utterance(4, 1, t_max * hop, full["sr"]).astype(np.float32)
    got = ssp.librosa_mfcc(sig[: (t_max - 1) * hop], **full)
    want = ofe.librosa_mfcc(sig[: (t_max - 1) * hop], **full)
    assert got.shape == want.shape == (13, t_max)
    err = float((np.abs(got - want) / np.maximum(1.0, np.abs(want))).max())
    note(f"librosa {preset} T={t_max}", err)
    assert err <= 1e-4
    with pytest.raises(NotImplementedError):
        ssp.librosa_mfcc(sig, **full)


# ------------------------------------------------------------------------------------------------ delta and CMVN
@pytest.mark.gpu
@pytest.mark.parametrize("N", DELTA_N)
def test_delta_matches_float64(gpu, N):
    """T = 1, 2, N, N + 1, 2N + 1 and 500 at F = 1, 13, 39 and 257, where edge padding decides every output."""
    torch = gpu
    den = 2.0 * sum(n * n for n in range(1, N + 1))
    rs = np.random.RandomState(N)
    worst = 0.0
    for T in sorted({1, 2, N, N + 1, 2 * N + 1, 500}):
        for F in DELTA_F:
            x = (rs.standard_normal((T, F)) * rs.uniform(0.1, 30.0, size=F) + rs.uniform(-50, 50, size=F)).astype(np.float32)
            out = torch.full((T, F), float("nan"), dtype=torch.float32, device="cuda")
            log = run("ssp_delta", P(dev(x)), T, F, N, P(out))
            assert log == {"delta_kernel": 1}, log
            x64 = x.astype(np.float64)
            want = ofe.delta(x64, N)
            t = np.arange(T)
            mag = sum(n * (np.abs(x64[np.minimum(t + n, T - 1)]) + np.abs(x64[np.maximum(t - n, 0)])) for n in range(1, N + 1))
            bound = mag * (N + 3) * U32 / den
            err = np.abs(out.cpu().numpy() - want)
            assert (err <= bound).all(), (N, T, F)
            worst = max(worst, float((err / np.maximum(bound, 1e-300)).max()))
    note(f"delta N={N} (error / bound)", worst)


def cmvn_bound(x, want, T, F):
    """4 sqrt(n) 2^-24 on the mean (of mean |x|) and on the variance, n = the sequential terms of the kernel's sums."""
    fj = np.minimum(F - 256 * (np.arange(F) // 256), 256)
    g = np.maximum(256 // fj, 1)
    n = np.ceil(T / g) + g + 2
    r = 4.0 * np.sqrt(n) * U32
    x64 = x.astype(np.float64)
    sd = x64.std(axis=0)
    sd = np.where(sd < 10 * np.finfo(np.float32).eps, 1.0, sd)
    return r * (np.abs(x64).mean(axis=0) + np.abs(x64 - x64.mean(axis=0))) / sd + r * np.abs(want)


@pytest.mark.gpu
@pytest.mark.parametrize("F", CMVN_F)
def test_cmvn_matches_float64(gpu, F):
    """Utterances of 3, 0, 1 (std 0 -> 1), 700 and 40 frames in one launch, cepstrum-like columns (a large-mean
    first column), the column-block loop beyond 256 columns."""
    torch = gpu
    lens = [3, 0, 1, 700, 40]
    offs = offsets(lens)
    rs = np.random.RandomState(F)
    scale_ = rs.uniform(0.3, 8.0, size=F)
    mean = rs.uniform(-20, 20, size=F)
    mean[0], scale_[0] = 60.0, 0.3
    x = (rs.standard_normal((int(offs[-1]), F)) * scale_ + mean).astype(np.float32)
    out = torch.full(x.shape, float("nan"), dtype=torch.float32, device="cuda")
    log = run("ssp_cmvn", P(dev(x)), P(dev(offs)), len(lens), F, P(out))
    assert log == {"cmvn_kernel": 1}, log
    got = out.cpu().numpy().astype(np.float64)
    worst = 0.0
    for u, T in enumerate(lens):
        if T == 0:
            continue
        sl = slice(offs[u], offs[u + 1])
        x64 = x[sl].astype(np.float64)
        sd = x64.std(axis=0)
        want = (x64 - x64.mean(axis=0)) / np.where(sd < 10 * np.finfo(np.float32).eps, 1.0, sd)
        if T == 1:
            assert (got[sl] == 0).all()
            continue
        err = np.abs(got[sl] - want)
        bound = cmvn_bound(x[sl], want, T, F)
        assert (err <= bound).all(), (F, u)
        worst = max(worst, float(err.max()))
    note(f"cmvn F={F} (absolute)", worst)


@pytest.mark.gpu
def test_cmvn_of_a_long_utterance(gpu):
    """200 000 frames of 39 columns with a mean-60, spread-0.3 first column: the float32 sums' error against float64."""
    torch = gpu
    T, F = 200000, 39
    rs = np.random.RandomState(7)
    scale_ = np.linspace(0.3, 8.0, F)
    mean = rs.uniform(-5, 5, size=F)
    mean[0] = 60.0
    x = (rs.standard_normal((T, F)) * scale_ + mean).astype(np.float32)
    out = torch.empty(x.shape, dtype=torch.float32, device="cuda")
    log = run("ssp_cmvn", P(dev(x)), P(dev(np.array([0, T], np.int64))), 1, F, P(out))
    assert log == {"cmvn_kernel": 1}, log
    x64 = x.astype(np.float64)
    want = (x64 - x64.mean(axis=0)) / x64.std(axis=0)
    err = np.abs(out.cpu().numpy() - want)
    bound = cmvn_bound(x, want, T, F)
    note("cmvn T=200000 F=39 (absolute)", float(err.max()))
    note("cmvn T=200000 F=39 (error / bound)", float((err / bound).max()))
    assert (err <= bound).all()


# ------------------------------------------------------------------------------------------------ M-step and MAP
def host_stats(M, K, D, seed, empty=(), frames=None):
    """Float64 statistics (n (M, K), f (M, K, D), s (M, K, D)) of plausible data, with n = 0 at the given (m, k) and,
    given ``frames``, sum_k n = frames[m]."""
    rs = np.random.RandomState(seed)
    n = rs.gamma(0.7, 40.0, size=(M, K))
    for m, k in empty:
        n[m, k] = 0.0
    if frames is not None:
        tot = n.sum(axis=1)
        n *= np.divide(np.asarray(frames, dtype=np.float64), tot, out=np.zeros(M), where=tot > 0)[:, None]
    mu = rs.standard_normal((M, K, D)) * 3.0
    var = rs.uniform(0.2, 2.0, size=(M, K, D))
    f = n[..., None] * mu
    s = n[..., None] * (var + mu * mu)
    return n, f, s


def sum_depth(K, threads):
    """Sequential additions on the longest path of the kernel's block sum of K terms, plus numpy's pairwise sum."""
    return math.ceil(K / threads) + 5 + threads // 32 + math.ceil(math.log2(max(K, 2))) + 2


@pytest.mark.gpu
@pytest.mark.parametrize("K", GMM_K)
def test_mstep_matches_float64(gpu, K):
    """Three models per launch, components with n = 0, K x D above the 1024-thread block."""
    torch = gpu
    M, D = 3, (1, 13, 39)[K % 3]
    n, f, s = host_stats(M, K, D, K, empty=[(0, 0), (2, K - 1), (1, K // 2)])
    eps = np.finfo(np.float64).eps
    ow = torch.empty((M, K), dtype=torch.float64, device="cuda")
    omu, ovar = (torch.empty((M, K, D), dtype=torch.float64, device="cuda") for _ in range(2))
    log = run("ssp_gmm_mstep", P(dev(n)), P(dev(f)), P(dev(s)), M, K, D, 1e-6, 10 * eps, P(ow), P(omu), P(ovar))
    assert log == {"gmm_mstep_kernel": 1}, log
    gw, gmu, gvar = (t.cpu().numpy() for t in (ow, omu, ovar))
    errs = [0.0, 0.0, 0.0]
    for m in range(M):
        w, mu, var = ogmm.m_step(n[m], f[m], s[m], 1e-6, eps)
        nk = n[m] + 10 * eps
        bounds = (sum_depth(K, kernel_bounds()["MSTEP_THREADS"]) * U64 * w, 2 * U64 * np.abs(mu),
                  6 * U64 * (np.abs(s[m] / nk[:, None]) + mu * mu + 1e-6))
        for i, (g, want, bound) in enumerate(zip((gw[m], gmu[m], gvar[m]), (w, mu, var), bounds)):
            err = np.abs(g - want)
            assert (err <= bound).all(), (K, m, ("weights", "means", "variances")[i])
            errs[i] = max(errs[i], float((err / np.maximum(bound, 1e-300)).max()))
    for i, what in enumerate(("weights", "means", "variances")):
        note(f"mstep K={K} D={D} {what} (error / bound)", errs[i])


@pytest.mark.gpu
@pytest.mark.parametrize("K", GMM_K)
def test_map_adapt_kernel_matches_float64(gpu, K):
    """Four speakers per launch (one of no frames), components with n = 0, every flags combination, relevance 16 and
    0: the kernel equals the oracle's MAP on the same float64 statistics, and nothing without data leaves the UBM."""
    torch = gpu
    S, D = 4, (1, 13, 39)[K % 3]
    lens = [500, 0, 700, 300]                                # speaker 1 has no frames
    n, f, s = host_stats(S, K, D, 100 + K, empty=[(0, 0), (2, K - 1)] + [(1, k) for k in range(K)], frames=lens)
    seg = offsets(lens)
    w, mu, var = synth.synth_ubm(K, D, seed=K)
    d_n, d_f, d_s, d_seg, d_w, d_mu, d_var = (dev(a) for a in (n, f, s, seg, w, mu, var))
    errs = {}
    for relevance in (16.0, 0.0):
        for flags in range(8):
            adapt = tuple(a for bit, a in ((1, "means"), (2, "weights"), (4, "variances")) if flags & bit)
            ow = torch.full((S, K), float("nan"), dtype=torch.float64, device="cuda")
            omu, ovar = (torch.full((S, K, D), float("nan"), dtype=torch.float64, device="cuda") for _ in range(2))
            log = run("ssp_gmm_map_adapt", P(d_n), P(d_f), P(d_s), P(d_seg), S, P(d_w), P(d_mu), P(d_var), K, D, relevance,
                      flags, P(ow), P(omu), P(ovar))
            assert log == {"gmm_map_kernel": 1}, log
            gw, gmu, gvar = (t.cpu().numpy() for t in (ow, omu, ovar))
            assert np.isfinite(gw).all() and np.isfinite(gmu).all() and np.isfinite(gvar).all(), (relevance, flags)
            for sp in range(S):
                rw, rmu, rvar = ogmm.map_adapt(n[sp], f[sp], s[sp], w, mu, var, int(seg[sp + 1] - seg[sp]), relevance, adapt)
                safe = np.maximum(n[sp], np.finfo(np.float64).tiny)[:, None]
                ex, ex2 = np.abs(f[sp] / safe), np.abs(s[sp] / safe)
                bounds = (sum_depth(K, kernel_bounds()["MAP_THREADS"]) * U64 * np.abs(rw) + 4 * U64 * np.abs(w),
                          8 * U64 * (ex + np.abs(mu)),
                          8 * U64 * (ex2 + var + mu * mu + rmu * rmu) + 24 * U64 * np.abs(rmu) * (ex + np.abs(mu)))
                for i, (g, want, bound) in enumerate(zip((gw[sp], gmu[sp], gvar[sp]), (rw, rmu, rvar), bounds)):
                    err = np.abs(g - want)
                    assert (err <= bound).all(), (K, relevance, flags, sp, i)
                    key = ("weights", "means", "variances")[i]
                    errs[key] = max(errs.get(key, 0.0), float((err / np.maximum(bound, 1e-300)).max()))
            # no data, no change: the empty speaker and the empty components keep the UBM's means and variances
            for sp, k in ((1, slice(None)), (0, 0), (2, K - 1)):
                np.testing.assert_array_equal(gmu[sp][k], mu[k])
                if not flags & 4:
                    np.testing.assert_array_equal(gvar[sp][k], var[k])
            if flags & 2:
                np.testing.assert_allclose(gw[1], w / w.sum(), rtol=8 * sum_depth(K, kernel_bounds()["MAP_THREADS"]) * U64)
    for key, e in errs.items():
        note(f"map K={K} D={D} {key} (error / bound)", e)


@pytest.mark.gpu
def test_map_adapt_without_data_keeps_the_ubm(gpu):
    """``ssp.map_adapt`` with a speaker of no frames and a component no frame reaches, at relevance 16 and 0: every
    output is finite, and what has no data keeps the UBM's parameters (weights renormalised)."""
    import speech_signal_processing_b200 as ssp

    K, D = 16, 13
    w, mu, var = synth.synth_ubm(K, D, seed=9)
    mu[5] += 60.0          # no frame below reaches this component: its responsibilities underflow to 0
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    a = synth.sample_gmm(w, mu - np.eye(K)[5][:, None] * 60.0, var, 400, seed=1)
    b = synth.sample_gmm(w, mu - np.eye(K)[5][:, None] * 60.0, var, 300, seed=2)
    frames = [a, np.zeros((0, D), np.float32), b]
    every = ("means", "weights", "variances")
    for relevance in (16.0, 0.0):
        ow, omu, ovar = (t.cpu().numpy() for t in ssp.map_adapt(ubm, frames, relevance=relevance, adapt=every))
        assert np.isfinite(ow).all() and np.isfinite(omu).all() and np.isfinite(ovar).all(), relevance
        np.testing.assert_allclose(ow[1], w / w.sum(), rtol=1e-14)
        np.testing.assert_array_equal(omu[1], mu)
        var_tol = 4 * U64 * (var + mu * mu)      # (var + mu^2) - mu^2
        assert (np.abs(ovar[1] - var) <= var_tol).all()
        for sp in (0, 2):
            np.testing.assert_array_equal(omu[sp][5], mu[5])
            assert (np.abs(ovar[sp][5] - var[5]) <= var_tol[5]).all()
            n, f, s, _ = ogmm.suff_stats(frames[sp].astype(np.float64), w, mu, var)
            assert n[5] == 0.0
            rw, rmu, rvar = ogmm.map_adapt(n, f, s, w, mu, var, len(frames[sp]), relevance, every)
            # the tolerances of tests/test_gpu_gmm.py::test_map_adapt_matches_oracle (tensor-core statistics)
            np.testing.assert_allclose(omu[sp], rmu, atol=2e-4)
            np.testing.assert_allclose(ow[sp], rw, atol=1e-5)
            np.testing.assert_allclose(ovar[sp], rvar, rtol=1e-3, atol=1e-3)
            note(f"map_adapt relevance {relevance} speaker {sp} means", float(np.abs(omu[sp] - rmu).max()))


# ------------------------------------------------------------------------------------------------ VAD
def vad_cfg(shift, n_blocks, normalize, pcm_dtype):
    from speech_signal_processing_b200 import _lib

    return _lib.VadCfg(256, shift, n_blocks, normalize, pcm_dtype, 1e-8)


def vad_run(sigs, shift, n_blocks, normalize, pcm_dtype):
    """ssp_vad_features over a batch: (zcr, power, entropy) as float64 numpy, frame offsets."""
    import torch

    lens = [len(s) for s in sigs]
    soffs = offsets(lens)
    foffs = offsets([-(-n // shift) for n in lens])
    cat = np.concatenate(sigs).astype(np.int16 if pcm_dtype == 0 else np.float32)
    total = int(foffs[-1])
    z = torch.full((total,), float("nan"), dtype=torch.float32, device="cuda")
    p = torch.full((total,), float("nan"), dtype=torch.float64, device="cuda")
    e = torch.full((total,), float("nan"), dtype=torch.float32, device="cuda")
    cfg = vad_cfg(shift, n_blocks, normalize, pcm_dtype)
    log = run("ssp_vad_features", P(dev(cat)), P(dev(soffs)), len(sigs), C.byref(cfg), P(dev(foffs)), P(z), P(p), P(e))
    assert log == {"vad_features_kernel": 1}, log
    return z.cpu().numpy().astype(np.float64), p.cpu().numpy(), e.cpu().numpy().astype(np.float64), foffs


def check_vad(key, sigs, got, shift, n_blocks, normalize):
    z, p, e, foffs = got
    worst = [0.0, 0.0]
    for u, s in enumerate(sigs):
        sl = slice(foffs[u], foffs[u + 1])
        if len(s) == 0:
            assert foffs[u + 1] == foffs[u]
            continue
        wz, wp, we = vad_ref(s, shift, n_blocks, normalize)
        assert len(wz) == foffs[u + 1] - foffs[u]
        np.testing.assert_array_equal(z[sl], wz, err_msg=f"{key} zcr {u}")
        same_nonfinite(p[sl], wp, key)
        same_nonfinite(e[sl], we, key)
        fin = np.isfinite(wp)
        rel = np.abs(p[sl][fin] - wp[fin]) / np.maximum(np.abs(wp[fin]), 1e-300)
        assert (rel <= 1e-12).all() and np.array_equal(p[sl][fin] == 0, wp[fin] == 0), f"{key} energy {u}"
        fin = np.isfinite(we)
        ent = np.abs(e[sl][fin] - we[fin])
        assert (ent <= ENT_ATOL).all(), f"{key} entropy {u}: {ent.max():.3e}"
        if rel.size:
            worst[0] = max(worst[0], float(rel.max()))
        if ent.size:
            worst[1] = max(worst[1], float(ent.max()))
    note(f"{key} energy (relative)", worst[0])
    note(f"{key} entropy (absolute)", worst[1])


def vad_signals(seed, pcm_dtype):
    """Utterances of 0, 1, 255, 256 and 257 samples, speech, speech with a full-scale -32768 sample, and silence."""
    sp = synth.synth_utterance(seed % 5, seed, 6000)
    sigs = [sp[100 : 100 + n] for n in VAD_LENS] + [sp[:3000], sp[2000:4711].copy()]
    sigs[-1][100] = -32768
    sigs.append(np.zeros(700, np.int16))
    sigs.append(sp[-1333:])
    if pcm_dtype == 1:
        rs = np.random.RandomState(seed)
        sigs = [(s.astype(np.float64) / 32768.0 * rs.uniform(0.01, 3.0)).astype(np.float32) for s in sigs]
    return sigs


@pytest.mark.gpu
@pytest.mark.parametrize("shift", VAD_SHIFTS)
def test_vad_features_match_float64(gpu, shift):
    """Every hop from 1 to 256 with 1, 3, 10 and 32 sub-bands, with and without peak normalisation, int16 and float32
    PCM: the silent utterance's NaNs stay inside its own frames."""
    for n_blocks in VAD_BLOCKS:
        for normalize in (1, 0):
            for pcm_dtype in (0, 1):
                sigs = vad_signals(shift + n_blocks, pcm_dtype)
                got = vad_run(sigs, shift, n_blocks, normalize, pcm_dtype)
                key = f"vad hop {shift} blocks {n_blocks} normalize {normalize} {('int16', 'float32')[pcm_dtype]}"
                check_vad(key, sigs, got, shift, n_blocks, normalize)
                silent = len(sigs) - 2
                in_silence = np.zeros(len(got[1]), bool)
                in_silence[got[3][silent] : got[3][silent + 1]] = True
                assert np.isfinite(got[1][~in_silence]).all() and np.isfinite(got[2][~in_silence]).all()
                assert np.isnan(got[1][in_silence]).all() == bool(normalize)


@pytest.mark.gpu
def test_vad_rejects_out_of_range_configurations(gpu):
    torch = gpu
    buf = torch.zeros(1024, dtype=torch.float64, device="cuda")
    offs = dev(np.array([0, 256], np.int64))
    foffs = dev(np.array([0, 1], np.int64))
    for shift, n_blocks in [(s, 10) for s in VAD_SHIFT_REJECT] + [(128, b) for b in VAD_BLOCK_REJECT]:
        cfg = vad_cfg(shift, n_blocks, 1, 0)
        rejected("ssp_vad_features", P(buf), P(offs), 1, C.byref(cfg), P(foffs), P(buf), P(buf), P(buf))
    cfg = vad_cfg(128, 10, 1, 0)
    cfg.frame_len = 512
    rejected("ssp_vad_features", P(buf), P(offs), 1, C.byref(cfg), P(foffs), P(buf), P(buf), P(buf))


@pytest.mark.gpu
def test_vad_features_more_than_65535_utterances(gpu):
    """70 000 short utterances in one launch: every frame written, and the utterances past the 65 535th (and a sample
    of the others) equal to the reference."""
    rs = np.random.RandomState(3)
    n = 70000
    lens = rs.randint(1, 400, size=n)
    base = synth.synth_utterance(1, 9, 200000)
    starts = rs.randint(0, len(base) - 400, size=n)
    sigs = [base[a : a + m] for a, m in zip(starts, lens)]
    got = vad_run(sigs, 128, 10, 0, 0)
    assert np.isfinite(got[0]).all() and np.isfinite(got[1]).all() and np.isfinite(got[2]).all()
    pick = sorted(set(range(65530, n, 7)) | set(rs.randint(0, 65530, size=300).tolist()))
    z, p, e, foffs = got
    sub = []
    for u in pick:
        sl = slice(foffs[u], foffs[u + 1])
        sub.append((sigs[u], z[sl], p[sl], e[sl]))
    zs = np.concatenate([s[1] for s in sub])
    ps = np.concatenate([s[2] for s in sub])
    es = np.concatenate([s[3] for s in sub])
    check_vad("vad 70000 utterances", [s[0] for s in sub], (zs, ps, es, offsets([len(s[1]) for s in sub])), 128, 10, 0)


@pytest.mark.gpu
def test_vad_detect_matches_the_oracle(gpu):
    """Random feature tracks, ragged, many utterances per launch, over min_len, ampl, amph and zcr_gate: decisions
    equal to oracle.vad.detect (utterances where the reference itself raises IndexError are skipped)."""
    torch = gpu
    rs = np.random.RandomState(5)
    compared = 0
    for trial, (min_len, ampl, amph, gate) in enumerate([(16, 0.3, 12.0, 35.0), (0, 0.3, 12.0, 35.0), (1, 1.0, 8.0, 25.0),
                                                          (5, 0.05, 3.0, 10.5), (40, 2.0, 20.0, 60.0), (16, 0.3, 12.0, 0.0)]):
        lens = rs.randint(0, 400, size=257)
        lens[:3] = (0, 1, 2)
        zs, ps = [], []
        for n in lens:
            p = np.abs(rs.standard_normal(n)) * rs.choice([0.05, 1.0, 25.0], size=n, p=[0.3, 0.3, 0.4])
            if n > 2:
                r = rs.randint(0, n - 1)
                p[r : r + rs.randint(0, 80)] = 30.0
                if rs.rand() < 0.5:
                    p[0] = 0.01
            zs.append((rs.randint(0, 80, size=n) * (p > 0.1)).astype(np.float32))
            ps.append(p)
        foffs = offsets(lens)
        out = torch.full((int(foffs[-1]),), 7, dtype=torch.uint8, device="cuda")
        log = run("ssp_vad_detect", P(dev(np.concatenate(zs))), P(dev(np.concatenate(ps))), P(dev(foffs)), len(lens), gate, ampl,
                  amph, min_len, P(out))
        assert log == {"vad_detect_kernel": 1}, log
        got = out.cpu().numpy()
        assert set(np.unique(got)) <= {0, 1}
        for u in range(len(lens)):
            try:
                want = ov.detect(zs[u], ps[u], gate, ampl, amph, min_len)[:, 0]
            except IndexError:
                continue
            assert np.array_equal(got[foffs[u] : foffs[u + 1]], want.astype(np.uint8)), (trial, u)
            compared += 1
    assert compared > 1000
    note("vad_detect utterances compared", compared)
