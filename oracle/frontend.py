"""numpy (float64) restatement of the reference front-ends.  TEST INFRASTRUCTURE ONLY.

Every function cites the reference (or third-party upstream) lines it follows.
See ``oracle/__init__.py`` for what is pinned and what is "parity unpinned".
"""
from __future__ import annotations

import math

import numpy as np

# ----------------------------------------------------------------------------
# shared pieces
# ----------------------------------------------------------------------------


def dct2_ortho_matrix(n_out: int, n_in: int, first: int = 0) -> np.ndarray:
    """Rows ``first .. first+n_out-1`` of the orthonormal DCT-II of length ``n_in``.

    scipy ``dct(x, type=2, norm='ortho')`` as used at utils/processing.py:106.
    """
    k = np.arange(first, first + n_out)[:, None].astype(np.float64)
    n = np.arange(n_in)[None, :].astype(np.float64)
    m = np.cos(np.pi * k * (2.0 * n + 1.0) / (2.0 * n_in)) * math.sqrt(2.0 / n_in)
    m[(k[:, 0] == 0)] *= math.sqrt(0.5)
    return m


def delta(feat: np.ndarray, N: int = 2) -> np.ndarray:
    """GMM_UBM.py:53-69 -- regression deltas with edge padding.

    delta_t = sum_{n=-N..N} n * c_{t+n} / (2 * sum_{n=1..N} n^2)
    """
    if N < 1:
        raise ValueError("N must be an integer >= 1")
    feat = np.asarray(feat)
    T = feat.shape[0]
    denom = 2.0 * sum(i * i for i in range(1, N + 1))
    idx = np.arange(T)
    out = np.zeros(feat.shape, dtype=np.float64)
    f64 = feat.astype(np.float64)
    for n in range(1, N + 1):
        hi = np.minimum(idx + n, T - 1)
        lo = np.maximum(idx - n, 0)
        out += n * (f64[hi] - f64[lo])
    return (out / denom).astype(feat.dtype if feat.dtype.kind == "f" else np.float64)


def scale(x: np.ndarray) -> np.ndarray:
    """sklearn.preprocessing.scale(X) as called at GMM_UBM.py:93 (axis=0, ddof=0).

    sklearn/preprocessing/_data.py:127,260-285: std below 10*eps is replaced by 1.
    """
    x = np.asarray(x)
    x64 = x.astype(np.float64)
    mean = x64.mean(axis=0)
    xc = x64 - mean
    std = np.sqrt((xc * xc).mean(axis=0))
    # _data.py:266-277: a mean that could not be represented exactly leaves a residue; sklearn removes it once more
    mean_1 = xc.mean(axis=0)
    if not np.allclose(mean_1, 0):
        xc = xc - mean_1
    std = np.where(std < 10 * np.finfo(x64.dtype).eps, 1.0, std)
    out = xc / std
    # _data.py:281-296: ... and again after the division when the deviation itself is at rounding level (a column that
    # is constant up to the inexact mean comes out as 0, not as +-1)
    mean_2 = out.mean(axis=0)
    if not np.allclose(mean_2, 0):
        out = out - mean_2
    return out.astype(x.dtype if x.dtype.kind == "f" else np.float64)


# ----------------------------------------------------------------------------
# utils/processing.py (in-repo front-end)
# ----------------------------------------------------------------------------


def processing_fbank(fs: float, nfft: int):
    """utils/processing.py:42-88 -- 13 linear + 27 log area-normalised triangles
    evaluated on the two-sided bin grid k*fs/nfft, k = 0..nfft-1."""
    n_lin, n_log = 13, 27
    n_filt = n_lin + n_log
    freqs = np.zeros(n_filt + 2)
    freqs[:n_lin] = 133.33 + np.arange(n_lin) * (200.0 / 3.0)
    freqs[n_lin:] = freqs[n_lin - 1] * 1.0711703 ** np.arange(1, n_log + 3)
    heights = 2.0 / (freqs[2:] - freqs[:-2])
    fb = np.zeros((n_filt, nfft))
    grid = np.arange(nfft) / float(nfft) * fs
    for i in range(n_filt):
        lo, ce, hi = freqs[i], freqs[i + 1], freqs[i + 2]
        b_lo = int(math.floor(lo * nfft / fs))
        b_ce = int(math.floor(ce * nfft / fs))
        b_hi = int(math.floor(hi * nfft / fs))
        up = np.arange(b_lo + 1, b_ce + 1)
        dn = np.arange(b_ce + 1, b_hi + 1)
        fb[i, up] = heights[i] / (ce - lo) * (grid[up] - lo)
        fb[i, dn] = heights[i] / (hi - ce) * (hi - grid[dn])
    return fb, freqs


def processing_enframe(sig: np.ndarray, frame_size: int = 400, step: int = 160) -> np.ndarray:
    """utils/processing.py:19-38 -- ceil(N/step) frames, zero-padded tail, symmetric
    Hamming window; returns (frame_size, n_frames) like the reference."""
    sig = np.asarray(sig, dtype=np.float64)
    n = sig.shape[0]
    n_frames = int(math.ceil(n / step))
    padded = np.zeros((n_frames - 1) * step + frame_size if n_frames > 0 else 0)
    padded[: min(n, padded.shape[0])] = sig[: padded.shape[0]]
    idx = np.arange(frame_size)[:, None] + step * np.arange(n_frames)[None, :]
    k = np.arange(frame_size)
    window = 0.54 - 0.46 * np.cos(2.0 * np.pi * k / (frame_size - 1))
    return padded[idx] * window[:, None]


def processing_mfcc(sig: np.ndarray, fs: float = 8000, frame_size: int = 512, step: int = 256) -> np.ndarray:
    """utils/processing.py:110-144 (MFCC) + :91-107 (stMFCC): per frame
    |FFT_n(x)|/n over all n = frame_size bins, log10(X.fbank^T + 1e-8), DCT-II ortho,
    first 13 coefficients (c0 kept)."""
    nfft = int(frame_size)
    fb, _ = processing_fbank(fs, nfft)
    frames = processing_enframe(sig, frame_size, step)  # (nfft, T)
    spec = np.abs(np.fft.fft(frames, axis=0)) / nfft  # (nfft, T) two-sided magnitude
    mspec = np.log10(fb @ spec + 1e-8)  # (40, T)
    return (dct2_ortho_matrix(13, fb.shape[0]) @ mspec).T  # (T, 13)


# ----------------------------------------------------------------------------
# SIDEKIT mfcc (what GMM_UBM.py:89 actually calls) -- PARITY UNPINNED
# ----------------------------------------------------------------------------


def hz2mel(f):
    return 2595.0 * np.log10(1.0 + np.asarray(f, dtype=np.float64) / 700.0)


def mel2hz(m):
    return 700.0 * (10.0 ** (np.asarray(m, dtype=np.float64) / 2595.0) - 1.0)


def sidekit_trfbank(fs, nfft, lowfreq, maxfreq, nlinfilt, nlogfilt):
    """SIDEKIT 1.3 frontend/features.py ``trfbank`` with nlinfilt == 0: nlogfilt
    triangles equally spaced in mel between lowfreq and maxfreq, area-normalised
    (height 2/(hi-lo)), weights linear in Hz, one-sided grid of nfft/2+1 bins; the
    falling edge drops its last bin (``rid[:-1]``)."""
    if nlinfilt != 0:
        raise NotImplementedError("oracle restates the nlinfilt == 0 branch only")
    nfilt = nlogfilt
    mels = hz2mel(lowfreq) + np.arange(nfilt + 2) * (hz2mel(maxfreq) - hz2mel(lowfreq)) / (nfilt + 1)
    freqs = mel2hz(mels)
    heights = 2.0 / (freqs[2:] - freqs[:-2])
    fb = np.zeros((nfilt, nfft // 2 + 1))
    grid = np.arange(nfft) / float(nfft) * fs
    for i in range(nfilt):
        lo, ce, hi = freqs[i], freqs[i + 1], freqs[i + 2]
        up = np.arange(math.floor(lo * nfft / fs) + 1, math.floor(ce * nfft / fs) + 1, dtype=int)
        dn = np.arange(math.floor(ce * nfft / fs) + 1, min(math.floor(hi * nfft / fs) + 1, nfft), dtype=int)
        fb[i, up] = heights[i] / (ce - lo) * (grid[up] - lo)
        dn = dn[:-1]
        fb[i, dn] = heights[i] / (hi - ce) * (hi - grid[dn])
    return fb, freqs


def sidekit_frames(sig: np.ndarray, win: int, shift: int) -> np.ndarray:
    """SIDEKIT ``framing``: floor((N-win)/shift)+1 frames, no padding."""
    sig = np.asarray(sig, dtype=np.float64)
    n_frames = (sig.shape[0] - win) // shift + 1
    if n_frames < 1:
        return np.zeros((0, win))
    idx = np.arange(win)[None, :] + shift * np.arange(n_frames)[:, None]
    return sig[idx]


def sidekit_mfcc(sig, lowfreq=100, maxfreq=8000, nlinfilt=0, nlogfilt=24, nwin=0.025, fs=16000,
                 nceps=13, shift=0.01, get_spec=False, get_mspec=False, prefac=0.97):
    """SIDEKIT 1.3 ``mfcc`` (signature as bound at GMM_UBM.py:20 / called :89).

    framing 400/160 without padding -> per-frame pre-emphasis (y[0] = x[0] - p*x[0]) ->
    log-energy = ln(sum y^2) -> Hanning -> rFFT(512) power -> 24 mel triangles ->
    ln -> DCT-II ortho, coefficients 1..nceps (c0 dropped).
    Returns [ceps (T,nceps), log_energy (T,), spec|None, mspec|None].
    """
    win = int(round(nwin * fs))
    hop = int(shift * fs)
    nfft = 2 ** int(math.ceil(math.log2(win)))
    framed = sidekit_frames(sig, win, hop)
    prev = np.concatenate([framed[:, :1], framed[:, :-1]], axis=1)
    framed = framed - prefac * prev
    log_energy = np.log((framed ** 2).sum(axis=1))
    k = np.arange(win)
    window = 0.5 - 0.5 * np.cos(2.0 * np.pi * k / (win - 1))  # numpy.hanning
    mag = np.fft.rfft(framed * window, nfft, axis=-1)
    spec = mag.real ** 2 + mag.imag ** 2
    fb, _ = sidekit_trfbank(fs, nfft, lowfreq, maxfreq, nlinfilt, nlogfilt)
    mspec = np.log(spec @ fb.T)
    ceps = mspec @ dct2_ortho_matrix(nceps, fb.shape[0], first=1).T
    return [ceps, log_energy, spec if get_spec else None, mspec if get_mspec else None]


# ----------------------------------------------------------------------------
# python_speech_features mfcc (BASELINE config 1 "26 mel") -- PARITY UNPINNED
# ----------------------------------------------------------------------------


def _round_half_up(x: float) -> int:
    return int(math.floor(x + 0.5))


def psf_filterbanks(nfilt=26, nfft=512, samplerate=16000, lowfreq=0, highfreq=None):
    """python_speech_features ``get_filterbanks``: unit-peak triangles on integer bins
    floor((nfft+1)*hz/fs)."""
    highfreq = highfreq or samplerate / 2
    melpoints = np.linspace(hz2mel(lowfreq), hz2mel(highfreq), nfilt + 2)
    bins = np.floor((nfft + 1) * mel2hz(melpoints) / samplerate).astype(int)
    fb = np.zeros((nfilt, nfft // 2 + 1))
    for j in range(nfilt):
        for i in range(bins[j], bins[j + 1]):
            fb[j, i] = (i - bins[j]) / (bins[j + 1] - bins[j])
        for i in range(bins[j + 1], bins[j + 2]):
            fb[j, i] = (bins[j + 2] - i) / (bins[j + 2] - bins[j + 1])
    return fb


def psf_mfcc(sig, samplerate=16000, winlen=0.025, winstep=0.01, numcep=13, nfilt=26, nfft=512,
             lowfreq=0, highfreq=None, preemph=0.97, ceplifter=22, appendEnergy=True):
    """python_speech_features 0.6 ``mfcc`` with its defaults (rectangular window)."""
    sig = np.asarray(sig, dtype=np.float64)
    sig = np.concatenate([sig[:1], sig[1:] - preemph * sig[:-1]])
    flen = _round_half_up(winlen * samplerate)
    fstep = _round_half_up(winstep * samplerate)
    n = sig.shape[0]
    n_frames = 1 if n <= flen else 1 + int(math.ceil((n - flen) / fstep))
    padded = np.zeros((n_frames - 1) * fstep + flen)
    padded[:n] = sig
    idx = np.arange(flen)[None, :] + fstep * np.arange(n_frames)[:, None]
    frames = padded[idx]
    pspec = np.abs(np.fft.rfft(frames, nfft, axis=-1)) ** 2 / nfft
    eps = np.finfo(float).eps
    energy = pspec.sum(axis=1)
    energy = np.where(energy == 0, eps, energy)
    feat = pspec @ psf_filterbanks(nfilt, nfft, samplerate, lowfreq, highfreq).T
    feat = np.where(feat == 0, eps, feat)
    feat = np.log(feat) @ dct2_ortho_matrix(numcep, nfilt).T
    if ceplifter > 0:
        feat = feat * (1.0 + (ceplifter / 2.0) * np.sin(np.pi * np.arange(numcep) / ceplifter))
    if appendEnergy:
        feat[:, 0] = np.log(energy)
    return feat


# ----------------------------------------------------------------------------
# the reference feature recipe: extract_feature (GMM_UBM.py:72-118)
# ----------------------------------------------------------------------------


def features(sig, preset="sidekit", delta_order=1, cmvn=True, **kw):
    """GMM_UBM.py:89-93 for one utterance: cepstra -> delta -> hstack -> scale.

    delta_order 1 is the reference (26-d); 2 adds delta(delta(c)) (39-d, SURVEY F5).
    """
    if preset == "sidekit":
        c = sidekit_mfcc(sig, **kw)[0]
    elif preset == "psf":
        c = psf_mfcc(sig, **kw)
    elif preset == "processing":
        c = processing_mfcc(sig, **kw)
    else:
        raise NameError(preset)
    parts = [c]
    d = c
    for _ in range(delta_order):
        d = delta(d)
        parts.append(d)
    f = np.hstack(parts)
    return scale(f) if cmvn else f


# ----------------------------------------------------------------------------
# sidekit plp (GMM_UBM.py:20 binds it, :94-99 calls it for feature_type == 'PLP') -- PARITY UNPINNED
# ----------------------------------------------------------------------------
# SIDEKIT is absent from the container (see sidekit_mfcc above).  Its ``plp`` is a port of Ellis' rastamat
# (rastaplp.m: powspec -> audspec -> rasta -> postaud -> dolpc -> lpc2cep -> lifter); the restatement below follows
# that published algorithm with SIDEKIT's defaults (nwin=0.025, fs=16000, plp_order=13, shift=0.01, prefac=0.97,
# rasta=True) and the same framing / pre-emphasis / window / FFT front half as ``sidekit_mfcc``.


def hz2bark(f):
    return 6.0 * np.arcsinh(np.asarray(f, dtype=np.float64) / 600.0)


def bark2hz(z):
    return 600.0 * np.sinh(np.asarray(z, dtype=np.float64) / 6.0)


def fft2barkmx(nfft, fs, nfilts=0, width=1.0, minfreq=0.0, maxfreq=None):
    """rastamat fft2barkmx: Bark-spaced trapezoid-in-log filters, 10^min(0, min(hif, -2.5 lof)/width)."""
    maxfreq = fs / 2.0 if maxfreq is None else maxfreq
    min_bark = hz2bark(minfreq)
    nyqbark = hz2bark(maxfreq) - min_bark
    if nfilts == 0:
        nfilts = int(math.ceil(nyqbark)) + 1
    step = nyqbark / (nfilts - 1)
    binbarks = hz2bark(np.arange(nfft // 2 + 1) * fs / nfft)
    wts = np.zeros((nfilts, nfft // 2 + 1))
    for i in range(nfilts):
        mid = min_bark + i * step
        lof = binbarks - mid - 0.5
        hif = binbarks - mid + 0.5
        wts[i] = 10.0 ** (np.minimum(0.0, np.minimum(hif, -2.5 * lof) / width))
    return wts


def rasta_filter_coefficients():
    numer = np.arange(-2, 3, dtype=np.float64)
    numer = -numer / np.sum(numer * numer)     # [0.2, 0.1, 0, -0.1, -0.2]
    return numer, np.array([1.0, -0.94])


def rasta_filt(x):
    """rastamat rastafilt on (T, nbands) log spectra, filtering along time: the FIR part alone runs over the first
    four frames to set the state (their outputs are zeroed), the full IIR filter continues from that state."""
    from scipy.signal import lfilter

    numer, denom = rasta_filter_coefficients()
    x = np.asarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    n0 = min(4, x.shape[0])
    _, z = lfilter(numer, [1.0], x[:n0], axis=0, zi=np.zeros((4, x.shape[1])))
    if x.shape[0] > 4:
        y[4:], _ = lfilter(numer, denom, x[4:], axis=0, zi=z)
    return y


def postaud_weights(nbands, fmax):
    """rastamat postaud (Bark): equal-loudness weights at the band centres."""
    cf = bark2hz(np.linspace(0.0, hz2bark(fmax), nbands))
    fsq = cf ** 2
    ftmp = fsq + 1.6e5
    return (fsq / ftmp) ** 2 * ((fsq + 1.44e6) / (fsq + 9.61e6))


def levinson(r, order):
    """Levinson-Durbin per row of r (T, >= order + 1): returns a (T, order + 1) with a[:, 0] = 1 and the error e (T,)."""
    r = np.asarray(r, dtype=np.float64)
    t = r.shape[0]
    a = np.zeros((t, order + 1))
    a[:, 0] = 1.0
    e = r[:, 0].copy()
    for i in range(1, order + 1):
        acc = r[:, i].copy()
        for j in range(1, i):
            acc += a[:, j] * r[:, i - j]
        k = -acc / e
        prev = a.copy()
        for j in range(1, i):
            a[:, j] = prev[:, j] + k * prev[:, i - j]
        a[:, i] = k
        e = e * (1.0 - k * k)
    return a, e


def sidekit_plp(sig, nwin=0.025, fs=16000, plp_order=13, shift=0.01, get_spec=False, get_mspec=False, prefac=0.97,
                rasta=True):
    """Restatement of SIDEKIT ``plp`` (rastamat ``rastaplp``).  Returns ``[ceps (T, plp_order), log_energy (T,), None, None]``."""
    win = int(round(nwin * fs))
    hop = int(shift * fs)
    nfft = 2 ** int(math.ceil(math.log2(win)))
    framed = sidekit_frames(sig, win, hop)
    prev = np.concatenate([framed[:, :1], framed[:, :-1]], axis=1)
    framed = framed - prefac * prev
    log_energy = np.log((framed ** 2).sum(axis=1))
    k = np.arange(win)
    window = 0.5 - 0.5 * np.cos(2.0 * np.pi * k / (win - 1))
    mag = np.fft.rfft(framed * window, nfft, axis=-1)
    powspec = mag.real ** 2 + mag.imag ** 2                              # (T, 257)
    wts = fft2barkmx(nfft, fs, 0, 1.0, 0.0, fs / 2.0)                    # (21, 257) at 16 kHz
    asp = powspec @ wts.T                                                # (T, nbands)
    return [plp_post(asp, plp_order, fs / 2.0, rasta), log_energy, None, None]


def plp_post(asp, plp_order, fmax, rasta=True):
    """The back half of ``rastaplp`` on critical-band energies asp (T, nbands): rasta -> postaud -> dolpc -> lpc2cep ->
    lifter.  Returns the liftered cepstra (T, plp_order)."""
    order = plp_order - 1
    nbands = asp.shape[1]
    if rasta:
        asp = np.exp(rasta_filt(np.log(asp)))
    post = (postaud_weights(nbands, fmax)[None, :] * asp) ** 0.33
    post[:, 0] = post[:, 1]
    post[:, -1] = post[:, -2]
    # dolpc: autocorrelation = real IDFT of the even-symmetric extension, then Levinson-Durbin
    ext = np.concatenate([post, post[:, nbands - 2 : 0 : -1]], axis=1)   # (T, 2 (nbands - 1))
    r = np.real(np.fft.ifft(ext, axis=1))[:, : order + 1]
    a, e = levinson(r, order)
    lpc = a / e[:, None]
    # lpc2cep
    ncep = order + 1
    cep = np.zeros((lpc.shape[0], ncep))
    cep[:, 0] = -np.log(lpc[:, 0])
    norm = lpc / lpc[:, :1]
    for n in range(1, ncep):
        s = np.zeros(lpc.shape[0])
        for m in range(1, n):
            s += (n - m) * norm[:, m] * cep[:, n - m]
        cep[:, n] = -(norm[:, n] + s / n)
    lift = np.concatenate([[1.0], np.arange(1, ncep, dtype=np.float64) ** 0.6])
    return cep * lift[None, :]


# ----------------------------------------------------------------------------
# librosa.feature.mfcc (MFCC_DTW.py:27-30 ``MFCC_lib``) -- PARITY UNPINNED
# ----------------------------------------------------------------------------
# librosa is absent from the container and un-pinned (requirements.txt).  Restated from its published algorithm with
# the defaults the reference call relies on: ``librosa.feature.mfcc(y, sr=8000, n_mfcc=13)`` -> melspectrogram
# (n_fft=2048, hop_length=512, periodic Hann, center=True with reflect padding, power 2, 128 Slaney mel bands with
# area normalisation, fmin 0, fmax sr/2) -> power_to_db (ref 1, amin 1e-10, top_db 80 against the maximum of the
# whole utterance) -> DCT-II ortho, first n_mfcc rows.  torchaudio's MFCC transform (same conventions, an independent
# implementation) is the cross-check in tests/test_oracle.py.


def slaney_hz_to_mel(f):
    f = np.asarray(f, dtype=np.float64)
    f_sp = 200.0 / 3.0
    min_log_hz, logstep = 1000.0, math.log(6.4) / 27.0
    lin = f / f_sp
    return np.where(f >= min_log_hz, min_log_hz / f_sp + np.log(np.maximum(f, min_log_hz) / min_log_hz) / logstep, lin)


def slaney_mel_to_hz(m):
    m = np.asarray(m, dtype=np.float64)
    f_sp = 200.0 / 3.0
    min_log_hz, logstep = 1000.0, math.log(6.4) / 27.0
    min_log_mel = min_log_hz / f_sp
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), f_sp * m)


def librosa_mel_filters(sr, n_fft, n_mels=128, fmin=0.0, fmax=None):
    """``librosa.filters.mel(sr, n_fft, n_mels, fmin, fmax, htk=False, norm='slaney')`` -> (n_mels, n_fft//2+1)."""
    fmax = sr / 2.0 if fmax is None else fmax
    fftfreqs = np.arange(n_fft // 2 + 1) * (sr / float(n_fft))
    mel_f = slaney_mel_to_hz(np.linspace(slaney_hz_to_mel(fmin), slaney_hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = mel_f[:, None] - fftfreqs[None, :]
    w = np.zeros((n_mels, n_fft // 2 + 1))
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        w[i] = np.maximum(0.0, np.minimum(lower, upper))
    w *= (2.0 / (mel_f[2 : n_mels + 2] - mel_f[:n_mels]))[:, None]
    return w


def librosa_mfcc(y, sr=8000, n_mfcc=13, n_fft=2048, hop_length=512, n_mels=128, fmin=0.0, fmax=None, top_db=80.0,
                 center=True, pad_mode="reflect", amin=1e-10):
    """``librosa.feature.mfcc`` -> (n_mfcc, T) like librosa (MFCC_DTW.py:28 then takes ``.T.flatten()``)."""
    y = np.asarray(y, dtype=np.float64)
    if center:
        y = np.pad(y, n_fft // 2, mode=pad_mode)
    if len(y) < n_fft:
        return np.zeros((n_mfcc, 0))
    T = 1 + (len(y) - n_fft) // hop_length
    win = 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(n_fft) / n_fft)  # scipy get_window('hann', fftbins=True)
    frames = np.stack([y[t * hop_length : t * hop_length + n_fft] for t in range(T)]) * win
    power = np.abs(np.fft.rfft(frames, n_fft, axis=1)) ** 2
    mel = power @ librosa_mel_filters(sr, n_fft, n_mels, fmin, fmax).T
    db = 10.0 * np.log10(np.maximum(amin, mel))  # ref = 1.0 -> the reference term is 10 log10(max(amin, 1)) = 0
    if top_db is not None:
        db = np.maximum(db, db.max() - top_db)
    return (db @ dct2_ortho_matrix(n_mfcc, n_mels).T).T


def mfcc_lib(raw_signal, n_mfcc=13):
    """MFCC_DTW.py:27-30 ``MFCC_lib``: float32 cast, sr=8000, flattened frame-major."""
    return librosa_mfcc(np.asarray(raw_signal).astype("float32"), sr=8000, n_mfcc=n_mfcc).T.flatten()
