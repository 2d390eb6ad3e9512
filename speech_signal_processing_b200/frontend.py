"""Host side of the fused front-end kernel, behind the reference's own entry points.

Drop-ins (same names, arguments and return conventions as the reference's callees):

* :func:`mfcc`  -- ``sidekit.frontend.features.mfcc`` as bound at GMM_UBM.py:20 and called at
  GMM_UBM.py:89, UI/GMM_UBM_GUI.py:91: returns ``[ceps, log_energy, None, None]``.
* :func:`MFCC`  -- ``utils.processing.MFCC`` (utils/processing.py:110-144).
* :func:`delta` -- ``GMM_UBM.delta`` (GMM_UBM.py:53-69).
* :func:`scale` -- ``sklearn.preprocessing.scale`` as called at GMM_UBM.py:93.
* :func:`extract_feature` -- ``GMM_UBM.extract_feature`` (GMM_UBM.py:72-118), batched: ONE kernel
  launch for the whole list instead of a Python loop per utterance and per frame.

The conventions that differ between recipes (framing, window, pre-emphasis, spectrum, filterbank,
log, DCT rows, lifter, energy) are tables + a small config struct; the kernel is the same.
Tables are computed here in float64 and uploaded once per :class:`FrontEnd`.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field

import numpy as np

from . import _lib

# --------------------------------------------------------------------------------------------
# host-side table builders
# --------------------------------------------------------------------------------------------


def _mel(f):
    return 2595.0 * np.log10(1.0 + np.asarray(f, dtype=np.float64) / 700.0)


def _imel(m):
    return 700.0 * (np.power(10.0, np.asarray(m, dtype=np.float64) / 2595.0) - 1.0)


def _area_triangles(edges_hz: np.ndarray, nfft: int, fs: float, n_bins: int, drop_last_falling: bool) -> np.ndarray:
    """Area-normalised triangles (height 2/(hi-lo)) sampled on the FFT bin grid k*fs/nfft with
    the talkbox bin rule: rising edge on bins floor(lo*nfft/fs)+1 .. floor(ce*nfft/fs), falling
    edge on floor(ce*nfft/fs)+1 .. floor(hi*nfft/fs) (utils/processing.py:72-86)."""
    n_filt = len(edges_hz) - 2
    fb = np.zeros((n_filt, n_bins))
    hz = np.arange(n_bins) * (fs / nfft)
    for m in range(n_filt):
        lo, ce, hi = edges_hz[m : m + 3]
        height = 2.0 / (hi - lo)
        k_lo, k_ce, k_hi = (int(math.floor(v * nfft / fs)) for v in (lo, ce, hi))
        rise = np.arange(k_lo + 1, min(k_ce, n_bins - 1) + 1)
        last = min(k_hi + 1, nfft) - 1
        if drop_last_falling:
            last -= 1
        fall = np.arange(k_ce + 1, min(last, n_bins - 1) + 1)
        fb[m, rise] = height / (ce - lo) * (hz[rise] - lo)
        fb[m, fall] = height / (hi - ce) * (hi - hz[fall])
    return fb


def sidekit_filterbank(fs, nfft, lowfreq, maxfreq, nlogfilt):
    edges = _imel(_mel(lowfreq) + np.arange(nlogfilt + 2) * ((_mel(maxfreq) - _mel(lowfreq)) / (nlogfilt + 1)))
    return _area_triangles(edges, nfft, fs, nfft // 2 + 1, drop_last_falling=True)


def _talkbox_edges() -> np.ndarray:
    """The 42 triangle corner frequencies of utils/processing.py:49-63: 13 linear (133.33 Hz + k * 66.67) and 29
    log-spaced (x 1.0711703) points."""
    edges = np.zeros(42)
    edges[:13] = 133.33 + (200.0 / 3.0) * np.arange(13)
    edges[13:] = edges[12] * 1.0711703 ** np.arange(1, 30)
    return edges


def mfccInitFilterBanks(fs, nfft):
    """``utils.processing.mfccInitFilterBanks`` (utils/processing.py:42-88): ``(fbank (40, nfft), freqs (42,))`` on the
    reference's TWO-sided bin grid k*fs/nfft, k < nfft.  A host-side table (it is what :func:`processing_recipe` folds
    onto nfft/2+1 bins and uploads), not a kernel."""
    edges = _talkbox_edges()
    return _area_triangles(edges, int(nfft), fs, int(nfft), drop_last_falling=False), edges


def processing_filterbank(fs, nfft):
    """utils/processing.py:42-88 evaluated on ALL nfft bins, then folded onto 0..nfft/2: the
    reference multiplies the two-sided magnitude spectrum (|X[k]| == |X[nfft-k]|) by a filterbank
    whose edges can exceed fs/2 (they do at fs = 8000)."""
    two_sided = _area_triangles(_talkbox_edges(), nfft, fs, nfft, drop_last_falling=False)
    half = nfft // 2
    fb = two_sided[:, : half + 1].copy()
    mirror = two_sided[:, :half:-1]  # bins nfft-1 ... half+1 fold onto 1 ... (half-1 for even nfft, half for odd)
    fb[:, 1 : 1 + mirror.shape[1]] += mirror
    return fb


def psf_filterbank(fs, nfft, nfilt=26, lowfreq=0.0, highfreq=None):
    highfreq = highfreq or fs / 2.0
    pts = np.floor((nfft + 1) * _imel(np.linspace(_mel(lowfreq), _mel(highfreq), nfilt + 2)) / fs).astype(int)
    fb = np.zeros((nfilt, nfft // 2 + 1))
    k = np.arange(nfft // 2 + 1)
    for m in range(nfilt):
        a, b, c = pts[m : m + 3]
        up = (k >= a) & (k < b)
        dn = (k >= b) & (k < c)
        fb[m, up] = (k[up] - a) / max(b - a, 1)
        fb[m, dn] = (c - k[dn]) / max(c - b, 1)
    return fb


def dct_rows(n_out: int, n_in: int, first: int = 0) -> np.ndarray:
    k = np.arange(first, first + n_out, dtype=np.float64)[:, None]
    n = np.arange(n_in, dtype=np.float64)[None, :]
    m = np.sqrt(2.0 / n_in) * np.cos(np.pi * k * (2.0 * n + 1.0) / (2.0 * n_in))
    m[k[:, 0] == 0] /= np.sqrt(2.0)
    return m


@dataclass
class Recipe:
    """Everything the kernel needs that is a convention rather than arithmetic."""
    name: str
    frame_len: int
    frame_shift: int
    nfft: int
    window: np.ndarray
    fbank: np.ndarray            # (n_filt, nfft/2+1)
    dct: np.ndarray              # (n_ceps, n_filt)
    framing: int = 0
    preemph_mode: int = 0
    preemph: float = 0.0
    spec_type: int = 0
    spec_scale: float = 1.0
    log_type: int = 0
    log_add: float = 0.0
    log_zero_floor: float = 0.0
    energy_mode: int = 0
    extra: dict = field(default_factory=dict)


def _pow2_at_least(n: int) -> int:
    return 1 << int(math.ceil(math.log2(n)))


def sidekit_recipe(lowfreq=100, maxfreq=8000, nlinfilt=0, nlogfilt=24, nwin=0.025, fs=16000, nceps=13, shift=0.01,
                   prefac=0.97) -> Recipe:
    """SIDEKIT 1.3 ``mfcc`` defaults (the function GMM_UBM.py:89 calls; parity unpinned, SURVEY 8(c))."""
    if nlinfilt != 0:
        raise NotImplementedError("nlinfilt != 0 is not supported")
    flen, hop = int(round(nwin * fs)), int(shift * fs)
    nfft = _pow2_at_least(flen)
    return Recipe("sidekit", flen, hop, nfft, np.hanning(flen), sidekit_filterbank(fs, nfft, lowfreq, maxfreq, nlogfilt),
                  dct_rows(nceps, nlogfilt, first=1), framing=0, preemph_mode=1, preemph=prefac, energy_mode=1)


def psf_recipe(samplerate=16000, winlen=0.025, winstep=0.01, numcep=13, nfilt=26, nfft=512, lowfreq=0, highfreq=None,
               preemph=0.97, ceplifter=22, appendEnergy=True) -> Recipe:
    """python_speech_features 0.6 ``mfcc`` defaults (BASELINE config 1's "26 mel"; parity unpinned)."""
    flen, hop = int(math.floor(winlen * samplerate + 0.5)), int(math.floor(winstep * samplerate + 0.5))
    d = dct_rows(numcep, nfilt)
    if ceplifter > 0:
        d = d * (1.0 + (ceplifter / 2.0) * np.sin(np.pi * np.arange(numcep) / ceplifter))[:, None]
    return Recipe("psf", flen, hop, nfft, np.ones(flen), psf_filterbank(samplerate, nfft, nfilt, lowfreq, highfreq), d,
                  framing=1, preemph_mode=2 if preemph else 0, preemph=preemph, spec_scale=1.0 / nfft,
                  log_zero_floor=float(np.finfo(float).eps), energy_mode=2 if appendEnergy else 0)


def _hz2bark(f):
    return 6.0 * np.arcsinh(np.asarray(f, dtype=np.float64) / 600.0)


def bark_filterbank(fs, nfft, nfilts=0, width=1.0, minfreq=0.0, maxfreq=None):
    """rastamat ``fft2barkmx`` (what SIDEKIT's ``plp`` -> ``audspec`` uses): (nfilts, nfft/2+1)."""
    maxfreq = fs / 2.0 if maxfreq is None else maxfreq
    min_bark = float(_hz2bark(minfreq))
    nyqbark = float(_hz2bark(maxfreq)) - min_bark
    if nfilts == 0:
        nfilts = int(math.ceil(nyqbark)) + 1
    step = nyqbark / (nfilts - 1)
    binbarks = _hz2bark(np.arange(nfft // 2 + 1) * fs / nfft)
    mid = min_bark + step * np.arange(nfilts)[:, None]
    lof, hif = binbarks[None, :] - mid - 0.5, binbarks[None, :] - mid + 0.5
    return 10.0 ** (np.minimum(0.0, np.minimum(hif, -2.5 * lof) / width))


def plp_recipe(nwin=0.025, fs=16000, plp_order=13, shift=0.01, prefac=0.97, rasta=True) -> Recipe:
    """SIDEKIT ``plp`` defaults (GMM_UBM.py:94-99; a port of rastamat ``rastaplp``; parity unpinned like ``mfcc``).
    The front-end kernel produces the critical-band energies (Bark filterbank, no log, identity "DCT"); the tables of
    the back half (``ssp_plp_post``) ride in ``extra``."""
    flen, hop = int(round(nwin * fs)), int(shift * fs)
    nfft = _pow2_at_least(flen)
    fb = bark_filterbank(fs, nfft)
    nb, nc = fb.shape[0], int(plp_order)
    cf = 600.0 * np.sinh(np.linspace(0.0, float(_hz2bark(fs / 2.0)), nb) / 6.0)
    fsq = cf ** 2
    eql = (fsq / (fsq + 1.6e5)) ** 2 * ((fsq + 1.44e6) / (fsq + 9.61e6))
    n = 2 * (nb - 1)
    k, i = np.arange(nc)[:, None], np.arange(nb)[None, :]
    idft = 2.0 * np.cos(2.0 * np.pi * k * i / n) / n
    idft[:, 0] = 1.0 / n
    idft[:, nb - 1] = ((-1.0) ** np.arange(nc)) / n
    lift = np.concatenate([[1.0], np.arange(1, nc, dtype=np.float64) ** 0.6])
    return Recipe("plp", flen, hop, nfft, np.hanning(flen), fb, np.eye(nb), framing=0, preemph_mode=1, preemph=prefac,
                  log_type=2, energy_mode=1, extra={"eql": eql, "idft": idft, "lift": lift, "rasta": bool(rasta), "n_ceps": nc})


def _slaney_mel(f):
    f = np.asarray(f, dtype=np.float64)
    return np.where(f >= 1000.0, 15.0 + np.log(np.maximum(f, 1000.0) / 1000.0) * (27.0 / math.log(6.4)), f * (3.0 / 200.0))


def _slaney_imel(m):
    m = np.asarray(m, dtype=np.float64)
    return np.where(m >= 15.0, 1000.0 * np.exp((math.log(6.4) / 27.0) * (m - 15.0)), m * (200.0 / 3.0))


def slaney_filterbank(sr, n_fft, n_mels=128, fmin=0.0, fmax=None):
    """``librosa.filters.mel`` defaults (Slaney mel scale, area-normalised triangles evaluated at the bin centres)."""
    fmax = sr / 2.0 if fmax is None else float(fmax)
    hz = np.arange(n_fft // 2 + 1) * (sr / float(n_fft))
    edges = _slaney_imel(np.linspace(_slaney_mel(fmin), _slaney_mel(fmax), n_mels + 2))
    fb = np.zeros((n_mels, n_fft // 2 + 1))
    for i in range(n_mels):
        lo, ce, hi = edges[i : i + 3]
        fb[i] = np.maximum(0.0, np.minimum((hz - lo) / (ce - lo), (hi - hz) / (hi - ce))) * (2.0 / (hi - lo))
    return fb


def librosa_recipe(sr=8000, n_mfcc=13, n_fft=2048, hop_length=512, n_mels=128, fmin=0.0, fmax=None, top_db=80.0,
                   center=True, pad_mode="reflect", amin=1e-10) -> Recipe:
    """``librosa.feature.mfcc(y, sr=8000, n_mfcc=13)`` as MFCC_DTW.py:27-30 calls it (parity unpinned: librosa is absent
    and un-pinned; SURVEY 8(c)).  The fused kernel produces the log-mel power in dB per frame (identity "DCT"); the
    utterance-wide ``top_db`` clip and the DCT (``ssp_mel_db_post``) ride in ``extra``."""
    if pad_mode not in ("reflect", "constant"):
        raise NotImplementedError(f"pad_mode {pad_mode!r} (reflect and constant are built)")
    n = int(n_fft)
    if not 64 <= n <= 4096:
        raise NotImplementedError("n_fft must lie in [64, 4096]")
    win = 0.5 - 0.5 * np.cos(2.0 * np.pi * np.arange(n) / n)  # periodic Hann (scipy get_window, fftbins=True)
    framing = (3 if pad_mode == "reflect" else 4) if center else 0
    return Recipe("librosa", n, int(hop_length), n, win, slaney_filterbank(sr, n, n_mels, fmin, fmax), np.eye(int(n_mels)),
                  framing=framing, log_type=3, log_zero_floor=float(amin),
                  extra={"dct": dct_rows(int(n_mfcc), int(n_mels)), "top_db": -1.0 if top_db is None else float(top_db),
                         "n_ceps": int(n_mfcc)})


def processing_recipe(fs=8000, frameSize=512, step=256) -> Recipe:
    """utils/processing.py:110-144 ``MFCC``: Hamming, no pre-emphasis (line 34 is commented out),
    magnitude/n spectrum, 40 talkbox triangles, log10(. + 1e-8), 13 cepstra incl. c0."""
    n = int(frameSize)
    if not 64 <= n <= 4096:
        raise NotImplementedError("frameSize (= FFT length at utils/processing.py:129) must lie in [64, 4096]")
    k = np.arange(n)
    ham = 0.54 - 0.46 * np.cos(2.0 * np.pi * k / (n - 1))
    return Recipe("processing", n, int(step), n, ham, processing_filterbank(fs, n), dct_rows(13, 40), framing=2,
                  spec_type=1, spec_scale=1.0 / n, log_type=1, log_add=1e-8)


# --------------------------------------------------------------------------------------------
# device-side front-end object
# --------------------------------------------------------------------------------------------


class FrontEnd:
    """A recipe uploaded to the GPU.  ``extract`` runs the fused kernel on a batch of utterances."""

    def __init__(self, recipe: Recipe, delta_order: int = 0, delta_n: int = 2, cmvn: bool = False, device=None):
        torch = _lib.require_cuda()
        self.lib = _lib.load()
        self.recipe = recipe
        self.delta_order, self.delta_n, self.cmvn = int(delta_order), int(delta_n), bool(cmvn)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.index is None:   # "cuda": the current device, named, so that tensors on it compare equal
            self.device = torch.device("cuda", torch.cuda.current_device())
        fb = np.asarray(recipe.fbank, dtype=np.float64)
        if fb.shape[1] != recipe.nfft // 2 + 1:
            raise ValueError("filterbank must have nfft/2+1 columns")
        starts, lens, offs, weights = [], [], [], []
        for row in fb:
            nz = np.nonzero(row)[0]
            s, e = (int(nz[0]), int(nz[-1]) + 1) if nz.size else (0, 0)
            starts.append(s)
            lens.append(e - s)
            offs.append(sum(len(w) for w in weights))
            weights.append(row[s:e])
        wcat = np.concatenate(weights) if weights and sum(lens) else np.zeros(1)

        def up(a, dt):
            return torch.as_tensor(np.ascontiguousarray(a, dtype=dt), device=self.device)

        self.t_window = up(recipe.window, np.float32)
        self.t_fb_start, self.t_fb_len, self.t_fb_off = up(starts, np.int32), up(lens, np.int32), up(offs, np.int32)
        self.t_fb_w = up(wcat, np.float32)
        self.t_dct = up(recipe.dct, np.float32)
        self.n_ceps = int(recipe.dct.shape[0])
        self.out_dim = self.n_ceps * (1 + self.delta_order)

    def _cfg(self, pcm_dtype: int) -> _lib.FrontendCfg:
        r = self.recipe
        return _lib.FrontendCfg(r.frame_len, r.frame_shift, r.nfft, r.fbank.shape[0], self.n_ceps, r.framing,
                                r.preemph_mode, r.preemph, r.spec_type, r.spec_scale, r.log_type, r.log_add,
                                r.log_zero_floor, r.energy_mode, self.delta_order, self.delta_n, int(self.cmvn), pcm_dtype)

    def num_frames(self, n_samples: int) -> int:
        cfg = self._cfg(0)
        return int(self.lib.ssp_frontend_num_frames(C.byref(cfg), int(n_samples)))

    def frame_counts(self, lens) -> np.ndarray:
        """Frames per utterance for an array of sample counts (the rule of ``ssp_frontend_num_frames``, vectorised)."""
        r = self.recipe
        lens = np.asarray(lens, dtype=np.int64)
        if r.framing == 0:
            nfr = np.where(lens < r.frame_len, 0, (lens - r.frame_len) // r.frame_shift + 1)
        elif r.framing == 1:
            nfr = np.where(lens <= r.frame_len, 1, 1 + -(-(lens - r.frame_len) // r.frame_shift))
        elif r.framing == 2:
            nfr = -(-lens // r.frame_shift)
        else:
            nfr = 1 + lens // r.frame_shift
        return np.where(lens <= 0, 0, nfr).astype(np.int64)

    # -- host entry: list of 1-D numpy signals -----------------------------------------------
    def pack_host(self, signals):
        """Concatenate utterances into one pinned host buffer + offsets (int16 stays int16).  A
        :class:`~speech_signal_processing_b200.wavio.PcmBatch` (``read_wav_batch``) already is one: no copy."""
        torch = _lib.require_cuda()
        from .wavio import PcmBatch

        if isinstance(signals, PcmBatch):
            pcm = signals.pcm if isinstance(signals.pcm, torch.Tensor) else torch.from_numpy(signals.pcm)
            return pcm, np.asarray(signals.sample_offsets, dtype=np.int64)
        sigs = [np.asarray(s) for s in signals]
        for s in sigs:
            if s.ndim != 1:
                raise ValueError("each utterance must be a 1-D array of samples")
        all_i16 = all(s.dtype == np.int16 for s in sigs)
        dt = np.int16 if all_i16 else np.float32
        lens = np.array([len(s) for s in sigs], dtype=np.int64)
        offs = np.zeros(len(sigs) + 1, dtype=np.int64)
        np.cumsum(lens, out=offs[1:])
        host = torch.empty(int(offs[-1]), dtype=torch.int16 if all_i16 else torch.float32, pin_memory=True)
        hv = host.numpy()
        for s, o in zip(sigs, offs[:-1]):
            hv[o : o + len(s)] = s.astype(dt, copy=False)
        return host, offs

    @_lib.on_device
    def extract(self, signals, want_log_energy: bool = False):
        """signals: list of 1-D arrays, or a PcmBatch.  Returns (feats (sum T, out_dim) cuda float32,
        frame_offsets np.int64 (n+1,), log_energy cuda float32 | None)."""
        host, offs = self.pack_host(signals)
        pcm = host.to(self.device, non_blocking=True)
        return self.extract_device(pcm, offs, want_log_energy)

    # -- device entry: PCM already resident in HBM --------------------------------------------
    @_lib.on_device
    def extract_device(self, pcm, sample_offsets: np.ndarray, want_log_energy: bool = False, out=None):
        """``pcm``: 1-D contiguous int16 / float32 tensor on ``self.device``; ``sample_offsets``: 1-D integer host array,
        never decreasing, within ``[0, len(pcm)]`` (it need not start at 0); ``out``: ``(total frames, out_dim)``
        contiguous float32 on the device, or None.  Anything else raises before a launch (a PCM dtype other than int16 /
        float32 is a ``TypeError``, the rest ``ValueError``): the kernel reads ``pcm`` as packed samples and writes
        ``out`` as packed rows."""
        torch = _lib.require_cuda()
        if pcm.dtype == torch.int16:
            pcm_dtype = 0
        elif pcm.dtype == torch.float32:
            pcm_dtype = 1
        else:
            raise TypeError("PCM must be int16 or float32")
        if pcm.dim() != 1 or not pcm.is_contiguous() or pcm.device != self.device:
            raise ValueError(f"PCM must be a 1-D contiguous tensor on {self.device} (got {pcm.dim()}-D, stride "
                             f"{tuple(pcm.stride())}, on {pcm.device})")
        cfg = self._cfg(pcm_dtype)
        sample_offsets = np.asarray(sample_offsets)
        if sample_offsets.ndim != 1 or sample_offsets.dtype.kind not in "iu" or len(sample_offsets) == 0:
            raise ValueError("sample_offsets must be a non-empty 1-D integer array")
        sample_offsets = sample_offsets.astype(np.int64, copy=False)
        if sample_offsets[0] < 0 or sample_offsets[-1] > pcm.shape[0] or np.any(sample_offsets[1:] < sample_offsets[:-1]):
            raise ValueError(f"sample_offsets must never decrease and stay within [0, {pcm.shape[0]}] (the PCM's samples)")
        n_utts = len(sample_offsets) - 1
        r = self.recipe
        nfr = self.frame_counts(np.diff(sample_offsets))
        frame_offsets = np.zeros(n_utts + 1, dtype=np.int64)
        np.cumsum(nfr, out=frame_offsets[1:])
        total = int(frame_offsets[-1])
        if out is None:
            out = torch.empty((total, self.out_dim), dtype=torch.float32, device=self.device)
        elif (tuple(out.shape) != (total, self.out_dim) or out.dtype != torch.float32 or not out.is_contiguous()
              or out.device != self.device):
            raise ValueError(f"out must be a contiguous ({total}, {self.out_dim}) float32 tensor on {self.device} (got "
                             f"{tuple(out.shape)} {out.dtype} on {out.device})")
        log_e = torch.empty(total, dtype=torch.float32, device=self.device) if want_log_energy else None
        if n_utts == 0 or total == 0:
            return out, frame_offsets, log_e
        max_fused = int(self.lib.ssp_frontend_max_frames(C.byref(cfg)))
        if int(nfr.max()) > max_fused and r.framing >= 3:
            raise NotImplementedError(f"centred framing: utterances beyond {max_fused} frames are not chunked")
        if int(nfr.max()) > max_fused:
            self._extract_mixed(pcm, pcm_dtype, sample_offsets, frame_offsets, nfr, max_fused, out, log_e)
            return out, frame_offsets, log_e
        d_soff = torch.as_tensor(sample_offsets, device=self.device)
        d_foff = torch.as_tensor(frame_offsets, device=self.device)
        rc = self.lib.ssp_frontend_batch(
            _lib.ptr(pcm), _lib.ptr(d_soff), n_utts, C.byref(cfg), _lib.ptr(self.t_window), _lib.ptr(self.t_fb_start),
            _lib.ptr(self.t_fb_len), _lib.ptr(self.t_fb_off), _lib.ptr(self.t_fb_w), _lib.ptr(self.t_dct),
            _lib.ptr(d_foff), int(nfr.max()), _lib.ptr(out), _lib.ptr(log_e), _lib.stream_ptr())
        _lib.check(rc, "ssp_frontend_batch")
        self._keep = (d_soff, d_foff)  # keep the offset tensors alive until the stream has consumed them
        return out, frame_offsets, log_e


    # -- utterances too long for the single-pass kernel (its per-utterance cepstra live in shared memory) ------------
    def _launch(self, pcm, cfg, soff, foff, max_t, out, log_e):
        torch = _lib.require_cuda()
        d_soff = torch.as_tensor(np.ascontiguousarray(soff, dtype=np.int64), device=self.device)
        d_foff = torch.as_tensor(np.ascontiguousarray(foff, dtype=np.int64), device=self.device)
        rc = self.lib.ssp_frontend_batch(
            _lib.ptr(pcm), _lib.ptr(d_soff), len(soff) - 1, C.byref(cfg), _lib.ptr(self.t_window), _lib.ptr(self.t_fb_start),
            _lib.ptr(self.t_fb_len), _lib.ptr(self.t_fb_off), _lib.ptr(self.t_fb_w), _lib.ptr(self.t_dct),
            _lib.ptr(d_foff), int(max_t), _lib.ptr(out), _lib.ptr(log_e), _lib.stream_ptr())
        _lib.check(rc, "ssp_frontend_batch")
        self._keep_long = getattr(self, "_keep_long", []) + [d_soff, d_foff]

    def _extract_mixed(self, pcm, pcm_dtype, soff, foff, nfr, max_fused, out, log_e):
        """Batch with utterances longer than the fused kernel's shared-memory bound (~35 s at 39-d).  Runs of short
        utterances go through the fused kernel unchanged.  A long utterance is cut into chunks of whole frames that
        the kernel turns into raw cepstra (each chunk a "virtual utterance"; frames are self-contained), then
        ``ssp_delta`` (once or twice) and ``ssp_cmvn`` run over the whole utterance -- three to five launches per
        long utterance instead of one."""
        torch = _lib.require_cuda()
        r = self.recipe
        self._keep_long = []
        long_ix = np.nonzero(nfr > max_fused)[0]
        cfg_full = self._cfg(pcm_dtype)
        # ---- runs of short utterances between the long ones
        edges = [-1] + [int(i) for i in long_ix] + [len(nfr)]
        for a, b in zip(edges[:-1], edges[1:]):
            lo, hi = a + 1, b
            if hi > lo and int(nfr[lo:hi].sum()) > 0:
                self._launch(pcm, cfg_full, soff[lo : hi + 1], foff[lo : hi + 1], int(nfr[lo:hi].max()), out, log_e)
        # ---- long utterances
        raw = FrontEnd.__new__(FrontEnd)
        raw.__dict__.update(self.__dict__)
        raw.delta_order, raw.cmvn = 0, False
        nc = self.n_ceps
        for u in long_ix:
            t = int(nfr[u])
            src, mode_cfg = pcm, raw._cfg(pcm_dtype)
            s0 = int(soff[u])
            if r.preemph_mode == 2:
                # whole-signal pre-emphasis crosses chunk borders: apply it up front (y[0] = x[0]) and switch it off
                x = pcm[s0 : int(soff[u + 1])].to(torch.float32)
                y = x.clone()
                y[1:] -= r.preemph * x[:-1]
                src, s0 = y, 0
                mode_cfg = raw._cfg(1)
                mode_cfg.preemph_mode = 0
            n_samp = int(soff[u + 1] - soff[u])
            chunk = int(self.lib.ssp_frontend_max_frames(C.byref(mode_cfg)))
            chunk = max(1, min(chunk, 2048))
            f_lo = np.arange(0, t, chunk, dtype=np.int64)
            f_hi = np.minimum(f_lo + chunk, t)
            c_soff = np.concatenate([s0 + f_lo * r.frame_shift, [0]])
            # every chunk but the last ends with its last frame; sample_offsets must be non-decreasing pairs, so each
            # chunk gets its own (start, end) pair through a two-entry offsets array per launch group
            ceps = torch.empty((t, nc), dtype=torch.float32, device=self.device)
            le = torch.empty(t, dtype=torch.float32, device=self.device) if log_e is not None else None
            for k in range(len(f_lo)):
                start = int(c_soff[k])
                last = k == len(f_lo) - 1
                stop = s0 + n_samp if last else start + int(f_hi[k] - f_lo[k] - 1) * r.frame_shift + r.frame_len
                self._launch(src, mode_cfg, np.array([start, min(stop, s0 + n_samp)]), np.array([0, int(f_hi[k] - f_lo[k])]),
                             int(f_hi[k] - f_lo[k]), ceps[int(f_lo[k]) :], le[int(f_lo[k]) :] if le is not None else None)
            cols = [ceps]
            for _ in range(self.delta_order):
                d = torch.empty_like(ceps)
                _lib.check(self.lib.ssp_delta(_lib.ptr(cols[-1]), t, nc, self.delta_n, _lib.ptr(d), _lib.stream_ptr()), "ssp_delta")
                cols.append(d)
            feats = torch.cat(cols, dim=1) if len(cols) > 1 else ceps
            dst = out[int(foff[u]) : int(foff[u + 1])]
            if self.cmvn:
                offs = torch.tensor([0, t], dtype=torch.int64, device=self.device)
                _lib.check(self.lib.ssp_cmvn(_lib.ptr(feats), _lib.ptr(offs), 1, feats.shape[1], _lib.ptr(dst), _lib.stream_ptr()), "ssp_cmvn")
                self._keep_long.append(offs)
            else:
                dst.copy_(feats)
            if log_e is not None:
                log_e[int(foff[u]) : int(foff[u + 1])].copy_(le)
            self._keep_long += [ceps, feats, src]


_FRONTENDS: dict = {}


def _cached(key, make):
    """Front-ends of the numpy drop-ins, one per (parameters, CURRENT device): the tables live on a device."""
    torch = _lib.require_cuda()
    key = (key, torch.cuda.current_device())
    fe = _FRONTENDS.get(key)
    if fe is None:
        fe = _FRONTENDS[key] = make()
    return fe


# --------------------------------------------------------------------------------------------
# drop-ins with the reference's signatures (numpy in, numpy out)
# --------------------------------------------------------------------------------------------


def mfcc(input_sig, lowfreq=100, maxfreq=8000, nlinfilt=0, nlogfilt=24, nwin=0.025, fs=16000, nceps=13, shift=0.01,
         get_spec=False, get_mspec=False, prefac=0.97):
    """``sidekit.frontend.features.mfcc`` (GMM_UBM.py:20,89): ``[ceps (T,nceps), log_energy (T,), None, None]``."""
    if get_spec or get_mspec:
        raise NotImplementedError("get_spec / get_mspec are not produced by the fused kernel")
    key = ("sidekit", lowfreq, maxfreq, nlinfilt, nlogfilt, nwin, fs, nceps, shift, prefac)
    fe = _cached(key, lambda: FrontEnd(sidekit_recipe(lowfreq, maxfreq, nlinfilt, nlogfilt, nwin, fs, nceps, shift, prefac)))
    feats, _, log_e = fe.extract([np.asarray(input_sig)], want_log_energy=True)
    return [feats.cpu().numpy(), log_e.cpu().numpy(), None, None]


class PlpFrontEnd:
    """PLP cepstra for a batch of utterances: the fused kernel up to the critical-band energies, ``ssp_plp_post`` for
    RASTA / equal loudness / LPC / cepstra, then (optionally) ``ssp_delta`` per utterance and ``ssp_cmvn``."""

    def __init__(self, recipe: Recipe | None = None, delta_order: int = 0, delta_n: int = 2, cmvn: bool = False, device=None):
        torch = _lib.require_cuda()
        self.recipe = recipe or plp_recipe()
        self.bands = FrontEnd(self.recipe, delta_order=0, cmvn=False, device=device)
        self.device, self.lib = self.bands.device, self.bands.lib
        ex = self.recipe.extra
        self.n_ceps = int(ex["n_ceps"])
        self.delta_order, self.delta_n, self.cmvn = int(delta_order), int(delta_n), bool(cmvn)
        self.out_dim = self.n_ceps * (1 + self.delta_order)
        up = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=self.device)  # noqa: E731
        self.t_eql, self.t_idft, self.t_lift = up(ex["eql"]), up(ex["idft"]), up(ex["lift"])

    @_lib.on_device
    def extract(self, signals, want_log_energy: bool = False):
        """Returns (feats (sum T, out_dim) cuda float32, frame_offsets np.int64, log_energy | None)."""
        torch = _lib.require_cuda()
        bands, offs, log_e = self.bands.extract(signals, want_log_energy)
        total, nb = int(offs[-1]), bands.shape[1]
        ceps = torch.empty((total, self.n_ceps), dtype=torch.float32, device=self.device)
        d_off = torch.as_tensor(offs, device=self.device)
        if total:
            _lib.check(self.lib.ssp_plp_post(_lib.ptr(bands), _lib.ptr(d_off), len(offs) - 1, nb, self.n_ceps, _lib.ptr(self.t_eql),
                                             _lib.ptr(self.t_idft), _lib.ptr(self.t_lift), int(self.recipe.extra["rasta"]),
                                             _lib.ptr(ceps), _lib.stream_ptr()), "ssp_plp_post")
        feats = ceps
        if self.delta_order and total:
            cols = [ceps]
            for _ in range(self.delta_order):
                d = torch.empty_like(ceps)
                for u in range(len(offs) - 1):  # GMM_UBM.delta pads at the utterance edges: one launch per utterance
                    lo, hi = int(offs[u]), int(offs[u + 1])
                    if hi > lo:
                        _lib.check(self.lib.ssp_delta(_lib.ptr(cols[-1][lo:]), hi - lo, self.n_ceps, self.delta_n, _lib.ptr(d[lo:]),
                                                      _lib.stream_ptr()), "ssp_delta")
                cols.append(d)
            feats = torch.cat(cols, dim=1)
        if self.cmvn and total:
            out = torch.empty_like(feats)
            _lib.check(self.lib.ssp_cmvn(_lib.ptr(feats), _lib.ptr(d_off), len(offs) - 1, feats.shape[1], _lib.ptr(out),
                                         _lib.stream_ptr()), "ssp_cmvn")
            feats = out
        self._keep = (d_off, bands, ceps)
        return feats, offs, log_e


class MelDbFrontEnd:
    """librosa-convention MFCC for a batch of utterances: the fused kernel up to the log-mel power in dB,
    ``ssp_mel_db_post`` for the utterance-wide ``top_db`` clip and the DCT."""

    def __init__(self, recipe: Recipe | None = None, device=None):
        torch = _lib.require_cuda()
        self.recipe = recipe or librosa_recipe()
        self.bands = FrontEnd(self.recipe, delta_order=0, cmvn=False, device=device)
        self.device, self.lib = self.bands.device, self.bands.lib
        ex = self.recipe.extra
        self.n_ceps = self.out_dim = int(ex["n_ceps"])
        self.top_db = float(ex["top_db"])
        self.t_dct = torch.as_tensor(np.ascontiguousarray(ex["dct"], dtype=np.float32), device=self.device)

    @_lib.on_device
    def extract(self, signals):
        """Returns (ceps (sum T, n_mfcc) cuda float32, frame_offsets np.int64)."""
        torch = _lib.require_cuda()
        mel_db, offs, _ = self.bands.extract(signals)
        total, nm = int(offs[-1]), mel_db.shape[1]
        ceps = torch.empty((total, self.n_ceps), dtype=torch.float32, device=self.device)
        d_off = torch.as_tensor(offs, device=self.device)
        if total:
            _lib.check(self.lib.ssp_mel_db_post(_lib.ptr(mel_db), _lib.ptr(d_off), len(offs) - 1, nm, self.n_ceps,
                                                _lib.ptr(self.t_dct), self.top_db, _lib.ptr(ceps), _lib.stream_ptr()),
                       "ssp_mel_db_post")
        self._keep = (d_off, mel_db)
        return ceps, offs


def librosa_mfcc(y, sr=8000, n_mfcc=13, **kwargs):
    """``librosa.feature.mfcc(y, sr=sr, n_mfcc=n_mfcc, ...)`` (MFCC_DTW.py:28): (n_mfcc, T) float32."""
    key = ("librosa", sr, n_mfcc, tuple(sorted(kwargs.items())))
    fe = _cached(key, lambda: MelDbFrontEnd(librosa_recipe(sr=sr, n_mfcc=n_mfcc, **kwargs)))
    ceps, _ = fe.extract([np.asarray(y, dtype=np.float32)])
    return np.ascontiguousarray(ceps.cpu().numpy().T)


def MFCC_lib(raw_signal, n_mfcc=13):
    """``MFCC_DTW.MFCC_lib`` (MFCC_DTW.py:27-30): librosa MFCC at sr=8000, frame-major, flattened."""
    return librosa_mfcc(np.asarray(raw_signal).astype("float32"), sr=8000, n_mfcc=n_mfcc).T.flatten()


def plp(input_sig, nwin=0.025, fs=16000, plp_order=13, shift=0.01, get_spec=False, get_mspec=False, prefac=0.97, rasta=True):
    """``sidekit.frontend.features.plp`` (GMM_UBM.py:20,94): ``[ceps (T, plp_order), log_energy (T,), None, None]``."""
    if get_spec or get_mspec:
        raise NotImplementedError("get_spec / get_mspec are not produced by the fused kernel")
    key = ("plp", nwin, fs, plp_order, shift, prefac, rasta)
    fe = _cached(key, lambda: PlpFrontEnd(plp_recipe(nwin, fs, plp_order, shift, prefac, rasta)))
    feats, _, log_e = fe.extract([np.asarray(input_sig)], want_log_energy=True)
    return [feats.cpu().numpy(), log_e.cpu().numpy(), None, None]


def MFCC(raw_signal, fs=8000, frameSize=512, step=256):
    """``utils.processing.MFCC`` (utils/processing.py:110-144): (ceil(N/step), 13) float64."""
    fe = _cached(("processing", fs, frameSize, step), lambda: FrontEnd(processing_recipe(fs, frameSize, step)))
    feats, _, _ = fe.extract([np.asarray(raw_signal)])
    return feats.cpu().numpy().astype(np.float64)


def delta(feat, N=2):
    """``GMM_UBM.delta`` (GMM_UBM.py:53-69)."""
    if N < 1:
        raise ValueError("N must be an integer >= 1")
    torch = _lib.require_cuda()
    feat = np.asarray(feat)
    x = torch.as_tensor(np.ascontiguousarray(feat, dtype=np.float32), device="cuda")
    out = torch.empty_like(x)
    if x.numel():
        _lib.check(_lib.load().ssp_delta(_lib.ptr(x), x.shape[0], x.shape[1], int(N), _lib.ptr(out), _lib.stream_ptr()),
                   "ssp_delta")
    return out.cpu().numpy().astype(feat.dtype if feat.dtype.kind == "f" else np.float64)


def scale(X):
    """``sklearn.preprocessing.scale(X)`` as called at GMM_UBM.py:93 (axis 0, ddof 0, zero std -> 1)."""
    torch = _lib.require_cuda()
    X = np.asarray(X)
    x = torch.as_tensor(np.ascontiguousarray(X, dtype=np.float32), device="cuda")
    out = torch.empty_like(x)
    offs = torch.tensor([0, x.shape[0]], dtype=torch.int64, device="cuda")
    if x.numel():
        _lib.check(_lib.load().ssp_cmvn(_lib.ptr(x), _lib.ptr(offs), 1, x.shape[1], _lib.ptr(out), _lib.stream_ptr()), "ssp_cmvn")
    return out.cpu().numpy().astype(X.dtype if X.dtype.kind == "f" else np.float64)


class _Preprocessing:
    """Stand-in for the ``sklearn.preprocessing`` module name bound at GMM_UBM.py:18."""
    scale = staticmethod(scale)


preprocessing = _Preprocessing()


def extract_feature(x, y, is_train=False, feature_type="MFCC", delta_order=1, recipe: Recipe | None = None):
    """``GMM_UBM.extract_feature`` (GMM_UBM.py:72-118) for the whole list in one launch.

    Returns ``(train_data, feature, y)`` if ``is_train`` else ``(feature, y)`` exactly like the
    reference: ``feature`` is a list of (T, 26) arrays (cepstra + delta, CMVN per utterance),
    ``train_data[label]`` their per-speaker vertical stack.  ``delta_order=2`` gives the 39-d
    north-star features.
    """
    # only the default recipes are cached; a caller's Recipe object gets a fresh front-end (caching under id(recipe)
    # would hand a recycled id the stale tables)
    if feature_type == "PLP":      # GMM_UBM.py:94-99
        make = lambda: PlpFrontEnd(recipe, delta_order=delta_order, delta_n=2, cmvn=True)  # noqa: E731
        fe = make() if recipe is not None else _cached(("xf-plp", delta_order, 2), make)
    elif feature_type == "MFCC":
        make = lambda: FrontEnd(recipe or sidekit_recipe(), delta_order=delta_order, delta_n=2, cmvn=True)  # noqa: E731
        fe = make() if recipe is not None else _cached(("xf-sidekit", delta_order, 2), make)
    else:
        raise NameError(feature_type)  # GMM_UBM.py:100-101
    feats, offs, _ = fe.extract(list(x))
    host = feats.cpu().numpy()
    feature = [host[offs[i] : offs[i + 1]] for i in range(len(x))]
    if not is_train:
        return feature, y
    train_data = {}
    order = {}
    for i, lab in enumerate(y):
        order.setdefault(lab, []).append(i)
    for lab, idx in order.items():
        train_data[lab] = np.vstack([feature[i] for i in idx])
    return train_data, feature, y
