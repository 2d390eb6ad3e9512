"""GMM-UBM speaker identification: UBM training, MAP enrolment, batched scoring, and the
reference's ``GMM()`` entry point.

* :func:`GMM` has the signature and printed output of ``GMM_UBM.GMM`` (GMM_UBM.py:134-199): one
  GMM per speaker + a UBM on the pooled frames, ``pred[j, i] = GMM[i].score(x_j) - UBM.score(x_j)``,
  argmax accuracy, models pickled under ``Model/`` as stock sklearn estimators.
* :func:`map_adapt` is the enrolment the reference's report describes but its code never does
  (SURVEY F4): relevance MAP of the UBM from per-speaker statistics, all speakers in one launch.
* :func:`identify` scores every test utterance against every speaker model (+ the UBM) in one
  kernel launch and returns the LLR matrix and the argmax decisions (GMM_UBM.py:191-197).
* :func:`install` rebinds the module-level names of an imported ``GMM_UBM`` module
  (GMM_UBM.py:16-20) to this package, which is the whole integration.
"""
from __future__ import annotations

import os
import pickle as pkl
import time

import numpy as np

from . import _lib
from . import frontend as fe
from .wavio import read_wav_batch
from .mixture import (SINGLE_PASS_MIN_COMPONENTS, GaussianMixture, ModelSet, SharedModelSet, check_top_c, concat_utterances,
                      fit_batch, resolve_precision, stacked_params)


def map_adapt(ubm: GaussianMixture, speaker_frames, relevance: float = 16.0, adapt=("means",), device=None):
    """Enrol speakers by relevance MAP (Reynolds, Quatieri & Dunn 2000, eq. 11-14).

    ``speaker_frames``: list (one entry per speaker) of (T_s, D) arrays, or ``(feats, seg_offsets)``
    already on the GPU.  Returns ``(weights (S,K), means (S,K,D), variances (S,K,D))`` as float64
    CUDA tensors, ready for :class:`ModelSet`.
    """
    torch = _lib.require_cuda()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    feats, seg = concat_utterances(speaker_frames, dev)
    ms = ubm._model_set()
    n, f, s, _ = ms.stats(feats, seg)
    n_spk, k, d = len(seg) - 1, ms.n_comp, ms.n_feat
    flags = (1 if "means" in adapt else 0) | (2 if "weights" in adapt else 0) | (4 if "variances" in adapt else 0)
    ow = torch.empty((n_spk, k), dtype=torch.float64, device=dev)
    omu = torch.empty((n_spk, k, d), dtype=torch.float64, device=dev)
    ovar = torch.empty((n_spk, k, d), dtype=torch.float64, device=dev)
    uw, umu, uvar = ms._params
    d_seg = torch.as_tensor(seg, device=dev)
    rc = ms.lib.ssp_gmm_map_adapt(_lib.ptr(n), _lib.ptr(f), _lib.ptr(s), _lib.ptr(d_seg), n_spk, _lib.ptr(uw), _lib.ptr(umu),
                                  _lib.ptr(uvar), k, d, float(relevance), flags, _lib.ptr(ow), _lib.ptr(omu), _lib.ptr(ovar),
                                  _lib.stream_ptr())
    _lib.check(rc, "ssp_gmm_map_adapt")
    torch.cuda.current_stream().synchronize()
    return ow, omu, ovar


def map_enrol(ubm: GaussianMixture, speaker_frames, relevance: float = 16.0, adapt=("means",), device=None):
    """MAP enrolment straight into a model set that carries the UBM as model S (``ubm_index``).

    The default, mean-only enrolment gives the form the shared-variance scoring kernel wants: a :class:`SharedModelSet`
    of the S adapted mean sets plus the UBM's own means, all with the UBM's weights and variances.
    ``identify(utts, map_enrol(...))`` then gives the LLR matrix of GMM_UBM.py:191-197 with one kernel launch and a
    per-speaker contraction of D + 2 instead of 2D + 2.  An ``adapt`` that includes ``"weights"`` or ``"variances"``
    gives ``ModelSet.with_ubm(*map_adapt(...), ubm)``: the general scoring kernel, and top-C scoring through
    :meth:`ModelSet.score_top_c`."""
    torch = _lib.require_cuda()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    if "weights" in adapt or "variances" in adapt:
        return ModelSet.with_ubm(*map_adapt(ubm, speaker_frames, relevance=relevance, adapt=adapt, device=dev), ubm, device=dev)
    _, mu, _ = map_adapt(ubm, speaker_frames, relevance=relevance, adapt=("means",), device=dev)
    uw, umu, uvar = ubm._model_set()._params
    return SharedModelSet.with_ubm(uw[0], uvar[0], mu, umu, device=dev)


def _base_params(model):
    """(weights (K,), variances (K, D)) of a fitted GaussianMixture-like or a single-model ModelSet as numpy, else None."""
    if isinstance(model, ModelSet):
        if model.n_models != 1:
            return None
        w, _, var = model._params
        return w[0].cpu().numpy(), var[0].cpu().numpy()
    return np.asarray(model.weights_), np.asarray(model.covariances_)


def _shares_base(weights, variances, ubm=None) -> bool:
    """True if every speaker of the (S,K) / (S,K,D) numpy stacks carries the same weights and variances -- and, given a
    ``ubm``, those are KNOWN to be the UBM's (mean-only MAP models adapted from it)."""
    if not SharedModelSet.shares_base(weights, variances):
        return False
    if ubm is None:
        return True
    base = _base_params(ubm)
    return base is not None and np.array_equal(base[0], weights[0]) and np.array_equal(base[1], variances[0])


def _ubm_means(ubm):
    return ubm._params[1] if isinstance(ubm, ModelSet) else np.asarray(ubm.means_)


def _llr(scores, k):
    """(pred (N, S) numpy, argmax (N,)) from the scores of a set whose column ``k`` is the UBM: every other column minus
    column ``k``."""
    keep = [i for i in range(scores.shape[1]) if i != k]
    pred = (scores[:, keep] - scores[:, k : k + 1]).cpu().numpy()
    return pred, pred.argmax(axis=1)


def _top_c_set(speakers, ubm, dev):
    """(set that selects by its UBM member, column of the UBM) for top-C scoring: a :class:`ModelSet` from
    :meth:`ModelSet.with_ubm` (speakers adapted in weights and variances too) or a :class:`SharedModelSet` whose
    reference member is the UBM; or the refusal: no UBM is a ``ValueError``, speakers that do not share the UBM's weights
    and variances a ``NotImplementedError``."""
    if isinstance(speakers, ModelSet) and speakers.ubm_index is not None and ubm is None:
        return speakers, speakers.ubm_index
    if isinstance(speakers, SharedModelSet) and ubm is None:
        k = getattr(speakers, "ubm_index", None)
        if k is None:
            raise ValueError("top_c scores against a UBM: pass ubm=, or a SharedModelSet from map_enrol")
        if k != speakers.ref_model:
            raise NotImplementedError("top_c selects by the reference member of the set, which must be its UBM "
                                      f"(ref_model {speakers.ref_model}, ubm_index {k})")
        return speakers, k
    if ubm is None:
        raise ValueError("top_c scores against a UBM: pass ubm=, or a SharedModelSet from map_enrol")
    if isinstance(ubm, ModelSet) and ubm.n_models != 1:
        raise ValueError("ubm must be ONE model")
    if isinstance(speakers, SharedModelSet):
        w, var, mu = (t.cpu().numpy() for t in speakers._params)
        sw, svar, smu = w[None], var[None], mu
    elif isinstance(speakers, ModelSet):
        sw, smu, svar = (t.cpu().numpy() for t in speakers._params)
    else:
        sw, smu, svar = stacked_params(speakers)
    if not _shares_base(sw, svar, ubm):
        raise NotImplementedError("top_c needs speaker models that share the UBM's weights and variances (mean-only MAP "
                                  "enrolment): there is no component correspondence otherwise")
    sms = SharedModelSet.with_ubm(sw[0], svar[0], smu, _ubm_means(ubm), device=dev)
    return sms, sms.ubm_index


def _exact_set(speakers, ubm, precision, dev):
    """(model set that scores ``speakers`` exactly at ``precision``, column of the UBM in it or None -- then the UBM, if
    any, is scored on its own)."""
    if isinstance(speakers, (SharedModelSet, ModelSet)) and getattr(speakers, "ubm_index", None) is not None and ubm is None:
        return speakers, speakers.ubm_index   # map_enrol / with_ubm: the UBM rides along as one of the models
    if isinstance(speakers, SharedModelSet):
        return (speakers if precision in ("tf32", "auto") else speakers.expand()), None
    if isinstance(speakers, ModelSet):
        return speakers, None
    sw, smu, svar = stacked_params(speakers)
    single_pass = precision == "tf32" or (precision == "auto" and sw.shape[1] >= SINGLE_PASS_MIN_COMPONENTS)
    # mean-only MAP speakers (e.g. unpickled models adapted from this UBM): shared-variance kernel, with the UBM as one
    # more mean set
    if single_pass and smu.shape[2] <= 39 and _shares_base(sw, svar, ubm):
        try:
            if ubm is None:
                return SharedModelSet(sw[0], svar[0], smu, device=dev), None
            sms = SharedModelSet.with_ubm(sw[0], svar[0], smu, _ubm_means(ubm), device=dev)
            return sms, sms.ubm_index
        except NotImplementedError:   # parameters outside the FP16 range of that kernel: general kernel below
            pass
    return ModelSet(sw, smu, svar, device=dev), None


def identify(utts, speakers, ubm=None, precision="auto", device=None, top_c=None):
    """LLR matrix and decisions for all (utterance, speaker) pairs (GMM_UBM.py:191-197).

    ``speakers``: :class:`ModelSet` / :class:`SharedModelSet`, or list of fitted GaussianMixture-likes.  ``ubm``: fitted
    GaussianMixture-like, single-model :class:`ModelSet`, or None.  Returns ``(pred (N,S) float64 numpy, argmax (N,)
    int64)``; ``pred`` is always the LLR ``speaker score - UBM score`` when a UBM is given, whichever kernel serves the
    call.  The UBM term is constant per utterance, so decisions depend on the speaker scores only (SURVEY F9); it is
    evaluated ONCE per utterance, not once per speaker.  A set with a ``ubm_index`` (:func:`map_enrol`,
    :meth:`ModelSet.with_ubm`) given without ``ubm`` carries its UBM: it is scored in the same launch as the speakers and
    ``pred`` is the LLR against it.

    ``precision``: "auto" (default) keeps every LLR within 1e-3 absolute of float64: one TF32 pass for models of
    >= 512 components (mean-only MAP sets then go through the shared-variance kernel), three passes (FP32-grade) for
    smaller ones, FP32 CUDA cores for D > 39.  "tf32" forces the single pass, "tf32x2" / "tf32x3" / "fp32" the others.

    ``top_c``: None (default) scores exactly as above.  An integer C scores by top-C fast scoring
    (:meth:`SharedModelSet.score_top_c` / :meth:`ModelSet.score_top_c`, Reynolds et al. 2000): every frame under every
    speaker over the C components the UBM ranks highest for it, always at FP32 grade (``precision`` is ignored).  The
    speakers must be known to be adapted from the UBM: a :func:`map_enrol` set (any ``adapt``), a
    :meth:`ModelSet.with_ubm` set, or mean-only MAP models with a ``ubm`` of the same weights and variances
    (``NotImplementedError`` otherwise: a list of models whose weights or variances differ from the UBM's may have been
    trained independently, and then there is no component correspondence); without a UBM it is a ``ValueError``.
    """
    torch = _lib.require_cuda()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    with torch.cuda.device(dev):
        if top_c is not None:
            sms, k = _top_c_set(speakers, ubm, dev)
            check_top_c(top_c, sms.n_comp)
            feats, offs = concat_utterances(utts, dev)
            return _llr(sms.score_top_c(feats, offs, c=top_c)[0], k)
        feats, offs = concat_utterances(utts, dev)
        ms, k = _exact_set(speakers, ubm, precision, dev)
        if k is not None:   # one launch scores speakers and UBM (a SharedModelSet has its one precision rung)
            scores, _ = ms.score(feats, offs) if isinstance(ms, SharedModelSet) else ms.score(feats, offs, precision=precision)
            return _llr(scores, k)
        scores, _ = ms.score(feats, offs, precision=precision)
        if ubm is not None:
            ums = ubm if isinstance(ubm, ModelSet) else ModelSet(ubm.weights_, ubm.means_, ubm.covariances_, device=dev)
            if ums.n_models != 1:
                raise ValueError("ubm must be ONE model (got a ModelSet of %d)" % ums.n_models)
            # same rung as the speakers: the model-side rounding of a shared base then cancels in the LLR
            base_prec = resolve_precision(precision, ms.n_comp, ms.n_feat)
            ubm_score, _ = ums.score(feats, offs, precision=base_prec)
            scores = scores - ubm_score
        pred = scores.cpu().numpy()
        return pred, pred.argmax(axis=1)


# frames one wave of the persistent scoring kernels covers: 148 CTAs x 256-frame units
_WAVE_FRAMES = 148 * 256


def split_for_overlap(frame_counts, head_fraction: float = 0.1, min_frames: int = 4 * _WAVE_FRAMES) -> int:
    """Utterances in the head part of a two-part pipelined batch: about ``head_fraction`` of the frames, rounded to
    whole waves of the persistent scoring kernel so that cutting the batch does not add a partly filled wave.  0 means
    "do not split" (batch too small for the overlap to pay)."""
    cum = np.cumsum(np.asarray(frame_counts, dtype=np.int64))
    total = int(cum[-1]) if len(cum) else 0
    if total < min_frames or len(cum) < 2:
        return 0
    waves = max(1, int(round(head_fraction * total / _WAVE_FRAMES)))
    n = int(np.searchsorted(cum, waves * _WAVE_FRAMES, side="right"))
    if not 0 < n < len(cum):  # less than a wave or two in total: cut at the plain fraction
        n = int(np.searchsorted(cum, head_fraction * total, side="right"))
    return n if 0 < n < len(cum) else 0


def identify_pcm(host_pcm, sample_offsets, front_end, speakers, ubm_index=None, precision="auto", out=None,
                 head_fraction: float = 0.1, min_split_frames: int = 4 * _WAVE_FRAMES, top_c=None):
    """Raw PCM on the host -> speaker decisions on the host, for one batch of utterances: the front-end of
    GMM_UBM.py:129 and the scoring / argmax of :191-197 as one call.

    ``host_pcm``: 1-D int16 / float32 torch tensor (pinned memory makes the copies asynchronous) or numpy array with all
    utterances back to back; ``sample_offsets``: int64 (N+1,); ``front_end``: :class:`FrontEnd`; ``speakers``:
    :class:`ModelSet` / :class:`SharedModelSet`; ``ubm_index``: the model whose score is subtracted (and excluded from
    the argmax), or None.  The host-to-device copy is cut in two at an utterance boundary: the head (about a tenth of
    the frames, whole scoring waves) is copied on the current stream and goes straight into the front-end and scoring
    kernels while a side stream copies the rest, so all but the head's transfer is hidden behind compute.
    ``top_c``: None scores exactly; an integer C scores by top-C fast scoring (:meth:`SharedModelSet.score_top_c` /
    :meth:`ModelSet.score_top_c`, ``precision`` ignored), which needs ``ubm_index`` to name the set's UBM: the reference
    member of a :class:`SharedModelSet`, or the ``ubm_index`` of a :class:`ModelSet` (a :func:`map_enrol` set and its
    ``ubm_index``, whatever it adapted).
    Returns ``(decisions (N,) int64 host tensor, total_frames)``; the call returns after the decisions have landed."""
    torch = _lib.require_cuda()
    dev = front_end.device
    if top_c is not None:
        if ubm_index is None:
            raise ValueError("top_c scores against a UBM: pass ubm_index")
        ubm_member = speakers.ref_model if isinstance(speakers, SharedModelSet) else getattr(speakers, "ubm_index", None)
        if ubm_member is None or int(ubm_index) % speakers.n_models != ubm_member:
            raise NotImplementedError("top_c needs a SharedModelSet whose reference member is the UBM, or a ModelSet whose "
                                      "ubm_index is the UBM (ubm_index)")
        check_top_c(top_c, speakers.n_comp)
    if isinstance(host_pcm, np.ndarray):
        host_pcm = torch.from_numpy(np.ascontiguousarray(host_pcm))
    sample_offsets = np.asarray(sample_offsets, dtype=np.int64)
    n_utts = len(sample_offsets) - 1
    if out is None:
        out = torch.empty(n_utts, dtype=torch.int64, pin_memory=True)
    if n_utts == 0:
        return out, 0
    nfr = front_end.frame_counts(np.diff(sample_offsets))
    n_head = split_for_overlap(nfr, head_fraction, min_split_frames)
    cur = torch.cuda.current_stream(dev)
    pcm = torch.empty(int(sample_offsets[-1] - sample_offsets[0]), dtype=host_pcm.dtype, device=dev)
    base = int(sample_offsets[0])
    parts = [(0, n_utts)] if n_head == 0 else [(0, n_head), (n_head, n_utts)]
    ready = []
    side = None
    for k, (lo, hi) in enumerate(parts):
        a, b = int(sample_offsets[lo]) - base, int(sample_offsets[hi]) - base
        if k == 0:
            pcm[a:b].copy_(host_pcm[base + a : base + b], non_blocking=True)
            ready.append(None)
        else:
            side = _side_stream(dev)
            side.wait_stream(cur)  # the buffer was allocated on the current stream
            with torch.cuda.stream(side):
                pcm[a:b].copy_(host_pcm[base + a : base + b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(side)
            ready.append(ev)
    dec = torch.empty(n_utts, dtype=torch.int64, device=dev)
    total = 0
    for (lo, hi), ev in zip(parts, ready):
        if ev is not None:
            cur.wait_event(ev)
        offs = sample_offsets[lo : hi + 1] - base
        feats, foffs, _ = front_end.extract_device(pcm, offs)
        total += int(foffs[-1])
        if top_c is None:
            scores, _ = speakers.score(feats, foffs, precision=precision)
        else:
            scores, _ = speakers.score_top_c(feats, foffs, c=top_c)
        if ubm_index is not None:
            k = int(ubm_index) % scores.shape[1]
            llr = scores - scores[:, k : k + 1]
            llr[:, k] = -float("inf")
            scores = llr
        torch.argmax(scores, dim=1, out=dec[lo:hi])
    out.copy_(dec, non_blocking=True)
    cur.synchronize()
    return out, total


def chunk_features(audio, feature_type="MFCC", fs=16000, seconds=1.0):
    """The feature side of ``records()`` in the final GUI (UI/tmp.py:301-326): the recording is cut into whole chunks of
    ``seconds`` (a trailing partial chunk is dropped, :305-307), every chunk goes through ``mfcc(chunk)[0]``,
    ``plp(chunk)[0]`` or both side by side (``'MFCC_PLP'``, :311-319) -- no deltas -- and ``preprocessing.scale``
    (:321).  All chunks share ONE upload and one front-end launch per feature type: a chunk is a pair of offsets into
    the recording.  Returns a list of (T, F) float32 arrays, one per chunk."""
    torch = _lib.require_cuda()
    audio = np.asarray(audio)
    if audio.ndim == 2:
        audio = audio[:, 0]
    n = int(round(seconds * fs))
    n_chunks = len(audio) // n
    if n_chunks == 0:
        return []
    chunks = [audio[i * n : (i + 1) * n] for i in range(n_chunks)]
    if feature_type == "MFCC":
        front = fe._cached(("chunk-mfcc", fs), lambda: fe.FrontEnd(fe.sidekit_recipe(fs=fs), delta_order=0, cmvn=True))
        feats, offs, _ = front.extract(chunks)
    elif feature_type == "PLP":
        front = fe._cached(("chunk-plp", fs), lambda: fe.PlpFrontEnd(fe.plp_recipe(fs=fs), delta_order=0, cmvn=True))
        feats, offs, _ = front.extract(chunks)
    elif feature_type == "MFCC_PLP":
        f_m = fe._cached(("chunk-mfcc-raw", fs), lambda: fe.FrontEnd(fe.sidekit_recipe(fs=fs), delta_order=0, cmvn=False))
        f_p = fe._cached(("chunk-plp-raw", fs), lambda: fe.PlpFrontEnd(fe.plp_recipe(fs=fs), delta_order=0, cmvn=False))
        a, offs, _ = f_m.extract(chunks)
        b, offs_p, _ = f_p.extract(chunks)
        assert np.array_equal(offs, offs_p)
        both = torch.cat([a, b], dim=1).contiguous()
        feats = torch.empty_like(both)
        d_off = torch.as_tensor(offs, device=both.device)
        if both.numel():
            _lib.check(_lib.load().ssp_cmvn(_lib.ptr(both), _lib.ptr(d_off), len(offs) - 1, both.shape[1], _lib.ptr(feats),
                                            _lib.stream_ptr()), "ssp_cmvn")
    else:
        raise NameError(feature_type)
    host = feats.cpu().numpy()
    return [host[offs[i] : offs[i + 1]] for i in range(n_chunks)]


def chunk_identify(features, gmms, ubm, precision="auto"):
    """``_GMM_test`` of the final GUI (UI/tmp.py:337-349) and ``test`` of the GMM-UBM GUI (UI/GMM_UBM_GUI.py:102-113)
    for a list of chunk feature matrices: ``pred[j, i] = GMM[i].score(x_j) - UBM.score(x_j)`` in one launch, the GUI's
    "probability" ``exp(pred.max(1)) / exp(pred).sum(1)`` and the argmax.  Returns ``(pred, prob, decisions)``."""
    pred, who = identify(features, gmms, ubm, precision=precision)
    prob = np.exp(pred.max(axis=1)) / np.exp(pred).sum(axis=1)
    return pred, prob, who


_SIDE_STREAMS: dict = {}


def _side_stream(dev):
    torch = _lib.require_cuda()
    key = (dev.type, dev.index)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev)
    return _SIDE_STREAMS[key]


label_encoder: dict = {}


def list_wavs(path="dataset/ASR_GMM"):
    """The files ``GMM_UBM.load_data`` reads, in its order (``os.listdir`` of ``path/<speaker>/<session>/``), with their
    labels; fills the module-level ``label_encoder`` the way GMM_UBM.py:36-38 does."""
    files, y = [], []
    for num, speaker in enumerate(os.listdir(path)):
        label_encoder[speaker] = num
        spk_dir = os.path.join(path, speaker)
        for session in os.listdir(spk_dir):
            ses_dir = os.path.join(spk_dir, session)
            for wav in os.listdir(ses_dir):
                files.append(os.path.join(ses_dir, wav))
                y.append(num)
    return files, y


def load_batch(path="dataset/ASR_GMM"):
    """``load_data`` without the list: ``(PcmBatch, y)`` -- every file of the tree decoded by worker threads straight into
    one pinned staging buffer (:func:`~speech_signal_processing_b200.wavio.read_wav_batch`), ready for ONE upload and ONE
    front-end launch (``FrontEnd.extract(batch)``)."""
    files, y = list_wavs(path)
    return read_wav_batch(files), y


def load_data(path="dataset/ASR_GMM"):
    """``GMM_UBM.load_data`` (GMM_UBM.py:24-50): walk ``path/<speaker>/<session>/<wav>``, encode speakers in directory
    order into the module-level ``label_encoder``.  Returns ``(x, y)``: list of int16 arrays, list of labels.  The
    files are decoded in one batch (headers first, then ``readinto`` the slices of one pinned buffer from worker threads)
    and ``x`` holds views of that buffer; a tree with anything but 16-bit PCM files is read file by file with
    ``scipy.io.wavfile.read`` as the reference does (utils/tools.py:45-47).  Stereo files keep their first channel (the
    handling MFCC_DTW.py:141-144 applies)."""
    t0 = time.time()
    print("Loading data...")
    files, y = list_wavs(path)
    try:
        x = read_wav_batch(files).utterances()
    except ValueError:
        from scipy.io import wavfile

        x = []
        for f in files:
            _, audio = wavfile.read(f)
            x.append(audio[:, 0] if audio.ndim == 2 else audio)
    print("Complete! Spend {:.2f}s".format(time.time() - t0))
    return x, y


def load_extract(test_size=0.3, path="dataset/ASR_GMM", delta_order=1):
    """``GMM_UBM.load_extract`` (GMM_UBM.py:121-131): load, split per utterance with ``random_state=0``
    (sklearn's ``train_test_split`` permutation: ``RandomState(0).permutation(n)``, test = first ceil(test_size*n)),
    then ONE front-end launch per split."""
    x, y = load_data(path)
    n = len(x)
    n_test = int(np.ceil(test_size * n))
    perm = np.random.RandomState(0).permutation(n)
    test_idx, train_idx = perm[:n_test], perm[n_test:]
    train_data, x_train, y_train = fe.extract_feature([x[i] for i in train_idx], [y[i] for i in train_idx], is_train=True,
                                                      delta_order=delta_order)
    x_test, y_test = fe.extract_feature([x[i] for i in test_idx], [y[i] for i in test_idx], delta_order=delta_order)
    return train_data, x_train, y_train, x_test, y_test


def main(path="dataset/ASR_GMM"):
    """``GMM_UBM.main`` (GMM_UBM.py:202-204)."""
    train_data, x_train, y_train, x_test, y_test = load_extract(path=path)
    return GMM(train_data, x_train, y_train, x_test, y_test, model=False)


def GMM(train, x_train, y_train, x_test, y_test, n_components=16, model=False, label_encoder=None, random_state=None,
        precision="auto"):
    """``GMM_UBM.GMM`` (GMM_UBM.py:134-199) on the GPU; prints the reference's result line and
    returns ``(acc_train, acc_test, pred_test)`` (the reference returns None).

    ``label_encoder`` defaults to this module's global of the same name, like the reference's
    (GMM_UBM.py:21,154); if that is empty the speakers are the sorted keys of ``train``.
    """
    print("Train GMM-UBM model !")
    t0 = time.time()
    enc = label_encoder if label_encoder is not None else globals()["label_encoder"]
    speakers = list(enc.values()) if enc else sorted(train.keys())
    if model:
        print("load model from file...")
        with open("Model/GMM_MFCC_model.pkl", "rb") as f:
            gmms = [GaussianMixture.from_sklearn(g) if not isinstance(g, GaussianMixture) else g for g in pkl.load(f)]
        with open("Model/UBM_MFCC_model.pkl", "rb") as f:
            u = pkl.load(f)
            ubm = GaussianMixture.from_sklearn(u) if not isinstance(u, GaussianMixture) else u
    else:
        print("Train GMM!")
        # the per-speaker loop of GMM_UBM.py:154-160 as ONE batched EM: a statistics call per iteration for all speakers
        gmms = fit_batch([train[spk] for spk in speakers], n_components=n_components, covariance_type="diag",
                         random_state=random_state)
        print("Train UBM!")
        ubm_train = np.vstack([train[spk] for spk in speakers])
        ubm = GaussianMixture(n_components=n_components, covariance_type="diag", random_state=random_state).fit(ubm_train)
        os.makedirs("Model", exist_ok=True)
        with open("Model/GMM_MFCC_model.pkl", "wb") as f:
            pkl.dump([g.to_sklearn() for g in gmms], f)
        with open("Model/UBM_MFCC_model.pkl", "wb") as f:
            pkl.dump(ubm.to_sklearn(), f)
    valid, arg_train = identify(x_train, gmms, ubm, precision=precision)
    acc_train = float((arg_train == np.array(y_train)).sum() / len(x_train))
    pred, arg = identify(x_test, gmms, ubm, precision=precision)
    acc = float((arg == np.array(y_test)).sum() / len(x_test))
    print("spend {:.2f}s, train acc {:.2%}, test acc {:.2%}".format(time.time() - t0, acc_train, acc))
    return acc_train, acc, pred


def install(gmm_ubm_module):
    """Rebind the names GMM_UBM.py:16-20 imports so the reference script runs on the GPU:

        import GMM_UBM, speech_signal_processing_b200 as ssp
        ssp.install(GMM_UBM)
        GMM_UBM.main()

    ``mfcc`` returns the cepstra array (the contract ``delta(mfcc(x))`` at GMM_UBM.py:89-90 needs;
    the stock sidekit list return raises there -- SURVEY F6).
    """
    def mfcc_cepstra(sig, **kw):
        return fe.mfcc(sig, **kw)[0]

    def plp_cepstra(sig, **kw):
        return fe.plp(sig, **kw)[0]

    gmm_ubm_module.mfcc = mfcc_cepstra
    gmm_ubm_module.plp = plp_cepstra
    gmm_ubm_module.delta = fe.delta
    gmm_ubm_module.preprocessing = fe.preprocessing
    gmm_ubm_module.GaussianMixture = GaussianMixture
    return gmm_ubm_module
