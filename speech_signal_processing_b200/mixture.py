"""Diagonal-covariance GMM on the GPU behind sklearn's ``GaussianMixture`` surface.

The reference binds ``sklearn.mixture.GaussianMixture`` at GMM_UBM.py:16 and uses exactly
``GaussianMixture(n_components=K, covariance_type='diag').fit(X)`` (:158-160, :169-170) and
``.score(X)`` (:185, :194), plus pickling of the fitted objects (:173-179).  :class:`GaussianMixture`
mirrors that surface (same constructor names, attributes and error behaviour) and adds the rest of
sklearn's inference calls (``predict_proba``, ``predict``, ``fit_predict``, ``bic``, ``aic``); the arithmetic runs
in the CUDA library: ``ssp_gmm_pack_models`` / ``ssp_gmm_score`` / ``ssp_gmm_stats`` /
``ssp_gmm_posteriors`` / ``ssp_gmm_mstep``.  :class:`ModelSet` + :func:`score_matrix` are the batched form the reference
lacks (all utterances x all models in one launch instead of S*N*2 Python calls).
"""
from __future__ import annotations

import ctypes as C
import warnings

import numpy as np

from . import _lib

PRECISIONS = {"fp32": _lib.PREC_FP32, "tf32": _lib.PREC_TF32, "tf32x2": _lib.PREC_TF32X2, "tf32x3": _lib.PREC_TF32X3}
# Below this many components the single-pass TF32 rounding no longer averages out to 1e-4 of the utterance score /
# 1e-3 of an LLR (SURVEY 8(c)); "auto" then takes the 3-pass (FP32-grade) tensor rung.
SINGLE_PASS_MIN_COMPONENTS = 512
# GaussianMixture.predict_proba computes the posteriors in frame chunks of at most this many bytes of float32 output, so
# the device buffer stays bounded whatever the number of frames
PROBA_CHUNK_BYTES = 1 << 30


def resolve_precision(precision: str, n_comp: int, n_feat: int) -> str:
    """``"auto"`` -> the cheapest rung that keeps LLRs within 1e-3 absolute: tensor cores whenever the contraction
    fits the tcgen05 tile (2D + 2 <= 80), one TF32 pass for large models, three for small ones."""
    if precision != "auto":
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)} or 'auto' (got {precision!r})")
        return precision
    if 2 * n_feat + 2 > 80:
        return "fp32"
    return "tf32" if n_comp >= SINGLE_PASS_MIN_COMPONENTS else "tf32x3"


def _as_feats(x, device):
    """numpy (T, D) or torch tensor -> contiguous float32 CUDA tensor."""
    torch = _lib.require_cuda()
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.float32).contiguous()
    x = np.asarray(x)
    if x.ndim != 2:
        raise ValueError(f"Expected 2D array, got {x.ndim}D array instead")
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32), device=device)


def device_frames(feats, offsets, device, what="feats"):
    """The one rule for frames a caller hands the GMM and DTW kernels on the device -> ``offsets`` as np.int64.

    ``feats`` must be a 2-D float32 torch tensor on ``device`` with contiguous rows (a row range ``x[a:b]`` is fine, a
    column slice or a transpose is not); ``offsets`` a 1-D integer host array that starts at 0, never decreases and ends
    at ``feats.shape[0]`` (empty utterances are allowed).  Anything else raises ``ValueError`` before a launch: the
    kernels read ``feats`` as packed float32 rows through the offsets, so another dtype or layout would be read as
    wrong numbers, and bad offsets would send them past the buffer.  Nothing is converted: a float64 copy of an EM run's
    frames would cost as much HBM as the frames themselves.  Checked on the host, with no device read-back."""
    import torch

    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if not isinstance(feats, torch.Tensor):
        raise ValueError(f"{what}: expected a torch tensor on {device}, got {type(feats).__name__}")
    if feats.dim() != 2 or feats.dtype != torch.float32:
        raise ValueError(f"{what}: expected a 2-D float32 tensor, got {feats.dim()}-D {feats.dtype}")
    if feats.device != device:
        raise ValueError(f"{what}: the tensor is on {feats.device}, the kernels run on {device}")
    if not feats.is_contiguous():
        raise ValueError(f"{what}: rows must be contiguous (stride ({feats.shape[1]}, 1), got {tuple(feats.stride())}); "
                         "pass .contiguous()")
    offs = np.asarray(offsets)
    if offs.ndim != 1 or offs.dtype.kind not in "iu" or len(offs) == 0:
        raise ValueError(f"{what}: offsets must be a non-empty 1-D integer array (got {offs.ndim}-D {offs.dtype})")
    offs = offs.astype(np.int64, copy=False)
    if offs[0] != 0 or offs[-1] != feats.shape[0] or np.any(offs[1:] < offs[:-1]):
        raise ValueError(f"{what}: offsets must start at 0, never decrease and end at the {feats.shape[0]} rows of the "
                         f"tensor (got {offs[0]} .. {offs[-1]})")
    return offs


def concat_utterances(utts, device):
    """list of (T_i, D) arrays -> (feats (sum T, D) cuda, frame_offsets np.int64); a ``(feats, offsets)`` tuple of device
    frames is passed through after :func:`device_frames` has checked it."""
    torch = _lib.require_cuda()
    if isinstance(utts, tuple) and len(utts) == 2 and isinstance(utts[0], torch.Tensor):
        return utts[0], device_frames(utts[0], utts[1], device)
    lens = np.array([len(u) for u in utts], dtype=np.int64)
    offs = np.zeros(len(utts) + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    d = np.asarray(utts[0]).shape[1]
    host = torch.empty((int(offs[-1]), d), dtype=torch.float32, pin_memory=True)
    hv = host.numpy()
    for u, o in zip(utts, offs[:-1]):
        hv[o : o + len(u)] = u
    return host.to(device, non_blocking=True), offs


def _as_params(a, device):
    """A model parameter (numpy or torch) as a contiguous float64 tensor on ``device``."""
    torch = _lib.require_cuda()
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=torch.float64).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=device)


def stacked_params(models):
    """(weights (S,K), means (S,K,D), covariances (S,K,D)) numpy of a list of fitted GaussianMixture-likes."""
    return (np.stack([np.asarray(m.weights_) for m in models]), np.stack([np.asarray(m.means_) for m in models]),
            np.stack([np.asarray(m.covariances_) for m in models]))


def _upload_frames(ms, feats, offsets):
    """What every call of a model set ``ms`` starts with: :func:`device_frames`, the feature-width check and the upload of
    the offsets, which ``ms`` keeps alive until its next call so that the stream has consumed them before they are
    freed.  Returns (offsets on the device, number of segments, total frames)."""
    torch = _lib.require_cuda()
    offsets = device_frames(feats, offsets, ms.device)
    if feats.shape[1] != ms.n_feat:
        raise ValueError(f"X has {feats.shape[1]} features, but the models expect {ms.n_feat}")
    ms._keep = torch.as_tensor(offsets, device=ms.device)
    return ms._keep, len(offsets) - 1, int(offsets[-1])


class ModelSet:
    """``n_models`` diagonal GMMs with the same (K, D), packed once in HBM for the scoring kernels."""

    def __init__(self, weights, means, variances, device=None):
        torch = _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        w, mu, var = (_as_params(a, self.device) for a in (weights, means, variances))
        if mu.dim() == 2:
            w, mu, var = w[None], mu[None], var[None]
        if mu.dim() != 3 or var.shape != mu.shape or w.shape != mu.shape[:2]:
            raise ValueError("expected weights (S,K), means (S,K,D), variances (S,K,D)")
        self.n_models, self.n_comp, self.n_feat = (int(v) for v in mu.shape)
        self.dims = _lib.GmmDims(self.n_models, self.n_comp, self.n_feat)
        nbytes = int(self.lib.ssp_gmm_pack_bytes(C.byref(self.dims)))
        if nbytes <= 0:
            raise ValueError(f"unsupported GMM dims K={self.n_comp} D={self.n_feat} (need 1 <= D <= 80)")
        self.pack = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._ws = StatsWorkspace(self.device)  # the calls given no workspace of their own
        self.ubm_index = None   # set by with_ubm
        self.repack(w, mu, var)

    @classmethod
    def with_ubm(cls, weights, means, variances, ubm, device=None):
        """Speakers MAP-adapted from ``ubm`` in any of weights, means and variances (``weights`` (S,K), ``means`` and
        ``variances`` (S,K,D), e.g. :func:`~speech_signal_processing_b200.ubm.map_adapt`) and the UBM as one set: the UBM
        is model S and ``ubm_index`` names it.  That declares that component c of every speaker is component c of the UBM,
        which :meth:`score_top_c` needs, and lets ``identify`` score the UBM in the same launch as the speakers.  ``ubm``:
        a fitted GaussianMixture-like or a one-model :class:`ModelSet`.  Weights and variances must be positive and finite
        (``ValueError`` otherwise, before anything is launched): the top-C table takes their logarithms, and a variance
        MAP at relevance 0 gives a component of one frame a zero variance."""
        torch = _lib.require_cuda()
        dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if isinstance(ubm, ModelSet):
            if ubm.n_models != 1:
                raise ValueError(f"ubm must be ONE model (got a ModelSet of {ubm.n_models})")
            ubm_params = ubm._params
        else:
            ubm_params = (ubm.weights_, ubm.means_, ubm.covariances_)
        w, mu, var = (_as_params(a, dev) for a in (weights, means, variances))
        uw, umu, uvar = (_as_params(a, dev) for a in ubm_params)
        if mu.dim() != 3 or var.shape != mu.shape or w.shape != mu.shape[:2] or umu.numel() != mu.shape[1] * mu.shape[2] \
                or uvar.numel() != umu.numel() or uw.numel() != mu.shape[1]:
            raise ValueError("expected weights (S,K), means (S,K,D), variances (S,K,D) and a UBM of the same K and D")
        w, mu, var = (torch.cat([a, u.reshape(1, *a.shape[1:])]) for a, u in ((w, uw), (mu, umu), (var, uvar)))
        for name, a in (("weights", w), ("variances", var)):
            if not bool((torch.isfinite(a) & (a > 0)).all().item()):
                raise ValueError(f"{name} must be positive and finite (the speakers' and the UBM's)")
        ms = cls(w, mu, var, device=dev)
        ms.ubm_index = ms.n_models - 1
        return ms

    @_lib.on_device
    def repack(self, w, mu, var):
        """Re-derive the packed operands from (device, float64) parameters -- one tiny kernel."""
        self._params = (w, mu, var)
        self._topc = None   # score_top_c's UBM set and table are rebuilt from the new parameters
        _lib.check(self.lib.ssp_gmm_pack_models(_lib.ptr(w), _lib.ptr(mu), _lib.ptr(var), C.byref(self.dims),
                                                _lib.ptr(self.pack), _lib.stream_ptr()), "ssp_gmm_pack_models")

    def _image_frames(self, fn, name, total, ws_bytes, workspace, reuse_images, *args):
        """``fn(*args, workspace, ws_bytes, reuse_images, stream)``: one of the calls that turn the frames into operand
        images in a :class:`StatsWorkspace`.  Without a ``workspace`` the set's own serves and its images are rebuilt (its
        frames may be another call's).  The workspace holds valid images only after a call that imaged frames."""
        if workspace is None:
            workspace, reuse_images = self._ws, False
        buf = workspace.reserve(ws_bytes)
        _lib.check(fn(*args, _lib.ptr(buf) if ws_bytes else None, ws_bytes, int(bool(reuse_images) and workspace.valid),
                      _lib.stream_ptr()), name)
        if total:
            workspace.valid = True

    # ---------------------------------------------------------------------------------------
    @_lib.on_device
    def score(self, feats, frame_offsets, precision="auto", want_frame_lse=False):
        """(scores (n_utts, n_models) cuda float64, frame_lse (n_models, total) cuda float32 | None).
        ``precision``: "fp32" (CUDA cores), "tf32" / "tf32x2" / "tf32x3" (tcgen05, 1 / 2 / 3 passes of 11-bit operands; the
        single pass streams FP16 images of the models) or "auto"
        (:func:`resolve_precision`)."""
        torch = _lib.require_cuda()
        precision = resolve_precision(precision, self.n_comp, self.n_feat)
        d_off, n_utts, total = _upload_frames(self, feats, frame_offsets)
        scores = torch.empty((n_utts, self.n_models), dtype=torch.float64, device=self.device)
        lse = torch.empty((self.n_models, total), dtype=torch.float32, device=self.device) if want_frame_lse else None
        rc = self.lib.ssp_gmm_score(_lib.ptr(feats), _lib.ptr(d_off), n_utts, total, _lib.ptr(self.pack),
                                    C.byref(self.dims), PRECISIONS[precision], _lib.ptr(scores), _lib.ptr(lse),
                                    _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_score")
        return scores, lse

    @_lib.on_device
    def stats(self, feats, seg_offsets, workspace=None, reuse_images=False):
        """N (S,K), F (S,K,D), S2 (S,K,D), loglik (S,) float64 cuda: every segment under this set's single model, or
        -- if the set holds one model per segment -- segment s under model s (models trained together, :func:`fit_batch`).

        ``workspace``: a :class:`StatsWorkspace` shared between calls (and model sets) on the SAME ``feats`` /
        ``seg_offsets``; ``reuse_images=True`` then skips the preparation pass that turns the frames into tensor-core
        operand images (EM iterations: the frames never change).  Default: a workspace owned by this model set."""
        torch = _lib.require_cuda()
        d_off, n_segs, total = _upload_frames(self, feats, seg_offsets)
        if self.n_models != 1 and self.n_models != n_segs:
            raise ValueError("statistics are taken under one model for all segments (the UBM), or under one model per "
                             f"segment (got {self.n_models} models for {n_segs} segments)")
        k, d = self.n_comp, self.n_feat
        n = torch.zeros((n_segs, k), dtype=torch.float64, device=self.device)
        f = torch.zeros((n_segs, k, d), dtype=torch.float64, device=self.device)
        s = torch.zeros((n_segs, k, d), dtype=torch.float64, device=self.device)
        ll = torch.zeros(n_segs, dtype=torch.float64, device=self.device)
        lse = torch.empty(max(total, 1), dtype=torch.float32, device=self.device)
        self._image_frames(self.lib.ssp_gmm_stats, "ssp_gmm_stats", total,
                           int(self.lib.ssp_gmm_stats_workspace_bytes(C.byref(self.dims), total, n_segs)), workspace,
                           reuse_images, _lib.ptr(feats), _lib.ptr(d_off), n_segs, total, _lib.ptr(self.pack),
                           C.byref(self.dims), _lib.ptr(lse), _lib.ptr(n), _lib.ptr(f), _lib.ptr(s), _lib.ptr(ll))
        self._keep = (d_off, lse)
        return n, f, s, ll


    @_lib.on_device
    def posteriors(self, feats, seg_offsets, resp=True, labels=False, workspace=None, reuse_images=False):
        """(resp (T, K) float32 cuda | None, labels (T,) int64 cuda | None, frame_lse (T,) float32 cuda | None): frame
        posteriors and/or the most probable component of every frame (lowest index on ties), under this set's single
        model or -- one model per segment -- segment s under model s, as in :meth:`stats`.  ``frame_lse`` (the per-frame
        log-likelihood) comes with ``resp``; labels alone skip the log-sum-exp pass and return None there.

        Always FP32 grade (``ssp_gmm_posteriors``): the 3 x BF16 tensor-core logits of :meth:`stats` for D <= 39, the
        FP32 CUDA-core kernels above.  ``workspace`` / ``reuse_images`` as in :meth:`stats`, whose workspace (and frame
        images) this call shares."""
        torch = _lib.require_cuda()
        d_off, n_segs, total = _upload_frames(self, feats, seg_offsets)
        if self.n_models != 1 and self.n_models != n_segs:
            raise ValueError("posteriors are taken under one model for all segments, or under one model per segment "
                             f"(got {self.n_models} models for {n_segs} segments)")
        if not (resp or labels):
            raise ValueError("posteriors: ask for resp, labels or both")
        g = torch.empty((total, self.n_comp), dtype=torch.float32, device=self.device) if resp else None
        lab = torch.empty(total, dtype=torch.int64, device=self.device) if labels else None
        lse = torch.empty(total, dtype=torch.float32, device=self.device) if resp else None
        self._image_frames(self.lib.ssp_gmm_posteriors, "ssp_gmm_posteriors", total,
                           int(self.lib.ssp_gmm_posteriors_workspace_bytes(C.byref(self.dims), total, n_segs)), workspace,
                           reuse_images, _lib.ptr(feats), _lib.ptr(d_off), n_segs, total, _lib.ptr(self.pack),
                           C.byref(self.dims), _lib.ptr(g), _lib.ptr(lab), _lib.ptr(lse))
        return g, lab, lse

    @_lib.on_device
    def top_components(self, feats, seg_offsets, c, workspace=None, reuse_images=False):
        """(idx (T, C) int32 cuda, logit (T, C) float32 cuda): the C components with the largest weighted
        log-probability ``log w_c + log N(x_t; c)`` for every frame, in descending order and the lower index first on
        equal values -- the Gaussian selection of top-C fast scoring (:meth:`SharedModelSet.score_top_c`).  One-model
        sets, D <= 39, 1 <= c <= min(K, 64).  FP32 grade: the tensor-core logits of :meth:`posteriors`, whose workspace
        (and frame images) this call shares; ``workspace`` / ``reuse_images`` as in :meth:`stats`."""
        torch = _lib.require_cuda()
        d_off, n_segs, total = _upload_frames(self, feats, seg_offsets)
        if self.n_models != 1:
            raise ValueError(f"top_components selects under one model (got a set of {self.n_models})")
        c = check_top_c(c, self.n_comp)
        idx = torch.empty((total, c), dtype=torch.int32, device=self.device)
        logit = torch.empty((total, c), dtype=torch.float32, device=self.device)
        self._image_frames(self.lib.ssp_gmm_top_components, "ssp_gmm_top_components", total,
                           int(self.lib.ssp_gmm_top_components_workspace_bytes(C.byref(self.dims), total, n_segs, c)),
                           workspace, reuse_images, _lib.ptr(feats), _lib.ptr(d_off), n_segs, total, _lib.ptr(self.pack),
                           C.byref(self.dims), c, _lib.ptr(idx), _lib.ptr(logit))
        return idx, logit

    @_lib.on_device
    def score_top_c(self, feats, frame_offsets, c=5, want_frame_lse=False):
        """Top-C fast scoring (Reynolds, Quatieri & Dunn 2000) of a set from :meth:`with_ubm`, whose speakers are
        MAP-adapted from the UBM in weights and variances as well as means: (scores (n_utts, n_models) cuda float64,
        frame_lse (n_models, total) cuda float32 | None).  For every frame the C components the UBM (``ubm_index``) ranks
        highest are selected (:meth:`top_components`), and every model is scored over those C components only:
        ``log sum_{c in S_t} w_s,c N(x_t; mu_s,c, var_s,c)``, averaged over the frames of each utterance (0 for an empty
        one).  With ``c = n_comp`` it is the exact score.  Always FP32 grade: FP32-grade selection logits, the difference
        from the UBM as FP32 FMAs on frames centred on the UBM's component mean, double utterance sums.  A set without
        ``ubm_index`` is a ``ValueError``, D > 39 a ``NotImplementedError``; neither launches anything."""
        if self.ubm_index is None:
            raise ValueError("top-C scoring selects under the UBM: build the set with ModelSet.with_ubm (ubm_index)")
        return _score_top_c(self, feats, frame_offsets, c, want_frame_lse, self.lib.ssp_gmm_score_topc_adapted,
                            "ssp_gmm_score_topc_adapted")

    def _topc_tables(self):
        """(the UBM as a one-model set (selection), the ``ssp_gmm_pack_topc_adapted`` table, the scoring's scratch), made
        on first use and dropped by :meth:`repack`."""
        torch = _lib.require_cuda()
        if self._topc is None:
            nbytes = int(self.lib.ssp_gmm_topc_adapted_pack_bytes(C.byref(self.dims)))
            if nbytes <= 0:
                raise NotImplementedError(f"top-C scoring takes D <= 39 (got D = {self.n_feat})")
            w, mu, var = self._params
            k = self.ubm_index
            ref = ModelSet(w[k][None], mu[k][None], var[k][None], device=self.device)
            pack = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.ssp_gmm_pack_topc_adapted(_lib.ptr(w), _lib.ptr(mu), _lib.ptr(var), C.byref(self.dims), k,
                                                          _lib.ptr(pack), _lib.stream_ptr()), "ssp_gmm_pack_topc_adapted")
            self._topc = (ref, pack, StatsWorkspace(self.device))
        return self._topc


# widest selection the top-C kernels keep per frame
MAX_TOP_C = 64


def check_top_c(c, n_comp):
    """``c`` as an int in [1, min(n_comp, MAX_TOP_C)], else ``ValueError``."""
    if isinstance(c, bool) or not isinstance(c, (int, np.integer)) or not 1 <= int(c) <= min(n_comp, MAX_TOP_C):
        raise ValueError(f"top-C needs an integer C in [1, min(K = {n_comp}, {MAX_TOP_C})] (got {c!r})")
    return int(c)


def _score_top_c(ms, feats, frame_offsets, c, want_frame_lse, score_fn, name):
    """The top-C call of :class:`SharedModelSet` and :class:`ModelSet`: the selection under the set's UBM, then
    ``score_fn`` (``ssp_gmm_score_topc`` / ``ssp_gmm_score_topc_adapted``) on the table of ``ms._topc_tables()``."""
    torch = _lib.require_cuda()
    d_off, n_utts, total = _upload_frames(ms, feats, frame_offsets)
    c = check_top_c(c, ms.n_comp)
    ref, pack, scratch = ms._topc_tables()
    idx, logit = ref.top_components(feats, np.array([0, total], dtype=np.int64), c)
    scores = torch.empty((n_utts, ms.n_models), dtype=torch.float64, device=ms.device)
    lse = torch.empty((ms.n_models, total), dtype=torch.float32, device=ms.device) if want_frame_lse else None
    ws_bytes = int(ms.lib.ssp_gmm_score_topc_workspace_bytes(C.byref(ms.dims), c, total))
    ws = scratch.reserve(ws_bytes)
    rc = score_fn(_lib.ptr(feats), _lib.ptr(d_off), n_utts, total, _lib.ptr(idx), _lib.ptr(logit), c, _lib.ptr(pack),
                  C.byref(ms.dims), _lib.ptr(scores), _lib.ptr(lse), _lib.ptr(ws) if ws_bytes else None, ws_bytes,
                  _lib.stream_ptr())
    _lib.check(rc, name)
    ms._keep = (d_off, idx, logit)
    return scores, lse


class StatsWorkspace:
    """Grow-only device scratch of the GMM calls that take a workspace.  ``ssp_gmm_stats``, ``ssp_gmm_posteriors`` and
    ``ssp_gmm_top_components`` lay it out alike (operand images of the frames + log-sum-exp partials): ``valid`` says that
    it holds the images of the frames it was last used with; growing it invalidates them."""

    def __init__(self, device):
        self.device, self.buf, self.valid = device, None, False

    def reserve(self, nbytes: int):
        torch = _lib.require_cuda()
        if nbytes and (self.buf is None or self.buf.numel() < nbytes):
            self.buf = None  # release before growing: the images of a large run are tens of GB
            self.buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self.valid = False
        return self.buf


class SharedModelSet:
    """``n_models`` diagonal GMMs that share ONE weight vector and ONE variance matrix and differ in their means --
    what mean-only MAP enrolment from a UBM yields (:func:`~speech_signal_processing_b200.ubm.map_adapt` with
    ``adapt=("means",)``).  Scored by the shared-variance tensor kernel (``ssp_gmm_score_shared``): the part of the
    log-likelihood common to all models -- the logit of the reference member ``ref_model`` (the UBM), evaluated to FP32
    grade in three FP16 passes -- is computed once per frame block; the per-model contraction is D + 2 long instead of
    2D + 2 and acts on ``means[s] - means[ref_model]`` in FP16 operands (the 11-bit significand of TF32), so its rounding
    scales with the distance from the reference and cancels in log-likelihood ratios against it.  Results equal
    :class:`ModelSet` ``.score(precision="tf32")`` on the expanded set to that rung's rounding or better.  Needs
    D <= 39 and parameters inside FP16's range (``NotImplementedError`` otherwise: use :meth:`expand` / :class:`ModelSet`)."""

    def __init__(self, weights, variances, means, ref_model=-1, device=None):
        torch = _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        w, var, mu = (_as_params(a, self.device) for a in (weights, variances, means))
        if mu.dim() == 2:
            mu = mu[None]
        if w.dim() != 1 or var.dim() != 2 or mu.dim() != 3 or mu.shape[1:] != var.shape or w.shape[0] != var.shape[0]:
            raise ValueError("expected weights (K,), variances (K,D), means (S,K,D)")
        self.n_models, self.n_comp, self.n_feat = (int(v) for v in mu.shape)
        self.ref_model = int(ref_model) % self.n_models
        self.dims = _lib.GmmDims(self.n_models, self.n_comp, self.n_feat)
        nbytes = int(self.lib.ssp_gmm_shared_pack_bytes(C.byref(self.dims)))
        if nbytes <= 0:
            raise ValueError(f"unsupported dims K={self.n_comp} D={self.n_feat} for the shared-variance kernel (need D <= 39)")
        self.pack = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ssp_gmm_pack_shared(_lib.ptr(w), _lib.ptr(var), _lib.ptr(mu), C.byref(self.dims),
                                                    self.ref_model, _lib.ptr(self.pack), _lib.stream_ptr()),
                       "ssp_gmm_pack_shared")
        self._params = (w, var, mu)
        self._ws = None    # score's scratch, made when the scoring first needs one (more than one L2 group of models)
        self._topc = None

    @classmethod
    def with_ubm(cls, weights, variances, speaker_means, ubm_means, device=None):
        """Speakers (S,K,D means) and their UBM (K,D means) with the same weights and variances as one set: the UBM is
        model S, the reference member, and ``ubm_index`` names it."""
        torch = _lib.require_cuda()
        dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        speaker_means, ubm_means = _as_params(speaker_means, dev), _as_params(ubm_means, dev)
        sms = cls(weights, variances, torch.cat([speaker_means, ubm_means.reshape(1, *speaker_means.shape[1:])]),
                  ref_model=-1, device=dev)
        sms.ubm_index = sms.n_models - 1
        return sms

    @staticmethod
    def shares_base(weights, variances) -> bool:
        """True if every model of an (S,K) / (S,K,D) parameter stack has the first model's weights and variances."""
        torch = _lib.require_cuda()
        if isinstance(weights, torch.Tensor):
            return bool((weights == weights[:1]).all().item() and (variances == variances[:1]).all().item())
        weights, variances = np.asarray(weights), np.asarray(variances)
        return bool((weights == weights[:1]).all() and (variances == variances[:1]).all())

    @_lib.on_device
    def score(self, feats, frame_offsets, precision="tf32", want_frame_lse=False):
        """(scores (n_utts, n_models) cuda float64, frame_lse (n_models, total) cuda float32 | None)."""
        torch = _lib.require_cuda()
        if precision not in ("tf32", "auto"):
            raise ValueError("the shared-variance kernel has one precision rung (11-bit operands, FP32-grade common part); expand() to a ModelSet for the "
                             "other precisions")
        d_off, n_utts, total = _upload_frames(self, feats, frame_offsets)
        scores = torch.empty((n_utts, self.n_models), dtype=torch.float64, device=self.device)
        lse = torch.empty((self.n_models, total), dtype=torch.float32, device=self.device) if want_frame_lse else None
        ws_bytes = int(self.lib.ssp_gmm_score_shared_workspace_bytes(C.byref(self.dims), total))
        if ws_bytes and self._ws is None:
            self._ws = StatsWorkspace(self.device)
        ws = self._ws.reserve(ws_bytes) if ws_bytes else None
        rc = self.lib.ssp_gmm_score_shared(_lib.ptr(feats), _lib.ptr(d_off), n_utts, total, _lib.ptr(self.pack),
                                           C.byref(self.dims), _lib.ptr(scores), _lib.ptr(lse),
                                           _lib.ptr(ws) if ws_bytes else None, ws_bytes, _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_score_shared")
        return scores, lse

    @_lib.on_device
    def score_top_c(self, feats, frame_offsets, c=5, want_frame_lse=False):
        """Top-C fast scoring (Reynolds, Quatieri & Dunn 2000): (scores (n_utts, n_models) cuda float64, frame_lse
        (n_models, total) cuda float32 | None).  For every frame the C components the reference member ``ref_model`` (the
        UBM) ranks highest are selected (:meth:`ModelSet.top_components`), and every model is scored over those C
        components only: ``log sum_{c in S_t} w_c N(x_t; mu_s,c, var_c)``, averaged over the frames of each utterance (0 for
        an empty one).  An approximation with its own definition: with ``c = n_comp`` it is the exact score.  Always FP32
        grade (FP32-grade selection logits, FP32 difference terms, double utterance sums)."""
        return _score_top_c(self, feats, frame_offsets, c, want_frame_lse, self.lib.ssp_gmm_score_topc, "ssp_gmm_score_topc")

    def _topc_tables(self):
        """(the reference member as a one-model set (selection), the component-major (a, b) table (scoring), the
        scoring's scratch), made on first use."""
        torch = _lib.require_cuda()
        if self._topc is None:
            w, var, mu = self._params
            ref = ModelSet(w[None], mu[self.ref_model][None], var[None], device=self.device)
            pack = torch.empty(int(self.lib.ssp_gmm_topc_pack_bytes(C.byref(self.dims))), dtype=torch.uint8, device=self.device)
            _lib.check(self.lib.ssp_gmm_pack_topc(_lib.ptr(var), _lib.ptr(mu), C.byref(self.dims), self.ref_model,
                                                  _lib.ptr(pack), _lib.stream_ptr()), "ssp_gmm_pack_topc")
            self._topc = (ref, pack, StatsWorkspace(self.device))
        return self._topc

    def expand(self) -> "ModelSet":
        """The same models as a general :class:`ModelSet` (weights and variances replicated)."""
        w, var, mu = self._params
        return ModelSet(w[None].expand(self.n_models, -1), mu, var[None].expand(self.n_models, -1, -1), device=self.device)


def score_matrix(utts, models, precision="auto", device=None):
    """``pred[j, i] = models[i].score(utts[j])`` for all pairs in one launch (GMM_UBM.py:182-185,
    191-194 without the Python double loop).  ``models``: list of fitted :class:`GaussianMixture`
    (or anything with ``weights_/means_/covariances_``) or a :class:`ModelSet`.  Returns float64 numpy."""
    torch = _lib.require_cuda()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    ms = models if isinstance(models, ModelSet) else ModelSet(*stacked_params(models), device=dev)
    feats, offs = concat_utterances(utts, dev)
    scores, _ = ms.score(feats, offs, precision=precision)
    return scores.cpu().numpy()


def _nk_eps(X):
    """sklearn's floor on the component counts of the M-step: 10 eps of the input's dtype (float32 input keeps
    float32, anything else is taken as float64)."""
    torch = _lib.require_cuda()
    f32 = (isinstance(X, torch.Tensor) and X.dtype == torch.float32) or (isinstance(X, np.ndarray) and X.dtype == np.float32)
    return 10.0 * float(np.finfo(np.float32 if f32 else np.float64).eps)


def _check_sample_counts(counts, k):
    """sklearn's refusal of a model fitted to fewer than 2 or fewer than ``k`` frames."""
    for cnt in counts:
        if cnt < 2:
            raise ValueError(f"Found array with {cnt} sample(s) while a minimum of 2 is required.")
        if cnt < k:
            raise ValueError(f"Expected n_samples >= n_components but got n_components = {k}, n_samples = {cnt}")


class GaussianMixture:
    """GPU drop-in for ``sklearn.mixture.GaussianMixture(covariance_type='diag')``.

    Same constructor arguments and fitted attributes as sklearn 1.9 (``weights_``, ``means_``,
    ``covariances_``, ``precisions_``, ``precisions_cholesky_``, ``converged_``, ``n_iter_``,
    ``lower_bound_``, ``lower_bounds_``).  ``init_params='kmeans'`` runs a GPU Lloyd iteration from
    random frames (sklearn's KMeans++ stream is not reproduced: the reference leaves
    ``random_state=None``, so its own runs are not reproducible either -- SURVEY F7); parity with
    sklearn is defined for given ``weights_init/means_init/precisions_init``.

    Inference beyond ``score`` follows sklearn too: ``predict_proba`` (float64 posteriors), ``predict`` and
    ``fit_predict`` (int64 labels, the lowest component index on ties), ``bic`` and ``aic``.  Posteriors and labels are
    always computed at FP32 grade (``ssp_gmm_posteriors``: 3 x BF16 tensor-core logits for D <= 39, FP32 CUDA cores
    above), whatever ``precision`` says.

    ``precision`` selects the scoring kernel of ``score`` / ``score_samples``: ``"fp32"`` (default: CUDA-core
    FMA, ~1e-7 relative, safe for any data) or ``"tf32"`` (tcgen05 tensor cores; meant for CMVN-normalised
    features, where the single-pass TF32 operand rounding stays within 1e-4 relative of the utterance score --
    on un-normalised data with |x - mu| >> sigma the expanded form loses digits).  The batched
    :func:`score_matrix` / ``identify`` default to ``"tf32"``.

    ``comm``: optional :class:`speech_signal_processing_b200.dist.Comm`; when given, ``fit`` treats X as
    this rank's shard of the frames and all-reduces the statistics tensor each EM iteration (NCCL).
    """

    def __init__(self, n_components=1, *, covariance_type="diag", tol=1e-3, reg_covar=1e-6, max_iter=100, n_init=1,
                 init_params="kmeans", weights_init=None, means_init=None, precisions_init=None, random_state=None,
                 warm_start=False, verbose=0, verbose_interval=10, precision="fp32", comm=None):
        self.n_components = n_components
        self.covariance_type = covariance_type
        self.tol = tol
        self.reg_covar = reg_covar
        self.max_iter = max_iter
        self.n_init = n_init
        self.init_params = init_params
        self.weights_init = weights_init
        self.means_init = means_init
        self.precisions_init = precisions_init
        self.random_state = random_state
        self.warm_start = warm_start
        self.verbose = verbose
        self.verbose_interval = verbose_interval
        self.precision = precision
        self.comm = comm
        self._ms = None

    # ------------------------------------------------------------------ pickling (GMM_UBM.py:173-179)
    def __getstate__(self):
        st = dict(self.__dict__)
        st["_ms"] = None
        st["comm"] = None
        return st

    # ------------------------------------------------------------------ helpers
    def _check(self):
        if self.covariance_type != "diag":
            raise NotImplementedError("only covariance_type='diag' (the reference's setting, GMM_UBM.py:158) is implemented")
        if self.n_components < 1:
            raise ValueError(f"Invalid value for 'n_components': {self.n_components}")

    def _model_set(self):
        if self._ms is None:
            if not hasattr(self, "means_"):
                raise AttributeError("This GaussianMixture instance is not fitted yet. Call 'fit' first.")
            self._ms = ModelSet(self.weights_, self.means_, self.covariances_)
        return self._ms

    def _rng(self):
        return self.random_state if isinstance(self.random_state, np.random.RandomState) else np.random.RandomState(self.random_state)

    def _set_fitted(self, weights, means, covariances, converged, n_iter, lower_bound):
        self.weights_, self.means_, self.covariances_ = (np.asarray(a, dtype=np.float64) for a in (weights, means, covariances))
        self.precisions_cholesky_ = 1.0 / np.sqrt(self.covariances_)
        self.precisions_ = self.precisions_cholesky_ ** 2
        self.converged_, self.n_iter_, self.lower_bound_ = bool(converged), int(n_iter), float(lower_bound)
        self._ms = None

    def _finish_em(self, weights, means, covariances, converged, n_iter, lower_bound, bounds):
        """sklearn's end of ``fit``: the non-convergence warning, the refusal of ill-defined covariances, the fitted
        attributes."""
        if not converged and self.max_iter > 0:
            warnings.warn("Best performing initialization did not converge. Try different init parameters, or "
                          "increase max_iter, tol, or check for degenerate data.", UserWarning)
        if not np.all(np.isfinite(covariances)) or np.any(covariances <= 0):
            raise ValueError("Fitting the mixture model failed because some components have ill-defined empirical "
                             "covariance (for instance caused by singleton or collapsed samples). Try to decrease the "
                             "number of components, increase reg_covar, or scale the input data.")
        self._set_fitted(weights, means, covariances, converged, n_iter, lower_bound)
        self.lower_bounds_ = bounds

    # ------------------------------------------------------------------ EM
    def _em_step(self, ms, feats, seg, workspace, nk_eps, w, mu, var, timed=False):
        """One E+M step on device: the statistics of segment s under model s (``ssp_gmm_stats``), summed over the ranks of
        ``comm`` in ONE all-reduce of ``[N, F, S, loglik, frames]``, then the M-step of every model into (w, mu, var).
        Returns (N, loglik) on the device and the frames of every segment on the host, all summed over the ranks."""
        torch = _lib.require_cuda()
        counts = np.diff(seg).astype(np.float64)
        n, f, s, ll = ms.stats(feats, seg, workspace=workspace, reuse_images=True)
        reduce = self.comm is not None and self.comm.world_size > 1
        if reduce:
            parts = (n, f, s, ll, torch.as_tensor(counts, device=feats.device))
            flat = torch.cat([t.reshape(-1) for t in parts])
            # bench.py: a list to append (start, end) CUDA events of the EM loop's all-reduce to
            timing = getattr(self, "allreduce_events", None) if timed else None
            if timing is not None:
                timing.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
                timing[-1][0].record()
            flat = self.comm.allreduce_sum(flat)
            if timing is not None:
                timing[-1][1].record()
            n, f, s, ll, counts = (v.view(t.shape) for v, t in zip(flat.split([t.numel() for t in parts]), parts))
        rc = ms.lib.ssp_gmm_mstep(_lib.ptr(n), _lib.ptr(f), _lib.ptr(s), ms.n_models, ms.n_comp, ms.n_feat,
                                  float(self.reg_covar), float(nk_eps), _lib.ptr(w), _lib.ptr(mu), _lib.ptr(var),
                                  _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_mstep")
        return n, ll, counts.cpu().numpy() if reduce else counts

    def _em(self, feats, seg, workspace, w, mu, var, nk_eps):
        """The EM loop of :meth:`fit` (S = 1) and :func:`fit_batch`: S models from (w (S,K), mu, var (S,K,D)), segment s
        of ``feats`` under model s, each to its own convergence as :func:`fit_batch` describes; the lower bound is the mean
        frame log-likelihood under the parameters the E-step used.  Returns (w, mu, var, lower bound (S,), bounds of
        every iteration (S lists), converged (S,), n_iter (S,))."""
        torch = _lib.require_cuda()
        ms = ModelSet(w, mu, var, device=feats.device)
        lower = np.full(ms.n_models, -np.inf)
        bounds = [[] for _ in range(ms.n_models)]
        converged = np.zeros(ms.n_models, dtype=bool)
        n_iter = np.zeros(ms.n_models, dtype=np.int64)
        for it in range(1, self.max_iter + 1):
            active = ~converged
            if not active.any():
                break
            ms.repack(w, mu, var)
            if active.all():  # the M-step in place
                _, ll, cnt = self._em_step(ms, feats, seg, workspace, nk_eps, w, mu, var, timed=True)
            else:
                w_new, mu_new, var_new = torch.empty_like(w), torch.empty_like(mu), torch.empty_like(var)
                _, ll, cnt = self._em_step(ms, feats, seg, workspace, nk_eps, w_new, mu_new, var_new, timed=True)
                keep = torch.as_tensor(active, device=feats.device)
                w = torch.where(keep[:, None], w_new, w)
                mu = torch.where(keep[:, None, None], mu_new, mu)
                var = torch.where(keep[:, None, None], var_new, var)
            now = ll.cpu().numpy() / cnt          # the one host synchronisation of the iteration (a second with comm)
            for i in np.nonzero(active)[0]:
                bounds[i].append(float(now[i]))
                n_iter[i] = it
                if abs(now[i] - lower[i]) < self.tol:
                    converged[i] = True
                lower[i] = now[i]
        return w, mu, var, lower, bounds, converged, n_iter

    def _kmeans_init(self, feats, seg, rs, w, mu, var, nk_eps, iters=10, workspace=None):
        """Lloyd iterations as hard EM: equal weights, one small shared variance, so posteriors are
        (numerically) one-hot; empty clusters are re-seeded from random frames.  Ends with sklearn's
        ``_initialize(X, resp)`` M-step from those assignments."""
        torch = _lib.require_cuda()
        n_frames, d = feats.shape
        k = self.n_components
        comm = self.comm if (self.comm is not None and self.comm.world_size > 1) else None

        def seed_rows(count, avoid=None):
            """`count` seed frames, identical on every rank (rank 0 draws from its shard): k-means++
            D^2 sampling (the seeding sklearn's KMeans uses) over a random subsample of <= 20k frames;
            control logic on device tensors, no host round trip per seed."""
            rows = torch.zeros((count, d), dtype=torch.float64, device=feats.device)
            if comm is None or comm.rank == 0:
                m = int(min(n_frames, max(20 * k, 4096)))
                # indices WITH replacement: a permutation of all frames (rs.choice(replace=False)) is 288 MB of host
                # work at 36 M frames, and duplicates among <= 20k of millions of frames are harmless for seeding
                pick = rs.permutation(n_frames)[:m] if n_frames <= 4 * m else rs.randint(n_frames, size=m)
                sub = feats[torch.as_tensor(pick, device=feats.device)].to(torch.float64)
                u = torch.as_tensor(rs.uniform(size=count), device=feats.device)
                if avoid is None:
                    rows[0] = sub[int(rs.randint(m))]
                    d2 = ((sub - rows[0]) ** 2).sum(dim=1)
                    start = 1
                else:
                    d2 = torch.cdist(sub, avoid).min(dim=1).values ** 2
                    start = 0
                for i in range(start, count):
                    j = torch.searchsorted(d2.cumsum(0), u[i] * d2.sum()).clamp_(max=m - 1)
                    rows[i] = sub[j]
                    d2 = torch.minimum(d2, ((sub - rows[i]) ** 2).sum(dim=1))
            return comm.broadcast(rows.contiguous()) if comm is not None else rows

        def reduced(t):
            return comm.allreduce_sum(t) if comm is not None else t

        mu.copy_(seed_rows(k)[None])
        cnt = reduced(torch.tensor([float(n_frames)], dtype=torch.float64, device=feats.device))
        m1 = reduced(feats.to(torch.float64).sum(dim=0)) / cnt
        m2 = reduced((feats.to(torch.float64) ** 2).sum(dim=0)) / cnt
        gvar = (m2 - m1 * m1).clamp_min(1e-12)
        # one spherical variance: the hard assignment is then the nearest centre in Euclidean distance
        sharp = (0.02 * gvar.mean()).expand(1, k, d).contiguous()
        w.fill_(1.0 / k)
        ms = ModelSet(w, mu, sharp, device=feats.device)
        for it in range(iters + 1):
            ms.repack(w, mu, sharp)
            n, _, _ = self._em_step(ms, feats, seg, workspace, nk_eps, w, mu, var)
            empty = (n[0] < 0.5).nonzero().flatten()
            if it == iters:
                # clusters still empty after the last Lloyd step would enter EM with mean 0 / var reg_covar; sklearn's
                # KMeans relocates them instead -- give each a frame far from every centre and the global variance
                if empty.numel():
                    mu[0, empty] = seed_rows(int(empty.numel()), avoid=mu[0])
                    var[0, empty] = gvar
                    w[0, empty] = 1.0 / n_frames if comm is None else 1.0 / float(cnt.item())
                    w /= w.sum()
                break
            w.fill_(1.0 / k)
            if empty.numel():
                mu[0, empty] = seed_rows(int(empty.numel()), avoid=mu[0])

    def _initial_parameters(self, feats, seg, rs, nk_eps, do_init=True, workspace=None):
        """(w (1,K), mu (1,K,D), var (1,K,D)) float64 on the device: warm start, k-means / random initialisation
        (sklearn/mixture/_base.py:120-129) and the user's ``*_init`` overrides."""
        torch = _lib.require_cuda()
        dev, (k, d) = feats.device, (self.n_components, feats.shape[1])
        w = torch.empty((1, k), dtype=torch.float64, device=dev)
        mu = torch.empty((1, k, d), dtype=torch.float64, device=dev)
        var = torch.empty((1, k, d), dtype=torch.float64, device=dev)
        if not do_init:
            w.copy_(torch.as_tensor(self.weights_)[None]); mu.copy_(torch.as_tensor(self.means_)[None])
            var.copy_(torch.as_tensor(self.covariances_)[None])
            return w, mu, var
        have_all = self.weights_init is not None and self.means_init is not None and self.precisions_init is not None
        if not have_all:
            if self.init_params not in ("kmeans", "k-means++", "random_from_data", "random"):
                raise ValueError(f"Invalid value for 'init_params': {self.init_params}")
            self._kmeans_init(feats, seg, rs, w, mu, var, nk_eps,
                              iters=10 if self.init_params in ("kmeans", "k-means++") else 0, workspace=workspace)
        if self.weights_init is not None:
            w.copy_(torch.as_tensor(np.asarray(self.weights_init, dtype=np.float64))[None])
        if self.means_init is not None:
            mu.copy_(torch.as_tensor(np.asarray(self.means_init, dtype=np.float64))[None])
        if self.precisions_init is not None:
            var.copy_(1.0 / torch.as_tensor(np.asarray(self.precisions_init, dtype=np.float64))[None])
        return w, mu, var

    def fit(self, X, y=None):
        """Estimate parameters with EM (sklearn/mixture/_base.py:203-312)."""
        self._fit(X)
        return self

    def fit_predict(self, X, y=None):
        """``fit(X)``, then the label of every frame from a final E-step under the best parameters (sklearn
        _base.py ``fit_predict``), so that it equals ``fit(X).predict(X)``.  The final E-step reuses the frames' operand
        images of the EM run."""
        feats, workspace = self._fit(X)
        _, labels, _ = self._model_set().posteriors(feats, np.array([0, feats.shape[0]]), resp=False, labels=True,
                                                    workspace=workspace, reuse_images=True)
        return labels.cpu().numpy()

    def _fit(self, X):
        """EM; returns the device frames and the :class:`StatsWorkspace` holding their operand images."""
        torch = _lib.require_cuda()
        self._check()
        dev = torch.device(f"cuda:{torch.cuda.current_device()}")
        feats = _as_feats(X, dev)
        seg = np.array([0, feats.shape[0]], dtype=np.int64)
        _check_sample_counts(np.diff(seg), self.n_components)
        nk_eps = _nk_eps(X)
        rs = self._rng()

        do_init = not (self.warm_start and hasattr(self, "converged_"))
        best = None
        workspace = StatsWorkspace(dev)  # the frames' operand images are built by the first statistics call and reused
        for _init in range(self.n_init if do_init else 1):
            w, mu, var = self._initial_parameters(feats, seg, rs, nk_eps, do_init, workspace)
            w, mu, var, lower, bounds, converged, n_iter = self._em(feats, seg, workspace, w, mu, var, nk_eps)
            if best is None or lower[0] > best[0] or best[0] == -np.inf:
                best = (lower[0], w[0], mu[0], var[0], n_iter[0], converged[0], bounds[0])
        lower, w, mu, var, n_iter, converged, bounds = best
        self._finish_em(w.cpu().numpy(), mu.cpu().numpy(), var.cpu().numpy(), converged, n_iter, lower, bounds)
        return feats, workspace

    # ------------------------------------------------------------------ scoring
    def score_samples(self, X):
        """Per-frame log-likelihood (sklearn/mixture/_base.py:373)."""
        ms = self._model_set()
        feats = _as_feats(X, ms.device)
        _, lse = ms.score(feats, np.array([0, feats.shape[0]]), precision=self.precision, want_frame_lse=True)
        return lse[0].cpu().numpy().astype(np.float64)

    def score(self, X, y=None):
        """Mean per-frame log-likelihood (sklearn/mixture/_base.py:393) -- what GMM_UBM.py:185 calls."""
        ms = self._model_set()
        feats = _as_feats(X, ms.device)
        scores, _ = ms.score(feats, np.array([0, feats.shape[0]]), precision=self.precision)
        return float(scores[0, 0].item())

    # ------------------------------------------------------------------ posteriors and model selection
    def _frames(self, X):
        ms = self._model_set()
        feats = _as_feats(X, ms.device)
        if feats.shape[1] != ms.n_feat:
            raise ValueError(f"X has {feats.shape[1]} features, but GaussianMixture is expecting {ms.n_feat} features as input.")
        return ms, feats

    def predict_proba(self, X):
        """Posterior of every component for every frame, float64 (T, K) (sklearn/mixture/_base.py ``predict_proba``).
        Computed at FP32 grade whatever ``precision`` says (``ssp_gmm_posteriors``), in frame chunks of at most
        ``PROBA_CHUNK_BYTES`` of device output, each copied into the host result as it completes."""
        ms, feats = self._frames(X)
        n, k = feats.shape[0], ms.n_comp
        out = np.empty((n, k), dtype=np.float64)
        step = max(1, PROBA_CHUNK_BYTES // (4 * k))
        workspace = StatsWorkspace(ms.device)
        for a in range(0, n, step):
            b = min(n, a + step)
            g, _, _ = ms.posteriors(feats[a:b], np.array([0, b - a]), resp=True, workspace=workspace)
            out[a:b] = g.cpu().numpy()
        return out

    def predict(self, X):
        """Most probable component of every frame, int64 (T,) (sklearn/mixture/_base.py ``predict``; the lowest index
        on ties).  FP32 grade whatever ``precision`` says."""
        ms, feats = self._frames(X)
        _, labels, _ = ms.posteriors(feats, np.array([0, feats.shape[0]]), resp=False, labels=True)
        return labels.cpu().numpy()

    def _n_parameters(self):
        """Free parameters of a diagonal model: K D variances, K D means and K - 1 weights."""
        k, d = np.shape(self.means_)
        return int(2 * k * d + k - 1)

    def bic(self, X):
        """Bayesian information criterion on X (sklearn/mixture/_gaussian_mixture.py ``bic``); lower is better."""
        n = int(X.shape[0]) if hasattr(X, "shape") else len(X)
        return -2.0 * self.score(X) * n + self._n_parameters() * np.log(n)

    def aic(self, X):
        """Akaike information criterion on X (sklearn/mixture/_gaussian_mixture.py ``aic``); lower is better."""
        n = int(X.shape[0]) if hasattr(X, "shape") else len(X)
        return -2.0 * self.score(X) * n + 2 * self._n_parameters()

    # ------------------------------------------------------------------ interchange (SURVEY 8(f).1)
    @classmethod
    def from_params(cls, weights, means, covariances, **kw):
        gm = cls(n_components=len(weights), **kw)
        gm._set_fitted(weights, means, covariances, True, 0, -np.inf)
        return gm

    @classmethod
    def from_sklearn(cls, sk, **kw):
        """Adopt a fitted (e.g. unpickled ``Model/GMM_MFCC_model.pkl``) sklearn GaussianMixture."""
        if sk.covariance_type != "diag":
            raise NotImplementedError("only diag covariances")
        return cls.from_params(sk.weights_, sk.means_, sk.covariances_, **kw)

    def to_sklearn(self):
        """A stock sklearn estimator carrying these parameters, so the reference's GUIs / pickles
        (UI/GMM_UBM_GUI.py:77-80) consume GPU-trained models unchanged."""
        from sklearn.mixture import GaussianMixture as SkGM

        sk = SkGM(n_components=self.n_components, covariance_type="diag", tol=self.tol, reg_covar=self.reg_covar,
                  max_iter=self.max_iter)
        sk.weights_, sk.means_, sk.covariances_ = self.weights_, self.means_, self.covariances_
        sk.precisions_cholesky_ = self.precisions_cholesky_
        sk.precisions_ = self.precisions_
        sk.converged_, sk.n_iter_, sk.lower_bound_ = self.converged_, self.n_iter_, self.lower_bound_
        sk.n_features_in_ = self.means_.shape[1]
        return sk


def fit_batch(X_list, n_components=1, **kwargs):
    """``[GaussianMixture(n_components, **kwargs).fit(X) for X in X_list]`` -- the per-speaker training loop of
    GMM_UBM.py:154-165 -- with the EM iterations of ALL models batched: one ``ssp_gmm_stats`` call per iteration scores
    segment s (speaker s's frames) under model s, one ``ssp_gmm_mstep`` launch updates every model, and ONE host
    read-back per iteration carries all lower bounds.  A model that has converged (sklearn's ``abs(change) < tol`` rule,
    per model) keeps the parameters of its converging iteration while the others go on, so every model ends with the
    ``n_iter_`` / parameters its own loop would have produced.  Initialisation (k-means or the ``*_init`` arguments,
    which may be per-model lists) runs per model, exactly as in :meth:`GaussianMixture.fit`.

    Returns the list of fitted :class:`GaussianMixture`.  ``n_init > 1``, ``warm_start`` and ``comm`` fall back to the
    plain loop."""
    torch = _lib.require_cuda()
    n_models = len(X_list)
    per_model = {key: kwargs.pop(key) for key in ("weights_init", "means_init", "precisions_init") if key in kwargs}

    def ctor_kwargs(i):
        out = dict(kwargs)
        for key, val in per_model.items():
            out[key] = None if val is None else (val[i] if isinstance(val, (list, tuple)) or np.ndim(val) == (3 if key != "weights_init" else 2) else val)
        return out

    gms = [GaussianMixture(n_components=n_components, **ctor_kwargs(i)) for i in range(n_models)]
    if n_models == 0:
        return gms
    g0 = gms[0]
    g0._check()
    if g0.n_init != 1 or g0.warm_start or g0.comm is not None or n_models > 1024:
        return [gm.fit(x) for gm, x in zip(gms, X_list)]
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    feats, seg = concat_utterances([np.asarray(x) if not isinstance(x, torch.Tensor) else x.cpu().numpy() for x in X_list], dev)
    d, k = feats.shape[1], n_components
    if 2 * d + 2 > 80:  # per-segment models need the tensor-core statistics kernels
        return [gm.fit(x) for gm, x in zip(gms, X_list)]
    _check_sample_counts(np.diff(seg), k)
    nk_eps = _nk_eps(X_list[0])
    # ---- initial parameters, per model (same code and RNG use as fit())
    w = torch.empty((n_models, k), dtype=torch.float64, device=dev)
    mu = torch.empty((n_models, k, d), dtype=torch.float64, device=dev)
    var = torch.empty((n_models, k, d), dtype=torch.float64, device=dev)
    for i, gm in enumerate(gms):
        fi = feats[int(seg[i]) : int(seg[i + 1])]
        wi, mi, vi = gm._initial_parameters(fi, np.array([0, fi.shape[0]], dtype=np.int64), gm._rng(), nk_eps, True, StatsWorkspace(dev))
        w[i], mu[i], var[i] = wi[0], mi[0], vi[0]
    # ---- batched EM
    w, mu, var, lower, bounds, converged, n_iter = g0._em(feats, seg, StatsWorkspace(dev), w, mu, var, nk_eps)
    hw, hmu, hvar = w.cpu().numpy(), mu.cpu().numpy(), var.cpu().numpy()
    for i, gm in enumerate(gms):
        gm._finish_em(hw[i], hmu[i], hvar[i], converged[i], n_iter[i], lower[i], bounds[i])
    return gms
