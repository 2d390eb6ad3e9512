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


def concat_utterances(utts, device):
    """list of (T_i, D) arrays -> (feats (sum T, D) cuda, frame_offsets np.int64)."""
    torch = _lib.require_cuda()
    if isinstance(utts, tuple) and len(utts) == 2 and isinstance(utts[0], torch.Tensor):
        return utts[0].contiguous(), np.asarray(utts[1], dtype=np.int64)
    lens = np.array([len(u) for u in utts], dtype=np.int64)
    offs = np.zeros(len(utts) + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    d = np.asarray(utts[0]).shape[1]
    host = torch.empty((int(offs[-1]), d), dtype=torch.float32, pin_memory=True)
    hv = host.numpy()
    for u, o in zip(utts, offs[:-1]):
        hv[o : o + len(u)] = u
    return host.to(device, non_blocking=True), offs


class ModelSet:
    """``n_models`` diagonal GMMs with the same (K, D), packed once in HBM for the scoring kernels."""

    def __init__(self, weights, means, variances, device=None):
        torch = _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")

        def dev(a):
            if isinstance(a, torch.Tensor):
                return a.to(device=self.device, dtype=torch.float64).contiguous()
            return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=self.device)

        w, mu, var = dev(weights), dev(means), dev(variances)
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
        self.repack(w, mu, var)

    @_lib.on_device
    def repack(self, w, mu, var):
        """Re-derive the packed operands from (device, float64) parameters -- one tiny kernel."""
        self._params = (w, mu, var)
        _lib.check(self.lib.ssp_gmm_pack_models(_lib.ptr(w), _lib.ptr(mu), _lib.ptr(var), C.byref(self.dims),
                                                _lib.ptr(self.pack), _lib.stream_ptr()), "ssp_gmm_pack_models")

    # ---------------------------------------------------------------------------------------
    @_lib.on_device
    def score(self, feats, frame_offsets, precision="auto", want_frame_lse=False):
        """(scores (n_utts, n_models) cuda float64, frame_lse (n_models, total) cuda float32 | None).
        ``precision``: "fp32" (CUDA cores), "tf32" / "tf32x2" / "tf32x3" (tcgen05, 1 / 2 / 3 passes of 11-bit operands; the
        single pass streams FP16 images of the models) or "auto"
        (:func:`resolve_precision`)."""
        torch = _lib.require_cuda()
        frame_offsets = np.asarray(frame_offsets, dtype=np.int64)
        n_utts, total = len(frame_offsets) - 1, int(frame_offsets[-1])
        precision = resolve_precision(precision, self.n_comp, self.n_feat)
        if feats.shape[1] != self.n_feat:
            raise ValueError(f"X has {feats.shape[1]} features, but the models expect {self.n_feat}")
        d_off = torch.as_tensor(frame_offsets, device=self.device)
        scores = torch.empty((n_utts, self.n_models), dtype=torch.float64, device=self.device)
        lse = torch.empty((self.n_models, total), dtype=torch.float32, device=self.device) if want_frame_lse else None
        rc = self.lib.ssp_gmm_score(_lib.ptr(feats), _lib.ptr(d_off), n_utts, total, _lib.ptr(self.pack),
                                    C.byref(self.dims), PRECISIONS[precision], _lib.ptr(scores), _lib.ptr(lse),
                                    _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_score")
        self._keep = d_off
        return scores, lse

    @_lib.on_device
    def stats(self, feats, seg_offsets, workspace=None, reuse_images=False):
        """N (S,K), F (S,K,D), S2 (S,K,D), loglik (S,) float64 cuda: every segment under this set's single model, or
        -- if the set holds one model per segment -- segment s under model s (models trained together, :func:`fit_batch`).

        ``workspace``: a :class:`StatsWorkspace` shared between calls (and model sets) on the SAME ``feats`` /
        ``seg_offsets``; ``reuse_images=True`` then skips the preparation pass that turns the frames into tensor-core
        operand images (EM iterations: the frames never change).  Default: a workspace owned by this model set."""
        torch = _lib.require_cuda()
        seg_offsets = np.asarray(seg_offsets, dtype=np.int64)
        n_segs, total = len(seg_offsets) - 1, int(seg_offsets[-1])
        if self.n_models != 1 and self.n_models != n_segs:
            raise ValueError("statistics are taken under one model for all segments (the UBM), or under one model per "
                             f"segment (got {self.n_models} models for {n_segs} segments)")
        k, d = self.n_comp, self.n_feat
        n = torch.zeros((n_segs, k), dtype=torch.float64, device=self.device)
        f = torch.zeros((n_segs, k, d), dtype=torch.float64, device=self.device)
        s = torch.zeros((n_segs, k, d), dtype=torch.float64, device=self.device)
        ll = torch.zeros(n_segs, dtype=torch.float64, device=self.device)
        lse = torch.empty(max(total, 1), dtype=torch.float32, device=self.device)
        d_off = torch.as_tensor(seg_offsets, device=self.device)
        ws_bytes = int(self.lib.ssp_gmm_stats_workspace_bytes(C.byref(self.dims), total, n_segs))
        if workspace is None:
            workspace = getattr(self, "_ws", None)
            if workspace is None:
                workspace = self._ws = StatsWorkspace(self.device)
            reuse_images = False
        buf = workspace.reserve(ws_bytes)
        rc = self.lib.ssp_gmm_stats(_lib.ptr(feats), _lib.ptr(d_off), n_segs, total, _lib.ptr(self.pack),
                                    C.byref(self.dims), _lib.ptr(lse), _lib.ptr(n), _lib.ptr(f), _lib.ptr(s), _lib.ptr(ll),
                                    _lib.ptr(buf) if ws_bytes else None, ws_bytes, int(bool(reuse_images) and workspace.valid),
                                    _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_stats")
        workspace.valid = True
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
        seg_offsets = np.asarray(seg_offsets, dtype=np.int64)
        n_segs, total = len(seg_offsets) - 1, int(seg_offsets[-1])
        if self.n_models != 1 and self.n_models != n_segs:
            raise ValueError("posteriors are taken under one model for all segments, or under one model per segment "
                             f"(got {self.n_models} models for {n_segs} segments)")
        if feats.shape[1] != self.n_feat:
            raise ValueError(f"X has {feats.shape[1]} features, but the models expect {self.n_feat}")
        if not (resp or labels):
            raise ValueError("posteriors: ask for resp, labels or both")
        g = torch.empty((total, self.n_comp), dtype=torch.float32, device=self.device) if resp else None
        lab = torch.empty(total, dtype=torch.int64, device=self.device) if labels else None
        lse = torch.empty(total, dtype=torch.float32, device=self.device) if resp else None
        d_off = torch.as_tensor(seg_offsets, device=self.device)
        ws_bytes = int(self.lib.ssp_gmm_posteriors_workspace_bytes(C.byref(self.dims), total, n_segs))
        if workspace is None:
            workspace = getattr(self, "_ws", None)
            if workspace is None:
                workspace = self._ws = StatsWorkspace(self.device)
            reuse_images = False
        buf = workspace.reserve(ws_bytes)
        rc = self.lib.ssp_gmm_posteriors(_lib.ptr(feats), _lib.ptr(d_off), n_segs, total, _lib.ptr(self.pack),
                                         C.byref(self.dims), _lib.ptr(g), _lib.ptr(lab), _lib.ptr(lse),
                                         _lib.ptr(buf) if ws_bytes else None, ws_bytes,
                                         int(bool(reuse_images) and workspace.valid), _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_posteriors")
        workspace.valid = True
        self._keep = d_off
        return g, lab, lse


class StatsWorkspace:
    """Scratch of ``ssp_gmm_stats`` and ``ssp_gmm_posteriors`` (operand images of the frames + log-sum-exp partials; the
    two calls lay it out alike).  ``valid`` says that it holds the images of the frames it was last used with; growing it
    invalidates them."""

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

        def dev(a):
            if isinstance(a, torch.Tensor):
                return a.to(device=self.device, dtype=torch.float64).contiguous()
            return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=self.device)

        w, var, mu = dev(weights), dev(variances), dev(means)
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
        self._ws = None

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
        frame_offsets = np.asarray(frame_offsets, dtype=np.int64)
        n_utts, total = len(frame_offsets) - 1, int(frame_offsets[-1])
        if feats.shape[1] != self.n_feat:
            raise ValueError(f"X has {feats.shape[1]} features, but the models expect {self.n_feat}")
        d_off = torch.as_tensor(frame_offsets, device=self.device)
        scores = torch.empty((n_utts, self.n_models), dtype=torch.float64, device=self.device)
        lse = torch.empty((self.n_models, total), dtype=torch.float32, device=self.device) if want_frame_lse else None
        ws_bytes = int(self.lib.ssp_gmm_score_shared_workspace_bytes(C.byref(self.dims), total))
        if ws_bytes and (self._ws is None or self._ws.numel() < ws_bytes):
            self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        rc = self.lib.ssp_gmm_score_shared(_lib.ptr(feats), _lib.ptr(d_off), n_utts, total, _lib.ptr(self.pack),
                                           C.byref(self.dims), _lib.ptr(scores), _lib.ptr(lse),
                                           _lib.ptr(self._ws) if ws_bytes else None, ws_bytes, _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_score_shared")
        self._keep = d_off
        return scores, lse

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
    ms = models if isinstance(models, ModelSet) else ModelSet(
        np.stack([np.asarray(m.weights_) for m in models]), np.stack([np.asarray(m.means_) for m in models]),
        np.stack([np.asarray(m.covariances_) for m in models]), device=dev)
    feats, offs = concat_utterances(utts, dev)
    scores, _ = ms.score(feats, offs, precision=precision)
    return scores.cpu().numpy()


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

    def _set_params_from_device(self, w, mu, var):
        self.weights_ = w.cpu().numpy()
        self.means_ = mu.cpu().numpy()
        self.covariances_ = var.cpu().numpy()
        self.precisions_cholesky_ = 1.0 / np.sqrt(self.covariances_)
        self.precisions_ = self.precisions_cholesky_ ** 2

    # ------------------------------------------------------------------ EM
    def _em_iteration(self, ms, feats, seg, n_total, nk_eps, w, mu, var, workspace=None):
        """One E+M step on device.  Returns the lower bound (mean frame log-likelihood under the
        parameters the E-step used)."""
        torch = _lib.require_cuda()
        n, f, s, ll = ms.stats(feats, seg, workspace=workspace, reuse_images=True)
        if self.comm is not None and self.comm.world_size > 1:
            k, d = ms.n_comp, ms.n_feat
            cnt = torch.tensor([float(feats.shape[0])], dtype=torch.float64, device=feats.device)
            flat = torch.cat([n.reshape(-1), f.reshape(-1), s.reshape(-1), ll.reshape(-1), cnt])
            timing = getattr(self, "allreduce_events", None)  # bench.py: a list to append (start, end) CUDA events to
            if timing is not None:
                timing.append((torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)))
                timing[-1][0].record()
            flat = self.comm.allreduce_sum(flat)
            if timing is not None:
                timing[-1][1].record()
            n, f, s = flat[:k].reshape(1, k), flat[k : k + k * d].reshape(1, k, d), flat[k + k * d : k + 2 * k * d].reshape(1, k, d)
            ll, n_total = flat[k + 2 * k * d : k + 2 * k * d + 1], float(flat[-1].item())
        rc = ms.lib.ssp_gmm_mstep(_lib.ptr(n), _lib.ptr(f), _lib.ptr(s), 1, ms.n_comp, ms.n_feat, float(self.reg_covar),
                                  float(nk_eps), _lib.ptr(w), _lib.ptr(mu), _lib.ptr(var), _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_mstep")
        return float(ll.item()) / n_total, n

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
            n, f, s, _ = ms.stats(feats, seg, workspace=workspace, reuse_images=True)
            if comm is not None:
                flat = reduced(torch.cat([n.reshape(-1), f.reshape(-1), s.reshape(-1)]))
                n, f, s = flat[:k].reshape(1, k), flat[k : k + k * d].reshape(1, k, d), flat[k + k * d :].reshape(1, k, d)
            rc = ms.lib.ssp_gmm_mstep(_lib.ptr(n), _lib.ptr(f), _lib.ptr(s), 1, k, d, float(self.reg_covar), float(nk_eps),
                                      _lib.ptr(w), _lib.ptr(mu), _lib.ptr(var), _lib.stream_ptr())
            _lib.check(rc, "ssp_gmm_mstep")
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
        x_dtype = X.dtype if isinstance(X, np.ndarray) and X.dtype in (np.float32, np.float64) else np.float64
        if isinstance(X, torch.Tensor):
            x_dtype = np.float32 if X.dtype == torch.float32 else np.float64
        feats = _as_feats(X, dev)
        n_frames, d = feats.shape
        k = self.n_components
        if n_frames < 2:
            raise ValueError(f"Found array with {n_frames} sample(s) while a minimum of 2 is required.")
        if n_frames < k:
            raise ValueError("Expected n_samples >= n_components "
                             f"but got n_components = {k}, n_samples = {n_frames}")
        nk_eps = 10.0 * float(np.finfo(x_dtype).eps)
        seg = np.array([0, n_frames], dtype=np.int64)
        rs = self.random_state if isinstance(self.random_state, np.random.RandomState) else np.random.RandomState(self.random_state)

        do_init = not (self.warm_start and hasattr(self, "converged_"))
        best = None
        workspace = StatsWorkspace(dev)  # the frames' operand images are built by the first statistics call and reused
        for _init in range(self.n_init if do_init else 1):
            w, mu, var = self._initial_parameters(feats, seg, rs, nk_eps, do_init, workspace)
            ms = ModelSet(w, mu, var, device=dev)
            lower, bounds, converged, n_iter = -np.inf, [], False, 0
            for n_iter in range(1, self.max_iter + 1):
                prev = lower
                ms.repack(w, mu, var)
                lower, _ = self._em_iteration(ms, feats, seg, float(n_frames), nk_eps, w, mu, var, workspace)
                bounds.append(lower)
                if abs(lower - prev) < self.tol:
                    converged = True
                    break
            if best is None or lower > best[0] or best[0] == -np.inf:
                best = (lower, w.clone(), mu.clone(), var.clone(), n_iter, converged, bounds)
        lower, w, mu, var, n_iter, converged, bounds = best
        if not converged and self.max_iter > 0:
            warnings.warn("Best performing initialization did not converge. Try different init parameters, or "
                          "increase max_iter, tol, or check for degenerate data.", UserWarning)
        self._set_params_from_device(w[0], mu[0], var[0])
        if not np.all(np.isfinite(self.covariances_)) or np.any(self.covariances_ <= 0):
            raise ValueError("Fitting the mixture model failed because some components have ill-defined empirical "
                             "covariance (for instance caused by singleton or collapsed samples). Try to decrease the "
                             "number of components, increase reg_covar, or scale the input data.")
        self.converged_, self.n_iter_, self.lower_bound_, self.lower_bounds_ = converged, n_iter, lower, bounds
        self._ms = None
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
        gm.weights_ = np.asarray(weights, dtype=np.float64)
        gm.means_ = np.asarray(means, dtype=np.float64)
        gm.covariances_ = np.asarray(covariances, dtype=np.float64)
        gm.precisions_cholesky_ = 1.0 / np.sqrt(gm.covariances_)
        gm.precisions_ = gm.precisions_cholesky_ ** 2
        gm.converged_, gm.n_iter_, gm.lower_bound_ = True, 0, -np.inf
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
    counts = np.diff(seg)
    for cnt in counts:
        if cnt < 2:
            raise ValueError(f"Found array with {cnt} sample(s) while a minimum of 2 is required.")
        if cnt < k:
            raise ValueError(f"Expected n_samples >= n_components but got n_components = {k}, n_samples = {cnt}")
    x_dtypes = [np.float32 if (isinstance(x, torch.Tensor) and x.dtype == torch.float32) or
                (isinstance(x, np.ndarray) and x.dtype == np.float32) else np.float64 for x in X_list]
    nk_eps = 10.0 * float(np.finfo(x_dtypes[0]).eps)
    # ---- initial parameters, per model (same code and RNG use as fit())
    w = torch.empty((n_models, k), dtype=torch.float64, device=dev)
    mu = torch.empty((n_models, k, d), dtype=torch.float64, device=dev)
    var = torch.empty((n_models, k, d), dtype=torch.float64, device=dev)
    for i, gm in enumerate(gms):
        rs = gm.random_state if isinstance(gm.random_state, np.random.RandomState) else np.random.RandomState(gm.random_state)
        fi = feats[int(seg[i]) : int(seg[i + 1])]
        wi, mi, vi = gm._initial_parameters(fi, np.array([0, fi.shape[0]], dtype=np.int64), rs, nk_eps, True, StatsWorkspace(dev))
        w[i], mu[i], var[i] = wi[0], mi[0], vi[0]
    # ---- batched EM
    ms = ModelSet(w, mu, var, device=dev)
    workspace = StatsWorkspace(dev)
    t_counts = torch.as_tensor(counts.astype(np.float64), device=dev)
    w_new, mu_new, var_new = torch.empty_like(w), torch.empty_like(mu), torch.empty_like(var)
    lower = np.full(n_models, -np.inf)
    bounds = [[] for _ in range(n_models)]
    converged = np.zeros(n_models, dtype=bool)
    n_iter = np.zeros(n_models, dtype=np.int64)
    for it in range(1, g0.max_iter + 1):
        active = ~converged
        if not active.any():
            break
        ms.repack(w, mu, var)
        n, f, s, ll = ms.stats(feats, seg, workspace=workspace, reuse_images=True)
        rc = ms.lib.ssp_gmm_mstep(_lib.ptr(n), _lib.ptr(f), _lib.ptr(s), n_models, k, d, float(g0.reg_covar), float(nk_eps),
                                  _lib.ptr(w_new), _lib.ptr(mu_new), _lib.ptr(var_new), _lib.stream_ptr())
        _lib.check(rc, "ssp_gmm_mstep")
        now = (ll / t_counts).cpu().numpy()          # the one host synchronisation of the iteration
        keep = torch.as_tensor(active, device=dev)
        w = torch.where(keep[:, None], w_new, w)
        mu = torch.where(keep[:, None, None], mu_new, mu)
        var = torch.where(keep[:, None, None], var_new, var)
        for i in np.nonzero(active)[0]:
            bounds[i].append(float(now[i]))
            n_iter[i] = it
            if abs(now[i] - lower[i]) < g0.tol:
                converged[i] = True
            lower[i] = now[i]
    hw, hmu, hvar = w.cpu().numpy(), mu.cpu().numpy(), var.cpu().numpy()
    for i, gm in enumerate(gms):
        if not converged[i] and gm.max_iter > 0:
            warnings.warn("Best performing initialization did not converge. Try different init parameters, or "
                          "increase max_iter, tol, or check for degenerate data.", UserWarning)
        gm.weights_, gm.means_, gm.covariances_ = hw[i], hmu[i], hvar[i]
        gm.precisions_cholesky_ = 1.0 / np.sqrt(gm.covariances_)
        gm.precisions_ = gm.precisions_cholesky_ ** 2
        if not np.all(np.isfinite(gm.covariances_)) or np.any(gm.covariances_ <= 0):
            raise ValueError("Fitting the mixture model failed because some components have ill-defined empirical "
                             "covariance (for instance caused by singleton or collapsed samples). Try to decrease the "
                             "number of components, increase reg_covar, or scale the input data.")
        gm.converged_, gm.n_iter_, gm.lower_bound_, gm.lower_bounds_ = bool(converged[i]), int(n_iter[i]), float(lower[i]), bounds[i]
        gm._ms = None
    return gms
