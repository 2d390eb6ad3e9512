"""Dynamic time warping on the GPU: the template-matching stage of the reference's MFCC+DTW recogniser.

``MFCC_DTW.py`` imports ``accelerated_dtw`` from the ``dtw`` package and runs it between every test utterance and
every template in a Python double loop, then takes the nearest template.  :func:`accelerated_dtw` is the drop-in for
one pair (dtw 1.4 semantics, float64 numpy out); :func:`dtw_matrix` / :func:`dtw_identify` are the batched form the
reference lacks: all pairs in one launch of ``dtw_kernel`` (``ssp_dtw_batch``).

Semantics (dtw 1.4, symmetric step pattern, no window, no slope weights): ``C = cdist(x, y, dist)`` for ``dist`` in
``'euclidean'``, ``'sqeuclidean'``, ``'cityblock'``; ``D[i, j] = C[i, j] + min(D[i-1, j-1], D[i-1, j], D[i, j-1])``
with ``D[-1, -1] = 0`` and the rest of row / column -1 at ``inf``; the distance is ``D[n-1, m-1]``.  The kernels
compute in FP32 (difference form, ~1e-6 relative).  ``fastdtw`` is not provided: it is an approximation, and an exact
replacement would change its results.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .mixture import concat_utterances

METRICS = {"euclidean": 0, "sqeuclidean": 1, "cityblock": 2}


def _metric(dist) -> int:
    if callable(dist) or not isinstance(dist, str) or dist not in METRICS:
        raise NotImplementedError(f"dist must be one of {sorted(METRICS)} (got {dist!r}); callables and other scipy "
                                  "metrics are not implemented on the GPU")
    return METRICS[dist]


def max_len(dim: int) -> int:
    """Longest sequence the kernels hold on their shared-memory side at this feature width (0: unsupported ``dim``).
    A pair needs only its SHORTER sequence within it (the distance is symmetric)."""
    return int(_lib.load().ssp_dtw_max_len(int(dim)))


def _sequence(a, what: str) -> np.ndarray:
    a = np.asarray(a)
    if a.ndim == 1:
        a = a.reshape(-1, 1)
    if a.ndim != 2:
        raise ValueError(f"{what}: expected a 1-D or 2-D array, got {a.ndim}-D")
    if len(a) == 0 or a.shape[1] == 0:
        raise ValueError(f"{what}: empty sequence")
    return np.ascontiguousarray(a, dtype=np.float32)


def _check_len(n: int, dim: int) -> None:
    limit = max_len(dim)
    if limit == 0:
        raise NotImplementedError(f"dim {dim} is not supported (1 <= dim <= 64)")
    if n > limit:
        raise NotImplementedError(f"sequences of {n} frames at dim {dim}: the shorter side of a pair may have at most "
                                  f"{limit} frames")


def _traceback(D0):
    """dtw 1.4 ``_traceback`` over the padded accumulated matrix: ties go to the diagonal, then i - 1, then j - 1."""
    i, j = np.array(D0.shape) - 2
    p, q = [i], [j]
    while i > 0 or j > 0:
        tb = np.argmin((D0[i, j], D0[i, j + 1], D0[i + 1, j]))
        if tb == 0:
            i -= 1
            j -= 1
        elif tb == 1:
            i -= 1
        else:
            j -= 1
        p.append(i)
        q.append(j)
    return np.array(p[::-1]), np.array(q[::-1])


def accelerated_dtw(x, y, dist, warp=1):
    """``dtw.accelerated_dtw`` (dtw 1.4): returns ``(d, C, D, path)`` as float64 numpy, ``path = (rows, cols)``.

    ``d = D[-1, -1]`` is not normalised (dtw < 1.4 returned ``D[-1, -1] / (n + m)``).  1-D inputs are ``(n, 1)``; an
    empty input is a ``ValueError``; a callable ``dist``, another metric name or ``warp != 1`` is
    ``NotImplementedError``.  ``C`` and ``D`` come from ``dtw_full_kernel``; the traceback runs on the host, O(n + m).
    """
    metric = _metric(dist)
    if warp != 1:
        raise NotImplementedError(f"warp={warp!r}: only warp=1 is implemented")
    x, y = _sequence(x, "x"), _sequence(y, "y")
    if x.shape[1] != y.shape[1]:
        raise ValueError(f"x and y have different feature widths ({x.shape[1]} and {y.shape[1]})")
    dim = x.shape[1]
    swap = len(y) > len(x)          # the shorter sequence goes to shared memory; D is exactly symmetric
    a, b = (y, x) if swap else (x, y)
    _check_len(len(b), dim)
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    da, db = torch.as_tensor(a, device=dev), torch.as_tensor(b, device=dev)
    cost = torch.empty((len(a), len(b)), dtype=torch.float32, device=dev)
    acc = torch.empty_like(cost)
    _lib.check(lib.ssp_dtw_full(_lib.ptr(da), len(a), _lib.ptr(db), len(b), dim, metric, _lib.ptr(cost), _lib.ptr(acc),
                                _lib.stream_ptr()), "ssp_dtw_full")
    C = cost.cpu().numpy().astype(np.float64)
    D = acc.cpu().numpy().astype(np.float64)
    if swap:
        C, D = np.ascontiguousarray(C.T), np.ascontiguousarray(D.T)
    if len(x) == 1:
        path = np.zeros(len(y)), range(len(y))
    elif len(y) == 1:
        path = range(len(x)), np.zeros(len(x))
    else:
        D0 = np.full((len(x) + 1, len(y) + 1), np.inf)
        D0[0, 0] = 0.0
        D0[1:, 1:] = D
        path = _traceback(D0)
    return D[-1, -1], C, D, path


def _ragged(seqs, dev, what):
    """list of (n_i, dim) / (n_i,) arrays, or a ``(device_feats, offsets)`` tuple -> (feats, offsets numpy, dim)."""
    torch = _lib.require_cuda()
    if isinstance(seqs, tuple) and len(seqs) == 2 and isinstance(seqs[0], torch.Tensor):
        feats, offs = seqs
        if feats.ndim != 2 or feats.dtype != torch.float32 or feats.device != dev:
            raise ValueError(f"{what}: device features must be a 2-D float32 tensor on {dev}")
        feats, offs = concat_utterances((feats, offs), dev)
        if len(offs) < 2 or offs[0] != 0 or offs[-1] != len(feats) or np.any(np.diff(offs) < 1):
            raise ValueError(f"{what}: offsets must start at 0, end at the frame count, and give every sequence a frame")
        return feats, offs, feats.shape[1]
    seqs = [_sequence(s, f"{what}[{k}]") for k, s in enumerate(seqs)]
    if not seqs:
        raise ValueError(f"{what}: no sequences")
    dim = seqs[0].shape[1]
    if any(s.shape[1] != dim for s in seqs):
        raise ValueError(f"{what}: sequences of different feature widths")
    feats, offs = concat_utterances(seqs, dev)
    return feats, offs, dim


def dtw_matrix(queries, templates, dist="euclidean", device=None):
    """``out[a, b] = accelerated_dtw(queries[a], templates[b], dist)[0]`` for all pairs in one ``dtw_kernel`` launch.

    ``queries`` / ``templates``: lists of ``(n, dim)`` (or 1-D) arrays, or ``(device_feats, offsets)`` tuples as
    :func:`score_matrix` takes them.  Whichever set has the shorter longest sequence is staged in shared memory, so
    that set's longest sequence must be within :func:`max_len` ``(dim)``.  Returns ``(n_q, n_r)`` float64 numpy."""
    metric = _metric(dist)
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    with torch.cuda.device(dev):
        qf, qo, qd = _ragged(queries, dev, "queries")
        rf, ro, rd = _ragged(templates, dev, "templates")
        if qd != rd:
            raise ValueError(f"queries and templates have different feature widths ({qd} and {rd})")
        q_max, r_max = int(np.diff(qo).max()), int(np.diff(ro).max())
        swap = q_max < r_max        # the set with the shorter longest sequence is the shared-memory side
        rows, row_offs, cols, col_offs = (rf, ro, qf, qo) if swap else (qf, qo, rf, ro)
        col_max = min(q_max, r_max)
        _check_len(col_max, qd)
        out = torch.empty((len(row_offs) - 1, len(col_offs) - 1), dtype=torch.float32, device=dev)
        d_row = torch.as_tensor(row_offs, device=dev)
        d_col = torch.as_tensor(col_offs, device=dev)
        _lib.check(lib.ssp_dtw_batch(_lib.ptr(rows), _lib.ptr(d_row), len(row_offs) - 1, _lib.ptr(cols), _lib.ptr(d_col),
                                     len(col_offs) - 1, qd, metric, col_max, _lib.ptr(out), _lib.stream_ptr()),
                   "ssp_dtw_batch")
        res = out.cpu().numpy().astype(np.float64)
    return np.ascontiguousarray(res.T) if swap else res


def dtw_identify(queries, templates, template_labels, dist="euclidean", device=None):
    """Nearest-template identification (MFCC_DTW.py's test loop): ``(distances, predicted_labels)`` where
    ``predicted_labels[a] = template_labels[argmin_b distances[a, b]]`` (the first minimum wins, as ``np.argmin``)."""
    labels = np.asarray(template_labels)
    d = dtw_matrix(queries, templates, dist=dist, device=device)
    if len(labels) != d.shape[1]:
        raise ValueError(f"{len(labels)} labels for {d.shape[1]} templates")
    return d, labels[np.argmin(d, axis=1)]
