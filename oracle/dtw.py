"""Float64 restatement of dtw 1.4 ``accelerated_dtw`` (the ``dtw`` package MFCC_DTW.py imports) -- TEST
INFRASTRUCTURE ONLY.

``dtw`` is absent here and unpinned in the reference's requirements: **parity unpinned**.  Restated from the
package's published 1.4 source:

* 1-D inputs become ``(n, 1)``; ``C = cdist(x, y, dist)``;
* ``D0`` is ``(n + 1, m + 1)`` with ``D0[0, 0] = 0`` and the rest of row / column 0 at ``inf``; with ``warp = 1``
  ``D0[i+1, j+1] = C[i, j] + min(D0[i, j], D0[i, j+1], D0[i+1, j])`` (diagonal, up, left);
* the distance is ``D[-1, -1]`` (dtw < 1.4 divided it by ``n + m``);
* the path is the traceback from the end cell, ``argmin`` of (diagonal, up, left) -- the first minimum wins -- and a
  length-1 input on either side is special-cased.

:func:`accelerated_dtw` is the literal loop; :func:`dtw_distance_antidiag` computes the same ``D`` one anti-diagonal
at a time with numpy (larger sizes, and the CPU arm of ``benchmarks/dtw_bench.py``).
"""
from __future__ import annotations

import numpy as np
from scipy.spatial.distance import cdist


def _as_2d(a):
    a = np.asarray(a, dtype=np.float64)
    return a.reshape(-1, 1) if a.ndim == 1 else a


def traceback(D0):
    """The package's ``_traceback`` over the padded matrix ``D0``."""
    i, j = np.array(D0.shape) - 2
    p, q = [i], [j]
    while (i > 0) or (j > 0):
        tb = np.argmin((D0[i, j], D0[i, j + 1], D0[i + 1, j]))
        if tb == 0:
            i -= 1
            j -= 1
        elif tb == 1:
            i -= 1
        else:
            j -= 1
        p.insert(0, i)
        q.insert(0, j)
    return np.array(p), np.array(q)


def accelerated_dtw(x, y, dist, warp=1):
    """``(d, C, D, path)`` exactly as the package's loop computes it (float64)."""
    assert len(x)
    assert len(y)
    x, y = _as_2d(x), _as_2d(y)
    r, c = len(x), len(y)
    D0 = np.zeros((r + 1, c + 1))
    D0[0, 1:] = np.inf
    D0[1:, 0] = np.inf
    D1 = D0[1:, 1:]
    D0[1:, 1:] = cdist(x, y, dist)
    C = D1.copy()
    for i in range(r):
        for j in range(c):
            min_list = [D0[i, j]]
            for k in range(1, warp + 1):
                min_list += [D0[min(i + k, r), j], D0[i, min(j + k, c)]]
            D1[i, j] += min(min_list)
    if len(x) == 1:
        path = np.zeros(len(y)), range(len(y))
    elif len(y) == 1:
        path = range(len(x)), np.zeros(len(x))
    else:
        path = traceback(D0)
    return D1[-1, -1], C, D1, path


def accumulated_antidiag(C):
    """``D`` of the warp-1 recurrence over the cost matrix ``C``, one anti-diagonal per numpy step."""
    n, m = C.shape
    D0 = np.full((n + 1, m + 1), np.inf)
    D0[0, 0] = 0.0
    for s in range(n + m - 1):           # cells with i + j == s
        i = np.arange(max(0, s - m + 1), min(n, s + 1))
        j = s - i
        D0[i + 1, j + 1] = C[i, j] + np.minimum(D0[i, j], np.minimum(D0[i, j + 1], D0[i + 1, j]))
    return D0[1:, 1:]


def dtw_distance_antidiag(x, y, dist="euclidean"):
    """DTW distance (float64) through :func:`accumulated_antidiag`."""
    return float(accumulated_antidiag(cdist(_as_2d(x), _as_2d(y), dist))[-1, -1])


def dtw_matrix(queries, templates, dist="euclidean"):
    """``(n_q, n_r)`` float64 distances, pair by pair."""
    return np.array([[dtw_distance_antidiag(q, t, dist) for t in templates] for q in queries])
