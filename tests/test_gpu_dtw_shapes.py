"""DTW kernels (``dtw_kernel`` / ``dtw_full_kernel``) at every feature-width bucket and at the size bounds, against the
float64 oracle of dtw 1.4 ``accelerated_dtw``.

The kernels are compiled once per width bucket (``dim_bucket`` in ``csrc/dtw.cu``): each bucket has its own unrolled
cost loop, zero padding and shared-memory row stride.  The tests that need no device (the oracle helper, the coverage
guard) run everywhere; the others are marked ``gpu`` one by one.
"""
import os
import time

import numpy as np
import pytest
from scipy.spatial.distance import cdist

from oracle import dtw as odtw

# Same bound as tests/test_gpu_dtw.py: FP32 sums of non-negative terms along a path of up to n + m cells.  A numpy
# emulation of the FP32 recurrence (C rounded to FP32, FP32 min-plus, anti-diagonal order) stayed within 3e-6 at
# 6 456 x 6 000 frames, dim 1, for all three metrics.
RTOL = 2e-5
METRICS = ("euclidean", "sqeuclidean", "cityblock")
# the top of every width bucket and the first width of the next (the coverage guard below derives the buckets)
WIDTHS = [1, 2, 3, 4, 5, 8, 9, 13, 14, 16, 17, 20, 21, 26, 27, 32, 33, 39, 40, 48, 49, 63, 64]
BUCKET_TOPS = [1, 2, 4, 8, 13, 16, 20, 26, 32, 39, 48, 64]
# one width per bucket for the bit-exact test: the first of each, so that all but the two narrowest pad
EXACT_WIDTHS = [1, 2, 3, 5, 9, 14, 17, 21, 27, 33, 40, 49]
# sequence lengths around the 32-row strips of a warp and the M = max(m, 32) steps between two rows of a lane
EDGE_LENS = [1, 2, 31, 32, 33, 63, 64, 65, 97]
# warps that serve more than one row-side sequence: launch_db caps grid.y at 65 535 CTAs of 8 warps
GRID_Y_ROWS = 65535 * 8
# the overflow test runs one warp for over 2^31 serial steps (271 s on a B200 at 1 000 W); it runs
# only when this variable is set to a non-empty value
LONG_ENV = "SSP_TEST_DTW_LONG"


@pytest.fixture(scope="module")
def lib():
    from speech_signal_processing_b200 import _lib, build

    build.build()
    return _lib.load()


@pytest.fixture(scope="module")
def ssp():
    import speech_signal_processing_b200 as ssp

    return ssp


def _cost(a, b, dist):
    """Row-wise local cost of frame pairs a[k], b[k] (float64)."""
    d = a - b
    if dist == "cityblock":
        return np.abs(d).sum(axis=1)
    s = (d * d).sum(axis=1)
    return np.sqrt(s) if dist == "euclidean" else s


def dtw_distance_two_diagonals(x, y, dist):
    """float64 DTW distance of dtw 1.4 keeping only the last two anti-diagonals of the padded accumulated matrix D0
    (O(n + m) memory: the full D of a 6 456 x 6 456 pair is 330 MB).  Entry a of a diagonal array is row a of D0."""
    x = np.asarray(x, dtype=np.float64).reshape(len(x), -1)
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    n, m = len(x), len(y)
    d2 = np.full(n + 1, np.inf)      # padded diagonal t - 2
    d1 = np.full(n + 1, np.inf)      # padded diagonal t - 1 (diagonal 1 is all border)
    d2[0] = 0.0                      # D0[0, 0]
    cur = np.empty(n + 1)
    for t in range(2, n + m + 1):    # cells D0[a, t - a] with 1 <= a <= n, 1 <= t - a <= m
        a = np.arange(max(1, t - m), min(n, t - 1) + 1)
        cur.fill(np.inf)
        cur[a] = _cost(x[a - 1], y[t - a - 1], dist) + np.minimum(d2[a - 1], np.minimum(d1[a - 1], d1[a]))
        d2, d1, cur = d1, cur, d2
    return float(d1[n])


def _buckets(lib):
    """[(first, top)] of every width bucket: ssp_dtw_max_len(dim) divides the shared memory by a per-frame size that
    depends on the bucket only (its row stride is distinct for every bucket), so it changes exactly where the bucket
    does; it is 0 beyond the widest."""
    lens = []
    while lib.ssp_dtw_max_len(len(lens) + 1) > 0:
        lens.append(int(lib.ssp_dtw_max_len(len(lens) + 1)))
    out, first = [], 1
    for d in range(1, len(lens) + 1):
        if d == len(lens) or lens[d] != lens[d - 1]:
            out.append((first, d))
            first = d + 1
    return out


# ------------------------------------------------------------------------------------------------ no device needed
def test_width_lists_cover_every_bucket(lib):
    buckets = _buckets(lib)
    assert len(buckets) >= 12 and buckets[0][0] == 1
    assert [top for _, top in buckets] == BUCKET_TOPS
    for first, top in buckets:
        assert top in WIDTHS, (first, top)
        assert sum(first <= w <= top for w in EXACT_WIDTHS) == 1, (first, top)
    for (_, top), (first, _) in zip(buckets, buckets[1:]):
        assert first == top + 1 and first in WIDTHS
    assert max(WIDTHS) == buckets[-1][1] and all(lib.ssp_dtw_max_len(w) > 0 for w in WIDTHS)


@pytest.mark.parametrize("dist", METRICS)
def test_two_diagonal_helper_equals_the_oracle(dist):
    rs = np.random.RandomState(1)
    for n, m, d in [(1, 1, 1), (1, 7, 3), (9, 1, 2), (2, 2, 1), (33, 31, 5), (40, 97, 13), (65, 64, 1)]:
        x, y = rs.randn(n, d), rs.randn(m, d)
        want = odtw.accumulated_antidiag(cdist(x, y, dist))[-1, -1]
        # the local costs are summed in another order than cdist's: equal to the last bits
        assert np.isclose(dtw_distance_two_diagonals(x, y, dist), want, rtol=1e-13, atol=0)
        assert np.isclose(dtw_distance_two_diagonals(y, x, dist), odtw.accelerated_dtw(y, x, dist)[0], rtol=1e-13, atol=0)


# ------------------------------------------------------------------------------------------------ GPU
def _rel(got, want):
    return np.abs(got - want) / np.maximum(np.abs(want), 1e-30)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", WIDTHS)
def test_every_bucket_on_boundary_lengths(ssp, dim):
    rs = np.random.RandomState(100 + dim)
    Q = [rs.randn(n, dim).astype(np.float32) for n in rs.permutation(EDGE_LENS)]
    R = [rs.randn(n, dim).astype(np.float32) for n in EDGE_LENS[::-1]]
    worst = 0.0
    for dist in METRICS:
        got = ssp.dtw_matrix(Q, R, dist)
        want = odtw.dtw_matrix([q.astype(np.float64) for q in Q], [r.astype(np.float64) for r in R], dist)
        rel = _rel(got, want)
        worst = max(worst, float(rel.max()))
        assert rel.max() <= RTOL, (dist, rel.max())
        # one longer template moves the queries to the shared-memory side: the same distances, bit for bit
        longer = rs.randn(98, dim).astype(np.float32)
        swapped = ssp.dtw_matrix(Q, R + [longer], dist)
        assert np.array_equal(swapped[:, : len(R)], got)
    print(f"dim {dim}: worst relative deviation {worst:.2e}")


def _int_seq(rs, n, dim):
    return rs.randint(0, 4, size=(n, dim)).astype(np.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", EXACT_WIDTHS)
@pytest.mark.parametrize("dist", ["cityblock", "sqeuclidean"])
def test_accelerated_dtw_is_exact_at_every_bucket(ssp, dim, dist):
    """Values in {0..3}: every C and D entry is an integer below 2^24 (at most 9 * 64 per cell over < 400 cells), exact
    in FP32, so d, C, D and the path (with the many ties of small integers) equal the float64 oracle bit for bit."""
    rs = np.random.RandomState(dim)
    for n, m in [(1, 1), (1, 33), (33, 1), (2, 2), (31, 33), (33, 31), (32, 32), (64, 65), (97, 63), (130, 3), (5, 200)]:
        x, y = _int_seq(rs, n, dim), _int_seq(rs, m, dim)
        d, C, D, path = ssp.accelerated_dtw(x, y, dist)
        rd, rC, rD, rpath = odtw.accelerated_dtw(x, y, dist)
        assert d == rd and np.array_equal(C, rC) and np.array_equal(D, rD), (n, m)
        assert np.array_equal(np.asarray(path[0]), np.asarray(rpath[0])), (n, m)
        assert np.array_equal(np.asarray(path[1]), np.asarray(rpath[1])), (n, m)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", BUCKET_TOPS)
def test_template_at_the_length_bound(ssp, dim):
    """A template of exactly max_len(dim) frames (the shared-memory side at its largest dynamic allocation) against a
    longer row-side query and a short one."""
    from speech_signal_processing_b200 import dtw

    L = dtw.max_len(dim)
    dist = METRICS[dim % 3]
    rs = np.random.RandomState(200 + dim)
    t = rs.randn(L, dim).astype(np.float32)
    q_long, q_short = rs.randn(L + 33, dim).astype(np.float32), rs.randn(97, dim).astype(np.float32)
    got = ssp.dtw_matrix([q_long, q_short], [t], dist)[:, 0]
    want = np.array([dtw_distance_two_diagonals(q, t, dist) for q in (q_long, q_short)])
    rel = _rel(got, want)
    print(f"dim {dim} ({dist}), template {L} frames: relative deviation {rel[0]:.2e} (query {L + 33} frames), "
          f"{rel[1]:.2e} (query 97 frames)")
    assert rel.max() <= RTOL, rel


@pytest.mark.gpu
def test_accelerated_dtw_at_the_length_bound(ssp):
    """dtw_full_kernel with its largest dynamic shared memory: x of exactly max_len(64) frames is the shorter sequence
    (the shared-memory side), y a little longer.  Integer data keeps every value exact, so C, D and the path equal
    the oracle's bit for bit."""
    from speech_signal_processing_b200 import dtw

    L = dtw.max_len(64)
    rs = np.random.RandomState(64)
    x, y = _int_seq(rs, L, 64), _int_seq(rs, L + 5, 64)
    d, C, D, path = ssp.accelerated_dtw(x, y, "sqeuclidean")
    rd, rC, rD, rpath = odtw.accelerated_dtw(x, y, "sqeuclidean")
    assert D.shape == (L, L + 5) and rD.max() < 2 ** 24
    assert d == rd and np.array_equal(C, rC) and np.array_equal(D, rD)
    assert np.array_equal(np.asarray(path[0]), rpath[0]) and np.array_equal(np.asarray(path[1]), rpath[1])


@pytest.mark.gpu
def test_warps_loop_over_more_rows_than_grid_y_holds(ssp):
    """More row-side sequences than 65 535 x 8 warps: a warp serves sequences q and q + 524 280 one after the other
    and reuses its row buffer.  Long sequences sit on both sides of that index (some in the same warp, one after
    the other); every other sequence has one frame, whose distance is the closed form sum_j C[0, j]."""
    import torch

    from speech_signal_processing_b200 import _lib

    dim, n_rows = 5, GRID_Y_ROWS + 40_000
    rs = np.random.RandomState(300)
    lens = np.ones(n_rows, dtype=np.int64)
    long_idx = np.array([0, 7, 1000, 300_001, GRID_Y_ROWS - 1, GRID_Y_ROWS, GRID_Y_ROWS + 7, GRID_Y_ROWS + 1000,
                         GRID_Y_ROWS + 39_999])
    lens[long_idx] = rs.randint(33, 101, size=len(long_idx))
    lens[long_idx[0]] = 100
    offs = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    x = rs.randn(int(offs[-1]), dim).astype(np.float32)
    T = [rs.randn(m, dim).astype(np.float32) for m in (1, 31, 32, 33, 64, 80)]   # all shorter than the longest query
    dev = torch.device("cuda", torch.cuda.current_device())
    _lib.load().ssp_reset_launch_count()
    got = ssp.dtw_matrix((torch.as_tensor(x, device=dev), offs), T, "euclidean")
    assert _lib.launch_log() == {"dtw_kernel": 1}
    assert got.shape == (n_rows, len(T))
    single = np.setdiff1d(np.arange(n_rows), long_idx)
    xs = x[offs[single]].astype(np.float64)
    for b, t in enumerate(T):
        want = np.zeros(len(single))
        for row in t.astype(np.float64):
            want += np.sqrt(((xs - row) ** 2).sum(axis=1))
        assert _rel(got[single, b], want).max() <= RTOL, b
    Q_long = [x[offs[i] : offs[i + 1]] for i in long_idx]
    want = odtw.dtw_matrix([q.astype(np.float64) for q in Q_long], [t.astype(np.float64) for t in T], "euclidean")
    assert _rel(got[long_idx], want).max() <= RTOL
    assert np.array_equal(got[long_idx], ssp.dtw_matrix(Q_long, T, "euclidean"))


@pytest.mark.gpu
@pytest.mark.skipif(not os.environ.get(LONG_ENV),
                    reason=f"over 2^31 serial steps of one warp: 271 s on a B200; set {LONG_ENV}=1 to run it")
def test_step_count_beyond_int32(ssp):
    """A 6 456-frame template and a row of 10 644 257 frames at dim 1: ceil(n / 32) * 6 456 + 31 steps exceed
    INT32_MAX (the first row length that does).  Constant sequences one apart under cityblock: every C is 1 and the
    distance is exactly n, an integer below 2^24."""
    from speech_signal_processing_b200 import dtw

    L, n = dtw.max_len(1), 10_644_257
    assert L == 6456 and -(-n // 32) * L + 31 > 2 ** 31 - 1
    t0 = time.perf_counter()
    got = ssp.dtw_matrix([np.ones(n, dtype=np.float32)], [np.zeros(L, dtype=np.float32)], "cityblock")
    print(f"{n} x {L} frames: {time.perf_counter() - t0:.1f} s")
    assert got[0, 0] == n
