"""DTW oracle (dtw 1.4 ``accelerated_dtw`` restated in float64) and the host-only side of the GPU path.  No GPU needed."""
import ctypes as C

import numpy as np
import pytest

from oracle import dtw as odtw


def test_distance_to_itself_is_zero():
    x = np.random.RandomState(0).randn(17, 5)
    for dist in ("euclidean", "sqeuclidean", "cityblock"):
        d, cost, acc, (p, q) = odtw.accelerated_dtw(x, x, dist)
        assert d == 0.0
        assert (p == q).all() and len(p) == len(x)   # the diagonal


def test_repeated_frames_are_free():
    x = np.random.RandomState(1).randn(12, 3)
    stretched = np.repeat(x, [1, 3, 1, 2, 1, 1, 4, 1, 1, 2, 1, 1], axis=0)
    for dist in ("euclidean", "sqeuclidean", "cityblock"):
        assert odtw.accelerated_dtw(x, stretched, dist)[0] == 0.0
        assert odtw.accelerated_dtw(stretched, x, dist)[0] == 0.0


def test_hand_worked_cityblock():
    # C = |x_i - y_j| for x = [0, 1, 3], y = [0, 2, 3]:
    #   C = [[0, 2, 3], [1, 1, 2], [3, 1, 0]]
    #   D = [[0, 2, 5], [1, 1, 3], [4, 2, 1]]  ->  d = 1 along (0,0) (1,1) (2,2)
    d, cost, acc, (p, q) = odtw.accelerated_dtw(np.array([0.0, 1, 3]), np.array([0.0, 2, 3]), "cityblock")
    assert (cost == [[0, 2, 3], [1, 1, 2], [3, 1, 0]]).all()
    assert (acc == [[0, 2, 5], [1, 1, 3], [4, 2, 1]]).all()
    assert d == 1.0
    assert list(p) == [0, 1, 2] and list(q) == [0, 1, 2]
    # unequal lengths: x = [1, 2, 3, 3], y = [1, 3]: D = [[0, 2], [1, 1], [3, 1], [5, 1]] -> 1
    d, _, acc, (p, q) = odtw.accelerated_dtw(np.array([1.0, 2, 3, 3]), np.array([1.0, 3]), "cityblock")
    assert (acc == [[0, 2], [1, 1], [3, 1], [5, 1]]).all() and d == 1.0
    assert list(p) == [0, 1, 2, 3] and list(q) == [0, 0, 1, 1]   # from (2, 1), diagonal (1, 0) and up (1, 1) tie: diagonal


def test_length_one_special_cases():
    y = np.array([1.0, 4, 2, 2])
    d, cost, acc, path = odtw.accelerated_dtw(np.array([2.0]), y, "cityblock")
    assert d == 1 + 2 + 0 + 0 and (acc[0] == np.cumsum(cost[0])).all()
    assert (path[0] == 0).all() and list(path[1]) == [0, 1, 2, 3]
    d, cost, acc, path = odtw.accelerated_dtw(y, np.array([2.0]), "cityblock")
    assert d == 3 and list(path[0]) == [0, 1, 2, 3] and (path[1] == 0).all()


@pytest.mark.parametrize("dist", ["euclidean", "sqeuclidean", "cityblock"])
def test_loop_and_antidiagonal_oracles_agree(dist):
    rs = np.random.RandomState(2)
    for n, m, d in [(1, 1, 1), (1, 9, 2), (9, 1, 2), (23, 31, 13), (40, 7, 3), (33, 65, 1)]:
        x, y = rs.randn(n, d), rs.randn(m, d)
        _, cost, acc, _ = odtw.accelerated_dtw(x, y, dist)
        assert np.array_equal(odtw.accumulated_antidiag(cost), acc)
        assert odtw.dtw_distance_antidiag(x, y, dist) == acc[-1, -1]


def test_benchmark_reference_equals_the_oracle():
    """benchmarks/dtw_bench.py checks the GPU against its own float64 recurrence (scripts there do not import the
    oracle); it must be the oracle's."""
    from benchmarks.dtw_bench import dtw_float64

    rs = np.random.RandomState(5)
    for n, m, d in [(1, 1, 1), (1, 7, 13), (8, 1, 1), (37, 50, 13), (90, 33, 1)]:
        x, y = rs.randn(n, d), rs.randn(m, d)
        for dist in ("euclidean", "sqeuclidean", "cityblock"):
            assert dtw_float64(x, y, dist) == odtw.accelerated_dtw(x, y, dist)[0]


def test_path_properties():
    rs = np.random.RandomState(3)
    for n, m in [(2, 2), (5, 19), (30, 12), (41, 41)]:
        x, y = rs.randn(n, 4), rs.randn(m, 4)
        d, cost, acc, (p, q) = odtw.accelerated_dtw(x, y, "euclidean")
        assert (p[0], q[0]) == (0, 0) and (p[-1], q[-1]) == (n - 1, m - 1)
        steps = set(zip(np.diff(p), np.diff(q)))
        assert steps <= {(1, 0), (0, 1), (1, 1)}
        assert np.isclose(cost[p, q].sum(), d, rtol=1e-12)


def test_traceback_of_the_package_equals_the_oracle():
    """The host-side traceback of ``ssp.accelerated_dtw`` is the oracle's (same D, same tie rule)."""
    from speech_signal_processing_b200 import dtw

    rs = np.random.RandomState(4)
    for n, m in [(2, 3), (17, 9), (25, 40)]:
        x, y = rs.randint(0, 3, (n, 2)).astype(float), rs.randint(0, 3, (m, 2)).astype(float)   # many ties
        _, _, acc, path = odtw.accelerated_dtw(x, y, "cityblock")
        D0 = np.full((n + 1, m + 1), np.inf)
        D0[0, 0] = 0
        D0[1:, 1:] = acc
        got = dtw._traceback(D0)
        assert np.array_equal(got[0], path[0]) and np.array_equal(got[1], path[1])


@pytest.fixture(scope="module")
def lib():
    from speech_signal_processing_b200 import _lib, build

    build.build()
    return _lib.load()


def test_max_len_bounds(lib):
    lens = [int(lib.ssp_dtw_max_len(d)) for d in range(1, 65)]
    assert all(a >= b for a, b in zip(lens, lens[1:])), lens     # non-increasing in dim
    assert lens[0] >= 13 * 157            # flattened MFCC_lib output of a 10 s utterance at 8 kHz
    assert lens[38] >= 1000               # 1 000 frames of 39-d features
    assert lens[63] > 0
    assert lib.ssp_dtw_max_len(0) == 0 and lib.ssp_dtw_max_len(65) == 0
    from speech_signal_processing_b200 import dtw

    assert dtw.max_len(39) == lens[38]


def test_entry_points_reject_bad_arguments_without_the_gpu(lib):
    assert lib.ssp_dtw_batch(None, None, 1, None, None, 1, 13, 0, 10, None, None) == -1
    assert b"null" in lib.ssp_last_error()
    p = C.c_void_p(16)   # never dereferenced: the checks come first
    assert lib.ssp_dtw_batch(p, p, 1, p, p, 1, 13, 7, 10, p, None) == -1                       # unknown metric
    assert lib.ssp_dtw_batch(p, p, 1, p, p, 1, 13, 0, lib.ssp_dtw_max_len(13) + 1, p, None) == -3   # too long
    assert lib.ssp_dtw_full(p, 0, p, 3, 13, 0, p, p, None) == -1                                  # empty
    assert lib.ssp_dtw_full(p, 3, p, 3, 65, 0, p, p, None) == -3                                  # dim


def test_python_layer_validates_before_the_device():
    import speech_signal_processing_b200 as ssp

    with pytest.raises(NotImplementedError, match="euclidean"):
        ssp.accelerated_dtw(np.ones(3), np.ones(3), lambda a, b: 0.0)
    with pytest.raises(NotImplementedError):
        ssp.accelerated_dtw(np.ones(3), np.ones(3), "chebyshev")
    with pytest.raises(NotImplementedError, match="warp"):
        ssp.accelerated_dtw(np.ones(3), np.ones(3), "euclidean", warp=2)
    with pytest.raises(ValueError, match="empty"):
        ssp.accelerated_dtw(np.ones(0), np.ones(3), "euclidean")
    with pytest.raises(ValueError, match="widths"):
        ssp.accelerated_dtw(np.ones((3, 2)), np.ones((3, 3)), "euclidean")


def test_dtw_matrix_without_a_device_raises():
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(_lib.SspError, match="no CPU fallback"):
        ssp.dtw_matrix([np.ones((4, 2))], [np.ones((5, 2))])
