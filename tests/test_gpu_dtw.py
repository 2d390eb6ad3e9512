"""DTW on the GPU (``dtw_kernel`` / ``dtw_full_kernel``) against the float64 oracle of dtw 1.4 ``accelerated_dtw``."""
import numpy as np
import pytest

from oracle import dtw as odtw

pytestmark = pytest.mark.gpu

# The kernels accumulate C and D in FP32 along a path of up to n + m cells of non-negative terms (no cancellation):
# the relative deviation from float64 measured over this file's sets is ~1e-6 (ragged sets, lengths 1..400); the bound
# leaves an order of magnitude of headroom.
RTOL = 2e-5
METRICS = ("euclidean", "sqeuclidean", "cityblock")


@pytest.fixture(scope="module")
def ssp():
    import speech_signal_processing_b200 as ssp

    return ssp


def _ragged(rs, count, dim, lo=1, hi=400):
    lens = rs.randint(lo, hi + 1, size=count)
    lens[0], lens[-1] = lo, hi
    return [rs.randn(n, dim).astype(np.float32) for n in lens]


@pytest.mark.parametrize("dim", [1, 13, 26, 39])
def test_dtw_matrix_matches_oracle_on_ragged_sets(ssp, dim):
    rs = np.random.RandomState(dim)
    Q, R = _ragged(rs, 6, dim), _ragged(rs, 5, dim)
    worst = 0.0
    for dist in METRICS:
        got = ssp.dtw_matrix(Q, R, dist)
        want = odtw.dtw_matrix([q.astype(np.float64) for q in Q], [r.astype(np.float64) for r in R], dist)
        assert got.shape == (6, 5) and got.dtype == np.float64
        rel = np.abs(got - want) / np.maximum(want, 1e-30)
        worst = max(worst, float(rel.max()))
        assert rel.max() <= RTOL, (dist, rel.max())
    print(f"dim {dim}: max relative deviation {worst:.2e}")


def _int_seq(rs, n, dim):
    return rs.randint(0, 4, size=(n, dim)).astype(np.float64)


@pytest.mark.parametrize("dist", ["cityblock", "sqeuclidean"])
def test_accelerated_dtw_is_exact_on_integer_data(ssp, dist):
    """Integer data: every C, D value is an integer below 2^24, exact in FP32, so d, C, D and the path (with the
    many ties small integers make) equal the float64 oracle bit for bit."""
    rs = np.random.RandomState(7)
    shapes = [(1, 1), (1, 9), (9, 1), (2, 2), (31, 33), (33, 31), (32, 32), (70, 45), (45, 70), (130, 3), (5, 200)]
    for n, m in shapes:
        for dim in (1, 3):
            x, y = _int_seq(rs, n, dim), _int_seq(rs, m, dim)
            if dim == 1:
                x, y = x[:, 0], y[:, 0]    # 1-D inputs are (n, 1)
            d, C, D, path = ssp.accelerated_dtw(x, y, dist)
            rd, rC, rD, rpath = odtw.accelerated_dtw(x, y, dist)
            assert d == rd and np.array_equal(C, rC) and np.array_equal(D, rD), (n, m, dim)
            assert C.dtype == np.float64 and D.shape == (n, m)
            assert np.array_equal(np.asarray(path[0]), np.asarray(rpath[0]))
            assert np.array_equal(np.asarray(path[1]), np.asarray(rpath[1]))


def test_a_pair_does_not_depend_on_the_batch_and_roles_swap_exactly(ssp):
    rs = np.random.RandomState(11)
    Q = _ragged(rs, 9, 13, hi=150)
    R = _ragged(rs, 7, 13, hi=90)       # shorter longest sequence: R is the shared-memory side
    for dist in METRICS:
        full = ssp.dtw_matrix(Q, R, dist)
        sub = ssp.dtw_matrix([Q[5], Q[2]], [R[6], R[0], R[3]], dist)
        assert np.array_equal(sub, full[np.ix_([5, 2], [6, 0, 3])])
        single = ssp.dtw_matrix([Q[4]], [R[1]], dist)
        assert single[0, 0] == full[4, 1]
        assert np.array_equal(ssp.dtw_matrix(R, Q, dist), full.T)
        # a set with the longer longest sequence on the template side takes the other role
        assert np.array_equal(ssp.dtw_matrix([R[2], R[0]], Q, dist), full[:, [2, 0]].T)
        # the drop-in computes the same distance as the batched kernel
        assert ssp.accelerated_dtw(Q[4], R[1], dist)[0] == full[4, 1]


def test_device_tuple_inputs(ssp):
    import torch

    from speech_signal_processing_b200.mixture import concat_utterances

    rs = np.random.RandomState(12)
    Q, R = _ragged(rs, 4, 13, hi=60), _ragged(rs, 3, 13, hi=60)
    dev = torch.device("cuda", torch.cuda.current_device())
    want = ssp.dtw_matrix(Q, R)
    assert np.array_equal(ssp.dtw_matrix(concat_utterances(Q, dev), concat_utterances(R, dev)), want)


def test_length_bound_and_errors(ssp):
    from speech_signal_processing_b200 import dtw

    rs = np.random.RandomState(13)
    for dim in (1, 39):
        L = dtw.max_len(dim)
        a, b = rs.randn(L, dim), rs.randn(L + 1, dim)
        got = ssp.dtw_matrix([a], [b, a[:7]], "sqeuclidean")      # the shorter side of every pair is within the bound
        assert np.isfinite(got).all()
        if dim == 39:
            assert np.isclose(got[0, 1], odtw.dtw_distance_antidiag(a.astype(np.float32), a[:7].astype(np.float32),
                                                                    "sqeuclidean"), rtol=RTOL)
        with pytest.raises(NotImplementedError, match="frames"):
            ssp.dtw_matrix([b], [b])
        d, C, D, _ = ssp.accelerated_dtw(a[:300], b, "cityblock")
        assert D.shape == (300, L + 1) and d == D[-1, -1]
        with pytest.raises(NotImplementedError):
            ssp.accelerated_dtw(b, b, "euclidean")
    x = rs.randn(5, 13)
    with pytest.raises(ValueError, match="empty"):
        ssp.dtw_matrix([x, x[:0]], [x])
    with pytest.raises(ValueError, match="empty"):
        ssp.accelerated_dtw(x[:0], x, "euclidean")
    with pytest.raises(ValueError, match="widths"):
        ssp.dtw_matrix([x], [rs.randn(5, 12)])
    with pytest.raises(ValueError, match="widths"):
        ssp.accelerated_dtw(x, rs.randn(5, 12), "euclidean")
    with pytest.raises(NotImplementedError):
        ssp.dtw_matrix([x], [x], dist=lambda u, v: 0.0)
    with pytest.raises(NotImplementedError):
        ssp.accelerated_dtw(x, x, lambda u, v: 0.0)
    with pytest.raises(NotImplementedError, match="warp"):
        ssp.accelerated_dtw(x, x, "euclidean", warp=2)
    with pytest.raises(NotImplementedError):
        ssp.dtw_matrix([rs.randn(4, 65)], [rs.randn(4, 65)])


def test_identify_synthetic_words(ssp):
    """MFCC_DTW.py's recogniser on synthetic "words" (one class per synthetic speaker): 8 kHz audio of 1-3 s,
    ``ssp.MFCC`` features (512 / 256), three templates per class; the GPU's nearest template is the float64 oracle's
    for every query whose top-2 margin exceeds the tolerance."""
    from speech_signal_processing_b200 import synth

    rs = np.random.RandomState(14)
    x, y = synth.synth_corpus(6, 8, 24000, fs=8000)
    feats = [ssp.MFCC(s[: rs.randint(8000, 24001)], fs=8000) for s in x]
    is_template = np.tile(np.arange(8) < 3, 6)
    T = [f for f, t in zip(feats, is_template) if t]
    T_lab = [c for c, t in zip(y, is_template) if t]
    Q = [f for f, t in zip(feats, is_template) if not t]
    Q_lab = np.array([c for c, t in zip(y, is_template) if not t])
    d, pred = ssp.dtw_identify(Q, T, T_lab)
    want = odtw.dtw_matrix([q.astype(np.float32).astype(np.float64) for q in Q],
                           [t.astype(np.float32).astype(np.float64) for t in T], "euclidean")
    assert np.abs(d - want).max() <= RTOL * want.max()
    top2 = np.sort(want, axis=1)[:, :2]
    clear = (top2[:, 1] - top2[:, 0]) > 2 * RTOL * top2[:, 1]
    assert clear.sum() >= len(Q) // 2
    ref = np.asarray(T_lab)[np.argmin(want, axis=1)]
    assert (pred[clear] == ref[clear]).all()
    print(f"{clear.sum()} of {len(Q)} queries with a clear margin; accuracy {(pred == Q_lab).mean():.2f}")


def test_launch_log_names_the_kernels(ssp):
    from speech_signal_processing_b200 import _lib

    rs = np.random.RandomState(15)
    _lib.load().ssp_reset_launch_count()
    ssp.dtw_matrix([rs.randn(20, 13)], [rs.randn(30, 13), rs.randn(10, 13)])
    assert _lib.launch_log() == {"dtw_kernel": 1}
    _lib.load().ssp_reset_launch_count()
    ssp.accelerated_dtw(rs.randn(20, 13), rs.randn(30, 13), "euclidean")
    assert _lib.launch_log() == {"dtw_full_kernel": 1}
