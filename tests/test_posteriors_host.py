"""Host-side checks of the posterior entry points (size query, argument checks, no CPU fallback) and of the float64
predict / predict_proba / bic / aic restatements the GPU tests use, against live sklearn 1.9.  Runs without a GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import gmm as ogmm


def predict(x, weights, means, variances):
    """sklearn _base.py ``predict`` restated in float64: argmax of the weighted log-probability (lowest index on ties)."""
    return ogmm.weighted_log_prob(x, weights, means, variances).argmax(axis=1)


def n_parameters(n_comp, n_feat):
    """_gaussian_mixture.py ``_n_parameters`` (diag): K D variances + K D means + K - 1 weights."""
    return 2 * n_comp * n_feat + n_comp - 1


def bic(x, weights, means, variances):
    """_gaussian_mixture.py ``bic``: -2 n score + p log n."""
    n, (k, d) = np.asarray(x).shape[0], np.shape(means)
    return -2.0 * ogmm.score(x, weights, means, variances) * n + n_parameters(k, d) * np.log(n)


def aic(x, weights, means, variances):
    """_gaussian_mixture.py ``aic``: -2 n score + 2 p."""
    n, (k, d) = np.asarray(x).shape[0], np.shape(means)
    return -2.0 * ogmm.score(x, weights, means, variances) * n + 2 * n_parameters(k, d)


@pytest.fixture(scope="module")
def lib():
    from speech_signal_processing_b200 import _lib, build

    build.build()
    return _lib.load()


def test_workspace_query(lib):
    from speech_signal_processing_b200 import _lib

    q = lib.ssp_gmm_posteriors_workspace_bytes
    for dims in [(1, 16, 81), (0, 16, 13), (1, 0, 13), (1, 16, 0), (2, 16, 40)]:
        assert q(C.byref(_lib.GmmDims(*dims)), 1000, 2) == 0, dims
    assert q(None, 1000, 1) == 0
    assert q(C.byref(_lib.GmmDims(1, 16, 13)), -1, 1) == 0
    assert q(C.byref(_lib.GmmDims(1, 16, 13)), 10, -1) == 0
    # tensor-core widths: the layout (and size) of the statistics workspace, so one buffer serves both calls
    for dims, t, s in [((1, 512, 39), 100000, 1), ((7, 129, 13), 5000, 7), ((1, 1, 1), 1, 1)]:
        d = C.byref(_lib.GmmDims(*dims))
        assert q(d, t, s) == lib.ssp_gmm_stats_workspace_bytes(d, t, s) > 0
    # CUDA-core widths: per-segment sums and the per-frame log-likelihood
    assert q(C.byref(_lib.GmmDims(1, 64, 40)), 1000, 3) >= 4 * 1000 + 8 * 3


def test_null_arguments_fail_without_touching_the_gpu(lib):
    from speech_signal_processing_b200 import _lib

    d = _lib.GmmDims(1, 16, 13)
    fake = C.c_void_p(4096)  # never dereferenced: every check below fails before any device work
    f = lib.ssp_gmm_posteriors
    assert f(None, None, 1, 10, None, None, fake, None, None, None, 0, 0, None) == -1
    assert f(None, None, 1, 10, None, C.byref(d), None, None, None, None, 0, 0, None) == -1
    assert b"NULL" in lib.ssp_last_error()
    assert f(None, None, 1, 10, None, C.byref(d), fake, None, None, None, 0, 0, None) == -1
    assert b"null" in lib.ssp_last_error()
    assert f(fake, fake, 1, 10, fake, C.byref(d), None, fake, None, None, 0, 0, None) == -1
    assert b"workspace" in lib.ssp_last_error()
    assert f(fake, fake, 2, 10, fake, C.byref(_lib.GmmDims(3, 16, 13)), fake, None, None, fake, 1 << 20, 0, None) == -1
    assert f(fake, fake, -1, 10, fake, C.byref(d), fake, None, None, fake, 1 << 20, 0, None) == -1


def test_methods_have_no_cpu_fallback():
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib, synth

    if torch.cuda.is_available():
        pytest.skip("checks the behaviour without a CUDA device")
    w, mu, var = synth.synth_ubm(4, 3, seed=0)
    x = synth.sample_gmm(w, mu, var, 50, seed=1)
    gm = ssp.GaussianMixture.from_params(w, mu, var)
    for fn in (gm.predict_proba, gm.predict, gm.bic, gm.aic, ssp.GaussianMixture(n_components=4).fit_predict):
        with pytest.raises(_lib.SspError, match="no CPU fallback"):
            fn(x)
    with pytest.raises(AttributeError):
        ssp.GaussianMixture(n_components=4).predict(x)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_float64_restatements_match_sklearn(dtype):
    from sklearn.mixture import GaussianMixture as SkGM

    from speech_signal_processing_b200 import synth

    k, d = 12, 7
    w, mu, var = synth.synth_ubm(k, d, seed=3, spread=1.0)
    x = synth.sample_gmm(w, mu, var, 3000, seed=4).astype(dtype)
    sk = SkGM(n_components=k, covariance_type="diag")
    sk.weights_, sk.means_, sk.covariances_ = w, mu, var
    sk.precisions_cholesky_ = 1.0 / np.sqrt(var)
    sk.precisions_ = 1.0 / var
    sk.n_features_in_ = d
    # sklearn squares float32 frames in float32; the oracle works in float64 throughout
    atol = 1e-5 if dtype == np.float32 else 1e-12
    np.testing.assert_allclose(ogmm.responsibilities(x, w, mu, var)[1], sk.predict_proba(x), rtol=0, atol=atol)
    wlp = np.sort(ogmm.weighted_log_prob(x, w, mu, var), axis=1)
    ok = wlp[:, -1] - wlp[:, -2] > 1e-3
    assert ok.mean() > 0.99
    np.testing.assert_array_equal(predict(x, w, mu, var)[ok], sk.predict(x)[ok])
    if dtype == np.float64:
        np.testing.assert_array_equal(predict(x, w, mu, var), sk.predict(x))
    assert n_parameters(k, d) == sk._n_parameters()
    rtol = 1e-6 if dtype == np.float32 else 1e-12
    np.testing.assert_allclose(bic(x, w, mu, var), sk.bic(x), rtol=rtol)
    np.testing.assert_allclose(aic(x, w, mu, var), sk.aic(x), rtol=rtol)
