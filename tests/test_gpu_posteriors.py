"""Frame posteriors and labels on the GPU (``ssp_gmm_posteriors``, ``ModelSet.posteriors`` and the sklearn methods
``predict_proba`` / ``predict`` / ``fit_predict`` / ``bic`` / ``aic``) against sklearn 1.9 and the float64 oracle, at the
tile and tile-pair edges of K, on both sides of the tensor-core / CUDA-core width bound, on ragged and per-model
segments, with the kernels that served each call asserted."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import speech_signal_processing_b200 as ssp  # noqa: E402
from oracle import gmm as ogmm  # noqa: E402
from speech_signal_processing_b200 import _lib, mixture, synth  # noqa: E402

# Stated bounds (FP32-grade logits: 3 x BF16 tensor products for D <= 39, FP32 FMA above): every posterior within
# PROBA_ATOL of float64, every row sum within ROWSUM_ATOL of 1.  Labels are compared on the frames whose float64 top-2
# margin of the weighted log-probability exceeds MARGIN.
PROBA_ATOL = 1e-4
ROWSUM_ATOL = 2e-5
MARGIN = 1e-3
# the per-frame log-likelihood that comes with the posteriors: the FP32-grade tolerance of test_gpu_gmm.py
LSE_RTOL = 5e-5

LSE = {"em_plan_kernel", "em_prep_kernel", "gmm_em_lse_kernel", "em_merge_kernel"}
TENSOR = {
    "resp": LSE | {"gmm_em_post_kernel<resp>"},
    "labels": {"em_plan_kernel", "em_prep_kernel", "gmm_em_post_kernel<labels>", "em_label_merge_kernel"},
    "both": LSE | {"gmm_em_post_kernel<resp+labels>", "em_label_merge_kernel"},
}
SIMT = {"resp": {"gmm_score_simt_kernel", "gmm_post_simt_kernel"}, "labels": {"gmm_post_simt_kernel"},
        "both": {"gmm_score_simt_kernel", "gmm_post_simt_kernel"}}


def torch():
    return _lib.require_cuda()


def reference(x, w, mu, var):
    """float64 (frame lse, gamma, labels, top-2 margin) of the weighted log-probability."""
    wlp = ogmm.weighted_log_prob(x, w, mu, var)
    lse = ogmm.logsumexp(wlp, axis=1)
    top = np.sort(wlp, axis=1)[:, -2:] if wlp.shape[1] > 1 else np.concatenate([wlp - np.inf, wlp], axis=1)
    return lse, np.exp(wlp - lse[:, None]), wlp.argmax(axis=1), top[:, 1] - top[:, 0]


def check(case, got_g, got_lab, x, w, mu, var, got_lse=None):
    lse, g, lab, margin = reference(x, w, mu, var)
    msg = f"{case}:"
    if got_g is not None:
        err = float(np.abs(got_g - g).max()) if g.size else 0.0
        rs = float(np.abs(got_g.sum(axis=1) - 1.0).max()) if g.size else 0.0
        msg += f" max|gamma - f64| {err:.2e}, max|row sum - 1| {rs:.2e}"
        assert err <= PROBA_ATOL, msg
        assert rs <= ROWSUM_ATOL, msg
    if got_lse is not None:
        lerr = float((np.abs(got_lse - lse) / np.maximum(1.0, np.abs(lse))).max())
        msg += f", frame lse {lerr:.2e} rel"
        assert lerr <= LSE_RTOL, msg
    if got_lab is not None:
        ok = margin > MARGIN
        msg += f", labels on {int(ok.sum())} of {len(ok)} frames ({int((~ok).sum())} below the margin)"
        np.testing.assert_array_equal(got_lab[ok], lab[ok], err_msg=msg)
    print(msg)


def model(k, d, seed):
    w, mu, var = synth.synth_ubm(k, d, seed=seed, spread=1.0)
    return w, mu, var


def frames(w, mu, var, lens, seed):
    x = synth.sample_gmm(w, mu, var, int(sum(lens)), seed=seed)
    offs = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    return x, offs


# ------------------------------------------------------------------------------------------------ sklearn parity
@pytest.mark.parametrize("tag", ["s", "m"])
def test_predict_proba_matches_sklearn_fixture(golden, tag):
    g = golden("sklearn_gmm.npz")
    gm = ssp.GaussianMixture.from_params(g[f"{tag}_w"], g[f"{tag}_mu"], g[f"{tag}_var"], precision="tf32")
    got = gm.predict_proba(g[f"{tag}_x"])
    assert got.dtype == np.float64 and got.shape == g[f"{tag}_proba"].shape
    err = float(np.abs(got - g[f"{tag}_proba"]).max())
    rs = float(np.abs(got.sum(axis=1) - 1).max())
    print(f"fixture {tag}: max|gamma - sklearn| {err:.2e}, max|row sum - 1| {rs:.2e}")
    assert err <= PROBA_ATOL and rs <= ROWSUM_ATOL
    lab = gm.predict(g[f"{tag}_x"])
    assert lab.dtype == np.int64
    check(f"fixture {tag} labels", None, lab, g[f"{tag}_x"], g[f"{tag}_w"], g[f"{tag}_mu"], g[f"{tag}_var"])


def sk_model(w, mu, var):
    from sklearn.mixture import GaussianMixture as SkGM

    sk = SkGM(n_components=len(w), covariance_type="diag")
    sk.weights_, sk.means_, sk.covariances_ = w, mu, var
    sk.precisions_cholesky_ = 1.0 / np.sqrt(var)
    sk.precisions_ = 1.0 / var
    sk.n_features_in_ = mu.shape[1]
    sk.converged_, sk.n_iter_, sk.lower_bound_ = True, 0, -np.inf
    return sk


@pytest.mark.parametrize("tag", ["s", "m", "l"])
def test_predict_proba_predict_bic_aic_match_live_sklearn(golden, tag):
    g = golden("sklearn_gmm.npz")
    w, mu, var, x = g[f"{tag}_w"], g[f"{tag}_mu"], g[f"{tag}_var"], g[f"{tag}_x"]
    sk = sk_model(w, mu, var)
    gm = ssp.GaussianMixture.from_params(w, mu, var)
    err = float(np.abs(gm.predict_proba(x) - sk.predict_proba(x)).max())
    print(f"live sklearn {tag}: max|gamma - sklearn| {err:.2e}")
    assert err <= PROBA_ATOL
    _, _, _, margin = reference(x, w, mu, var)
    ok = margin > MARGIN
    print(f"live sklearn {tag}: labels compared on {int(ok.sum())} of {len(ok)} frames")
    np.testing.assert_array_equal(gm.predict(x)[ok], sk.predict(x)[ok])
    k, d = mu.shape
    assert gm._n_parameters() == sk._n_parameters() == 2 * k * d + k - 1
    for fn in ("bic", "aic"):
        want = getattr(sk, fn)(x)
        assert abs(getattr(gm, fn)(x) - want) <= 1e-6 * abs(want), fn


def test_errors_follow_sklearn():
    w, mu, var = model(4, 5, 0)
    with pytest.raises(AttributeError):
        ssp.GaussianMixture(n_components=4).predict_proba(np.zeros((3, 5)))
    with pytest.raises(AttributeError):
        ssp.GaussianMixture(n_components=4).predict(np.zeros((3, 5)))
    gm = ssp.GaussianMixture.from_params(w, mu, var)
    for fn in (gm.predict_proba, gm.predict):
        with pytest.raises(ValueError):
            fn(np.zeros((3, 4), dtype=np.float32))


def test_duplicated_component_gives_equal_posteriors_and_the_lower_label():
    for d in (13, 40):
        w, mu, var = model(8, d, 1)
        mu[5], var[5] = mu[2], var[2]
        w[5] = w[2]
        w /= w.sum()
        x = (mu[2] + 0.3 * np.random.RandomState(2).standard_normal((500, d))).astype(np.float32)
        gm = ssp.GaussianMixture.from_params(w, mu, var)
        g = gm.predict_proba(x)
        np.testing.assert_array_equal(g[:, 2], g[:, 5])
        lab = gm.predict(x)
        assert (lab == 2).sum() > 400 and not (lab == 5).any(), np.bincount(lab)


def test_fit_predict_equals_fit_then_predict():
    w, mu, var = model(16, 13, 3)
    x = synth.sample_gmm(w, mu, var, 6000, seed=4)
    gm = ssp.GaussianMixture(n_components=16, random_state=0, max_iter=20)
    lab = gm.fit_predict(x)
    assert lab.dtype == np.int64 and lab.shape == (6000,)
    np.testing.assert_array_equal(lab, gm.predict(x))
    check("fit_predict", None, lab, x, gm.weights_, gm.means_, gm.covariances_)


@pytest.mark.parametrize("tag", ["s", "m"])
def test_fit_predict_from_fixed_init_matches_sklearn(golden, tag):
    from sklearn.mixture import GaussianMixture as SkGM

    g = golden("sklearn_gmm.npz")
    w, mu, var, x = g[f"{tag}_w"], g[f"{tag}_mu"], g[f"{tag}_var"], g[f"{tag}_x"]
    kw = dict(n_components=len(w), covariance_type="diag", weights_init=w, means_init=mu, precisions_init=1.0 / var,
              max_iter=100)
    sk = SkGM(**kw)
    want = sk.fit_predict(x)
    got = ssp.GaussianMixture(**kw).fit_predict(x)
    _, _, _, margin = reference(x, sk.weights_, sk.means_, sk.covariances_)
    ok = margin > MARGIN
    print(f"fit_predict {tag}: labels compared on {int(ok.sum())} of {len(ok)} frames")
    np.testing.assert_array_equal(got[ok], want[ok])


# ------------------------------------------------------------------------------------------------ bounds
@pytest.mark.parametrize("d", [1, 13, 26, 39, 40, 80])
@pytest.mark.parametrize("k", [1, 127, 128, 129, 255, 256, 257, 1024])
def test_posteriors_at_every_bound(k, d):
    w, mu, var = model(k, d, 10 + k + d)
    x, offs = frames(w, mu, var, [1, 63, 64, 65, 300, 2, 129], seed=k * 100 + d)
    ms = ssp.ModelSet(w, mu, var)
    feats = torch().as_tensor(x, device="cuda")
    want = TENSOR if d <= 39 else SIMT
    for mode, (resp, labels) in {"resp": (True, False), "labels": (False, True), "both": (True, True)}.items():
        lib = _lib.load()
        lib.ssp_reset_launch_count()
        g, lab, lse = ms.posteriors(feats, offs, resp=resp, labels=labels)
        assert set(_lib.launch_log()) == want[mode], (mode, _lib.launch_log())
        assert (g is None) != resp and (lab is None) != labels and (lse is None) != resp
        check(f"K={k} D={d} {mode}", None if g is None else g.cpu().numpy(), None if lab is None else lab.cpu().numpy(),
              x, w, mu, var, None if lse is None else lse.cpu().numpy())


@pytest.mark.parametrize("k,d", [(129, 26), (256, 39), (64, 13)])
def test_per_segment_models(k, d):
    lens = [1, 63, 64, 65, 300, 128]
    params = [model(k, d, 50 + s) for s in range(len(lens))]
    x = np.concatenate([synth.sample_gmm(*params[s], n, seed=60 + s) for s, n in enumerate(lens)])
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    ms = ssp.ModelSet(*(np.stack([p[i] for p in params]) for i in range(3)))
    _lib.load().ssp_reset_launch_count()
    g, lab, lse = ms.posteriors(torch().as_tensor(x, device="cuda"), offs, resp=True, labels=True)
    assert set(_lib.launch_log()) == TENSOR["both"]
    g, lab, lse = g.cpu().numpy(), lab.cpu().numpy(), lse.cpu().numpy()
    for s in range(len(lens)):
        a, b = offs[s], offs[s + 1]
        check(f"per-segment K={k} D={d} segment {s} ({b - a} frames)", g[a:b], lab[a:b], x[a:b], *params[s], got_lse=lse[a:b])


def test_many_segments_under_one_model():
    w, mu, var = model(200, 20, 7)
    lens = np.random.RandomState(8).randint(1, 140, size=700)
    lens[::50] = 0
    x, offs = frames(w, mu, var, lens, seed=9)
    g, lab, lse = ssp.ModelSet(w, mu, var).posteriors(torch().as_tensor(x, device="cuda"), offs, resp=True, labels=True)
    check(f"{len(lens)} segments", g.cpu().numpy(), lab.cpu().numpy(), x, w, mu, var, lse.cpu().numpy())


@pytest.mark.parametrize("k,d,n_models", [(129, 13, 1), (256, 13, 1), (128, 39, 3), (100, 40, 1), (256, 80, 1)])
def test_padding_is_never_written(k, d, n_models):
    """Canary-filled outputs larger than T x K / T: only the live frames and components are written."""
    t = torch()
    lens = [1, 63, 64, 65, 300] if n_models == 1 else [65, 1, 130]
    params = [model(k, d, 70 + s) for s in range(n_models)]
    x = np.concatenate([synth.sample_gmm(*params[s % n_models], n, seed=80 + s) for s, n in enumerate(lens)])
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    ms = ssp.ModelSet(*(np.stack([p[i] for p in params]) for i in range(3)))
    total, pad = int(offs[-1]), 4096
    resp = t.full((total * k + pad,), -7.0, dtype=t.float32, device="cuda")
    lab = t.full((total + pad,), -7, dtype=t.int64, device="cuda")
    lse = t.full((total + pad,), -7.0, dtype=t.float32, device="cuda")
    lib = _lib.load()
    ws_bytes = int(lib.ssp_gmm_posteriors_workspace_bytes(C.byref(ms.dims), total, len(lens)))
    ws = t.empty(ws_bytes, dtype=t.uint8, device="cuda")
    feats, d_off = t.as_tensor(x, device="cuda"), t.as_tensor(offs, device="cuda")
    rc = lib.ssp_gmm_posteriors(feats.data_ptr(), d_off.data_ptr(), len(lens), total, ms.pack.data_ptr(), C.byref(ms.dims),
                                resp.data_ptr(), lab.data_ptr(), lse.data_ptr(), ws.data_ptr(), ws_bytes, 0, _lib.stream_ptr())
    _lib.check(rc, "ssp_gmm_posteriors")
    r, lb, ls = resp.cpu().numpy(), lab.cpu().numpy(), lse.cpu().numpy()
    assert (r[total * k:] == -7.0).all() and (lb[total:] == -7).all() and (ls[total:] == -7.0).all()
    assert not (r[: total * k] == -7.0).any() and not (lb[:total] == -7).any()
    g = r[: total * k].reshape(total, k)
    for s in range(len(lens)):
        a, b = offs[s], offs[s + 1]
        check(f"canary K={k} D={d} models={n_models} segment {s}", g[a:b], lb[a:b], x[a:b], *params[s % n_models],
              got_lse=ls[a:b])


# ------------------------------------------------------------------------------------------------ sharing and errors
def test_stats_then_posteriors_share_the_frame_images():
    w, mu, var = model(300, 39, 11)
    x, offs = frames(w, mu, var, [1000, 77, 2500], seed=12)
    feats = torch().as_tensor(x, device="cuda")
    ms = ssp.ModelSet(w, mu, var)
    fresh = ms.posteriors(feats, offs, resp=True, labels=True)
    ws = mixture.StatsWorkspace(ms.device)
    ms.stats(feats, offs, workspace=ws)
    lib = _lib.load()
    lib.ssp_reset_launch_count()
    shared = ms.posteriors(feats, offs, resp=True, labels=True, workspace=ws, reuse_images=True)
    log = _lib.launch_log()
    assert "em_prep_kernel" not in log and "em_plan_kernel" not in log, log
    for a, b in zip(fresh, shared):
        assert t_equal(a, b)
    # and the other way round: posteriors prepare, stats reuse
    ws2 = mixture.StatsWorkspace(ms.device)
    ms.posteriors(feats, offs, resp=False, labels=True, workspace=ws2)
    n1 = ms.stats(feats, offs, workspace=ws2, reuse_images=True)
    n0 = ms.stats(feats, offs)
    for a, b in zip(n0[:3], n1[:3]):
        np.testing.assert_allclose(a.cpu().numpy(), b.cpu().numpy(), rtol=1e-9, atol=1e-9)


def t_equal(a, b):
    return bool((a == b).all().item())


def test_labels_alone_run_no_log_sum_exp_pass():
    w, mu, var = model(512, 39, 13)
    x, offs = frames(w, mu, var, [5000], seed=14)
    lib = _lib.load()
    lib.ssp_reset_launch_count()
    gm = ssp.GaussianMixture.from_params(w, mu, var)
    gm.predict(x)
    log = _lib.launch_log()
    assert "gmm_em_lse_kernel" not in log and "em_merge_kernel" not in log and "gmm_em_post_kernel<labels>" in log, log


@pytest.mark.parametrize("d", [13, 40])
def test_chunked_predict_proba_equals_one_device_call(monkeypatch, d):
    k = 96
    w, mu, var = model(k, d, 15)
    x = synth.sample_gmm(w, mu, var, 7000, seed=16)
    gm = ssp.GaussianMixture.from_params(w, mu, var)
    ms = gm._model_set()
    g, _, _ = ms.posteriors(torch().as_tensor(x, device="cuda"), np.array([0, len(x)]))
    monkeypatch.setattr(mixture, "PROBA_CHUNK_BYTES", 4 * k * 2048)
    lib = _lib.load()
    lib.ssp_reset_launch_count()
    got = gm.predict_proba(x)
    served = "gmm_em_post_kernel<resp>" if d <= 39 else "gmm_post_simt_kernel"
    assert _lib.launch_log()[served] == 4
    np.testing.assert_array_equal(got, g.cpu().numpy().astype(np.float64))


def test_argument_errors():
    w, mu, var = model(16, 13, 17)
    x, offs = frames(w, mu, var, [10, 20], seed=18)
    feats = torch().as_tensor(x, device="cuda")
    ms = ssp.ModelSet(w, mu, var)
    with pytest.raises(ValueError):
        ms.posteriors(feats, offs, resp=False, labels=False)
    with pytest.raises(ValueError):
        ms.posteriors(feats[:, :12].contiguous(), offs)
    with pytest.raises(ValueError):
        ssp.ModelSet(np.stack([w] * 3), np.stack([mu] * 3), np.stack([var] * 3)).posteriors(feats, offs)
    # the C entry point itself: both outputs NULL, n_models neither 1 nor n_segs
    lib = _lib.load()
    d_off = torch().as_tensor(offs, device="cuda")
    assert lib.ssp_gmm_posteriors(feats.data_ptr(), d_off.data_ptr(), 2, 30, ms.pack.data_ptr(), C.byref(ms.dims), None,
                                  None, None, None, 0, 0, _lib.stream_ptr()) == -1
    dims3 = _lib.GmmDims(3, 16, 13)
    assert lib.ssp_gmm_posteriors(feats.data_ptr(), d_off.data_ptr(), 2, 30, ms.pack.data_ptr(), C.byref(dims3), None,
                                  feats.data_ptr(), None, None, 0, 0, _lib.stream_ptr()) == -1
    # per-segment models beyond the tensor-core width
    w40, mu40, var40 = model(16, 40, 19)
    x40, _ = frames(w40, mu40, var40, [10, 20], seed=20)
    ms40 = ssp.ModelSet(np.stack([w40] * 2), np.stack([mu40] * 2), np.stack([var40] * 2))
    with pytest.raises(NotImplementedError):
        ms40.posteriors(torch().as_tensor(x40, device="cuda"), offs)
