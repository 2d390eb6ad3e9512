"""Top-C fast scoring on the GPU (``ssp_gmm_top_components``, ``ssp_gmm_score_topc``, ``ModelSet.top_components``,
``SharedModelSet.score_top_c``, ``identify(top_c=)`` / ``identify_pcm(top_c=)``) against the float64 oracle: the selection
at the tile edges of K and every width of the tensor-core path, the scores on the GPU's own selection at model-tile and
chunk edges, extreme adaptation, the public entry points, and the refusals with the kernels that served each call."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import speech_signal_processing_b200 as ssp  # noqa: E402
from oracle import gmm as ogmm  # noqa: E402
from speech_signal_processing_b200 import _lib, synth  # noqa: E402
from test_topc_host import score_top_c, top_components  # noqa: E402

MARGIN = 1e-3          # float64 gap below which two logits may come out in either order (the posteriors tests' margin)
LOGIT_RTOL = 1e-4      # the posteriors path's bound (|gamma - float64| <= 1e-4, i.e. ~1e-4 on a leading logit), relative to max(1, |L|)
SCORE_RTOL = 2e-5      # utterance scores
LLR_ATOL = 1e-3        # identify's contract
SELECT = {"em_plan_kernel", "em_prep_kernel", "gmm_em_post_kernel<topc>", "em_topc_merge_kernel"}
SCORE = {"topc_hist_kernel", "topc_scan_kernel", "topc_scatter_kernel", "topc_product_kernel", "topc_combine_kernel",
         "topc_finalize_kernel"}


def torch():
    return _lib.require_cuda()


def dev_frames(x):
    return torch().as_tensor(np.ascontiguousarray(x, dtype=np.float32), device="cuda")


def offsets(lens):
    offs = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    return offs


def check_selection(case, idx, logit, x, w, mu, var):
    """idx / logit (T, C) from the GPU against the float64 weighted log-probability."""
    c = idx.shape[1]
    wlp = ogmm.weighted_log_prob(x, w, mu, var)
    ref_idx, _ = top_components(x, w, mu, var, c)
    srt = -np.sort(-wlp, axis=1)
    # index sets: equal wherever the C-th and (C+1)-th logits are MARGIN apart
    sep = srt[:, c - 1] - srt[:, c] > MARGIN if c < wlp.shape[1] else np.ones(len(x), bool)
    got_sets, ref_sets = np.sort(idx, axis=1), np.sort(ref_idx, axis=1)
    bad = np.nonzero(sep & (got_sets != ref_sets).any(axis=1))[0]
    assert bad.size == 0, f"{case}: index sets differ at frames {bad[:5]}"
    # order: descending logits, the lower index first on equal ones; the float64 order wherever it is MARGIN-separated
    assert (logit[:, :-1] >= logit[:, 1:]).all(), case
    tie = logit[:, :-1] == logit[:, 1:]
    assert (idx[:, :-1][tie] < idx[:, 1:][tie]).all(), case
    gaps = -np.diff(srt[:, : min(c + 1, wlp.shape[1])], axis=1)
    clear = (gaps > MARGIN).all(axis=1)
    np.testing.assert_array_equal(idx[clear], ref_idx[clear], err_msg=case)
    ref_logit = np.take_along_axis(wlp, idx.astype(np.int64), axis=1)
    err = float((np.abs(logit - ref_logit) / np.maximum(1.0, np.abs(ref_logit))).max())
    assert err <= LOGIT_RTOL, f"{case}: logit error {err:.2e}"
    print(f"{case}: {int(sep.sum())} of {len(x)} frames separated, {int(clear.sum())} in full order, logit {err:.2e} rel")


# ------------------------------------------------------------------------------------------------ selection
@pytest.mark.parametrize("d", [1, 13, 26, 39])
@pytest.mark.parametrize("k", [1, 5, 64, 65, 128, 129, 1024, 2048])
def test_selection_matches_float64(k, d):
    w, mu, var = synth.synth_ubm(k, d, seed=k + d, spread=1.0)
    x = synth.sample_gmm(w, mu, var, 700, seed=d)
    ms = ssp.ModelSet(w, mu, var)
    feats = dev_frames(x)
    ws = ssp.mixture.StatsWorkspace(ms.device)
    for n, c in enumerate([c for c in (1, 2, 5, 16, 64) if c <= k]):
        idx, logit = ms.top_components(feats, [0, len(x)], c, workspace=ws, reuse_images=n > 0)
        assert idx.shape == (len(x), c) and idx.dtype == torch().int32 and logit.dtype == torch().float32
        check_selection(f"K={k} D={d} C={c}", idx.cpu().numpy(), logit.cpu().numpy(), x, w, mu, var)


def test_exact_ties_go_to_the_lower_index():
    w, mu, var = synth.synth_ubm(130, 13, seed=3, spread=1.0)
    for a, b in ((7, 3), (70, 129), (64, 63)):  # duplicates inside a half tile, across tiles, across half tiles
        mu[b], var[b], w[b] = mu[a], var[a], w[a]
    w = w / w.sum()
    x = synth.sample_gmm(w, mu, var, 500, seed=4)
    idx, logit = ssp.ModelSet(w, mu, var).top_components(dev_frames(x), [0, len(x)], 16)
    idx, logit = idx.cpu().numpy(), logit.cpu().numpy()
    for a, b in ((7, 3), (70, 129), (64, 63)):
        lo, hi = min(a, b), max(a, b)
        both = (idx == lo).any(axis=1) & (idx == hi).any(axis=1)
        assert both.any()
        pos_lo = np.argmax(idx == lo, axis=1)[both]
        pos_hi = np.argmax(idx == hi, axis=1)[both]
        assert (pos_hi == pos_lo + 1).all()
        np.testing.assert_array_equal(logit[both, pos_lo], logit[both, pos_hi])
    check_selection("duplicates", idx, logit, x, w, mu, var)


# ------------------------------------------------------------------------------------------------ scores
def shared_set(s, k, d, seed, shift=0.35):
    w, mu, var = synth.synth_ubm(k, d, seed=seed, spread=1.0)
    means = np.concatenate([synth.synth_speaker_means(mu, s - 1, seed=seed + 1, shift=shift), mu[None]]) if s > 1 else mu[None]
    return w, var, means


def check_scores(case, sms, feats, offs, x, c, w, var, means, ref):
    scores, lse = sms.score_top_c(feats, offs, c=c, want_frame_lse=True)
    idx, _ = sms._topc[0].top_components(feats, [0, len(x)], c)
    want, want_frame = score_top_c(x, offs, w, var, means, ref, c, idx=idx.cpu().numpy())
    got = scores.cpu().numpy()
    rel = float((np.abs(got - want) / np.maximum(1.0, np.abs(want))).max())
    llr_err = float(np.abs((got - got[:, ref : ref + 1]) - (want - want[:, ref : ref + 1])).max())
    frame_err = float((np.abs(lse.cpu().numpy() - want_frame) / np.maximum(1.0, np.abs(want_frame))).max()) if len(x) else 0.0
    print(f"{case}: scores {rel:.2e} rel, LLR {llr_err:.2e} abs, frame values {frame_err:.2e} rel")
    assert rel <= SCORE_RTOL, case
    assert llr_err <= LLR_ATOL, case
    assert frame_err <= 5e-5, case
    empty = np.diff(offs) == 0
    assert (got[empty] == 0.0).all()
    return got


@pytest.mark.parametrize("s", [1, 2, 255, 256, 257, 1001])
def test_scores_match_float64_on_the_gpu_selection(s):
    chunk = int(_lib.load().ssp_gmm_topc_chunk_frames())
    k, d, c = 64, 13, 5
    w, var, means = shared_set(s, k, d, seed=s)
    # ragged utterances: empty, one frame, around a 128-frame unit, 30 s, and one across each chunk boundary
    lens = [0, 1, 127, 128, 129, 2998, 0, chunk - 3000, 7, chunk + 11, 5]
    offs = offsets(lens)
    x = synth.sample_gmm(w, means[-1], var, int(offs[-1]), seed=s + 7)
    sms = ssp.SharedModelSet(w, var, means, ref_model=-1)
    check_scores(f"S={s}", sms, dev_frames(x), offs, x, c, w, var, means, s - 1)


@pytest.mark.parametrize("k,d", [(16, 13), (64, 39)])
def test_c_equal_to_k_is_the_exact_score(k, d):
    w, var, means = shared_set(3, k, d, seed=k)
    lens = [300, 0, 17]
    offs = offsets(lens)
    x = synth.sample_gmm(w, means[0], var, int(offs[-1]), seed=1)
    sms = ssp.SharedModelSet(w, var, means, ref_model=-1)
    got, _ = sms.score_top_c(dev_frames(x), offs, c=k)
    got = got.cpu().numpy()
    for u in (0, 2):
        for s_ in range(3):
            want = ogmm.score(x[offs[u] : offs[u + 1]], w, means[s_], var)
            assert abs(got[u, s_] - want) <= SCORE_RTOL * max(1.0, abs(want)), (u, s_, got[u, s_], want)
    assert (got[1] == 0.0).all()


def test_extreme_adaptation_stays_finite():
    k, d, c = 64, 13, 5
    w, var, means = shared_set(3, k, d, seed=5)
    means[0] = means[-1] + 8.0 * np.sqrt(var)   # every component 8 sigma away in every dimension
    offs = offsets([400, 250])
    x = synth.sample_gmm(w, means[-1], var, int(offs[-1]), seed=2)
    sms = ssp.SharedModelSet(w, var, means, ref_model=-1)
    got = check_scores("extreme", sms, dev_frames(x), offs, x, c, w, var, means, 2)
    assert np.isfinite(got).all()
    assert (got[:, 2] - got[:, 0]).min() > 200.0   # the distance the case is about


# ------------------------------------------------------------------------------------------------ public entry points
def enrolled(k=64, d=39, n_spk=12, seed=0):
    w, mu, var = synth.synth_ubm(k, d, seed=seed, spread=1.0)
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    spk_mu = synth.synth_speaker_means(mu, n_spk, seed=seed + 1, shift=0.5)
    enrol = [synth.sample_gmm(w, spk_mu[i], var, 600, seed=100 + i) for i in range(n_spk)]
    tests = [synth.sample_gmm(w, spk_mu[i % n_spk], var, 150 + 37 * i, seed=200 + i) for i in range(2 * n_spk)]
    return ubm, enrol, tests


def test_identify_top_c_matches_the_oracle():
    ubm, enrol, tests = enrolled()
    sms = ssp.map_enrol(ubm, enrol)
    pred, arg = ssp.identify(tests, sms, top_c=5)
    w, var, means = (t.cpu().numpy() for t in sms._params)
    x = np.concatenate(tests)
    offs = offsets([len(t) for t in tests])
    idx, _ = sms._topc[0].top_components(dev_frames(x), [0, len(x)], 5)
    want, _ = score_top_c(x, offs, w, var, means, sms.ubm_index, 5, idx=idx.cpu().numpy())
    want = want[:, :-1] - want[:, -1:]
    err = float(np.abs(pred - want).max())
    print(f"identify(top_c=5): LLR {err:.2e} abs of float64")
    assert err <= LLR_ATOL
    top = np.sort(want, axis=1)
    ok = top[:, -1] - top[:, -2] > MARGIN
    np.testing.assert_array_equal(arg[ok], want.argmax(axis=1)[ok])
    # a list of mean-only MAP models with the UBM gives the same matrix
    gms = [ssp.GaussianMixture.from_params(w, means[i], var) for i in range(len(enrol))]
    pred2, _ = ssp.identify(tests, gms, ubm, top_c=5)
    np.testing.assert_allclose(pred2, pred, rtol=0, atol=1e-9)


def test_identify_pcm_top_c_equals_identify():
    torch_ = torch()
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True)
    pcm = [synth.synth_utterance(i % 4, i, n_samples=16000 + 800 * i) for i in range(12)]
    soffs = offsets([len(p) for p in pcm])
    host = torch_.from_numpy(np.concatenate(pcm))
    feats, foffs, _ = fe.extract_device(host.to("cuda"), soffs)
    w, mu, var = synth.synth_ubm(64, 39, seed=0, spread=1.0)
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    x = feats.cpu().numpy()
    sms = ssp.map_enrol(ubm, [x[foffs[i] : foffs[i + 1]] for i in range(4)])
    pred, _ = ssp.identify((feats, foffs), sms, top_c=5)
    want = pred.argmax(axis=1)
    dec, total = ssp.identify_pcm(host, soffs, fe, sms, ubm_index=sms.ubm_index, top_c=5)
    assert total == int(foffs[-1])
    np.testing.assert_array_equal(dec.numpy(), want)
    # the two-part pipeline: the tail copied on the side stream
    dec2, _ = ssp.identify_pcm(host, soffs, fe, sms, ubm_index=sms.ubm_index, top_c=5, min_split_frames=1, head_fraction=0.3)
    np.testing.assert_array_equal(dec2.numpy(), want)


# ------------------------------------------------------------------------------------------------ refusals and launches
def test_refusals_launch_nothing():
    torch_ = torch()
    lib = _lib.load()
    w, mu, var = synth.synth_ubm(16, 13, seed=0, spread=1.0)
    ms = ssp.ModelSet(w, mu, var)
    x = synth.sample_gmm(w, mu, var, 100, seed=0)
    feats = dev_frames(x)
    sms = ssp.SharedModelSet(w, var, np.stack([mu, mu + 0.1]), ref_model=-1)
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    other = ssp.GaussianMixture.from_params(w, mu, var * 1.5)
    pair = ssp.ModelSet(np.stack([w, w]), np.stack([mu, mu]), np.stack([var, var]))
    w40, mu40, var40 = synth.synth_ubm(16, 40, seed=0, spread=1.0)
    ms40 = ssp.ModelSet(w40, mu40, var40)
    x40 = dev_frames(np.zeros((10, 40)))
    xt = dev_frames(np.zeros((13, 100))).t()
    torch_.cuda.synchronize()
    before = lib.ssp_launch_count()
    refusals = [
        (ValueError, lambda: ms.top_components(feats, [0, 100], 0)),
        (ValueError, lambda: ms.top_components(feats, [0, 100], 17)),
        (ValueError, lambda: ms.top_components(feats, [0, 100], 2.0)),
        (ValueError, lambda: sms.score_top_c(feats, [0, 100], c=65)),
        (ValueError, lambda: pair.top_components(feats, [0, 100], 2)),
        (ValueError, lambda: ms.top_components(x, [0, 100], 2)),                                   # numpy frames
        (ValueError, lambda: ms.top_components(feats.double(), [0, 100], 2)),                      # float64
        (ValueError, lambda: ms.top_components(xt, [0, 100], 2)),                                  # transposed
        (ValueError, lambda: ms.top_components(feats, [0, 99], 2)),                                # offsets short of the rows
        (ValueError, lambda: sms.score_top_c(feats, [0, 50, 40, 100], c=2)),                       # decreasing offsets
        (ValueError, lambda: ssp.identify((feats, np.array([0, 100])), [ubm], None, top_c=2)),     # no UBM
        (NotImplementedError, lambda: ssp.identify((feats, np.array([0, 100])), [other], ubm, top_c=2)),
        (NotImplementedError, lambda: ms40.top_components(x40, [0, 10], 2)),                       # D = 40
    ]
    for exc, call in refusals:
        with pytest.raises(exc):
            call()
        assert lib.ssp_launch_count() == before
    p = 1 << 20
    dims = C.byref(_lib.GmmDims(1, 16, 13))
    assert lib.ssp_gmm_top_components(p, p, 1, 10, p, dims, 2, p, p, p + 4, 1 << 30, 0, None) == -1
    assert b"16-byte aligned" in lib.ssp_last_error()
    sdims = C.byref(_lib.GmmDims(2, 16, 13))
    assert lib.ssp_gmm_score_topc(p, p, 1, 10, p, p, 2, p, sdims, p, None, p + 8, 1 << 30, None) == -1
    assert b"16-byte aligned" in lib.ssp_last_error()
    assert lib.ssp_gmm_score_topc(p, p, 1, 10, p, p, 17, p, sdims, p, None, p, 1 << 30, None) == -1
    assert lib.ssp_gmm_top_components(p, p, 1, 10, p, dims, 2, None, p, p, 1 << 30, 0, None) == -1
    assert lib.ssp_gmm_top_components(p, p, 1, 10, p, dims, 2, p, p, p, 16, 0, None) == -1   # short workspace
    assert lib.ssp_launch_count() == before


def test_launch_log_and_reused_images():
    lib = _lib.load()
    w, mu, var = synth.synth_ubm(128, 39, seed=1, spread=1.0)
    ms = ssp.ModelSet(w, mu, var)
    x = synth.sample_gmm(w, mu, var, 1000, seed=1)
    feats = dev_frames(x)
    ws = ssp.mixture.StatsWorkspace(ms.device)
    lib.ssp_reset_launch_count()
    first = ms.top_components(feats, [0, 1000], 5, workspace=ws)
    assert _lib.launch_log() == {name: 1 for name in SELECT}
    # the posteriors of the same frames and a second selection run on the images the first call prepared
    lib.ssp_reset_launch_count()
    _, labels, _ = ms.posteriors(feats, [0, 1000], resp=False, labels=True, workspace=ws, reuse_images=True)
    again = ms.top_components(feats, [0, 1000], 5, workspace=ws, reuse_images=True)
    log = _lib.launch_log()
    assert "em_plan_kernel" not in log and "em_prep_kernel" not in log, log
    assert log["gmm_em_post_kernel<topc>"] == 1 and log["em_topc_merge_kernel"] == 1
    np.testing.assert_array_equal(again[0].cpu().numpy(), first[0].cpu().numpy())
    np.testing.assert_array_equal(first[0][:, 0].long().cpu().numpy(), labels.cpu().numpy())
    sms = ssp.SharedModelSet(w, var, np.stack([mu + 0.2, mu]), ref_model=-1)
    sms.score_top_c(feats, [0, 1000], c=5)   # builds the reference set and the table
    lib.ssp_reset_launch_count()
    sms.score_top_c(feats, [0, 400, 1000], c=5)
    assert set(_lib.launch_log()) == SELECT | SCORE, _lib.launch_log()
