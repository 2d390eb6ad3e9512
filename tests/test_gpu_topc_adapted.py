"""Top-C fast scoring of speakers MAP-adapted in weights and variances as well as means, on the GPU
(``ssp_gmm_pack_topc_adapted``, ``ssp_gmm_score_topc_adapted``, ``ModelSet.with_ubm``, ``ModelSet.score_top_c``,
``map_enrol(adapt=)``, ``identify(top_c=)`` / ``identify_pcm(top_c=)`` on such sets) against the float64 definition of
tests/test_topc_adapted_host.py on the GPU's own selection: model-tile and chunk edges, every feature width, every adapt
combination, known answers, extreme adaptation, the public entry points, and the refusals with the kernels that served
each call."""
import ctypes as C
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import speech_signal_processing_b200 as ssp  # noqa: E402
from oracle import gmm as ogmm  # noqa: E402
from speech_signal_processing_b200 import _lib, synth  # noqa: E402
from test_gpu_topc import LLR_ATOL, SCORE_RTOL, SELECT  # noqa: E402
from test_topc_adapted_host import score_top_c_adapted  # noqa: E402

ADAPTS = [combo for r in (1, 2, 3) for combo in itertools.combinations(("means", "weights", "variances"), r)]
ALL = ("means", "weights", "variances")
SCORE = {"topc_hist_kernel", "topc_scan_kernel", "topc_scatter_kernel", "topc_adapted_product_kernel", "topc_combine_kernel",
         "topc_finalize_kernel"}


def torch():
    return _lib.require_cuda()


def dev_frames(x):
    return torch().as_tensor(np.ascontiguousarray(x, dtype=np.float32), device="cuda")


def offsets(lens):
    offs = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    return offs


def synthetic_set(n_spk, k, d, seed):
    """(ModelSet.with_ubm of n_spk synthetic adapted speakers, UBM (w, mu, var)): every speaker's means shifted, weights
    tilted and variances scaled per component, as full MAP enrolment moves them."""
    w, mu, var = synth.synth_ubm(k, d, seed=seed, spread=1.0)
    rs = np.random.RandomState(seed + 1)
    smu = synth.synth_speaker_means(mu, n_spk, seed=seed + 2, shift=0.35) if n_spk else np.zeros((0, k, d))
    sw = w[None] * rs.uniform(0.5, 1.5, size=(n_spk, k))
    sw /= sw.sum(axis=1, keepdims=True)
    svar = var[None] * rs.uniform(0.6, 1.6, size=(n_spk, k, d))
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    return ssp.ModelSet.with_ubm(sw, smu, svar, ubm), (w, mu, var)


def check_scores(case, ms, feats, offs, x, c):
    """score_top_c of ``ms`` against the float64 definition on the GPU's own selection; prints the largest errors."""
    scores, lse = ms.score_top_c(feats, offs, c=c, want_frame_lse=True)
    idx, _ = ms._topc[0].top_components(feats, [0, len(x)], c)
    w, mu, var = (t.cpu().numpy() for t in ms._params)
    r = ms.ubm_index
    want, want_frame = score_top_c_adapted(x, offs, w, mu, var, r, c, idx=idx.cpu().numpy())
    got = scores.cpu().numpy()
    rel = float((np.abs(got - want) / np.maximum(1.0, np.abs(want))).max())
    llr_err = float(np.abs((got - got[:, r : r + 1]) - (want - want[:, r : r + 1])).max())
    frame_err = float((np.abs(lse.cpu().numpy() - want_frame) / np.maximum(1.0, np.abs(want_frame))).max()) if len(x) else 0.0
    print(f"{case}: scores {rel:.2e} rel, LLR {llr_err:.2e} abs, frame values {frame_err:.2e} rel")
    assert np.isfinite(got).all(), case
    assert rel <= SCORE_RTOL, case
    assert llr_err <= LLR_ATOL, case
    assert frame_err <= 5e-5, case
    assert (got[np.diff(offs) == 0] == 0.0).all(), case
    return got


# ------------------------------------------------------------------------------------------------ model tiles and chunks
@pytest.mark.parametrize("s", [1, 127, 128, 129, 300])
def test_model_tiles_and_chunk_edges(s):
    chunk = int(_lib.load().ssp_gmm_topc_chunk_frames())
    ms, (w, mu, var) = synthetic_set(s - 1, 32, 13, seed=s)
    assert ms.n_models == s
    for t in (chunk - 1, chunk, chunk + 1, 2 * chunk + 1):
        lens = [0, 1, 127, 0, t - 135, 1, 6]   # empty and one-frame utterances, one across every chunk boundary
        offs = offsets(lens)
        assert offs[-1] == t
        x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=t)
        check_scores(f"S={s} T={t}", ms, dev_frames(x), offs, x, 5)


# ------------------------------------------------------------------------------------------------ widths
@pytest.mark.parametrize("k", [5, 129])
@pytest.mark.parametrize("d", list(range(1, 40)))
def test_every_feature_width(d, k):
    ms, (w, mu, var) = synthetic_set(4, k, d, seed=d)
    offs = offsets([150, 0, 1, 210])
    x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=d + k)
    feats = dev_frames(x)
    for c in (1, min(k, 64)):
        check_scores(f"D={d} (NQ={(2 * d + 1 + 3) // 4}) K={k} C={c}", ms, feats, offs, x, c)


# ------------------------------------------------------------------------------------------------ adapt combinations
def enrolment(k=64, d=13, n_spk=6, seed=0, spread=1.0, shift=0.5):
    """UBM, speakers' enrolment frames (speaker 0 has none, speaker 1 three) and test frames."""
    w, mu, var = synth.synth_ubm(k, d, seed=seed, spread=spread)
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    spk_mu = synth.synth_speaker_means(mu, n_spk, seed=seed + 1, shift=shift)
    n = [0, 3] + [400 + 100 * i for i in range(n_spk - 2)]
    enrol = [synth.sample_gmm(w, spk_mu[i], var * (0.6 + 0.2 * i), n[i], seed=100 + i).reshape(n[i], d) for i in range(n_spk)]
    tests = [synth.sample_gmm(w, spk_mu[i % n_spk], var * (0.6 + 0.2 * (i % n_spk)), 120 + 31 * i, seed=200 + i)
             for i in range(2 * n_spk)]
    return ubm, enrol, tests


@pytest.mark.parametrize("adapt,relevance", [(a, 16.0) for a in ADAPTS] + [(a, 0.0) for a in ADAPTS if "variances" not in a])
def test_adapt_combinations(adapt, relevance):
    # variance MAP without the means subtracts the UBM's squared mean (mu_ubm^2) from the adapted second moment, which goes
    # negative where a speaker's frames sit away from the UBM's means: a UBM of small means and speakers close to it keep
    # every adapted variance positive (the least is 0.33 of the UBM's, by the float64 oracle)
    ubm, enrol, tests = enrolment(spread=0.5, shift=0.1)
    ms = ssp.ModelSet.with_ubm(*ssp.map_adapt(ubm, enrol, relevance=relevance, adapt=adapt), ubm)
    x = np.concatenate(tests)
    offs = offsets([len(t) for t in tests] + [0])
    feats = dev_frames(x)
    for c in (1, 5):
        got = check_scores(f"adapt={'+'.join(adapt)} r={relevance:g} C={c}", ms, feats, offs, x, c)
        # the speaker enrolled on no frames kept the UBM's parameters: its LLR is exactly 0
        assert (got[:, 0] - got[:, ms.ubm_index] == 0.0).all()


# ------------------------------------------------------------------------------------------------ known answers
@pytest.mark.parametrize("k", [1, 5, 64])
def test_c_equal_to_k_is_the_exact_score(k):
    ms, (w, mu, var) = synthetic_set(3, k, 13, seed=k)
    offs = offsets([300, 0, 17])
    x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=1)
    feats = dev_frames(x)
    got = check_scores(f"K={k} C=K", ms, feats, offs, x, k)
    exact, _ = ms.score(feats, offs, precision="fp32")
    exact = exact.cpu().numpy()
    sw, smu, svar = (t.cpu().numpy() for t in ms._params)
    for u in (0, 2):
        for s in range(ms.n_models):
            want = ogmm.score(x[offs[u] : offs[u + 1]], sw[s], smu[s], svar[s])
            assert abs(got[u, s] - want) <= SCORE_RTOL * max(1.0, abs(want)), (u, s, got[u, s], want)
            assert abs(got[u, s] - exact[u, s]) <= SCORE_RTOL * max(1.0, abs(want)), (u, s, got[u, s], exact[u, s])
    assert (got[1] == 0.0).all()


def test_mean_only_speakers_agree_with_the_shared_path():
    ubm, enrol, tests = enrolment(d=39)
    w, mu, var = ssp.map_adapt(ubm, enrol, adapt=("means",))
    ms = ssp.ModelSet.with_ubm(w, mu, var, ubm)
    sms = ssp.map_enrol(ubm, enrol)
    x = np.concatenate(tests)
    offs = offsets([len(t) for t in tests])
    feats = dev_frames(x)
    for c in (1, 5, 64):
        a = ms.score_top_c(feats, offs, c=c)[0].cpu().numpy()
        b = sms.score_top_c(feats, offs, c=c)[0].cpu().numpy()
        rel = float((np.abs(a - b) / np.maximum(1.0, np.abs(b))).max())
        llr = float(np.abs((a[:, :-1] - a[:, -1:]) - (b[:, :-1] - b[:, -1:])).max())
        print(f"C={c}: ModelSet.with_ubm vs SharedModelSet: scores {rel:.2e} rel, LLR {llr:.2e} abs")
        assert rel <= SCORE_RTOL and llr <= LLR_ATOL


def test_extreme_adaptation_stays_finite():
    k, d = 64, 13
    w, mu, var = synth.synth_ubm(k, d, seed=5, spread=1.0)
    far = mu + 8.0 * np.sqrt(var)                          # every component 8 sigma away in every dimension
    sw = np.stack([w, w, w, w, np.roll(w, 1)])
    smu = np.stack([far, mu, mu, far, far])
    svar = np.stack([var, 4.0 * var, var / 4.0, 4.0 * var, var / 4.0])
    ms = ssp.ModelSet.with_ubm(sw, smu, svar, ssp.GaussianMixture.from_params(w, mu, var))
    offs = offsets([400, 250])
    x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=2)
    for c in (1, 5, 64):
        got = check_scores(f"extreme C={c}", ms, dev_frames(x), offs, x, c)
        assert (got[:, ms.ubm_index] - got[:, 0]).min() > 200.0   # the distance the case is about


# ------------------------------------------------------------------------------------------------ public entry points
def test_identify_top_c_and_exact_on_a_fully_adapted_set():
    ubm, enrol, tests = enrolment(k=64, d=39, n_spk=12)
    ms = ssp.map_enrol(ubm, enrol, adapt=ALL)
    assert isinstance(ms, ssp.ModelSet) and ms.ubm_index == ms.n_models - 1 == 12
    x = np.concatenate(tests)
    offs = offsets([len(t) for t in tests])
    sw, smu, svar = (t.cpu().numpy() for t in ms._params)
    u = ms.ubm_index
    # top-C
    pred, arg = ssp.identify(tests, ms, top_c=5)
    idx, _ = ms._topc[0].top_components(dev_frames(x), [0, len(x)], 5)
    want, _ = score_top_c_adapted(x, offs, sw, smu, svar, u, 5, idx=idx.cpu().numpy())
    want = want[:, :u] - want[:, u:]
    # exact, the UBM scored in the same launch: identify runs what one ModelSet.score runs
    lib = _lib.load()
    lib.ssp_reset_launch_count()
    pred_x, arg_x = ssp.identify(tests, ms)
    log = _lib.launch_log()
    lib.ssp_reset_launch_count()
    ms.score(dev_frames(x), offs)
    assert log == _lib.launch_log(), log
    want_x = np.array([[ogmm.score(t, sw[s], smu[s], svar[s]) for s in range(u + 1)] for t in tests])
    want_x = want_x[:, :u] - want_x[:, u:]
    for name, p, a, wnt in (("top-C", pred, arg, want), ("exact", pred_x, arg_x, want_x)):
        err = float(np.abs(p - wnt).max())
        top = np.sort(wnt, axis=1)
        clear = top[:, -1] - top[:, -2] > 2 * LLR_ATOL
        print(f"identify {name}: LLR {err:.2e} abs of float64, {int(clear.sum())} of {len(tests)} decisions clear")
        assert err <= LLR_ATOL
        np.testing.assert_array_equal(a[clear], wnt.argmax(axis=1)[clear])


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
    ms = ssp.map_enrol(ubm, [x[foffs[i] : foffs[i + 1]] for i in range(4)], adapt=ALL)
    pred, _ = ssp.identify((feats, foffs), ms, top_c=5)
    want = pred.argmax(axis=1)
    dec, total = ssp.identify_pcm(host, soffs, fe, ms, ubm_index=ms.ubm_index, top_c=5)
    assert total == int(foffs[-1])
    np.testing.assert_array_equal(dec.numpy(), want)
    dec2, _ = ssp.identify_pcm(host, soffs, fe, ms, ubm_index=ms.ubm_index, top_c=5, min_split_frames=1, head_fraction=0.3)
    np.testing.assert_array_equal(dec2.numpy(), want)


# ------------------------------------------------------------------------------------------------ refusals and launches
def test_refusals_launch_nothing():
    torch_ = torch()
    lib = _lib.load()
    w, mu, var = synth.synth_ubm(16, 13, seed=0, spread=1.0)
    ubm = ssp.GaussianMixture.from_params(w, mu, var)
    ms = ssp.ModelSet.with_ubm(np.stack([w, w]), np.stack([mu + 0.1, mu]), np.stack([var, 2 * var]), ubm)
    plain = ssp.ModelSet(np.stack([w, w]), np.stack([mu + 0.1, mu]), np.stack([var, 2 * var]))
    x = synth.sample_gmm(w, mu, var, 100, seed=0)
    feats = dev_frames(x)
    w40, mu40, var40 = synth.synth_ubm(16, 40, seed=0, spread=1.0)
    ms40 = ssp.ModelSet.with_ubm(w40[None], mu40[None], var40[None], ssp.GaussianMixture.from_params(w40, mu40, var40))
    x40 = dev_frames(np.zeros((10, 40)))
    zero_var, neg_w, nan_var = var.copy(), w.copy(), var.copy()
    zero_var[3, 2], neg_w[5], nan_var[0, 0] = 0.0, -0.1, np.nan
    torch_.cuda.synchronize()
    before = lib.ssp_launch_count()
    refusals = [
        (ValueError, lambda: plain.score_top_c(feats, [0, 100], c=2)),                          # no ubm_index
        (ValueError, lambda: ssp.identify((feats, np.array([0, 100])), plain, top_c=2)),        # no UBM at all
        (NotImplementedError, lambda: ms40.score_top_c(x40, [0, 10], c=2)),                      # D = 40
        (ValueError, lambda: ms.score_top_c(feats, [0, 100], c=0)),
        (ValueError, lambda: ms.score_top_c(feats, [0, 100], c=17)),                             # C > K
        (ValueError, lambda: ms.score_top_c(feats, [0, 100], c=2.0)),
        (ValueError, lambda: ssp.ModelSet.with_ubm(w[None], mu[None], zero_var[None], ubm)),
        (ValueError, lambda: ssp.ModelSet.with_ubm(neg_w[None], mu[None], var[None], ubm)),
        (ValueError, lambda: ssp.ModelSet.with_ubm(w[None], mu[None], nan_var[None], ubm)),
        (ValueError, lambda: ssp.ModelSet.with_ubm(w[None], mu[None], var[None],
                                                   ssp.GaussianMixture.from_params(w, mu, zero_var))),
        (ValueError, lambda: ms.score_top_c(feats.double(), [0, 100], c=2)),                     # float64 frames
        (ValueError, lambda: ms.score_top_c(feats, [0, 99], c=2)),                               # offsets short of the rows
    ]
    for exc, call in refusals:
        with pytest.raises(exc):
            call()
        assert lib.ssp_launch_count() == before
    w65, mu65, var65 = synth.synth_ubm(128, 13, seed=0, spread=1.0)
    big = ssp.ModelSet.with_ubm(w65[None], mu65[None], var65[None], ssp.GaussianMixture.from_params(w65, mu65, var65))
    torch_.cuda.synchronize()
    before = lib.ssp_launch_count()
    with pytest.raises(ValueError):
        big.score_top_c(dev_frames(np.zeros((5, 13))), [0, 5], c=65)                           # C > 64
    # the C ABI, with made-up pointers: every call returns before anything dereferences them
    p = 1 << 20
    dims = C.byref(_lib.GmmDims(2, 16, 13))
    assert lib.ssp_gmm_pack_topc_adapted(p, p, p, dims, 2, p, None) == -1                      # ref_model out of range
    assert b"ref_model" in lib.ssp_last_error()
    assert lib.ssp_gmm_pack_topc_adapted(p, p, p, dims, -1, p, None) == -1
    assert lib.ssp_gmm_pack_topc_adapted(p, None, p, dims, 1, p, None) == -1                   # null pointer
    assert b"null" in lib.ssp_last_error()
    assert lib.ssp_gmm_pack_topc_adapted(p, p, p, dims, 1, p + 4, None) == -1                  # misaligned pack
    assert lib.ssp_gmm_pack_topc_adapted(p, p, p, C.byref(_lib.GmmDims(2, 16, 40)), 1, p, None) == -1
    assert lib.ssp_gmm_topc_adapted_pack_bytes(C.byref(_lib.GmmDims(2, 16, 40))) == 0
    assert lib.ssp_gmm_topc_adapted_pack_bytes(dims) == (16 * 2 * 28 + 16 * 16) * 4
    score = lib.ssp_gmm_score_topc_adapted
    assert score(p, p, 1, 10, p, p, 2, p + 8, dims, p, None, p, 1 << 30, None) == -1           # misaligned pack
    assert b"16-byte aligned" in lib.ssp_last_error()
    assert score(p, p, 1, 10, p, p, 2, p, dims, p, None, p + 8, 1 << 30, None) == -1           # misaligned workspace
    assert b"16-byte aligned" in lib.ssp_last_error()
    assert score(p, p, 1, 10, p, p, 2, p, dims, p, None, p, 16, None) == -1                    # short workspace
    assert score(p, p, 1, 10, p, p, 0, p, dims, p, None, p, 1 << 30, None) == -1               # C = 0
    assert score(p, p, 1, 10, p, p, 17, p, dims, p, None, p, 1 << 30, None) == -1              # C > K
    assert score(p, p, 1, 10, p, p, 2, p, C.byref(_lib.GmmDims(2, 16, 40)), p, None, p, 1 << 30, None) == -1
    assert score(p, p, 1, 10, None, p, 2, p, dims, p, None, p, 1 << 30, None) == -1            # null idx
    assert lib.ssp_launch_count() == before


def test_launch_log_and_cached_table():
    lib = _lib.load()
    ms, (w, mu, var) = synthetic_set(3, 128, 39, seed=1)
    x = synth.sample_gmm(w, mu, var, 1000, seed=1)
    feats = dev_frames(x)
    lib.ssp_reset_launch_count()
    ms.score_top_c(feats, [0, 1000], c=5)     # builds the UBM set and the table: the pack runs once
    first = _lib.launch_log()
    assert first["topc_adapted_pack_kernel"] == 1 and "topc_pack_kernel" not in first and "topc_product_kernel" not in first
    lib.ssp_reset_launch_count()
    ms.score_top_c(feats, [0, 400, 1000], c=5)
    assert set(_lib.launch_log()) == SELECT | SCORE, _lib.launch_log()
    assert all(n == 1 for n in _lib.launch_log().values()), _lib.launch_log()
    # repack drops the table: the next call builds it from the new parameters
    wp, mp, vp = ms._params
    ms.repack(wp, mp, vp * 1.1)
    lib.ssp_reset_launch_count()
    again, _ = ms.score_top_c(feats, [0, 1000], c=5)
    assert _lib.launch_log()["topc_adapted_pack_kernel"] == 1
    check_scores("after repack", ms, feats, np.array([0, 1000]), x, 5)
