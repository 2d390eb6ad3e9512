"""The oracle restatements against fixtures produced by the unmodified reference
(tests/golden/make_golden.py) and against sklearn 1.9.0 live.  CPU only."""
import numpy as np
import pytest

from oracle import frontend as ofe
from oracle import gmm as ogmm


def test_processing_mfcc_matches_reference(golden):
    g = golden("processing_mfcc.npz")
    for tag in "abcd":
        fs, fsz, step = (int(v) for v in g[f"{tag}_cfg"])
        got = ofe.processing_mfcc(g[f"{tag}_sig"], fs, fsz, step)
        ref = g[f"{tag}_mfcc"]
        assert got.shape == ref.shape
        np.testing.assert_allclose(got, ref, rtol=0, atol=1e-9)


def test_processing_fbank_and_enframe(golden):
    g = golden("processing_mfcc.npz")
    fb, fr = ofe.processing_fbank(16000, 512)
    np.testing.assert_allclose(fb, g["fbank_16k_512"], atol=1e-14)
    np.testing.assert_allclose(fr, g["freqs_16k_512"], atol=1e-9)
    np.testing.assert_allclose(ofe.processing_fbank(8000, 512)[0], g["fbank_8k_512"], atol=1e-14)
    np.testing.assert_allclose(ofe.processing_enframe(g["a_sig"], 400, 160), g["enframe_a"], atol=1e-9)


def test_delta_matches_reference(golden):
    g = golden("delta.npz")
    i = 0
    while f"x{i}" in g.files:
        got = ofe.delta(g[f"x{i}"], int(g[f"n{i}"]))
        np.testing.assert_allclose(got, g[f"d{i}"], atol=1e-13)
        i += 1
    assert i >= 8
    # known answer: interior of a ramp has delta == slope (SURVEY section 4 item 5)
    d = ofe.delta(g["ramp"], 2)
    np.testing.assert_allclose(d, g["ramp_d"], atol=1e-13)
    np.testing.assert_allclose(d[2:-2], np.tile([[1.0, -2.0]], (16, 1)), atol=1e-13)
    with pytest.raises(ValueError):
        ofe.delta(g["ramp"], 0)


def test_scale_matches_sklearn(golden):
    g = golden("sklearn_gmm.npz")
    np.testing.assert_allclose(ofe.scale(g["scale_x"]), g["scale_y"], atol=1e-10)
    y = ofe.scale(g["scale_x"])
    np.testing.assert_allclose(y.mean(axis=0), 0, atol=1e-10)
    keep = np.arange(26) != 3
    np.testing.assert_allclose(y.std(axis=0)[keep], 1, atol=1e-10)
    np.testing.assert_allclose(y[:, 3], 0, atol=1e-12)


@pytest.mark.parametrize("tag", ["s", "m", "l"])
def test_gmm_score_matches_sklearn(golden, tag):
    g = golden("sklearn_gmm.npz")
    w, mu, var, x = g[f"{tag}_w"], g[f"{tag}_mu"], g[f"{tag}_var"], g[f"{tag}_x"]
    np.testing.assert_allclose(ogmm.score_samples(x, w, mu, var), g[f"{tag}_score_samples"], rtol=1e-12, atol=1e-10)
    assert abs(ogmm.score(x, w, mu, var) - float(g[f"{tag}_score"])) < 1e-10
    if f"{tag}_proba" in g.files:
        np.testing.assert_allclose(ogmm.responsibilities(x, w, mu, var)[1], g[f"{tag}_proba"], atol=1e-12)


@pytest.mark.parametrize("tag", ["s", "m"])
@pytest.mark.parametrize("iters", [1, 3, 100])
def test_em_trajectory_matches_sklearn(golden, tag, iters):
    g = golden("sklearn_gmm.npz")
    w, mu, var, x = g[f"{tag}_w"], g[f"{tag}_mu"], g[f"{tag}_var"], g[f"{tag}_x"]
    w2, mu2, var2, n_iter, conv, bounds = ogmm.em_fit(x, w, mu, var, max_iter=iters)
    assert n_iter == int(g[f"{tag}_fit{iters}_niter"])
    assert conv == bool(g[f"{tag}_fit{iters}_conv"])
    np.testing.assert_allclose(w2, g[f"{tag}_fit{iters}_w"], rtol=1e-8, atol=1e-12)
    np.testing.assert_allclose(mu2, g[f"{tag}_fit{iters}_mu"], rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(var2, g[f"{tag}_fit{iters}_var"], rtol=1e-7, atol=1e-9)
    assert abs(bounds[-1] - float(g[f"{tag}_fit{iters}_lb"])) < 1e-9


def test_identify_matches_reference_pipeline(golden):
    """GMM_UBM.py:191-197 pred matrix recomputed by the oracle from the reference-trained models."""
    g = golden("pipeline.npz")
    models = [(g["gmm_w"][i], g["gmm_mu"][i], g["gmm_var"][i]) for i in range(g["gmm_w"].shape[0])]
    ubm = (g["ubm_w"], g["ubm_mu"], g["ubm_var"])
    pred, arg = ogmm.identify(list(g["feat_test"]), models, ubm)
    np.testing.assert_allclose(pred, g["pred"], rtol=1e-10, atol=1e-9)
    acc = (arg == g["y_test"]).mean()
    assert f"test acc {acc:.2%}" in str(g["printed"])


def test_features_recipe_matches_reference_extract_feature(golden):
    """oracle.features == GMM_UBM.extract_feature (with the sidekit restatement as mfcc)."""
    g = golden("pipeline.npz")
    for j in range(3):
        got = ofe.features(g["x_test"][j], preset="sidekit", delta_order=1, cmvn=True)
        np.testing.assert_allclose(got, g["feat_test"][j], atol=1e-9)


def test_sidekit_shape_witness():
    """report/final.pdf p.5, d_vector.py:81-91: 1 s @ 16 kHz -> 98 x 13 cepstra."""
    from speech_signal_processing_b200 import synth

    out = ofe.sidekit_mfcc(synth.synth_utterance(1, 1, 16000))
    assert out[0].shape == (98, 13) and out[1].shape == (98,) and out[2] is None and out[3] is None
    assert ofe.sidekit_mfcc(synth.synth_utterance(1, 1, 48000))[0].shape == (298, 13)


def test_psf_known_answers():
    from speech_signal_processing_b200 import synth

    sig = synth.synth_utterance(2, 0, 48000)
    c = ofe.psf_mfcc(sig)
    assert c.shape == (299, 13)  # 1 + ceil((48000-400)/160)
    fb = ofe.psf_filterbanks()
    assert fb.shape == (26, 257) and np.isclose(fb.max(), 1.0)


def test_dct_orthonormal():
    m = ofe.dct2_ortho_matrix(24, 24)
    np.testing.assert_allclose(m @ m.T, np.eye(24), atol=1e-12)
    from scipy.fft import dct

    x = np.random.RandomState(0).standard_normal(24)
    np.testing.assert_allclose(m @ x, dct(x, type=2, norm="ortho"), atol=1e-12)


def test_single_gaussian_closed_form():
    x = np.array([[0.5, -1.0], [2.0, 0.0]])
    mu, var = np.array([[0.0, 1.0]]), np.array([[2.0, 0.5]])
    want = -0.5 * (2 * np.log(2 * np.pi) + np.log(var).sum() + ((x - mu) ** 2 / var).sum(axis=1))
    np.testing.assert_allclose(ogmm.score_samples(x, np.array([1.0]), mu, var), want, atol=1e-12)


def test_map_adapt_limits():
    from speech_signal_processing_b200 import synth

    w, mu, var = synth.synth_ubm(8, 5, seed=2)
    x = synth.sample_gmm(w, mu + 0.5, var, 500, seed=3).astype(np.float64)
    n, f, s, _ = ogmm.suff_stats(x, w, mu, var)
    _, m_inf, _ = ogmm.map_adapt(n, f, s, w, mu, var, 500, relevance=1e12)
    np.testing.assert_allclose(m_inf, mu, atol=1e-6)  # r -> inf keeps the UBM
    _, m_0, _ = ogmm.map_adapt(n, f, s, w, mu, var, 500, relevance=1e-12)
    np.testing.assert_allclose(m_0, f / n[:, None], atol=1e-6)  # r -> 0 is the ML mean
    w2, m2, v2 = ogmm.map_adapt(n, f, s, w, mu, var, 500, adapt=("means", "weights", "variances"))
    assert np.isclose(w2.sum(), 1.0) and (v2 > 0).all()


def test_map_adapt_without_data_keeps_the_ubm():
    """A speaker of no frames, and a component no frame reaches (also at relevance 0), keep the UBM's parameters."""
    from speech_signal_processing_b200 import synth

    every = ("means", "weights", "variances")
    w, mu, var = synth.synth_ubm(8, 5, seed=4)
    z = np.zeros(8)
    for r in (16.0, 0.0):
        got = ogmm.map_adapt(z, np.zeros((8, 5)), np.zeros((8, 5)), w, mu, var, 0, relevance=r, adapt=every)
        for g, want in zip(got, (w / w.sum(), mu, var)):
            assert np.isfinite(g).all()
            np.testing.assert_allclose(g, want, rtol=1e-12, atol=0)   # var + mu^2 - mu^2 rounds
    x = synth.sample_gmm(w, mu + 0.5, var, 400, seed=5).astype(np.float64)
    n, f, s, _ = ogmm.suff_stats(x, w, mu, var)
    n[3], f[3], s[3] = 0.0, 0.0, 0.0
    for r in (16.0, 0.0):
        w2, m2, v2 = ogmm.map_adapt(n, f, s, w, mu, var, 400, relevance=r, adapt=every)
        assert np.isfinite(w2).all() and np.isfinite(m2).all() and np.isfinite(v2).all()
        np.testing.assert_array_equal(m2[3], mu[3])
        np.testing.assert_allclose(v2[3], var[3], rtol=1e-12)
        a = n / (n + r) if r else (n > 0).astype(float)
        want_w = a * n / 400 + (1 - a) * w
        np.testing.assert_allclose(w2, want_w / want_w.sum(), rtol=1e-14)
    np.testing.assert_allclose(ogmm.map_adapt(n, f, s, w, mu, var, 400, relevance=0.0)[1][n > 0], (f / n[:, None])[n > 0],
                               rtol=1e-14)


def test_vad_matches_reference(golden):
    """oracle.vad against the unmodified VAD.py (framing, ZCR, energy, spectral entropy, both detectors)."""
    from oracle import vad as ov

    g = golden("vad.npz")
    for i in range(int(g["n_cases"])):
        frames = ov.enframe(ov.wav_normalise(g[f"sig{i}"]))
        if f"frames{i}" in g:
            assert np.array_equal(frames, g[f"frames{i}"])
        z, p, e = ov.feature(frames)
        assert np.array_equal(ov.zcr(frames), g[f"zcr_raw{i}"])
        assert np.array_equal(z, g[f"zcr{i}"])
        np.testing.assert_allclose(p, g[f"power{i}"], rtol=1e-12)
        np.testing.assert_allclose(e, g[f"entropy{i}"], rtol=1e-9, atol=1e-12)
        assert np.array_equal(ov.detect(z, p), g[f"det{i}"])
        assert np.array_equal(ov.detect(z, p, zcr_gate=25, ampl=1.0, amph=8), g[f"det_b{i}"])
        assert np.array_equal(ov.frequency(e), g[f"freq{i}"])


def test_plp_building_blocks_known_answers():
    """sidekit's plp is unpinned (package absent); its building blocks are checked against independent computations:
    Levinson-Durbin vs a Toeplitz solve, the LPC -> cepstrum recursion vs the FFT cepstrum of the all-pole spectrum,
    the RASTA filter vs scipy.signal.lfilter from rest, the Bark filterbank's shape facts, and the output shape the
    reference's report quotes for 1 s of audio (98 frames)."""
    from scipy.linalg import solve_toeplitz
    from scipy.signal import lfilter

    from speech_signal_processing_b200 import synth

    rs = np.random.RandomState(0)
    # Levinson: a[1:] solves R a = -r[1:], error = r0 + sum a_k r_k
    x = rs.standard_normal((5, 400))
    r = np.array([[np.dot(row[: 400 - k], row[k:]) for k in range(13)] for row in x])
    a, e = ofe.levinson(r, 12)
    for i in range(5):
        sol = solve_toeplitz(r[i, :12], -r[i, 1:13])
        np.testing.assert_allclose(a[i, 1:], sol, rtol=1e-8, atol=1e-10)
        np.testing.assert_allclose(e[i], r[i, 0] + np.dot(a[i, 1:], r[i, 1:13]), rtol=1e-10)
    # LPC -> cepstrum: c_n of log(1 / A(z)) from the recursion == inverse FFT of the log all-pole spectrum
    poles = 0.6 * np.exp(1j * np.array([0.4, 1.3, 2.2]))
    poly = np.real(np.poly(np.concatenate([poles, poles.conj()])))          # A(z) = 1 + a1 z^-1 + ...
    n_fft = 4096
    log_h = -np.log(np.fft.fft(poly, n_fft))
    cep_fft = np.real(np.fft.ifft(log_h))[:7]
    cep = np.zeros(7)
    for n in range(1, 7):
        s = sum((n - m) * poly[m] * cep[n - m] for m in range(1, n))
        cep[n] = -(poly[n] + s / n)
    np.testing.assert_allclose(cep[1:], cep_fft[1:], atol=1e-9)
    # RASTA: after the four warm-up frames the output is the IIR filter continued from the FIR state
    z = rs.standard_normal((50, 3))
    y = ofe.rasta_filt(z)
    assert np.all(y[:4] == 0.0)
    numer, denom = ofe.rasta_filter_coefficients()
    np.testing.assert_allclose(numer, [0.2, 0.1, 0.0, -0.1, -0.2])
    full_fir = lfilter(numer, [1.0], z, axis=0)
    np.testing.assert_allclose(y[4], full_fir[4] , atol=1e-12)               # first IIR output has no feedback term yet
    np.testing.assert_allclose(y[5], full_fir[5] + 0.94 * y[4], atol=1e-12)
    # Bark filterbank at 16 kHz / 512: 21 bands, unit peaks, centre frequencies increasing
    w = ofe.fft2barkmx(512, 16000)
    assert w.shape == (21, 257) and np.isclose(w.max(axis=1)[1:-1], 1.0, atol=0.2).all()
    assert (np.diff(w.argmax(axis=1)) > 0).all()
    out = ofe.sidekit_plp(synth.synth_utterance(1, 2, 16000))
    assert out[0].shape == (98, 13) and out[1].shape == (98,) and np.isfinite(out[0]).all()


def test_librosa_restatement_agrees_with_torchaudio():
    """librosa is absent (parity unpinned); torchaudio's MFCC transform implements the same conventions independently
    (Slaney mel / area norm, centred reflect-padded STFT, power_to_db with top_db 80, DCT-II ortho) -- a cross-check of
    the restatement, not a pin.  MFCC_DTW.py:27-30."""
    torch = pytest.importorskip("torch")
    torchaudio = pytest.importorskip("torchaudio")
    from speech_signal_processing_b200 import synth

    sig = synth.synth_utterance(3, 1, 12000, 8000).astype(np.float64)
    tr = torchaudio.transforms.MFCC(sample_rate=8000, n_mfcc=13, dct_type=2, norm="ortho", log_mels=False, melkwargs=dict(
        n_fft=2048, hop_length=512, n_mels=128, center=True, pad_mode="reflect", power=2.0, norm="slaney", mel_scale="slaney",
        f_min=0.0, f_max=4000.0)).double()
    want = tr(torch.from_numpy(sig)).numpy()
    got = ofe.librosa_mfcc(sig)
    assert got.shape == want.shape == (13, 1 + 12000 // 512)
    # torchaudio builds its filterbank in float32: agreement to ~1e-7 relative on values up to ~900
    np.testing.assert_allclose(got, want, rtol=2e-6, atol=1e-3)
    assert ofe.mfcc_lib(sig.astype(np.int16)).shape == (13 * 24,)


def test_librosa_known_answers():
    # Slaney mel scale: linear below 1 kHz (200/3 Hz per mel), log above; the two branches meet at 1 kHz = 15 mel
    assert ofe.slaney_hz_to_mel(1000.0) == pytest.approx(15.0)
    assert ofe.slaney_hz_to_mel(200.0) == pytest.approx(3.0)
    assert ofe.slaney_mel_to_hz(ofe.slaney_hz_to_mel(3210.0)) == pytest.approx(3210.0)
    assert ofe.slaney_hz_to_mel(6400.0) == pytest.approx(15.0 + 27.0)  # log step: 27 mel per factor 6.4
    fb = ofe.librosa_mel_filters(8000, 2048)
    assert fb.shape == (128, 1025) and (fb >= 0).all() and (fb.sum(axis=1) > 0).all()
    # area normalisation: every triangle integrates to ~1 over frequency
    np.testing.assert_allclose(fb.sum(axis=1) * (8000 / 2048), 1.0, atol=0.08)
    # digital silence: every band sits at amin -> -100 dB everywhere -> only c0 is non-zero
    c = ofe.librosa_mfcc(np.zeros(4096))
    np.testing.assert_allclose(c[0], -100.0 * np.sqrt(128), rtol=1e-12)
    np.testing.assert_allclose(c[1:], 0.0, atol=1e-9)
    # a tone far above the floor: the top_db clip holds every band within 80 dB of the maximum
    t = np.arange(8000) / 8000.0
    tone = 1e4 * np.sin(2 * np.pi * 440.0 * t)
    c_clip = ofe.librosa_mfcc(tone)
    c_free = ofe.librosa_mfcc(tone, top_db=None)
    assert np.abs(c_clip - c_free).max() > 1.0
    assert c_clip.shape == (13, 1 + 8000 // 512)


def test_config1_reference_run_is_reproduced_by_the_oracle(golden, config1_corpus):
    """BASELINE configs[0] at its stated size: the models the unmodified GMM_UBM.GMM() trained (fixture), scored by the
    oracle on oracle features of the regenerated audio, reproduce the reference's LLR matrix and decisions."""
    import zlib

    g = golden("config1.npz")
    _, x_te, _, y_te = config1_corpus
    assert zlib.crc32(np.concatenate(x_te).tobytes()) == int(g["audio_crc"]), "synthetic audio differs from the fixture's"
    assert list(y_te) == list(g["y_test"])
    feats = [ofe.features(x, preset="sidekit", delta_order=1, cmvn=True) for x in x_te]
    np.testing.assert_allclose(feats[0], g["feat_first"], atol=2e-5)   # the reference path is float32 after the spectrum
    np.testing.assert_allclose(feats[-1], g["feat_last"], atol=2e-5)
    np.testing.assert_allclose([np.abs(f).mean() for f in feats], g["feat_abs_mean"], rtol=1e-5)
    mu, var = g["gmm_mu"].astype(np.float64), g["gmm_var"].astype(np.float64)
    pred = np.array([[ogmm.score(f, g["gmm_w"][i], mu[i], var[i]) for i in range(10)] for f in feats])
    pred -= np.array([ogmm.score(f, g["ubm_w"], g["ubm_mu"].astype(np.float64), g["ubm_var"].astype(np.float64)) for f in feats])[:, None]
    np.testing.assert_allclose(pred, g["pred"], rtol=0, atol=5e-4)
    assert (pred.argmax(axis=1) == g["pred"].argmax(axis=1)).all()
    assert (pred.argmax(axis=1) == np.asarray(y_te)).mean() == 1.0 and "test acc 100.00%" in str(g["printed"])


def test_sidekit_restatement_known_answers():
    """Properties the sidekit restatement must have whatever the absent package's exact code is (parity unpinned):
    the published conventions of SURVEY 8(c) -- mel-spaced area-normalised triangles between 100 Hz and 8 kHz, a pure
    tone lands in the band whose centre is nearest, per-frame pre-emphasis, frame energy of the un-windowed frame."""
    fb, edges = ofe.sidekit_trfbank(16000, 512, 100, 8000, 0, 24)
    assert fb.shape == (24, 257) and edges.shape == (26,)
    assert edges[0] == pytest.approx(100.0) and edges[-1] == pytest.approx(8000.0)
    np.testing.assert_allclose(np.diff(ofe.hz2mel(edges)), np.diff(ofe.hz2mel(edges))[0], rtol=1e-9)  # equal mel steps
    assert ofe.hz2mel(1000.0) == pytest.approx(2595.0 * np.log10(1.0 + 1000.0 / 700.0))  # report/GMM_UBM.pdf p.4
    assert (fb >= 0).all() and (fb.sum(axis=1) > 0).all()
    peak_bin = fb.argmax(axis=1)
    assert (np.diff(peak_bin) > 0).all()                                   # bands ordered in frequency
    centre_bin = np.floor(edges[1:-1] * 512 / 16000).astype(int)
    assert (np.abs(peak_bin - centre_bin) <= 1).all()                      # each triangle peaks at its centre bin
    # pure tones: the strongest band is one whose passband contains the tone
    t = np.arange(16000) / 16000.0
    for f0 in (300.0, 1000.0, 2500.0, 6000.0):
        tone = np.round(8000.0 * np.sin(2 * np.pi * f0 * t)).astype(np.int16)
        framed = ofe.sidekit_frames(tone.astype(np.float64), 400, 160)
        framed = framed - 0.97 * np.concatenate([framed[:, :1], framed[:, :-1]], axis=1)
        spec = np.abs(np.fft.rfft(framed * np.hanning(400), 512, axis=1)) ** 2
        band = int((spec @ fb.T).mean(axis=0).argmax())
        assert edges[band] < f0 < edges[band + 2], (f0, band)
    # frame log-energy is that of the pre-emphasised, un-windowed frame; first sample uses itself as predecessor
    sig = np.arange(1, 801, dtype=np.float64)
    out = ofe.sidekit_mfcc(sig)
    fr = ofe.sidekit_frames(sig, 400, 160)
    pre = fr - 0.97 * np.concatenate([fr[:, :1], fr[:, :-1]], axis=1)
    np.testing.assert_allclose(out[1], np.log((pre ** 2).sum(axis=1)), rtol=1e-6)
    assert fr.shape == (3, 400) and fr[1, 0] == 161.0
    # c0 is dropped: adding a gain changes no cepstrum (log-spectrum offset lives in c0 only)
    a = ofe.sidekit_mfcc(1000.0 * np.sin(2 * np.pi * 440.0 * t) + 50 * np.cos(2 * np.pi * 3000.0 * t))[0]
    b = ofe.sidekit_mfcc(4000.0 * np.sin(2 * np.pi * 440.0 * t) + 200 * np.cos(2 * np.pi * 3000.0 * t))[0]
    np.testing.assert_allclose(a, b, atol=2e-3)


def test_delta_and_scale_properties():
    """GMM_UBM.delta / preprocessing.scale restatements: linearity, constant and ramp inputs, idempotence."""
    from hypothesis import given, settings
    from hypothesis import strategies as st
    from hypothesis.extra import numpy as hnp
    import warnings

    from sklearn import preprocessing

    @settings(max_examples=40, deadline=None, derandomize=True, database=None)
    @given(hnp.arrays(np.float64, st.tuples(st.integers(1, 40), st.integers(1, 6)), elements=st.floats(-1e3, 1e3)),
           st.integers(1, 4), st.floats(-5, 5))
    def prop(x, n, a):
        d = ofe.delta(x, n)
        assert d.shape == x.shape
        np.testing.assert_allclose(ofe.delta(a * x, n), a * d, atol=1e-9 * (1 + np.abs(x).max()))   # homogeneous
        np.testing.assert_allclose(ofe.delta(x + 3.25, n), d, atol=1e-9 * (1 + np.abs(x).max()))     # offsets vanish
        s = ofe.scale(x)
        np.testing.assert_allclose(s.mean(axis=0), 0.0, atol=1e-7)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            np.testing.assert_allclose(s, preprocessing.scale(x), atol=1e-9)   # incl. columns constant up to rounding

    prop()
    ramp = np.arange(30, dtype=np.float64)[:, None] * np.array([[2.0, -0.5]])
    d = ofe.delta(ramp, 2)
    np.testing.assert_allclose(d[2:-2], np.tile([[2.0, -0.5]], (26, 1)), atol=1e-12)  # interior = slope
    np.testing.assert_allclose(d[0], np.array([2.0, -0.5]) * (1 * 1 + 2 * 2) / 10.0, atol=1e-12)  # edge padding: (c1-c0)+2(c2-c0) over 10


def test_librosa_restatement_agrees_with_transformers_audio_utils():
    """Second independent cross-check of the librosa restatement (parity unpinned): ``transformers.audio_utils`` is a
    numpy re-implementation written to reproduce librosa's mel filters and dB spectrogram."""
    au = pytest.importorskip("transformers.audio_utils")
    from speech_signal_processing_b200 import synth

    mf = au.mel_filter_bank(num_frequency_bins=1025, num_mel_filters=128, min_frequency=0.0, max_frequency=4000.0,
                            sampling_rate=8000, norm="slaney", mel_scale="slaney")
    np.testing.assert_allclose(mf.T, ofe.librosa_mel_filters(8000, 2048), atol=1e-13)
    for n in (12000, 3000):
        sig = synth.synth_utterance(3, n % 5, n, 8000).astype(np.float64)
        db = au.spectrogram(sig, au.window_function(2048, "hann", periodic=True), frame_length=2048, hop_length=512,
                            fft_length=2048, power=2.0, center=True, pad_mode="reflect", mel_filters=mf, log_mel="dB",
                            reference=1.0, min_value=1e-10, db_range=80.0)
        np.testing.assert_allclose(ofe.dct2_ortho_matrix(13, 128) @ db, ofe.librosa_mfcc(sig), atol=1e-4)


def test_sidekit_filterbank_against_an_independent_htk_mel_implementation():
    """The sidekit ``trfbank`` restatement (parity unpinned) against ``transformers.audio_utils.mel_filter_bank`` with
    the HTK mel scale and area normalisation: identical weights (1e-16) wherever the restatement is non-zero; the only
    difference is the quirk SURVEY 8(c) attributes to SIDEKIT -- the last bin of each falling edge is dropped
    (``rid[:-1]``), one bin per filter except the last, whose edge ends on the Nyquist bin."""
    au = pytest.importorskip("transformers.audio_utils")
    fb, _ = ofe.sidekit_trfbank(16000, 512, 100, 8000, 0, 24)
    mf = au.mel_filter_bank(num_frequency_bins=257, num_mel_filters=24, min_frequency=100.0, max_frequency=8000.0,
                            sampling_rate=16000, norm="slaney", mel_scale="htk").T
    nz = fb > 0
    np.testing.assert_allclose(fb[nz], mf[nz], atol=1e-15)
    extra = np.argwhere(np.abs(fb - mf) > 1e-12)
    assert all(fb[i, j] == 0.0 for i, j in extra)
    assert np.bincount(extra[:, 0], minlength=24).tolist() == [1] * 23 + [0]
    for i, j in extra:  # the dropped bin is the last one of the falling edge
        assert j == np.nonzero(mf[i])[0][-1]
