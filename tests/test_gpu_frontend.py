"""Parity of the fused front-end kernel (through the C ABI) with the oracle / reference fixtures."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import speech_signal_processing_b200 as ssp  # noqa: E402
from oracle import frontend as ofe  # noqa: E402
from speech_signal_processing_b200 import synth  # noqa: E402

# SURVEY 8(c): |delta| <= 1e-4 * max(1, |c|) against the float64 restatement
def assert_ceps_close(got, want, tol=1e-4):
    assert got.shape == want.shape
    err = np.abs(got.astype(np.float64) - want) / np.maximum(1.0, np.abs(want))
    assert err.max() <= tol, f"max scaled error {err.max():.3e}"


def test_processing_MFCC_matches_reference_outputs(golden):
    """utils.processing.MFCC run unmodified (fixtures) vs the kernel with the 'processing' tables."""
    g = golden("processing_mfcc.npz")
    for tag in "abcd":  # c: frameSize 400 = FFT length 400 (utils/processing.py:129) -> the direct-DFT path
        fs, fsz, step = (int(v) for v in g[f"{tag}_cfg"])
        got = ssp.MFCC(g[f"{tag}_sig"], fs, fsz, step)
        assert got.dtype == np.float64
        assert_ceps_close(got, g[f"{tag}_mfcc"])


@pytest.mark.parametrize("fs,frame_size,step", [(8000, 200, 80), (16000, 400, 160), (8000, 255, 100), (16000, 1000, 400),
                                                (16000, 480, 160), (8000, 434, 200), (16000, 90, 45), (16000, 162, 80)])
def test_processing_MFCC_any_frame_size_matches_oracle(fs, frame_size, step):
    """Frame sizes that are not a power of two against the oracle restatement (itself pinned by the reference outputs
    of cases a-d): 200 / 400 / 1000 / 480 / 90 / 162 take the mixed-radix FFT (half = 2^a 3^b 5^c), 255 (odd) and 434
    (2 * 7 * 31) the direct DFT."""
    sig = synth.synth_utterance(4, frame_size % 89, 2 * fs + 123, fs)
    got = ssp.MFCC(sig, fs, frame_size, step)
    want = ofe.processing_mfcc(sig, fs, frame_size, step)
    assert_ceps_close(got, want)


@pytest.mark.parametrize("n_samples", [16000, 48000, 400, 12345])
def test_sidekit_mfcc_matches_oracle(n_samples):
    sig = synth.synth_utterance(5, n_samples % 97, n_samples)
    out = ssp.mfcc(sig)
    want = ofe.sidekit_mfcc(sig)
    assert isinstance(out, list) and len(out) == 4 and out[2] is None and out[3] is None
    assert out[0].dtype == np.float32
    assert_ceps_close(out[0], want[0])
    np.testing.assert_allclose(out[1], want[1], rtol=1e-5)


def test_sidekit_shape_witness():
    assert ssp.mfcc(synth.synth_utterance(1, 1, 16000))[0].shape == (98, 13)  # report/final.pdf p.5


def test_too_short_utterance_gives_zero_frames():
    out = ssp.mfcc(synth.synth_utterance(1, 2, 399))
    assert out[0].shape == (0, 13) and out[1].shape == (0,)


def test_float_pcm_equals_int16_pcm():
    sig = synth.synth_utterance(7, 3, 16000)
    a = ssp.mfcc(sig)[0]
    b = ssp.mfcc(sig.astype(np.float64))[0]
    # int16 PCM takes the direct-load path, float PCM the staged one: two inlined copies of the frame pipeline whose FMA
    # contractions differ in the last bit
    np.testing.assert_allclose(a, b, rtol=0, atol=1e-5)


def test_psf_recipe_matches_oracle():
    sig = synth.synth_utterance(9, 0, 16000 + 77)
    fe = ssp.FrontEnd(ssp.psf_recipe())
    feats, offs, _ = fe.extract([sig])
    want = ofe.psf_mfcc(sig)
    assert offs[-1] == want.shape[0]
    assert_ceps_close(feats.cpu().numpy(), want)


def test_delta_matches_reference(golden):
    g = golden("delta.npz")
    i = 0
    while f"x{i}" in g.files:
        got = ssp.delta(g[f"x{i}"], int(g[f"n{i}"]))
        np.testing.assert_allclose(got, g[f"d{i}"], atol=2e-6)
        i += 1
    with pytest.raises(ValueError):
        ssp.delta(g["x0"], 0)


def test_scale_matches_sklearn(golden):
    g = golden("sklearn_gmm.npz")
    got = ssp.scale(g["scale_x"])
    np.testing.assert_allclose(got, g["scale_y"], atol=2e-5)
    assert np.all(got[:, 3] == 0)  # constant column: std 0 -> divisor 1


def pipeline_train_audio(g):
    """The training half of pipeline.npz's corpus, regenerated from the seeds the fixture was made with and split the way
    GMM_UBM.py:125 does; the fixture holds its CRC instead of 0.7 MB of PCM."""
    import zlib

    from sklearn.model_selection import train_test_split

    x, y = synth.synth_corpus(4, 8, 16000)
    x_tr, _, y_tr, _ = train_test_split(x, y, test_size=0.3, random_state=0)
    assert zlib.crc32(np.stack(x_tr).tobytes()) == int(g["x_train_crc"]), "synthetic audio differs from the fixture's"
    assert list(y_tr) == list(g["y_train"])
    return x_tr


def test_extract_feature_matches_reference_pipeline(golden):
    """GMM_UBM.extract_feature (run unmodified with the sidekit restatement as mfcc) vs ONE launch."""
    g = golden("pipeline.npz")
    x = list(g["x_test"])
    feature, y = ssp.extract_feature(x, list(g["y_test"]))
    assert len(feature) == len(x)
    for j in range(len(x)):
        assert feature[j].shape == (98, 26)
        np.testing.assert_allclose(feature[j], g["feat_test"][j], atol=2e-4)
    train, feature, y = ssp.extract_feature(pipeline_train_audio(g), list(g["y_train"]), is_train=True)
    assert sorted(train) == sorted(set(g["y_train"].tolist()))
    lab0 = int(g["y_train"][0])
    np.testing.assert_allclose(train[lab0][:98], g["feat_train0"], atol=2e-4)


def test_39_dim_features_ragged_batch():
    """c + delta + delta-delta with CMVN on a ragged batch == oracle per utterance."""
    lens = [16000, 400, 20000, 399, 4321, 48000, 16001, 8000]  # (utterances 4 and 7 start on odd samples)
    sigs = [synth.synth_utterance(3 + i, i, n) for i, n in enumerate(lens)]
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True)
    feats, offs, _ = fe.extract(sigs)
    feats = feats.cpu().numpy()
    assert feats.shape[1] == 39
    for i, s in enumerate(sigs):
        got = feats[offs[i] : offs[i + 1]]
        if len(s) < 400:
            assert got.shape[0] == 0
            continue
        want = ofe.features(s, preset="sidekit", delta_order=2, cmvn=True)
        assert got.shape == want.shape
        np.testing.assert_allclose(got, want, atol=5e-4)


def test_long_utterance_30s():
    sig = synth.synth_utterance(2, 5, 480000)
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=False)
    feats, offs, _ = fe.extract([sig])
    assert offs[-1] == 2998
    c = ofe.sidekit_mfcc(sig)[0]
    want = np.hstack([c, ofe.delta(c), ofe.delta(ofe.delta(c))])
    assert_ceps_close(feats.cpu().numpy(), want)


def test_utterances_beyond_the_fused_bound_take_the_chunked_path():
    """60 s (5998 frames) does not fit the single-pass kernel's shared memory: chunks of whole frames -> raw cepstra,
    then ssp_delta / ssp_cmvn over the utterance.  Same numbers as the oracle; short neighbours are untouched."""
    long1 = synth.synth_utterance(2, 6, 16000 * 60)
    long2 = synth.synth_utterance(4, 1, 16000 * 45 + 123)
    short = [synth.synth_utterance(1, k, 16000 * 2 + 77 * k) for k in range(3)]
    out = ssp.mfcc(long1)                                              # the reference's entry point, 13-d
    want = ofe.sidekit_mfcc(long1)
    assert out[0].shape == want[0].shape == (5998, 13)
    assert_ceps_close(out[0], want[0])
    np.testing.assert_allclose(out[1], want[1], rtol=2e-5)            # frame log-energy
    batch = [short[0], long1, short[1], short[2], long2]
    for preset, recipe in (("sidekit", ssp.sidekit_recipe()), ("psf", ssp.psf_recipe())):
        fe = ssp.FrontEnd(recipe, delta_order=2, cmvn=True)
        feats, offs, _ = fe.extract(batch)
        feats = feats.cpu().numpy()
        for j, sig in enumerate(batch):
            ref = ofe.features(sig, preset=preset, delta_order=2, cmvn=True)
            got = feats[offs[j] : offs[j + 1]]
            assert got.shape == ref.shape
            np.testing.assert_allclose(got, ref, atol=2e-3 if preset == "psf" else 5e-4)


# ------------------------------------------------------------------------------------------------
# PLP (sidekit.frontend.features.plp, GMM_UBM.py:94-99): front-end kernel with a Bark filterbank + ssp_plp_post
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rasta", [True, False])
def test_plp_matches_oracle(rasta):
    """Against the float64 restatement of sidekit / rastamat PLP (parity unpinned like sidekit's mfcc: the package is
    absent).  Stated tolerance: 2e-3 absolute on liftered cepstra of magnitude 0.1 .. 10 (float32 power spectrum,
    everything after the critical-band energies in double)."""
    for n in (16000, 48000, 4000):
        sig = synth.synth_utterance(7, n % 89, n)
        got = ssp.plp(sig, rasta=rasta)
        want = ofe.sidekit_plp(sig, rasta=rasta)
        assert got[0].shape == want[0].shape and got[0].shape[1] == 13
        np.testing.assert_allclose(got[0], want[0], rtol=0, atol=2e-3)
        np.testing.assert_allclose(got[1], want[1], rtol=2e-5)
        assert got[2] is None and got[3] is None


def test_extract_feature_plp_batched():
    """GMM_UBM.extract_feature(feature_type='PLP'): plp -> delta -> hstack -> scale, for the whole list at once."""
    x, y = synth.synth_corpus(3, 3, 16000)
    train, feats, labels = ssp.extract_feature(x, y, is_train=True, feature_type="PLP")
    assert labels is y and len(feats) == len(x) and set(train) == set(y)
    for sig, f in zip(x, feats):
        c = ofe.sidekit_plp(sig)[0]
        ref = ofe.scale(np.hstack([c, ofe.delta(c)]))
        assert f.shape == ref.shape == (98, 26)
        np.testing.assert_allclose(f, ref, rtol=0, atol=2e-2)   # CMVN divides by per-column std (~0.02 .. 0.5)
    with pytest.raises(NameError):
        ssp.extract_feature(x, y, feature_type="LPCC")


@pytest.mark.parametrize("n_samples", [12000, 24000, 700, 1])
def test_MFCC_lib_matches_oracle(n_samples):
    """MFCC_DTW.MFCC_lib (librosa.feature.mfcc at sr=8000; MFCC_DTW.py:27-30): centred, mirror-padded frames of 2048,
    128 Slaney mel bands, dB with the utterance-wide 80 dB clip, DCT -- fused kernel + ssp_mel_db_post."""
    sig = synth.synth_utterance(6, n_samples % 11, n_samples, 8000)
    got = ssp.MFCC_lib(sig)
    want = ofe.mfcc_lib(sig)
    assert got.shape == want.shape == (13 * (1 + n_samples // 512),)
    assert_ceps_close(got, want)


def test_librosa_mfcc_options_match_oracle():
    sig = synth.synth_utterance(8, 2, 9000, 8000)
    for kw in (dict(pad_mode="constant"), dict(center=False), dict(top_db=None), dict(n_fft=512, hop_length=128, n_mels=40),
               dict(n_fft=400, hop_length=160, n_mels=40, sr=16000)):
        full = dict(sr=8000, n_mfcc=13)
        full.update(kw)
        got = ssp.librosa_mfcc(sig.astype(np.float32), **full)
        want = ofe.librosa_mfcc(sig.astype(np.float32), **full)
        assert got.shape == want.shape and got.shape[0] == 13
        assert_ceps_close(got, want)


def test_wav_batch_goes_to_the_front_end_without_a_repack(tmp_path):
    """read_wav_batch -> FrontEnd.extract(batch): the pinned staging buffer is uploaded as it is; same features as the
    list of arrays scipy returns for the same files (mono and stereo, ragged)."""
    from scipy.io import wavfile

    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True)
    paths, sigs = [], []
    for i, n in enumerate((16000, 4000, 48000, 399, 9000)):
        sig = synth.synth_utterance(i, 70, n_samples=n)
        if i == 2:
            sig = np.stack([sig, sig[::-1]], axis=1)
        p = tmp_path / f"u{i}.wav"
        wavfile.write(str(p), 16000, sig)
        paths.append(p)
        sigs.append(sig[:, 0] if sig.ndim == 2 else sig)
    batch = ssp.read_wav_batch(paths)
    assert batch.pcm.is_pinned()
    host, offs = fe.pack_host(batch)
    assert host.data_ptr() == batch.pcm.data_ptr()
    f_batch, o_batch, _ = fe.extract(batch)
    f_list, o_list, _ = fe.extract(sigs)
    assert np.array_equal(o_batch, o_list)
    assert bool((f_batch == f_list).all())
