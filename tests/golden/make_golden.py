#!/usr/bin/env python
"""Generate the committed golden fixtures by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference and sklearn 1.9.0):

    python tests/golden/make_golden.py [processing|sklearn|pipeline|vad|config1 ...]

Writes small ``.npz`` files next to this script.  The reference modules are imported
through ``oracle.ref_shims`` (stub modules for the absent GUI/audio packages).

Fixtures
--------
processing_mfcc.npz   utils/processing.py::MFCC / enframe / mfccInitFilterBanks outputs
delta.npz             GMM_UBM.py::delta outputs
sklearn_gmm.npz       sklearn GaussianMixture(diag) score_samples / predict_proba / fit
                      trajectory from fixed initial parameters, preprocessing.scale
vad.npz               VAD.py::enframe / ZCR / energy / spectrum_entropy / feature / VAD_detection / VAD_frequency
                      on synthetic bursts-in-noise signals
config1.npz           BASELINE configs[0] at its stated size (10 speakers x 30 utterances x 3 s, 64 components) through the
                      unmodified GMM_UBM.py::extract_feature + GMM(): reference-trained models, LLR matrix, accuracy line
pipeline.npz          GMM_UBM.py::extract_feature + GMM() end to end on synthetic audio with
                      the sidekit restatement plugged in as ``mfcc`` and a seeded
                      GaussianMixture (random_state only; everything else stock)
"""
from __future__ import annotations

import contextlib
import functools
import io
import os
import pickle
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import frontend as ofe  # noqa: E402
from oracle import ref_shims  # noqa: E402
from speech_signal_processing_b200 import synth  # noqa: E402


def gen_processing():
    proc = ref_shims.load("utils.processing")
    out = {}
    cases = [("a", 8000, 512, 256, 4000), ("b", 16000, 512, 160, 4800), ("c", 16000, 400, 160, 4000),
             ("d", 8000, 256, 128, 1500)]
    for tag, fs, fsz, step, n in cases:
        sig = synth.synth_utterance(3, ord(tag), n, fs)
        out[f"{tag}_sig"] = sig
        out[f"{tag}_cfg"] = np.array([fs, fsz, step])
        out[f"{tag}_mfcc"] = proc.MFCC(sig, fs, fsz, step)
    fb, fr = proc.mfccInitFilterBanks(16000, 512)
    out["fbank_16k_512"] = fb
    out["freqs_16k_512"] = fr
    fb, fr = proc.mfccInitFilterBanks(8000, 512)
    out["fbank_8k_512"] = fb
    out["enframe_a"] = proc.enframe(out["a_sig"].astype(np.float64), 400, 160)
    np.savez_compressed(os.path.join(HERE, "processing_mfcc.npz"), **out)


def gen_delta(gu):
    rs = np.random.RandomState(7)
    out = {}
    for i, (t, f, n) in enumerate([(1, 13, 2), (2, 13, 2), (3, 5, 2), (4, 13, 2), (5, 13, 2), (37, 13, 2), (50, 13, 1), (50, 13, 3),
                                   (298, 13, 2)]):
        x = rs.standard_normal((t, f))
        out[f"x{i}"] = x
        out[f"n{i}"] = np.array(n)
        out[f"d{i}"] = gu.delta(x, n)
    ramp = np.arange(20, dtype=np.float64)[:, None] * np.array([[1.0, -2.0]])
    out["ramp"] = ramp
    out["ramp_d"] = gu.delta(ramp, 2)
    np.savez_compressed(os.path.join(HERE, "delta.npz"), **out)


def gen_sklearn():
    from sklearn import preprocessing
    from sklearn.mixture import GaussianMixture

    out = {}
    for tag, k, d, n in [("s", 8, 5, 400), ("m", 64, 26, 1000), ("l", 128, 39, 600)]:
        w, mu, var = synth.synth_ubm(k, d, seed=11 + k)
        x = synth.sample_gmm(w, mu * 0.9, var * 1.3, n, seed=k).astype(np.float64)
        import warnings

        gm = GaussianMixture(n_components=k, covariance_type="diag")
        # load fixed parameters the way an unpickled model carries them (GMM_UBM.py:141-146)
        gm.weights_, gm.means_, gm.covariances_ = w, mu, var
        gm.precisions_cholesky_ = 1.0 / np.sqrt(var)
        out[f"{tag}_w"], out[f"{tag}_mu"], out[f"{tag}_var"], out[f"{tag}_x"] = w, mu, var, x
        out[f"{tag}_score_samples"] = gm.score_samples(x)
        out[f"{tag}_score"] = np.array(gm.score(x))
        if k <= 64:
            # on a 2^-52 grid (no value moves by more than 1.2e-16, far inside the tests' 1e-12): most entries become
            # exact zeros, which takes 0.5 MB off the fixture
            out[f"{tag}_proba"] = np.round(gm.predict_proba(x) * 2.0 ** 52) / 2.0 ** 52
        # EM trajectory from fixed init, stock tolerances
        for iters in (1, 3, 100):
            g2 = GaussianMixture(n_components=k, covariance_type="diag", weights_init=w, means_init=mu,
                                 precisions_init=1.0 / var, max_iter=iters)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                g2.fit(x)
            out[f"{tag}_fit{iters}_w"] = g2.weights_
            out[f"{tag}_fit{iters}_mu"] = g2.means_
            out[f"{tag}_fit{iters}_var"] = g2.covariances_
            out[f"{tag}_fit{iters}_niter"] = np.array(g2.n_iter_)
            out[f"{tag}_fit{iters}_lb"] = np.array(g2.lower_bound_)
            out[f"{tag}_fit{iters}_conv"] = np.array(g2.converged_)
    rs = np.random.RandomState(3)
    xs = rs.standard_normal((57, 26)) * rs.uniform(0.1, 30, size=(1, 26)) + rs.uniform(-50, 50, size=(1, 26))
    xs[:, 3] = 4.25  # constant column -> std 0 -> divisor 1
    out["scale_x"] = xs
    out["scale_y"] = preprocessing.scale(xs)
    out["scale_y32"] = preprocessing.scale(xs.astype(np.float32))
    np.savez_compressed(os.path.join(HERE, "sklearn_gmm.npz"), **out)


def gen_pipeline():
    """Reference extract_feature + GMM() on 4 synthetic speakers x 6 utterances of 1 s."""
    from sklearn.mixture import GaussianMixture

    def mfcc_cepstra(sig, **kw):  # GMM_UBM.py:89 omits the [0] (SURVEY F6); contract = cepstra ndarray
        return ofe.sidekit_mfcc(sig, **kw)[0]

    gu = ref_shims.load("GMM_UBM", sidekit_mfcc=mfcc_cepstra)
    gu.mfcc = mfcc_cepstra
    gen_delta(gu)

    n_spk, n_utt, n_samp, k = 4, 8, 16000, 4
    x, y = synth.synth_corpus(n_spk, n_utt, n_samp)
    from sklearn.model_selection import train_test_split

    x_tr, x_te, y_tr, y_te = train_test_split(x, y, test_size=0.3, random_state=0)  # GMM_UBM.py:125
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
        train, f_tr, y_tr2 = gu.extract_feature(x=x_tr, y=y_tr, is_train=True)
        f_te, y_te2 = gu.extract_feature(x=x_te, y=y_te)
    gu.label_encoder.clear()
    gu.label_encoder.update({f"spk{i}": i for i in range(n_spk)})
    gu.GaussianMixture = functools.partial(GaussianMixture, random_state=0)
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
                gu.GMM(train, f_tr, y_tr2, f_te, y_te2, n_components=k, model=False)
            with open("Model/GMM_MFCC_model.pkl", "rb") as f:
                gmms = pickle.load(f)
            with open("Model/UBM_MFCC_model.pkl", "rb") as f:
                ubm = pickle.load(f)
        finally:
            os.chdir(cwd)
    line = [ln for ln in buf.getvalue().splitlines() if "train acc" in ln][-1]
    pred = np.zeros((len(f_te), len(gmms)))
    for i in range(len(gmms)):
        for j in range(len(f_te)):
            pred[j, i] = gmms[i].score(f_te[j]) - ubm.score(f_te[j])  # GMM_UBM.py:194
    import zlib

    out = {  # the training audio is regenerated from the seeds by the test: only its CRC is stored
        "x_test": np.stack(x_te), "y_test": np.array(y_te2), "x_train_crc": np.array(zlib.crc32(np.stack(x_tr).tobytes())),
        "y_train": np.array(y_tr2),
        "feat_test": np.stack(f_te).astype(np.float64), "feat_train0": np.asarray(f_tr[0], dtype=np.float64),
        "gmm_w": np.stack([g.weights_ for g in gmms]), "gmm_mu": np.stack([g.means_ for g in gmms]),
        "gmm_var": np.stack([g.covariances_ for g in gmms]),
        "ubm_w": ubm.weights_, "ubm_mu": ubm.means_, "ubm_var": ubm.covariances_,
        "pred": pred, "printed": np.array(line),
    }
    np.savez_compressed(os.path.join(HERE, "pipeline.npz"), **out)
    print("reference GMM() printed:", line)


CONFIG1 = dict(n_spk=10, n_utt=30, n_samp=48000, k=64)  # BASELINE configs[0] at its stated size


def config1_split():
    """The corpus and the reference's own split (GMM_UBM.py:125) of BASELINE configs[0]; shared with the GPU test, which
    regenerates the audio from the seeds instead of shipping 29 MB of PCM."""
    from sklearn.model_selection import train_test_split

    x, y = synth.synth_corpus(CONFIG1["n_spk"], CONFIG1["n_utt"], CONFIG1["n_samp"])
    return train_test_split(x, y, test_size=0.3, random_state=0)


def gen_config1():
    """BASELINE configs[0] ("GMM_UBM.py default pipeline on CPU: 13-dim MFCC ... + 64-comp diag GMM, 10 speakers,
    synthetic audio") run through the UNMODIFIED reference extract_feature + GMM() (sidekit restatement plugged in as
    ``mfcc``, seeded GaussianMixture).  Stored: the reference-trained models, the LLR matrix ``pred`` of the 90 test
    utterances (GMM_UBM.py:191-194), the printed accuracy line and a fingerprint of audio + features."""
    import zlib

    from sklearn.mixture import GaussianMixture

    def mfcc_cepstra(sig, **kw):
        return ofe.sidekit_mfcc(sig, **kw)[0]

    gu = ref_shims.load("GMM_UBM", sidekit_mfcc=mfcc_cepstra)
    gu.mfcc = mfcc_cepstra
    x_tr, x_te, y_tr, y_te = config1_split()
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        train, f_tr, y_tr2 = gu.extract_feature(x=x_tr, y=y_tr, is_train=True)
        f_te, y_te2 = gu.extract_feature(x=x_te, y=y_te)
    gu.label_encoder.clear()
    gu.label_encoder.update({f"spk{i}": i for i in range(CONFIG1["n_spk"])})
    gu.GaussianMixture = functools.partial(GaussianMixture, random_state=0)
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(io.StringIO()):
                gu.GMM(train, f_tr, y_tr2, f_te, y_te2, n_components=CONFIG1["k"], model=False)
            with open("Model/GMM_MFCC_model.pkl", "rb") as f:
                gmms = pickle.load(f)
            with open("Model/UBM_MFCC_model.pkl", "rb") as f:
                ubm = pickle.load(f)
        finally:
            os.chdir(cwd)
    line = [ln for ln in buf.getvalue().splitlines() if "train acc" in ln][-1]
    pred = np.zeros((len(f_te), len(gmms)))
    for i in range(len(gmms)):
        for j in range(len(f_te)):
            pred[j, i] = gmms[i].score(f_te[j]) - ubm.score(f_te[j])  # GMM_UBM.py:194
    out = {
        "y_test": np.array(y_te2), "pred": pred, "printed": np.array(line),
        "audio_crc": np.array(zlib.crc32(np.concatenate(x_te).tobytes())),
        "feat_first": np.asarray(f_te[0], dtype=np.float64), "feat_last": np.asarray(f_te[-1], dtype=np.float64),
        "feat_abs_mean": np.array([np.abs(f).mean() for f in f_te]),
        "gmm_w": np.stack([g.weights_ for g in gmms]), "gmm_mu": np.stack([g.means_ for g in gmms]).astype(np.float32),
        "gmm_var": np.stack([g.covariances_ for g in gmms]).astype(np.float32),
        "ubm_w": ubm.weights_, "ubm_mu": ubm.means_.astype(np.float32), "ubm_var": ubm.covariances_.astype(np.float32),
    }
    # the models are stored in float32 (half the bytes); pred is recomputed from the stored parameters so that the
    # fixture is self-consistent (the float32 rounding of a parameter moves a score by ~1e-6)
    def sk(wt, m, v):
        e = GaussianMixture(n_components=len(wt), covariance_type="diag")
        e.weights_, e.means_, e.covariances_ = wt, m.astype(np.float64), v.astype(np.float64)
        e.precisions_cholesky_ = 1 / np.sqrt(e.covariances_)
        return e

    u32 = sk(out["ubm_w"], out["ubm_mu"], out["ubm_var"])
    g32 = [sk(out["gmm_w"][i], out["gmm_mu"][i], out["gmm_var"][i]) for i in range(len(gmms))]
    pred32 = np.array([[g.score(f) - u32.score(f) for g in g32] for f in f_te])
    assert np.abs(pred32 - pred).max() < 1e-4 and (pred32.argmax(1) == pred.argmax(1)).all()
    out["pred"] = pred32
    sorted_llr = np.sort(pred32, axis=1)
    out["min_top2_margin"] = np.array((sorted_llr[:, -1] - sorted_llr[:, -2]).min())
    np.savez_compressed(os.path.join(HERE, "config1.npz"), **out)
    print("config 1: reference GMM() printed:", line, "| min top-2 LLR margin", float(out["min_top2_margin"]))


def vad_signal(seed: int, n: int, bursts):
    """int16 test signal for the VAD: noise floor + voiced bursts (harmonics) + one unvoiced (noisy) burst."""
    rs = np.random.RandomState(seed)
    t = np.arange(n) / 8000.0
    x = 40.0 * rs.standard_normal(n)
    for lo, hi, f0, amp in bursts:
        seg = slice(lo, hi)
        if f0 > 0:
            x[seg] += amp * (np.sin(2 * np.pi * f0 * t[seg]) + 0.5 * np.sin(2 * np.pi * 2 * f0 * t[seg] + 0.3))
        else:
            x[seg] += amp * rs.standard_normal(hi - lo)
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


VAD_CASES = [
    (1, 24000, [(3000, 9000, 140.0, 9000.0), (9000, 10500, 0.0, 1500.0), (15000, 21000, 210.0, 6000.0)]),
    (2, 16000, [(200, 7000, 110.0, 12000.0), (7600, 8200, 180.0, 8000.0), (12000, 15990, 160.0, 10000.0)]),  # run reaches the end
    (3, 9000, [(0, 4000, 250.0, 7000.0)]),                                                                     # speech from frame 0
    (4, 5000, [(2000, 2050, 500.0, 20000.0)]),                                                                 # noise + a click: no speech
    (5, 20011, [(2500, 5200, 95.0, 11000.0), (5300, 9000, 0.0, 4000.0), (11000, 11900, 300.0, 9000.0), (13000, 19000, 130.0, 3000.0)]),
]


def gen_vad():
    """VAD.py (SURVEY 8(f).4) on synthetic signals: framing, per-frame features, both detectors."""
    ref_shims._stub("bayes_opt", BayesianOptimization=object)
    ref_shims._stub("seaborn")
    vad = ref_shims.load("VAD")
    out = {"n_cases": np.array(len(VAD_CASES))}
    for i, (seed, n, bursts) in enumerate(VAD_CASES):
        sig = vad_signal(seed, n, bursts)
        wave = sig / (max(abs(sig.astype(np.int64))))          # VAD.py:133 (abs in int64: no int16 wrap at -32768)
        frames = vad.enframe(wave)
        with contextlib.redirect_stdout(io.StringIO()):
            z, p, e = vad.feature(frames)
        out[f"sig{i}"] = sig
        if frames.shape[1] <= 80:
            out[f"frames{i}"] = frames   # the larger ones are re-derived in the tests (enframe is pinned by the small ones)
        out[f"zcr_raw{i}"] = vad.ZCR(frames)
        out[f"zcr{i}"], out[f"power{i}"], out[f"entropy{i}"] = z, p, e
        out[f"det{i}"] = vad.VAD_detection(z, p)
        out[f"det_b{i}"] = vad.VAD_detection(z, p, zcr_gate=25, ampl=1.0, amph=8)
        out[f"freq{i}"] = vad.VAD_frequency(e)
    np.savez_compressed(os.path.join(HERE, "vad.npz"), **out)
    print("vad.npz: speech frames per case", [int(out[f"det{i}"].sum()) for i in range(len(VAD_CASES))])


if __name__ == "__main__":
    if not ref_shims.available():
        sys.exit("reference tree not found; fixtures can only be generated in the build container")
    only = set(sys.argv[1:])
    for name, fn in (("processing", gen_processing), ("sklearn", gen_sklearn), ("pipeline", gen_pipeline), ("vad", gen_vad),
                     ("config1", gen_config1)):
        if not only or name in only:
            fn()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
