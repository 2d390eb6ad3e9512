"""Top-C fast scoring on the host: the float64 definition the GPU tests hold the kernels to (``top_components`` /
``score_top_c``, built on the float64 GMM maths of oracle/gmm.py), its known answers, and the float64 restatement
benchmarks/topc_bench.py checks the GPU with, held equal to it."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import gmm as ogmm  # noqa: E402
from speech_signal_processing_b200 import synth  # noqa: E402


def top_components(x, weights, means, variances, c):
    """Gaussian selection of top-C fast scoring (Reynolds, Quatieri & Dunn 2000): for every frame the C components with the
    largest log w_c + log N(x_t; c), in descending order, the lower index first on equal values.  Returns (idx (T, C),
    logit (T, C))."""
    wlp = ogmm.weighted_log_prob(x, weights, means, variances)
    idx = np.argsort(-wlp, axis=1, kind="stable")[:, :c]
    return idx, np.take_along_axis(wlp, idx, axis=1)


def score_top_c(x, frame_offsets, weights, variances, means, ref_model, c, idx=None):
    """Top-C fast scoring of models that share ``weights`` (K,) and ``variances`` (K, D) and differ in ``means`` (S, K, D):
    l_s(t) = log sum_{c in S_t} exp(log w_c + log N(x_t; means[s, c], variances[c])), S_t the top C of the reference
    member ``means[ref_model]`` (or the given ``idx`` (T, C)); utterance score = mean of l_s(t) over its frames (0 for an
    empty utterance).  Returns (scores (n_utts, S), frame values (S, T))."""
    x = np.asarray(x, dtype=np.float64)
    means = np.asarray(means, dtype=np.float64)
    if idx is None:
        idx, _ = top_components(x, weights, means[ref_model], variances, c)
    idx = np.asarray(idx, dtype=np.int64)
    frame = np.empty((means.shape[0], x.shape[0]))
    for s in range(means.shape[0]):
        sel = np.take_along_axis(ogmm.weighted_log_prob(x, weights, means[s], variances), idx, axis=1)
        frame[s] = ogmm.logsumexp(sel, axis=1)
    offs = np.asarray(frame_offsets, dtype=np.int64)
    scores = np.zeros((len(offs) - 1, means.shape[0]))
    for u in range(len(offs) - 1):
        if offs[u + 1] > offs[u]:
            scores[u] = frame[:, offs[u] : offs[u + 1]].mean(axis=1)
    return scores, frame


def case(s=4, k=12, d=5, lens=(30, 0, 1, 17), seed=0):
    w, mu, var = synth.synth_ubm(k, d, seed=seed, spread=1.0)
    means = np.concatenate([synth.synth_speaker_means(mu, s - 1, seed=seed + 1, shift=0.4), mu[None]])
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    x = synth.sample_gmm(w, mu, var, int(offs[-1]), seed=seed + 2)
    return x, offs, w, var, means


def test_c_equal_to_k_is_the_exact_score():
    x, offs, w, var, means = case()
    got, _ = score_top_c(x, offs, w, var, means, 3, c=12)
    for u in range(len(offs) - 1):
        for s in range(means.shape[0]):
            want = ogmm.score(x[offs[u] : offs[u + 1]], w, means[s], var) if offs[u + 1] > offs[u] else 0.0
            assert abs(got[u, s] - want) < 1e-12 * max(1.0, abs(want))


def test_c_equal_to_one_is_the_mean_of_the_best_weighted_log_probability():
    x, offs, w, var, means = case()
    got, _ = score_top_c(x, offs, w, var, means, 3, c=1)
    ref_best = ogmm.weighted_log_prob(x, w, means[3], var).argmax(axis=1)
    for s in range(means.shape[0]):
        wlp = ogmm.weighted_log_prob(x, w, means[s], var)
        per_frame = wlp[np.arange(len(x)), ref_best]
        np.testing.assert_allclose(got[0, s], per_frame[: offs[1]].mean(), rtol=1e-13)
        if s == 3:
            np.testing.assert_allclose(per_frame, wlp.max(axis=1), rtol=1e-13)


def test_duplicated_components_resolve_to_the_lower_index():
    w, mu, var = synth.synth_ubm(8, 3, seed=1, spread=1.0)
    mu[5], var[5], w[5] = mu[2], var[2], w[2]
    x = synth.sample_gmm(w / w.sum(), mu, var, 200, seed=3)
    idx, logit = top_components(x, w, mu, var, 8)
    pos2 = np.argmax(idx == 2, axis=1)
    pos5 = np.argmax(idx == 5, axis=1)
    assert (pos5 == pos2 + 1).all()
    assert (np.diff(logit, axis=1) <= 0).all()


def test_reference_member_llr_is_zero():
    x, offs, w, var, means = case()
    got, _ = score_top_c(x, offs, w, var, means, 3, c=3)
    llr = got - got[:, 3:4]
    assert (llr[:, 3] == 0.0).all()


def test_bench_restatement_equals_the_oracle():
    from benchmarks.topc_bench import reference_top_c

    x, offs, w, var, means = case(s=5, k=20, d=7, lens=(40, 0, 3, 25))
    for c in (1, 3, 20):
        idx, _ = top_components(x, w, means[-1], var, c)
        want, _ = score_top_c(x, offs, w, var, means, 4, c, idx=idx)
        np.testing.assert_allclose(reference_top_c(x, offs, w, var, means, idx), want, rtol=1e-12, atol=1e-12)
