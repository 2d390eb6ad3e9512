"""Top-C fast scoring of speakers MAP-adapted in weights and variances as well as means, on the host: the float64
definition the GPU tests hold ``ssp_gmm_score_topc_adapted`` to (``score_top_c_adapted``, built on oracle/gmm.py), its
known answers, the centred difference table the kernels use, and the float64 restatement
benchmarks/topc_adapted_bench.py checks the GPU with, held equal to the definition."""
import itertools
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import gmm as ogmm  # noqa: E402
from speech_signal_processing_b200 import synth  # noqa: E402
from test_topc_host import score_top_c, top_components  # noqa: E402

ADAPTS = [combo for r in (1, 2, 3) for combo in itertools.combinations(("means", "weights", "variances"), r)]


def score_top_c_adapted(x, frame_offsets, weights, means, variances, ref_model, c, idx=None):
    """Top-C fast scoring of models adapted from the reference member ``ref_model``, each with its own ``weights`` (S, K),
    ``means`` and ``variances`` (S, K, D): l_s(t) = log sum_{c in S_t} exp(log w_s,c + log N(x_t; mu_s,c, var_s,c)), S_t
    the top C of the reference member (or the given ``idx`` (T, C)); utterance score = mean of l_s(t) over its frames (0
    for an empty utterance).  Returns (scores (n_utts, S), frame values (S, T))."""
    x = np.asarray(x, dtype=np.float64)
    w, mu, var = (np.asarray(a, dtype=np.float64) for a in (weights, means, variances))
    if idx is None:
        idx, _ = top_components(x, w[ref_model], mu[ref_model], var[ref_model], c)
    idx = np.asarray(idx, dtype=np.int64)
    frame = np.empty((mu.shape[0], x.shape[0]))
    for s in range(mu.shape[0]):
        sel = np.take_along_axis(ogmm.weighted_log_prob(x, w[s], mu[s], var[s]), idx, axis=1)
        frame[s] = ogmm.logsumexp(sel, axis=1)
    offs = np.asarray(frame_offsets, dtype=np.int64)
    scores = np.zeros((len(offs) - 1, mu.shape[0]))
    for u in range(len(offs) - 1):
        if offs[u + 1] > offs[u]:
            scores[u] = frame[:, offs[u] : offs[u + 1]].mean(axis=1)
    return scores, frame


def centred_table(weights, means, variances, ref_model):
    """float64 restatement of the ssp_gmm_pack_topc_adapted table: (a, b (S, K, D), k (S, K)) with
    L_s,c(t) - L_r,c(t) = k + a . y + b . y^2, y = x_t - mu_r,c."""
    w, mu, var = (np.asarray(a, dtype=np.float64) for a in (weights, means, variances))
    delta = mu - mu[ref_model][None]
    a = delta / var
    b = -0.5 * (1.0 / var - 1.0 / var[ref_model][None])
    k = np.log(w / w[ref_model][None]) - 0.5 * np.log(var / var[ref_model][None]).sum(axis=2) - 0.5 * (delta ** 2 / var).sum(axis=2)
    return a, b, k


def adapted_set(adapt, n_spk=4, k=12, d=5, relevance=16.0, seed=0, n_enrol=(40, 0, 3, 200)):
    """(ubm (w, mu, var), speakers + UBM as stacks (S + 1, ...), member index of the UBM): speakers MAP-adapted by the
    float64 oracle from seeded enrolment frames of shifted means (one speaker of no frames, one of three)."""
    w, mu, var = synth.synth_ubm(k, d, seed=seed, spread=1.0)
    spk_mu = synth.synth_speaker_means(mu, n_spk, seed=seed + 1, shift=0.5)
    sw, smu, svar = [], [], []
    for i in range(n_spk):
        xe = synth.sample_gmm(w, spk_mu[i], var * (0.7 + 0.2 * i), n_enrol[i % len(n_enrol)], seed=seed + 10 + i)
        if len(xe):
            n, f, s, _ = ogmm.suff_stats(xe, w, mu, var)
        else:
            n, f, s = np.zeros(k), np.zeros((k, d)), np.zeros((k, d))
        nw, nm, nv = ogmm.map_adapt(n, f, s, w, mu, var, len(xe), relevance=relevance, adapt=adapt)
        sw.append(nw), smu.append(nm), svar.append(nv)
    return (w, mu, var), np.stack(sw + [w]), np.stack(smu + [mu]), np.stack(svar + [var]), n_spk


def frames(w, mu, var, lens=(30, 0, 1, 17), seed=5):
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    return synth.sample_gmm(w, mu, var, int(offs[-1]), seed=seed), offs


@pytest.mark.parametrize("adapt", ADAPTS)
def test_c_equal_to_k_is_the_exact_score(adapt):
    (w, mu, var), sw, smu, svar, r = adapted_set(adapt)
    x, offs = frames(w, mu, var)
    got, _ = score_top_c_adapted(x, offs, sw, smu, svar, r, c=12)
    for u in range(len(offs) - 1):
        for s in range(sw.shape[0]):
            xs = x[offs[u] : offs[u + 1]]
            want = ogmm.score(xs, sw[s], smu[s], svar[s]) if len(xs) else 0.0
            assert abs(got[u, s] - want) < 1e-12 * max(1.0, abs(want)), (adapt, u, s)


def test_mean_only_stacks_equal_the_shared_definition():
    (w, mu, var), sw, smu, svar, r = adapted_set(("means",))
    x, offs = frames(w, mu, var)
    for c in (1, 3, 12):
        got, got_frame = score_top_c_adapted(x, offs, sw, smu, svar, r, c)
        want, want_frame = score_top_c(x, offs, w, var, smu, r, c)
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(got_frame, want_frame)


@pytest.mark.parametrize("adapt", ADAPTS)
def test_ubm_member_llr_is_zero(adapt):
    (w, mu, var), sw, smu, svar, r = adapted_set(adapt)
    x, offs = frames(w, mu, var)
    got, _ = score_top_c_adapted(x, offs, sw, smu, svar, r, c=3)
    assert ((got - got[:, r : r + 1])[:, r] == 0.0).all()


def test_c_equal_to_one_is_the_mean_of_the_speaker_logit_at_the_ubm_best_component():
    (w, mu, var), sw, smu, svar, r = adapted_set(("means", "weights", "variances"))
    x, offs = frames(w, mu, var)
    got, _ = score_top_c_adapted(x, offs, sw, smu, svar, r, c=1)
    best = ogmm.weighted_log_prob(x, w, mu, var).argmax(axis=1)
    for s in range(sw.shape[0]):
        per_frame = ogmm.weighted_log_prob(x, sw[s], smu[s], svar[s])[np.arange(len(x)), best]
        np.testing.assert_allclose(got[0, s], per_frame[: offs[1]].mean(), rtol=1e-13)
        np.testing.assert_allclose(got[3, s], per_frame[offs[3] :].mean(), rtol=1e-13)


# relevance 0 for the combinations without variances: variance MAP at relevance 0 gives a component of one frame a zero
# variance, which ModelSet.with_ubm refuses
@pytest.mark.parametrize("adapt,relevance", [(a, 16.0) for a in ADAPTS] + [(a, 0.0) for a in ADAPTS if "variances" not in a])
def test_centred_table_equals_the_logit_difference(adapt, relevance):
    (w, mu, var), sw, smu, svar, r = adapted_set(adapt, relevance=relevance)
    x, _ = frames(w, mu, var, lens=(300,))
    a, b, k = centred_table(sw, smu, svar, r)
    lr = ogmm.weighted_log_prob(x, sw[r], smu[r], svar[r])
    y = x[:, None, :] - smu[r][None]                                    # (T, K, D)
    for s in range(sw.shape[0]):
        want = ogmm.weighted_log_prob(x, sw[s], smu[s], svar[s]) - lr
        got = k[s][None] + (a[s][None] * y).sum(axis=2) + (b[s][None] * y * y).sum(axis=2)
        err = np.abs(got - want) / np.maximum(1.0, np.abs(want))
        assert err.max() <= 1e-12, (adapt, relevance, s, err.max())
    # the UBM member has a row of exact zeros; so does the speaker enrolled on no frames in what MAP leaves bit-exact (its
    # means; its renormalised weights and its variances var + mu^2 - mu^2 may move by an ulp)
    assert (a[r] == 0).all() and (b[r] == 0).all() and (k[r] == 0).all()
    assert (a[1] == 0).all()
    if "variances" not in adapt:
        assert (b[1] == 0).all()
        if "weights" not in adapt:
            assert (k[1] == 0).all()


def test_bench_restatement_equals_the_definition():
    from benchmarks.topc_adapted_bench import reference_top_c_adapted

    (w, mu, var), sw, smu, svar, r = adapted_set(("means", "weights", "variances"), k=20, d=7)
    x, offs = frames(w, mu, var, lens=(40, 0, 3, 25))
    for c in (1, 3, 20):
        idx, _ = top_components(x, w, mu, var, c)
        want, _ = score_top_c_adapted(x, offs, sw, smu, svar, r, c, idx=idx)
        np.testing.assert_allclose(reference_top_c_adapted(x, offs, sw, smu, svar, idx), want, rtol=1e-12, atol=1e-12)
