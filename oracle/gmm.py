"""numpy (float64) restatement of the diag-covariance GMM maths the reference
reaches through sklearn.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Reference call sites: GMM_UBM.py:158-160,169-170 (fit), :185,194 (score).
sklearn lines cited are sklearn 1.9.0 (``sklearn/mixture/_gaussian_mixture.py``,
``sklearn/mixture/_base.py``), the reference's own (un-pinned) dependency.
"""
from __future__ import annotations

import numpy as np

LOG_2PI = float(np.log(2.0 * np.pi))


def log_gaussian_prob(x, means, variances):
    """_gaussian_mixture.py:536-553 (diag branch): log N(x_t; mu_c, diag var_c), (T, K)."""
    x = np.asarray(x, dtype=np.float64)
    means = np.asarray(means, dtype=np.float64)
    prec = 1.0 / np.asarray(variances, dtype=np.float64)
    d = x.shape[1]
    log_det = 0.5 * np.log(prec).sum(axis=1)
    quad = (means ** 2 * prec).sum(axis=1) - 2.0 * x @ (means * prec).T + (x * x) @ prec.T
    return -0.5 * (d * LOG_2PI + quad) + log_det


def weighted_log_prob(x, weights, means, variances):
    """_base.py:513-525: log w_c + log N(x_t | c)."""
    return log_gaussian_prob(x, means, variances) + np.log(np.asarray(weights, dtype=np.float64))


def logsumexp(a, axis=1):
    m = a.max(axis=axis, keepdims=True)
    return (m + np.log(np.exp(a - m).sum(axis=axis, keepdims=True))).squeeze(axis)


def score_samples(x, weights, means, variances):
    """_base.py:373: per-frame log-likelihood."""
    return logsumexp(weighted_log_prob(x, weights, means, variances), axis=1)


def score(x, weights, means, variances):
    """_base.py:393: mean per-frame log-likelihood (what GMM_UBM.py:185 subtracts)."""
    return float(score_samples(x, weights, means, variances).mean())


def responsibilities(x, weights, means, variances):
    """_base.py:552-582: (frame log-lik, posterior gamma)."""
    wlp = weighted_log_prob(x, weights, means, variances)
    lse = logsumexp(wlp, axis=1)
    return lse, np.exp(wlp - lse[:, None])


def suff_stats(x, weights, means, variances):
    """Zeroth/first/second order statistics N (K,), F (K,D), S (K,D) and sum of frame
    log-likelihoods -- the quantities _gaussian_mixture.py:312-313,250-252 forms as
    resp.T @ [1, X, X*X]."""
    x = np.asarray(x, dtype=np.float64)
    lse, gamma = responsibilities(x, weights, means, variances)
    return gamma.sum(axis=0), gamma.T @ x, gamma.T @ (x * x), float(lse.sum())


def m_step(n, f, s, reg_covar=1e-6, eps=None):
    """_gaussian_mixture.py:312-313 (nk + 10 eps), :250-252 (diag covariances),
    :898 (weights normalised by their sum)."""
    if eps is None:
        eps = np.finfo(np.float64).eps
    nk = n + 10.0 * eps
    means = f / nk[:, None]
    variances = s / nk[:, None] - means ** 2 + reg_covar
    weights = nk / nk.sum()
    return weights, means, variances


def em_fit(x, weights, means, variances, max_iter=100, tol=1e-3, reg_covar=1e-6, eps=None):
    """_base.py:258-312: EM loop from given initial parameters.  Returns
    (weights, means, variances, n_iter, converged, lower_bounds)."""
    x = np.asarray(x, dtype=np.float64)
    lower = -np.inf
    bounds = []
    converged = False
    n_iter = 0
    for n_iter in range(1, max_iter + 1):
        prev = lower
        n, f, s, ll = suff_stats(x, weights, means, variances)
        weights, means, variances = m_step(n, f, s, reg_covar, eps)
        lower = ll / x.shape[0]
        bounds.append(lower)
        if abs(lower - prev) < tol:
            converged = True
            break
    return weights, means, variances, n_iter, converged, bounds


def map_adapt(n, f, s, weights, means, variances, n_frames, relevance=16.0,
              adapt=("means",)):
    """Reynolds, Quatieri & Dunn (2000) eq. 11-14 relevance MAP from UBM statistics.

    alpha_c = n_c / (n_c + r); mu^_c = alpha E_c[x] + (1-alpha) mu_c
    (optionally) w^_c ~ alpha n_c / T + (1-alpha) w_c, renormalised;
    var^_c = alpha E_c[x^2] + (1-alpha)(var_c + mu_c^2) - mu^_c^2.
    A speaker or component without data keeps the UBM's parameters: alpha = 0 where n_c = 0 (also at relevance 0),
    and the weight term alpha n_c / T is 0 for a speaker of T = 0 frames.
    The reference has no MAP code (SURVEY F4): parity unpinned, defined by formula.
    """
    n = np.asarray(n, dtype=np.float64)
    alpha = np.divide(n, n + relevance, out=np.zeros_like(n), where=n > 0)[:, None]
    safe = np.maximum(n, np.finfo(np.float64).tiny)[:, None]
    ex = f / safe
    ex2 = s / safe
    new_means = alpha * ex + (1.0 - alpha) * means if "means" in adapt else np.array(means, dtype=np.float64)
    new_w = np.array(weights, dtype=np.float64)
    if "weights" in adapt:
        new_w = (alpha[:, 0] * n / n_frames if n_frames > 0 else 0.0) + (1.0 - alpha[:, 0]) * weights
        new_w = new_w / new_w.sum()
    new_var = np.array(variances, dtype=np.float64)
    if "variances" in adapt:
        new_var = alpha * ex2 + (1.0 - alpha) * (variances + np.asarray(means) ** 2) - new_means ** 2
    return new_w, new_means, new_var


def identify(utts, models, ubm=None):
    """GMM_UBM.py:182-197: pred[j, i] = GMM[i].score(x_j) - UBM.score(x_j); argmax over i."""
    pred = np.zeros((len(utts), len(models)))
    for j, x in enumerate(utts):
        base = score(x, *ubm) if ubm is not None else 0.0
        for i, m in enumerate(models):
            pred[j, i] = score(x, *m) - base
    return pred, pred.argmax(axis=1)
