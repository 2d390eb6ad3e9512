"""GMM kernels at every feature-width specialisation and component-tile edge, against the float64 oracle.

Each width class has its own instantiation: the CUDA-core kernels pad D to DP in {16, 32, 40, 64, 80}; the tensor
rungs contract over KD = roundup(2D + 2, 8) (TF32 images) or KDb = roundup(2D + 2, 16) (FP16 / BF16 images); the
shared-variance kernel over KS = roundup(D + 2, 16).  Components are padded to tiles of 128 (64 in the shared-variance
kernel).  The layout restatement and the coverage guard need no device; every other test is marked ``gpu``.
"""
import ctypes as C
import warnings

import numpy as np
import pytest

from oracle import gmm as ogmm

EM_TENSOR_KERNELS = {"em_plan_kernel", "em_prep_kernel", "gmm_em_lse_kernel", "em_merge_kernel", "gmm_em_stats_kernel"}
EM_SIMT_KERNELS = {"gmm_score_simt_kernel", "gmm_stats_simt_kernel"}

# widths: the tensor scoring rungs (D <= 39), the CUDA-core kernels beyond, the tensor statistics, the shared variance
SCORE_WIDTHS = [1, 2, 3, 4, 7, 8, 15, 16, 17, 23, 24, 31, 32, 33, 38, 39]
SCORE_COMPONENTS = [1, 2, 127, 129]
SIMT_WIDTHS = [40, 41, 63, 64, 65, 79, 80]
STATS_WIDTHS = [1, 2, 3, 7, 8, 15, 16, 23, 24, 31, 32, 39]
STATS_COMPONENTS = [1, 127, 129]
SV_WIDTHS = [1, 14, 15, 30, 31, 39]
SV_COMPONENTS = [1, 63, 64, 65]
UTT_LENS = [1, 2, 127, 128, 129, 300]
SEG_LENS = [0, 1, 63, 64, 65]          # the statistics workspace pads segments to 64 frames

# Per-frame error bound of a log-likelihood: c * u * (sum_d |x_d mu_d / var_d| + x_d^2 / (2 var_d) + |const| + 1)
# for the component where it is largest (log-sum-exp moves by at most the largest logit error).  The sum is what
# the contraction adds up; the 1 covers the FP32 exponentials and logarithm.  u is the unit roundoff of the
# operands: 2^-11 (11-bit significands of TF32 / FP16) when the frame or the model is rounded once, 2^-22 when both
# are split into two pieces (3-pass rung) and for the FP32 CUDA-core kernel.  The statistics kernels form their logits
# from three products of BF16 hi / lo pieces (8-bit significands): u = 2^-18.  The shared-variance kernel's reference
# member (common part split in FP16 pieces) has no derived bound here: u = 2^-16 is set from its measured error.
# Largest errors measured on a B200 (1 000 W), in units of u * terms: fp32 1.05, tf32 0.73, tf32x2 0.45, tf32x3 4.4
# (D = 1, K = 1), shared-variance speakers 0.10 and reference member 1.9 (D = 1, K = 1), statistics log-likelihood 0.56.
# Every test prints its largest ratio (profiles/r3b_pytest_gpu_widths.log).
U = {"fp32": 2.0 ** -22, "tf32": 2.0 ** -11, "tf32x2": 2.0 ** -11, "tf32x3": 2.0 ** -22, "stats": 2.0 ** -18,
     "sv_reference": 2.0 ** -16}
C_BOUND = 8.0
# posteriors enter the statistics GEMM as FP16 (11-bit significand)
U_GAMMA = 2.0 ** -11
# ... and the frame values v (x and x^2) as FP16 hi + lo pieces: within 2^-22 |v| in FP16's normal range, and within half the
# smallest FP16 subnormal below 2^-14 (x^2 of every |x| < 2^-7): an absolute 2^-25 per frame and unit of posterior
X_FLOOR = 2.0 ** -25


@pytest.fixture(scope="module")
def lib():
    from speech_signal_processing_b200 import _lib, build

    build.build()
    return _lib.load()


# ------------------------------------------------------------------------------------------------ layout restatement
def pad_feat(d):
    return next(p for p in (16, 32, 40, 64, 80) if d <= p)


def _up(x, g):
    return (x + g - 1) // g * g


def kd(d):
    return _up(2 * d + 2, 8)


def kdb(d):
    return _up(2 * d + 2, 16)


def ks(d):
    return _up(d + 2, 16)


def pack_bytes(n_models, k, d):
    """make_layout in csrc/common.cuh: bytes of the packed-model buffer, 0 when D is outside [1, 80]."""
    if not 1 <= d <= 80:
        return 0
    kp = _up(k, 128)
    o = _up(n_models * kp * pad_feat(d) * 8, 128)             # CUDA-core rows (float2)
    o = _up(o + n_models * kp * 4, 128)                       # constants
    o = _up(o + n_models * kp * kd(d) * 4, 128)               # TF32 images
    o = _up(o + n_models * kp * kd(d) * 4, 128)               # their residuals
    if 2 * d + 2 <= 80:
        if n_models <= 1024:
            o = _up(o + n_models * (kp // 128) * 512 * kdb(d), 128)   # BF16 hi + lo images (statistics)
        o = _up(o + n_models * kp * kdb(d) * 2, 128)          # FP16 images
        o = _up(o + n_models * kp * kdb(d) * 2, 128)          # FP16 residuals
        o = _up(o + 128, 128)                                 # range flag
    return o


def sv_smem_bytes(ks_, kq, stages=12, slots=6, chunk=32, unit=256, tile=64):
    return 2 * unit * kq * 2 + stages * tile * ks_ * 2 + 2 * chunk * unit * 4 + (2 * stages + 2 * slots + 2) * 8 + 16 + unit * 4


def shared_pack_bytes(n_models, k, d):
    """make_sv_layout in csrc/common.cuh: 0 when KS > 64 or the kernel's shared memory exceeds 227 KB (D > 39)."""
    if d < 1 or ks(d) > 64 or sv_smem_bytes(ks(d), kdb(d)) > 232448:
        return 0
    return (_up(k, 64) // 64) * (n_models + 4) * 64 * ks(d) * 2 + 128


def test_layout_restatement_matches_the_library(lib):
    from speech_signal_processing_b200 import _lib

    for d in range(0, 83):
        for n_models, k in ((1, 1), (1, 129), (3, 64), (1025, 65)):
            dims = _lib.GmmDims(n_models, k, d)
            assert lib.ssp_gmm_pack_bytes(C.byref(dims)) == pack_bytes(n_models, k, d), (n_models, k, d)
            assert lib.ssp_gmm_shared_pack_bytes(C.byref(dims)) == shared_pack_bytes(n_models, k, d), (n_models, k, d)


def _steps(f, widths):
    """[(top, first)] of every run of equal f over the widths: where a specialisation changes."""
    return [(d, d + 1) for d in widths[:-1] if f(d) != f(d + 1)]


def test_width_lists_cover_every_boundary():
    tensor = [d for d in range(1, 81) if pack_bytes(1, 1, d) and kd(d) <= 80]       # the tensor rungs' widths
    assert tensor == list(range(1, 40))
    widest = tensor[-1]
    fp32_scored = set(SCORE_WIDTHS) | set(SIMT_WIDTHS)
    for top, first in _steps(pad_feat, list(range(1, 81))):                          # CUDA-core DP
        assert {top, first} <= fp32_scored, (top, first)
    assert {1, 80} <= fp32_scored
    for top, first in _steps(kdb, tensor):                                            # FP16 / BF16 images
        assert {top, first} <= set(SCORE_WIDTHS) and {top, first} <= set(STATS_WIDTHS), (top, first)
    assert kd(3) == 8 and kd(4) == 16 and {1, 3, 4, widest} <= set(SCORE_WIDTHS)      # single TF32 k-step, widest
    assert {1, widest} <= set(STATS_WIDTHS) and {widest + 1, 80} <= set(SIMT_WIDTHS)
    sv = [d for d in range(1, 81) if shared_pack_bytes(1, 1, d)]
    assert sv == list(range(1, sv[-1] + 1))
    for top, first in _steps(ks, sv):
        assert {top, first} <= set(SV_WIDTHS), (top, first)
    assert {1, sv[-1]} <= set(SV_WIDTHS)
    # component tiles: a single component, one real component in the last 128- (64-) tile, a full tile
    assert {1, 127, 129} <= set(SCORE_COMPONENTS) | set(STATS_COMPONENTS) and {1, 63, 64, 65} <= set(SV_COMPONENTS)


# ------------------------------------------------------------------------------------------------ helpers
def _models(k, d, n_models, seed):
    """n_models diagonal GMMs (S, K) / (S, K, D): distinct means and variances per model."""
    from speech_signal_processing_b200 import synth

    ws, mus, vs = [], [], []
    for s in range(n_models):
        w, mu, var = synth.synth_ubm(k, d, seed=seed + s)
        ws.append(w)
        mus.append(mu)
        vs.append(var * (1.0 + 0.3 * s))
    return np.stack(ws), np.stack(mus), np.stack(vs)


def _frames(w, mu, var, lens, seed):
    from speech_signal_processing_b200 import synth

    x = synth.sample_gmm(w, mu, var, max(sum(lens), 1), seed=seed)[: sum(lens)]
    return x, np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


def frame_bound_terms(x, w, mu, var):
    """Per frame, max over the components of sum_d |x mu / var| + x^2 / (2 var) + |const| + 1 (float64)."""
    x = np.asarray(x, dtype=np.float64)
    prec = 1.0 / var
    const = np.log(w) - 0.5 * (x.shape[1] * ogmm.LOG_2PI + (mu * mu * prec).sum(axis=1)) + 0.5 * np.log(prec).sum(axis=1)
    terms = np.abs(x) @ np.abs(mu * prec).T + 0.5 * (x * x) @ prec.T + np.abs(const)[None] + 1.0
    return terms.max(axis=1)


def _check_scores(got, lse, x, offs, w, mu, var, u, what):
    """Utterance scores (n_utts, S) and per-frame log-likelihoods (S, T) against the oracle within the frame bound;
    returns the largest error as a multiple of u * terms (the constant the bound must exceed)."""
    worst = 0.0
    for s in range(len(w)):
        ref = ogmm.score_samples(x, w[s], mu[s], var[s])
        unit = u * frame_bound_terms(x, w[s], mu[s], var[s])
        err = np.abs(lse[s].astype(np.float64) - ref)
        worst = max(worst, float((err / unit).max()))
        assert (err <= C_BOUND * unit).all(), (what, s, float((err / unit).max()))
        for j in range(len(offs) - 1):
            lo, hi = offs[j], offs[j + 1]
            if hi == lo:
                continue
            e = abs(got[j, s] - ref[lo:hi].mean())
            assert e <= C_BOUND * unit[lo:hi].mean(), (what, s, j, e)
    return worst


# ------------------------------------------------------------------------------------------------ scoring
@pytest.mark.gpu
@pytest.mark.parametrize("d", SCORE_WIDTHS)
def test_scoring_rungs_at_every_tensor_width(d):
    """fp32, tf32, tf32x2 and tf32x3 at the tensor widths; K cycles through 1, 2, 127, 129 (a diagonal of D x K)."""
    import torch

    import speech_signal_processing_b200 as ssp

    k = SCORE_COMPONENTS[SCORE_WIDTHS.index(d) % len(SCORE_COMPONENTS)]
    w, mu, var = _models(k, d, 2, seed=10 * d + k)
    x, offs = _frames(w[0], mu[0], var[0], UTT_LENS, seed=d)
    ms = ssp.ModelSet(w, mu, var)
    feats = torch.as_tensor(x, device=ms.device)
    report = []
    for precision in ("fp32", "tf32", "tf32x2", "tf32x3"):
        got, lse = ms.score(feats, offs, precision=precision, want_frame_lse=True)
        c = _check_scores(got.cpu().numpy(), lse.cpu().numpy(), x, offs, w, mu, var, U[precision], precision)
        report.append(f"{precision} {c:.2f}")
    print(f"D {d} K {k}: largest error / (u * terms): " + ", ".join(report))


@pytest.mark.gpu
@pytest.mark.parametrize("d", SIMT_WIDTHS)
def test_cuda_core_widths_scoring_and_statistics(d):
    """D > 39: fp32 scoring and ssp_gmm_stats on the CUDA-core kernels (DP = 64 and 80 included)."""
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    k = SCORE_COMPONENTS[SIMT_WIDTHS.index(d) % len(SCORE_COMPONENTS)]
    w, mu, var = _models(k, d, 2, seed=20 * d + k)
    x, offs = _frames(w[0], mu[0], var[0], UTT_LENS, seed=d)
    ms = ssp.ModelSet(w, mu, var)
    feats = torch.as_tensor(x, device=ms.device)
    got, lse = ms.score(feats, offs, precision="fp32", want_frame_lse=True)
    c = _check_scores(got.cpu().numpy(), lse.cpu().numpy(), x, offs, w, mu, var, U["fp32"], "fp32")
    print(f"D {d} K {k}: largest error / (u * terms): fp32 {c:.2f}")
    seg_x, seg = _frames(w[0], mu[0], var[0], SEG_LENS + [300], seed=d + 1)
    ms1 = ssp.ModelSet(w[:1], mu[:1], var[:1])
    _lib.load().ssp_reset_launch_count()
    stats = ms1.stats(torch.as_tensor(seg_x, device=ms.device), seg)
    assert set(_lib.launch_log()) == EM_SIMT_KERNELS, _lib.launch_log()
    _check_stats(stats, seg_x, seg, lambda s: (w[0], mu[0], var[0]))


# ------------------------------------------------------------------------------------------------ statistics
def _check_stats(stats, x, seg, model_of):
    """N, F, S, loglik per segment against the oracle.  A posterior g_tc is off by its FP16 rounding (2^-11 of itself)
    and by the error of its logit and of the frame's log-likelihood (each within C_BOUND * u * terms_t): a statistic
    sum_t g_tc v_t within sum_t g_tc (e_t |v_t| + X_FLOOR), e_t = 2 * 2^-11 + 2 * C_BOUND * u * terms_t.  The N of all components
    sums to the segment length (a padded frame would add one).  Returns the largest log-likelihood error in units of
    u * terms."""
    n, f, s, ll = (t.cpu().numpy() for t in stats)
    worst = 0.0
    for i in range(len(seg) - 1):
        xs = x[seg[i] : seg[i + 1]].astype(np.float64)
        ln = len(xs)
        if ln == 0:
            assert np.all(n[i] == 0) and np.all(f[i] == 0) and np.all(s[i] == 0) and ll[i] == 0
            continue
        w, mu, var = model_of(i)
        lse, g = ogmm.responsibilities(xs, w, mu, var)
        rn, rf, rs_ = g.sum(axis=0), g.T @ xs, g.T @ (xs * xs)
        terms = frame_bound_terms(xs, w, mu, var)
        ge = g * (2 * U_GAMMA + 2 * C_BOUND * U["stats"] * terms)[:, None]
        floor = 1e-9 * ln
        assert (np.abs(n[i] - rn) <= ge.sum(axis=0) + floor).all(), (i, np.abs(n[i] - rn).max())
        assert (np.abs(f[i] - rf) <= ge.T @ np.abs(xs) + X_FLOOR * rn[:, None] + floor).all(), (i, np.abs(f[i] - rf).max())
        assert (np.abs(s[i] - rs_) <= ge.T @ (xs * xs) + X_FLOOR * rn[:, None] + floor).all(), (i, np.abs(s[i] - rs_).max())
        assert abs(n[i].sum() - ln) <= 2 * U_GAMMA * ln
        assert abs(ll[i] - lse.sum()) <= C_BOUND * U["stats"] * terms.sum()
        worst = max(worst, abs(ll[i] - lse.sum()) / (U["stats"] * terms.sum()))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("k", STATS_COMPONENTS)
@pytest.mark.parametrize("d", STATS_WIDTHS)
def test_tensor_statistics_at_every_width(d, k):
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import _lib

    w, mu, var = _models(k, d, 1, seed=30 * d + k)
    lens = SEG_LENS + [300, 0]
    x, seg = _frames(w[0], mu[0] * 0.9, var[0] * 1.2, lens, seed=d + k)
    ms = ssp.ModelSet(w, mu, var)
    _lib.load().ssp_reset_launch_count()
    stats = ms.stats(torch.as_tensor(x, device=ms.device), seg)
    assert set(_lib.launch_log()) == EM_TENSOR_KERNELS, _lib.launch_log()
    c = _check_stats(stats, x, seg, lambda i: (w[0], mu[0], var[0]))
    print(f"D {d} K {k}: largest log-likelihood error / (u * terms): {c:.2f}")
    if k == 1:                                         # every posterior is 1: N is the segment length
        assert np.array_equal(stats[0].cpu().numpy()[:, 0], np.asarray(lens, dtype=np.float64))


@pytest.mark.gpu
def test_per_segment_model_statistics_at_the_width_edges():
    """ssp_gmm_stats with one model per segment (what fit_batch runs) at D = 1 and D = 39 against the oracle."""
    import torch

    import speech_signal_processing_b200 as ssp

    for d in (1, 39):
        lens = [64, 1, 65, 0, 300]
        w, mu, var = _models(129, d, len(lens), seed=40 + d)
        x, seg = _frames(w[0], mu[0], var[0], lens, seed=d)
        ms = ssp.ModelSet(w, mu, var)
        stats = ms.stats(torch.as_tensor(x, device=ms.device), seg)
        _check_stats(stats, x, seg, lambda i: (w[i], mu[i], var[i]))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 39])
def test_fit_batch_at_the_width_edges(d):
    """fit_batch (per-segment models, one statistics call per iteration) equals the per-model loop and, for one EM
    iteration, the float64 oracle's E + M step."""
    import speech_signal_processing_b200 as ssp

    k, lens = 4, [300, 64, 65]
    xs, inits = [], []
    for i, n in enumerate(lens):
        w, mu, var = _models(k, d, 1, seed=50 + i)
        xs.append(_frames(w[0], mu[0], var[0], [n], seed=60 + i)[0])
        inits.append((w[0], mu[0] + 0.2, np.ones_like(var[0])))
    kw = dict(covariance_type="diag", max_iter=1, weights_init=[a for a, _, _ in inits],
              means_init=[b for _, b, _ in inits], precisions_init=[1.0 / c for _, _, c in inits])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        batched = ssp.fit_batch(xs, n_components=k, **kw)
        looped = [ssp.GaussianMixture(n_components=k, covariance_type="diag", max_iter=1, weights_init=a, means_init=b,
                                      precisions_init=1.0 / c).fit(x) for x, (a, b, c) in zip(xs, inits)]
    eps = np.finfo(np.float32).eps
    for x, (a, b, c), gb, gl in zip(xs, inits, batched, looped):
        assert abs(gb.lower_bound_ - gl.lower_bound_) <= 1e-7 * abs(gl.lower_bound_)
        np.testing.assert_allclose(gb.means_, gl.means_, rtol=0, atol=1e-6)
        np.testing.assert_allclose(gb.covariances_, gl.covariances_, rtol=1e-5, atol=1e-8)
        n, f, s, ll = ogmm.suff_stats(x.astype(np.float64), a, b, c)
        rw, rmu, rvar = ogmm.m_step(n, f, s, 1e-6, eps)
        terms = frame_bound_terms(x, a, b, c)
        assert abs(gb.lower_bound_ - ll / len(x)) <= C_BOUND * U["stats"] * terms.mean()
        # the posteriors' FP16 rounding (2^-11 of each term) bounds the statistics, hence these parameters
        np.testing.assert_allclose(gb.weights_, rw, rtol=1e-3, atol=1e-6)
        assert (np.abs(gb.means_ - rmu) <= 1e-3 * (1 + np.abs(rmu))).all()
        np.testing.assert_allclose(gb.covariances_, rvar, rtol=1e-3, atol=1e-6)


# ------------------------------------------------------------------------------------------------ shared variance
@pytest.mark.gpu
@pytest.mark.parametrize("k", SV_COMPONENTS)
@pytest.mark.parametrize("d", SV_WIDTHS)
def test_shared_variance_kernel_at_every_width(d, k):
    """The per-model contraction has KS = roundup(D + 2, 16) columns and components come in tiles of 64.  Against
    the oracle (the speakers' differences from the reference carry 11-bit operands, the reference member itself is
    FP32 grade) and against expand() scored by the FP32 kernel."""
    import torch

    import speech_signal_processing_b200 as ssp
    from speech_signal_processing_b200 import synth

    w, mu, var = synth.synth_ubm(k, d, seed=70 + d + k)
    means = np.concatenate([synth.synth_speaker_means(mu, 2, seed=71 + d, shift=0.3), mu[None]])   # last = reference
    x, offs = _frames(w, means[0], var, UTT_LENS, seed=d + k)
    sms = ssp.SharedModelSet(w, var, means)
    feats = torch.as_tensor(x, device=sms.device)
    got, lse = sms.score(feats, offs, want_frame_lse=True)
    got, lse = got.cpu().numpy(), lse.cpu().numpy()
    W, V = np.tile(w, (3, 1)), np.tile(var, (3, 1, 1))
    worst = _check_scores(got[:, :2], lse[:2], x, offs, W[:2], means[:2], V[:2], U["tf32"], "shared variance")
    ref_c = _check_scores(got[:, 2:], lse[2:], x, offs, W[2:], means[2:], V[2:], U["sv_reference"], "reference member")
    gen, gen_lse = sms.expand().score(feats, offs, precision="fp32", want_frame_lse=True)
    _check_scores(gen.cpu().numpy(), gen_lse.cpu().numpy(), x, offs, W, means, V, U["fp32"], "expand fp32")
    unit = U["tf32"] * np.stack([frame_bound_terms(x, w, m, var) for m in means])
    assert (np.abs(lse - gen_lse.cpu().numpy()) <= 2 * C_BOUND * unit).all()
    print(f"D {d} K {k}: largest error / (u * terms): speakers {worst:.2f}, reference member {ref_c:.2f}")


# ------------------------------------------------------------------------------------------------ rejections
@pytest.mark.gpu
def test_rejections_beyond_each_width_limit():
    import torch

    import speech_signal_processing_b200 as ssp

    w, mu, var = _models(8, 40, 2, seed=80)
    x, offs = _frames(w[0], mu[0], var[0], [5, 7], seed=80)
    ms = ssp.ModelSet(w, mu, var)
    feats = torch.as_tensor(x, device=ms.device)
    for precision in ("tf32", "tf32x2", "tf32x3"):       # the tensor scoring rungs stop at D = 39
        with pytest.raises(NotImplementedError, match="contraction"):
            ms.score(feats, offs, precision=precision)
    w81, mu81, var81 = _models(8, 81, 1, seed=81)
    with pytest.raises(ValueError, match="D <= 80"):
        ssp.ModelSet(w81, mu81, var81)
    with pytest.raises(ValueError, match="D <= 39"):
        ssp.SharedModelSet(w[0], var[0], mu)
    # per-segment models need the tensor statistics kernels: at D = 40 ssp_gmm_stats refuses them cleanly ...
    with pytest.raises(NotImplementedError, match="per-segment models"):
        ms.stats(feats, offs)
    # ... so fit_batch trains such models one by one, with the result of the per-model loop
    kw = dict(covariance_type="diag", max_iter=2, weights_init=w[0], means_init=mu[0], precisions_init=1.0 / var[0])
    x2, seg2 = _frames(w[0], mu[0], var[0], [40, 40], seed=82)
    parts = [x2[: seg2[1]], x2[seg2[1] :]]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        batched = ssp.fit_batch(parts, n_components=8, **kw)
        looped = [ssp.GaussianMixture(n_components=8, **kw).fit(p) for p in parts]
    for a, b in zip(batched, looped):     # (float64 atomics: the same sums in another order)
        assert abs(a.lower_bound_ - b.lower_bound_) <= 1e-12 * abs(b.lower_bound_)
        np.testing.assert_allclose(a.means_, b.means_, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(a.covariances_, b.covariances_, rtol=1e-9, atol=1e-12)
