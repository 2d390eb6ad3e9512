"""The public entry points on every input form they accept, against float64, and on every form they refuse.

The kernel suites feed the kernels what the library builds for itself: a contiguous float32 buffer on the current
device, on the default stream, with offsets that are a prefix sum from 0.  Callers also pass their own device tensors
(``(feats, offsets)`` tuples, ``ModelSet`` / ``SharedModelSet`` features, ``FrontEnd.extract_device`` PCM and ``out``).
Here:

- accepted forms reach the kernels and give the float64 oracle's numbers at the bounds the kernel suites derive
  (``test_gpu_gmm_widths``, ``test_gpu_posteriors``, ``test_gpu_frontend_paths``, ``test_gpu_dtw_shapes``): features
  4 bytes past a 16-byte boundary, a side stream whose writes are still in flight, every input form of
  ``GaussianMixture``, PCM offsets that do not start at 0, ``identify_pcm`` with split and unsplit batches, and
  workspaces at the weakest alignment the C ABI accepts;
- refused forms (float64, strided, host or other-device tensors, bad offsets, strided PCM, a wrong ``out``, a misaligned
  workspace) raise before anything is launched: ``ssp_launch_count`` does not move.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import dtw as odtw
from oracle import frontend as ofe
from oracle import gmm as ogmm
from test_gpu_dtw_shapes import RTOL as DTW_RTOL
from test_gpu_frontend_paths import check as check_ceps
from test_gpu_frontend_paths import kernel_of, load_path
from test_gpu_frontend_paths import reference as fe_reference
from test_gpu_gmm_widths import U, _check_scores, _check_stats, _frames, _models
from test_gpu_posteriors import MARGIN, SIMT, TENSOR
from test_gpu_posteriors import check as check_post

pytestmark = pytest.mark.gpu

RUNGS = ("fp32", "tf32", "tf32x2", "tf32x3")
UTT_LENS = [1, 127, 128, 129, 300]
SEG_LENS = [0, 1, 63, 64, 65, 300]
# ~10 ms of GPU time at the B200's clock: the side stream's write of the inputs is still running when the entry point
# enqueues its kernels, so a kernel put on any other stream would read the buffer before it holds the frames
SLEEP_CYCLES = 20_000_000


@pytest.fixture(scope="module")
def torch():
    import torch

    from speech_signal_processing_b200 import _lib

    _lib.load()
    torch.cuda.set_device(0)
    return torch


def ssp_mod():
    import speech_signal_processing_b200 as ssp

    return ssp


def launches():
    from speech_signal_processing_b200 import _lib

    return _lib.launch_count()


def reset_log():
    from speech_signal_processing_b200 import _lib

    _lib.load().ssp_reset_launch_count()


def launch_log():
    from speech_signal_processing_b200 import _lib

    return set(_lib.launch_log())


def off16(torch, x, dev="cuda:0"):
    """``x`` as a (T, D) float32 device tensor whose base sits 4 bytes past a 16-byte boundary: a row range of a
    flat buffer, NaN around it."""
    flat = torch.full((x.size + 8,), float("nan"), dtype=torch.float32, device=dev)
    v = flat[1 : 1 + x.size].view(x.shape)
    v.copy_(torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32)))
    assert v.data_ptr() % 16 == 4 and v.is_contiguous()
    return v


def shared_set(k, d, seed):
    """Weights (K,), variances (K, D), means (3, K, D): two speakers shifted from a UBM whose means are the last set."""
    from speech_signal_processing_b200 import synth

    w, mu, var = synth.synth_ubm(k, d, seed=seed)
    return w, var, np.concatenate([synth.synth_speaker_means(mu, 2, seed=seed + 1, shift=0.3), mu[None]])


def check_shared(got, lse, x, offs, w, var, means):
    W, V = np.tile(w, (len(means), 1)), np.tile(var, (len(means), 1, 1))
    _check_scores(got[:, :-1], lse[:-1], x, offs, W[:-1], means[:-1], V[:-1], U["tf32"], "shared variance")
    _check_scores(got[:, -1:], lse[-1:], x, offs, W[-1:], means[-1:], V[-1:], U["sv_reference"], "reference member")


# ================================================================================================ accepted forms
@pytest.mark.parametrize("d", [13, 39, 40])
def test_features_4_bytes_past_a_16_byte_boundary(torch, d):
    """Every GMM kernel reads frames from a base that is only 4-byte aligned (what a row range such as the chunks of
    ``predict_proba`` gives): the four scoring rungs, the shared-variance kernel, statistics and posteriors on the tensor
    path (D <= 39) and the CUDA-core path (D > 39)."""
    ssp = ssp_mod()
    k = 64
    w, mu, var = _models(k, d, 2, seed=400 + d)
    x, offs = _frames(w[0], mu[0], var[0], UTT_LENS, seed=d)
    ms = ssp.ModelSet(w, mu, var)
    feats = off16(torch, x)
    for precision in RUNGS if d <= 39 else ("fp32",):
        got, lse = ms.score(feats, offs, precision=precision, want_frame_lse=True)
        c = _check_scores(got.cpu().numpy(), lse.cpu().numpy(), x, offs, w, mu, var, U[precision], precision)
        print(f"D {d} {precision}: largest error / (u * terms) {c:.2f}")
    if d <= 39:
        sw, svar, smeans = shared_set(k, d, seed=410 + d)
        xs, soffs = _frames(sw, smeans[0], svar, UTT_LENS, seed=d + 1)
        got, lse = ssp.SharedModelSet(sw, svar, smeans).score(off16(torch, xs), soffs, want_frame_lse=True)
        check_shared(got.cpu().numpy(), lse.cpu().numpy(), xs, soffs, sw, svar, smeans)
    xg, seg = _frames(w[0], mu[0], var[0], SEG_LENS, seed=d + 2)
    ms1 = ssp.ModelSet(w[:1], mu[:1], var[:1])
    fg = off16(torch, xg)
    c = _check_stats(ms1.stats(fg, seg), xg, seg, lambda i: (w[0], mu[0], var[0]))
    print(f"D {d} statistics: largest log-likelihood error / (u * terms) {c:.2f}")
    kernels = TENSOR if d <= 39 else SIMT
    for mode in ("resp", "labels", "both"):
        reset_log()
        g, lab, lse = ms1.posteriors(fg, seg, resp=mode != "labels", labels=mode != "resp")
        assert launch_log() == kernels[mode], launch_log()
        check_post(f"D {d} {mode}", None if g is None else g.cpu().numpy(), None if lab is None else lab.cpu().numpy(),
                   xg, w[0], mu[0], var[0], None if lse is None else lse.cpu().numpy())


@pytest.mark.parametrize("d", [13, 40])
def test_dtw_from_features_4_bytes_past_a_16_byte_boundary(torch, d):
    ssp = ssp_mod()
    rs = np.random.RandomState(d)
    q_lens, r_lens = [1, 17, 40], [5, 33, 64, 2]
    q = rs.standard_normal((sum(q_lens), d)).astype(np.float32)
    r = rs.standard_normal((sum(r_lens), d)).astype(np.float32)
    qo, ro = np.concatenate([[0], np.cumsum(q_lens)]), np.concatenate([[0], np.cumsum(r_lens)])
    Q = [q[a:b] for a, b in zip(qo[:-1], qo[1:])]
    R = [r[a:b] for a, b in zip(ro[:-1], ro[1:])]
    for dist in ("euclidean", "sqeuclidean", "cityblock"):
        got = ssp.dtw_matrix((off16(torch, q), qo), (off16(torch, r), ro), dist)
        want = odtw.dtw_matrix([s.astype(np.float64) for s in Q], [s.astype(np.float64) for s in R], dist)
        rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-30)
        assert rel.max() <= DTW_RTOL, (dist, rel.max())
        np.testing.assert_array_equal(got, ssp.dtw_matrix(Q, R, dist))


# ------------------------------------------------------------------------------------------------ side stream
def _as_host(out):
    import torch

    return [o.cpu().numpy() if isinstance(o, torch.Tensor) else np.asarray(o) for o in out if o is not None]


def _run(torch, fn, side):
    """fn() on the default stream, or on a fresh side stream behind a spin kernel; fn writes its inputs with torch ops
    on that stream first (nothing synchronises before the entry point enqueues its work)."""
    cur = torch.cuda.current_stream()
    s = torch.cuda.Stream() if side else cur
    s.wait_stream(cur)
    with torch.cuda.stream(s):
        if side:
            torch.cuda._sleep(SLEEP_CYCLES)
        out = _as_host(fn())
    s.synchronize()
    return out


def _stream_cases(torch, d):
    """name -> (fn, exact): every public entry point that takes device frames or PCM.  ``exact``: the result is
    reproducible bit for bit (the statistics sum posteriors with double-precision atomics: their order varies)."""
    ssp = ssp_mod()
    from speech_signal_processing_b200 import synth

    dev = torch.device("cuda:0")
    k = 64
    w, mu, var = _models(k, d, 3, seed=500 + d)
    x, offs = _frames(w[0], mu[0], var[0], UTT_LENS, seed=d)
    xg, seg = _frames(w[0], mu[0], var[0], SEG_LENS, seed=d + 1)
    src_x, src_g = torch.as_tensor(x, device=dev), torch.as_tensor(xg, device=dev)
    src_p = [torch.as_tensor(a, device=dev) for a in (w, mu, var)]
    ubm = ssp.GaussianMixture.from_params(w[2], mu[2], var[2])
    speakers = [ssp.GaussianMixture.from_params(w[i], mu[i], var[i]) for i in range(2)]

    def fresh(t):
        return t.clone()   # a torch op on the current stream writes the buffer the entry point reads

    def model_set():
        return ssp.ModelSet(*(fresh(t) for t in src_p))   # the pack kernel and its range-flag read-back on this stream

    cases = {}
    for precision in RUNGS if d <= 39 else ("fp32",):
        cases[f"ModelSet.score {precision}"] = (
            lambda p=precision: model_set().score(fresh(src_x), offs, precision=p, want_frame_lse=True), True)
    cases["score_matrix"] = (lambda: [ssp.score_matrix((fresh(src_x), offs), model_set(), precision="fp32")], True)
    cases["identify"] = (lambda: ssp.identify((fresh(src_x), offs), speakers, ubm, precision="fp32"), True)
    one = [fresh(t[:1]) for t in src_p]
    cases["ModelSet.stats"] = (lambda: ssp.ModelSet(*(fresh(t) for t in one)).stats(fresh(src_g), seg), False)
    cases["ModelSet.posteriors"] = (
        lambda: ssp.ModelSet(*(fresh(t) for t in one)).posteriors(fresh(src_g), seg, resp=True, labels=True), True)
    cases["map_adapt"] = (lambda: ssp.map_adapt(ubm, (fresh(src_g), seg), adapt=("means", "weights", "variances")), False)
    if d <= 39:
        sw, svar, smeans = shared_set(k, d, seed=510 + d)
        src_s = [torch.as_tensor(a, device=dev) for a in (sw, svar, smeans)]
        cases["SharedModelSet.score"] = (
            lambda: ssp.SharedModelSet(*(fresh(t) for t in src_s)).score(fresh(src_x), offs, want_frame_lse=True), True)
        cases["map_enrol + score"] = (
            lambda: ssp.map_enrol(ubm, (fresh(src_g), seg)).score(fresh(src_x), offs, want_frame_lse=True), False)
    q_offs = np.array([0, 1, 128, 257, 557])
    cases["dtw_matrix"] = (lambda: [ssp.dtw_matrix((fresh(src_x[:557]), q_offs), (fresh(src_x[1:129]), [0, 128]))], True)
    cases["dtw_identify"] = (
        lambda: ssp.dtw_identify((fresh(src_x[:557]), q_offs), (fresh(src_x[1:129]), [0, 1, 128]), [7, 8]), True)
    sigs = [synth.synth_utterance(s, 0, n) for s, n in enumerate((16000, 4001, 400))]
    pcm = torch.as_tensor(np.concatenate(sigs), device=dev)
    soff = np.concatenate([[0], np.cumsum([len(s) for s in sigs])])
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True)
    cases["FrontEnd.extract_device"] = (lambda: fe.extract_device(fresh(pcm), soff, want_log_energy=True), True)
    if d == 39:
        host = torch.as_tensor(np.concatenate(sigs)).pin_memory()
        ms3 = ssp.ModelSet(w, mu, var)
        cases["identify_pcm"] = (lambda: [ssp.identify_pcm(host, soff, fe, ms3, ubm_index=2, min_split_frames=1)[0]], True)
    return cases


@pytest.mark.parametrize("d", [13, 39, 40])
def test_every_entry_point_on_a_side_stream(torch, d):
    """All work is enqueued on the caller's current stream (ssp_b200.h: "all work is enqueued on `stream`"), the pack
    entry points' FP16-range read-back included: on a side stream whose write of the inputs is still in flight, every
    entry point gives the default stream's results, bit for bit where the computation is reproducible (DESIGN 4.1), and
    to 1e-12 relative where double-precision atomics sum the statistics."""
    for name, (fn, exact) in _stream_cases(torch, d).items():
        want = _run(torch, fn, side=False)
        got = _run(torch, fn, side=True)
        assert len(got) == len(want), name
        for a, b in zip(got, want):
            assert np.isfinite(b).all(), name
            if exact:
                np.testing.assert_array_equal(a, b, err_msg=name)
            else:
                np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12 * np.abs(b).max(), err_msg=name)


# ------------------------------------------------------------------------------------------------ GaussianMixture
@pytest.mark.parametrize("d", [13, 40])
def test_gaussian_mixture_takes_every_array_form(torch, d):
    """sklearn's surface converts whatever it is given: numpy float64 / float32 / Fortran order, CPU torch, CUDA float64
    and a strided CUDA view all give the contiguous float32 CUDA tensor's results bit for bit, and those match float64."""
    ssp = ssp_mod()
    k = 32
    w, mu, var = _models(k, d, 1, seed=600 + d)
    w, mu, var = w[0], mu[0], var[0]
    x, _ = _frames(w, mu, var, [700], seed=d)
    gm = ssp.GaussianMixture.from_params(w, mu, var)
    dev = torch.device("cuda:0")
    wide = torch.full((len(x), d + 3), float("nan"), device=dev)
    wide[:, 1 : d + 1] = torch.as_tensor(x, device=dev)
    forms = {
        "numpy float64": x.astype(np.float64),
        "numpy float32": x,
        "numpy Fortran order": np.asfortranarray(x),
        "CPU torch": torch.as_tensor(x),
        "CUDA float64": torch.as_tensor(x.astype(np.float64), device=dev),
        "strided CUDA view": wide[:, 1 : d + 1],
    }
    base = torch.as_tensor(x, device=dev)

    def results(X):
        return gm.score(X), gm.score_samples(X), gm.predict_proba(X), gm.predict(X)

    want = results(base)
    _check_scores(np.array([[want[0]]]), want[1][None], x, np.array([0, len(x)]), w[None], mu[None], var[None], U["fp32"],
                  "GaussianMixture.score")
    check_post(f"D {d} GaussianMixture", want[2], want[3], x, w, mu, var)
    for name, X in forms.items():
        got = results(X)
        assert got[0] == want[0], name
        for a, b in zip(got[1:], want[1:]):
            np.testing.assert_array_equal(a, b, err_msg=name)


# ------------------------------------------------------------------------------------------------ front-end
@pytest.mark.parametrize("path", ["direct", "staged-int16", "float32"])
def test_extract_device_with_offsets_that_do_not_start_at_0(torch, path):
    """identify_pcm hands the tail of a split batch to extract_device as offsets into the whole buffer; each load path
    of the sidekit kernel (int16 from a 4-byte boundary, int16 from an odd sample, float32) reads from there."""
    ssp = ssp_mod()
    from speech_signal_processing_b200 import synth

    recipe = ssp.sidekit_recipe()
    lens = [4003, 4000, 401, 4008]
    sigs = [synth.synth_utterance(s, 1, n) for s, n in enumerate(lens)]
    lead = 4321                                            # samples before the first utterance: odd
    cat = np.concatenate([np.zeros(lead, dtype=np.int16)] + sigs)
    offs = lead + np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    dev = torch.device("cuda:0")
    if path == "float32":
        pcm = torch.as_tensor(cat.astype(np.float32), device=dev)
    else:
        shift = 0 if path == "direct" else 1               # a base 2 bytes past a 4-byte boundary
        buf = torch.zeros(len(cat) + 8, dtype=torch.int16, device=dev)
        pcm = buf[shift : shift + len(cat)]
        pcm.copy_(torch.as_tensor(cat))
    sk = kernel_of(recipe) == "frontend512_kernel"
    paths = {load_path(sk, pcm.element_size(), pcm.data_ptr(), int(o)) for o in offs[:-1]}
    assert paths == {"direct": {"direct-even", "direct-odd"}, "staged-int16": {"staged-int16"},
                     "float32": {"staged-float"}}[path], paths
    fe = ssp.FrontEnd(recipe)
    reset_log()
    feats, foffs, le = fe.extract_device(pcm, offs, want_log_energy=True)
    assert launch_log() == {kernel_of(recipe, int(path == "float32"))}, launch_log()
    feats = feats.cpu().numpy()
    for i, s in enumerate(sigs):
        want, _ = fe_reference(recipe, s)
        check_ceps(f"offset start {path}", feats[foffs[i] : foffs[i + 1]], want)


@pytest.mark.parametrize("host", ["numpy", "pinned torch"])
def test_identify_pcm_split_unsplit_and_offset(torch, host):
    """Split and unsplit batches, with a first sample offset above 0, from pageable numpy and pinned torch PCM: the
    decisions of the device path (extract_device + score) and of float64 features and scores."""
    ssp = ssp_mod()
    from speech_signal_processing_b200 import synth

    k, d, n_spk = 32, 39, 4
    w, mu, var = synth.synth_ubm(k, d, seed=7, spread=0.8)
    means = np.concatenate([synth.synth_speaker_means(mu, n_spk, seed=8, shift=0.4), mu[None]])
    ms = ssp.ModelSet(np.tile(w, (n_spk + 1, 1)), means, np.tile(var, (n_spk + 1, 1, 1)))
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True)
    sigs = [synth.synth_utterance(s % n_spk, s, 8000 + 997 * s) for s in range(9)]
    lead = 777
    cat = np.concatenate([synth.synth_utterance(0, 99, lead)] + sigs)
    offs = lead + np.concatenate([[0], np.cumsum([len(s) for s in sigs])]).astype(np.int64)
    hpcm = cat if host == "numpy" else torch.as_tensor(cat).pin_memory()
    # float64: features of the recipe, float64 scores, LLR against the UBM (model n_spk)
    llr = np.array([[ogmm.score(ofe.features(s, preset="sidekit", delta_order=2, cmvn=True), w, m, var) for m in means]
                    for s in sigs])
    llr = llr[:, :n_spk] - llr[:, n_spk:]
    top = np.sort(llr, axis=1)
    clear = top[:, -1] - top[:, -2] > MARGIN
    assert clear.sum() >= len(sigs) - 1
    feats, foffs, _ = fe.extract_device(torch.as_tensor(cat, device="cuda:0"), offs)
    scores, _ = ms.score(feats, foffs)
    device_dec = (scores[:, :n_spk] - scores[:, n_spk:]).argmax(dim=1).cpu().numpy()
    for split in (1, 1 << 40):
        n_head = ssp.ubm.split_for_overlap(fe.frame_counts(np.diff(offs)), 0.1, split)
        assert (n_head > 0) == (split == 1)
        dec, total = ssp.identify_pcm(hpcm, offs, fe, ms, ubm_index=n_spk, min_split_frames=split)
        assert total == int(foffs[-1])
        np.testing.assert_array_equal(dec.numpy(), device_dec)
        np.testing.assert_array_equal(dec.numpy()[clear], llr.argmax(axis=1)[clear])


# ------------------------------------------------------------------------------------------------ workspaces
@pytest.mark.parametrize("d", [13, 40])
def test_workspace_at_the_weakest_accepted_alignment(torch, d):
    """A statistics / posterior workspace 16 bytes into a larger uint8 buffer (the alignment ssp_gmm_stats and
    ssp_gmm_posteriors require) gives the results of an allocation-aligned one."""
    ssp = ssp_mod()
    from speech_signal_processing_b200.mixture import StatsWorkspace

    w, mu, var = _models(64, d, 1, seed=700 + d)
    x, seg = _frames(w[0], mu[0], var[0], SEG_LENS, seed=d)
    ms = ssp.ModelSet(w, mu, var)
    feats = torch.as_tensor(x, device="cuda:0")
    dims = ms.dims
    lib = ms.lib
    nbytes = max(int(lib.ssp_gmm_stats_workspace_bytes(C.byref(dims), len(x), len(seg) - 1)),
                 int(lib.ssp_gmm_posteriors_workspace_bytes(C.byref(dims), len(x), len(seg) - 1)))
    big = torch.empty(nbytes + 64, dtype=torch.uint8, device="cuda:0")
    sliced = StatsWorkspace(ms.device)
    sliced.buf = big[16 : 16 + nbytes]
    assert sliced.buf.data_ptr() % 32 == 16                 # 16-byte aligned and no more (the allocation is 512-aligned)
    results = []
    for ws in (StatsWorkspace(ms.device), sliced):
        stats = ms.stats(feats, seg, workspace=ws)
        _check_stats(stats, x, seg, lambda i: (w[0], mu[0], var[0]))
        post = ms.posteriors(feats, seg, resp=True, labels=True, workspace=ws)
        results.append(([t.cpu().numpy() for t in stats], [t.cpu().numpy() for t in post]))
    assert sliced.buf.data_ptr() == big.data_ptr() + 16    # the workspace was used, not reallocated
    (stats_a, post_a), (stats_b, post_b) = results
    for a, b in zip(post_b, post_a):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(stats_b, stats_a):                      # double-precision atomics: the order of the sums varies
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12 * np.abs(b).max())


# ================================================================================================ refused forms
def refused(fn, exc=ValueError, match=None):
    """fn raises exc and launches nothing."""
    before = launches()
    with pytest.raises(exc, match=match):
        fn()
    assert launches() == before


def test_refused_features_launch_nothing(torch):
    ssp = ssp_mod()
    d, k = 13, 64
    w, mu, var = _models(k, d, 2, seed=800)
    x, offs = _frames(w[0], mu[0], var[0], UTT_LENS, seed=800)
    dev = torch.device("cuda:0")
    ms, ms1 = ssp.ModelSet(w, mu, var), ssp.ModelSet(w[:1], mu[:1], var[:1])
    sw, svar, smeans = shared_set(k, d, seed=801)
    sms = ssp.SharedModelSet(sw, svar, smeans)
    ubm = ssp.GaussianMixture.from_params(w[0], mu[0], var[0])
    ubm._model_set()
    speakers = [ssp.GaussianMixture.from_params(w[1], mu[1], var[1])]
    good = torch.as_tensor(x, device=dev)
    wide = torch.zeros((len(x), d + 1), device=dev)
    wide[:, :d] = good
    forms = {
        "CUDA float64": (good.double(), offs, "float32"),
        "column slice": (wide[:, :d], offs, "contiguous"),
        "transpose": (good.T.contiguous().T, offs, "contiguous"),
        "CPU tensor": (good.cpu(), offs, "cpu"),
        "offsets decrease": (good, np.array([0, 200, 100, 685]), "offsets"),
        "offsets start above 0": (good, offs + 1, "offsets"),
        "offsets end beyond the rows": (good[:-1], offs, "offsets"),
    }
    for name, (f, o, match) in forms.items():
        refused(lambda: ms.score(f, o), match=match)
        refused(lambda: ms1.stats(f, o), match=match)
        refused(lambda: ms1.posteriors(f, o), match=match)
        refused(lambda: sms.score(f, o), match=match)
        refused(lambda: ssp.score_matrix((f, o), ms), match=match)
        refused(lambda: ssp.identify((f, o), speakers, ubm), match=match)
        refused(lambda: ssp.map_adapt(ubm, (f, o)), match=match)
        refused(lambda: ssp.map_enrol(ubm, (f, o)), match=match)
        refused(lambda: ssp.dtw_matrix((f, o), [x[:5]]), match=match)
        refused(lambda: ssp.dtw_identify([x[:5]], (f, o), np.arange(len(o) - 1)), match=match)
    # DTW keeps its own rule on top: every sequence has a frame
    refused(lambda: ssp.dtw_matrix((good, np.array([0, 0, len(x)])), [x[:5]]), match="every sequence")


def test_refused_pcm_and_out_launch_nothing(torch):
    ssp = ssp_mod()
    from speech_signal_processing_b200 import synth

    fe = ssp.FrontEnd(ssp.sidekit_recipe(), delta_order=2, cmvn=True)
    dev = torch.device("cuda:0")
    left, right = synth.synth_utterance(0, 0, 8000), synth.synth_utterance(1, 1, 8000)
    stereo = torch.as_tensor(np.stack([left, right], 1), device=dev)
    pcm = stereo[:, 0].contiguous()
    offs = np.array([0, 3000, 8000])
    total = int(fe.frame_counts(np.diff(offs)).sum())
    refused(lambda: fe.extract_device(stereo[:, 0], offs), match="contiguous")
    refused(lambda: fe.extract_device(stereo, offs), match="1-D")
    refused(lambda: fe.extract_device(pcm.cpu(), offs), match="cuda")
    refused(lambda: fe.extract_device(pcm.to(torch.int32), offs), TypeError)
    refused(lambda: fe.extract_device(pcm, np.array([0, 3000, 8001])), match="sample_offsets")
    refused(lambda: fe.extract_device(pcm, np.array([0, 3000, 2000])), match="sample_offsets")
    refused(lambda: fe.extract_device(pcm, np.array([-1, 3000])), match="sample_offsets")
    refused(lambda: fe.extract_device(pcm, np.array([0.0, 3000.0])), match="sample_offsets")
    for out in (torch.empty((total - 1, fe.out_dim), device=dev), torch.empty((total, fe.out_dim), dtype=torch.float64, device=dev),
                torch.empty((total, fe.out_dim)), torch.empty((fe.out_dim, total), device=dev).T):
        refused(lambda: fe.extract_device(pcm, offs, out=out), match="out")
    # the accepted forms of the same PCM: a contiguous copy, and an exact out
    out = torch.empty((total, fe.out_dim), device=dev)
    got, _, _ = fe.extract_device(pcm, offs, out=out)
    assert got.data_ptr() == out.data_ptr() and bool(torch.isfinite(out).all())


def test_misaligned_workspace_is_refused_at_the_c_abi(torch):
    """Workspaces 4, 8 or 12 bytes off a 16-byte boundary are SSP_EINVAL for ssp_gmm_stats, ssp_gmm_posteriors and
    ssp_gmm_score_shared, with real device buffers, before any launch; through ModelSet that is a ValueError."""
    ssp = ssp_mod()
    from speech_signal_processing_b200 import _lib
    from speech_signal_processing_b200.mixture import StatsWorkspace

    d, k = 13, 64
    w, mu, var = _models(k, d, 1, seed=900)
    x, seg = _frames(w[0], mu[0], var[0], SEG_LENS, seed=900)
    ms = ssp.ModelSet(w, mu, var)
    lib = ms.lib
    dev = torch.device("cuda:0")
    feats = torch.as_tensor(x, device=dev)
    d_seg = torch.as_tensor(seg, device=dev)
    n_segs, total = len(seg) - 1, len(x)
    nbytes = int(lib.ssp_gmm_stats_workspace_bytes(C.byref(ms.dims), total, n_segs))
    big = torch.empty(nbytes + 64, dtype=torch.uint8, device=dev)
    lse = torch.empty(total, device=dev)
    n, f, s, ll = (torch.zeros(m, dtype=torch.float64, device=dev) for m in (k, k * d, k * d, n_segs))
    resp = torch.empty((total, k), device=dev)
    sw, svar, smeans = shared_set(k, d, seed=901)
    sms = ssp.SharedModelSet(sw, svar, smeans)
    scores = torch.empty((n_segs, 3), dtype=torch.float64, device=dev)
    for off in (4, 8, 12):
        ws = big.data_ptr() + off
        before = launches()
        assert lib.ssp_gmm_stats(feats.data_ptr(), d_seg.data_ptr(), n_segs, total, ms.pack.data_ptr(), C.byref(ms.dims),
                                 lse.data_ptr(), n.data_ptr(), f.data_ptr(), s.data_ptr(), ll.data_ptr(), ws, nbytes, 0,
                                 _lib.stream_ptr()) == -1
        assert lib.ssp_gmm_posteriors(feats.data_ptr(), d_seg.data_ptr(), n_segs, total, ms.pack.data_ptr(),
                                      C.byref(ms.dims), resp.data_ptr(), None, lse.data_ptr(), ws, nbytes, 0,
                                      _lib.stream_ptr()) == -1
        assert lib.ssp_gmm_score_shared(feats.data_ptr(), d_seg.data_ptr(), n_segs, total, sms.pack.data_ptr(),
                                        C.byref(sms.dims), scores.data_ptr(), None, ws, nbytes, _lib.stream_ptr()) == -1
        assert b"16-byte aligned" in lib.ssp_last_error()
        assert launches() == before
        bad = StatsWorkspace(ms.device)
        bad.buf = big[off : off + nbytes]
        refused(lambda: ms.stats(feats, seg, workspace=bad), match="16-byte aligned")
        refused(lambda: ms.posteriors(feats, seg, workspace=bad), match="16-byte aligned")


def test_features_on_another_gpu_are_refused(torch):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ssp = ssp_mod()
    w, mu, var = _models(16, 13, 1, seed=1000)
    x, offs = _frames(w[0], mu[0], var[0], [5, 7], seed=1000)
    ms = ssp.ModelSet(w, mu, var, device="cuda:1")
    feats = torch.as_tensor(x, device="cuda:0")
    refused(lambda: ms.score(feats, offs), match="cuda:0")
    refused(lambda: ms.stats(feats, offs), match="cuda:0")
    refused(lambda: ms.posteriors(feats, offs), match="cuda:0")
    refused(lambda: ssp.score_matrix((feats, offs), ms, device="cuda:1"), match="cuda:0")
    fe = ssp.FrontEnd(ssp.sidekit_recipe(), device="cuda:1")
    refused(lambda: fe.extract_device(torch.zeros(4000, dtype=torch.int16, device="cuda:0"), [0, 4000]), match="cuda")
